// Metropolis-Hastings on the Darcy forward model (MCMC.model_mh with ces_b200.darcy.model / model_trunc): n_chains chains
// stepped in lockstep through the batched Darcy solver of darcy.cu, on the model's stream.
//
// The reference (ces/sample.py:121-196) calls model(theta) once per proposal.  Here one step evaluates every chain's
// proposal in one batched forward call, and nothing in the step loop waits for the host:
//   dmh_noise_kernel     Z (p x n_chains) ~ N(0, I) and u ~ U(0, 1) per chain (mh_chain_draw of rng.cuh: chain 0 consumes
//                        numpy's MT19937 stream, the others draw Philox noise keyed by (seed, step, chain)); prop <- cur
//   prop = b cur + a scales Z           one DMMA GEMM, a / b through the epilogue's alpha / beta (random walk a = b = 1,
//                                       pCN a = sqrt(beta), b = sqrt(1 - beta^2), ces/sample.py:198-202)
//   Gp = G(prop)                        darcy_forward_async: KL GEMM, exp, splines, CG, gather (n_obs x n_chains)
//   dmh_resid_kernel     R = Gp - y and, for the random walk, D = prop - mu; the step's largest CG iteration count to a
//                        device array
//   W = Ginv2 R,  Pz = Pinv D           DMMA GEMMs, Ginv2 = (2 Gamma)^-1 (no limit on n_obs or p)
//   chain_accept_kernel  (chains.cuh, with DmhPhi) Phi = sum R o W (+ 1/2 sum D o Pz), accept when log u < Phi_cur - Phi
//                        (a NaN rejects), state to the device samples buffer
// The initial Phi_cur is evaluated the same way at phi_point (the ensemble mean for chain 0, also on resume).  After the
// loop the iteration counts come back once: if any solve reached max_iter the call fails and names the first such step,
// and nothing else is copied back.  Otherwise samples, acceptances and numpy's generator state are copied back once.
#include <cstdio>
#include <vector>
#include "kernels.h"
#include "chains.cuh"
#include "rng.cuh"

namespace ces {

namespace {

constexpr int DMH_THREADS = CHAIN_THREADS;
constexpr uint32_t DMH_TAG = 0x4452u;       // Philox counter word of this sampler ("DR")

// Phi of chain c at the evaluated point: misfit sum_i R_i W_i, plus 1/2 sum_q D_q Pz_q unless pCN.  Fixed order.
struct DmhPhi {
    int k, pcn;
    const double *R, *W;        // k x ld
    const double *D, *Pz;       // p x ld
    __device__ double operator()(const ChainState& a, int c) const {
        double phi = 0.0;
        for (int i = 0; i < k; ++i) phi = fma(R[(size_t)i * a.ld + c], W[(size_t)i * a.ld + c], phi);
        if (!pcn) {
            double pp = 0.0;
            for (int q = 0; q < a.p; ++q) pp = fma(D[(size_t)q * a.ld + c], Pz[(size_t)q * a.ld + c], pp);
            phi = fma(0.5, pp, phi);
        }
        return phi;
    }
};

struct DarcyMhArgs {
    ChainState ch;
    int k, pcn;
    const double* y;            // k
    const double* mu;           // p   (random walk)
    double* Z;                  // p x ld   standard normals of the step
    double* D;                  // p x ld   prop - mu
    double* Pz;                 // p x ld   Pinv D
    double* Gp;                 // k x ld   forward map at prop
    double* R;                  // k x ld   Gp - y
    double* W;                  // k x ld   Ginv2 R
    int* step_iters;            // n_mcmc + 1: largest CG iteration count of the initial evaluation and of every step
    const int* iters;           // the Darcy model's device counters ([0]: largest count of its last forward call)
    DmhPhi phi() const { return DmhPhi{k, pcn, R, W, D, Pz}; }
};

// Block 0 stages numpy's generator state in shared memory for chain 0: the draws and the twist of the 624-word key are a
// long dependent sequence of accesses in one thread, at shared-memory rather than L2 latency.
__global__ void __launch_bounds__(DMH_THREADS) dmh_noise_kernel(const DarcyMhArgs a, int it) {
    __shared__ uint32_t mt_s[626];
    const ChainState& ch = a.ch;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const bool mt_block = ch.use_mt && blockIdx.x == 0;
    if (mt_block) {
        for (int i = threadIdx.x; i < 626; i += blockDim.x) mt_s[i] = ch.mt[i];
        __syncthreads();
    }
    if (c < ch.n_chains) {
        ch.u[c] = mh_chain_draw(ch.p, it, c, (mt_block && c == 0) ? mt_s : nullptr, ch.mt_gauss, ch.seed, DMH_TAG, a.Z + c,
                                (int)ch.ld);
        for (int q = 0; q < ch.p; ++q) ch.prop[(size_t)q * ch.ld + c] = ch.cur[(size_t)q * ch.ld + c];
    }
    if (mt_block) {
        __syncthreads();
        for (int i = threadIdx.x; i < 626; i += blockDim.x) ch.mt[i] = mt_s[i];
    }
}

// rows [0, k): R = Gp - y; rows [k, k + p): D = prop - mu (random walk only).  The forward call just before it on the
// stream left its largest CG iteration count in iters[0]: kept as step_iters[slot].
__global__ void __launch_bounds__(DMH_THREADS) dmh_resid_kernel(const DarcyMhArgs a, int slot) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
    if (c == 0 && row == 0) a.step_iters[slot] = a.iters[0];
    if (c >= a.ch.n_chains) return;
    const long long ld = a.ch.ld;
    if (row < a.k) {
        a.R[(size_t)row * ld + c] = a.Gp[(size_t)row * ld + c] - a.y[row];
    } else {
        const int q = row - a.k;
        a.D[(size_t)q * ld + c] = a.ch.prop[(size_t)q * ld + c] - a.mu[q];
    }
}

struct DmhOperators {
    const double *Ginv2, *Pinv, *scales;
    int64_t ldk, ldp;
};

// forward map, residuals (iteration count into step_iters[slot]) and the two quadratic forms' GEMMs at the points in prop
int dmh_evaluate(DarcyModel* m, const DarcyMhArgs& a, const DmhOperators& o, double tol, int max_iter, int slot) {
    cudaStream_t st = darcy_shape(m).st;
    const ChainState& ch = a.ch;
    CES_TRY(darcy_forward_async(m, ch.prop, ch.ld, ch.n_chains, a.Gp, ch.ld, 0, tol, max_iter));
    const dim3 grid((unsigned)ceil_div(ch.n_chains, DMH_THREADS), (unsigned)(a.k + (a.pcn ? 0 : ch.p)));
    dmh_resid_kernel<<<grid, DMH_THREADS, 0, st>>>(a, slot);
    CES_LAUNCHED(1);
    GemmCall w;                                     // W = Ginv2 R
    w.a_mode = A_MK; w.b_mode = B_KN;
    w.M = a.k; w.N = ch.n_chains; w.K = a.k;
    w.A = o.Ginv2; w.lda = o.ldk; w.B = a.R; w.ldb = ch.ld; w.C = a.W; w.ldc = ch.ld;
    CES_TRY(gemm(st, w));
    if (!a.pcn) {                                   // Pz = Pinv D
        GemmCall pz;
        pz.a_mode = A_MK; pz.b_mode = B_KN;
        pz.M = ch.p; pz.N = ch.n_chains; pz.K = ch.p;
        pz.A = o.Pinv; pz.lda = o.ldp; pz.B = a.D; pz.ldb = ch.ld; pz.C = a.Pz; pz.ldc = ch.ld;
        CES_TRY(gemm(st, pz));
    }
    return CES_OK;
}

int dmh_run(DarcyModel* m, const DarcyMhArgs& a, const DmhOperators& o, double beta, double tol, int max_iter) {
    cudaStream_t st = darcy_shape(m).st;
    const ChainState& ch = a.ch;
    const unsigned blocks = (unsigned)ceil_div(ch.n_chains, DMH_THREADS);
    CES_TRY(dmh_evaluate(m, a, o, tol, max_iter, 0));      // Phi_cur at phi_point (uploaded into prop)
    chain_init_kernel<<<blocks, DMH_THREADS, 0, st>>>(ch, a.phi());
    CES_LAUNCHED(1);
    GemmCall g;                                     // prop = b cur + a scales Z, prop pre-filled with cur
    g.a_mode = A_MK; g.b_mode = B_KN;
    g.M = ch.p; g.N = ch.n_chains; g.K = ch.p;
    g.A = o.scales; g.lda = o.ldp; g.B = a.Z; g.ldb = ch.ld; g.C = ch.prop; g.ldc = ch.ld;
    g.alpha = a.pcn ? sqrt(beta) : 1.0;
    g.beta = a.pcn ? sqrt(1.0 - beta * beta) : 1.0;
    for (int it = 0; it < ch.n_mcmc; ++it) {
        dmh_noise_kernel<<<blocks, DMH_THREADS, 0, st>>>(a, it);
        CES_LAUNCHED(1);
        CES_TRY(gemm(st, g));
        CES_TRY(dmh_evaluate(m, a, o, tol, max_iter, it + 1));
        chain_accept_kernel<<<blocks, DMH_THREADS, 0, st>>>(ch, a.phi(), it);
        CES_LAUNCHED(1);
    }
    // every solve converged?  Only then do the results (and numpy's advanced generator state) go back
    std::vector<int> iters((size_t)ch.n_mcmc + 1);
    CES_CUDA(cudaMemcpyAsync(iters.data(), a.step_iters, iters.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaStreamSynchronize(st));
    const int limit = darcy_max_iter(m, max_iter);
    for (size_t s = 0; s < iters.size(); ++s)
        if (iters[s] >= limit) {
            char msg[256];
            if (s == 0)
                snprintf(msg, sizeof(msg), "ces_darcy_mh: CG reached max_iter = %d without converging at the initial point "
                         "(step 0)", limit);
            else
                snprintf(msg, sizeof(msg), "ces_darcy_mh: CG reached max_iter = %d without converging in step %lld of %d",
                         limit, (long long)s, ch.n_mcmc);
            return fail(CES_ERR_STATE, "%s", msg);
        }
    return CES_OK;
}

}  // namespace

}  // namespace ces

using namespace ces;

extern "C" int ces_darcy_mh(void* model, double tol, int max_iter, const double* y_host, const double* Ginv2_host,
                            const double* mu_host, const double* Pinv_host, const double* scales_host, int pcn, double beta,
                            int64_t n_mcmc, int64_t n_chains, const double* start_host, const double* phi_point_host,
                            uint32_t* mt_state_host, double* mt_gauss_host, uint64_t seed, double* samples_host,
                            int32_t* accepted_host) {
    const ChainHost h{"ces_darcy_mh", n_mcmc, n_chains, pcn, y_host, scales_host, mu_host, Pinv_host, start_host,
                      phi_point_host, mt_state_host, mt_gauss_host, seed, samples_host, accepted_host};
    CES_TRY(chain_check(h));
    if (!Ginv2_host) return fail(CES_ERR_INVALID, "ces_darcy_mh: needs non-null arguments%s", "");
    DarcyModel* m = static_cast<DarcyModel*>(model);
    if (!m) return fail(CES_ERR_INVALID, "ces_darcy_mh: null model%s", "");
    const DarcyShape sh = darcy_shape(m);
    if (sh.n_obs < 1) return fail(CES_ERR_INVALID, "ces_darcy_mh: the model was created without an obs_index%s", "");
    const int p = sh.p, k = sh.n_obs;
    const int64_t ld = padded_ld(n_chains), ldk = padded_ld(k), ldp = padded_ld(p);
    ChainRun run(h, p, sh.st);
    DarcyMhArgs a;
    a.k = k; a.pcn = pcn ? 1 : 0;
    a.iters = sh.iters;
    DmhOperators o;
    o.ldk = ldk; o.ldp = ldp;
    CES_TRY(run.build([&] {
        a.ch = chain_state(run, ld);
        a.y = run.put(y_host, k);
        o.Ginv2 = run.put2d(Ginv2_host, k, k, ldk);
        a.mu = run.put(pcn ? nullptr : mu_host, p);
        o.Pinv = run.put2d(pcn ? nullptr : Pinv_host, p, p, ldp);
        o.scales = run.put2d(scales_host, p, p, ldp);
        a.Z = run.take((size_t)p * ld);
        a.D = run.take((size_t)p * ld);
        a.Pz = run.take((size_t)p * ld);
        a.Gp = run.take((size_t)k * ld);
        a.R = run.take((size_t)k * ld);
        a.W = run.take((size_t)k * ld);
        a.step_iters = run.take<int>((size_t)n_mcmc + 1);
    }));
    CES_TRY(dmh_run(m, a, o, beta, tol, max_iter));
    return run.copy_back();
}
