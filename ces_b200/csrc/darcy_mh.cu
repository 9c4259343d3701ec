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
//   dmh_resid_kernel     R = Gp - y and, for the random walk, D = prop - mu
//   W = Ginv2 R,  Pz = Pinv D           DMMA GEMMs, Ginv2 = (2 Gamma)^-1 (no limit on n_obs or p)
//   dmh_accept_kernel    Phi = sum R o W (+ 1/2 sum D o Pz), accept when log u < Phi_cur - Phi (a NaN rejects), state to
//                        the device samples buffer, and the step's largest CG iteration count to a device array
// The initial Phi_cur is evaluated the same way at phi_point (the ensemble mean for chain 0, also on resume).  After the
// loop the iteration counts come back once: if any solve reached max_iter the call fails and names the first such step,
// and nothing else is copied back.  Otherwise samples, acceptances and numpy's generator state are copied back once.
#include <climits>
#include <cstdio>
#include <vector>
#include "kernels.h"
#include "rng.cuh"

namespace ces {

namespace {

constexpr int DMH_THREADS = 128;
constexpr uint32_t DMH_TAG = 0x4452u;       // Philox counter word of this sampler ("DR")

struct DarcyMhArgs {
    int p, k, n_mcmc, n_chains, pcn, use_mt;
    long long ld;               // pitch of the p x n_chains / n_obs x n_chains state arrays (one chain per column)
    const double* y;            // k
    const double* mu;           // p   (random walk)
    double* cur;                // p x ld   current states
    double* prop;               // p x ld   proposals (the evaluated points)
    double* Z;                  // p x ld   standard normals of the step
    double* D;                  // p x ld   prop - mu
    double* Pz;                 // p x ld   Pinv D
    double* Gp;                 // k x ld   forward map at prop
    double* R;                  // k x ld   Gp - y
    double* W;                  // k x ld   Ginv2 R
    double* u;                  // n_chains: the accept test's uniform of this step
    double* phi_cur;            // n_chains
    double* samples;            // n_chains x (n_mcmc + 1) x p
    int* accepted;              // n_chains
    int* step_iters;            // n_mcmc + 1: largest CG iteration count of the initial evaluation and of every step
    const int* iters;           // the Darcy model's device counters ([0]: largest count of its last forward call)
    uint32_t* mt;               // 624 key words, pos, has_gauss
    double* mt_gauss;
    unsigned long long seed;
};

// Phi of chain c at the evaluated point: misfit sum_i R_i W_i, plus 1/2 sum_q D_q Pz_q unless pCN.  Fixed order.
__device__ double dmh_phi(const DarcyMhArgs& a, int c) {
    double phi = 0.0;
    for (int i = 0; i < a.k; ++i) phi = fma(a.R[(size_t)i * a.ld + c], a.W[(size_t)i * a.ld + c], phi);
    if (!a.pcn) {
        double pp = 0.0;
        for (int q = 0; q < a.p; ++q) pp = fma(a.D[(size_t)q * a.ld + c], a.Pz[(size_t)q * a.ld + c], pp);
        phi = fma(0.5, pp, phi);
    }
    return phi;
}

// Block 0 stages numpy's generator state in shared memory for chain 0: the draws and the twist of the 624-word key are a
// long dependent sequence of accesses in one thread, at shared-memory rather than L2 latency.
__global__ void __launch_bounds__(DMH_THREADS) dmh_noise_kernel(const DarcyMhArgs a, int it) {
    __shared__ uint32_t mt_s[626];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const bool mt_block = a.use_mt && blockIdx.x == 0;
    if (mt_block) {
        for (int i = threadIdx.x; i < 626; i += blockDim.x) mt_s[i] = a.mt[i];
        __syncthreads();
    }
    if (c < a.n_chains) {
        a.u[c] = mh_chain_draw(a.p, it, c, (mt_block && c == 0) ? mt_s : nullptr, a.mt_gauss, a.seed, DMH_TAG, a.Z + c,
                               (int)a.ld);
        for (int q = 0; q < a.p; ++q) a.prop[(size_t)q * a.ld + c] = a.cur[(size_t)q * a.ld + c];
    }
    if (mt_block) {
        __syncthreads();
        for (int i = threadIdx.x; i < 626; i += blockDim.x) a.mt[i] = mt_s[i];
    }
}

// rows [0, k): R = Gp - y; rows [k, k + p): D = prop - mu (random walk only)
__global__ void __launch_bounds__(DMH_THREADS) dmh_resid_kernel(const DarcyMhArgs a) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, row = blockIdx.y;
    if (c >= a.n_chains) return;
    if (row < a.k) {
        a.R[(size_t)row * a.ld + c] = a.Gp[(size_t)row * a.ld + c] - a.y[row];
    } else {
        const int q = row - a.k;
        a.D[(size_t)q * a.ld + c] = a.prop[(size_t)q * a.ld + c] - a.mu[q];
    }
}

// Phi_cur at the evaluated points (phi_point), then cur <- start: state 0 of every chain
__global__ void __launch_bounds__(DMH_THREADS) dmh_init_kernel(const DarcyMhArgs a, const double* __restrict__ start) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chains) return;
    a.phi_cur[c] = dmh_phi(a, c);
    double* out = a.samples + (size_t)c * (a.n_mcmc + 1) * a.p;
    for (int q = 0; q < a.p; ++q) {
        const double v = start[(size_t)c * a.p + q];
        a.cur[(size_t)q * a.ld + c] = v;
        out[q] = v;
    }
    a.accepted[c] = 0;
    if (c == 0) a.step_iters[0] = a.iters[0];
}

__global__ void __launch_bounds__(DMH_THREADS) dmh_accept_kernel(const DarcyMhArgs a, int it) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chains) return;
    const double phi_prop = dmh_phi(a, c);
    const bool take = log(a.u[c]) < a.phi_cur[c] - phi_prop;          // ces/sample.py:182; NaN compares false: rejected
    double* out = a.samples + ((size_t)c * (a.n_mcmc + 1) + it + 1) * a.p;
    for (int q = 0; q < a.p; ++q) {
        double x = a.cur[(size_t)q * a.ld + c];
        if (take) {
            x = a.prop[(size_t)q * a.ld + c];
            a.cur[(size_t)q * a.ld + c] = x;
        }
        out[q] = x;
    }
    if (take) {
        a.phi_cur[c] = phi_prop;
        a.accepted[c] += 1;
    }
    if (c == 0) a.step_iters[it + 1] = a.iters[0];
}

struct DmhOperators {
    const double *Ginv2, *Pinv, *scales;
    int64_t ldk, ldp;
};

// forward map, residuals and the two quadratic forms' GEMMs at the points in a.prop
int dmh_evaluate(DarcyModel* m, const DarcyMhArgs& a, const DmhOperators& o, double tol, int max_iter) {
    cudaStream_t st = darcy_shape(m).st;
    CES_TRY(darcy_forward_async(m, a.prop, a.ld, a.n_chains, a.Gp, a.ld, 0, tol, max_iter));
    const dim3 grid((unsigned)ceil_div(a.n_chains, DMH_THREADS), (unsigned)(a.k + (a.pcn ? 0 : a.p)));
    dmh_resid_kernel<<<grid, DMH_THREADS, 0, st>>>(a);
    CES_LAUNCHED(1);
    GemmCall w;                                     // W = Ginv2 R
    w.a_mode = A_MK; w.b_mode = B_KN;
    w.M = a.k; w.N = a.n_chains; w.K = a.k;
    w.A = o.Ginv2; w.lda = o.ldk; w.B = a.R; w.ldb = a.ld; w.C = a.W; w.ldc = a.ld;
    CES_TRY(gemm(st, w));
    if (!a.pcn) {                                   // Pz = Pinv D
        GemmCall pz;
        pz.a_mode = A_MK; pz.b_mode = B_KN;
        pz.M = a.p; pz.N = a.n_chains; pz.K = a.p;
        pz.A = o.Pinv; pz.lda = o.ldp; pz.B = a.D; pz.ldb = a.ld; pz.C = a.Pz; pz.ldc = a.ld;
        CES_TRY(gemm(st, pz));
    }
    return CES_OK;
}

int dmh_run(DarcyModel* m, const DarcyMhArgs& a, const DmhOperators& o, double beta, double tol, int max_iter,
            const double* start, uint32_t* ibuf, uint32_t* mt_state_host, double* mt_gauss_host, double* samples_host,
            int32_t* accepted_host) {
    cudaStream_t st = darcy_shape(m).st;
    const unsigned blocks = (unsigned)ceil_div(a.n_chains, DMH_THREADS);
    CES_TRY(dmh_evaluate(m, a, o, tol, max_iter));          // Phi_cur at phi_point (uploaded into prop)
    dmh_init_kernel<<<blocks, DMH_THREADS, 0, st>>>(a, start);
    CES_LAUNCHED(1);
    GemmCall g;                                     // prop = b cur + a scales Z, prop pre-filled with cur
    g.a_mode = A_MK; g.b_mode = B_KN;
    g.M = a.p; g.N = a.n_chains; g.K = a.p;
    g.A = o.scales; g.lda = o.ldp; g.B = a.Z; g.ldb = a.ld; g.C = a.prop; g.ldc = a.ld;
    g.alpha = a.pcn ? sqrt(beta) : 1.0;
    g.beta = a.pcn ? sqrt(1.0 - beta * beta) : 1.0;
    for (int it = 0; it < a.n_mcmc; ++it) {
        dmh_noise_kernel<<<blocks, DMH_THREADS, 0, st>>>(a, it);
        CES_LAUNCHED(1);
        CES_TRY(gemm(st, g));
        CES_TRY(dmh_evaluate(m, a, o, tol, max_iter));
        dmh_accept_kernel<<<blocks, DMH_THREADS, 0, st>>>(a, it);
        CES_LAUNCHED(1);
    }
    // every solve converged?  Only then do the results (and numpy's advanced generator state) go back
    std::vector<int> iters((size_t)a.n_mcmc + 1);
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
                         limit, (long long)s, a.n_mcmc);
            return fail(CES_ERR_STATE, "%s", msg);
        }
    const size_t nsamp = (size_t)a.n_chains * (a.n_mcmc + 1) * a.p;
    CES_CUDA(cudaMemcpyAsync(samples_host, a.samples, nsamp * sizeof(double), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaMemcpyAsync(accepted_host, a.accepted, (size_t)a.n_chains * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (mt_state_host) {
        CES_CUDA(cudaMemcpyAsync(mt_state_host, ibuf, 626 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        CES_CUDA(cudaMemcpyAsync(mt_gauss_host, a.mt_gauss, sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CES_CUDA(cudaStreamSynchronize(st));
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
    if (!y_host || !Ginv2_host || !scales_host || !start_host || !phi_point_host || !samples_host || !accepted_host ||
        (!pcn && (!mu_host || !Pinv_host)) || (mt_state_host && !mt_gauss_host) || n_mcmc < 1 || n_mcmc >= INT_MAX ||
        n_chains < 1 || n_chains > (1 << 24))
        return fail(CES_ERR_INVALID, "ces_darcy_mh: needs n_mcmc >= 1, 1 <= n_chains <= 2^24 and non-null arguments%s", "");
    DarcyModel* m = static_cast<DarcyModel*>(model);
    if (!m) return fail(CES_ERR_INVALID, "ces_darcy_mh: null model%s", "");
    const DarcyShape sh = darcy_shape(m);
    if (sh.n_obs < 1) return fail(CES_ERR_INVALID, "ces_darcy_mh: the model was created without an obs_index%s", "");
    const int p = sh.p, k = sh.n_obs;
    cudaStream_t st = sh.st;
    const int64_t ld = padded_ld(n_chains), ldk = padded_ld(k), ldp = padded_ld(p);
    if ((double)n_chains * (double)(n_mcmc + 1) * p * sizeof(double) > 4e18)
        return fail(CES_ERR_NOMEM, "ces_darcy_mh: the samples buffer is too large%s", "");
    const size_t nsamp = (size_t)n_chains * (n_mcmc + 1) * p;
    auto r16 = [](size_t n) -> size_t { return (n + 15) / 16 * 16; };      // every sub-buffer 128-byte aligned (TMA)
    const size_t n_state = r16(k) + r16((size_t)k * ldk) + r16(p) + 2 * r16((size_t)p * ldp) + 5 * r16((size_t)p * ld) +
                           3 * r16((size_t)k * ld) + 2 * r16(ld) + r16(1) + r16((size_t)n_chains * p);
    double* dbuf = nullptr;
    uint32_t* ibuf = nullptr;
    if (cudaMalloc(&dbuf, (n_state + nsamp) * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        return fail(CES_ERR_NOMEM, "ces_darcy_mh: allocation failed%s", "");
    }
    if (cudaMalloc(&ibuf, (626 + (size_t)n_chains + (size_t)n_mcmc + 1) * sizeof(uint32_t)) != cudaSuccess) {
        cudaFree(dbuf);
        cudaGetLastError();
        return fail(CES_ERR_NOMEM, "ces_darcy_mh: allocation failed%s", "");
    }
    int s = CES_OK;
    do {
        if (cudaMemsetAsync(dbuf, 0, n_state * sizeof(double), st) != cudaSuccess) { s = fail(CES_ERR_CUDA, "ces_darcy_mh: upload failed%s", ""); break; }
        double* q = dbuf;
        auto take = [&](size_t cnt) -> double* { double* d = q; q += r16(cnt); return d; };
        auto put = [&](const double* src, size_t cnt) -> double* {
            double* d = take(cnt);
            if (src && s == CES_OK && cudaMemcpyAsync(d, src, cnt * sizeof(double), cudaMemcpyHostToDevice, st) != cudaSuccess) s = CES_ERR_CUDA;
            return d;
        };
        auto put2d = [&](const double* src, int rows, int cols, int64_t pitch) -> double* {
            double* d = take((size_t)rows * pitch);
            if (src && s == CES_OK && cudaMemcpy2DAsync(d, pitch * sizeof(double), src, cols * sizeof(double), cols * sizeof(double),
                                                        rows, cudaMemcpyHostToDevice, st) != cudaSuccess) s = CES_ERR_CUDA;
            return d;
        };
        // the p x n_chains state arrays hold one chain per column: transpose the row-per-chain phi_point
        std::vector<double> phiT((size_t)p * ld, 0.0);
        for (int64_t c = 0; c < n_chains; ++c)
            for (int d = 0; d < p; ++d) phiT[(size_t)d * ld + c] = phi_point_host[(size_t)c * p + d];
        DarcyMhArgs a;
        a.p = p; a.k = k; a.n_mcmc = (int)n_mcmc; a.n_chains = (int)n_chains; a.pcn = pcn ? 1 : 0;
        a.use_mt = mt_state_host != nullptr;
        a.ld = ld;
        DmhOperators o;
        o.ldk = ldk; o.ldp = ldp;
        a.y = put(y_host, k);
        o.Ginv2 = put2d(Ginv2_host, k, k, ldk);
        a.mu = put(pcn ? nullptr : mu_host, p);
        o.Pinv = put2d(pcn ? nullptr : Pinv_host, p, p, ldp);
        o.scales = put2d(scales_host, p, p, ldp);
        a.cur = take((size_t)p * ld);
        a.prop = put(phiT.data(), (size_t)p * ld);
        a.Z = take((size_t)p * ld);
        a.D = take((size_t)p * ld);
        a.Pz = take((size_t)p * ld);
        a.Gp = take((size_t)k * ld);
        a.R = take((size_t)k * ld);
        a.W = take((size_t)k * ld);
        a.u = take(ld);
        a.phi_cur = take(ld);
        a.mt_gauss = put(mt_state_host ? mt_gauss_host : nullptr, 1);
        const double* start = put(start_host, (size_t)n_chains * p);
        a.samples = q;
        a.mt = ibuf;
        a.accepted = reinterpret_cast<int*>(ibuf + 626);
        a.step_iters = reinterpret_cast<int*>(ibuf + 626 + n_chains);
        a.iters = sh.iters;
        a.seed = seed;
        if (s == CES_OK && mt_state_host &&
            cudaMemcpyAsync(ibuf, mt_state_host, 626 * sizeof(uint32_t), cudaMemcpyHostToDevice, st) != cudaSuccess)
            s = CES_ERR_CUDA;
        if (s != CES_OK) { s = fail(CES_ERR_CUDA, "ces_darcy_mh: upload failed%s", ""); break; }
        s = dmh_run(m, a, o, beta, tol, max_iter, start, ibuf, mt_state_host, mt_gauss_host, samples_host, accepted_host);
    } while (0);
    cudaStreamSynchronize(st);          // nothing may still use the buffers (also after a failed enqueue)
    cudaFree(dbuf);
    cudaFree(ibuf);
    return s;
}
