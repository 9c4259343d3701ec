// Metropolis-Hastings on the TRUE forward model (MCMC.model_mh, ces/sample.py:121-196), whole chains on the device.
//
// The reference runs one chain, one Python iteration per proposal: proposal (random walk current + scales z, or pCN
// sqrt(1 - beta^2) current + sqrt(beta) scales z; :198-202), one forward evaluation enka.G(proposal, model) (:168), the
// misfit Phi = yg . solve(2 Gamma, yg) minus prior.logpdf unless pCN (:170-176), and the accept test
// log(uniform) < Phi_current - Phi_proposal (:182).  19 570 it/s on the linear model in the notebooks (BASELINE.md).
//
// Here one WARP owns one chain and the loop never leaves the kernel: lanes split the p rows of the proposal and of the
// prior term and the k rows of the forward map and of Gamma^-1 yg, the two quadratic forms are fixed-order shuffle
// reductions, and every state of the chain goes straight to the samples array in HBM.  Several chains run side by
// side (one warp each, four warps per CTA).
//
// Random numbers.  Chain 0 can consume the caller's numpy stream itself: the kernel carries the MT19937 state of
// numpy's global RandomState (624 words, position, cached Gaussian) and restates its legacy generators -- next_double =
// (a >> 5, b >> 6) / 2^53, the polar Box-Muller of legacy_gauss with its cached second variate, uniform() -- so it draws
// exactly the variates normal(0, 1, p) and uniform() would have produced, in the reference's order, and hands the
// advanced state back (integer-exact: the rejection loop and the consumption count depend only on exact IEEE
// products; the variates themselves can differ from glibc's in the last bit of log).  The other chains use Philox
// keyed by (seed, chain, iteration).
#include "kernels.h"
#include "chains.cuh"
#include "rng.cuh"

namespace ces {

namespace {

constexpr int MH_P_MAX = 32, MH_K_MAX = 64, MH_WARPS = 4;
constexpr uint32_t MH_TAG = 0x4d48u;        // Philox counter word of this sampler ("MH")

struct MhArgs {
    int p, k, n_mcmc, n_chains, map_kind, pcn, use_mt;
    double beta;
    const double* A; long long lda; const double* b;      // lineal / lineal_log (device)
    double par0, par1;                                      // elliptic / banana
    const double* y;            // k
    const double* Ginv2;        // k x k, (2 Gamma)^-1
    const double* mu;           // p     prior mean
    const double* Pinv;         // p x p prior precision
    const double* scales;       // p x p
    const double* start;        // n_chains x p  first state of every chain
    const double* phi_point;    // n_chains x p  point whose Phi is the initial Phi_current (the reference evaluates it at the
                                //               ensemble mean even when it resumes from the last sample, :141-166)
    double* samples;            // n_chains x (n_mcmc + 1) x p
    int* accepted;              // n_chains
    uint32_t* mt;               // 624 + 2 words: key, pos, has_gauss ; double cached gauss in mt_gauss
    double* mt_gauss;
    unsigned long long seed;
};

// Phi(x) for the point in xs[0..p) (shared memory of this warp): misfit (+ prior term unless pCN).  gs / ygs: scratch.
__device__ double mh_phi(const MhArgs& a, const double* xs, double* gs, double* ygs, double* ds, int lane) {
    const int p = a.p, k = a.k;
    // forward map (ces/utils.py:25-31, 39-42, 72-89, 116-122)
    if (a.map_kind == CES_MAP_LINEAL || a.map_kind == CES_MAP_LINEAL_LOG) {
        for (int m = lane; m < k; m += 32) {
            double s = 0.0;
            for (int q = 0; q < p; ++q) s = fma(a.A[(size_t)m * a.lda + q], a.map_kind == CES_MAP_LINEAL_LOG ? exp(xs[q]) : xs[q], s);
            gs[m] = a.b ? s + a.b[m] : s;
        }
    } else if (lane == 0) {
        const double u1 = xs[0], u2 = xs[1];
        if (a.map_kind == CES_MAP_ELLIPTIC) {
            const double e = exp(-u1), x1 = a.par0, x2 = a.par1;
            gs[0] = (u2 * x1) + (e * (-x1 * x1 + x1) * 0.5);
            gs[1] = (u2 * x2) + (e * (-x2 * x2 + x2) * 0.5);
        } else {
            gs[0] = u1 * a.par0;
            gs[1] = u2 / a.par0 - a.par1 * (u1 * u1 + a.par0 * a.par0);
        }
    }
    __syncwarp();
    for (int m = lane; m < k; m += 32) ygs[m] = gs[m] - a.y[m];
    __syncwarp();
    double part = 0.0;
    for (int m = lane; m < k; m += 32) {
        double t = 0.0;
        for (int n = 0; n < k; ++n) t = fma(a.Ginv2[(size_t)m * k + n], ygs[n], t);
        part = fma(ygs[m], t, part);            // yg . solve(2 Gamma, yg)   (:170, :174)
    }
    double phi = warp_sum(part);
    if (!a.pcn) {                               // - prior.logpdf(x) up to its constant (cancels in the ratio; :171-176)
        for (int q = lane; q < p; q += 32) ds[q] = xs[q] - a.mu[q];
        __syncwarp();
        double pp = 0.0;
        for (int q = lane; q < p; q += 32) {
            double t = 0.0;
            for (int n = 0; n < p; ++n) t = fma(a.Pinv[(size_t)q * p + n], ds[n], t);
            pp = fma(0.5 * ds[q], t, pp);
        }
        phi += warp_sum(pp);
    }
    __syncwarp();
    return phi;
}

__global__ void __launch_bounds__(32 * MH_WARPS) mh_chain_kernel(const MhArgs a) {
    __shared__ double sh[MH_WARPS][3 * MH_P_MAX + 2 * MH_K_MAX + MH_P_MAX + 2];
    __shared__ uint32_t mt_key[624];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int chain = blockIdx.x * MH_WARPS + warp;
    if (chain >= a.n_chains) return;
    double* cur = sh[warp];                 // p
    double* prop = cur + MH_P_MAX;          // p
    double* ds = prop + MH_P_MAX;           // p
    double* gs = ds + MH_P_MAX;             // k
    double* ygs = gs + MH_K_MAX;            // k
    double* zs = ygs + MH_K_MAX;            // p normals + 1 uniform
    const int p = a.p;
    const bool mt_chain = a.use_mt && chain == 0;
    Mt rng;
    rng.key = mt_key; rng.pos = 0; rng.has_gauss = 0; rng.gauss = 0.0;
    if (mt_chain) {
        for (int i = lane; i < 624; i += 32) mt_key[i] = a.mt[i];
        rng.pos = (int)a.mt[624];
        rng.has_gauss = (int)a.mt[625];
        rng.gauss = a.mt_gauss[0];
    }
    // The reference's banana model draws np.random.normal(0, 1, [2]) in EVERY evaluation, noise switched on or not
    // (ces/utils.py:122: flag_noise * chol(Gamma).dot(normal)): the stream chain consumes those two variates where the
    // reference does -- before the first evaluation and between the proposal's normals and the accept test's uniform.
    const int forward_draws = a.map_kind == CES_MAP_BANANA ? 2 : 0;
    if (mt_chain && lane == 0)
        for (int q = 0; q < forward_draws; ++q) (void)mt_gauss(rng);
    for (int q = lane; q < p; q += 32) prop[q] = a.phi_point[(size_t)chain * p + q];
    __syncwarp();
    double phi_cur = mh_phi(a, prop, gs, ygs, ds, lane);
    double* out = a.samples + (size_t)chain * (a.n_mcmc + 1) * p;
    for (int q = lane; q < p; q += 32) { cur[q] = a.start[(size_t)chain * p + q]; out[q] = cur[q]; }
    __syncwarp();
    const double a_cur = a.pcn ? sqrt(1.0 - a.beta * a.beta) : 1.0, a_z = a.pcn ? sqrt(a.beta) : 1.0;     // :198-202
    int acc = 0;
    for (int it = 0; it < a.n_mcmc; ++it) {
        // ---- z ~ N(0, I_p), u ~ U(0, 1), in the order np.random.normal(0, 1, p) then np.random.uniform() draw them
        if (mt_chain) {
            if (lane == 0) {
                for (int q = 0; q < p; ++q) zs[q] = mt_gauss(rng);
                for (int q = 0; q < forward_draws; ++q) (void)mt_gauss(rng);
                zs[p] = mt_double(rng);
            }
        } else {
            for (int q2 = lane; 2 * q2 < p; q2 += 32) {             // Box-Muller pairs (2 q2, 2 q2 + 1)
                philox_normal_pair(a.seed, it, chain, q2, MH_TAG, &zs[2 * q2], 2 * q2 + 1 < p ? &zs[2 * q2 + 1] : nullptr);
            }
            if (lane == 31) zs[p] = philox_accept_uniform(a.seed, it, chain, MH_TAG);
        }
        __syncwarp();
        for (int q = lane; q < p; q += 32) {
            double s = 0.0;
            for (int n = 0; n < p; ++n) s = fma(a.scales[(size_t)q * p + n], zs[n], s);      // np.matmul(scales, z)
            prop[q] = a.pcn ? a_cur * cur[q] + a_z * s : cur[q] + s;
        }
        __syncwarp();
        const double phi_prop = mh_phi(a, prop, gs, ygs, ds, lane);
        const bool take = log(zs[p]) < phi_cur - phi_prop;         // :182  (NaN compares false: the proposal is rejected)
        if (take) {
            for (int q = lane; q < p; q += 32) cur[q] = prop[q];
            phi_cur = phi_prop;
            ++acc;
        }
        __syncwarp();
        for (int q = lane; q < p; q += 32) out[(size_t)(it + 1) * p + q] = cur[q];
    }
    if (lane == 0) a.accepted[chain] = acc;
    if (mt_chain) {
        __syncwarp();
        for (int i = lane; i < 624; i += 32) a.mt[i] = mt_key[i];
        if (lane == 0) { a.mt[624] = (uint32_t)rng.pos; a.mt[625] = (uint32_t)rng.has_gauss; a.mt_gauss[0] = rng.gauss; }
    }
}

}  // namespace

}  // namespace ces

using namespace ces;

extern "C" int ces_mcmc_model_mh(void* stream, int map_kind, int64_t p, int64_t k, const double* A_dev, int64_t lda,
                                 const double* b_dev, const double* params_host, const double* y_host,
                                 const double* Ginv2_host, const double* mu_host, const double* Pinv_host,
                                 const double* scales_host, int pcn, double beta, int64_t n_mcmc, int64_t n_chains,
                                 const double* start_host, const double* phi_point_host, uint32_t* mt_state_host,
                                 double* mt_gauss_host, uint64_t seed, double* samples_host, int32_t* accepted_host) {
    const ChainHost h{"ces_mcmc_model_mh", n_mcmc, n_chains, pcn, y_host, scales_host, mu_host, Pinv_host, start_host,
                      phi_point_host, mt_state_host, mt_gauss_host, seed, samples_host, accepted_host};
    CES_TRY(chain_check(h));
    if (p < 1 || p > MH_P_MAX || k < 1 || k > MH_K_MAX || !Ginv2_host)
        return fail(CES_ERR_INVALID, "ces_mcmc_model_mh: needs 1 <= p <= 32, 1 <= k <= 64 and non-null arguments%s", "");
    if (map_kind < CES_MAP_LINEAL || map_kind > CES_MAP_BANANA) return fail(CES_ERR_INVALID, "ces_mcmc_model_mh: unknown map kind%s", "");
    if ((map_kind == CES_MAP_LINEAL || map_kind == CES_MAP_LINEAL_LOG) ? !A_dev : (!params_host || p != 2 || k != 2))
        return fail(CES_ERR_INVALID, "ces_mcmc_model_mh: the map needs A (lineal) or two parameters with p = k = 2%s", "");
    ChainRun run(h, (int)p, static_cast<cudaStream_t>(stream));
    MhArgs a;
    a.p = (int)p; a.k = (int)k; a.n_mcmc = (int)n_mcmc; a.n_chains = (int)n_chains; a.map_kind = map_kind; a.pcn = pcn ? 1 : 0;
    a.use_mt = mt_state_host != nullptr;
    a.beta = beta;
    a.A = A_dev; a.lda = lda; a.b = b_dev;
    a.par0 = params_host ? params_host[0] : 0.0; a.par1 = params_host ? params_host[1] : 0.0;
    a.seed = seed;
    CES_TRY(run.build([&] {
        a.y = run.put(y_host, k);
        a.Ginv2 = run.put(Ginv2_host, (size_t)k * k);
        a.mu = run.put(mu_host, p);
        a.Pinv = run.put(Pinv_host, (size_t)p * p);
        a.scales = run.put(scales_host, (size_t)p * p);
        a.start = run.put(start_host, (size_t)n_chains * p);
        a.phi_point = run.put(phi_point_host, (size_t)n_chains * p);
        a.samples = run.samples;
        a.accepted = run.accepted;
        a.mt = run.mt;
        a.mt_gauss = run.mt_gauss;
    }));
    mh_chain_kernel<<<(unsigned)ceil_div(n_chains, MH_WARPS), 32 * MH_WARPS, 0, run.st>>>(a);
    CES_LAUNCHED(1);
    return run.copy_back();
}
