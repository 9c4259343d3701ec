// Emulate stage: exact Gaussian-process emulators of the whitened forward map (ces_b200/emulate.py) and
// Metropolis-Hastings chains through them (MCMC.emulator_mh).
//
// Model (one independent GP per whitened output i < k; training inputs X (p x n), outputs Y = T G - ybar (k x n)):
//   theta_i = [log sf2, log l_1..l_p, log sn2]                (sklearn's theta of C*RBF(ARD)+White, or C*Matern(ARD)+White)
//   D_d = (x_d - z_d)^2 / l_d^2,  r^2 = sum_d D_d,  k(x, z) = K_f(r) with the family fixed per model (ces_gp_set_kernel):
//             SE  sf2 exp(-r^2/2)          Matern12  sf2 exp(-r)
//             Matern32  sf2 (1 + sqrt3 r) exp(-sqrt3 r)          Matern52  sf2 (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r)
//   K = k(X, X) + (sn2 + jitter) I,  L = chol(K),  alpha = K^-1 y_i
//   LML     = -1/2 y_i^T alpha - sum log L_jj - n/2 log 2 pi
//   dLML/dtheta_j = 1/2 sum_ab W_ab dK_ab/dtheta_j,  W = alpha alpha^T - K^-1
//             dK/dlog sf2 = K_f,  dK/dlog l_d = sf2 g(r) D_d,  dK/dlog sn2 = sn2 I   (K_f: no noise, no jitter)
//             g(r): SE exp(-r^2/2) (so sf2 g = K_f),  Matern12 exp(-r) / r and 0 at r = 0 (sklearn's convention),
//                   Matern32 3 exp(-sqrt3 r),  Matern52 5/3 (1 + sqrt5 r) exp(-sqrt5 r)
//   mean_i(u) = ybar_i + k_i(u)^T alpha_i,   var_i(u) = max(sf2 - ||L_i^-1 k_i(u)||^2, 0)   (latent f, no sn2)
//   Phi(u)  = 1/2 sum_i (ytil_i - mean_i)^2 / (1 + var_i) + 1/2 sum_i log(1 + var_i)   [use_variance]
//             1/2 sum_i (ytil_i - mean_i)^2                                            [otherwise]
//
// Device layout.  Covariance blocks are assembled by one tile kernel batched over outputs on blockIdx.z, from the
// coordinates divided by the lengthscales and staged in shared memory (p <= 32).  The family is a template parameter
// of the covariance and gradient kernels, dispatched once per launch; r^2 always comes from direct differences (no
// |a|^2 + |b|^2 - 2 a.b expansion, which cancels near r = 0).  The factorisations are the DMMA
// Cholesky / triangular solves of chol.cu.  The gradient is one pass over the lower triangle of K that recomputes K_f
// on the fly and contracts it with W into p + 2 per-CTA partial sums, finished in fixed order by one more kernel: no
// atomics, so repeated calls are bit-identical (the L-BFGS fit relies on it).  Conditioning keeps L_i^-1 explicitly,
// stacked over outputs with n padded to the GEMM's 128-row box and zero padding, so that one prediction of m points is
//   K*_i (n x m, assembled)  ->  V_i = L_i^-1 K*_i (one batched lower-triangular DMMA GEMM)  ->  mean / var (column pass).
// A chain step is a propose kernel, that prediction for every chain's proposal at once, and an accept kernel; states go
// to a device samples buffer that is copied back once at the end.
#include <vector>
#include "kernels.h"
#include "chains.cuh"
#include "rng.cuh"

namespace ces {

namespace {

constexpr int GP_P_MAX = 32, GP_K_MAX = 64, GP_TB = 32, GP_PAD = GEMM_BM, GP_RHS_LD = 16;
constexpr int GP_PROPOSE_THREADS = 128;

__device__ __forceinline__ void stage_scaled(double (*s)[GP_TB + 1], const double* P, long long ld, int n0, int n, int p,
                                             const double* th) {
    for (int e = threadIdx.x; e < p * GP_TB; e += blockDim.x) {
        const int d = e / GP_TB, j = e % GP_TB;
        s[d][j] = (n0 + j < n) ? P[(size_t)d * ld + n0 + j] / exp(th[1 + d]) : 0.0;
    }
}

__device__ __forceinline__ double scaled_dist2(const double (*sa)[GP_TB + 1], const double (*sb)[GP_TB + 1], int r, int c, int p) {
    double s = 0.0;
    for (int d = 0; d < p; ++d) {
        const double t = sa[d][r] - sb[d][c];
        s = fma(t, t, s);
    }
    return s;
}

// The covariance family (CES_GP_*) as a function of the scaled squared distance r2 = r^2: gp_kf = K_f / sf2 and
// gp_g = g(r), the weight of D_d in dK/dlog l_d = sf2 g(r) D_d.  gp_g is not used for SE, where g = K_f / sf2.
constexpr double GP_SQRT3 = 1.7320508075688772935, GP_SQRT5 = 2.2360679774997896964;

template <int KIND> __device__ __forceinline__ double gp_kf(double r2);
template <> __device__ __forceinline__ double gp_kf<CES_GP_SE>(double r2) { return exp(-0.5 * r2); }
template <> __device__ __forceinline__ double gp_kf<CES_GP_MATERN12>(double r2) { return exp(-sqrt(r2)); }
template <> __device__ __forceinline__ double gp_kf<CES_GP_MATERN32>(double r2) {
    const double t = GP_SQRT3 * sqrt(r2);
    return (1.0 + t) * exp(-t);
}
template <> __device__ __forceinline__ double gp_kf<CES_GP_MATERN52>(double r2) {
    const double t = GP_SQRT5 * sqrt(r2);
    return (1.0 + t + t * t / 3.0) * exp(-t);
}

template <int KIND> __device__ __forceinline__ double gp_g(double r2);
template <> __device__ __forceinline__ double gp_g<CES_GP_MATERN12>(double r2) {
    if (r2 == 0.0) return 0.0;                      // sklearn's value at r = 0: D_d = 0 there, so dK/dlog l_d = 0
    const double r = sqrt(r2);
    return exp(-r) / r;
}
template <> __device__ __forceinline__ double gp_g<CES_GP_MATERN32>(double r2) { return 3.0 * exp(-GP_SQRT3 * sqrt(r2)); }
template <> __device__ __forceinline__ double gp_g<CES_GP_MATERN52>(double r2) {
    const double t = GP_SQRT5 * sqrt(r2);
    return (5.0 / 3.0) * (1.0 + t) * exp(-t);
}

// out_z[r][c] = k_z(A[:, r], B[:, c]) for r < nr, c < nc (+ sn2 + jitter where `train` and r == c); rows nr <= r < nr_pad
// are written as zeros.  train: only tiles on or below the diagonal (the Cholesky reads the lower triangle).
// Output z uses theta row z0 + z.
template <int KIND>
__global__ void __launch_bounds__(256) gp_cov_kernel(const double* __restrict__ A, long long lda, int nr, int nr_pad,
                                                     const double* __restrict__ B, long long ldb, int nc, int p,
                                                     const double* __restrict__ theta, int z0, double jitter, int train,
                                                     double* __restrict__ out, long long ldo, long long out_batch) {
    __shared__ double sa[GP_P_MAX][GP_TB + 1], sb[GP_P_MAX][GP_TB + 1];
    const int tr = blockIdx.y, tc = blockIdx.x, z = blockIdx.z;
    if (train && tc > tr) return;
    const double* th = theta + (size_t)(z0 + z) * (p + 2);
    const int r0 = tr * GP_TB, c0 = tc * GP_TB;
    stage_scaled(sa, A, lda, r0, nr, p, th);
    stage_scaled(sb, B, ldb, c0, nc, p, th);
    __syncthreads();
    const double sf2 = exp(th[0]), diag = exp(th[p + 1]) + jitter;
    double* o = out + (size_t)z * out_batch;
    const int c = threadIdx.x & 31;
    for (int r = threadIdx.x >> 5; r < GP_TB; r += 8) {
        const int gr = r0 + r, gc = c0 + c;
        if (gr >= nr_pad || gc >= nc) continue;
        double v = 0.0;
        if (gr < nr) {
            v = sf2 * gp_kf<KIND>(scaled_dist2(sa, sb, r, c, p));
            if (train && gr == gc) v += diag;
        }
        o[(size_t)gr * ldo + gc] = v;
    }
}

// One CTA per 32 x 32 tile on or below the diagonal of K (linear index blockIdx.x): M_ab = w_ab W_ab K_f,ab and
// M'_ab = w_ab W_ab sf2 g(r_ab) with W = alpha alpha^T - K^-1 and w_ab the multiplicity of the pair in the full matrix
// (2 off the diagonal, 1 on it), then part[tile] = { sum M, sum M' (s_ad - s_bd)^2 for d < p, sum_a W_aa }.
// For SE, M' = M: the same value, kept in the same register.
template <int KIND>
__global__ void __launch_bounds__(256) gp_grad_kernel(const double* __restrict__ X, long long ldx, int n, int p,
                                                      const double* __restrict__ th, const double* __restrict__ Kinv,
                                                      long long ldk, const double* __restrict__ alpha, long long lda,
                                                      double* __restrict__ part) {
    __shared__ double sa[GP_P_MAX][GP_TB + 1], sb[GP_P_MAX][GP_TB + 1], sm[GP_TB][GP_TB + 1];
    __shared__ double red[8][GP_P_MAX + 2];
    const int t = blockIdx.x;
    int tr = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
    while ((tr + 1) * (tr + 2) / 2 <= t) ++tr;
    while (tr * (tr + 1) / 2 > t) --tr;
    const int tc = t - tr * (tr + 1) / 2;
    const int r0 = tr * GP_TB, c0 = tc * GP_TB;
    stage_scaled(sa, X, ldx, r0, n, p, th);
    stage_scaled(sb, X, ldx, c0, n, p, th);
    __syncthreads();
    const double sf2 = exp(th[0]);
    const int c = threadIdx.x & 31, w = threadIdx.x >> 5;
    double s_f = 0.0, s_tr = 0.0;
    for (int r = w; r < GP_TB; r += 8) {
        const int gr = r0 + r, gc = c0 + c;
        double m = 0.0, mg = 0.0;
        if (gr < n && gc < n && (tr != tc || c <= r)) {
            const double W = alpha[(size_t)gr * lda] * alpha[(size_t)gc * lda] - Kinv[(size_t)gr * ldk + gc];
            const double r2 = scaled_dist2(sa, sb, r, c, p);
            const double wW = (gr == gc ? 1.0 : 2.0) * W;
            m = wW * (sf2 * gp_kf<KIND>(r2));
            if constexpr (KIND == CES_GP_SE) mg = m;
            else mg = wW * (sf2 * gp_g<KIND>(r2));
            if (gr == gc) s_tr += W;
        }
        sm[r][c] = mg;
        s_f += m;
    }
    __syncthreads();
    double s_d = 0.0;                   // thread (d = lane, group w): rows w, w + 8, ... of the tile, dimension d
    if (c < p) {
        for (int r = w; r < GP_TB; r += 8)
            for (int cc = 0; cc < GP_TB; ++cc) {
                const double dd = sa[c][r] - sb[c][cc];
                s_d = fma(sm[r][cc] * dd, dd, s_d);
            }
    }
    s_f = warp_sum(s_f);
    s_tr = warp_sum(s_tr);
    red[w][c] = s_d;
    if (c == 0) { red[w][GP_P_MAX] = s_f; red[w][GP_P_MAX + 1] = s_tr; }
    __syncthreads();
    double* out = part + (size_t)t * (p + 2);
    const int j = threadIdx.x;
    if (j < p + 2) {
        const int col = j == 0 ? GP_P_MAX : (j <= p ? j - 1 : GP_P_MAX + 1);
        double s = 0.0;
        for (int g = 0; g < 8; ++g) s += red[g][col];
        out[j] = s;
    }
}

// terms[0] = sum log L_jj, terms[1] = y . alpha  (one CTA, fixed-order reduction)
__global__ void __launch_bounds__(256) gp_terms_kernel(const double* __restrict__ L, long long ldl, const double* __restrict__ y,
                                                       const double* __restrict__ alpha, long long lda, int n,
                                                       double* __restrict__ terms) {
    __shared__ double scratch[32];
    double ld = 0.0, ya = 0.0;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        ld += log(L[(size_t)j * ldl + j]);
        ya = fma(y[j], alpha[(size_t)j * lda], ya);
    }
    ld = block_sum(ld, scratch);
    if (threadIdx.x == 0) terms[0] = ld;
    __syncthreads();
    ya = block_sum(ya, scratch);
    if (threadIdx.x == 0) terms[1] = ya;
}

// out_z = [LML, dLML/dtheta (p + 2)] from the per-output terms and (with grad) the per-tile partials, summed in tile order.
__global__ void gp_finish_kernel(const double* __restrict__ terms, const double* __restrict__ part, int ntiles, int p, int n,
                                 const double* __restrict__ theta, int grad, double* __restrict__ out) {
    const int z = blockIdx.x, j = threadIdx.x;
    const int np2 = p + 2;
    double* o = out + (size_t)z * (np2 + 1);
    if (j == 0) o[0] = -0.5 * terms[2 * z + 1] - terms[2 * z] - 0.5 * n * 1.8378770664093454836;   // log 2 pi
    if (!grad || j >= np2) return;
    const double* pz = part + (size_t)z * ntiles * np2;
    double s = 0.0;
    for (int t = 0; t < ntiles; ++t) s += pz[(size_t)t * np2 + j];
    if (j == np2 - 1) s *= exp(theta[(size_t)z * np2 + np2 - 1]);
    o[1 + j] = 0.5 * s;
}

// mean[z][j] = ybar_z + sum_r alpha_z[r] KS_z[r][j],  var[z][j] = max(sf2_z - sum_r V_z[r][j]^2, 0)
__global__ void __launch_bounds__(128) gp_column_kernel(const double* __restrict__ KS, const double* __restrict__ V, long long ld,
                                                        long long batch, const double* __restrict__ alpha, long long npad,
                                                        const double* __restrict__ ybar, const double* __restrict__ theta, int p,
                                                        int n, int m, double* __restrict__ mean, long long ldm,
                                                        double* __restrict__ var, long long ldv) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, z = blockIdx.y;
    if (j >= m) return;
    const double* ks = KS + (size_t)z * batch + j;
    const double* v = V + (size_t)z * batch + j;
    const double* al = alpha + (size_t)z * npad;
    double mu0 = 0.0, mu1 = 0.0, q0 = 0.0, q1 = 0.0;
    int r = 0;
    for (; r + 1 < n; r += 2) {
        mu0 = fma(al[r], ks[(size_t)r * ld], mu0);
        mu1 = fma(al[r + 1], ks[(size_t)(r + 1) * ld], mu1);
        const double a = v[(size_t)r * ld], b = v[(size_t)(r + 1) * ld];
        q0 = fma(a, a, q0);
        q1 = fma(b, b, q1);
    }
    if (r < n) {
        mu0 = fma(al[r], ks[(size_t)r * ld], mu0);
        const double a = v[(size_t)r * ld];
        q0 = fma(a, a, q0);
    }
    mean[(size_t)z * ldm + j] = ybar[z] + (mu0 + mu1);
    var[(size_t)z * ldv + j] = fmax(exp(theta[(size_t)z * (p + 2)]) - (q0 + q1), 0.0);
}

// Phi of chain c at its evaluated point (column c of prop) from its predicted mean / var: emulated misfit, plus the prior
// term 1/2 (x - mu)^T Pinv (x - mu) unless pCN.  One thread, fixed order.
struct GpPhi {
    int k, use_variance, pcn;
    const double* ytil;         // k
    const double* mean;         // k x ld
    const double* var;          // k x ld
    const double* mu;           // p
    const double* Pinv;         // p x p
    __device__ double operator()(const ChainState& a, int c) const {
        const double* x = a.prop;
        double phi = 0.0;
        for (int i = 0; i < k; ++i) {
            const double r = ytil[i] - mean[(size_t)i * a.ld + c];
            if (use_variance) {
                const double s = 1.0 + var[(size_t)i * a.ld + c];
                phi += r * r / s + log(s);
            } else {
                phi = fma(r, r, phi);
            }
        }
        phi *= 0.5;
        if (!pcn) {
            double pp = 0.0;
            for (int q = 0; q < a.p; ++q) {
                double t = 0.0;
                for (int m = 0; m < a.p; ++m) t = fma(Pinv[(size_t)q * a.p + m], x[(size_t)m * a.ld + c] - mu[m], t);
                pp = fma(0.5 * (x[(size_t)q * a.ld + c] - mu[q]), t, pp);
            }
            phi += pp;
        }
        return phi;
    }
};

// z ~ N(0, I_p) and u ~ U(0, 1) per chain (chain 0 from numpy's stream when use_mt), proposal = random walk / pCN.
__global__ void __launch_bounds__(GP_PROPOSE_THREADS) gp_propose_kernel(const ChainState a, const double* scales, int pcn,
                                                                       double beta, int it) {
    __shared__ double zs[GP_P_MAX][GP_PROPOSE_THREADS];
    __shared__ double sc[GP_P_MAX * GP_P_MAX];
    const int p = a.p;
    for (int e = threadIdx.x; e < p * p; e += blockDim.x) sc[e] = scales[e];
    __syncthreads();
    const int c = blockIdx.x * blockDim.x + threadIdx.x, tid = threadIdx.x;
    if (c >= a.n_chains) return;
    a.u[c] = mh_chain_draw(p, it, c, (a.use_mt && c == 0) ? a.mt : nullptr, a.mt_gauss, a.seed, 0x4750u, &zs[0][tid],
                           GP_PROPOSE_THREADS);
    const double a_cur = pcn ? sqrt(1.0 - beta * beta) : 1.0, a_z = pcn ? sqrt(beta) : 1.0;
    for (int q = 0; q < p; ++q) {
        double s = 0.0;
        for (int m = 0; m < p; ++m) s = fma(sc[q * p + m], zs[m][tid], s);       // np.matmul(scales, z)
        const double x = a.cur[(size_t)q * a.ld + c];
        a.prop[(size_t)q * a.ld + c] = pcn ? a_cur * x + a_z * s : x + s;
    }
}

// the instantiations per family, indexed by CES_GP_*: the one dispatch of every covariance / gradient launch
constexpr int GP_KINDS = 4;
decltype(&gp_cov_kernel<CES_GP_SE>) const GP_COV_KERNEL[GP_KINDS] = {
    gp_cov_kernel<CES_GP_SE>, gp_cov_kernel<CES_GP_MATERN12>, gp_cov_kernel<CES_GP_MATERN32>, gp_cov_kernel<CES_GP_MATERN52>};
decltype(&gp_grad_kernel<CES_GP_SE>) const GP_GRAD_KERNEL[GP_KINDS] = {
    gp_grad_kernel<CES_GP_SE>, gp_grad_kernel<CES_GP_MATERN12>, gp_grad_kernel<CES_GP_MATERN32>, gp_grad_kernel<CES_GP_MATERN52>};

}  // namespace

// ------------------------------------------------------------------------------------------------ host side
struct GpModel {
    cudaStream_t st = nullptr;
    int p = 0, k = 0, n = 0;
    int kind = CES_GP_SE;       // covariance family (ces_gp_set_kernel)
    int64_t ldn = 0, npad = 0;
    double* X = nullptr;        // p x n (ldn)
    double* Y = nullptr;        // k x n (ldn), whitened and centred
    double* ybar = nullptr;     // k
    double* theta = nullptr;    // k x (p + 2): scratch of ces_gp_lml
    double* K = nullptr;        // n x ldn: K, then L
    double* Kinv = nullptr;     // n x ldn
    double* Lblk = nullptr;     // inverses of the diagonal blocks of L (round_up(n, 64) x CHOL_NB)
    double* rhs = nullptr;      // n x GP_RHS_LD: column 0 = y, then alpha
    double* part = nullptr;     // k x ntiles x (p + 2)
    double* terms = nullptr;    // k x 2
    double* res = nullptr;      // k x (p + 3)
    int* info = nullptr;        // k
    int ntiles = 0;
    // conditioning (ces_gp_condition)
    bool conditioned = false;
    double* ctheta = nullptr;   // k x (p + 2)
    double* LI = nullptr;       // k x npad x npad: L_i^-1, zero padded
    double* calpha = nullptr;   // k x npad, zero padded
    // prediction scratch, grown on demand
    int64_t m_cap = 0;
    double* KS = nullptr;       // k x npad x ld(m)
    double* V = nullptr;        // k x npad x ld(m)
    std::vector<void*> allocs;
};

namespace {

int gp_alloc(GpModel* g, void** p, size_t bytes) {
    if (cudaMalloc(p, bytes) != cudaSuccess) {
        cudaGetLastError();
        *p = nullptr;
        return fail(CES_ERR_NOMEM, "ces_gp: device allocation of %s%lld bytes failed", "", (long long)bytes);
    }
    g->allocs.push_back(*p);
    return CES_OK;
}

void gp_free(GpModel* g, void* p) {
    if (!p) return;
    cudaFree(p);
    for (auto& q : g->allocs)
        if (q == p) q = nullptr;
}

int gp_ntiles(int n) {
    const int t = (int)ceil_div(n, GP_TB);
    return t * (t + 1) / 2;
}

// K_z (lower triangle, + (sn2 + jitter) I) of output z, with theta row z of `theta`
int gp_assemble_train(GpModel* g, const double* theta, int z, double jitter) {
    const unsigned t = (unsigned)ceil_div(g->n, GP_TB);
    GP_COV_KERNEL[g->kind]<<<dim3(t, t, 1), 256, 0, g->st>>>(g->X, g->ldn, g->n, g->n, g->X, g->ldn, g->n, g->p, theta, z,
                                                             jitter, 1, g->K, g->ldn, 0);
    CES_LAUNCHED(1);
    return CES_OK;
}

// factor K in place and solve alpha = K^-1 y_z into column 0 of rhs
int gp_factor_solve(GpModel* g, int z) {
    CES_TRY(potrf_lower(g->st, g->K, g->ldn, g->n, g->Lblk, CHOL_NB, g->info + z));
    CES_CUDA(cudaMemcpy2DAsync(g->rhs, GP_RHS_LD * sizeof(double), g->Y + (size_t)z * g->ldn, sizeof(double), sizeof(double),
                               g->n, cudaMemcpyDeviceToDevice, g->st));
    CES_TRY(trsm_lower(g->st, g->K, g->ldn, g->n, g->Lblk, CHOL_NB, g->rhs, GP_RHS_LD, GP_RHS_LD, false));
    CES_TRY(trsm_lower(g->st, g->K, g->ldn, g->n, g->Lblk, CHOL_NB, g->rhs, GP_RHS_LD, GP_RHS_LD, true));
    return CES_OK;
}

int gp_read_info(GpModel* g, int z0, int z1, const char* what) {
    std::vector<int> info((size_t)(z1 - z0));
    CES_CUDA(cudaMemcpyAsync(info.data(), g->info + z0, info.size() * sizeof(int), cudaMemcpyDeviceToHost, g->st));
    CES_CUDA(cudaStreamSynchronize(g->st));
    for (int z = z0; z < z1; ++z)
        if (info[z - z0] != 0) {
            CES_CUDA(cudaMemsetAsync(g->info, 0, (size_t)g->k * sizeof(int), g->st));
            return fail(CES_ERR_NOT_SPD, what, "", (long long)z);
        }
    return CES_OK;
}

int gp_predict(GpModel* g, const double* U, int64_t ldu, int64_t m, double* mean, int64_t ldm, double* var, int64_t ldv) {
    const int64_t ldq = padded_ld(m);
    if (m > g->m_cap || ldq > padded_ld(g->m_cap)) {
        gp_free(g, g->KS);
        gp_free(g, g->V);
        g->KS = g->V = nullptr;
        g->m_cap = 0;
        const size_t bytes = (size_t)g->k * g->npad * ldq * sizeof(double);
        CES_TRY(gp_alloc(g, (void**)&g->KS, bytes));
        CES_TRY(gp_alloc(g, (void**)&g->V, bytes));
        g->m_cap = m;
    }
    const int64_t ld = padded_ld(g->m_cap), batch = g->npad * ld;
    GP_COV_KERNEL[g->kind]<<<dim3((unsigned)ceil_div(m, GP_TB), (unsigned)(g->npad / GP_TB), (unsigned)g->k), 256, 0, g->st>>>(
        g->X, g->ldn, g->n, (int)g->npad, U, ldu, (int)m, g->p, g->ctheta, 0, 0.0, 0, g->KS, ld, batch);
    CES_LAUNCHED(1);
    GemmCall c;                                     // V_i = L_i^-1 K*_i for every output at once
    c.a_mode = A_MK; c.b_mode = B_KN;
    c.M = g->n; c.N = (int)m; c.K = g->n;
    c.A = g->LI; c.lda = g->npad;
    c.B = g->KS; c.ldb = ld;
    c.C = g->V; c.ldc = ld;
    c.flags = GEMM_A_LOWER_TRI;
    c.batch = g->k; c.a_batch_rows = g->npad; c.b_batch_rows = g->npad; c.c_batch_elems = batch;
    CES_TRY(gemm(g->st, c));
    gp_column_kernel<<<dim3((unsigned)ceil_div(m, 128), (unsigned)g->k), 128, 0, g->st>>>(
        g->KS, g->V, ld, batch, g->calpha, g->npad, g->ybar, g->ctheta, g->p, g->n, (int)m, mean, ldm, var, ldv);
    CES_LAUNCHED(1);
    return CES_OK;
}

}  // namespace

}  // namespace ces

using namespace ces;

extern "C" int ces_gp_create(void* stream, int64_t p, int64_t k, int64_t n, const double* X_host, const double* Y_host,
                             const double* ybar_host, void** out) {
    if (!out) return fail(CES_ERR_INVALID, "ces_gp_create: null output%s", "");
    *out = nullptr;
    if (p < 1 || p > GP_P_MAX || k < 1 || k > GP_K_MAX || n < 2 || n > (1 << 20) || !X_host || !Y_host || !ybar_host)
        return fail(CES_ERR_INVALID, "ces_gp_create: needs 1 <= p <= 32, 1 <= k <= 64, n >= 2 and non-null inputs%s", "");
    GpModel* g = new GpModel();
    g->st = static_cast<cudaStream_t>(stream);
    g->p = (int)p; g->k = (int)k; g->n = (int)n;
    g->ldn = padded_ld(n);
    g->npad = round_up(n, GP_PAD);
    g->ntiles = gp_ntiles((int)n);
    int s = CES_OK;
    do {
        const size_t nn = (size_t)n * g->ldn * sizeof(double);
        if ((s = gp_alloc(g, (void**)&g->X, (size_t)p * g->ldn * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->Y, (size_t)k * g->ldn * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->ybar, (size_t)k * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->theta, (size_t)k * (p + 2) * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->ctheta, (size_t)k * (p + 2) * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->K, nn)) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->Kinv, nn)) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->Lblk, (size_t)round_up(n, CHOL_NB) * CHOL_NB * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->rhs, (size_t)n * GP_RHS_LD * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->part, (size_t)k * g->ntiles * (p + 2) * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->terms, (size_t)k * 2 * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->res, (size_t)k * (p + 3) * sizeof(double))) != CES_OK) break;
        if ((s = gp_alloc(g, (void**)&g->info, (size_t)k * sizeof(int))) != CES_OK) break;
        if (cudaMemcpy2DAsync(g->X, g->ldn * sizeof(double), X_host, n * sizeof(double), n * sizeof(double), p,
                              cudaMemcpyHostToDevice, g->st) != cudaSuccess ||
            cudaMemcpy2DAsync(g->Y, g->ldn * sizeof(double), Y_host, n * sizeof(double), n * sizeof(double), k,
                              cudaMemcpyHostToDevice, g->st) != cudaSuccess ||
            cudaMemcpyAsync(g->ybar, ybar_host, k * sizeof(double), cudaMemcpyHostToDevice, g->st) != cudaSuccess ||
            cudaMemsetAsync(g->rhs, 0, (size_t)n * GP_RHS_LD * sizeof(double), g->st) != cudaSuccess ||
            cudaMemsetAsync(g->info, 0, (size_t)k * sizeof(int), g->st) != cudaSuccess ||
            cudaStreamSynchronize(g->st) != cudaSuccess) {
            s = fail(CES_ERR_CUDA, "ces_gp_create: upload failed%s", "");
            break;
        }
    } while (0);
    if (s != CES_OK) {
        for (void* q : g->allocs) if (q) cudaFree(q);
        delete g;
        return s;
    }
    *out = g;
    return CES_OK;
}

extern "C" int ces_gp_destroy(void* h) {
    if (!h) return CES_OK;
    GpModel* g = static_cast<GpModel*>(h);
    cudaStreamSynchronize(g->st);
    for (void* q : g->allocs) if (q) cudaFree(q);
    delete g;
    return CES_OK;
}

extern "C" int ces_gp_set_kernel(void* h, int kind) {
    GpModel* g = static_cast<GpModel*>(h);
    if (!g || kind < 0 || kind >= GP_KINDS)
        return fail(CES_ERR_INVALID, "ces_gp_set_kernel: needs a model and a kind CES_GP_SE .. CES_GP_MATERN52, got %s%lld", "",
                    (long long)kind);
    g->kind = kind;
    g->conditioned = false;
    return CES_OK;
}

extern "C" int ces_gp_lml(void* h, int64_t i0, int64_t i1, const double* theta_host, double jitter, double* lml_host,
                          double* grad_host) {
    GpModel* g = static_cast<GpModel*>(h);
    if (!g || !theta_host || !lml_host || i0 < 0 || i1 <= i0 || i1 > (g ? g->k : 0) || !(jitter >= 0.0))
        return fail(CES_ERR_INVALID, "ces_gp_lml: needs a model, 0 <= i0 < i1 <= k, jitter >= 0 and non-null theta / lml%s", "");
    const int np2 = g->p + 2, nz = (int)(i1 - i0);
    double* th = g->theta + (size_t)i0 * np2;
    CES_CUDA(cudaMemcpyAsync(th, theta_host, (size_t)nz * np2 * sizeof(double), cudaMemcpyHostToDevice, g->st));
    for (int z = (int)i0; z < (int)i1; ++z) {
        const double* thz = g->theta + (size_t)z * np2;
        CES_TRY(gp_assemble_train(g, g->theta, z, jitter));
        CES_TRY(gp_factor_solve(g, z));
        gp_terms_kernel<<<1, 256, 0, g->st>>>(g->K, g->ldn, g->Y + (size_t)z * g->ldn, g->rhs, GP_RHS_LD, g->n, g->terms + 2 * z);
        CES_LAUNCHED(1);
        if (grad_host) {
            CES_TRY(spd_inverse_from_factor(g->st, g->K, g->ldn, g->n, g->Lblk, CHOL_NB, g->Kinv, g->ldn));
            GP_GRAD_KERNEL[g->kind]<<<(unsigned)g->ntiles, 256, 0, g->st>>>(g->X, g->ldn, g->n, g->p, thz, g->Kinv, g->ldn,
                                                                           g->rhs, GP_RHS_LD,
                                                                           g->part + (size_t)z * g->ntiles * np2);
            CES_LAUNCHED(1);
        }
    }
    gp_finish_kernel<<<(unsigned)nz, 64, 0, g->st>>>(g->terms + 2 * i0, g->part + (size_t)i0 * g->ntiles * np2, g->ntiles,
                                                     g->p, g->n, th, grad_host ? 1 : 0, g->res);
    CES_LAUNCHED(1);
    std::vector<double> res((size_t)nz * (np2 + 1));
    CES_CUDA(cudaMemcpyAsync(res.data(), g->res, res.size() * sizeof(double), cudaMemcpyDeviceToHost, g->st));
    CES_TRY(gp_read_info(g, (int)i0, (int)i1, "ces_gp_lml: K of output %s%lld is not positive definite"));
    for (int z = 0; z < nz; ++z) {
        lml_host[z] = res[(size_t)z * (np2 + 1)];
        if (grad_host)
            for (int j = 0; j < np2; ++j) grad_host[(size_t)z * np2 + j] = res[(size_t)z * (np2 + 1) + 1 + j];
    }
    return CES_OK;
}

extern "C" int ces_gp_condition(void* h, const double* theta_host, double jitter) {
    GpModel* g = static_cast<GpModel*>(h);
    if (!g || !theta_host || !(jitter >= 0.0))
        return fail(CES_ERR_INVALID, "ces_gp_condition: needs a model, theta and jitter >= 0%s", "");
    g->conditioned = false;
    const int np2 = g->p + 2;
    if (!g->LI || !g->calpha) {
        CES_TRY(gp_alloc(g, (void**)&g->LI, (size_t)g->k * g->npad * g->npad * sizeof(double)));
        CES_TRY(gp_alloc(g, (void**)&g->calpha, (size_t)g->k * g->npad * sizeof(double)));
    }
    CES_CUDA(cudaMemsetAsync(g->LI, 0, (size_t)g->k * g->npad * g->npad * sizeof(double), g->st));
    CES_CUDA(cudaMemsetAsync(g->calpha, 0, (size_t)g->k * g->npad * sizeof(double), g->st));
    CES_CUDA(cudaMemcpyAsync(g->ctheta, theta_host, (size_t)g->k * np2 * sizeof(double), cudaMemcpyHostToDevice, g->st));
    for (int z = 0; z < g->k; ++z) {
        CES_TRY(gp_assemble_train(g, g->ctheta, z, jitter));
        CES_TRY(gp_factor_solve(g, z));
        CES_CUDA(cudaMemcpy2DAsync(g->calpha + (size_t)z * g->npad, sizeof(double), g->rhs, GP_RHS_LD * sizeof(double),
                                   sizeof(double), g->n, cudaMemcpyDeviceToDevice, g->st));
        double* LIz = g->LI + (size_t)z * g->npad * g->npad;
        CES_TRY(set_identity(g->st, LIz, g->npad, g->n));
        CES_TRY(trsm_lower(g->st, g->K, g->ldn, g->n, g->Lblk, CHOL_NB, LIz, g->npad, g->n, false));
    }
    CES_TRY(gp_read_info(g, 0, g->k, "ces_gp_condition: K of output %s%lld is not positive definite"));
    g->conditioned = true;
    return CES_OK;
}

extern "C" int ces_gp_predict(void* h, const double* U_dev, int64_t ldu, int64_t m, double* mean_dev, int64_t ldm,
                              double* var_dev, int64_t ldv) {
    GpModel* g = static_cast<GpModel*>(h);
    if (!g || !U_dev || !mean_dev || !var_dev || m < 1 || ldu < m || ldm < m || ldv < m)
        return fail(CES_ERR_INVALID, "ces_gp_predict: needs a model, m >= 1, leading dimensions >= m and non-null arrays%s", "");
    if (!g->conditioned) return fail(CES_ERR_STATE, "ces_gp_predict: call ces_gp_condition first%s", "");
    return gp_predict(g, U_dev, ldu, m, mean_dev, ldm, var_dev, ldv);
}

extern "C" int ces_gp_mh(void* h, const double* ytil_host, int use_variance, const double* mu_host, const double* Pinv_host,
                         const double* scales_host, int pcn, double beta, int64_t n_mcmc, int64_t n_chains,
                         const double* start_host, const double* phi_point_host, uint32_t* mt_state_host,
                         double* mt_gauss_host, uint64_t seed, double* samples_host, int32_t* accepted_host) {
    const ChainHost ch{"ces_gp_mh", n_mcmc, n_chains, pcn, ytil_host, scales_host, mu_host, Pinv_host, start_host,
                       phi_point_host, mt_state_host, mt_gauss_host, seed, samples_host, accepted_host};
    CES_TRY(chain_check(ch));
    GpModel* g = static_cast<GpModel*>(h);
    if (!g) return fail(CES_ERR_INVALID, "ces_gp_mh: null model%s", "");
    if (!g->conditioned) return fail(CES_ERR_STATE, "ces_gp_mh: call ces_gp_condition first%s", "");
    const int p = g->p, k = g->k;
    const int64_t ld = padded_ld(n_chains);
    ChainRun run(ch, p, g->st);
    ChainState a;
    GpPhi phi;
    phi.k = k; phi.use_variance = use_variance ? 1 : 0; phi.pcn = pcn ? 1 : 0;
    const double* scales = nullptr;
    double *mean = nullptr, *var = nullptr;
    CES_TRY(run.build([&] {
        a = chain_state(run, ld);
        phi.ytil = run.put(ytil_host, k);
        phi.mu = run.put(pcn ? nullptr : mu_host, p);
        phi.Pinv = run.put(pcn ? nullptr : Pinv_host, (size_t)p * p);
        scales = run.put(scales_host, (size_t)p * p);
        phi.mean = mean = run.take((size_t)k * ld);
        phi.var = var = run.take((size_t)k * ld);
    }));
    CES_TRY(gp_predict(g, a.prop, ld, n_chains, mean, ld, var, ld));
    const unsigned blocks = (unsigned)ceil_div(n_chains, CHAIN_THREADS);
    chain_init_kernel<<<blocks, CHAIN_THREADS, 0, g->st>>>(a, phi);
    CES_LAUNCHED(1);
    for (int it = 0; it < a.n_mcmc; ++it) {
        gp_propose_kernel<<<(unsigned)ceil_div(n_chains, GP_PROPOSE_THREADS), GP_PROPOSE_THREADS, 0, g->st>>>(a, scales, pcn,
                                                                                                          beta, it);
        CES_LAUNCHED(1);
        CES_TRY(gp_predict(g, a.prop, ld, n_chains, mean, ld, var, ld));
        chain_accept_kernel<<<blocks, CHAIN_THREADS, 0, g->st>>>(a, phi, it);
        CES_LAUNCHED(1);
    }
    return run.copy_back();
}
