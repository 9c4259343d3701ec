// Whole ensemble Kalman update in ONE single-CTA kernel for small problems (p <= 8, k <= 16, J <= 512), e.g.
// BASELINE config 1 (d = 2, k = 10, J = 100, 1000 steps) where the general path's ~20 launches are pure latency.
//
// Same arithmetic as the phases (ces/calibrate.py:418-529): one thread per particle, the ensemble in shared
// memory, D never stored -- thread j accumulates its column of V = U~ D while streaming over the particles i
// (d_ij = e_i . w_j / J), together with the Frobenius sum.  Step size, chol(C^uu) (and the implicit-prior factor for
// the semi-implicit rule) are computed by thread 0 between two barriers.
//
// The noise form is a template parameter ENS of the kernels.  false: the reference's sqrt(2h) chol(C^uu) xi with a p x J
// xi.  true (CES_NOISE_ENSEMBLE): sqrt(2h / n_C) U~ xi with a J x J xi, read from the caller's matrix or drawn in the
// kernel from the stream of ces_fill_ensemble_noise; chol(C^uu) is then not formed.
#include "kernels.h"
#include "rng.cuh"

namespace ces {

constexpr int SP = SMALL_P_MAX, SK = SMALL_K_MAX;

struct SmallArgs {
    int p, k, J, rule, ts_kind;
    double fixed_h, switch_;
    const double *U, *G, *xi;
    long long ldu, ldg, ldxi;
    double* out;
    long long ldo;
    const double *y, *mu, *ustar, *bprior;
    const double *ginv_diag, *Ginv;      // one of them (diagonal / dense Gamma^-1, ld = ldk)
    const double *sinv_diag, *sig_diag, *Sinv, *Sigma0;   // diagonal or dense prior (ld = ldp)
    long long ldk, ldp;
    double* S;                           // device scalars (StepScalars layout; S_INFO reports a failed pivot)
};

// Column j of V = U~ D with D = (1/J) E^T W never stored, and this column's share of ||D||_F^2: the one loop of the step
// that is O(J) per thread.  K and P are compile-time trip counts (the generic, predicated form of this loop spent 87 % of
// the kernel on branches and address arithmetic -- 166 instructions per particle pair for 13 useful DFMAs); four
// independent particles i are in flight per trip, so the FMA chains of d overlap.
template <int KK, int PP>
__device__ __forceinline__ void interaction_column(const double* __restrict__ Es, const double* __restrict__ Uts, int J, int p,
                                                   const double (&w)[SMALL_K_MAX], double invJ, double (&v)[SMALL_P_MAX],
                                                   double& ssq) {
    double s0 = 0.0, s1 = 0.0;
    int i = 0;
    for (; i + 1 < J; i += 2) {
        double d0 = 0.0, d1 = 0.0;
#pragma unroll
        for (int m = 0; m < KK; ++m) {
            d0 = fma(Es[m * J + i], w[m], d0);
            d1 = fma(Es[m * J + i + 1], w[m], d1);
        }
        d0 *= invJ; d1 *= invJ;
        s0 = fma(d0, d0, s0); s1 = fma(d1, d1, s1);
#pragma unroll
        for (int q = 0; q < PP; ++q)
            if (q < p) v[q] = fma(Uts[q * J + i + 1], d1, fma(Uts[q * J + i], d0, v[q]));
    }
    if (i < J) {
        double d0 = 0.0;
#pragma unroll
        for (int m = 0; m < KK; ++m) d0 = fma(Es[m * J + i], w[m], d0);
        d0 *= invJ;
        s0 = fma(d0, d0, s0);
#pragma unroll
        for (int q = 0; q < PP; ++q)
            if (q < p) v[q] = fma(Uts[q * J + i], d0, v[q]);
    }
    ssq += s0 + s1;
}

template <int KK>
__device__ __forceinline__ void interaction_column_p(const double* Es, const double* Uts, int J, int p, const double (&w)[SMALL_K_MAX],
                                                     double invJ, double (&v)[SMALL_P_MAX], double& ssq) {
    if (p <= 2) interaction_column<KK, 2>(Es, Uts, J, p, w, invJ, v, ssq);
    else if (p <= 4) interaction_column<KK, 4>(Es, Uts, J, p, w, invJ, v, ssq);
    else interaction_column<KK, 8>(Es, Uts, J, p, w, invJ, v, ssq);
}

// Column j of the ensemble noise before its scale: n = sum_s U~[:, s] xi[s, j], s in order, P a compile-time trip count as
// in interaction_column.  xi != nullptr: the caller's J x J matrix (ld ldxi).  Otherwise the Box-Muller pair of (s, j >> 1)
// (rng.cuh ensemble_noise_pair) is drawn once per step: of threads 2m and 2m + 1, the even one draws the pairs of the even
// rows s and the odd one those of the odd rows, and each hands its partner the partner's half of the pair by a shuffle.
// Four rows per trip put two independent draws in flight per thread (a CTA of J threads has few warps to hide the latency
// of log / sincospi).  Both forms read xi[s, j] in the same order into the same FMAs, so the stream and its fill give
// bit-identical columns.  Every lane of the CTA must call it (the shuffles); a lane past J gets values nobody reads.
template <int PP>
__device__ __forceinline__ void ensemble_noise_column(const double* __restrict__ Uts, int J, int p, int j, const double* xi,
                                                      long long ldxi, unsigned long long seed, unsigned long long step,
                                                      double (&n)[SMALL_P_MAX]) {
    const bool on = j < J, odd = j & 1;
    for (int s0 = 0; s0 < J; s0 += 4) {
        double x[4];
        if (xi) {
#pragma unroll
            for (int r = 0; r < 4; ++r) x[r] = (on && s0 + r < J) ? xi[(size_t)(s0 + r) * ldxi + j] : 0.0;
        } else {
            const double2 za = ensemble_noise_pair(seed, step, (unsigned long long)(s0 + odd), (unsigned long long)(j >> 1));
            const double2 zb = ensemble_noise_pair(seed, step, (unsigned long long)(s0 + 2 + odd), (unsigned long long)(j >> 1));
            const double oa = __shfl_xor_sync(0xffffffffu, odd ? za.x : za.y, 1);
            const double ob = __shfl_xor_sync(0xffffffffu, odd ? zb.x : zb.y, 1);
            x[0] = odd ? oa : za.x; x[1] = odd ? za.y : oa;
            x[2] = odd ? ob : zb.x; x[3] = odd ? zb.y : ob;
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (s0 + r < J)
#pragma unroll
                for (int q = 0; q < PP; ++q)
                    if (q < p) n[q] = fma(Uts[q * J + s0 + r], x[r], n[q]);
    }
}

__device__ __forceinline__ void block_reduce5(double (&v)[5], double (*scratch)[32], bool take_max4) {
    // sums of v[0..3] (+ v[4]: sum, or max when take_max4); every thread returns the totals
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int q = 0; q < 5; ++q) v[q] = (q == 4 && take_max4) ? warp_max(v[q]) : warp_sum(v[q]);
    __syncthreads();
    if (lane == 0)
#pragma unroll
        for (int q = 0; q < 5; ++q) scratch[q][wid] = v[q];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 5; ++q) {
        double t = 0.0;
        for (int w = 0; w < nw; ++w) t = (q == 4 && take_max4) ? fmax(t, scratch[q][w]) : t + scratch[q][w];
        v[q] = t;
    }
}

// One update by the whole CTA (one thread per particle).  Every thread of the CTA must call it (barriers inside); it
// returns with the new column written to a.out and the step scalars in a.S (thread 0), without a trailing barrier.
// ENS: the ensemble noise, xi = a.xi (J x J, ld a.ldxi) or the stream at (seed, step); eki takes ENS = false.
template <bool ENS>
__device__ __forceinline__ void small_step_body(const SmallArgs& a, double* sm, double (*scratch)[32], unsigned long long seed,
                                                unsigned long long step) {
    const int p = a.p, k = a.k, J = a.J;
    double* Es = sm;                    // k x J   E = G - mean
    double* Uts = Es + (size_t)k * J;   // p x J   U~ = U - mean
    double* mean = Uts + (size_t)p * J; // k + p
    double* Cs = mean + (SK + SP);      // p x p   C^uu
    double* Ls = Cs + SP * SP;          // p x p   chol(C^uu)
    double* Ms = Ls + SP * SP;          // p x p   chol(Sigma0 + h C)   (eks)
    double* cb = Ms + SP * SP;          // p       C Sigma0^-1 mu       (eks)
    double* sc = cb + SP;               // scalars: h, sqrt2h (ENS: sqrt(2h / n_C) in place of sqrt2h)
    const int j = threadIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    const bool on = j < J;

    // ---- load this particle, stage raw values in shared memory for the row means
    double u[SP], g[SK];
#pragma unroll
    for (int q = 0; q < SP; ++q) { u[q] = (on && q < p) ? a.U[(size_t)q * a.ldu + j] : 0.0; if (on && q < p) Uts[(size_t)q * J + j] = u[q]; }
#pragma unroll
    for (int m = 0; m < SK; ++m) { g[m] = (on && m < k) ? a.G[(size_t)m * a.ldg + j] : 0.0; if (on && m < k) Es[(size_t)m * J + j] = g[m]; }
    __syncthreads();
    for (int row = wid; row < k + p; row += nw) {           // one warp per row
        const double* src = row < k ? Es + (size_t)row * J : Uts + (size_t)(row - k) * J;
        double s = 0.0;
        for (int i = lane; i < J; i += 32) s += src[i];
        s = warp_sum(s);
        if (lane == 0) mean[row] = s / (double)J;
    }
    __syncthreads();

    // ---- centring, W = Gamma^-1 R, Z = Sigma0^-1 (U - mu), per-particle diagnostics (:427-435)
    double w[SK], z[SP], ut[SP];
    double red[5] = {0.0, 0.0, 0.0, 0.0, 0.0};   // ssq, self-bias, bias, self-bias-data, bias-data
    {
        double e[SK], r[SK];
#pragma unroll
        for (int m = 0; m < SK; ++m) {
            e[m] = (on && m < k) ? g[m] - mean[m] : 0.0;
            r[m] = (on && m < k) ? g[m] - a.y[m] : 0.0;
        }
        double qe = 0.0, qr = 0.0;
#pragma unroll
        for (int m = 0; m < SK; ++m) {
            double wm = 0.0, wem = 0.0;
            if (m < k) {
                if (a.Ginv) {
#pragma unroll
                    for (int n = 0; n < SK; ++n)
                        if (n < k) { const double gi = a.Ginv[(size_t)m * a.ldk + n]; wm += gi * r[n]; wem += gi * e[n]; }
                } else {
                    const double gi = a.ginv_diag[m];
                    wm = gi * r[m]; wem = gi * e[m];
                }
            }
            w[m] = wm;
            qe += e[m] * wem;
            qr += r[m] * wm;
        }
#pragma unroll
        for (int q = 0; q < SP; ++q) {
            ut[q] = (on && q < p) ? u[q] - mean[k + q] : 0.0;
            if (on && q < p) {
                red[1] += ut[q] * ut[q];
                const double db = u[q] - a.ustar[q];
                red[2] += db * db;
            }
        }
#pragma unroll
        for (int q = 0; q < SP; ++q) {
            double zq = 0.0;
            if (on && q < p) {
                if (a.Sinv) {
#pragma unroll
                    for (int n = 0; n < SP; ++n) if (n < p) zq += a.Sinv[(size_t)q * a.ldp + n] * (u[n] - a.mu[n]);
                } else {
                    zq = a.sinv_diag[q] * (u[q] - a.mu[q]);
                }
            }
            z[q] = zq;
        }
        red[3] = on ? qe * qe : 0.0;
        red[4] = on ? qr * qr : 0.0;
        __syncthreads();                      // everyone has read the raw rows: overwrite them with E and U~
        if (on) {
#pragma unroll
            for (int m = 0; m < SK; ++m) if (m < k) Es[(size_t)m * J + j] = e[m];
#pragma unroll
            for (int q = 0; q < SP; ++q) if (q < p) Uts[(size_t)q * J + j] = ut[q];
        }
    }
    __syncthreads();

    // ---- column j of V = U~ D, D = (1/J) E^T W never stored (:429, :484); Frobenius sum (:248)
    double v[SP];
#pragma unroll
    for (int q = 0; q < SP; ++q) v[q] = 0.0;
    if (on) {
        const double invJ = 1.0 / (double)J;
        switch (k) {
#define CES_IC(KK) case KK: interaction_column_p<KK>(Es, Uts, J, p, w, invJ, v, red[0]); break;
            CES_IC(1) CES_IC(2) CES_IC(3) CES_IC(4) CES_IC(5) CES_IC(6) CES_IC(7) CES_IC(8)
            CES_IC(9) CES_IC(10) CES_IC(11) CES_IC(12) CES_IC(13) CES_IC(14) CES_IC(15) CES_IC(16)
#undef CES_IC
            default: break;
        }
    }
    // ---- C^uu = U~ U~^T / (J-1) (+1e-8 I); 1/J for the semi-implicit rule (:424, :476, :512)
    const double cscale = (a.rule == CES_RULE_EKS) ? 1.0 / (double)J : 1.0 / (double)(J - 1);
    for (int pair = wid; pair < p * p; pair += nw) {
        const int ra = pair / p, rb = pair % p;
        if (rb > ra) continue;
        double s = 0.0;
        for (int i = lane; i < J; i += 32) s += Uts[(size_t)ra * J + i] * Uts[(size_t)rb * J + i];
        s = warp_sum(s);
        if (lane == 0) {
            const double c = s * cscale + (ra == rb ? 1e-8 : 0.0);
            Cs[ra * SP + rb] = c;
            Cs[rb * SP + ra] = c;
        }
    }
    block_reduce5(red, scratch, false);       // also orders the writes of Cs before thread 0 reads them

    // ---- drift of aldi_constant needs max|.| before h (:515-519)
    const double alphaJ = (double)(p + 1) / (double)J;
    double cz[SP];
#pragma unroll
    for (int q = 0; q < SP; ++q) {
        double s = 0.0;
        if (q < p)
#pragma unroll
            for (int n = 0; n < SP; ++n) if (n < p) s += Cs[q * SP + n] * z[n];
        cz[q] = s;
    }
    double maxdrift = 0.0;
    if (a.rule == CES_RULE_ALDI_CONSTANT) {
        double md[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
        if (on)
#pragma unroll
            for (int q = 0; q < SP; ++q) if (q < p) md[4] = fmax(md[4], fabs(-v[q] - cz[q] + a.switch_ * alphaJ * ut[q]));
        block_reduce5(md, scratch, true);
        maxdrift = md[4];
    }

    if (threadIdx.x == 0) {
        double h;
        if (a.rule == CES_RULE_ALDI_CONSTANT) h = 0.1 / maxdrift;
        else if (a.ts_kind == CES_TS_FIXED) h = a.fixed_h;
        else h = 1.0 / (sqrt(red[0]) + 1e-8);
        sc[0] = h;
        sc[1] = sqrt(2.0 * h);
        a.S[S_INFO] = 0.0;
        a.S[S_SSQ] = red[0]; a.S[S_SELF_BIAS] = red[1]; a.S[S_BIAS] = red[2]; a.S[S_SELF_DATA] = red[3]; a.S[S_BIAS_DATA] = red[4];
        a.S[S_MAXDRIFT] = maxdrift; a.S[S_H] = h; a.S[S_SQRT2H] = sc[1]; a.S[S_NEG_H] = -h; a.S[S_H_ALPHA] = h * alphaJ;
        if constexpr (ENS) {
            // sqrt(2h / n_C), n_C of the rule's own C^uu (api.cu ens_inv_nc)
            const double inv_nc = (a.rule == CES_RULE_EKS) ? 1.0 / (double)J : 1.0 / (double)(J - 1);
            sc[1] = sqrt(2.0 * h * inv_nc);
            a.S[S_ENS_ALPHA] = sc[1];
        }
        // chol(C^uu) (:446, :487, :526; not with ENS), and chol(Sigma0 + h C) for the implicit prior step (:443, SURVEY.md F6)
        for (int pass = ENS ? 1 : 0; pass < ((a.rule == CES_RULE_EKS) ? 2 : 1); ++pass) {
            double* Lm = pass == 0 ? Ls : Ms;
            for (int r = 0; r < p; ++r)
                for (int c = 0; c <= r; ++c) {
                    double x = Cs[r * SP + c];
                    if (pass == 1) {
                        x *= h;
                        x += a.Sigma0 ? a.Sigma0[(size_t)r * a.ldp + c] : (r == c ? a.sig_diag[r] : 0.0);
                    }
                    for (int t = 0; t < c; ++t) x -= Lm[r * SP + t] * Lm[c * SP + t];
                    if (r == c) {
                        if (!(x > 0.0) && a.S[S_INFO] == 0.0) a.S[S_INFO] = (double)(r + 1);
                        Lm[r * SP + r] = sqrt(x);
                    } else {
                        Lm[r * SP + c] = x / Lm[c * SP + c];
                    }
                }
        }
        if (a.rule == CES_RULE_EKS)
            for (int r = 0; r < p; ++r) {
                double s = 0.0;
                for (int n = 0; n < p; ++n) s += Cs[r * SP + n] * a.bprior[n];
                cb[r] = s;
            }
    }
    __syncthreads();
    double noise[SP];
    if constexpr (ENS) {
#pragma unroll
        for (int q = 0; q < SP; ++q) noise[q] = 0.0;
        if (p <= 2) ensemble_noise_column<2>(Uts, J, p, j, a.xi, a.ldxi, seed, step, noise);
        else if (p <= 4) ensemble_noise_column<4>(Uts, J, p, j, a.xi, a.ldxi, seed, step, noise);
        else ensemble_noise_column<8>(Uts, J, p, j, a.xi, a.ldxi, seed, step, noise);
    }
    if (!on) return;                    // (no barrier follows inside this function)

    // ---- assemble U_{n+1}[:, j]
    const double h = sc[0], s2h = sc[1];
    if constexpr (!ENS) {
#pragma unroll
        for (int q = 0; q < SP; ++q) {
            double s = 0.0;
            if (q < p && a.rule != CES_RULE_EKI)
#pragma unroll
                for (int n = 0; n < SP; ++n) if (n <= q) s += Ls[q * SP + n] * a.xi[(size_t)n * a.ldxi + j];
            noise[q] = s;
        }
    }
    double o[SP];
    if (a.rule == CES_RULE_ALDI) {
#pragma unroll
        for (int q = 0; q < SP; ++q) o[q] = u[q] - h * v[q] - h * cz[q] + h * alphaJ * ut[q] + s2h * noise[q];
    } else if (a.rule == CES_RULE_ALDI_CONSTANT) {
#pragma unroll
        for (int q = 0; q < SP; ++q) o[q] = u[q] + h * (-v[q] - cz[q] + a.switch_ * alphaJ * ut[q]) + s2h * noise[q];
    } else if (a.rule == CES_RULE_EKI) {
#pragma unroll
        for (int q = 0; q < SP; ++q) o[q] = u[q] - h * v[q];
    } else {
        double t[SP];
#pragma unroll
        for (int q = 0; q < SP; ++q) t[q] = (q < p) ? u[q] - h * v[q] + h * cb[q] : 0.0;
#pragma unroll
        for (int q = 0; q < SP; ++q)            // forward substitution with chol(Sigma0 + h C)
            if (q < p) {
                double s = t[q];
#pragma unroll
                for (int n = 0; n < SP; ++n) if (n < q) s -= Ms[q * SP + n] * t[n];
                t[q] = s / Ms[q * SP + q];
            }
#pragma unroll
        for (int qq = SP - 1; qq >= 0; --qq)    // backward substitution
            if (qq < p) {
                double s = t[qq];
#pragma unroll
                for (int n = 0; n < SP; ++n) if (n > qq && n < p) s -= Ms[n * SP + qq] * t[n];
                t[qq] = s / Ms[qq * SP + qq];
            }
#pragma unroll
        for (int q = 0; q < SP; ++q) {
            double s = 0.0;
            if (q < p) {
                if (a.Sigma0) {
#pragma unroll
                    for (int n = 0; n < SP; ++n) if (n < p) s += a.Sigma0[(size_t)q * a.ldp + n] * t[n];
                } else {
                    s = a.sig_diag[q] * t[q];
                }
            }
            o[q] = s + s2h * noise[q];
        }
    }
#pragma unroll
    for (int q = 0; q < SP; ++q) if (q < p) a.out[(size_t)q * a.ldo + j] = o[q];
}

template <bool ENS>
__global__ void __launch_bounds__(512, 1) small_step_kernel(const SmallArgs a, unsigned long long seed, unsigned long long step) {
    extern __shared__ double sm[];
    __shared__ double scratch[5][32];
    small_step_body<ENS>(a, sm, scratch, seed, step);
}

// ---- the whole sampling.run loop of a small problem in ONE launch (BASELINE config 1: d = 2, k = 10, J = 100, T = 1000).
// Per iteration (ces/calibrate.py:341-388): forward map of every particle (enka.G_ens, :351-352; the ces.utils maps),
// update (small_step_body), cumulative pseudo-time (:262-265) and the stopping rule t > t_tol (:387-388).  The chain of
// ensembles IS the trace: iteration i reads U from slot i of Utrace and writes slot i + 1, the forward outputs go to
// Gtrace, the step scalars of every iteration to Sall -- the host downloads them once at the end.  No launch, no host
// round trip and no PCIe transfer happens between iterations.
struct SmallRunArgs {
    SmallArgs base;                     // problem data, rule, step-size rule (U / G / xi / out / S are set per iteration)
    int T, map_kind, have_t0;
    double t0, t_tol;
    const double* A; long long lda;     // lineal / lineal_log: k x p (ld = lda), b: k or nullptr
    const double* b;
    double par0, par1;                  // elliptic (x1, x2) / banana (a, b)
    double* Utrace;                     // (T + 1) x p x J
    double* Gtrace;                     // (T + 1) x k x J
    const double* Xi;                   // T x p x J
    double* Sall;                       // T x S_COUNT
    double* tvec;                       // T cumulative times
    int* nsteps;                        // [0]: updates performed
    unsigned long long seed, step0;     // ENS without an explicit xi: iteration i draws the stream at (seed, step0 + i)
};

__device__ __forceinline__ void small_forward(const SmallRunArgs& r, const double* U, double* G, int j) {
    const int p = r.base.p, k = r.base.k, J = r.base.J;
    if (r.map_kind == CES_MAP_LINEAL || r.map_kind == CES_MAP_LINEAL_LOG) {
        double u[SP];
#pragma unroll
        for (int q = 0; q < SP; ++q) {
            u[q] = q < p ? U[(size_t)q * J + j] : 0.0;
            if (r.map_kind == CES_MAP_LINEAL_LOG && q < p) u[q] = exp(u[q]);
        }
        for (int m = 0; m < k; ++m) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < SP; ++q) if (q < p) s = fma(r.A[(size_t)m * r.lda + q], u[q], s);
            G[(size_t)m * J + j] = r.b ? s + r.b[m] : s;
        }
    } else if (r.map_kind == CES_MAP_ELLIPTIC) {
        const double u1 = U[j], u2 = U[J + j], e = exp(-u1), x1 = r.par0, x2 = r.par1;
        G[j] = (u2 * x1) + (e * (-x1 * x1 + x1) * 0.5);
        G[J + j] = (u2 * x2) + (e * (-x2 * x2 + x2) * 0.5);
    } else {                            // banana
        const double u1 = U[j], u2 = U[J + j];
        G[j] = u1 * r.par0;
        G[J + j] = u2 / r.par0 - r.par1 * (u1 * u1 + r.par0 * r.par0);
    }
}

template <bool ENS>
__global__ void __launch_bounds__(512, 1) small_run_kernel(const SmallRunArgs r) {
    extern __shared__ double sm[];
    __shared__ double scratch[5][32];
    __shared__ double t_acc;
    __shared__ int stop;
    const int p = r.base.p, k = r.base.k, J = r.base.J;
    const int j = threadIdx.x;
    const bool on = j < J;
    if (j == 0) { t_acc = r.t0; stop = 0; }
    int it = 0;
    for (; it < r.T; ++it) {
        const double* Ucur = r.Utrace + (size_t)it * p * J;
        double* Gcur = r.Gtrace + (size_t)it * k * J;
        if (on) small_forward(r, Ucur, Gcur, j);            // own column: read back by the same thread below
        SmallArgs a = r.base;
        a.U = Ucur; a.ldu = J; a.G = Gcur; a.ldg = J;
        if constexpr (!ENS) { a.xi = r.Xi ? r.Xi + (size_t)it * p * J : nullptr; a.ldxi = J; }   // ENS: one J x J xi or NULL
        a.out = r.Utrace + (size_t)(it + 1) * p * J; a.ldo = J;
        a.S = r.Sall + (size_t)it * S_COUNT;
        small_step_body<ENS>(a, sm, scratch, r.seed, r.step0 + (unsigned long long)it);
        __syncthreads();                                    // every column of slot it + 1 is written, a.S is complete
        if (j == 0) {
            const double h = a.S[S_H];
            t_acc = (it == 0 && !r.have_t0) ? h : t_acc + h;    // ces/calibrate.py:262-265
            r.tvec[it] = t_acc;
            if (t_acc > r.t_tol || a.S[S_INFO] != 0.0 || !(h == h)) stop = 1;    // :387-388; failed pivot / NaN: the host raises
        }
        __syncthreads();
        if (stop) { ++it; break; }
    }
    // the final forward evaluation of the last ensemble (:390-398)
    if (on) small_forward(r, r.Utrace + (size_t)it * p * J, r.Gtrace + (size_t)it * k * J, j);
    if (j == 0) r.nsteps[0] = it;
}

bool small_step_eligible(int64_t p, int64_t k, int64_t J) {
    return p <= SMALL_P_MAX && k <= SMALL_K_MAX && J <= 512 && J >= 2;
}

static size_t small_smem(const SmallStepCall& c) {
    return ((size_t)(c.k + c.p) * c.J + (SK + SP) + 3 * SP * SP + SP + 8) * sizeof(double);
}

// Dynamic shared memory above 48 KB for one kernel (each kernel keeps its own setting per device).
template <auto Kernel>
static int allow_smem(size_t smem) {
    static size_t configured_of[kMaxDevices] = {};
    size_t& configured = configured_of[device_slot()];
    if (smem > 48 * 1024 && smem > configured) {
        CES_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    return CES_OK;
}

int small_step(cudaStream_t st, const SmallStepCall& c) {
    SmallArgs a;
    a.p = (int)c.p; a.k = (int)c.k; a.J = (int)c.J; a.rule = c.rule; a.ts_kind = c.ts_kind;
    a.fixed_h = c.fixed_h; a.switch_ = c.switch_;
    a.U = c.U; a.G = c.G; a.xi = c.xi; a.ldu = c.ldu; a.ldg = c.ldg; a.ldxi = c.ldxi;
    a.out = c.out; a.ldo = c.ldo;
    a.y = c.y; a.mu = c.mu; a.ustar = c.ustar; a.bprior = c.bprior;
    a.ginv_diag = c.ginv_diag; a.Ginv = c.Ginv; a.sinv_diag = c.sinv_diag; a.sig_diag = c.sig_diag;
    a.Sinv = c.Sinv; a.Sigma0 = c.Sigma0; a.ldk = c.ldk; a.ldp = c.ldp;
    a.S = c.S;
    const int threads = (int)round_up(c.J, 32);
    const size_t smem = small_smem(c);
    if (c.ensemble) {
        CES_TRY(allow_smem<small_step_kernel<true>>(smem));
        small_step_kernel<true><<<1, threads, smem, st>>>(a, c.seed, c.step);
    } else {
        CES_TRY(allow_smem<small_step_kernel<false>>(smem));
        small_step_kernel<false><<<1, threads, smem, st>>>(a, 0, 0);
    }
    CES_LAUNCHED(1);
    return CES_OK;
}

int small_run(cudaStream_t st, const SmallStepCall& c, const SmallRunCall& rc) {
    SmallRunArgs r;
    SmallArgs& a = r.base;
    a.p = (int)c.p; a.k = (int)c.k; a.J = (int)c.J; a.rule = c.rule; a.ts_kind = c.ts_kind;
    a.fixed_h = c.fixed_h; a.switch_ = c.switch_;
    a.U = nullptr; a.G = nullptr; a.xi = nullptr; a.ldu = a.ldg = a.ldxi = a.ldo = c.J; a.out = nullptr;
    a.y = c.y; a.mu = c.mu; a.ustar = c.ustar; a.bprior = c.bprior;
    a.ginv_diag = c.ginv_diag; a.Ginv = c.Ginv; a.sinv_diag = c.sinv_diag; a.sig_diag = c.sig_diag;
    a.Sinv = c.Sinv; a.Sigma0 = c.Sigma0; a.ldk = c.ldk; a.ldp = c.ldp;
    a.S = nullptr;
    r.T = (int)rc.T; r.map_kind = rc.map_kind; r.have_t0 = rc.have_t0; r.t0 = rc.t0; r.t_tol = rc.t_tol;
    r.A = rc.A; r.lda = rc.lda; r.b = rc.b; r.par0 = rc.par0; r.par1 = rc.par1;
    r.Utrace = rc.Utrace; r.Gtrace = rc.Gtrace; r.Xi = rc.Xi; r.Sall = rc.Sall; r.tvec = rc.tvec; r.nsteps = rc.nsteps;
    r.seed = c.seed; r.step0 = c.step;
    const int threads = (int)round_up(c.J, 32);
    const size_t smem = small_smem(c);
    if (c.ensemble) {
        a.xi = c.xi; a.ldxi = c.ldxi;   // one J x J xi for every iteration, or NULL (the stream)
        CES_TRY(allow_smem<small_run_kernel<true>>(smem));
        small_run_kernel<true><<<1, threads, smem, st>>>(r);
    } else {
        CES_TRY(allow_smem<small_run_kernel<false>>(smem));
        small_run_kernel<false><<<1, threads, smem, st>>>(r);
    }
    CES_LAUNCHED(1);
    return CES_OK;
}

}  // namespace ces
