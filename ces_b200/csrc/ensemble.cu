// Bandwidth-bound ensemble kernels: row sums over particles, centring, per-particle quadratic
// forms for the diagnostics, step-size scalars and the final assembly of U_{n+1}.
// Reference arithmetic: ces/calibrate.py:423-435, 459-467, 475-488 (see DESIGN.md kernel table).
#include "kernels.h"
#include "rng.cuh"

namespace ces {

// ------------------------------------------------------------------------------------------
// Row sums over the particle axis: out[r] = sum_j X[r, j], j < cols.   One CTA per row.
// 16-byte loads when the row is 16-byte aligned, four loads in flight per thread.
template <bool VEC>
__global__ void __launch_bounds__(256) row_sums_kernel(const double* __restrict__ X, long long ld, long long cols,
                                                       double* __restrict__ out) {
    __shared__ double scratch[32];
    const double* row = X + (size_t)blockIdx.x * ld;
    double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
    if (VEC) {
        const long long n2 = cols >> 1;
        const double2* r2 = reinterpret_cast<const double2*>(row);
        long long i = threadIdx.x;
        for (; i + 3 * 256 < n2; i += 4 * 256) {
            const double2 a = r2[i], b = r2[i + 256], c = r2[i + 512], d = r2[i + 768];
            s0 += a.x + a.y; s1 += b.x + b.y; s2 += c.x + c.y; s3 += d.x + d.y;
        }
        for (; i < n2; i += 256) { const double2 a = r2[i]; s0 += a.x + a.y; }
        if ((cols & 1) && threadIdx.x == 0) s1 += row[cols - 1];
    } else {
        long long i = threadIdx.x;
        for (; i + 3 * 256 < cols; i += 4 * 256) {
            s0 += row[i]; s1 += row[i + 256]; s2 += row[i + 512]; s3 += row[i + 768];
        }
        for (; i < cols; i += 256) s0 += row[i];
    }
    const double tot = block_sum((s0 + s1) + (s2 + s3), scratch);
    if (threadIdx.x == 0) out[blockIdx.x] = tot;
}

int row_sums(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, double* out) {
    if (rows < 1) return CES_OK;
    const bool vec = ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && (ld % 2 == 0);
    if (vec) row_sums_kernel<true><<<(unsigned)rows, 256, 0, st>>>(X, ld, cols, out);
    else     row_sums_kernel<false><<<(unsigned)rows, 256, 0, st>>>(X, ld, cols, out);
    CES_LAUNCHED(1);
    return CES_OK;
}

// ------------------------------------------------------------------------------------------
// Centring of the forward-output ensemble (ces/calibrate.py:427-428):
//   E = G - mean_J(G),  R = G - y,  and either W = R * ginv (diagonal Gamma) or R itself (dense
//   Gamma; W = Gamma^-1 R follows as a GEMM).  Also c = mean - y (k-vector), written by column-block 0.
// Thread = 2 adjacent particles x CENTRE_ROWS rows; columns >= cols (padding up to ldo) get zeros.
constexpr int CENTRE_ROWS = 8;

template <bool VEC>
__global__ void __launch_bounds__(256) centre_g_kernel(const double* __restrict__ G, long long ldg, int k, long long cols,
                                                       const double* __restrict__ sums, double inv_J,
                                                       const double* __restrict__ y, const double* __restrict__ ginv_diag,
                                                       double* __restrict__ E, double* __restrict__ W, long long ldo,
                                                       double* __restrict__ cvec) {
    const long long j = 2 * ((long long)blockIdx.x * 256 + threadIdx.x);
    if (j >= ldo) return;
    const int m0 = blockIdx.y * CENTRE_ROWS;
#pragma unroll
    for (int r = 0; r < CENTRE_ROWS; ++r) {
        const int m = m0 + r;
        if (m >= k) break;
        const double mean = sums[m] * inv_J, ym = y[m];
        const double gs = ginv_diag ? ginv_diag[m] : 1.0;
        double g0 = 0.0, g1 = 0.0;
        const bool in0 = j < cols, in1 = j + 1 < cols;
        if (VEC) {
            if (in1) { const double2 v = *reinterpret_cast<const double2*>(G + (size_t)m * ldg + j); g0 = v.x; g1 = v.y; }
            else if (in0) g0 = G[(size_t)m * ldg + j];
        } else {
            if (in0) g0 = G[(size_t)m * ldg + j];
            if (in1) g1 = G[(size_t)m * ldg + j + 1];
        }
        double2 e, w;
        e.x = in0 ? g0 - mean : 0.0;        e.y = in1 ? g1 - mean : 0.0;
        w.x = in0 ? (g0 - ym) * gs : 0.0;   w.y = in1 ? (g1 - ym) * gs : 0.0;
        *reinterpret_cast<double2*>(E + (size_t)m * ldo + j) = e;
        *reinterpret_cast<double2*>(W + (size_t)m * ldo + j) = w;
        if (blockIdx.x == 0 && threadIdx.x == 0) cvec[m] = mean - ym;
    }
}

int centre_g(cudaStream_t st, const double* G, int64_t ldg, int64_t k, int64_t cols, const double* sums, double inv_J,
             const double* y, const double* ginv_diag, double* E, double* W, int64_t ldo, double* cvec) {
    const bool vec = ((reinterpret_cast<uintptr_t>(G) & 15) == 0) && (ldg % 2 == 0);
    dim3 grid((unsigned)ceil_div(ldo, 512), (unsigned)ceil_div(k, CENTRE_ROWS));
    if (vec) centre_g_kernel<true><<<grid, 256, 0, st>>>(G, ldg, (int)k, cols, sums, inv_J, y, ginv_diag, E, W, ldo, cvec);
    else     centre_g_kernel<false><<<grid, 256, 0, st>>>(G, ldg, (int)k, cols, sums, inv_J, y, ginv_diag, E, W, ldo, cvec);
    CES_LAUNCHED(1);
    return CES_OK;
}

// Centring of the parameter ensemble (ces/calibrate.py:423, 475, 485):
//   Ut = U - mean_J(U);  Z = (U - mu) * sinv (diagonal Sigma0) or U - mu (dense; Z = Sigma0^-1 (.) follows
//   as a GEMM).  Per-particle partial sums over this CTA's rows for the two parameter-space diagnostics
//   (:432-433): q_self[j] += Ut_ij^2, q_bias[j] += (U_ij - ustar_i)^2  -> qpart[2][gridDim.y][ldo].
template <bool VEC>
__global__ void __launch_bounds__(256) centre_u_kernel(const double* __restrict__ U, long long ldu, int p, long long cols,
                                                       const double* __restrict__ sums, double inv_J,
                                                       const double* __restrict__ mu, const double* __restrict__ ustar,
                                                       const double* __restrict__ sinv_diag, double* __restrict__ Ut,
                                                       double* __restrict__ Z, long long ldo, double* __restrict__ qpart,
                                                       int rows_per_cta) {
    const long long j = 2 * ((long long)blockIdx.x * 256 + threadIdx.x);
    if (j >= ldo) return;
    const int i0 = blockIdx.y * rows_per_cta;
    double qs0 = 0, qs1 = 0, qb0 = 0, qb1 = 0;
    const bool in0 = j < cols, in1 = j + 1 < cols;
#pragma unroll 4
    for (int r = 0; r < rows_per_cta; ++r) {
        const int i = i0 + r;
        if (i >= p) break;
        const double mean = sums[i] * inv_J, mui = mu[i], us = ustar[i];
        const double ss = sinv_diag ? sinv_diag[i] : 1.0;
        double u0 = 0.0, u1 = 0.0;
        if (VEC) {
            if (in1) { const double2 v = *reinterpret_cast<const double2*>(U + (size_t)i * ldu + j); u0 = v.x; u1 = v.y; }
            else if (in0) u0 = U[(size_t)i * ldu + j];
        } else {
            if (in0) u0 = U[(size_t)i * ldu + j];
            if (in1) u1 = U[(size_t)i * ldu + j + 1];
        }
        double2 t, z;
        t.x = in0 ? u0 - mean : 0.0;         t.y = in1 ? u1 - mean : 0.0;
        z.x = in0 ? (u0 - mui) * ss : 0.0;   z.y = in1 ? (u1 - mui) * ss : 0.0;
        *reinterpret_cast<double2*>(Ut + (size_t)i * ldo + j) = t;
        if (Z) *reinterpret_cast<double2*>(Z + (size_t)i * ldo + j) = z;
        qs0 += t.x * t.x; qs1 += t.y * t.y;
        if (in0) qb0 += (u0 - us) * (u0 - us);
        if (in1) qb1 += (u1 - us) * (u1 - us);
    }
    double* q_self = qpart + (size_t)blockIdx.y * ldo;
    double* q_bias = qpart + ((size_t)gridDim.y + blockIdx.y) * ldo;
    *reinterpret_cast<double2*>(q_self + j) = make_double2(qs0, qs1);
    *reinterpret_cast<double2*>(q_bias + j) = make_double2(qb0, qb1);
}

// Rows handled by one CTA of the kernels that emit per-particle partial sums: enough CTAs for ~4 waves
// of 148 SMs, and few enough row blocks that the partial-sum pass stays small.
int form_rows_per_cta(int64_t rows, int64_t ld) {
    const int64_t col_blocks = ceil_div(ld, 512);
    int64_t target = 592 / col_blocks;
    if (target < 1) target = 1;
    int64_t rpc = round_up(ceil_div(rows, target), 8);
    return (int)(rpc < 8 ? 8 : rpc);
}
int form_row_blocks(int64_t rows, int64_t ld) { return (int)ceil_div(rows, form_rows_per_cta(rows, ld)); }

int centre_u(cudaStream_t st, const double* U, int64_t ldu, int64_t p, int64_t cols, const double* sums, double inv_J,
             const double* mu, const double* ustar, const double* sinv_diag, double* Ut, double* Z, int64_t ldo,
             double* qpart) {
    const bool vec = ((reinterpret_cast<uintptr_t>(U) & 15) == 0) && (ldu % 2 == 0);
    const int rpc = form_rows_per_cta(p, ldo);
    dim3 grid((unsigned)ceil_div(ldo, 512), (unsigned)ceil_div(p, rpc));
    if (vec) centre_u_kernel<true><<<grid, 256, 0, st>>>(U, ldu, (int)p, cols, sums, inv_J, mu, ustar, sinv_diag, Ut, Z, ldo, qpart, rpc);
    else     centre_u_kernel<false><<<grid, 256, 0, st>>>(U, ldu, (int)p, cols, sums, inv_J, mu, ustar, sinv_diag, Ut, Z, ldo, qpart, rpc);
    CES_LAUNCHED(1);
    return CES_OK;
}

// Per-particle data-space quadratic forms (ces/calibrate.py:434-435) without the reference's two
// extra J x J products:  with W = Gamma^-1 R, c = mean - y, z = Gamma^-1 c and R = E + c 1^T,
//   e_j^T Gamma^-1 e_j = sum_m E_mj (W_mj - z_m),      r_j^T Gamma^-1 r_j = sum_m (E_mj + c_m) W_mj.
// Partial sums over this CTA's rows -> qpart[2][gridDim.y][ld].
__global__ void __launch_bounds__(256) data_forms_kernel(const double* __restrict__ E, const double* __restrict__ W,
                                                         long long ld, int k, const double* __restrict__ cvec,
                                                         const double* __restrict__ zvec, double* __restrict__ qpart,
                                                         int rows_per_cta) {
    const long long j = 2 * ((long long)blockIdx.x * 256 + threadIdx.x);
    if (j >= ld) return;
    const int m0 = blockIdx.y * rows_per_cta;
    double qe0 = 0, qe1 = 0, qr0 = 0, qr1 = 0;
#pragma unroll 4
    for (int r = 0; r < rows_per_cta; ++r) {
        const int m = m0 + r;
        if (m >= k) break;
        const double2 e = *reinterpret_cast<const double2*>(E + (size_t)m * ld + j);
        const double2 w = *reinterpret_cast<const double2*>(W + (size_t)m * ld + j);
        const double c = cvec[m], z = zvec[m];
        qe0 += e.x * (w.x - z); qe1 += e.y * (w.y - z);
        qr0 += (e.x + c) * w.x; qr1 += (e.y + c) * w.y;
    }
    double* q_e = qpart + (size_t)blockIdx.y * ld;
    double* q_r = qpart + ((size_t)gridDim.y + blockIdx.y) * ld;
    *reinterpret_cast<double2*>(q_e + j) = make_double2(qe0, qe1);
    *reinterpret_cast<double2*>(q_r + j) = make_double2(qr0, qr1);
}

int data_forms(cudaStream_t st, const double* E, const double* W, int64_t ld, int64_t k, const double* cvec,
               const double* zvec, double* qpart) {
    const int rpc = form_rows_per_cta(k, ld);
    dim3 grid((unsigned)ceil_div(ld, 512), (unsigned)ceil_div(k, rpc));
    data_forms_kernel<<<grid, 256, 0, st>>>(E, W, ld, (int)k, cvec, zvec, qpart, rpc);
    CES_LAUNCHED(1);
    return CES_OK;
}

// part[0][b] = sum_{j in block b} f(sum_y qpart[0][y][j]), part[1][b] likewise for qpart[1]; j < cols;
// f = identity (SQUARE=false) or square (SQUARE=true).  One column per thread, fixed order.
template <bool SQUARE>
__global__ void __launch_bounds__(256) finish_forms_kernel(const double* __restrict__ qpart, int ny, long long ld,
                                                           long long cols, double* __restrict__ part) {
    __shared__ double scratch[32];
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    double a0 = 0.0, a1 = 0.0;
    if (j < cols) {
        double q0 = 0.0, q1 = 0.0;
        for (int y = 0; y < ny; ++y) {
            q0 += qpart[(size_t)y * ld + j];
            q1 += qpart[((size_t)ny + y) * ld + j];
        }
        a0 = SQUARE ? q0 * q0 : q0;
        a1 = SQUARE ? q1 * q1 : q1;
    }
    const double t0 = block_sum(a0, scratch);
    const double t1 = block_sum(a1, scratch);
    if (threadIdx.x == 0) { part[blockIdx.x] = t0; part[gridDim.x + blockIdx.x] = t1; }
}
// out[0] = sum part[0][:], out[1] = sum part[1][:]  (one CTA, fixed order -> deterministic)
__global__ void __launch_bounds__(256) finish_pair_kernel(const double* __restrict__ part, int n, double* __restrict__ out) {
    __shared__ double scratch[32];
    double a0 = 0.0, a1 = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) { a0 += part[i]; a1 += part[n + i]; }
    const double t0 = block_sum(a0, scratch);
    const double t1 = block_sum(a1, scratch);
    if (threadIdx.x == 0) { out[0] = t0; out[1] = t1; }
}

// `part` holds 2 * ceil(cols / 256) doubles of scratch.
int finish_forms(cudaStream_t st, const double* qpart, int ny, int64_t ld, int64_t cols, bool square, double* part,
                 double* out) {
    const int nb = (int)ceil_div(cols < 1 ? 1 : cols, 256);
    if (square) finish_forms_kernel<true><<<nb, 256, 0, st>>>(qpart, ny, ld, cols, part);
    else        finish_forms_kernel<false><<<nb, 256, 0, st>>>(qpart, ny, ld, cols, part);
    finish_pair_kernel<<<1, 256, 0, st>>>(part, nb, out);
    CES_LAUNCHED(2);
    return CES_OK;
}

// out[r] = sum_j X[r, j]^2  (rows of a matrix whose Frobenius norm is wanted: timestep_method(D, ...), :248)
__global__ void __launch_bounds__(256) row_sumsq_kernel(const double* __restrict__ X, long long ld, long long cols,
                                                        double* __restrict__ out) {
    __shared__ double scratch[32];
    const double* row = X + (size_t)blockIdx.x * ld;
    double s = 0.0;
    for (long long i = threadIdx.x; i < cols; i += 256) s += row[i] * row[i];
    const double t = block_sum(s, scratch);
    if (threadIdx.x == 0) out[blockIdx.x] = t;
}
int row_sumsq(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, double* out) {
    row_sumsq_kernel<<<(unsigned)rows, 256, 0, st>>>(X, ld, cols, out);
    CES_LAUNCHED(1);
    return CES_OK;
}

// out[0] = sum of n doubles, fixed order (one CTA).
__global__ void __launch_bounds__(1024) sum_vector_kernel(const double* __restrict__ v, long long n, double* __restrict__ out) {
    __shared__ double scratch[32];
    double a = 0.0;
    for (long long i = threadIdx.x; i < n; i += 1024) a += v[i];
    const double t = block_sum(a, scratch);
    if (threadIdx.x == 0) out[0] = t;
}
int sum_vector(cudaStream_t st, const double* v, int64_t n, double* out) {
    sum_vector_kernel<<<1, 1024, 0, st>>>(v, n, out);
    CES_LAUNCHED(1);
    return CES_OK;
}

// y = M x for a small dense row-major matrix (n x n): z = Gamma^-1 c, b = Sigma0^-1 mu ...  One warp per row.
__global__ void __launch_bounds__(256) matvec_kernel(const double* __restrict__ M, long long ld, int n,
                                                     const double* __restrict__ x, double* __restrict__ y) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= n) return;
    double a = 0.0;
    for (int c = lane; c < n; c += 32) a += M[(size_t)row * ld + c] * x[c];
    a = warp_sum(a);
    if (lane == 0) y[row] = a;
}
int matvec(cudaStream_t st, const double* M, int64_t ld, int64_t n, const double* x, double* y) {
    matvec_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, st>>>(M, ld, (int)n, x, y);
    CES_LAUNCHED(1);
    return CES_OK;
}
__global__ void scale_vector_kernel(const double* __restrict__ d, const double* __restrict__ x, double* __restrict__ y, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = d[i] * x[i];
}
int scale_vector(cudaStream_t st, const double* d, const double* x, double* y, int64_t n) {
    scale_vector_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(d, x, y, (int)n);
    CES_LAUNCHED(1);
    return CES_OK;
}

// ------------------------------------------------------------------------------------------
// Step-size scalars (ces/calibrate.py:247-260, 519).  S layout: see StepScalars in kernels.h.
//   kind 0: hk = 1 / (sqrt(ssq) + 1e-8)          (default, :248)
//   kind 1: hk = fixed                           ('constant', :253; 'mix' after spin-up, :260)
//   kind 2: hk = 0.1 / max|drift|                ('aldi_constant', :519)
//   inv_nc > 0 (ensemble noise): S_ENS_ALPHA = sqrt(2 h / n_C), the scale of (U - ubar) xi; left untouched otherwise
__global__ void step_scalars_kernel(double* __restrict__ S, int kind, double fixed_h, double alpha_J, double inv_nc) {
    double h;
    if (kind == 0) h = 1.0 / (sqrt(S[S_SSQ]) + 1e-8);
    else if (kind == 1) h = fixed_h;
    else h = 0.1 / S[S_MAXDRIFT];
    S[S_H] = h;
    S[S_SQRT2H] = sqrt(2.0 * h);
    S[S_NEG_H] = -h;
    S[S_H_ALPHA] = h * alpha_J;
    if (inv_nc > 0.0) S[S_ENS_ALPHA] = sqrt(2.0 * h * inv_nc);
}
int step_scalars(cudaStream_t st, double* S, int kind, double fixed_h, double alpha_J, double inv_nc) {
    step_scalars_kernel<<<1, 1, 0, st>>>(S, kind, fixed_h, alpha_J, inv_nc);
    CES_LAUNCHED(1);
    return CES_OK;
}

// ------------------------------------------------------------------------------------------
// out = a*X + (*b_dev)*b*Y + (*c_dev)*c*Z   elementwise over rows x cols (any of the device scalars
// may be null = 1).  Used to assemble U + h*alpha_J*Ut - h*V (:484-486) before the two GEMMs that add
// the prior drift and the noise, and to form the aldi_constant drift (:515-517).
__global__ void __launch_bounds__(256) axpbypcz_kernel(int rows, long long cols, double a, const double* __restrict__ X,
                                                       long long ldx, double b, const double* __restrict__ b_dev,
                                                       const double* __restrict__ Y, long long ldy, double c,
                                                       const double* __restrict__ c_dev, const double* __restrict__ Z,
                                                       long long ldz, double* __restrict__ out, long long ldo) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    const int i = blockIdx.y;
    if (j >= cols) return;
    const double bb = b * (b_dev ? *b_dev : 1.0), cc = c * (c_dev ? *c_dev : 1.0);
    double v = a * X[(size_t)i * ldx + j];
    if (Y) v += bb * Y[(size_t)i * ldy + j];
    if (Z) v += cc * Z[(size_t)i * ldz + j];
    out[(size_t)i * ldo + j] = v;
}
int axpbypcz(cudaStream_t st, int64_t rows, int64_t cols, double a, const double* X, int64_t ldx, double b,
             const double* b_dev, const double* Y, int64_t ldy, double c, const double* c_dev, const double* Z,
             int64_t ldz, double* out, int64_t ldo) {
    dim3 grid((unsigned)ceil_div(cols, 256), (unsigned)rows);
    axpbypcz_kernel<<<grid, 256, 0, st>>>((int)rows, cols, a, X, ldx, b, b_dev, Y, ldy, c, c_dev, Z, ldz, out, ldo);
    CES_LAUNCHED(1);
    return CES_OK;
}

// max |X| over rows x cols -> out[0] (two launches: per-row maxima then one CTA).
__global__ void __launch_bounds__(256) row_absmax_kernel(const double* __restrict__ X, long long ld, long long cols,
                                                         double* __restrict__ out) {
    __shared__ double scratch[32];
    const double* row = X + (size_t)blockIdx.x * ld;
    double m = 0.0;
    for (long long i = threadIdx.x; i < cols; i += 256) m = fmax(m, fabs(row[i]));
    m = block_max(m, scratch);
    if (threadIdx.x == 0) out[blockIdx.x] = m;
}
__global__ void __launch_bounds__(1024) max_vector_kernel(const double* __restrict__ v, long long n, double* __restrict__ out) {
    __shared__ double scratch[32];
    double m = 0.0;
    for (long long i = threadIdx.x; i < n; i += 1024) m = fmax(m, v[i]);
    m = block_max(m, scratch);
    if (threadIdx.x == 0) out[0] = m;
}
int absmax(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, double* row_scratch, double* out) {
    row_absmax_kernel<<<(unsigned)rows, 256, 0, st>>>(X, ld, cols, row_scratch);
    max_vector_kernel<<<1, 1024, 0, st>>>(row_scratch, rows, out);
    CES_LAUNCHED(2);
    return CES_OK;
}

// Copy a rows x cols matrix between leading dimensions, zero-filling columns [cols, ldo).
__global__ void __launch_bounds__(256) pad_copy_kernel(const double* __restrict__ X, long long ldx, long long cols,
                                                       double* __restrict__ out, long long ldo) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    if (j >= ldo) return;
    out[(size_t)blockIdx.y * ldo + j] = j < cols ? X[(size_t)blockIdx.y * ldx + j] : 0.0;
}
int pad_copy(cudaStream_t st, const double* X, int64_t ldx, int64_t rows, int64_t cols, double* out, int64_t ldo) {
    dim3 grid((unsigned)ceil_div(ldo, 256), (unsigned)rows);
    pad_copy_kernel<<<grid, 256, 0, st>>>(X, ldx, cols, out, ldo);
    CES_LAUNCHED(1);
    return CES_OK;
}

// out[i][j] = diag[i] * X[i][j]  (row scaling: Sigma0 * X for diagonal Sigma0 in the implicit EKS solve).
__global__ void __launch_bounds__(256) row_scale_kernel(const double* __restrict__ diag, double* __restrict__ X,
                                                        long long ld, long long cols) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    if (j >= cols) return;
    X[(size_t)blockIdx.y * ld + j] *= diag[blockIdx.y];
}
// col_dot: partial sums over this CTA's rows of X[m, j] v[m] -> part[blockIdx.y][ld] (two columns per thread, as
// data_forms), then one fixed-order sum over the row blocks per column: deterministic.
__global__ void __launch_bounds__(256) col_dot_kernel(const double* __restrict__ X, long long ld, int rows,
                                                      const double* __restrict__ v, double* __restrict__ part,
                                                      int rows_per_cta) {
    const long long j = 2 * ((long long)blockIdx.x * 256 + threadIdx.x);
    if (j >= ld) return;
    const int m0 = blockIdx.y * rows_per_cta;
    double a0 = 0.0, a1 = 0.0;
#pragma unroll 4
    for (int r = 0; r < rows_per_cta; ++r) {
        const int m = m0 + r;
        if (m >= rows) break;
        const double2 x = *reinterpret_cast<const double2*>(X + (size_t)m * ld + j);
        const double w = v[m];
        a0 += x.x * w; a1 += x.y * w;
    }
    *reinterpret_cast<double2*>(part + (size_t)blockIdx.y * ld + j) = make_double2(a0, a1);
}
__global__ void __launch_bounds__(256) col_dot_finish_kernel(const double* __restrict__ part, int ny, long long ld,
                                                             long long cols, double* __restrict__ out) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    if (j >= cols) return;
    double s = 0.0;
    for (int y = 0; y < ny; ++y) s += part[(size_t)y * ld + j];
    out[j] = s;
}
int col_dot(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, const double* v, double* part,
            double* out) {
    const int rpc = form_rows_per_cta(rows, ld);
    const int ny = (int)ceil_div(rows, rpc);
    col_dot_kernel<<<dim3((unsigned)ceil_div(ld, 512), (unsigned)ny), 256, 0, st>>>(X, ld, (int)rows, v, part, rpc);
    col_dot_finish_kernel<<<(unsigned)ceil_div(cols, 256), 256, 0, st>>>(part, ny, ld, cols, out);
    CES_LAUNCHED(2);
    return CES_OK;
}

// row_dot: one CTA per row, fixed-order block sum
__global__ void __launch_bounds__(256) row_dot_kernel(const double* __restrict__ X, long long ld, long long cols,
                                                      const double* __restrict__ v, double s, double* __restrict__ out) {
    __shared__ double scratch[32];
    const double* row = X + (size_t)blockIdx.x * ld;
    double a = 0.0;
    for (long long i = threadIdx.x; i < cols; i += 256) a += row[i] * v[i];
    const double t = block_sum(a, scratch);
    if (threadIdx.x == 0) out[blockIdx.x] = s * t;
}
int row_dot(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, const double* v, double s, double* out) {
    row_dot_kernel<<<(unsigned)rows, 256, 0, st>>>(X, ld, cols, v, s, out);
    CES_LAUNCHED(1);
    return CES_OK;
}

int row_scale(cudaStream_t st, const double* diag, double* X, int64_t ld, int64_t rows, int64_t cols) {
    dim3 grid((unsigned)ceil_div(cols, 256), (unsigned)rows);
    row_scale_kernel<<<grid, 256, 0, st>>>(diag, X, ld, cols);
    CES_LAUNCHED(1);
    return CES_OK;
}

// X[i][j] += v[i]  (adds the constant vector h*C*Sigma0^-1*mu to every particle, :445).
__global__ void __launch_bounds__(256) add_col_vector_kernel(double* __restrict__ X, long long ld, long long cols,
                                                             const double* __restrict__ v, double s,
                                                             const double* __restrict__ s_dev) {
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    if (j >= cols) return;
    X[(size_t)blockIdx.y * ld + j] += s * (s_dev ? *s_dev : 1.0) * v[blockIdx.y];
}
int add_col_vector(cudaStream_t st, double* X, int64_t ld, int64_t rows, int64_t cols, const double* v, double s,
                   const double* s_dev) {
    dim3 grid((unsigned)ceil_div(cols, 256), (unsigned)rows);
    add_col_vector_kernel<<<grid, 256, 0, st>>>(X, ld, cols, v, s, s_dev);
    CES_LAUNCHED(1);
    return CES_OK;
}

// ------------------------------------------------------------------------------------------
// Standard normal noise generated on the device (production alternative to the host numpy draw of
// ces/calibrate.py:447,488,527): Philox4x32-10 keyed by the seed, counter = (global element pair, step), two
// 53-bit uniforms per call turned into two normals by Box-Muller.  The value of element (row, global column)
// depends only on (seed, step, row, column), so a column-sharded ensemble draws what a single GPU would.
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
__global__ void __launch_bounds__(256) fill_normal_kernel(double* __restrict__ X, long long ld, int rows, long long cols,
                                                          long long col_offset, unsigned long long seed,
                                                          unsigned long long step) {
    // one thread per GLOBAL column pair (2g, 2g+1) that intersects this shard [col_offset, col_offset + cols): the
    // stream depends only on (seed, step, row, global column), so any sharding -- odd offsets and odd widths
    // included -- reproduces the columns of a single-GPU draw
    const unsigned long long gpair = ((unsigned long long)col_offset >> 1) + (unsigned long long)blockIdx.x * 256 + threadIdx.x;
    const int row = blockIdx.y;
    const long long j = (long long)(2 * gpair) - col_offset;               // local index of the pair's first column (may be -1)
    if (j >= cols) return;
    uint32_t c[4] = {(uint32_t)gpair, (uint32_t)(gpair >> 32), (uint32_t)row, (uint32_t)step};
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    const double two53 = 1.0 / 9007199254740992.0;      // (0, 1): the top 53-bit value would round to 1.0 without the fmin
    const double u1 = fmin(((double)((((unsigned long long)c[0] << 32) | c[1]) >> 11) + 0.5) * two53, 1.0 - two53);
    const double u2 = fmin(((double)((((unsigned long long)c[2] << 32) | c[3]) >> 11) + 0.5) * two53, 1.0 - two53);
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    if (j >= 0) X[(size_t)row * ld + j] = rad * cs;
    if (j + 1 < cols) X[(size_t)row * ld + j + 1] = rad * sn;
}
int fill_normal(cudaStream_t st, double* X, int64_t ld, int64_t rows, int64_t cols, int64_t col_offset, uint64_t seed,
                uint64_t step) {
    if (rows < 1 || cols < 1) return CES_OK;
    if (col_offset < 0) return fail(CES_ERR_INVALID, "fill_normal: negative column offset%s", "");
    const int64_t pairs = ((col_offset + cols - 1) >> 1) - (col_offset >> 1) + 1;
    dim3 grid((unsigned)ceil_div(pairs, 256), (unsigned)rows);
    fill_normal_kernel<<<grid, 256, 0, st>>>(X, ld, (int)rows, cols, col_offset, seed, step);
    CES_LAUNCHED(1);
    return CES_OK;
}

// A block of xi (J x J) of the ensemble noise sqrt(2h / n_C) (U - ubar) xi, elements as rng.cuh ensemble_noise_pair draws
// them.  An element depends only on (seed, step, global s, global j): any block of rows and columns, odd offsets included,
// reproduces what one GPU draws.  Rows go on blockIdx.y with a grid-stride loop (gridDim.y <= 65535 < J).
__global__ void __launch_bounds__(256) fill_ensemble_noise_kernel(double* __restrict__ X, long long ld, long long rows,
                                                                  long long cols, long long row_offset, long long col_offset,
                                                                  unsigned long long seed, unsigned long long step) {
    const unsigned long long gpair = ((unsigned long long)col_offset >> 1) + (unsigned long long)blockIdx.x * 256 + threadIdx.x;
    const long long j = (long long)(2 * gpair) - col_offset;               // local index of the pair's first column (may be -1)
    if (j >= cols) return;
    for (long long r = blockIdx.y; r < rows; r += gridDim.y) {
        const double2 z = ensemble_noise_pair(seed, step, (unsigned long long)(row_offset + r), gpair);
        double* row = X + (size_t)r * ld;
        if (j >= 0) row[j] = z.x;
        if (j + 1 < cols) row[j + 1] = z.y;
    }
}
int fill_ensemble_noise(cudaStream_t st, double* X, int64_t ld, int64_t rows, int64_t cols, int64_t row_offset,
                        int64_t col_offset, uint64_t seed, uint64_t step) {
    if (rows < 1 || cols < 1) return CES_OK;
    if (row_offset < 0 || col_offset < 0) return fail(CES_ERR_INVALID, "fill_ensemble_noise: negative offset%s", "");
    const int64_t pairs = ((col_offset + cols - 1) >> 1) - (col_offset >> 1) + 1;
    dim3 grid((unsigned)ceil_div(pairs, 256), (unsigned)(rows < 65535 ? rows : 65535));
    fill_ensemble_noise_kernel<<<grid, 256, 0, st>>>(X, ld, rows, cols, row_offset, col_offset, seed, step);
    CES_LAUNCHED(1);
    return CES_OK;
}

// M = Sigma0 + (*h) * C  (dense, p x p) or diag(sig) + (*h) * C.
__global__ void __launch_bounds__(256) form_implicit_kernel(const double* __restrict__ C, long long ldc,
                                                            const double* __restrict__ Sigma0, long long lds,
                                                            const double* __restrict__ sig_diag,
                                                            const double* __restrict__ h_dev, int p,
                                                            double* __restrict__ M, long long ldm) {
    const int j = blockIdx.x * 256 + threadIdx.x, i = blockIdx.y;
    if (j >= p) return;
    double v = (*h_dev) * C[(size_t)i * ldc + j];
    if (Sigma0) v += Sigma0[(size_t)i * lds + j];
    else if (i == j) v += sig_diag[i];
    M[(size_t)i * ldm + j] = v;
}
int form_implicit(cudaStream_t st, const double* C, int64_t ldc, const double* Sigma0, int64_t lds,
                  const double* sig_diag, const double* h_dev, int64_t p, double* M, int64_t ldm) {
    dim3 grid((unsigned)ceil_div(p, 256), (unsigned)p);
    form_implicit_kernel<<<grid, 256, 0, st>>>(C, ldc, Sigma0, lds, sig_diag, h_dev, (int)p, M, ldm);
    CES_LAUNCHED(1);
    return CES_OK;
}

}  // namespace ces
