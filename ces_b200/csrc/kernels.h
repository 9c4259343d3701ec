// Internal host-side interface between the translation units of libces_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "common.cuh"

namespace ces {

constexpr int GEMM_BM = 128, GEMM_BN = 128, GEMM_BK = 16;   // CTA tile of the DMMA GEMM

enum GemmFlags : int {
    GEMM_A_LOWER_TRI = 1,    // A (MK) is lower triangular: rows of tile tm need kk < (tm+1)*BM only
    GEMM_C_LOWER_ONLY = 2,   // compute only tiles with tn <= tm (symmetric result)
    GEMM_B_UPPER_TRI = 4,    // B (KN) is upper triangular: columns of tile tn need kk < (tn+1)*BN only
    GEMM_SERPENTINE_K = 8,   // odd waves of CTAs traverse the contraction axis backwards (L2 reuse across waves)
};

enum AMode : int { A_MK = 0, A_KM = 1 };
enum BMode : int { B_KN = 0, B_NK = 1 };

struct GemmCall {
    int a_mode = A_MK, b_mode = B_KN;
    int M = 0, N = 0, K = 0;
    const double* A = nullptr; int64_t lda = 0;
    const double* B = nullptr; int64_t ldb = 0;
    double* C = nullptr;       int64_t ldc = 0;
    double alpha = 1.0, beta = 0.0;
    const double* alpha_dev = nullptr;
    int flags = 0;
    int group_m = 0;
    double* ssq_partials = nullptr;   // [gemm_tiles(M,N)]
    int splits = 1;
    double* splitk_ws = nullptr;      // >= splits*M*N doubles; enables the reduce epilogue
    double diag_add = 0.0;            // reduce epilogue only
    // batched form: `batch` problems, operand rows shifted by z*{a,b}_batch_rows (0 = shared), C by z*c_batch_elems
    int64_t batch = 1, a_batch_rows = 0, b_batch_rows = 0, c_batch_elems = 0;
    // walk of the contraction axis (ces_gemm_ex): CTAs per wave (0 = SM count), serpentine -1 = CES_GEMM_SERPENTINE / on,
    // 0 = off, 1 = on
    int wave_ctas = 0, serpentine = -1;
};

int gemm(cudaStream_t st, const GemmCall& c);
int gemm_tiles(int M, int N);
int gemm_sm_count();   // SMs of the current device = CTAs of one wave of the GEMM (one CTA per SM)

// Device scalar block of a handle (doubles).
enum StepScalars : int {
    S_SSQ = 0,        // sum of squares of D (local until the host all-reduces it)
    S_SELF_BIAS = 1,  // sum_j |u_j - ubar|^2                (local partial sums of the four diagnostics)
    S_BIAS = 2,       // sum_j |u_j - ustar|^2
    S_SELF_DATA = 3,  // sum_j (e_j^T Gamma^-1 e_j)^2
    S_BIAS_DATA = 4,  // sum_j (r_j^T Gamma^-1 r_j)^2
    S_MAXDRIFT = 5,   // max |drift| (aldi_constant)
    S_H = 6, S_SQRT2H = 7, S_NEG_H = 8, S_H_ALPHA = 9,
    S_ENS_ALPHA = 10, // sqrt(2h / n_C): scale of the ensemble noise (U - ubar) xi (CES_NOISE_ENSEMBLE)
    S_INFO = 15,      // small path: 1 + index of the first non-positive Cholesky pivot (0 = ok)
    S_COUNT = 16,
};

// ensemble.cu
int row_sums(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, double* out);
int centre_g(cudaStream_t st, const double* G, int64_t ldg, int64_t k, int64_t cols, const double* sums, double inv_J,
             const double* y, const double* ginv_diag, double* E, double* W, int64_t ldo, double* cvec);
int centre_u(cudaStream_t st, const double* U, int64_t ldu, int64_t p, int64_t cols, const double* sums, double inv_J,
             const double* mu, const double* ustar, const double* sinv_diag, double* Ut, double* Z, int64_t ldo,
             double* qpart);
int form_rows_per_cta(int64_t rows, int64_t ld);
int form_row_blocks(int64_t rows, int64_t ld);
int data_forms(cudaStream_t st, const double* E, const double* W, int64_t ld, int64_t k, const double* cvec,
               const double* zvec, double* qpart);
int finish_forms(cudaStream_t st, const double* qpart, int ny, int64_t ld, int64_t cols, bool square, double* part,
                 double* out);
int sum_vector(cudaStream_t st, const double* v, int64_t n, double* out);
int row_sumsq(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, double* out);
int matvec(cudaStream_t st, const double* M, int64_t ld, int64_t n, const double* x, double* y);
int scale_vector(cudaStream_t st, const double* d, const double* x, double* y, int64_t n);
int step_scalars(cudaStream_t st, double* S, int kind, double fixed_h, double alpha_J, double inv_nc);
int axpbypcz(cudaStream_t st, int64_t rows, int64_t cols, double a, const double* X, int64_t ldx, double b,
             const double* b_dev, const double* Y, int64_t ldy, double c, const double* c_dev, const double* Z,
             int64_t ldz, double* out, int64_t ldo);
int absmax(cudaStream_t st, const double* X, int64_t ld, int64_t rows, int64_t cols, double* row_scratch, double* out);
int pad_copy(cudaStream_t st, const double* X, int64_t ldx, int64_t rows, int64_t cols, double* out, int64_t ldo);
int row_scale(cudaStream_t st, const double* diag, double* X, int64_t ld, int64_t rows, int64_t cols);
int add_col_vector(cudaStream_t st, double* X, int64_t ld, int64_t rows, int64_t cols, const double* v, double s,
                   const double* s_dev);
int fill_normal(cudaStream_t st, double* X, int64_t ld, int64_t rows, int64_t cols, int64_t col_offset, uint64_t seed,
                uint64_t step);
int fill_ensemble_noise(cudaStream_t st, double* X, int64_t ld, int64_t rows, int64_t cols, int64_t row_offset,
                        int64_t col_offset, uint64_t seed, uint64_t step);
int form_implicit(cudaStream_t st, const double* C, int64_t ldc, const double* Sigma0, int64_t lds,
                  const double* sig_diag, const double* h_dev, int64_t p, double* M, int64_t ldm);

// chol.cu -- blocked Cholesky and triangular solves built on the DMMA GEMM.
constexpr int CHOL_NB = 64;
// In-place lower Cholesky of the n x n SPD matrix A (row-major, ld).  The strict upper triangle is
// zeroed.  Linv receives the inverses of the CHOL_NB x CHOL_NB diagonal blocks of L, stacked:
// block b at Linv + b*CHOL_NB*ldinv (row-major, ldinv >= CHOL_NB, even).  *info_dev (device int)
// is set to (1 + index of the first non-positive pivot) on failure, left untouched otherwise.
int potrf_lower(cudaStream_t st, double* A, int64_t ld, int64_t n, double* Linv, int64_t ldinv, int* info_dev);
// B <- L^-1 B  (forward) / B <- L^-T B (backward) for an n x nrhs right-hand side (row-major, ldb).
int trsm_lower(cudaStream_t st, const double* L, int64_t ld, int64_t n, const double* Linv, int64_t ldinv,
               double* B, int64_t ldb, int64_t nrhs, bool transpose);
// Ainv <- A^-1 for SPD A given its factor (L, Linv): solves L L^T X = I.  Ainv is n x n, ld = ldo.
int spd_inverse_from_factor(cudaStream_t st, const double* L, int64_t ld, int64_t n, const double* Linv, int64_t ldinv,
                            double* Ainv, int64_t ldo);
int set_identity(cudaStream_t st, double* A, int64_t ld, int64_t n);

// eig.cu -- lambda_max(Gamma^-1 C) by Lanczos in the Gamma^-1 inner product (time_step='spectral')
int spectral_radius(cudaStream_t st, const double* C, int64_t ld, int64_t n, const double* Ginv, const double* ginv_diag,
                    double* work, int64_t mmax, double* lambda_host, int* steps_host);

// small.cu -- the whole update in one single-CTA kernel for small problems
constexpr int SMALL_P_MAX = 8, SMALL_K_MAX = 16;
struct SmallStepCall {
    int64_t p, k, J;
    int rule, ts_kind;
    double fixed_h, switch_;
    const double *U, *G, *xi;
    int64_t ldu, ldg, ldxi;
    double* out;
    int64_t ldo;
    const double *y, *mu, *ustar, *bprior, *ginv_diag, *Ginv, *sinv_diag, *sig_diag, *Sinv, *Sigma0;
    int64_t ldk, ldp;
    double* S;
};
bool small_step_eligible(int64_t p, int64_t k, int64_t J);
int small_step(cudaStream_t st, const SmallStepCall& c);
// the whole run loop (forward map + update per iteration, stopping rule) of a small problem in one launch
struct SmallRunCall {
    int64_t T;
    int map_kind, have_t0;
    double t0, t_tol;
    const double* A; int64_t lda; const double* b;
    double par0, par1;
    double *Utrace, *Gtrace;
    const double* Xi;
    double *Sall, *tvec;
    int* nsteps;
};
int small_run(cudaStream_t st, const SmallStepCall& c, const SmallRunCall& rc);

// darcy.cu -- the body of ces_darcy_forward without its final synchronisation (valid arguments assumed): enqueues the
// pipeline for U (p x cols) -> G on the model's stream and leaves the largest / summed CG iteration count of the call in
// the device ints `iters` of darcy_shape.  darcy_max_iter resolves the iteration limit (<= 0: the default, 40 N).
struct DarcyModel;
struct DarcyShape {
    int N, p, n_obs;
    cudaStream_t st;
    const int* iters;
};
int darcy_forward_async(DarcyModel* m, const double* U, int64_t ldu, int64_t cols, double* G, int64_t ldg, int full_solution,
                        double tol, int max_iter);
int darcy_max_iter(const DarcyModel* m, int max_iter);
DarcyShape darcy_shape(const DarcyModel* m);

// forward.cu
int exp_map(cudaStream_t st, const double* X, int64_t ldx, int64_t rows, int64_t cols, double* out, int64_t ldo);
int elliptic_map(cudaStream_t st, const double* U, int64_t ldu, int64_t cols, double x1, double x2, double* G, int64_t ldg);
int banana_map(cudaStream_t st, const double* U, int64_t ldu, int64_t cols, double a, double b, double* G, int64_t ldg);

}  // namespace ces
