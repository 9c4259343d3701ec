/* ces_b200 -- C ABI of the B200-native ensemble Kalman update (libces_b200.so).
 *
 * Drop-in boundary for the numpy update of agarbuno/ces `ces/calibrate.py`.  The reference has no
 * FFI of its own (it is pure Python); these entry points are what `ces_b200/calibrate.py` binds
 * through ctypes in place of the numpy/LAPACK calls of
 *     sampling.eks_update                (ces/calibrate.py:418-449)
 *     sampling.eks_update_aldi           (ces/calibrate.py:451-490)   default rule
 *     sampling.eks_update_aldi_constant  (ces/calibrate.py:492-529)
 *     sampling.timestep_method           (ces/calibrate.py:243-267)
 *     enka.G_ens over the ces.utils maps (ces/calibrate.py:106-130, ces/utils.py:5-122)
 * INTEGRATION.md shows the reference-side stub a maintainer would add.
 *
 * Conventions
 *   - plain C types only; every matrix is row-major float64 with an explicit leading dimension (in
 *     elements); ensembles are (p x J) and (k x J) with the particle index contiguous, exactly the
 *     reference's layout (ces/calibrate.py:56-57, 123).
 *   - `*_dev` pointers are CUDA device pointers, `*_host` pointers are host pointers.
 *   - every function returns an int status: 0 ok, <0 error (CES_ERR_*), message via ces_last_error().
 *     CES_ERR_NOT_SPD maps to numpy.linalg.LinAlgError on the Python side.  No C++ exception crosses.
 *   - a handle is not re-entrant; different handles may be used from different threads.  All work of a
 *     handle is issued on the stream given at creation.
 *   - multi-GPU: one handle per process/GPU, the ensemble is sharded by particle columns.  The library
 *     performs no communication itself; the host runs the collectives named below between the phases
 *     (torch.distributed / NCCL in ces_b200/calibrate.py).
 */
#ifndef CES_B200_H
#define CES_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CES_OK 0
#define CES_ERR_INVALID (-1)
#define CES_ERR_STATE (-2)
#define CES_ERR_ALIGN (-3)
#define CES_ERR_NOT_SPD (-4)
#define CES_ERR_CUDA (-5)
#define CES_ERR_NOMEM (-6)

/* update rules (ces/calibrate.py:364-369) */
#define CES_RULE_EKS 0            /* :418-449 semi-implicit, biased covariance                       */
#define CES_RULE_ALDI 1           /* :451-490 default                                                */
#define CES_RULE_ALDI_CONSTANT 2  /* :492-529 h = 0.1 / max|drift|                                   */
#define CES_RULE_EKI 3            /* U - h (U - ubar) D, the part shared by all three (SURVEY F3)    */

/* step-size rules (ces/calibrate.py:247-260) */
#define CES_TS_FROBENIUS 0        /* h = 1 / (||D||_F + 1e-8), :248                                  */
#define CES_TS_FIXED 1            /* h given by the caller ('constant', and 'mix' after spin-up)     */
#define CES_TS_KEEP 2             /* phase 4 keeps the h fixed earlier by ces_peek_step_size          */

/* formulation of the interaction term */
#define CES_FORM_INTERACTION 0    /* D = (1/J) E^T W formed in panels, V = U~ D (the reference's formulation) */
#define CES_FORM_FACTORED 1       /* V = (1/J)(U~ E^T) W, ||D||_F from Gram matrices; same update to rounding */

/* noise term of the noisy rules eks, aldi, aldi_constant (ces_set_noise); n_C = J for eks, J - 1 for aldi / aldi_constant */
#define CES_NOISE_CHOLESKY 0      /* sqrt(2h) chol(C^uu) xi, xi p x J: the reference's (default)     */
#define CES_NOISE_ENSEMBLE 1      /* sqrt(2h / n_C) (U - ubar) xi, xi J x J                           */

/* forward maps (ces/utils.py) */
#define CES_MAP_LINEAL 0          /* A theta + b           :25-31  */
#define CES_MAP_LINEAL_LOG 1      /* A exp(phi) + b        :39-42  */
#define CES_MAP_ELLIPTIC 2        /* :72-89  (p = 2, k = 2; params = {x1, x2})                       */
#define CES_MAP_BANANA 3          /* :116-122 (p = 2, k = 2; params = {a, b})                        */

/* covariance families of the GP emulator (ces_gp_set_kernel; GPflow's class names) */
#define CES_GP_SE 0               /* SquaredExponential (the default)                                 */
#define CES_GP_MATERN12 1         /* Matern12 = sklearn's Matern(nu=0.5)                              */
#define CES_GP_MATERN32 2         /* Matern32 = sklearn's Matern(nu=1.5)                              */
#define CES_GP_MATERN52 3         /* Matern52 = sklearn's Matern(nu=2.5)                              */

typedef struct ces_handle_s* ces_handle_t;

/* Library / build identification ("ces_b200 <version> sm_100a"). */
const char* ces_version(void);
/* Message of the last failing call on this thread. */
const char* ces_last_error(void);

/* Create the per-GPU state of one sampler: p parameters, k observations (enka.__init__,
 * ces/calibrate.py:14-22), J_local particle columns on this rank out of J_global, rank/nranks of the
 * column sharding (1 GPU: J_local = J_global, rank 0 of 1).  With nranks > 1 every rank must use the
 * same J_local (pad the last shard with zero columns and pass its true width to the phases through
 * `cols_local`).  `stream` is a cudaStream_t (NULL = legacy default stream).  `d_panel_bytes` bounds the
 * workspace of the J x J interaction matrix, which is formed in column panels (0 = 8 GiB default; < 0 = a
 * light handle for ces_forward_map only, without any update workspace). */
int ces_create(int64_t p, int64_t k, int64_t J_local, int64_t J_global, int rank, int nranks, int64_t cols_local,
               void* stream, int64_t d_panel_bytes, ces_handle_t* out);
int ces_destroy(ces_handle_t h);

/* Problem data, HOST pointers, copied and factorised once (the reference re-solves with Gamma three
 * times per step, ces/calibrate.py:429,434,435): y (k), Gamma (k x k, SPD, ld = k), Sigma0 = sampler.sigma
 * (p x p, SPD, ld = p), mu (p), ustar (p).  Diagonal Gamma / Sigma0 are detected and take the scaling
 * path.  Returns CES_ERR_NOT_SPD when a factorisation fails. */
int ces_set_problem(ces_handle_t h, const double* y_host, const double* Gamma_host, const double* Sigma0_host,
                    const double* mu_host, const double* ustar_host);

/* ---- the update, in phases (single GPU: call them back to back, or use ces_step) ------------------
 * phase 1  local row sums of G and U over the local particles -> sums_dev (k + p doubles)
 *          [host: all-reduce(sum) of ces_buffer("sums")]
 * phase 2  centring E, R, W = Gamma^-1 R, U~, Z = Sigma0^-1 (U - mu); local partial sums of the four
 *          diagnostics; local partial covariance U~ U~^T
 *          [host: all-reduce(sum) of "cuu"; all-gather of "e_all" and "ut_all" (rank-major blocks)]
 * phase 3  chol(C^uu) (Cholesky noise only); D = (1/J) E^T W by source block and column panel with sum of squares; V = U~ D
 *          [host: all-reduce(sum) of the first 5 doubles of "scalars"]
 * phase 4a (aldi_constant only) drift and its local max-abs  [host: all-reduce(max) of scalars[5]]
 * phase 4  step size, prior term, noise term (ces_set_noise), assembly of U_{n+1}; returns hk and the four diagnostics
 *          (self-bias, bias, self-bias-data, bias-data: ces/calibrate.py:432-435) on the host.
 * U, G, xi, U_out are device pointers to this rank's columns with leading dimensions ld*.  */
int ces_phase1_sums(ces_handle_t h, const double* U_dev, int64_t ldu, const double* G_dev, int64_t ldg);
int ces_phase2_centre(ces_handle_t h, int rule, const double* U_dev, int64_t ldu, const double* G_dev, int64_t ldg);
int ces_phase3_interact(ces_handle_t h, int rule, int skip_interaction);
/* Phase 3 in pieces, for overlapping the all-gather with compute: source blocks (rows of D) are processed in rotated
 * order (rank + i) % nranks, i in [first, first + count).  Block i = 0 is this rank's own E / U~ (already in place
 * after phase 2), so the host starts the all-gathers asynchronously, calls ces_phase3_blocks(h, rule, 0, 1), waits for
 * the collectives and calls ces_phase3_blocks(h, rule, 1, nranks - 1).  (first = 0 also starts chol(C^uu).) */
int ces_phase3_blocks(ces_handle_t h, int rule, int first, int count);
/* Non-default time_step modes ('constant', 'mix'; ces/calibrate.py:439-441, 470-473): after phase 3 (and its
 * all-reduce) ces_peek_step_size fixes and returns the step size hk this step uses; ces_phase3b_cpp forms the local
 * part of C^pp = cov(G, bias=True) = E E^T / J  [host: all-reduce(sum) of ces_buffer("cpp")]; ces_phase3c_resolve
 * recomputes D = (1/J) E^T (hk C^pp + Gamma)^-1 R and V = U~ D.  Phase 4 is then called with CES_TS_KEEP.  With a
 * caller-given hk ('constant') phase 3 may skip forming the Gamma-only D (skip_interaction = 1). */
int ces_peek_step_size(ces_handle_t h, int ts_kind, double fixed_h, double* hk_host);
int ces_phase3b_cpp(ces_handle_t h);
int ces_phase3c_resolve(ces_handle_t h, int rule);
/* time_step = 'spectral' (ces/calibrate.py:249-251: radspec = eigvals(D).real.max(), hk = 1 / radspec): after phase 3,
 * ces_phase3b_cpp and the all-reduce of "cpp", ces_phase3d_spectral returns lambda_max(Gamma^-1 C^pp), which equals the
 * largest eigenvalue of D (the non-zero spectrum of D = E^T (Gamma^-1 R / J) is that of Gamma^-1 R E^T / J = Gamma^-1 C^pp,
 * real and non-negative), by Lanczos in the Gamma^-1 inner product with full re-orthogonalisation; *lanczos_steps
 * receives the number of steps taken -- NEGATED when the iteration reached its cap (min(k, 768) steps) without two
 * agreeing estimates: the value is then only a lower bound of lambda_max.  Phase 4 is then called with CES_TS_FIXED
 * and 1 / radspec. */
int ces_phase3d_spectral(ces_handle_t h, double* radspec_host, int* lanczos_steps_host);
/* Factored formulation (opt-in; the same update to rounding without forming the J x J matrix):
 *   V = (1/J) (U~ E^T) W   and   ||D||_F^2 = sum((E E^T) o (W W^T)) / J^2.
 * ces_phase3f_products replaces phase 3: local parts of P1 = U~ E^T (d x k), GE = E E^T, GW = W W^T (k x k)
 * [host: all-reduce(sum) of ces_buffer "p1", "gram_e", "gram_w"]; ces_phase3f_finish forms V and the sum of squares
 * [host: all-reduce(sum) of scalars[0:5] as after phase 3].  No all-gather of E / U~ is needed in this form. */
int ces_phase3f_products(ces_handle_t h, int rule);
int ces_phase3f_finish(ces_handle_t h, int rule);
int ces_phase4a_drift(ces_handle_t h, double switch_);
int ces_phase4_update(ces_handle_t h, int rule, int ts_kind, double fixed_h, const double* U_dev, int64_t ldu,
                      const double* xi_dev, int64_t ldxi, double* Uout_dev, int64_t ldo, double* hk_host,
                      double* metrics_host /* [4] */);

/* Noise term of the noisy rules for the following steps (the setting stays on the handle until the next call; set
 * (seed, step) before each step).  CES_NOISE_CHOLESKY: the reference's sqrt(2h) chol(C^uu + 1e-8 I) xi with the p x J
 * xi passed to phase 4 / ces_step / ces_step_host.  CES_NOISE_ENSEMBLE:
 *     sqrt(2h / n_C) (U - ubar) xi,   xi in R^{J x J} i.i.d. N(0, 1),  xi[s, j]: source particle s, target particle j,
 * with n_C the normalisation of the rule's own C^uu (J for eks, J - 1 for aldi and aldi_constant).  Given U every column
 * is N(0, 2h (C^uu - 1e-8 I)) and lies in span(U - ubar); it costs 2 p J^2 flop and no factorisation (chol(C^uu) is not
 * computed in this mode).  The rest of the step is unchanged; eki has no noise term.  xi_dev == NULL: xi from Philox at
 * (seed, step), exactly as ces_fill_ensemble_noise draws it; otherwise a J_global x cols_local device matrix of this
 * rank's columns (row s = global particle s) with a 16-byte aligned base and an even ldxi >= cols_local (else
 * CES_ERR_ALIGN), which must stay valid until the step's phase 4 has run.  In ensemble mode the xi argument of phase 4,
 * ces_step and ces_step_host is ignored and may be NULL, and the single-kernel path of small problems is not taken.
 * CES_ERR_INVALID for an unknown kind or a NULL handle; ensemble mode with CES_FORM_FACTORED (which never gathers
 * U - ubar) is refused by ces_step, ces_host_begin and ces_phase3f_products.  No device work. */
int ces_set_noise(ces_handle_t h, int kind, uint64_t seed, uint64_t step, const double* xi_dev, int64_t ldxi);

/* One whole single-GPU step on device buffers (nranks must be 1). */
int ces_step(ces_handle_t h, int rule, int ts_kind, double fixed_h, double switch_, int formulation,
             const double* U_dev, int64_t ldu, const double* G_dev, int64_t ldg, const double* xi_dev, int64_t ldxi,
             double* Uout_dev, int64_t ldo, double* hk_host, double* metrics_host);

/* The same step on HOST buffers (dense, ld = J): host->device copies of U, G, xi and the device->host
 * copy of U_out happen inside the call.  This is the call behind sampling.eks_update*(numpy arrays)
 * (ces/calibrate.py:418, 451, 492).  The copies are pipelined against the arithmetic: G is uploaded in row chunks on a
 * copy stream, each chunk is summed and centred as it lands and the first column panel of D = (1/J) E^T W accumulates
 * over the rows received so far, U and xi follow behind; U_next is downloaded in column chunks while the next chunk is
 * still being assembled.  (Page-locked host buffers make the copies asynchronous; pageable ones still work.) */
int ces_step_host(ces_handle_t h, int rule, int ts_kind, double fixed_h, double switch_, int formulation,
                  const double* U_host, const double* G_host, const double* xi_host, double* Uout_host,
                  double* hk_host, double* metrics_host);
/* Gathers of the other ranks' E / U~ blocks over peer memory instead of an NCCL all-gather (one process per GPU on one
 * NVSwitch domain): ces_ipc_export writes the 64-byte CUDA IPC handles of this rank's "e_all" / "ut_all" buffers, the
 * host exchanges them once and calls ces_ipc_import for every peer.  Per step, after the all-reduce of "cuu" has been
 * queued, ces_peer_gather queues one device-to-device copy per peer block on a side stream (copy engines over NVLink:
 * no SM is taken from the own-block GEMMs that run meanwhile), and ces_peer_gather_wait makes the handle's stream wait
 * for them before ces_phase3_blocks(h, rule, 1, nranks - 1).  See csrc/api.cu for why no further handshake is needed. */
int ces_ipc_export(ces_handle_t h, void* e_handle /* 64 bytes */, void* ut_handle /* 64 bytes */);
int ces_ipc_import(ces_handle_t h, int peer_rank, const void* e_handle, const void* ut_handle);
int ces_peer_gather(ces_handle_t h);
int ces_peer_gather_wait(ces_handle_t h);
/* Per-phase timeline (profiles/): while enabled, the phases record named CUDA events on the streams they use
 * (ces_timeline_mark adds one on the handle's main stream, e.g. around a collective the host issues).
 * ces_timeline_read synchronises the device, returns the marks recorded since the last read as '\n'-separated names
 * and their times in ms relative to the first mark (-1: not comparable), and clears them. */
int ces_timeline_enable(ces_handle_t h, int on);
int ces_timeline_mark(ces_handle_t h, const char* name);
int ces_timeline_read(ces_handle_t h, char* names, int64_t names_cap, double* ms, int64_t ms_cap, int64_t* count);
/* The host step in pieces, for column-sharded callers (nranks > 1; ces_step_host is exactly this sequence with no
 * collectives).  Host arrays are this rank's dense shards: U_host, xi_host p x cols_local, G_host k x cols_local.
 *   ces_host_begin         queues every upload on the copy stream (G in *nchunks <= 8 row chunks with bounds[0..nchunks],
 *                          sized from the host->device rate measured on the previous call; then U, then xi) and returns
 *   for c in chunks:       ces_host_sums_g(c)     row sums of the chunk          [all-reduce "sums"[bounds[c]:bounds[c+1]]]
 *                          ces_host_centre_g(c, interact)   E, W rows; interact != 0: ces_host_interact_chunk(c) at once
 *                          ces_host_interact_chunk(c)       with several chunks: the own block's first D panel contracted
 *                                                 over these rows (accumulating; chunks in order).  A sharded caller defers
 *                                                 the last chunk's until the gathers of E / U~ have been started
 *   ces_host_sums_u        z, data-space diagnostics; row sums of U                   [all-reduce "sums"[k:k+p]]
 *   ces_host_centre_u      U~, Z, diagnostics, local C^uu                             [all-reduce "cuu"; all-gather "e_all", "ut_all"]
 *   ces_host_interact_own  starts chol(C^uu); the rest of the own block (runs while the gathers are in flight)
 *   [ces_phase3_blocks(h, rule, 1, nranks - 1)]                                       [all-reduce "scalars"[0:5]]
 *   [ces_phase4a_drift for aldi_constant                                              all-reduce(max) "scalars"[5:6]]
 *   ces_host_update        waits for xi, assembles U_next and downloads this rank's p x cols_local block into
 *                          Uout_host in overlapped column chunks; returns hk and the diagnostics like ces_phase4_update */
/* The row chunks ces_host_begin will use (bounds[0..n], returns n <= 8): a pure function, identical on every rank (no
 * handle, no device).  h2d_gbs <= 0: the nominal host->device rate for `nranks` processes. */
int ces_host_chunk_schedule(int64_t k, int64_t J_local, int64_t panel, int nranks, double h2d_gbs, int64_t* bounds /* [9] */);
int ces_host_begin(ces_handle_t h, int rule, int formulation, const double* U_host, const double* G_host,
                   const double* xi_host, int* nchunks_out, int64_t* bounds_out /* [9] */);
int ces_host_sums_g(ces_handle_t h, int chunk);
int ces_host_centre_g(ces_handle_t h, int chunk, int interact);
int ces_host_interact_chunk(ces_handle_t h, int chunk);
int ces_host_sums_u(ces_handle_t h);
int ces_host_centre_u(ces_handle_t h);
int ces_host_interact_own(ces_handle_t h);
int ces_host_update(ces_handle_t h, int ts_kind, double fixed_h, double* Uout_host, double* hk_host, double* metrics_host);
/* Device-pointer phases with a host destination: the next ces_phase4_update also copies this rank's p x cols_local
 * block of U_next to host_out (dense, ld = cols_local; column chunks overlapped with the assembly).  One-shot; NULL cancels. */
int ces_set_pending_output(ces_handle_t h, double* host_out);

/* The whole loop of sampling.run (ces/calibrate.py:341-398) for a SMALL single-GPU problem (p <= 8, k <= 16, J <= 512,
 * e.g. BASELINE config 1: d = 2, k = 10, J = 100, 1000 iterations) with one of the ces.utils maps as forward model, in ONE
 * kernel launch: per iteration the forward map, the update, the cumulative pseudo-time and the stopping rule t > t_tol.
 * U0_host: p x J.  xi_host: T x p x J pre-drawn N(0,1) noise (the caller's numpy stream), or NULL: device noise from
 * (seed, step0 + iteration).  t0 / have_t0: time reached by earlier runs of the same sampler (resume).  Outputs (host):
 * Utrace (n + 1) x p x J and Gtrace (n + 1) x k x J -- slot i is the ensemble before update i, slot n the final one --,
 * S_host n x 16 step scalars (layout of ces_buffer "scalars"; the four diagnostics are sums over particles), t_host n
 * cumulative times, *nsteps = n <= T updates performed.  A/b as in ces_forward_map (device), params_host its two scalars. */
int ces_small_run(ces_handle_t h, int rule, int ts_kind, double fixed_h, double switch_, int map_kind, const double* A_dev,
                  int64_t lda, const double* b_dev, const double* params_host, const double* U0_host, const double* xi_host,
                  uint64_t seed, uint64_t step0, int64_t T, double t0, int have_t0, double t_tol, double* Utrace_host,
                  double* Gtrace_host, double* S_host, double* t_host, int64_t* nsteps_host);

/* Batched forward map G[:, j] = model(U[:, j]) for this rank's columns (enka.G_ens, ces/calibrate.py:106-130).
 * CES_MAP_LINEAL / _LOG: A_dev is k x p (ld = lda, even, 16-byte aligned), b_dev is k doubles or NULL.
 * CES_MAP_ELLIPTIC / _BANANA: params_host holds the two scalars named above, A_dev/b_dev are NULL. */
int ces_forward_map(ces_handle_t h, int map_kind, const double* A_dev, int64_t lda, const double* b_dev,
                    const double* params_host, const double* U_dev, int64_t ldu, double* G_dev, int64_t ldg);

/* Named device buffers of the handle, for the host-side collectives and for tests:
 * "sums" (k+p), "cuu" (p x ldp), "e_all" (nranks x k x ldJ), "ut_all" (nranks x p x ldJ), "scalars" (16),
 * "w" (k x ldJ), "v" (p x ldJ), "chol" (p x ldp), "cpp" (k x ldk, after ces_phase3b_cpp), "d_panel".  rows/cols/ld may be NULL. */
int ces_buffer(ces_handle_t h, const char* name, double** ptr_dev, int64_t* rows, int64_t* cols, int64_t* ld);

/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
int64_t ces_launch_count(ces_handle_t h);

/* Optional device-side timing of the dominant kernel, the D = (1/J) E^T W GEMM: when enabled, phase 3
 * brackets every launch of it with CUDA events on the handle's stream.  ces_profile_read synchronises the
 * stream and returns the summed duration (ms), the number of launches and their algorithmic flops
 * (2 * k * rows * cols each) since the previous read. */
int ces_profile_enable(ces_handle_t h, int on);
int ces_profile_read(ces_handle_t h, double* gemm_d_ms, int64_t* launches, double* flops);

/* ---- batched 2-D Darcy forward model (ces/darcy.py:9-138 + utilities/mfiles/gaussrnd_coarse.m, solve_gwf.m) ------
 * ces_darcy_create: N x N mesh (16 <= N <= 128, N % 16 == 0), p active KL modes; HOST operators assembled by the
 * caller (ces_b200/darcy.py): PhiT (p x N^2, scaled 2-D inverse-DCT basis of the active modes), S (N x N, not-a-knot
 * spline cell centres -> nodes), S2 (N x N, nodes -> centres); obs_index (n_obs flat cell indices, row-major) or NULL.
 * ces_darcy_forward: U_dev (p x cols, ld = ldu) -> G_dev (n_obs x cols, or N^2 x cols when full_solution != 0), one
 * thread-block cluster per member running preconditioned CG (Jacobi scaling plus, for Nmesh in {32, 48, 64, 128}, a local
 * 4 x 4-node level and an
 * aggregation coarse level of at most 64 unknowns) to relative residual `tol` in the preconditioner norm (<= 0: 1e-13)
 * with at most max_iter iterations (<= 0: 40 N); *iters_host receives the largest iteration count of the batch.
 * Environment (experiments only): CES_DARCY_COARSE=0 disables the coarse level, CES_DARCY_CLUSTER=2|4|8 asks for a larger
 * cluster than the grid needs. */
int ces_darcy_create(int64_t N, int64_t p, const double* PhiT_host, const double* S_host, const double* S2_host,
                     const int64_t* obs_index_host, int64_t n_obs, void* stream, void** out);
int ces_darcy_destroy(void* model);
int ces_darcy_forward(void* model, const double* U_dev, int64_t ldu, int64_t cols, double* G_dev, int64_t ldg,
                      int full_solution, double tol, int max_iter, int* iters_host);
/* Statistics of the last ces_darcy_forward call (measurement only, bench.py): members solved, CG iterations summed
 * over the members, and the duration of the solver launches by CUDA events on the model's stream.  Synchronises. */
int ces_darcy_last_stats(void* model, int64_t* members, int64_t* total_iterations, double* solver_ms);

/* ---- batched 'pde'-type forward models (enka.G_pde_ens, ces/calibrate.py:132-168; ces/utils.py:124-447) --------------
 * One call integrates every particle from its own initial condition W0[:, j] with the parameters U[:, j] over the
 * uniform output grid t_i = i * dt_out, i < n_out, with `substeps` classical RK4 steps per output interval (the
 * reference uses adaptive scipy integrators, one particle per Python call), accumulates the model's window statistics
 * on the fly and returns them in G (n_obs x cols) and the final states in Wend (n_state x cols, may be NULL); traj
 * (may be NULL) receives the sampled trajectory, sample i of state variable v of particle j at [(i * n_state + v) * ldt + j]
 * (model.solve of a single particle).
 * Lorenz 63 (ces/utils.py:124-229): p <= 2 parameters (r, b) -- or (log r, log b) when log_params != 0 --, sigma = 10;
 *   G = means of (x, y, z, x^2, y^2, z^2, xy, xz, yz) over the last `window` samples of t[1:]  (:181-194).
 * Lorenz 96 (ces/utils.py:231-447): state = n_slow slow then n_slow * n_fast fast variables; U row i sets parameter
 *   param_slots[i] (0 h, 1 F, 2 log c, 3 b; defaults 1, 10, log 10, 10), which covers lorenz96 / Fc / Fb / hFb / hcb;
 *   statistics (:332-342) over the last `window` samples after the first `skip` (= spinup * freq + 1): out_mode 0 ->
 *   5 * n_slow rows; 1 -> their means over k (lorenz96_hom); 2 -> column out_col. */
int ces_lorenz63_forward(void* stream, int log_params, const double* U_dev, int64_t ldu, int64_t p, int64_t cols,
                         const double* W0_dev, int64_t ldw0, int64_t n_out, double dt_out, int substeps, int64_t window,
                         double* G_dev, int64_t ldg, double* Wend_dev, int64_t ldwe, double* traj_dev, int64_t ldt);
int ces_lorenz96_forward(void* stream, const int* param_slots, int n_slow, int n_fast, const double* U_dev, int64_t ldu,
                         int64_t p, int64_t cols, const double* W0_dev, int64_t ldw0, int64_t n_out, double dt_out,
                         int substeps, int64_t skip, int64_t window, int out_mode, int out_col, double* G_dev, int64_t ldg,
                         double* Wend_dev, int64_t ldwe, double* traj_dev, int64_t ldt);

/* Frobenius norm of a device matrix (sampling.timestep_method(D, ...) for callers that own an explicit D). */
int ces_frobenius(void* stream, const double* X_dev, int64_t ld, int64_t rows, int64_t cols, double* out_host);

/* N(0,1) noise on the device (production alternative to the host draw np.random.normal(0,1,[p,J]) of
 * ces/calibrate.py:447,488,527): Philox4x32-10 + Box-Muller.  Element (row, col_offset + col) depends only on
 * (seed, step, row, global column), so a column-sharded ensemble draws exactly what one GPU would (col_offset even). */
int ces_fill_normal(void* stream, uint64_t seed, uint64_t step, double* X_dev, int64_t ld, int64_t rows, int64_t cols,
                    int64_t col_offset);

/* The xi of CES_NOISE_ENSEMBLE on the device: rows [row_offset, row_offset + rows) (source particles) and columns
 * [col_offset, col_offset + cols) (target particles) into X_dev (ld >= cols).  Philox4x32-10 keyed by (seed low, seed high)
 * at the counter (j >> 1, 0x454E, s, step mod 2^32); even j takes the Box-Muller cosine, odd j the sine (the uniforms and
 * Box-Muller of ces_fill_normal).  Element (s, j) depends only on (seed, step, s, j), so any sharding of rows or columns
 * reproduces a single draw; counter word 1 keeps the stream apart from ces_fill_normal's. */
int ces_fill_ensemble_noise(void* stream, uint64_t seed, uint64_t step, double* X_dev, int64_t ld, int64_t rows,
                            int64_t cols, int64_t row_offset, int64_t col_offset);

/* ---- building blocks exported for tests and for callers that own their orchestration ---------------
 * C[M,N] = alpha * op(A) op(B) + beta * C on the FP64 tensor cores.  a_mode: 0 = A is M x K row-major,
 * 1 = A is stored K x M (i.e. A^T given); b_mode: 0 = B is K x N row-major, 1 = B stored N x K.
 * Operands need 16-byte aligned bases and even leading dimensions no smaller than their stored rows (lda >= K or M,
 * ldb >= N or K, ldc >= N; CES_ERR_INVALID otherwise). */
int ces_gemm(void* stream, int a_mode, int b_mode, int64_t M, int64_t N, int64_t K, double alpha, const double* A_dev,
             int64_t lda, const double* B_dev, int64_t ldb, double beta, double* C_dev, int64_t ldc);
/* In-place lower Cholesky of an n x n SPD matrix on the device (strict upper triangle zeroed). */
int ces_potrf(void* stream, double* A_dev, int64_t ld, int64_t n);
/* X = A^-1 B for SPD A (n x n) and B (n x nrhs), both on the device; A is overwritten by its factor. */
int ces_posv(void* stream, double* A_dev, int64_t lda, int64_t n, double* B_dev, int64_t ldb, int64_t nrhs);
/* Ainv = A^-1 (n x n, ld ldo) for SPD A on the device, through the blocked Cholesky and two triangular solves of the
 * identity (the inverse the GP gradient uses); A is overwritten by its factor.  CES_ERR_NOT_SPD names the failing pivot. */
int ces_potri(void* stream, double* A_dev, int64_t ld, int64_t n, double* Ainv_dev, int64_t ldo);

/* ---- test support: not part of the stable interface --------------------------------------------------------------
 * The whole DMMA GEMM family behind ces_gemm, for tests that pin each of its features:
 *   C[M,N] = alpha (* *alpha_dev) * sum_kk op(A)(m,kk) op(B)(kk,n) + beta * C  (+ diag_add on the diagonal)
 * flags: 1 = op(A) lower triangular (row tile tm reads kk < 128 (tm + 1) only, entries above the diagonal inside that
 * range must be zero), 2 = only tiles on or below the diagonal (square C; mirrored when a workspace is given),
 * 4 = op(B) upper triangular (column tile tn reads kk < 128 (tn + 1) only).  splits > 1 splits the contraction into
 * planes of splitk_ws (splits*M*N doubles) that a reduce kernel sums; with a workspace alpha / beta / diag_add are
 * applied there.  ssq_partials (no workspace, flag 2 excluded) receives one sum of squares of the stored values per
 * 128 x 128 tile and problem.  batch > 1: problem z shifts A's and B's stored rows by z*a_batch_rows / z*b_batch_rows
 * (0 = shared) and writes C + z*c_batch_elems, or, with a workspace, all problems are summed into C.  group_m (0 = 16):
 * row tiles per rasterisation group.  wave_ctas (0 = SM count) and serpentine (-1 = environment default, 0 = off,
 * 1 = on): odd waves of wave_ctas CTAs walk the contraction backwards.  struct_size must be sizeof(ces_gemm_desc), the
 * capacities (in doubles) must cover what the call writes; otherwise CES_ERR_INVALID before any device work. */
typedef struct ces_gemm_desc {
    int64_t struct_size;
    int32_t a_mode, b_mode;
    int64_t M, N, K;
    const double* A;
    int64_t lda;
    const double* B;
    int64_t ldb;
    double* C;
    int64_t ldc;
    double alpha, beta;
    const double* alpha_dev;
    int32_t flags, group_m, splits, wave_ctas, serpentine, reserved;
    double* splitk_ws;
    int64_t splitk_ws_elems;
    double diag_add;
    double* ssq_partials;
    int64_t ssq_partials_elems;
    int64_t batch, a_batch_rows, b_batch_rows, c_batch_elems;
} ces_gemm_desc;
int ces_gemm_ex(void* stream, const ces_gemm_desc* desc);

/* ---- Metropolis-Hastings on the true forward model: MCMC.model_mh (ces/sample.py:121-196) ---------------------------
 * n_chains independent chains of n_mcmc proposals, one warp per chain, the loop entirely on the device (csrc/mcmc.cu).
 * Forward model: one of the ces.utils maps (A_dev / b_dev / params_host as in ces_forward_map).  Host inputs:
 * y (k), Ginv2 = (2 Gamma)^-1 (k x k, dense), prior mean mu (p) and precision Pinv (p x p) -- unused with pcn != 0 --,
 * scales (p x p: delta * chol(cov(Ustar)), or chol(prior.cov) for pCN), beta (pCN), start (n_chains x p: first state of
 * every chain) and phi_point (n_chains x p: where the initial Phi_current is evaluated; the reference uses the ensemble
 * mean even when it resumes from its last sample).  Random numbers: with mt_state_host != NULL chain 0 consumes numpy's
 * global MT19937 stream exactly as np.random.normal(0, 1, p) followed by np.random.uniform() would -- mt_state_host =
 * 624 key words, position, has_gauss flag (626 uint32), *mt_gauss_host = the cached Gaussian; both are updated to the
 * state after the run --; every other chain (all of them with NULL) draws from Philox keyed by (seed, chain, iteration).
 * Outputs: samples (n_chains x (n_mcmc + 1) x p, state 0 = start) and the number of accepted proposals per chain.
 * Limits shared by every sampler (ces_darcy_mh, ces_gp_mh too): 1 <= n_mcmc < 2^31 - 1, 1 <= n_chains <= 2^24, mt_gauss_host
 * non-NULL whenever mt_state_host is, mu_host / Pinv_host non-NULL unless pcn; otherwise CES_ERR_INVALID before any
 * device work.  A samples buffer beyond 4e18 bytes returns CES_ERR_NOMEM.  Synchronises. */
int ces_mcmc_model_mh(void* stream, int map_kind, int64_t p, int64_t k, const double* A_dev, int64_t lda,
                      const double* b_dev, const double* params_host, const double* y_host, const double* Ginv2_host,
                      const double* mu_host, const double* Pinv_host, const double* scales_host, int pcn, double beta,
                      int64_t n_mcmc, int64_t n_chains, const double* start_host, const double* phi_point_host,
                      uint32_t* mt_state_host, double* mt_gauss_host, uint64_t seed, double* samples_host,
                      int32_t* accepted_host);

/* MCMC.model_mh on the Darcy models (csrc/darcy_mh.cu): n_chains chains of n_mcmc proposals stepped in lockstep on a
 * Darcy model created with an obs_index (ces_darcy_create), on that model's stream, with no host synchronisation inside
 * the step loop.  One step draws every chain's noise (random numbers exactly as ces_mcmc_model_mh: chain 0 from numpy's
 * stream when mt_state_host != NULL, the others from Philox keyed by (seed, step, chain)), forms the proposals
 * b cur + a scales z as one DMMA GEMM (random walk a = b = 1; pCN a = sqrt(beta), b = sqrt(1 - beta^2)), evaluates them in
 * one batched ces_darcy_forward pipeline (CG to `tol`, at most max_iter iterations; <= 0: the defaults of
 * ces_darcy_forward), and accepts with Phi = (G - y)^T Ginv2 (G - y) (+ 1/2 (u - mu)^T Pinv (u - mu) unless pCN) as
 * GEMMs, so p and n_obs are limited only by the model.  Arguments from y_host onwards as ces_mcmc_model_mh (p and
 * k = n_obs are the model's).  If any solve -- the initial one at phi_point or a proposal's -- reaches max_iter, returns
 * CES_ERR_STATE naming the first such step and leaves samples, acceptances and the generator state untouched.
 * The limits of ces_mcmc_model_mh apply (checked before the model); a model without obs_index also returns
 * CES_ERR_INVALID before any device work.  Synchronises. */
int ces_darcy_mh(void* model, double tol, int max_iter, const double* y_host, const double* Ginv2_host,
                 const double* mu_host, const double* Pinv_host, const double* scales_host, int pcn, double beta,
                 int64_t n_mcmc, int64_t n_chains, const double* start_host, const double* phi_point_host,
                 uint32_t* mt_state_host, double* mt_gauss_host, uint64_t seed, double* samples_host,
                 int32_t* accepted_host);

/* ---- Emulate: exact GP emulators of the whitened forward map and MH chains through them (csrc/emulate.cu) ----------
 * One GP per whitened output i < k on the training inputs X (p x n, row-major, one point per column) and outputs
 * Y = T G - ybar (k x n; T = diag(lam^-1/2) Q^T from Gamma = Q diag(lam) Q^T, ybar the row means), all fixed by the caller.
 * theta_i = [log sf2, log l_1..l_p, log sn2];  r^2 = sum_d (x_d - z_d)^2 / l_d^2;  k(x, z) by the model's family:
 *   CES_GP_SE sf2 exp(-r^2/2) (the default),  CES_GP_MATERN12 sf2 exp(-r),  CES_GP_MATERN32 sf2 (1 + sqrt3 r) exp(-sqrt3 r),
 *   CES_GP_MATERN52 sf2 (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r);
 * K = k(X, X) + (sn2 + jitter) I;  L = chol(K);  alpha = K^-1 y_i.  Limits: 1 <= p <= 32, 1 <= k <= 64, n >= 2 (n is
 * otherwise bounded by device memory: CES_ERR_NOMEM).  A K that is not positive definite returns CES_ERR_NOT_SPD.
 * ces_gp_create copies X, Y, ybar to the device on `stream`; every later call runs on that stream. */
int ces_gp_create(void* stream, int64_t p, int64_t k, int64_t n, const double* X_host, const double* Y_host,
                  const double* ybar_host, void** out);
int ces_gp_destroy(void* model);
/* Selects the covariance family (CES_GP_*) of every output.  Clears the conditioned state: ces_gp_predict and ces_gp_mh
 * return CES_ERR_STATE until ces_gp_condition runs again.  A NULL model or an unknown kind returns CES_ERR_INVALID.
 * No device work. */
int ces_gp_set_kernel(void* model, int kind);
/* LML_i = -1/2 y_i^T alpha - sum_j log L_jj - n/2 log 2 pi for outputs i0 <= i < i1 (theta_host: (i1 - i0) x (p + 2)) and,
 * with grad_host != NULL, dLML_i/dtheta_i = 1/2 sum_ab (alpha alpha^T - K^-1)_ab dK_ab/dtheta ((i1 - i0) x (p + 2)).
 * Fixed-order reductions: repeated calls return bit-identical results.  Synchronises. */
int ces_gp_lml(void* model, int64_t i0, int64_t i1, const double* theta_host, double jitter, double* lml_host,
               double* grad_host);
/* Conditions every output on theta_host (k x (p + 2)): keeps L_i^-1 and alpha_i for ces_gp_predict / ces_gp_mh. */
int ces_gp_condition(void* model, const double* theta_host, double jitter);
/* Latent-f prediction at the m points U (p x m on the device, ld ldu):  mean_i(u) = ybar_i + k_i(u)^T alpha_i,
 * var_i(u) = max(sf2_i - ||L_i^-1 k_i(u)||^2, 0), into mean / var (k x m on the device).  Asynchronous on the stream. */
int ces_gp_predict(void* model, const double* U_dev, int64_t ldu, int64_t m, double* mean_dev, int64_t ldm,
                   double* var_dev, int64_t ldv);
/* MCMC.emulator_mh: ces_mcmc_model_mh's chains (proposal, prior term, accept test, random numbers, outputs; arguments from
 * mu_host onwards as there) with the forward misfit replaced by the emulated one at the whitened data ytil_host (k):
 *   Phi(u) = 1/2 sum_i (ytil_i - mean_i(u))^2 / (1 + var_i(u)) + 1/2 sum_i log(1 + var_i(u))   (use_variance != 0)
 *   Phi(u) = 1/2 sum_i (ytil_i - mean_i(u))^2                                                  (use_variance == 0)
 * The limits of ces_mcmc_model_mh apply (checked before the model).  Needs ces_gp_condition.  Synchronises. */
int ces_gp_mh(void* model, const double* ytil_host, int use_variance, const double* mu_host, const double* Pinv_host,
              const double* scales_host, int pcn, double beta, int64_t n_mcmc, int64_t n_chains, const double* start_host,
              const double* phi_point_host, uint32_t* mt_state_host, double* mt_gauss_host, uint64_t seed,
              double* samples_host, int32_t* accepted_host);

#ifdef __cplusplus
}
#endif
#endif /* CES_B200_H */
