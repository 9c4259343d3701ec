// C ABI of libces_b200.so (include/ces_b200.h): handle, problem set-up, the phases of one update.
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <optional>
#include <string>
#include <vector>
#include "../../include/ces_b200.h"
#include "kernels.h"

using namespace ces;

struct ces_handle_s {
    int64_t p = 0, k = 0, Jl = 0, Jg = 0, cols = 0;
    int rank = 0, nranks = 1;
    int64_t ldJ = 0, ldp = 0, ldk = 0, ldD = 0, panel = 0;
    cudaStream_t st = nullptr;
    bool have_problem = false, gamma_diag = true, sigma_diag = true;
    bool forward_only = false;          // created for ces_forward_map only: no update workspace
    bool use_small = true;              // single-kernel path for small problems (CES_NO_SMALL_PATH=1 disables it)
    int last_rule = -1;
    // noise term of the noisy rules (ces_set_noise): the reference's sqrt(2h) chol(C^uu) xi, or sqrt(2h / n_C) (U - ubar) xi
    // with xi (J x J) from the Philox stream at (noise_seed, noise_step) or the caller's device matrix noise_xi
    int noise_kind = CES_NOISE_CHOLESKY;
    uint64_t noise_seed = 0, noise_step = 0;
    const double* noise_xi = nullptr;
    int64_t noise_ldxi = 0;
    // problem data (device)
    double *y = nullptr, *ginv_diag = nullptr, *Ginv = nullptr, *mu = nullptr, *ustar = nullptr;
    double *sinv_diag = nullptr, *sig_diag = nullptr, *Sinv = nullptr, *Sigma0 = nullptr, *bprior = nullptr;
    // per-step workspace (device)
    double *sums = nullptr, *cvec = nullptr, *zvec = nullptr, *S = nullptr, *qpart = nullptr, *rowscratch = nullptr, *formpart = nullptr;
    double *E_all = nullptr, *W = nullptr, *R = nullptr, *Ut_all = nullptr, *Z = nullptr, *Y = nullptr, *V = nullptr, *T = nullptr;
    double *xi_pad = nullptr, *expU = nullptr;
    double *Cuu = nullptr, *L = nullptr, *Linv = nullptr, *M = nullptr, *Minv = nullptr, *cb = nullptr;
    double *D = nullptr, *ssq_partials = nullptr, *splitk_ws = nullptr, *v_ws = nullptr;
    double *dvec = nullptr, *uc = nullptr;   // single GPU: c = E^T w0 (J) and U~ c / J (p), the rank-one part of D and V
    int64_t ssq_cap = 0, splitk_cap = 0, ssq_used = 0, v_ws_planes = 4;
    int syrk_splits = 1;
    int* info = nullptr;
    // factored formulation (D never formed): P1 = U~ E^T, Gram matrices of E and W
    double *P1 = nullptr, *GE = nullptr, *GW = nullptr, *gram_ws = nullptr, *gram_part = nullptr;
    int gram_splits = 1, p1_splits = 1;
    // K11 (time_step 'constant' / 'mix'): D re-solved with Gamma -> h*C^pp + Gamma
    std::vector<double> gamma_host;
    double *GammaD = nullptr, *Cpp = nullptr, *Mk = nullptr, *MkLinv = nullptr, *MkInv = nullptr, *Wr = nullptr, *cpp_ws = nullptr, *eig_ws = nullptr;
    double* zr = nullptr;               // M^-1 c: the w0 of the re-solve
    int cpp_splits = 1;
    // host staging
    double* hS = nullptr;   // pinned, S_COUNT doubles + 1 int
    int* hinfo = nullptr;
    double *stage_U = nullptr, *stage_G = nullptr, *stage_xi = nullptr, *stage_out = nullptr;
    double* pending_out = nullptr;      // host destination of stage_out, copied inside phase 4 before its final sync
    int64_t pending_rows = 0;
    // gathers of the other ranks' E / U~ blocks by copy engines over NVLink (ces_ipc_*, ces_peer_gather): IPC-mapped bases
    // of every peer's E_all / Ut_all, a stream for the pulls, an event each way
    std::vector<double*> peer_E, peer_Ut;
    cudaStream_t gather_st = nullptr;
    cudaEvent_t gather_go = nullptr, gather_done = nullptr;
    double* run_ws = nullptr;           // ces_small_run: trace / noise / scalars of a whole run
    int64_t run_ws_len = 0;
    int hb_nchunk = 1, hb_formulation = 0;   // state of a host step in progress (ces_host_begin ... ces_host_update)
    bool hb_have_xi = false;
    int64_t hb_bound[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    bool hb_timed = false;
    int hb_nchunk_prev = 1;
    cudaStream_t aux_st = nullptr;      // chol(C^uu) runs here, hidden behind the D / V GEMMs of the main stream
    cudaEvent_t cuu_ready = nullptr, chol_done = nullptr;
    bool chol_pending = false;
    cudaStream_t copy_st = nullptr;     // ces_step_host: uploads G (row chunks), U and xi while the main stream computes
    cudaEvent_t copy_ev = nullptr, start_ev = nullptr, u_ev = nullptr;
    cudaEvent_t g_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t up_begin = nullptr;     // timing pair around the upload of G: the measured host->device rate sizes the next call's chunks
    double h2d_gbs = 0.0;               // 0: not measured yet
    cudaStream_t out_st = nullptr;      // phase 4: downloads finished column chunks of U_next while the next chunk computes
    cudaEvent_t out_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    std::vector<void*> allocs;
    // optional per-phase timeline (ces_timeline_*): named CUDA events recorded on the stream a phase runs on
    bool timeline = false;
    std::vector<std::pair<std::string, cudaEvent_t>> marks;
    std::vector<cudaEvent_t> mark_pool;
    // optional event timing of the D = E^T W launches
    bool profile = false;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    double prof_flops = 0.0;
};

namespace {

const int64_t kLinvLd = CHOL_NB;

int dalloc(ces_handle_t h, double** out, int64_t n) {
    void* ptr = nullptr;
    const size_t bytes = (size_t)(n < 1 ? 1 : n) * sizeof(double);
    cudaError_t e = cudaMalloc(&ptr, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(CES_ERR_NOMEM, "cudaMalloc of %s%lld bytes failed", "", (long long)bytes);
    }
    e = cudaMemsetAsync(ptr, 0, bytes, h->st);
    if (e != cudaSuccess) return fail(CES_ERR_CUDA, "cudaMemset failed%s", "");
    h->allocs.push_back(ptr);
    *out = static_cast<double*>(ptr);
    return CES_OK;
}

// Timeline mark: a timing event on `s` (default: the main stream) when the timeline is enabled; free otherwise.
void mark(ces_handle_t h, const char* name, cudaStream_t s = nullptr) {
    if (!h->timeline) return;
    cudaEvent_t e;
    if (!h->mark_pool.empty()) { e = h->mark_pool.back(); h->mark_pool.pop_back(); }
    else if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, s ? s : h->st);
    h->marks.emplace_back(name, e);
}

double* e_block(ces_handle_t h, int r) { return h->E_all + (size_t)r * h->k * h->ldJ; }
double* ut_block(ces_handle_t h, int r) { return h->Ut_all + (size_t)r * h->p * h->ldJ; }

int check_info(ces_handle_t h, const char* what) {
    CES_CUDA(cudaMemcpyAsync(h->hinfo, h->info, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CES_CUDA(cudaStreamSynchronize(h->st));
    if (*h->hinfo != 0) {
        const int piv = *h->hinfo;
        CES_CUDA(cudaMemsetAsync(h->info, 0, sizeof(int), h->st));
        return fail(CES_ERR_NOT_SPD, "%s: matrix is not positive definite (pivot %lld)", what, (long long)piv);
    }
    return CES_OK;
}

bool is_diagonal(const double* A, int64_t n) {
    for (int64_t i = 0; i < n; ++i)
        for (int64_t j = 0; j < n; ++j)
            if (i != j && A[i * n + j] != 0.0) return false;
    return true;
}

// Upload a dense n x n host matrix into a padded device buffer (ld = padded_ld(n)).
int upload_square(ces_handle_t h, const double* host, int64_t n, double* dev, int64_t ld) {
    CES_CUDA(cudaMemcpy2DAsync(dev, ld * sizeof(double), host, n * sizeof(double), n * sizeof(double), n,
                               cudaMemcpyHostToDevice, h->st));
    return CES_OK;
}

// dst (n x n, ld) <- inverse of the SPD matrix src (n x n host), via device Cholesky.
int device_spd_inverse(ces_handle_t h, const double* host, int64_t n, double* dst, int64_t ld, const char* what) {
    double *F = nullptr, *Fi = nullptr;
    CES_CUDA(cudaMalloc(&F, (size_t)n * ld * sizeof(double)));
    cudaError_t e = cudaMalloc(&Fi, (size_t)round_up(n, CHOL_NB) * kLinvLd * sizeof(double));
    if (e != cudaSuccess) { cudaFree(F); cudaGetLastError(); return fail(CES_ERR_NOMEM, "cudaMalloc failed%s", ""); }
    int s = CES_OK;
    do {
        if (cudaMemsetAsync(F, 0, (size_t)n * ld * sizeof(double), h->st) != cudaSuccess) { s = CES_ERR_CUDA; break; }
        if ((s = upload_square(h, host, n, F, ld)) != CES_OK) break;
        if ((s = potrf_lower(h->st, F, ld, n, Fi, kLinvLd, h->info)) != CES_OK) break;
        if ((s = check_info(h, what)) != CES_OK) break;
        if ((s = spd_inverse_from_factor(h->st, F, ld, n, Fi, kLinvLd, dst, ld)) != CES_OK) break;
        if (cudaStreamSynchronize(h->st) != cudaSuccess) { s = fail(CES_ERR_CUDA, "device inverse failed%s", ""); break; }
    } while (0);
    cudaFree(F);
    cudaFree(Fi);
    return s;
}

bool ensemble_noise(ces_handle_t h) { return h->noise_kind == CES_NOISE_ENSEMBLE; }

// 1 / n_C of the rule's own C^uu (api.cu centre_u_all: J for eks, J - 1 otherwise) in ensemble-noise mode; 0 otherwise
double ens_inv_nc(ces_handle_t h, int rule) {
    if (!ensemble_noise(h) || rule == CES_RULE_EKI) return 0.0;
    return rule == CES_RULE_EKS ? 1.0 / (double)h->Jg : 1.0 / (double)(h->Jg - 1);
}

int valid(ces_handle_t h, bool need_problem) {
    if (!h) return fail(CES_ERR_INVALID, "null handle%s", "");
    if (need_problem && h->forward_only) return fail(CES_ERR_STATE, "this handle was created for forward maps only%s", "");
    if (need_problem && !h->have_problem) return fail(CES_ERR_STATE, "ces_set_problem has not been called%s", "");
    return CES_OK;
}

// The noise operand xi a step needs: the Cholesky noise of the noisy rules (EKI has no noise term, ensemble noise its own).
bool needs_xi(ces_handle_t h, int rule) { return rule != CES_RULE_EKI && !ensemble_noise(h); }

// The arguments of a step, checked by every entry point before any device work.  std::nullopt: the entry point takes no
// such argument (its rule is phase 2's).  CES_TS_KEEP (`keep_ok`) is for phase 4 only: it keeps ces_peek_step_size's h.
int check_step(ces_handle_t h, const char* who, std::optional<int> rule, std::optional<int> ts_kind, bool keep_ok,
               std::optional<int> formulation, bool have_ptrs, bool no_host_xi = true) {
    if (rule && (*rule < CES_RULE_EKS || *rule > CES_RULE_EKI)) return fail(CES_ERR_INVALID, "unknown update rule %s%lld", "", *rule);
    if (ts_kind && *ts_kind != CES_TS_FROBENIUS && *ts_kind != CES_TS_FIXED && !(keep_ok && *ts_kind == CES_TS_KEEP))
        return fail(CES_ERR_INVALID, "unknown step-size rule%s", "");
    if (formulation && *formulation != CES_FORM_INTERACTION && *formulation != CES_FORM_FACTORED)
        return fail(CES_ERR_INVALID, "unknown formulation%s", "");
    if (formulation == CES_FORM_FACTORED && ensemble_noise(h) && rule.value_or(h->last_rule) != CES_RULE_EKI)
        return fail(CES_ERR_INVALID, "ensemble noise needs the interaction formulation (the factored one never gathers U~)%s", "");
    if (!have_ptrs) return fail(CES_ERR_INVALID, "%s: null pointer", who);
    if (!no_host_xi) return fail(CES_ERR_INVALID, "%s: ensemble noise takes its xi from ces_set_noise, not xi_host", who);
    return CES_OK;
}

// Split-K count of a GEMM with `tiles` output tiles contracting over `contraction`: fill two waves of 148 SMs, with at
// most one split per k-block and at most 64.
int splitk_count(int64_t tiles, int64_t contraction) {
    int64_t sp = ceil_div(296, tiles);
    const int64_t kb = ceil_div(contraction, GEMM_BK);
    if (sp > kb) sp = kb;
    if (sp > 64) sp = 64;
    return sp < 1 ? 1 : (int)sp;
}

// Largest J of the single-CTA step with ensemble noise: its J^2 / 2 Box-Muller pairs per step run on one SM, the phases'
// noise pass on all of them.  Measured per iteration of sampling.run (p = 8, k = 16, B200): 0.88x the phases' time at
// J = 128, 1.04x at 192 (DESIGN.md section 4g, profiles/r08_bench_small_ensemble_noise.json).
constexpr int64_t kSmallEnsembleJMax = 128;

// The whole step in one single-CTA kernel (small problems, where launch latency dominates otherwise).
bool small_path(ces_handle_t h, int formulation) {
    return h->use_small && formulation == CES_FORM_INTERACTION && small_step_eligible(h->p, h->k, h->Jl) &&
           (!ensemble_noise(h) || h->Jl <= kSmallEnsembleJMax);
}

// The fields of a single-CTA call that come from the handle and the step's settings; operands are the caller's.
SmallStepCall small_call(ces_handle_t h, int rule, int ts_kind, double fixed_h, double switch_) {
    SmallStepCall c{};
    c.p = h->p; c.k = h->k; c.J = h->Jl; c.rule = rule; c.ts_kind = ts_kind; c.fixed_h = fixed_h; c.switch_ = switch_;
    c.y = h->y; c.mu = h->mu; c.ustar = h->ustar; c.bprior = h->bprior;
    c.ginv_diag = h->gamma_diag ? h->ginv_diag : nullptr; c.Ginv = h->gamma_diag ? nullptr : h->Ginv;
    c.sinv_diag = h->sinv_diag; c.sig_diag = h->sig_diag;
    c.Sinv = h->sigma_diag ? nullptr : h->Sinv; c.Sigma0 = h->sigma_diag ? nullptr : h->Sigma0;
    c.ldk = h->ldk; c.ldp = h->ldp;
    c.ensemble = ensemble_noise(h) && rule != CES_RULE_EKI;      // eki has no noise term: the same kernel either way
    if (c.ensemble) { c.xi = h->noise_xi; c.ldxi = h->noise_ldxi; c.seed = h->noise_seed; c.step = h->noise_step; }
    return c;
}

// The end of a step: download the step scalars and, when a host destination is pending (one-shot), U_next on the same
// synchronisation; refuse a factorisation of C^uu that failed; hand out hk and the metrics (sums over particles / J).
// The pivot is the device int of potrf (`pivot_on_device`) or S[S_INFO] (the single-CTA kernel).
int finish_step(ces_handle_t h, const double* Uout, int64_t ldo, bool pivot_on_device, double* hk_host, double* metrics_host) {
    cudaStream_t st = h->st;
    CES_CUDA(cudaMemcpyAsync(h->hS, h->S, S_COUNT * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (h->pending_out && h->cols > 0) {
        const size_t wbytes = h->cols * sizeof(double);
        if (ldo == h->cols) CES_CUDA(cudaMemcpyAsync(h->pending_out, Uout, (size_t)h->pending_rows * wbytes, cudaMemcpyDeviceToHost, st));
        else CES_CUDA(cudaMemcpy2DAsync(h->pending_out, wbytes, Uout, ldo * sizeof(double), wbytes, h->pending_rows, cudaMemcpyDeviceToHost, st));
    }
    h->pending_out = nullptr;
    if (pivot_on_device) {
        CES_TRY(check_info(h, "cov(U)"));   // synchronises the stream
    } else {
        CES_CUDA(cudaStreamSynchronize(st));
        if (h->hS[S_INFO] != 0.0)
            return fail(CES_ERR_NOT_SPD, "%s: matrix is not positive definite (pivot %lld)", "cov(U)", (long long)h->hS[S_INFO]);
    }
    if (hk_host) *hk_host = h->hS[S_H];
    if (metrics_host) {
        const double J = (double)h->Jg;
        metrics_host[0] = h->hS[S_SELF_BIAS] / J; metrics_host[1] = h->hS[S_BIAS] / J;
        metrics_host[2] = h->hS[S_SELF_DATA] / J; metrics_host[3] = h->hS[S_BIAS_DATA] / J;
    }
    return CES_OK;
}

}  // namespace

extern "C" {

const char* ces_version(void) { return "ces_b200 0.1.0 sm_100a"; }
const char* ces_last_error(void) { return g_last_error; }
int64_t ces_launch_count(ces_handle_t) { return g_launches; }

int ces_create(int64_t p, int64_t k, int64_t J_local, int64_t J_global, int rank, int nranks, int64_t cols_local,
               void* stream, int64_t d_panel_bytes, ces_handle_t* out) {
    if (!out) return fail(CES_ERR_INVALID, "ces_create: null output%s", "");
    *out = nullptr;
    if (p < 1 || k < 1 || J_local < 1 || J_global < 2 || nranks < 1 || rank < 0 || rank >= nranks || cols_local < 0 ||
        cols_local > J_local || J_local * nranks < J_global)
        return fail(CES_ERR_INVALID, "ces_create: inconsistent sizes%s", "");
    if (p > (1 << 20) || k > (1 << 20) || J_global > (1ll << 30))
        return fail(CES_ERR_INVALID, "ces_create: size out of range%s", "");
    ces_handle_t h = new ces_handle_s();
    h->p = p; h->k = k; h->Jl = J_local; h->Jg = J_global; h->cols = cols_local;
    h->rank = rank; h->nranks = nranks;
    h->st = static_cast<cudaStream_t>(stream);
    h->use_small = std::getenv("CES_NO_SMALL_PATH") == nullptr;
    h->ldJ = padded_ld(J_local);
    h->ldp = padded_ld(p);
    h->ldk = padded_ld(k);
    h->forward_only = d_panel_bytes < 0;
    if (d_panel_bytes <= 0) d_panel_bytes = 8ll << 30;
    // multi-rank: the D blocks of the other ranks' particles are formed by ONE batched launch, one slot each
    const int64_t slots = nranks > 1 ? nranks - 1 : 1;
    int64_t panel = d_panel_bytes / (8 * h->ldJ * slots);
    panel = panel / 128 * 128;
    if (panel < 128) panel = 128;
    if (panel > h->ldJ) panel = h->ldJ;
    h->panel = panel;
    h->ldD = panel;
    h->v_ws_planes = slots > 4 ? slots : 4;

    int s = CES_OK;
    const int nyk0 = form_row_blocks(k, h->ldJ), nyp0 = form_row_blocks(p, h->ldJ);
    const int ny = nyk0 > nyp0 ? nyk0 : nyp0;
    const int64_t tiles_per_rank = ceil_div(J_local, GEMM_BM) * ceil_div(J_local, GEMM_BN) + ceil_div(J_local, GEMM_BM) * ceil_div(J_local, panel);
    h->ssq_cap = tiles_per_rank * nranks + 16;
    h->syrk_splits = splitk_count(gemm_trap_tiles((int)p, (int)p), h->ldJ);   // C^uu: lower tiles only
    h->splitk_cap = h->syrk_splits * p * p;
#define A_(ptr, n) if (s == CES_OK && !h->forward_only) s = dalloc(h, &h->ptr, (n))
    A_(y, k); A_(ginv_diag, k); A_(mu, p); A_(ustar, p); A_(sinv_diag, p); A_(sig_diag, p); A_(bprior, p);
    A_(sums, k + p); A_(cvec, k); A_(zvec, k); A_(S, S_COUNT); A_(cb, p);
    A_(qpart, 2 * (int64_t)ny * h->ldJ); A_(formpart, 2 * ceil_div(h->ldJ, 256) + 2); A_(rowscratch, (p > k ? p : k));
    A_(E_all, (int64_t)nranks * k * h->ldJ); A_(W, k * h->ldJ);
    A_(Ut_all, (int64_t)nranks * p * h->ldJ); A_(Z, p * h->ldJ); A_(V, p * h->ldJ); A_(T, p * h->ldJ);
    A_(Cuu, p * h->ldp); A_(L, p * h->ldp); A_(Linv, round_up(p, CHOL_NB) * kLinvLd);
    A_(D, slots * h->ldJ * h->ldD);
    A_(ssq_partials, h->ssq_cap); A_(splitk_ws, h->splitk_cap);
    A_(dvec, h->ldJ); A_(uc, p);
#undef A_
    if (s == CES_OK) {
        void* ip = nullptr;
        if (cudaMalloc(&ip, sizeof(int)) != cudaSuccess) s = fail(CES_ERR_NOMEM, "cudaMalloc failed%s", "");
        else { h->info = static_cast<int*>(ip); h->allocs.push_back(ip); cudaMemsetAsync(ip, 0, sizeof(int), h->st); }
    }
    if (s == CES_OK) {
        void* hp = nullptr;
        if (cudaMallocHost(&hp, (S_COUNT + 2) * sizeof(double)) != cudaSuccess) s = fail(CES_ERR_NOMEM, "cudaMallocHost failed%s", "");
        else { h->hS = static_cast<double*>(hp); h->hinfo = reinterpret_cast<int*>(h->hS + S_COUNT); *h->hinfo = 0; }
    }
    if (s == CES_OK && cudaStreamSynchronize(h->st) != cudaSuccess) s = fail(CES_ERR_CUDA, "workspace initialisation failed%s", "");
    if (s != CES_OK) { ces_destroy(h); return s; }
    *out = h;
    return CES_OK;
}

int ces_destroy(ces_handle_t h) {
    if (!h) return CES_OK;
    cudaStreamSynchronize(h->st);
    if (h->aux_st) cudaStreamSynchronize(h->aux_st);
    if (h->copy_st) cudaStreamSynchronize(h->copy_st);
    for (void* ptr : h->allocs) cudaFree(ptr);
    if (h->run_ws) cudaFree(h->run_ws);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    for (auto& m : h->marks) cudaEventDestroy(m.second);
    for (cudaEvent_t e : h->mark_pool) cudaEventDestroy(e);
    if (h->cuu_ready) cudaEventDestroy(h->cuu_ready);
    if (h->chol_done) cudaEventDestroy(h->chol_done);
    if (h->aux_st) cudaStreamDestroy(h->aux_st);
    if (h->copy_ev) cudaEventDestroy(h->copy_ev);
    if (h->start_ev) cudaEventDestroy(h->start_ev);
    if (h->u_ev) cudaEventDestroy(h->u_ev);
    for (cudaEvent_t e : h->g_ev) if (e) cudaEventDestroy(e);
    if (h->up_begin) cudaEventDestroy(h->up_begin);
    for (cudaEvent_t e : h->out_ev) if (e) cudaEventDestroy(e);
    if (h->copy_st) cudaStreamDestroy(h->copy_st);
    if (h->out_st) { cudaStreamSynchronize(h->out_st); cudaStreamDestroy(h->out_st); }
    if (h->gather_st) { cudaStreamSynchronize(h->gather_st); cudaStreamDestroy(h->gather_st); }
    if (h->gather_go) cudaEventDestroy(h->gather_go);
    if (h->gather_done) cudaEventDestroy(h->gather_done);
    for (double* q : h->peer_E) if (q) cudaIpcCloseMemHandle(q);
    for (double* q : h->peer_Ut) if (q) cudaIpcCloseMemHandle(q);
    if (h->hS) cudaFreeHost(h->hS);
    delete h;
    cudaGetLastError();
    return CES_OK;
}

int ces_set_problem(ces_handle_t h, const double* y, const double* Gamma, const double* Sigma0, const double* mu,
                    const double* ustar) {
    CES_TRY(valid(h, false));
    if (h->forward_only) return fail(CES_ERR_STATE, "this handle was created for forward maps only%s", "");
    if (!y || !Gamma || !Sigma0 || !mu || !ustar) return fail(CES_ERR_INVALID, "ces_set_problem: null pointer%s", "");
    const int64_t p = h->p, k = h->k;
    h->have_problem = false;
    CES_CUDA(cudaMemcpyAsync(h->y, y, k * sizeof(double), cudaMemcpyHostToDevice, h->st));
    CES_CUDA(cudaMemcpyAsync(h->mu, mu, p * sizeof(double), cudaMemcpyHostToDevice, h->st));
    CES_CUDA(cudaMemcpyAsync(h->ustar, ustar, p * sizeof(double), cudaMemcpyHostToDevice, h->st));
    CES_CUDA(cudaStreamSynchronize(h->st));

    h->gamma_host.assign(Gamma, Gamma + k * k);
    if (h->GammaD) CES_TRY(upload_square(h, Gamma, k, h->GammaD, h->ldk));
    h->gamma_diag = is_diagonal(Gamma, k);
    if (h->gamma_diag) {
        std::vector<double> inv(k);
        for (int64_t i = 0; i < k; ++i) {
            if (!(Gamma[i * k + i] > 0.0)) return fail(CES_ERR_NOT_SPD, "Gamma: matrix is not positive definite (pivot %s%lld)", "", (long long)i + 1);
            inv[i] = 1.0 / Gamma[i * k + i];
        }
        CES_CUDA(cudaMemcpyAsync(h->ginv_diag, inv.data(), k * sizeof(double), cudaMemcpyHostToDevice, h->st));
        CES_CUDA(cudaStreamSynchronize(h->st));
    } else {
        if (!h->Ginv) { CES_TRY(dalloc(h, &h->Ginv, k * h->ldk)); }
        if (!h->R) { CES_TRY(dalloc(h, &h->R, k * h->ldJ)); }
        CES_TRY(device_spd_inverse(h, Gamma, k, h->Ginv, h->ldk, "Gamma"));
    }

    h->sigma_diag = is_diagonal(Sigma0, p);
    if (h->sigma_diag) {
        std::vector<double> inv(p), dg(p), bp(p);
        for (int64_t i = 0; i < p; ++i) {
            if (!(Sigma0[i * p + i] > 0.0)) return fail(CES_ERR_NOT_SPD, "sigma: matrix is not positive definite (pivot %s%lld)", "", (long long)i + 1);
            dg[i] = Sigma0[i * p + i];
            inv[i] = 1.0 / dg[i];
            bp[i] = mu[i] / dg[i];
        }
        CES_CUDA(cudaMemcpyAsync(h->sinv_diag, inv.data(), p * sizeof(double), cudaMemcpyHostToDevice, h->st));
        CES_CUDA(cudaMemcpyAsync(h->sig_diag, dg.data(), p * sizeof(double), cudaMemcpyHostToDevice, h->st));
        CES_CUDA(cudaMemcpyAsync(h->bprior, bp.data(), p * sizeof(double), cudaMemcpyHostToDevice, h->st));
        CES_CUDA(cudaStreamSynchronize(h->st));
    } else {
        if (!h->Sinv) { CES_TRY(dalloc(h, &h->Sinv, p * h->ldp)); }
        if (!h->Sigma0) { CES_TRY(dalloc(h, &h->Sigma0, p * h->ldp)); }
        if (!h->Y) { CES_TRY(dalloc(h, &h->Y, p * h->ldJ)); }
        CES_TRY(upload_square(h, Sigma0, p, h->Sigma0, h->ldp));
        CES_TRY(device_spd_inverse(h, Sigma0, p, h->Sinv, h->ldp, "sigma"));
        CES_TRY(matvec(h->st, h->Sinv, h->ldp, p, h->mu, h->bprior));
        CES_CUDA(cudaStreamSynchronize(h->st));
    }
    h->have_problem = true;
    return CES_OK;
}

int ces_phase1_sums(ces_handle_t h, const double* U, int64_t ldu, const double* G, int64_t ldg) {
    CES_TRY(valid(h, true));
    if (!U || !G || ldu < h->cols || ldg < h->cols) return fail(CES_ERR_INVALID, "phase1: bad ensemble pointers%s", "");
    mark(h, "phase1:begin");
    if (h->cols == 0) {
        CES_CUDA(cudaMemsetAsync(h->sums, 0, (h->k + h->p) * sizeof(double), h->st));
        return CES_OK;
    }
    CES_TRY(row_sums(h->st, G, ldg, h->k, h->cols, h->sums));
    CES_TRY(row_sums(h->st, U, ldu, h->p, h->cols, h->sums + h->k));
    mark(h, "phase1:end");
    return CES_OK;
}

// ---- phase 2 in pieces (ces_step_host pipelines them against the row-chunked upload of G) -----------------------
// Rows [r0, r0 + nr) of the forward outputs: E, W (diagonal Gamma) or R (dense), c = mean - y.  Row means are per row
// over the particles, so a row chunk is self-contained.
static int centre_g_rows(ces_handle_t h, const double* G, int64_t ldg, int64_t r0, int64_t nr) {
    const int64_t ld = h->ldJ;
    const double invJ = 1.0 / (double)h->Jg;
    double* E = e_block(h, h->rank) + r0 * ld;
    double* WR = (h->gamma_diag ? h->W : h->R) + r0 * ld;
    return centre_g(h->st, G + r0 * ldg, ldg, nr, h->cols, h->sums + r0, invJ, h->y + r0,
                    h->gamma_diag ? h->ginv_diag + r0 : nullptr, E, WR, ld, h->cvec + r0);
}

// After every row of G is centred: W = Gamma^-1 R for dense Gamma, z = Gamma^-1 c, data-space diagnostics.
static int finish_g(ces_handle_t h) {
    const int64_t k = h->k, ld = h->ldJ;
    cudaStream_t st = h->st;
    if (h->gamma_diag) {
        CES_TRY(scale_vector(st, h->ginv_diag, h->cvec, h->zvec, k));
    } else {
        GemmCall g;   // W = Gamma^-1 R   (K2 of SURVEY.md section 2.2)
        g.a_mode = A_MK; g.b_mode = B_KN;
        g.M = (int)k; g.N = (int)h->Jl; g.K = (int)k;
        g.A = h->Ginv; g.lda = h->ldk; g.B = h->R; g.ldb = ld; g.C = h->W; g.ldc = ld;
        CES_TRY(gemm(st, g));
        CES_TRY(matvec(st, h->Ginv, h->ldk, k, h->cvec, h->zvec));
    }
    const int nyk = form_row_blocks(k, ld);
    CES_TRY(data_forms(st, e_block(h, h->rank), h->W, ld, k, h->cvec, h->zvec, h->qpart));
    return finish_forms(st, h->qpart, nyk, ld, h->cols, true, h->formpart, h->S + S_SELF_DATA);
}

// Parameters: U~, Z, parameter-space diagnostics, local part of C^uu.
static int centre_u_all(ces_handle_t h, int rule, const double* U, int64_t ldu) {
    const int64_t p = h->p, k = h->k, ld = h->ldJ, cols = h->cols;
    const double invJ = 1.0 / (double)h->Jg;
    cudaStream_t st = h->st;
    double* Ut = ut_block(h, h->rank);
    const int nyp = form_row_blocks(p, ld);
    CES_TRY(centre_u(st, U, ldu, p, cols, h->sums + k, invJ, h->mu, h->ustar, h->sigma_diag ? h->sinv_diag : nullptr, Ut,
                     h->sigma_diag ? h->Z : h->Y, ld, h->qpart));
    CES_TRY(finish_forms(st, h->qpart, nyp, ld, cols, false, h->formpart, h->S + S_SELF_BIAS));
    if (!h->sigma_diag) {
        GemmCall g;   // Z = Sigma0^-1 (U - mu)
        g.a_mode = A_MK; g.b_mode = B_KN;
        g.M = (int)p; g.N = (int)h->Jl; g.K = (int)p;
        g.A = h->Sinv; g.lda = h->ldp; g.B = h->Y; g.ldb = ld; g.C = h->Z; g.ldc = ld;
        CES_TRY(gemm(st, g));
    }
    // --- local part of C^uu = U~ U~^T / (J-1) (+1e-8 I once)   (K6; :424 uses 1/J, :476/:512 use 1/(J-1))
    GemmCall g;
    g.a_mode = A_MK; g.b_mode = B_NK;
    g.M = (int)p; g.N = (int)p; g.K = (int)h->Jl;
    g.A = Ut; g.lda = ld; g.B = Ut; g.ldb = ld; g.C = h->Cuu; g.ldc = h->ldp;
    g.alpha = (rule == CES_RULE_EKS) ? 1.0 / (double)h->Jg : 1.0 / (double)(h->Jg - 1);
    g.flags = GEMM_C_LOWER_ONLY;
    g.splits = h->syrk_splits; g.splitk_ws = h->splitk_ws;
    g.diag_add = (h->rank == 0) ? 1e-8 : 0.0;
    return gemm(st, g);
}

int ces_phase2_centre(ces_handle_t h, int rule, const double* U, int64_t ldu, const double* G, int64_t ldg) {
    CES_TRY(valid(h, true));
    if (rule < CES_RULE_EKS || rule > CES_RULE_EKI) return fail(CES_ERR_INVALID, "unknown update rule %s%lld", "", rule);
    if (!U || !G) return fail(CES_ERR_INVALID, "phase2: null ensemble%s", "");
    h->last_rule = rule;
    mark(h, "phase2:begin");
    CES_TRY(centre_g_rows(h, G, ldg, 0, h->k));
    CES_TRY(finish_g(h));
    CES_TRY(centre_u_all(h, rule, U, ldu));
    mark(h, "phase2:end");
    return CES_OK;
}

// D = (1/J) E^T Wsrc by source block s (rows of D) and column panel (K3, K4); V = U~ D (K5).
// Source blocks (rows of D = particles of rank s) are taken in rotated order starting with this rank's own block:
// positions i in [first, first + count) map to s = (rank + i) % nranks, so the host can overlap the all-gather of the
// other ranks' E / U~ with position 0.  Consecutive positions whose s is contiguous in memory are processed by ONE
// batched D launch (blockIdx.y = block, one D slot each) and ONE batched V launch whose per-block partial products are
// summed by the split-K reduce kernel -- with P = 8 ranks and small shards a per-block launch has too few tiles to
// fill 148 SMs (256 tiles = 1.73 waves at Jl = 2048).
//
// A call may cover only part of the work (ces_step_host pipelines the interaction against the upload of G):
// column panels [c_begin, c_end) of this rank's particles, contraction rows [k_lo, k_hi) of the D GEMM -- chunks after
// the first accumulate into the panel (beta = 1; the sum of squares is taken from the stored values of the last
// chunk) --, and the D and V products separately.
struct InteractRange {
    int64_t c_begin = 0, c_end = -1;     // -1: Jl
    int64_t k_lo = 0, k_hi = -1;         // -1: k
    bool do_d = true, do_v = true;
    bool reset = true;                   // first call of a step: restart the sum-of-squares partials
    bool finish = true;                  // last call of a step: reduce the partials into S[S_SSQ]
};

// V = U~ D as a GEMM over the contraction K; split 2-4 ways when the d/128 x N/128 tiles quantise badly on 148 SMs
// (e.g. 512 tiles = 3.46 waves) and the partial planes fit the V workspace.
static int v_gemm(ces_handle_t h, GemmCall& g) {
    const double tiles = (double)gemm_tiles(g.M, g.N);
    int best = 1;
    double best_eff = 0.0;
    for (int sp = 1; sp <= 4; ++sp) {
        const double waves = tiles * sp / 148.0;
        const double eff = waves / ceil(waves);
        if (eff > best_eff + 0.02) { best_eff = eff; best = sp; }
        if (best_eff >= 0.97) break;
    }
    if (best > 1 && g.K >= 64 * best && (int64_t)best * g.N <= h->v_ws_planes * h->panel) {
        if (!h->v_ws) CES_TRY(dalloc(h, &h->v_ws, h->v_ws_planes * h->p * h->panel));
        g.splits = best;
        g.splitk_ws = h->v_ws;
    }
    return gemm(h->st, g);
}

// Event pair around a D launch (ces_profile_*), credited with the flops of the outputs it forms.
static int profile_begin(ces_handle_t h) {
    if (!h->profile) return CES_OK;
    while (h->ev_pool.size() < h->ev_used + 2) {
        cudaEvent_t e;
        CES_CUDA(cudaEventCreate(&e));
        h->ev_pool.push_back(e);
    }
    CES_CUDA(cudaEventRecord(h->ev_pool[h->ev_used], h->st));
    return CES_OK;
}
static int profile_end(ces_handle_t h, double flops) {
    if (!h->profile) return CES_OK;
    CES_CUDA(cudaEventRecord(h->ev_pool[h->ev_used + 1], h->st));
    h->ev_used += 2;
    h->prof_flops += flops;
    return CES_OK;
}

// Single GPU.  With R = E + c_g 1^T (c_g = mean - y) and W = B R for the symmetric B (Gamma^-1, or M^-1 in the re-solve):
//   J D = E^T W = S + c 1^T,   S = E^T B E  symmetric,   c = E^T w0,   w0 = B c_g.
// Column panel [a, b) of D forms only the lower trapezoid of S / J: D workspace row r stands for particle a + r, and the
// launch covers the tiles tn <= tm of E[:, a:J]^T W[:, a:b], storing (acc - c_i) / J (the row term on the last
// contraction chunk).  The strictly lower tiles of the panel's diagonal block are mirrored into its upper tiles; the rows
// above the panel (particles < a) are the transposes of earlier panels, whose products have already added them:
//   V[:, a:b] (+)= U~[:, a:J] Dws[0:J-a, :],    V[:, b:J] (+)= U~[:, a:b] Dws[b-a:J-a, :]^T,
// and once per step V += (U~ c / J) 1^T.  Every entry of D still comes from the J x J contraction: half the D flops of
// forming both triangles, the same V flops.  ||D||_F^2 is taken from the stored values plus the row term, a tile below
// the diagonal counting for its mirror too (GEMM_C_LOWER_TRAP).  `w0` must be ready when the last chunk of panel 0 runs.
static int symmetric_loops(ces_handle_t h, const double* Wsrc, const double* w0, bool accumulate_ssq, const InteractRange& rg) {
    const int64_t p = h->p, k = h->k, ld = h->ldJ, J = h->Jl;
    cudaStream_t st = h->st;
    if (rg.reset) h->ssq_used = 0;
    int64_t npart = h->ssq_used;
    const double invJ = 1.0 / (double)h->Jg;
    const int64_t c_end = rg.c_end < 0 ? J : rg.c_end;
    const int64_t k_lo = rg.k_lo, k_hi = rg.k_hi < 0 ? k : rg.k_hi;
    const bool last_chunk = (k_hi == k);
    double* E = e_block(h, 0);
    double* Ut = ut_block(h, 0);
    if (rg.do_d && last_chunk && rg.c_begin == 0) CES_TRY(col_dot(st, E, ld, k, J, w0, h->qpart, h->dvec));
    for (int64_t a = rg.c_begin; a < c_end; a += h->panel) {
        const int64_t nc = (c_end - a) < h->panel ? (c_end - a) : h->panel;
        const int64_t b = a + nc;
        if (rg.do_d) {
            GemmCall g1;
            g1.a_mode = A_KM; g1.b_mode = B_KN;
            g1.M = (int)(J - a); g1.N = (int)nc; g1.K = (int)(k_hi - k_lo);
            g1.A = E + k_lo * ld + a; g1.lda = ld;
            g1.B = Wsrc + k_lo * ld + a; g1.ldb = ld;
            g1.C = h->D; g1.ldc = h->ldD;
            g1.alpha = invJ;
            g1.beta = k_lo > 0 ? 1.0 : 0.0;
            g1.flags = GEMM_C_LOWER_TRAP;
            if (last_chunk) g1.row_vec = h->dvec + a;
            if (accumulate_ssq && last_chunk) {
                const int64_t tiles = gemm_trap_tiles(g1.M, g1.N);
                if (npart + tiles > h->ssq_cap) return fail(CES_ERR_STATE, "phase3: partial-sum buffer too small%s", "");
                g1.ssq_partials = h->ssq_partials + npart;
                npart += tiles;
            }
            CES_TRY(profile_begin(h));
            CES_TRY(gemm(st, g1));
            CES_TRY(profile_end(h, 2.0 * (double)g1.K * (double)gemm_trap_entries(g1.M, g1.N)));
            if (last_chunk) CES_TRY(mirror_lower_tiles(st, h->D, h->ldD, nc));
        }
        if (!rg.do_v) continue;
        GemmCall g2;
        g2.a_mode = A_MK; g2.b_mode = B_KN;
        g2.M = (int)p; g2.N = (int)nc; g2.K = (int)(J - a);
        g2.A = Ut + a; g2.lda = ld;
        g2.B = h->D; g2.ldb = h->ldD;
        g2.C = h->V + a; g2.ldc = ld;
        g2.beta = a > 0 ? 1.0 : 0.0;
        CES_TRY(v_gemm(h, g2));
        if (b < J) {
            GemmCall g3;
            g3.a_mode = A_MK; g3.b_mode = B_NK;
            g3.M = (int)p; g3.N = (int)(J - b); g3.K = (int)nc;
            g3.A = Ut + a; g3.lda = ld;
            g3.B = h->D + nc * h->ldD; g3.ldb = h->ldD;
            g3.C = h->V + b; g3.ldc = ld;
            g3.beta = a > 0 ? 1.0 : 0.0;
            CES_TRY(v_gemm(h, g3));
        }
    }
    h->ssq_used = npart;
    if (rg.do_v && c_end == J) {
        CES_TRY(row_dot(st, Ut, ld, p, J, h->dvec, invJ, h->uc));
        CES_TRY(add_col_vector(st, h->V, ld, p, J, h->uc, 1.0, nullptr));
    }
    if (accumulate_ssq && rg.finish) CES_TRY(sum_vector(st, h->ssq_partials, npart, h->S + S_SSQ));
    return CES_OK;
}

static int interaction_loops(ces_handle_t h, const double* Wsrc, const double* w0, bool accumulate_ssq, int first, int count,
                             const InteractRange& rg = InteractRange()) {
    if (h->nranks == 1) return symmetric_loops(h, Wsrc, w0, accumulate_ssq, rg);
    const int64_t p = h->p, k = h->k, ld = h->ldJ;
    cudaStream_t st = h->st;
    if (first == 0 && rg.reset) h->ssq_used = 0;
    int64_t npart = h->ssq_used;
    const double invJ = 1.0 / (double)h->Jg;
    const int64_t c_end = rg.c_end < 0 ? h->Jl : rg.c_end;
    const int64_t k_lo = rg.k_lo, k_hi = rg.k_hi < 0 ? k : rg.k_hi;
    const bool last_chunk = (k_hi == k);
    for (int64_t c0 = rg.c_begin; c0 < c_end; c0 += h->panel) {
        const int64_t nc = (c_end - c0) < h->panel ? (c_end - c0) : h->panel;
        int i = first;
        while (i < first + count) {
            const int s0 = (h->rank + i) % h->nranks;
            // run of positions with contiguous s (stops at the wrap-around); position 0 (own block) stays alone so
            // that it can run while the gathers are in flight
            int run = 1;
            if (i > 0)
                while (i + run < first + count && s0 + run < h->nranks) ++run;
            GemmCall g1;
            g1.a_mode = A_KM; g1.b_mode = B_KN;
            g1.M = (int)h->Jl; g1.N = (int)nc; g1.K = (int)(k_hi - k_lo);
            g1.A = e_block(h, s0) + k_lo * ld; g1.lda = ld;
            g1.B = Wsrc + k_lo * ld + c0; g1.ldb = ld;
            g1.C = h->D; g1.ldc = h->ldD;
            g1.alpha = invJ;
            g1.beta = k_lo > 0 ? 1.0 : 0.0;
            g1.batch = run; g1.a_batch_rows = k; g1.c_batch_elems = h->Jl * h->ldD;
            if (rg.do_d && accumulate_ssq && last_chunk) {
                const int64_t tiles = (int64_t)gemm_tiles(g1.M, g1.N) * run;
                if (npart + tiles > h->ssq_cap) return fail(CES_ERR_STATE, "phase3: partial-sum buffer too small%s", "");
                g1.ssq_partials = h->ssq_partials + npart;
                npart += tiles;
            }
            if (rg.do_d) {
                CES_TRY(profile_begin(h));
                CES_TRY(gemm(st, g1));
                CES_TRY(profile_end(h, 2.0 * (double)g1.K * (double)g1.M * (double)g1.N * run));
            }
            if (!rg.do_v) { i += run; continue; }
            GemmCall g2;
            g2.a_mode = A_MK; g2.b_mode = B_KN;
            g2.M = (int)p; g2.N = (int)nc; g2.K = (int)h->Jl;
            g2.A = ut_block(h, s0); g2.lda = ld;
            g2.B = h->D; g2.ldb = h->ldD;
            g2.C = h->V + c0; g2.ldc = ld;
            g2.beta = (i == 0) ? 0.0 : 1.0;
            if (run > 1) {
                // per-block partial products into workspace planes, summed (+ beta * V) by the reduce kernel
                if (!h->v_ws) CES_TRY(dalloc(h, &h->v_ws, h->v_ws_planes * p * h->panel));
                g2.batch = run; g2.a_batch_rows = p; g2.b_batch_rows = h->Jl;
                g2.splitk_ws = h->v_ws;
                CES_TRY(gemm(st, g2));
            } else {
                CES_TRY(v_gemm(h, g2));
            }
            i += run;
        }
    }
    h->ssq_used = npart;
    if (accumulate_ssq && rg.finish && first + count == h->nranks) CES_TRY(sum_vector(st, h->ssq_partials, npart, h->S + S_SSQ));
    return CES_OK;
}

static int start_cholesky(ces_handle_t h, int rule);

int ces_phase3_interact(ces_handle_t h, int rule, int skip_interaction) {
    CES_TRY(valid(h, true));
    if (rule != h->last_rule) return fail(CES_ERR_STATE, "phase3: rule differs from phase2%s", "");
    CES_TRY(start_cholesky(h, rule));
    if (skip_interaction) return CES_OK;       // 'constant' step size: D is formed once, by ces_phase3c_resolve
    mark(h, "phase3:begin");
    CES_TRY(interaction_loops(h, h->W, h->zvec, true, 0, h->nranks));
    mark(h, "phase3:end");
    return CES_OK;
}

int ces_phase3_blocks(ces_handle_t h, int rule, int first, int count) {
    CES_TRY(valid(h, true));
    if (rule != h->last_rule) return fail(CES_ERR_STATE, "phase3: rule differs from phase2%s", "");
    if (first < 0 || count < 0 || first + count > h->nranks) return fail(CES_ERR_INVALID, "phase3_blocks: bad block range%s", "");
    if (first == 0) CES_TRY(start_cholesky(h, rule));
    if (count == 0) return CES_OK;
    mark(h, first == 0 ? "phase3:own:begin" : "phase3:rest:begin");
    CES_TRY(interaction_loops(h, h->W, h->zvec, true, first, count));
    mark(h, first == 0 ? "phase3:own:end" : "phase3:rest:end");
    return CES_OK;
}

static int start_cholesky(ces_handle_t h, int rule) {
    const int64_t p = h->p;
    cudaStream_t st = h->st;
    // chol(C^uu)  (K7); EKI has no noise term and skips it.  Only the noise GEMM of phase 4 needs the factor, so it
    // is computed on a high-priority side stream while the main stream runs the D and V GEMMs (its ~50 small
    // launches would otherwise sit on the critical path: 3 % of a cfg3 step).  The ensemble noise needs no factor.
    if (rule != CES_RULE_EKI && !ensemble_noise(h)) {
        if (!h->aux_st) {
            int lo = 0, hi = 0;
            CES_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CES_CUDA(cudaStreamCreateWithPriority(&h->aux_st, cudaStreamNonBlocking, hi));
            CES_CUDA(cudaEventCreateWithFlags(&h->cuu_ready, cudaEventDisableTiming));
            CES_CUDA(cudaEventCreateWithFlags(&h->chol_done, cudaEventDisableTiming));
        }
        CES_CUDA(cudaEventRecord(h->cuu_ready, st));
        CES_CUDA(cudaStreamWaitEvent(h->aux_st, h->cuu_ready, 0));
        CES_CUDA(cudaMemcpy2DAsync(h->L, h->ldp * sizeof(double), h->Cuu, h->ldp * sizeof(double), p * sizeof(double), p,
                                   cudaMemcpyDeviceToDevice, h->aux_st));
        CES_TRY(potrf_lower(h->aux_st, h->L, h->ldp, p, h->Linv, kLinvLd, h->info));
        CES_CUDA(cudaEventRecord(h->chol_done, h->aux_st));
        h->chol_pending = true;
    }
    return CES_OK;
}

int ces_peek_step_size(ces_handle_t h, int ts_kind, double fixed_h, double* hk_host) {
    CES_TRY(valid(h, true));
    CES_TRY(check_step(h, "peek", std::nullopt, ts_kind, false, std::nullopt, true));
    const double alphaJ = (double)(h->p + 1) / (double)h->Jg;
    CES_TRY(step_scalars(h->st, h->S, ts_kind == CES_TS_FIXED ? 1 : 0, fixed_h, alphaJ, ens_inv_nc(h, h->last_rule)));
    CES_CUDA(cudaMemcpyAsync(h->hS, h->S, S_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->st));
    CES_CUDA(cudaStreamSynchronize(h->st));
    if (hk_host) *hk_host = h->hS[S_H];
    return CES_OK;
}

int ces_phase3b_cpp(ces_handle_t h) {
    CES_TRY(valid(h, true));
    const int64_t k = h->k, ld = h->ldJ;
    cudaStream_t st = h->st;
    if (!h->Cpp) {
        h->cpp_splits = splitk_count(gemm_trap_tiles((int)k, (int)k), ld);
        CES_TRY(dalloc(h, &h->Cpp, k * h->ldk));
        CES_TRY(dalloc(h, &h->cpp_ws, h->cpp_splits * k * k));
        CES_TRY(dalloc(h, &h->Mk, k * h->ldk));
        CES_TRY(dalloc(h, &h->MkInv, k * h->ldk));
        CES_TRY(dalloc(h, &h->MkLinv, round_up(k, CHOL_NB) * kLinvLd));
        CES_TRY(dalloc(h, &h->Wr, k * ld));
        CES_TRY(dalloc(h, &h->zr, k));
        CES_TRY(dalloc(h, &h->GammaD, k * h->ldk));
        if (!h->R) CES_TRY(dalloc(h, &h->R, k * ld));
        CES_TRY(upload_square(h, h->gamma_host.data(), k, h->GammaD, h->ldk));
    }
    // C^pp = cov(G, bias=True) = E E^T / J   (ces/calibrate.py:440, 472): local part, lower tiles, mirrored
    GemmCall g;
    g.a_mode = A_MK; g.b_mode = B_NK;
    g.M = (int)k; g.N = (int)k; g.K = (int)h->Jl;
    g.A = e_block(h, h->rank); g.lda = ld; g.B = g.A; g.ldb = ld; g.C = h->Cpp; g.ldc = h->ldk;
    g.alpha = 1.0 / (double)h->Jg;
    g.flags = GEMM_C_LOWER_ONLY;
    g.splits = h->cpp_splits; g.splitk_ws = h->cpp_ws;
    return gemm(st, g);
}

int ces_phase3c_resolve(ces_handle_t h, int rule) {
    CES_TRY(valid(h, true));
    if (rule != h->last_rule) return fail(CES_ERR_STATE, "phase3c: rule differs from phase2%s", "");
    if (!h->Cpp) return fail(CES_ERR_STATE, "phase3c: ces_phase3b_cpp has not run%s", "");
    const int64_t k = h->k, ld = h->ldJ;
    cudaStream_t st = h->st;
    // R = G - y: stored by phase 2 for dense Gamma, rebuilt as E + (mean - y) 1^T for diagonal Gamma
    if (h->gamma_diag) {
        CES_CUDA(cudaMemcpyAsync(h->R, e_block(h, h->rank), (size_t)k * ld * sizeof(double), cudaMemcpyDeviceToDevice, st));
        CES_TRY(add_col_vector(st, h->R, ld, k, h->cols, h->cvec, 1.0, nullptr));
    }
    // M = hk * C^pp + Gamma with the hk of ces_peek_step_size (device scalar), inverted through its Cholesky factor
    CES_TRY(form_implicit(st, h->Cpp, h->ldk, h->GammaD, h->ldk, nullptr, h->S + S_H, k, h->Mk, h->ldk));
    CES_TRY(potrf_lower(st, h->Mk, h->ldk, k, h->MkLinv, kLinvLd, h->info));
    CES_TRY(spd_inverse_from_factor(st, h->Mk, h->ldk, k, h->MkLinv, kLinvLd, h->MkInv, h->ldk));
    GemmCall g;
    g.a_mode = A_MK; g.b_mode = B_KN;
    g.M = (int)k; g.N = (int)h->Jl; g.K = (int)k;
    g.A = h->MkInv; g.lda = h->ldk; g.B = h->R; g.ldb = ld; g.C = h->Wr; g.ldc = ld;
    CES_TRY(gemm(st, g));
    CES_TRY(matvec(st, h->MkInv, h->ldk, k, h->cvec, h->zr));   // w0 = M^-1 c of the single-GPU schedule
    // the step size stays the one computed from the Gamma-only D (ces/calibrate.py:437 precedes :439-441)
    return interaction_loops(h, h->Wr, h->zr, false, 0, h->nranks);
}

// time_step='spectral' (ces/calibrate.py:249-251): radspec = eigvals(D).real.max() = lambda_max(Gamma^-1 C^pp), see eig.cu.
// Needs the (all-reduced) C^pp of ces_phase3b_cpp.
int ces_phase3d_spectral(ces_handle_t h, double* radspec_host, int* lanczos_steps_host) {
    CES_TRY(valid(h, true));
    if (!h->Cpp) return fail(CES_ERR_STATE, "phase3d: ces_phase3b_cpp has not run%s", "");
    const int64_t k = h->k;
    const int64_t mmax = k < 768 ? k : 768;
    if (!h->eig_ws) CES_TRY(dalloc(h, &h->eig_ws, (2 * (mmax + 1) + 2) * k + 4 * mmax + 8));
    return spectral_radius(h->st, h->Cpp, h->ldk, k, h->gamma_diag ? nullptr : h->Ginv, h->gamma_diag ? h->ginv_diag : nullptr,
                           h->eig_ws, mmax, radspec_host, lanczos_steps_host);
}

// ---- factored formulation: the same update without forming the J x J matrix -------------------------------------
//   V = U~ D = (1/J) (U~ E^T) W         (d x k) then (d x J):  4 d k J flops instead of 2 (k + d) J^2
//   ||D||_F^2 = sum((E E^T) o (W W^T)) / J^2          two k x k Gram matrices:  ~2 k^2 J flops (symmetric halves)
// Phase 3f-a forms the local parts of P1 = U~ E^T, GE = E E^T, GW = W W^T over this rank's columns
// [host: all-reduce(sum) of "p1", "gram_e", "gram_w"]; phase 3f-b finishes V and the sum of squares.
__global__ void __launch_bounds__(256) gram_dot_kernel(const double* __restrict__ A, const double* __restrict__ B, long long ld,
                                                       int n, double scale, double* __restrict__ part) {
    __shared__ double scratch[32];
    const int i = blockIdx.x;
    double a = 0.0;
    for (int j = threadIdx.x; j < n; j += 256) a += A[(size_t)i * ld + j] * B[(size_t)i * ld + j];
    const double t = block_sum(a, scratch);
    if (threadIdx.x == 0) part[i] = t * scale;
}

int ces_phase3f_products(ces_handle_t h, int rule) {
    CES_TRY(valid(h, true));
    if (rule != h->last_rule) return fail(CES_ERR_STATE, "phase3f: rule differs from phase2%s", "");
    CES_TRY(check_step(h, "phase3f", std::nullopt, std::nullopt, false, CES_FORM_FACTORED, true));
    const int64_t p = h->p, k = h->k, ld = h->ldJ;
    cudaStream_t st = h->st;
    if (!h->P1) {
        h->gram_splits = splitk_count(gemm_trap_tiles((int)k, (int)k), ld);
        // P1 has few (d/128 x k/128) tiles and a long contraction: split it so the tiles fill the machine
        h->p1_splits = splitk_count(gemm_tiles((int)p, (int)k), ld);
        const int64_t ws = h->gram_splits * k * k > h->p1_splits * p * k ? h->gram_splits * k * k : h->p1_splits * p * k;
        CES_TRY(dalloc(h, &h->P1, p * h->ldk));
        CES_TRY(dalloc(h, &h->GE, k * h->ldk));
        CES_TRY(dalloc(h, &h->GW, k * h->ldk));
        CES_TRY(dalloc(h, &h->gram_ws, ws));
        CES_TRY(dalloc(h, &h->gram_part, k));
    }
    // chol(C^uu) on the side stream, as in ces_phase3_interact
    CES_TRY(ces_phase3_interact(h, rule, 1));
    const double* E = e_block(h, h->rank);
    const double* Ut = ut_block(h, h->rank);
    GemmCall g;                                  // P1 = U~ E^T  (d x k), contraction over the local particles
    g.a_mode = A_MK; g.b_mode = B_NK;
    g.M = (int)p; g.N = (int)k; g.K = (int)h->Jl;
    g.A = Ut; g.lda = ld; g.B = E; g.ldb = ld; g.C = h->P1; g.ldc = h->ldk;
    g.splits = h->p1_splits; g.splitk_ws = h->gram_ws;
    CES_TRY(gemm(st, g));
    for (int which = 0; which < 2; ++which) {   // GE = E E^T, GW = W W^T (lower tiles, mirrored)
        GemmCall s2;
        s2.a_mode = A_MK; s2.b_mode = B_NK;
        s2.M = (int)k; s2.N = (int)k; s2.K = (int)h->Jl;
        s2.A = which == 0 ? E : h->W; s2.lda = ld; s2.B = s2.A; s2.ldb = ld;
        s2.C = which == 0 ? h->GE : h->GW; s2.ldc = h->ldk;
        s2.flags = GEMM_C_LOWER_ONLY;
        s2.splits = h->gram_splits; s2.splitk_ws = h->gram_ws;
        CES_TRY(gemm(st, s2));
    }
    return CES_OK;
}

int ces_phase3f_finish(ces_handle_t h, int rule) {
    CES_TRY(valid(h, true));
    if (rule != h->last_rule || !h->P1) return fail(CES_ERR_STATE, "phase3f_finish: ces_phase3f_products has not run%s", "");
    const int64_t p = h->p, k = h->k, ld = h->ldJ;
    cudaStream_t st = h->st;
    const double invJ = 1.0 / (double)h->Jg;
    GemmCall g;                                  // V = (1/J) P1 W
    g.a_mode = A_MK; g.b_mode = B_KN;
    g.M = (int)p; g.N = (int)h->Jl; g.K = (int)k;
    g.A = h->P1; g.lda = h->ldk; g.B = h->W; g.ldb = ld; g.C = h->V; g.ldc = ld;
    g.alpha = invJ;
    CES_TRY(gemm(st, g));
    // ||D||_F^2 = sum_ab GE_ab GW_ab / J^2.  Every rank holds the all-reduced Gram matrices, so the value is global:
    // only rank 0 contributes it to the scalar that the host all-reduces afterwards.
    gram_dot_kernel<<<(unsigned)k, 256, 0, st>>>(h->GE, h->GW, h->ldk, (int)k, invJ * invJ, h->gram_part);
    CES_LAUNCHED(1);
    if (h->rank == 0) CES_TRY(sum_vector(st, h->gram_part, k, h->S + S_SSQ));
    else CES_CUDA(cudaMemsetAsync(h->S + S_SSQ, 0, sizeof(double), st));
    return CES_OK;
}

int ces_phase4a_drift(ces_handle_t h, double switch_) {
    CES_TRY(valid(h, true));
    if (h->last_rule != CES_RULE_ALDI_CONSTANT) return fail(CES_ERR_STATE, "phase4a is for aldi_constant only%s", "");
    const int64_t p = h->p, ld = h->ldJ;
    cudaStream_t st = h->st;
    const double alphaJ = (double)(p + 1) / (double)h->Jg;
    // drift = -(U~ D) - C Sigma0^-1 (U - mu) + switch * alpha_J * U~     (:515-517)
    CES_TRY(axpbypcz(st, p, h->Jl, -1.0, h->V, ld, switch_ * alphaJ, nullptr, ut_block(h, h->rank), ld, 0.0, nullptr, nullptr,
                     0, h->T, ld));
    GemmCall g;
    g.a_mode = A_MK; g.b_mode = B_KN;
    g.M = (int)p; g.N = (int)h->Jl; g.K = (int)p;
    g.A = h->Cuu; g.lda = h->ldp; g.B = h->Z; g.ldb = ld; g.C = h->T; g.ldc = ld;
    g.alpha = -1.0; g.beta = 1.0;
    CES_TRY(gemm(st, g));
    CES_TRY(absmax(st, h->T, ld, p, h->cols, h->rowscratch, h->S + S_MAXDRIFT));
    return CES_OK;
}

// Ensemble noise (CES_NOISE_ENSEMBLE) for the local columns [c0, c0 + nc) of U_next, added into C (= Uout + c0):
//   C += sqrt(2h / n_C) sum_s U~_s xi[s's particles, the columns' global particles]
// over the source blocks s of every rank (all of U~ is on this rank after the gathers), column panel by column panel.
// Philox mode materialises each xi block in the D-panel workspace, which phase 4 no longer needs; it is not generated in
// the GEMM's producer, where every row tile of U~ would regenerate it on the FP64 pipe the DMMAs use.
static int add_ensemble_noise(ces_handle_t h, int64_t c0, int64_t nc, double* C, int64_t ldc) {
    cudaStream_t st = h->st;
    const int64_t col0 = (int64_t)h->rank * h->Jl;         // global particle of local column 0
    mark(h, "noise:begin");
    for (int64_t q0 = c0; q0 < c0 + nc; q0 += h->panel) {
        const int64_t nq = (c0 + nc - q0) < h->panel ? (c0 + nc - q0) : h->panel;
        for (int s = 0; s < h->nranks; ++s) {
            const int64_t lo = (int64_t)s * h->Jl < h->Jg ? (int64_t)s * h->Jl : h->Jg;
            const int64_t ks = (lo + h->Jl < h->Jg ? lo + h->Jl : h->Jg) - lo;     // particles of block s
            if (ks < 1) continue;
            GemmCall g;
            g.a_mode = A_MK; g.b_mode = B_KN;
            g.M = (int)h->p; g.N = (int)nq; g.K = (int)ks;
            g.A = ut_block(h, s); g.lda = h->ldJ;
            if (h->noise_xi) {
                g.B = h->noise_xi + lo * h->noise_ldxi + q0; g.ldb = h->noise_ldxi;
            } else {
                CES_TRY(fill_ensemble_noise(st, h->D, h->ldD, ks, nq, lo, col0 + q0, h->noise_seed, h->noise_step));
                g.B = h->D; g.ldb = h->ldD;
            }
            g.C = C + (q0 - c0); g.ldc = ldc;
            g.alpha_dev = h->S + S_ENS_ALPHA; g.beta = 1.0;
            CES_TRY(gemm(st, g));
        }
    }
    mark(h, "noise:end");
    return CES_OK;
}

int ces_phase4_update(ces_handle_t h, int rule, int ts_kind, double fixed_h, const double* U, int64_t ldu,
                      const double* xi, int64_t ldxi, double* Uout, int64_t ldo, double* hk_host, double* metrics_host) {
    CES_TRY(valid(h, true));
    if (rule != h->last_rule) return fail(CES_ERR_STATE, "phase4: rule differs from phase2%s", "");
    CES_TRY(check_step(h, "phase4", std::nullopt, ts_kind, true, std::nullopt, U && Uout && (xi || !needs_xi(h, rule))));
    const bool ens = ensemble_noise(h);
    const int64_t p = h->p, ld = h->ldJ;
    cudaStream_t st = h->st;
    const double alphaJ = (double)(p + 1) / (double)h->Jg;
    double* S = h->S;
    double* Ut = ut_block(h, h->rank);

    // noise operand: TMA needs a 16-byte aligned base and an even leading dimension
    const double* xi_use = ens ? nullptr : xi;         // ensemble mode ignores xi
    int64_t ldxi_use = ldxi;
    if (xi_use && (((reinterpret_cast<uintptr_t>(xi) & 15) != 0) || (ldxi & 1))) {
        if (!h->xi_pad) { CES_TRY(dalloc(h, &h->xi_pad, p * ld)); }
        CES_TRY(pad_copy(st, xi, ldxi, p, h->cols, h->xi_pad, ld));
        xi_use = h->xi_pad; ldxi_use = ld;
    }

    mark(h, "phase4:begin");
    if (h->chol_pending) {              // the factor of C^uu from the side stream
        CES_CUDA(cudaStreamWaitEvent(st, h->chol_done, 0));
        h->chol_pending = false;
    }
    mark(h, "phase4:chol_ready");
    const int kind = (rule == CES_RULE_ALDI_CONSTANT) ? 2 : (ts_kind == CES_TS_FIXED ? 1 : 0);
    if (ts_kind != CES_TS_KEEP || rule == CES_RULE_ALDI_CONSTANT) CES_TRY(step_scalars(st, S, kind, fixed_h, alphaJ, ens_inv_nc(h, rule)));

    GemmCall noise;   // += sqrt(2h) chol(C) xi     (K8; L lower triangular -> skip the zero blocks)
    noise.a_mode = A_MK; noise.b_mode = B_KN;
    noise.M = (int)p; noise.N = (int)h->cols; noise.K = (int)p;
    noise.A = h->L; noise.lda = h->ldp; noise.B = xi_use; noise.ldb = ldxi_use; noise.C = Uout; noise.ldc = ldo;
    noise.alpha_dev = S + S_SQRT2H; noise.beta = 1.0; noise.flags = GEMM_A_LOWER_TRI;

    // With a host destination (ces_step_host / ces_set_pending_output) the explicit rules finish U_next in column
    // chunks: chunk c is copied to the host on a second stream while chunk c + 1 is computed, so that only the last
    // chunk's download is exposed.  Chunk starts are multiples of 128 columns (TMA operand alignment).
    // Chunk widths are whole double-waves of the p x p GEMMs (2 x SMs tiles), so chunking adds no partial wave.  The
    // download (p x cols x 8 B over PCIe) takes longer than assembling U_next, so it should start as early as possible:
    // a first chunk of one unit, then the rest in three pieces; exposed = the first chunk's assembly + whatever of the
    // download the assembly could not cover.
    int64_t cstart[6] = {0, h->cols, h->cols, h->cols, h->cols, h->cols};
    int nchunks = 1;
    if (h->pending_out && rule != CES_RULE_EKS && h->cols >= 4096) {
        const int64_t tiles_m = ceil_div(p, p <= 64 ? 64 : GEMM_BM);
        int64_t unit_blocks = (2 * (int64_t)gemm_sm_count()) / tiles_m;
        if (unit_blocks < 1) unit_blocks = 1;
        int64_t unit = unit_blocks * GEMM_BN;
        const int64_t eighth = round_up(ceil_div(h->cols, 8), GEMM_BN);
        if (unit > eighth) unit = eighth;                       // few row tiles: a wave is wider than the ensemble
        const int64_t units = h->cols / unit;                   // whole units; the last chunk takes the remainder
        if (units >= 2) {
            cstart[nchunks++] = unit;
            const int64_t pieces = units - 1 >= 3 ? 3 : units - 1;
            for (int64_t i = 1; i < pieces; ++i) cstart[nchunks++] = unit + (units - 1) * i / pieces * unit;
        }
    }
    bool downloaded = false;
    if (nchunks > 1) {
        if (!h->out_st) {
            CES_CUDA(cudaStreamCreateWithFlags(&h->out_st, cudaStreamNonBlocking));
            for (cudaEvent_t& e : h->out_ev) CES_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        downloaded = true;
    }
    cstart[nchunks] = h->cols;
    for (int chunk = 0; chunk < nchunks && h->cols > 0 && rule != CES_RULE_EKS; ++chunk) {
        const int64_t c0 = cstart[chunk], nc = cstart[chunk + 1] - c0;
        GemmCall nz = noise;
        nz.N = (int)nc; nz.B = xi_use ? xi_use + c0 : nullptr; nz.C = Uout + c0;
        if (rule == CES_RULE_ALDI) {
            // U + h alpha_J U~ - h V - h C Z + sqrt(2h) L xi      (:484-488)
            CES_TRY(axpbypcz(st, p, nc, 1.0, U + c0, ldu, 1.0, S + S_H_ALPHA, Ut + c0, ld, 1.0, S + S_NEG_H, h->V + c0, ld,
                             Uout + c0, ldo));
            GemmCall g;
            g.a_mode = A_MK; g.b_mode = B_KN;
            g.M = (int)p; g.N = (int)nc; g.K = (int)p;
            g.A = h->Cuu; g.lda = h->ldp; g.B = h->Z + c0; g.ldb = ld; g.C = Uout + c0; g.ldc = ldo;
            g.alpha_dev = S + S_NEG_H; g.beta = 1.0;
            CES_TRY(gemm(st, g));
            CES_TRY(ens ? add_ensemble_noise(h, c0, nc, Uout + c0, ldo) : gemm(st, nz));
        } else if (rule == CES_RULE_ALDI_CONSTANT) {
            // U + h drift + sqrt(2h) L xi                         (:525-527)
            CES_TRY(axpbypcz(st, p, nc, 1.0, U + c0, ldu, 1.0, S + S_H, h->T + c0, ld, 0.0, nullptr, nullptr, 0, Uout + c0, ldo));
            CES_TRY(ens ? add_ensemble_noise(h, c0, nc, Uout + c0, ldo) : gemm(st, nz));
        } else {                                                   // EKI
            CES_TRY(axpbypcz(st, p, nc, 1.0, U + c0, ldu, 1.0, S + S_NEG_H, h->V + c0, ld, 0.0, nullptr, nullptr, 0, Uout + c0, ldo));
        }
        if (downloaded) {
            CES_CUDA(cudaEventRecord(h->out_ev[chunk], st));
            CES_CUDA(cudaStreamWaitEvent(h->out_st, h->out_ev[chunk], 0));
            CES_CUDA(cudaMemcpy2DAsync(h->pending_out + c0, h->cols * sizeof(double), Uout + c0, ldo * sizeof(double),
                                       nc * sizeof(double), h->pending_rows, cudaMemcpyDeviceToHost, h->out_st));
        }
    }
    if (h->cols > 0 && rule == CES_RULE_EKS) {
        {
            // semi-implicit EKS (:443-447) with (I + h C S^-1)^-1 = S (S + h C)^-1   (SURVEY.md F6)
            if (!h->M) { CES_TRY(dalloc(h, &h->M, p * h->ldp)); }
            if (!h->Minv) { CES_TRY(dalloc(h, &h->Minv, round_up(p, CHOL_NB) * kLinvLd)); }
            CES_TRY(form_implicit(st, h->Cuu, h->ldp, h->sigma_diag ? nullptr : h->Sigma0, h->ldp, h->sig_diag, S + S_H, p,
                                  h->M, h->ldp));
            CES_TRY(potrf_lower(st, h->M, h->ldp, p, h->Minv, kLinvLd, h->info));
            // T = U - h V + h C Sigma0^-1 mu
            CES_TRY(axpbypcz(st, p, h->cols, 1.0, U, ldu, 1.0, S + S_NEG_H, h->V, ld, 0.0, nullptr, nullptr, 0, h->T, ld));
            CES_TRY(matvec(st, h->Cuu, h->ldp, p, h->bprior, h->cb));
            CES_TRY(add_col_vector(st, h->T, ld, p, h->cols, h->cb, 1.0, S + S_H));
            CES_TRY(trsm_lower(st, h->M, h->ldp, p, h->Minv, kLinvLd, h->T, ld, h->cols, false));
            CES_TRY(trsm_lower(st, h->M, h->ldp, p, h->Minv, kLinvLd, h->T, ld, h->cols, true));
            if (h->sigma_diag) {
                CES_TRY(row_scale(st, h->sig_diag, h->T, ld, p, h->cols));
                CES_TRY(axpbypcz(st, p, h->cols, 1.0, h->T, ld, 0.0, nullptr, nullptr, 0, 0.0, nullptr, nullptr, 0, Uout, ldo));
            } else {
                GemmCall g;
                g.a_mode = A_MK; g.b_mode = B_KN;
                g.M = (int)p; g.N = (int)h->cols; g.K = (int)p;
                g.A = h->Sigma0; g.lda = h->ldp; g.B = h->T; g.ldb = ld; g.C = Uout; g.ldc = ldo;
                CES_TRY(gemm(st, g));
            }
            CES_TRY(ens ? add_ensemble_noise(h, 0, h->cols, Uout, ldo) : gemm(st, noise));
        }
    }
    mark(h, "phase4:computed");
    if (!downloaded) return finish_step(h, Uout, ldo, true, hk_host, metrics_host);
    mark(h, "phase4:downloaded", h->out_st);
    h->pending_out = nullptr;           // already on its way, chunk by chunk
    const int s = finish_step(h, Uout, ldo, true, hk_host, metrics_host);
    CES_CUDA(cudaStreamSynchronize(h->out_st));   // the host copy is complete whatever the status
    return s;
}

static int interaction_phase(ces_handle_t h, int rule, int formulation) {
    if (formulation == CES_FORM_FACTORED) {
        CES_TRY(ces_phase3f_products(h, rule));
        return ces_phase3f_finish(h, rule);
    }
    return ces_phase3_interact(h, rule, 0);
}

int ces_step(ces_handle_t h, int rule, int ts_kind, double fixed_h, double switch_, int formulation, const double* U,
             int64_t ldu, const double* G, int64_t ldg, const double* xi, int64_t ldxi, double* Uout, int64_t ldo,
             double* hk_host, double* metrics_host) {
    CES_TRY(valid(h, true));
    if (h->nranks != 1) return fail(CES_ERR_STATE, "ces_step is single-GPU; use the phases with nranks > 1%s", "");
    CES_TRY(check_step(h, "ces_step", rule, ts_kind, false, formulation, U && G && Uout && (xi || !needs_xi(h, rule))));
    if (small_path(h, formulation)) {
        SmallStepCall c = small_call(h, rule, ts_kind, fixed_h, switch_);
        c.U = U; c.G = G; c.ldu = ldu; c.ldg = ldg; c.out = Uout; c.ldo = ldo; c.S = h->S;
        if (!c.ensemble) { c.xi = xi; c.ldxi = ldxi; }
        h->last_rule = rule;
        CES_TRY(small_step(h->st, c));
        return finish_step(h, Uout, ldo, false, hk_host, metrics_host);
    }
    CES_TRY(ces_phase1_sums(h, U, ldu, G, ldg));
    CES_TRY(ces_phase2_centre(h, rule, U, ldu, G, ldg));
    CES_TRY(interaction_phase(h, rule, formulation));
    if (rule == CES_RULE_ALDI_CONSTANT) CES_TRY(ces_phase4a_drift(h, switch_));
    return ces_phase4_update(h, rule, ts_kind, fixed_h, U, ldu, xi, ldxi, Uout, ldo, hk_host, metrics_host);
}

// ---- the update on HOST buffers, as pieces (include/ces_b200.h: "host steps") -----------------------------------
// ces_step_host (single GPU) strings them together; a column-sharded caller runs its collectives in between.
static int host_staging(ces_handle_t h) {
    const int64_t p = h->p, k = h->k, ld = h->ldJ;
    if (!h->stage_U) {
        CES_TRY(dalloc(h, &h->stage_U, p * ld));
        CES_TRY(dalloc(h, &h->stage_G, k * ld));
        CES_TRY(dalloc(h, &h->stage_xi, p * ld));
        CES_TRY(dalloc(h, &h->stage_out, p * ld));
    }
    if (!h->copy_st) {
        CES_CUDA(cudaStreamCreateWithFlags(&h->copy_st, cudaStreamNonBlocking));
        CES_CUDA(cudaEventCreateWithFlags(&h->copy_ev, cudaEventDisableTiming));
        CES_CUDA(cudaEventCreateWithFlags(&h->start_ev, cudaEventDisableTiming));
        CES_CUDA(cudaEventCreateWithFlags(&h->u_ev, cudaEventDisableTiming));
        for (cudaEvent_t& e : h->g_ev) CES_CUDA(cudaEventCreate(&e));          // (timing enabled: the last one closes the rate measurement)
        CES_CUDA(cudaEventCreate(&h->up_begin));
    }
    return CES_OK;
}

static cudaError_t host_h2d(ces_handle_t h, double* dst, const double* src, int64_t rows, cudaStream_t s) {
    const int64_t w = h->cols, ld = h->ldJ;       // host arrays are dense: ld = cols_local
    if (rows < 1 || w < 1) return cudaSuccess;
    if (ld == w) return cudaMemcpyAsync(dst, src, (size_t)rows * w * sizeof(double), cudaMemcpyHostToDevice, s);
    return cudaMemcpy2DAsync(dst, ld * sizeof(double), src, w * sizeof(double), w * sizeof(double), rows, cudaMemcpyHostToDevice, s);
}

// Row chunks of the G upload of a host step: bounds[0..n] (n <= 8 chunks), returns n.  A PURE function of its arguments --
// every rank of a column-sharded step must arrive at the same chunks, because the caller all-reduces the means slice by
// slice: nothing rank-local (measured rates, this rank's column count) may enter when nranks > 1.
//   rho = time of the first-panel GEMM per row of G (2 J_l min(panel, J_l) flop at ~36 TF/s)
//       / time of the upload per row (8 J_l bytes at h2d_gbs; 0 = nominal for the process count, measured on this pool:
//         55 GB/s for 1-2 processes, ~40 for 4, ~21 each when eight upload at once).
// A first chunk of k/32 rows is the only exposed transfer; each following chunk may be rho times the previous one (its
// upload hides behind the previous chunk's GEMM): three chunks at rho ~ 6 (one GPU, 16384-column panel).  When that does
// not reach k within 8 chunks (uploads as slow as the GEMM: eight ranks) the rest is split evenly, so the contraction keeps
// pace with the arrival and only the last seventh remains when the upload ends.  Small shapes: one chunk.
int ces_host_chunk_schedule(int64_t k, int64_t J_local, int64_t panel, int nranks, double h2d_gbs, int64_t* bound /* [9] */) {
    if (!bound || k < 1) return 0;
    bound[0] = 0;
    for (int i = 1; i < 9; ++i) bound[i] = k;
    if (k < 256 || J_local < 2048) return 1;
    const double panel0 = (double)(panel < J_local ? panel : J_local);
    const double t_gemm = 2.0 * (double)J_local * panel0 / 36.0e12;
    double gbs = h2d_gbs;
    if (!(gbs > 1.0)) gbs = nranks <= 2 ? 55.0 : (nranks <= 4 ? 40.0 : 21.0);
    const double t_up = 8.0 * (double)J_local / (gbs * 1e9);
    double rho = 0.9 * t_gemm / t_up;
    if (rho > 8.0) rho = 8.0;
    const int64_t first = round_up(k / 32 > 16 ? k / 32 : 16, 16);
    constexpr int kMaxChunks = 8;
    int n = 1;
    int64_t at = first, size = first;
    bound[1] = first;
    bool fits = false;
    if (rho >= 1.5) {
        while (n < kMaxChunks) {
            size = round_up((int64_t)(size * rho), 16);
            if (at + size >= k || n == kMaxChunks - 1) {
                fits = (at + size >= k) || (k - at) <= (int64_t)(size * 1.2);
                bound[++n] = k;
                at = k;
                break;
            }
            at += size;
            bound[++n] = at;
        }
    }
    if (!fits) {
        const int64_t each = round_up(ceil_div(k - first, kMaxChunks - 1), 16);
        n = 1;
        at = first;
        while (at < k && n < kMaxChunks) { at = at + each < k ? at + each : k; bound[++n] = at; }
        bound[n] = k;
    }
    for (int i = n + 1; i < 9; ++i) bound[i] = k;
    return n;
}

int ces_host_begin(ces_handle_t h, int rule, int formulation, const double* U, const double* G, const double* xi,
                   int* nchunks_out, int64_t* bounds_out /* [9] */) {
    CES_TRY(valid(h, true));
    CES_TRY(check_step(h, "ces_host_begin", rule, std::nullopt, false, formulation, (U && G) || h->cols == 0));
    CES_TRY(host_staging(h));
    const int64_t p = h->p, k = h->k, ld = h->ldJ, w = h->cols;
    // ---- uploads, all on the copy stream, in the order the main stream needs them: G in row chunks (ces_host_chunk_schedule),
    // U, xi.  Row means are per row over the particles, so a row chunk of G can be summed and centred as soon as it has landed,
    // and the D GEMM of the first column panel (own block) contracts over the rows received so far (beta = 1 after the first).
    int64_t* bound = h->hb_bound;
    int nchunk = 1;
    bound[0] = 0;
    for (int i = 1; i < 9; ++i) bound[i] = k;
    if (formulation == CES_FORM_INTERACTION && h->gamma_diag) {
        double gbs = 0.0;                       // several ranks: the nominal rate of the process count (see the schedule)
        if (h->nranks == 1 && h->h2d_gbs > 1.0) gbs = h->h2d_gbs;
        nchunk = ces_host_chunk_schedule(k, h->Jl, h->panel, h->nranks, gbs, bound);
    }
    h->hb_nchunk = nchunk;
    h->hb_formulation = formulation;
    h->hb_have_xi = xi != nullptr;
    mark(h, "host:begin");
    CES_CUDA(cudaEventRecord(h->start_ev, h->st));                // after the previous step's readers of the staging buffers
    CES_CUDA(cudaStreamWaitEvent(h->copy_st, h->start_ev, 0));
    // the rate of the previous call's G upload (its events have completed: that call ended with a synchronisation)
    if (h->hb_timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->up_begin, h->g_ev[h->hb_nchunk_prev - 1]) == cudaSuccess && ms > 0.05f)
            h->h2d_gbs = (double)k * (double)w * 8.0 / (ms * 1e-3) * 1e-9;
        else cudaGetLastError();
    }
    static const char* up_names[8] = {"upload:G0", "upload:G1", "upload:G2", "upload:G3", "upload:G4", "upload:G5", "upload:G6", "upload:G7"};
    CES_CUDA(cudaEventRecord(h->up_begin, h->copy_st));
    for (int c = 0; c < nchunk; ++c) {
        CES_CUDA(host_h2d(h, h->stage_G + bound[c] * ld, G + bound[c] * w, bound[c + 1] - bound[c], h->copy_st));
        CES_CUDA(cudaEventRecord(h->g_ev[c], h->copy_st));
        mark(h, up_names[c], h->copy_st);
    }
    h->hb_timed = w > 0;
    h->hb_nchunk_prev = nchunk;
    CES_CUDA(host_h2d(h, h->stage_U, U, p, h->copy_st));
    CES_CUDA(cudaEventRecord(h->u_ev, h->copy_st));
    mark(h, "upload:U", h->copy_st);
    if (xi) {
        CES_CUDA(host_h2d(h, h->stage_xi, xi, p, h->copy_st));
        CES_CUDA(cudaEventRecord(h->copy_ev, h->copy_st));
        mark(h, "upload:xi", h->copy_st);
    }
    h->last_rule = rule;
    if (nchunks_out) *nchunks_out = nchunk;
    if (bounds_out) for (int i = 0; i < 9; ++i) bounds_out[i] = bound[i];
    return CES_OK;
}

int ces_host_sums_g(ces_handle_t h, int chunk) {
    CES_TRY(valid(h, true));
    if (chunk < 0 || chunk >= h->hb_nchunk) return fail(CES_ERR_INVALID, "ces_host_sums_g: bad chunk%s", "");
    const int64_t r0 = h->hb_bound[chunk], nr = h->hb_bound[chunk + 1] - r0;
    CES_CUDA(cudaStreamWaitEvent(h->st, h->g_ev[chunk], 0));
    if (h->cols == 0) { CES_CUDA(cudaMemsetAsync(h->sums + r0, 0, nr * sizeof(double), h->st)); return CES_OK; }
    return row_sums(h->st, h->stage_G + r0 * h->ldJ, h->ldJ, nr, h->cols, h->sums + r0);
}

int ces_host_interact_chunk(ces_handle_t h, int chunk);

int ces_host_centre_g(ces_handle_t h, int chunk, int interact) {
    CES_TRY(valid(h, true));
    if (chunk < 0 || chunk >= h->hb_nchunk) return fail(CES_ERR_INVALID, "ces_host_centre_g: bad chunk%s", "");
    const int64_t r0 = h->hb_bound[chunk], nr = h->hb_bound[chunk + 1] - r0;
    CES_TRY(centre_g_rows(h, h->stage_G, h->ldJ, r0, nr));
    if (interact) return ces_host_interact_chunk(h, chunk);
    return CES_OK;
}

// Own block, first column panel: contract over the rows of this chunk (no-op with a single chunk: ces_host_interact_own
// then does the whole block).  Chunks must be taken in order.
int ces_host_interact_chunk(ces_handle_t h, int chunk) {
    CES_TRY(valid(h, true));
    if (chunk < 0 || chunk >= h->hb_nchunk) return fail(CES_ERR_INVALID, "ces_host_interact_chunk: bad chunk%s", "");
    const int64_t r0 = h->hb_bound[chunk], nr = h->hb_bound[chunk + 1] - r0;
    if (h->hb_nchunk > 1) {
        // own block, first column panel: contract over the rows received so far
        static const char* ck[8] = {"centred:G0", "centred:G1", "centred:G2", "centred:G3", "centred:G4", "centred:G5", "centred:G6", "centred:G7"};
        static const char* dk[8] = {"D0:chunk0", "D0:chunk1", "D0:chunk2", "D0:chunk3", "D0:chunk4", "D0:chunk5", "D0:chunk6", "D0:chunk7"};
        InteractRange rg;
        rg.c_begin = 0; rg.c_end = h->panel < h->Jl ? h->panel : h->Jl; rg.k_lo = r0; rg.k_hi = r0 + nr;
        rg.do_v = false; rg.reset = (chunk == 0); rg.finish = false;
        mark(h, ck[chunk]);
        // the last chunk applies the rank-one row term, from z = Gamma^-1 c (finish_g recomputes the same z later)
        if (h->nranks == 1 && chunk == h->hb_nchunk - 1) CES_TRY(scale_vector(h->st, h->ginv_diag, h->cvec, h->zvec, h->k));
        CES_TRY(interaction_loops(h, h->W, h->zvec, true, 0, 1, rg));
        mark(h, dk[chunk]);
    }
    return CES_OK;
}

int ces_host_sums_u(ces_handle_t h) {
    CES_TRY(valid(h, true));
    CES_TRY(finish_g(h));
    CES_CUDA(cudaStreamWaitEvent(h->st, h->u_ev, 0));
    if (h->cols == 0) { CES_CUDA(cudaMemsetAsync(h->sums + h->k, 0, h->p * sizeof(double), h->st)); return CES_OK; }
    return row_sums(h->st, h->stage_U, h->ldJ, h->p, h->cols, h->sums + h->k);
}

int ces_host_centre_u(ces_handle_t h) {
    CES_TRY(valid(h, true));
    CES_TRY(centre_u_all(h, h->last_rule, h->stage_U, h->ldJ));
    mark(h, "centred:U+Cuu");
    return CES_OK;
}

// Own block: what is left of it after the chunks of ces_host_centre_g (V of the first panel, the remaining panels), or
// all of it (single chunk).  Also starts chol(C^uu) on the side stream, so C^uu must be final (all-reduced) by now.
int ces_host_interact_own(ces_handle_t h) {
    CES_TRY(valid(h, true));
    const int rule = h->last_rule;
    if (h->hb_formulation == CES_FORM_FACTORED) {
        if (h->nranks != 1) return fail(CES_ERR_STATE, "host steps: the factored formulation is single-GPU here%s", "");
        return interaction_phase(h, rule, CES_FORM_FACTORED);
    }
    CES_TRY(start_cholesky(h, rule));
    const bool whole = (h->nranks == 1);          // single GPU: the own block is the whole interaction
    if (h->hb_nchunk > 1) {
        const int64_t panel0 = h->panel < h->Jl ? h->panel : h->Jl;
        InteractRange rv;                         // V of the first panel, then the remaining panels as usual
        rv.c_begin = 0; rv.c_end = panel0; rv.do_d = false; rv.reset = false; rv.finish = whole && (panel0 >= h->Jl);
        CES_TRY(interaction_loops(h, h->W, h->zvec, true, 0, 1, rv));
        mark(h, "V0");
        if (panel0 < h->Jl) {
            InteractRange rr;
            rr.c_begin = panel0; rr.reset = false; rr.finish = whole;
            CES_TRY(interaction_loops(h, h->W, h->zvec, true, 0, 1, rr));
            mark(h, "panels:rest");
        }
        return CES_OK;
    }
    InteractRange all;
    all.finish = whole;
    return interaction_loops(h, h->W, h->zvec, true, 0, 1, all);
}

int ces_host_update(ces_handle_t h, int ts_kind, double fixed_h, double* Uout_host, double* hk_host, double* metrics_host) {
    CES_TRY(valid(h, true));
    if (!Uout_host && h->cols > 0) return fail(CES_ERR_INVALID, "ces_host_update: null output%s", "");
    if (h->hb_have_xi) CES_CUDA(cudaStreamWaitEvent(h->st, h->copy_ev, 0));
    // phase 4 downloads U_next (in column chunks, overlapped) and ends with a synchronisation (status + scalars)
    h->pending_out = h->cols > 0 ? Uout_host : nullptr;
    h->pending_rows = h->p;
    const int s4 = ces_phase4_update(h, h->last_rule, ts_kind, fixed_h, h->stage_U, h->ldJ, h->hb_have_xi ? h->stage_xi : nullptr,
                                     h->ldJ, h->stage_out, h->ldJ, hk_host, metrics_host);
    h->pending_out = nullptr;
    return s4;
}

int ces_step_host(ces_handle_t h, int rule, int ts_kind, double fixed_h, double switch_, int formulation, const double* U,
                  const double* G, const double* xi, double* Uout, double* hk_host, double* metrics_host) {
    CES_TRY(valid(h, true));
    if (h->nranks != 1) return fail(CES_ERR_STATE, "ces_step_host is single-GPU; use the ces_host_* pieces with nranks > 1%s", "");
    CES_TRY(check_step(h, "ces_step_host", rule, ts_kind, false, formulation, U && G && Uout && (xi || !needs_xi(h, rule))));
    const int64_t p = h->p, k = h->k, ld = h->ldJ;
    if (small_path(h, formulation)) {
        // tiny problems keep everything on one stream -- extra streams and events would cost more than the copies
        CES_TRY(host_staging(h));
        if (xi && !ensemble_noise(h)) CES_CUDA(host_h2d(h, h->stage_xi, xi, p, h->st));
        CES_CUDA(host_h2d(h, h->stage_U, U, p, h->st));
        CES_CUDA(host_h2d(h, h->stage_G, G, k, h->st));
        h->pending_out = Uout;
        h->pending_rows = p;
        const int s1 = ces_step(h, rule, ts_kind, fixed_h, switch_, formulation, h->stage_U, ld, h->stage_G, ld,
                                xi ? h->stage_xi : nullptr, ld, h->stage_out, ld, hk_host, metrics_host);
        h->pending_out = nullptr;
        return s1;
    }
    int nchunk = 1;
    CES_TRY(ces_host_begin(h, rule, formulation, U, G, xi, &nchunk, nullptr));
    for (int c = 0; c < nchunk; ++c) {
        CES_TRY(ces_host_sums_g(h, c));
        CES_TRY(ces_host_centre_g(h, c, 1));
    }
    CES_TRY(ces_host_sums_u(h));
    CES_TRY(ces_host_centre_u(h));
    CES_TRY(ces_host_interact_own(h));
    if (rule == CES_RULE_ALDI_CONSTANT) CES_TRY(ces_phase4a_drift(h, switch_));
    return ces_host_update(h, ts_kind, fixed_h, Uout, hk_host, metrics_host);
}

int ces_set_pending_output(ces_handle_t h, double* host_out) {
    CES_TRY(valid(h, true));
    h->pending_out = host_out;
    h->pending_rows = h->p;
    return CES_OK;
}

// The whole run loop of a small single-GPU problem in one launch (csrc/small.cu: small_run_kernel).
int ces_small_run(ces_handle_t h, int rule, int ts_kind, double fixed_h, double switch_, int map_kind, const double* A_dev,
                  int64_t lda, const double* b_dev, const double* params_host, const double* U0_host, const double* xi_host,
                  uint64_t seed, uint64_t step0, int64_t T, double t0, int have_t0, double t_tol, double* Utrace_host,
                  double* Gtrace_host, double* S_host, double* t_host, int64_t* nsteps_host) {
    CES_TRY(valid(h, true));
    if (h->nranks != 1) return fail(CES_ERR_STATE, "ces_small_run is single-GPU%s", "");
    const int64_t p = h->p, k = h->k, J = h->Jl;
    if (!small_step_eligible(p, k, J)) return fail(CES_ERR_INVALID, "ces_small_run: the problem is too large for the single-CTA path%s", "");
    CES_TRY(check_step(h, "ces_small_run", rule, ts_kind, false, std::nullopt, true, !(xi_host && ensemble_noise(h))));
    if (T < 1 || !U0_host || !Utrace_host || !Gtrace_host || !S_host || !t_host || !nsteps_host)
        return fail(CES_ERR_INVALID, "ces_small_run: bad argument%s", "");
    if (map_kind < CES_MAP_LINEAL || map_kind > CES_MAP_BANANA) return fail(CES_ERR_INVALID, "ces_small_run: unknown map kind%s", "");
    if ((map_kind == CES_MAP_LINEAL || map_kind == CES_MAP_LINEAL_LOG) ? !A_dev : (!params_host || p != 2 || k != 2))
        return fail(CES_ERR_INVALID, "ces_small_run: the map needs A (lineal) or two parameters with p = k = 2%s", "");
    cudaStream_t st = h->st;
    const int64_t nu = (T + 1) * p * J, ng = (T + 1) * k * J, nx = needs_xi(h, rule) ? T * p * J : 0;
    const int64_t total = nu + ng + nx + T * S_COUNT + T + 2;
    if (h->run_ws_len < total) {
        if (h->run_ws) cudaFree(h->run_ws);
        h->run_ws = nullptr; h->run_ws_len = 0;
        if (cudaMalloc(&h->run_ws, (size_t)total * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return fail(CES_ERR_NOMEM, "ces_small_run: workspace allocation failed%s", ""); }
        h->run_ws_len = total;
    }
    double* Ut = h->run_ws;
    double* Gt = Ut + nu;
    double* Xi = Gt + ng;
    double* Sall = Xi + nx;
    double* tv = Sall + T * S_COUNT;
    int* nst = reinterpret_cast<int*>(tv + T);
    CES_CUDA(cudaMemcpyAsync(Ut, U0_host, (size_t)p * J * sizeof(double), cudaMemcpyHostToDevice, st));
    if (nx > 0) {
        if (xi_host) CES_CUDA(cudaMemcpyAsync(Xi, xi_host, (size_t)nx * sizeof(double), cudaMemcpyHostToDevice, st));
        else for (int64_t it = 0; it < T; ++it) CES_TRY(fill_normal(st, Xi + it * p * J, J, p, J, 0, seed, step0 + (uint64_t)it));
    }
    SmallStepCall c = small_call(h, rule, ts_kind, fixed_h, switch_);   // operands: the run's own buffers
    c.ldu = c.ldg = c.ldo = J;
    if (!c.ensemble) c.ldxi = J;
    SmallRunCall rc;
    rc.T = T; rc.map_kind = map_kind; rc.have_t0 = have_t0; rc.t0 = t0; rc.t_tol = t_tol;
    rc.A = A_dev; rc.lda = lda; rc.b = b_dev;
    rc.par0 = params_host ? params_host[0] : 0.0; rc.par1 = params_host ? params_host[1] : 0.0;
    rc.Utrace = Ut; rc.Gtrace = Gt; rc.Xi = nx > 0 ? Xi : nullptr; rc.Sall = Sall; rc.tvec = tv; rc.nsteps = nst;
    h->last_rule = rule;
    CES_TRY(small_run(st, c, rc));
    int n = 0;
    CES_CUDA(cudaMemcpyAsync(&n, nst, sizeof(int), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaStreamSynchronize(st));
    if (n < 1 || n > T) return fail(CES_ERR_CUDA, "ces_small_run: kernel failure%s", "");
    CES_CUDA(cudaMemcpyAsync(Utrace_host, Ut, (size_t)(n + 1) * p * J * sizeof(double), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaMemcpyAsync(Gtrace_host, Gt, (size_t)(n + 1) * k * J * sizeof(double), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaMemcpyAsync(S_host, Sall, (size_t)n * S_COUNT * sizeof(double), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaMemcpyAsync(t_host, tv, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaStreamSynchronize(st));
    *nsteps_host = n;
    const double info = S_host[(size_t)(n - 1) * S_COUNT + S_INFO];
    if (info != 0.0) return fail(CES_ERR_NOT_SPD, "%s: matrix is not positive definite (pivot %lld)", "cov(U)", (long long)info);
    return CES_OK;
}

int ces_forward_map(ces_handle_t h, int map_kind, const double* A, int64_t lda, const double* b, const double* params,
                    const double* U, int64_t ldu, double* G, int64_t ldg) {
    CES_TRY(valid(h, false));
    if (!U || !G) return fail(CES_ERR_INVALID, "ces_forward_map: null ensemble%s", "");
    const int64_t p = h->p, k = h->k, cols = h->cols, ld = h->ldJ;
    if (cols == 0) return CES_OK;
    cudaStream_t st = h->st;
    if (map_kind == CES_MAP_LINEAL || map_kind == CES_MAP_LINEAL_LOG) {
        if (!A) return fail(CES_ERR_INVALID, "ces_forward_map: lineal needs A%s", "");
        const double* B = U;
        int64_t ldb = ldu;
        const bool misaligned = ((reinterpret_cast<uintptr_t>(U) & 15) != 0) || (ldu & 1);
        if (map_kind == CES_MAP_LINEAL_LOG || misaligned) {
            if (!h->expU) { CES_TRY(dalloc(h, &h->expU, p * ld)); }
            if (map_kind == CES_MAP_LINEAL_LOG) CES_TRY(exp_map(st, U, ldu, p, cols, h->expU, ld));
            else CES_TRY(pad_copy(st, U, ldu, p, cols, h->expU, ld));
            B = h->expU; ldb = ld;
        }
        GemmCall g;
        g.a_mode = A_MK; g.b_mode = B_KN;
        g.M = (int)k; g.N = (int)cols; g.K = (int)p;
        g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = G; g.ldc = ldg;
        CES_TRY(gemm(st, g));
        if (b) CES_TRY(add_col_vector(st, G, ldg, k, cols, b, 1.0, nullptr));
        return CES_OK;
    }
    if (map_kind == CES_MAP_ELLIPTIC || map_kind == CES_MAP_BANANA) {
        if (p != 2 || k != 2 || !params) return fail(CES_ERR_INVALID, "ces_forward_map: elliptic/banana need p = k = 2 and params%s", "");
        if (map_kind == CES_MAP_ELLIPTIC) return elliptic_map(st, U, ldu, cols, params[0], params[1], G, ldg);
        return banana_map(st, U, ldu, cols, params[0], params[1], G, ldg);
    }
    return fail(CES_ERR_INVALID, "ces_forward_map: unknown map kind %s%lld", "", map_kind);
}

// ---- gathers over peer memory (one process per GPU, all on one NVSwitch domain) ---------------------------------
// Every rank exports its E_all / Ut_all allocations as CUDA IPC handles, the host exchanges the 64-byte handles once
// (torch.distributed all_gather_object) and every rank maps its peers' buffers.  Per step, after the collective that
// follows the centring (the all-reduce of C^uu: when it has completed on this rank's stream, every peer has written
// its own E / U~ block), ces_peer_gather queues one device-to-device copy per peer and buffer on a side stream --
// copy engines over NVLink, no SM is taken from the own-block GEMMs that run meanwhile, unlike an NCCL all-gather --
// and ces_peer_gather_wait makes the main stream wait for them.  A peer overwrites its block only in the next step's
// centring, which is ordered after the all-reduce of the step scalars, which every rank enters only after its GEMMs
// on the pulled blocks: no further handshake is needed.
int ces_ipc_export(ces_handle_t h, void* e_handle, void* ut_handle) {
    CES_TRY(valid(h, false));
    if (h->forward_only || !e_handle || !ut_handle) return fail(CES_ERR_INVALID, "ces_ipc_export: bad argument%s", "");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CES_CUDA(cudaIpcGetMemHandle(static_cast<cudaIpcMemHandle_t*>(e_handle), h->E_all));
    CES_CUDA(cudaIpcGetMemHandle(static_cast<cudaIpcMemHandle_t*>(ut_handle), h->Ut_all));
    return CES_OK;
}

int ces_ipc_import(ces_handle_t h, int peer, const void* e_handle, const void* ut_handle) {
    CES_TRY(valid(h, false));
    if (h->forward_only || peer < 0 || peer >= h->nranks || peer == h->rank || !e_handle || !ut_handle)
        return fail(CES_ERR_INVALID, "ces_ipc_import: bad argument%s", "");
    if (h->peer_E.empty()) { h->peer_E.assign(h->nranks, nullptr); h->peer_Ut.assign(h->nranks, nullptr); }
    void *pe = nullptr, *pu = nullptr;
    cudaIpcMemHandle_t he, hu;
    memcpy(&he, e_handle, 64);
    memcpy(&hu, ut_handle, 64);
    CES_CUDA(cudaIpcOpenMemHandle(&pe, he, cudaIpcMemLazyEnablePeerAccess));
    CES_CUDA(cudaIpcOpenMemHandle(&pu, hu, cudaIpcMemLazyEnablePeerAccess));
    h->peer_E[peer] = static_cast<double*>(pe);
    h->peer_Ut[peer] = static_cast<double*>(pu);
    return CES_OK;
}

int ces_peer_gather(ces_handle_t h) {
    CES_TRY(valid(h, true));
    if (h->nranks < 2) return CES_OK;
    if ((int)h->peer_E.size() != h->nranks) return fail(CES_ERR_STATE, "ces_peer_gather: peers were not imported%s", "");
    if (!h->gather_st) {
        CES_CUDA(cudaStreamCreateWithFlags(&h->gather_st, cudaStreamNonBlocking));
        CES_CUDA(cudaEventCreateWithFlags(&h->gather_go, cudaEventDisableTiming));
        CES_CUDA(cudaEventCreateWithFlags(&h->gather_done, cudaEventDisableTiming));
    }
    CES_CUDA(cudaEventRecord(h->gather_go, h->st));
    CES_CUDA(cudaStreamWaitEvent(h->gather_st, h->gather_go, 0));
    const size_t eb = (size_t)h->k * h->ldJ, ub = (size_t)h->p * h->ldJ;
    // rotated order: at any moment every peer is read by a different rank; E first (the D GEMMs need it first)
    for (int pass = 0; pass < 2; ++pass)
        for (int i = 1; i < h->nranks; ++i) {
            const int s = (h->rank + i) % h->nranks;
            if (!h->peer_E[s] || !h->peer_Ut[s]) return fail(CES_ERR_STATE, "ces_peer_gather: peer %s%lld was not imported", "", s);
            if (pass == 0) CES_CUDA(cudaMemcpyAsync(h->E_all + s * eb, h->peer_E[s] + s * eb, eb * sizeof(double), cudaMemcpyDeviceToDevice, h->gather_st));
            else CES_CUDA(cudaMemcpyAsync(h->Ut_all + s * ub, h->peer_Ut[s] + s * ub, ub * sizeof(double), cudaMemcpyDeviceToDevice, h->gather_st));
        }
    CES_CUDA(cudaEventRecord(h->gather_done, h->gather_st));
    mark(h, "peer_gather:done", h->gather_st);
    return CES_OK;
}

int ces_peer_gather_wait(ces_handle_t h) {
    CES_TRY(valid(h, true));
    if (h->nranks < 2 || !h->gather_done) return CES_OK;
    CES_CUDA(cudaStreamWaitEvent(h->st, h->gather_done, 0));
    return CES_OK;
}

int ces_timeline_enable(ces_handle_t h, int on) {
    CES_TRY(valid(h, false));
    for (auto& m : h->marks) h->mark_pool.push_back(m.second);
    h->marks.clear();
    h->timeline = on != 0;
    return CES_OK;
}

int ces_timeline_mark(ces_handle_t h, const char* name) {
    CES_TRY(valid(h, false));
    mark(h, name ? name : "");
    return CES_OK;
}

int ces_timeline_read(ces_handle_t h, char* names, int64_t names_cap, double* ms, int64_t ms_cap, int64_t* count) {
    CES_TRY(valid(h, false));
    CES_CUDA(cudaDeviceSynchronize());
    int64_t n = 0;
    size_t used = 0;
    for (auto& m : h->marks) {
        if (n >= ms_cap) break;
        float t = 0.f;
        if (cudaEventElapsedTime(&t, h->marks[0].second, m.second) != cudaSuccess) { cudaGetLastError(); t = -1.f; }
        if (ms) ms[n] = t;
        if (names && used + m.first.size() + 2 <= (size_t)names_cap) {
            memcpy(names + used, m.first.c_str(), m.first.size());
            used += m.first.size();
            names[used++] = '\n';
            names[used] = 0;
        }
        ++n;
    }
    if (count) *count = n;
    for (auto& m : h->marks) h->mark_pool.push_back(m.second);
    h->marks.clear();
    return CES_OK;
}

int ces_profile_enable(ces_handle_t h, int on) {
    CES_TRY(valid(h, false));
    h->profile = on != 0;
    h->ev_used = 0;
    h->prof_flops = 0.0;
    return CES_OK;
}

int ces_profile_read(ces_handle_t h, double* gemm_d_ms, int64_t* launches, double* flops) {
    CES_TRY(valid(h, false));
    CES_CUDA(cudaStreamSynchronize(h->st));
    double total = 0.0;
    for (size_t i = 0; i + 1 < h->ev_used; i += 2) {
        float ms = 0.f;
        CES_CUDA(cudaEventElapsedTime(&ms, h->ev_pool[i], h->ev_pool[i + 1]));
        total += ms;
    }
    if (gemm_d_ms) *gemm_d_ms = total;
    if (launches) *launches = (int64_t)(h->ev_used / 2);
    if (flops) *flops = h->prof_flops;
    h->ev_used = 0;
    h->prof_flops = 0.0;
    return CES_OK;
}

int ces_buffer(ces_handle_t h, const char* name, double** ptr, int64_t* rows, int64_t* cols, int64_t* ld) {
    CES_TRY(valid(h, false));
    if (!name || !ptr) return fail(CES_ERR_INVALID, "ces_buffer: null argument%s", "");
    const std::string n(name);
    double* q = nullptr;
    int64_t r = 0, c = 0, l = 0;
    if (n == "sums") { q = h->sums; r = 1; c = h->k + h->p; l = c; }
    else if (n == "cuu") { q = h->Cuu; r = h->p; c = h->ldp; l = h->ldp; }
    else if (n == "chol") { q = h->L; r = h->p; c = h->ldp; l = h->ldp; }
    else if (n == "e_all") { q = h->E_all; r = h->nranks * h->k; c = h->ldJ; l = h->ldJ; }
    else if (n == "ut_all") { q = h->Ut_all; r = h->nranks * h->p; c = h->ldJ; l = h->ldJ; }
    else if (n == "scalars") { q = h->S; r = 1; c = S_COUNT; l = S_COUNT; }
    else if (n == "w") { q = h->W; r = h->k; c = h->ldJ; l = h->ldJ; }
    else if (n == "v") { q = h->V; r = h->p; c = h->ldJ; l = h->ldJ; }
    else if (n == "z") { q = h->Z; r = h->p; c = h->ldJ; l = h->ldJ; }
    else if (n == "p1") { q = h->P1; r = h->p; c = h->ldk; l = h->ldk; }
    else if (n == "gram_e") { q = h->GE; r = h->k; c = h->ldk; l = h->ldk; }
    else if (n == "gram_w") { q = h->GW; r = h->k; c = h->ldk; l = h->ldk; }
    else if (n == "cpp") { q = h->Cpp; r = h->k; c = h->ldk; l = h->ldk; }
    else if (n == "d_panel") { q = h->D; r = h->ldJ; c = h->ldD; l = h->ldD; }
    else return fail(CES_ERR_INVALID, "ces_buffer: unknown buffer '%s'", name);
    *ptr = q;
    if (rows) *rows = r;
    if (cols) *cols = c;
    if (ld) *ld = l;
    return CES_OK;
}

int ces_set_noise(ces_handle_t h, int kind, uint64_t seed, uint64_t step, const double* xi_dev, int64_t ldxi) {
    // arguments that need no handle first
    if (kind != CES_NOISE_CHOLESKY && kind != CES_NOISE_ENSEMBLE) return fail(CES_ERR_INVALID, "ces_set_noise: unknown noise kind %s%lld", "", kind);
    if (kind == CES_NOISE_ENSEMBLE && xi_dev && (((reinterpret_cast<uintptr_t>(xi_dev) & 15) != 0) || (ldxi & 1) || ldxi < 1))
        return fail(CES_ERR_ALIGN, "ces_set_noise: xi needs a 16-byte aligned base and an even leading dimension%s", "");
    CES_TRY(valid(h, false));
    if (kind == CES_NOISE_ENSEMBLE && h->Jg < 2) return fail(CES_ERR_INVALID, "ces_set_noise: ensemble noise needs J >= 2%s", "");
    if (kind == CES_NOISE_ENSEMBLE && xi_dev && ldxi < h->cols)
        return fail(CES_ERR_ALIGN, "ces_set_noise: leading dimension of xi below the local column count%s", "");
    h->noise_kind = kind;
    h->noise_seed = seed;
    h->noise_step = step;
    h->noise_xi = kind == CES_NOISE_ENSEMBLE ? xi_dev : nullptr;
    h->noise_ldxi = kind == CES_NOISE_ENSEMBLE && xi_dev ? ldxi : 0;
    return CES_OK;
}

int ces_fill_ensemble_noise(void* stream, uint64_t seed, uint64_t step, double* X, int64_t ld, int64_t rows, int64_t cols,
                            int64_t row_offset, int64_t col_offset) {
    if (!X || rows < 0 || cols < 0 || ld < cols || row_offset < 0 || col_offset < 0)
        return fail(CES_ERR_INVALID, "ces_fill_ensemble_noise: bad argument%s", "");
    return fill_ensemble_noise(static_cast<cudaStream_t>(stream), X, ld, rows, cols, row_offset, col_offset, seed, step);
}

int ces_fill_normal(void* stream, uint64_t seed, uint64_t step, double* X, int64_t ld, int64_t rows, int64_t cols,
                    int64_t col_offset) {
    if (!X || ld < cols) return fail(CES_ERR_INVALID, "ces_fill_normal: bad argument%s", "");
    return fill_normal(static_cast<cudaStream_t>(stream), X, ld, rows, cols, col_offset, seed, step);
}

int ces_frobenius(void* stream, const double* X, int64_t ld, int64_t rows, int64_t cols, double* out_host) {
    if (!X || !out_host || rows < 1 || cols < 1 || ld < cols) return fail(CES_ERR_INVALID, "ces_frobenius: bad argument%s", "");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* part = nullptr;
    CES_CUDA(cudaMalloc(&part, (size_t)(rows + 1) * sizeof(double)));
    int s = row_sumsq(st, X, ld, rows, cols, part);
    if (s == CES_OK) s = sum_vector(st, part, rows, part + rows);
    double v = 0.0;
    if (s == CES_OK && cudaMemcpyAsync(&v, part + rows, sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess) s = CES_ERR_CUDA;
    if (cudaStreamSynchronize(st) != cudaSuccess && s == CES_OK) s = fail(CES_ERR_CUDA, "ces_frobenius: kernel failure%s", "");
    cudaFree(part);
    if (s == CES_OK) *out_host = sqrt(v);
    return s;
}

// A leading dimension below the stored row width would make consecutive rows overlap.
static bool gemm_ld_ok(int a_mode, int b_mode, int64_t M, int64_t N, int64_t K, int64_t lda, int64_t ldb, int64_t ldc) {
    return lda >= (a_mode == A_MK ? K : M) && ldb >= (b_mode == B_KN ? N : K) && ldc >= N;
}

int ces_gemm(void* stream, int a_mode, int b_mode, int64_t M, int64_t N, int64_t K, double alpha, const double* A, int64_t lda,
             const double* B, int64_t ldb, double beta, double* C, int64_t ldc) {
    if (a_mode < 0 || a_mode > 1 || b_mode < 0 || b_mode > 1 || M > (1ll << 30) || N > (1ll << 30) || K > (1ll << 30))
        return fail(CES_ERR_INVALID, "ces_gemm: bad mode or size%s", "");
    if (!gemm_ld_ok(a_mode, b_mode, M, N, K, lda, ldb, ldc))
        return fail(CES_ERR_INVALID, "ces_gemm: leading dimension smaller than the operand's stored row%s", "");
    GemmCall g;
    g.a_mode = a_mode; g.b_mode = b_mode;
    g.M = (int)M; g.N = (int)N; g.K = (int)K;
    g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc;
    g.alpha = alpha; g.beta = beta;
    return gemm(static_cast<cudaStream_t>(stream), g);
}

int ces_gemm_ex(void* stream, const ces_gemm_desc* d) {
    if (!d || d->struct_size != (int64_t)sizeof(ces_gemm_desc))
        return fail(CES_ERR_INVALID, "ces_gemm_ex: null descriptor or struct_size != sizeof(ces_gemm_desc)%s", "");
    const int64_t lim = 1ll << 30;
    if (d->a_mode < 0 || d->a_mode > 1 || d->b_mode < 0 || d->b_mode > 1 || d->M < 1 || d->N < 1 || d->K < 1 || d->M > lim ||
        d->N > lim || d->K > lim || d->batch < 1 || d->batch > 65535 || d->a_batch_rows < 0 || d->b_batch_rows < 0 ||
        d->a_batch_rows > lim || d->b_batch_rows > lim || d->c_batch_elems < 0 || d->splits < 0 || d->splits > 65535 || d->group_m < 0 ||
        (d->flags & ~(GEMM_A_LOWER_TRI | GEMM_C_LOWER_ONLY | GEMM_B_UPPER_TRI | GEMM_C_LOWER_TRAP)) != 0)
        return fail(CES_ERR_INVALID, "ces_gemm_ex: bad mode, size, batch or flags%s", "");
    if (!gemm_ld_ok(d->a_mode, d->b_mode, d->M, d->N, d->K, d->lda, d->ldb, d->ldc))
        return fail(CES_ERR_INVALID, "ces_gemm_ex: leading dimension smaller than the operand's stored row%s", "");
    // capacities: the planes the kernel writes into the workspace and the partial slots of every tile of every problem
    const int64_t kb = ceil_div(d->K, GEMM_BK);
    const int64_t planes = d->batch > 1 ? d->batch : (d->splits > 1 ? (d->splits < kb ? d->splits : kb) : 1);
    if (d->splitk_ws && planes * d->M * d->N > d->splitk_ws_elems)
        return fail(CES_ERR_INVALID, "ces_gemm_ex: workspace smaller than (splits or batch) * M * N%s", "");
    const int64_t tiles = (d->flags & GEMM_C_LOWER_TRAP) && d->M >= d->N ? gemm_trap_tiles((int)d->M, (int)d->N)
                                                                           : (int64_t)gemm_tiles((int)d->M, (int)d->N);
    if (d->ssq_partials && tiles * d->batch > d->ssq_partials_elems)
        return fail(CES_ERR_INVALID, "ces_gemm_ex: partials buffer smaller than the launched tiles * batch%s", "");
    GemmCall g;
    g.a_mode = d->a_mode; g.b_mode = d->b_mode;
    g.M = (int)d->M; g.N = (int)d->N; g.K = (int)d->K;
    g.A = d->A; g.lda = d->lda; g.B = d->B; g.ldb = d->ldb; g.C = d->C; g.ldc = d->ldc;
    g.alpha = d->alpha; g.beta = d->beta; g.alpha_dev = d->alpha_dev;
    g.flags = d->flags; g.group_m = d->group_m;
    g.ssq_partials = d->ssq_partials;
    g.splits = d->splits; g.splitk_ws = d->splitk_ws; g.diag_add = d->diag_add;
    g.batch = d->batch; g.a_batch_rows = d->a_batch_rows; g.b_batch_rows = d->b_batch_rows; g.c_batch_elems = d->c_batch_elems;
    g.wave_ctas = d->wave_ctas; g.serpentine = d->serpentine;
    g.row_vec = d->row_vec;
    return gemm(static_cast<cudaStream_t>(stream), g);
}

int ces_potrf(void* stream, double* A, int64_t ld, int64_t n) {
    if (!A || n < 1 || ld < n) return fail(CES_ERR_INVALID, "ces_potrf: bad argument%s", "");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* Linv = nullptr;
    int* info = nullptr;
    CES_CUDA(cudaMalloc(&Linv, (size_t)round_up(n, CHOL_NB) * kLinvLd * sizeof(double)));
    if (cudaMalloc(&info, sizeof(int)) != cudaSuccess) { cudaFree(Linv); return fail(CES_ERR_NOMEM, "cudaMalloc failed%s", ""); }
    cudaMemsetAsync(info, 0, sizeof(int), st);
    int s = potrf_lower(st, A, ld, n, Linv, kLinvLd, info);
    int hinfo = 0;
    if (s == CES_OK && cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess) s = CES_ERR_CUDA;
    if (cudaStreamSynchronize(st) != cudaSuccess && s == CES_OK) s = fail(CES_ERR_CUDA, "ces_potrf: kernel failure%s", "");
    cudaFree(Linv);
    cudaFree(info);
    if (s == CES_OK && hinfo != 0) return fail(CES_ERR_NOT_SPD, "ces_potrf: matrix is not positive definite (pivot %s%lld)", "", hinfo);
    return s;
}

int ces_posv(void* stream, double* A, int64_t lda, int64_t n, double* B, int64_t ldb, int64_t nrhs) {
    if (!A || !B || n < 1 || nrhs < 1 || lda < n || ldb < nrhs) return fail(CES_ERR_INVALID, "ces_posv: bad argument%s", "");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* Linv = nullptr;
    int* info = nullptr;
    CES_CUDA(cudaMalloc(&Linv, (size_t)round_up(n, CHOL_NB) * kLinvLd * sizeof(double)));
    if (cudaMalloc(&info, sizeof(int)) != cudaSuccess) { cudaFree(Linv); return fail(CES_ERR_NOMEM, "cudaMalloc failed%s", ""); }
    cudaMemsetAsync(info, 0, sizeof(int), st);
    int s = potrf_lower(st, A, lda, n, Linv, kLinvLd, info);
    int hinfo = 0;
    if (s == CES_OK && cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess) s = CES_ERR_CUDA;
    if (s == CES_OK && cudaStreamSynchronize(st) != cudaSuccess) s = fail(CES_ERR_CUDA, "ces_posv: kernel failure%s", "");
    if (s == CES_OK && hinfo != 0) s = fail(CES_ERR_NOT_SPD, "ces_posv: matrix is not positive definite (pivot %s%lld)", "", hinfo);
    if (s == CES_OK) s = trsm_lower(st, A, lda, n, Linv, kLinvLd, B, ldb, nrhs, false);
    if (s == CES_OK) s = trsm_lower(st, A, lda, n, Linv, kLinvLd, B, ldb, nrhs, true);
    if (cudaStreamSynchronize(st) != cudaSuccess && s == CES_OK) s = fail(CES_ERR_CUDA, "ces_posv: kernel failure%s", "");
    cudaFree(Linv);
    cudaFree(info);
    return s;
}

int ces_potri(void* stream, double* A, int64_t ld, int64_t n, double* Ainv, int64_t ldo) {
    if (!A || !Ainv || n < 1 || ld < n || ldo < n) return fail(CES_ERR_INVALID, "ces_potri: bad argument%s", "");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double* Linv = nullptr;
    int* info = nullptr;
    CES_CUDA(cudaMalloc(&Linv, (size_t)round_up(n, CHOL_NB) * kLinvLd * sizeof(double)));
    if (cudaMalloc(&info, sizeof(int)) != cudaSuccess) { cudaFree(Linv); return fail(CES_ERR_NOMEM, "cudaMalloc failed%s", ""); }
    cudaMemsetAsync(info, 0, sizeof(int), st);
    int s = potrf_lower(st, A, ld, n, Linv, kLinvLd, info);
    int hinfo = 0;
    if (s == CES_OK && cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess) s = CES_ERR_CUDA;
    if (s == CES_OK && cudaStreamSynchronize(st) != cudaSuccess) s = fail(CES_ERR_CUDA, "ces_potri: kernel failure%s", "");
    if (s == CES_OK && hinfo != 0) s = fail(CES_ERR_NOT_SPD, "ces_potri: matrix is not positive definite (pivot %s%lld)", "", hinfo);
    if (s == CES_OK) s = spd_inverse_from_factor(st, A, ld, n, Linv, kLinvLd, Ainv, ldo);
    if (cudaStreamSynchronize(st) != cudaSuccess && s == CES_OK) s = fail(CES_ERR_CUDA, "ces_potri: kernel failure%s", "");
    cudaFree(Linv);
    cudaFree(info);
    return s;
}

}  // extern "C"
