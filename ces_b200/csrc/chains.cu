// Host side of the chain plumbing shared by the Metropolis-Hastings samplers (chains.cuh).
#include <climits>
#include "chains.cuh"

namespace ces {

int chain_check(const ChainHost& h) {
    if (h.n_mcmc < 1 || h.n_mcmc >= INT_MAX || h.n_chains < 1 || h.n_chains > (1 << 24) || !h.y || !h.scales || !h.start ||
        !h.phi_point || !h.samples || !h.accepted || (!h.pcn && (!h.mu || !h.Pinv)) || (h.mt_state && !h.mt_gauss))
        return fail(CES_ERR_INVALID, "%s: needs 1 <= n_mcmc < 2^31 - 1, 1 <= n_chains <= 2^24 and non-null arguments", h.who);
    return CES_OK;
}

ChainRun::~ChainRun() {
    if (!base_) return;
    cudaStreamSynchronize(st);         // nothing may still use the arena (also after a failed enqueue)
    cudaFree(base_);
}

// samples first: everything after them is zeroed by allocate()
void ChainRun::place() {
    used_ = 0;
    samples = take((size_t)h.n_chains * (h.n_mcmc + 1) * p);
    zero_from_ = used_;
    mt = put(h.mt_state, 626);
    mt_gauss = put(h.mt_state ? h.mt_gauss : nullptr, 1);
    accepted = take<int>(h.n_chains);
}

int ChainRun::allocate() {
    if ((double)h.n_chains * (double)(h.n_mcmc + 1) * p * sizeof(double) > 4e18)
        return fail(CES_ERR_NOMEM, "%s: the samples buffer is too large", h.who);
    if (cudaMalloc(&base_, used_) != cudaSuccess) {
        base_ = nullptr;
        cudaGetLastError();
        return fail(CES_ERR_NOMEM, "%s: allocation failed", h.who);
    }
    if (cudaMemsetAsync(base_ + zero_from_, 0, used_ - zero_from_, st) != cudaSuccess)
        return fail(CES_ERR_CUDA, "%s: upload failed", h.who);
    return CES_OK;
}

double* ChainRun::put2d(const double* src, int64_t rows, int64_t cols, int64_t pitch) {
    double* d = take((size_t)rows * pitch);
    if (base_ && src && err_ == cudaSuccess)
        err_ = cudaMemcpy2DAsync(d, pitch * sizeof(double), src, cols * sizeof(double), cols * sizeof(double), rows,
                                 cudaMemcpyHostToDevice, st);
    return d;
}

double* ChainRun::put_columns(const double* src, int64_t ld) {
    if (!base_) return take((size_t)p * ld);
    columns_.assign((size_t)p * ld, 0.0);
    for (int64_t c = 0; c < h.n_chains; ++c)
        for (int d = 0; d < p; ++d) columns_[(size_t)d * ld + c] = src[(size_t)c * p + d];
    return put(columns_.data(), columns_.size());
}

int ChainRun::copy_back() {
    CES_CUDA(cudaMemcpyAsync(h.samples, samples, (size_t)h.n_chains * (h.n_mcmc + 1) * p * sizeof(double),
                             cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaMemcpyAsync(h.accepted, accepted, (size_t)h.n_chains * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (h.mt_state) {
        CES_CUDA(cudaMemcpyAsync(h.mt_state, mt, 626 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        CES_CUDA(cudaMemcpyAsync(h.mt_gauss, mt_gauss, sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CES_CUDA(cudaStreamSynchronize(st));
    return CES_OK;
}

ChainState chain_state(ChainRun& run, int64_t ld) {
    const ChainHost& h = run.h;
    const int p = run.p;
    ChainState a;
    a.p = p; a.n_mcmc = (int)h.n_mcmc; a.n_chains = (int)h.n_chains; a.use_mt = h.mt_state != nullptr;
    a.ld = ld;
    a.cur = run.take((size_t)p * ld);
    a.prop = run.put_columns(h.phi_point, ld);
    a.u = run.take(ld);
    a.phi_cur = run.take(ld);
    a.start = run.put(h.start, (size_t)h.n_chains * p);
    a.samples = run.samples;
    a.accepted = run.accepted;
    a.mt = run.mt;
    a.mt_gauss = run.mt_gauss;
    a.seed = h.seed;
    return a;
}

}  // namespace ces
