// Chain plumbing shared by the Metropolis-Hastings samplers: ces_mcmc_model_mh (mcmc.cu, one warp per chain), ces_gp_mh
// (emulate.cu) and ces_darcy_mh (darcy_mh.cu), the last two stepping all chains in lockstep.  Lockstep chains share their
// state (ChainState) and their init / accept kernels, templated on a functor phi(a, c): Phi of chain c at a.prop.
#pragma once
#include <vector>
#include "kernels.h"

namespace ces {

// The arguments of every sampler entry point (include/ces_b200.h), as the caller passed them.
struct ChainHost {
    const char* who;                            // entry point, for messages
    int64_t n_mcmc, n_chains;
    int pcn;
    const double *y, *scales, *mu, *Pinv;       // y: the data (ytil for the emulator); mu, Pinv unused with pCN
    const double *start, *phi_point;            // n_chains x p, row per chain
    uint32_t* mt_state;                         // numpy's MT19937 state (626 words) or NULL
    double* mt_gauss;                           // its cached Gaussian
    unsigned long long seed;
    double* samples;                            // n_chains x (n_mcmc + 1) x p
    int32_t* accepted;                          // n_chains
};

// CES_ERR_INVALID naming the entry point, before any device work, unless 1 <= n_mcmc < 2^31 - 1 (n_mcmc + 1 states fit an
// int), 1 <= n_chains <= 2^24 and the pointers are non-null: mu and Pinv unless pCN, mt_gauss whenever mt_state.
int chain_check(const ChainHost& h);

// One device allocation per sampler call, freed (after a final synchronisation of the stream, on every path) when the
// ChainRun goes out of scope.  build(layout) runs the sampler's `layout` twice: once to measure, once after the
// allocation to place its buffers and enqueue its uploads.  The arena holds the samples buffer, numpy's generator state
// (uploaded), the acceptances and then the sampler's own buffers; every buffer starts 128-byte aligned (the TMA GEMMs need
// it) and everything but the samples buffer is zeroed before the uploads, so pitch padding holds zeros.  The first failed
// upload is kept and returned by build.
class ChainRun {
  public:
    ChainRun(const ChainHost& h_, int p_, cudaStream_t st_) : h(h_), p(p_), st(st_) {}
    ~ChainRun();
    ChainRun(const ChainRun&) = delete;
    ChainRun& operator=(const ChainRun&) = delete;

    template <class F> int build(F&& layout);

    template <class T = double> T* take(size_t n) {
        T* d = reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(base_) + used_);
        used_ += (n * sizeof(T) + 127) / 128 * 128;
        return d;
    }
    template <class T> T* put(const T* src, size_t n) {           // n elements, uploaded when src != NULL
        T* d = take<T>(n);
        if (base_ && src && err_ == cudaSuccess) err_ = cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, st);
        return d;
    }
    double* put2d(const double* src, int64_t rows, int64_t cols, int64_t pitch);    // rows x cols -> rows x pitch
    double* put_columns(const double* src, int64_t ld);            // row-per-chain src (n_chains x p) -> p x ld, chain c in column c

    // samples, acceptances and numpy's advanced generator state back to the host, every copy checked; synchronises
    int copy_back();

    const ChainHost h;
    const int p;
    const cudaStream_t st;
    double* samples = nullptr;
    int* accepted = nullptr;
    uint32_t* mt = nullptr;                     // 624 key words, position, has_gauss (NULL state: unused)
    double* mt_gauss = nullptr;

  private:
    void place();
    int allocate();

    char* base_ = nullptr;
    size_t used_ = 0, zero_from_ = 0;
    cudaError_t err_ = cudaSuccess;
    std::vector<double> columns_;               // the host source of put_columns, kept until the arena is freed
};

template <class F> int ChainRun::build(F&& layout) {
    place();
    layout();
    CES_TRY(allocate());
    place();
    layout();
    return err_ == cudaSuccess ? CES_OK : fail(CES_ERR_CUDA, "%s: upload failed", h.who);
}

// ---------------------------------------------------------------------------------------------- lockstep chains
constexpr int CHAIN_THREADS = 128;

// Every chain is a column of the p x ld state arrays.
struct ChainState {
    int p, n_mcmc, n_chains, use_mt;
    long long ld;               // pitch of the p x n_chains state arrays
    double* cur;                // p x ld   current states
    double* prop;               // p x ld   the evaluated points: phi_point, then each step's proposals
    double* u;                  // n_chains: the accept test's uniform of this step
    double* phi_cur;            // n_chains
    const double* start;        // n_chains x p: state 0 of every chain
    double* samples;            // n_chains x (n_mcmc + 1) x p
    int* accepted;              // n_chains
    uint32_t* mt;               // 624 key words, pos, has_gauss
    double* mt_gauss;
    unsigned long long seed;
};

// The lockstep state in the arena of `run` (call it inside the layout): phi_point uploaded into prop.
ChainState chain_state(ChainRun& run, int64_t ld);

// Phi_cur at the evaluated points (phi_point, in prop), then cur <- start: state 0 of every chain; no proposal accepted yet
template <class Phi>
__global__ void __launch_bounds__(CHAIN_THREADS) chain_init_kernel(const ChainState a, const Phi phi) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chains) return;
    a.phi_cur[c] = phi(a, c);
    double* out = a.samples + (size_t)c * (a.n_mcmc + 1) * a.p;
    for (int q = 0; q < a.p; ++q) {
        const double v = a.start[(size_t)c * a.p + q];
        a.cur[(size_t)q * a.ld + c] = v;
        out[q] = v;
    }
    a.accepted[c] = 0;
}

// accept the proposals of step it (in prop) when log u < Phi_cur - Phi (ces/sample.py:182; NaN compares false: the proposal
// is rejected), and write state it + 1 of every chain to the samples
template <class Phi>
__global__ void __launch_bounds__(CHAIN_THREADS) chain_accept_kernel(const ChainState a, const Phi phi, int it) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.n_chains) return;
    const double phi_prop = phi(a, c);
    const bool take = log(a.u[c]) < a.phi_cur[c] - phi_prop;
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
}


}  // namespace ces
