// Host launcher of the FP64 DMMA GEMM family (see gemm.cuh).
#include <cstdlib>
#include "gemm.cuh"
#include "kernels.h"

namespace ces {

thread_local char g_last_error[512] = "";
std::atomic<long long> g_launches{0};

template <int AM, int BM_, int ROWS>
static int launch_one(cudaStream_t st, const CUtensorMap& ma, const CUtensorMap& mb, const GemmArgs& a, dim3 grid) {
    static bool attr_set[kMaxDevices] = {};
    const int slot = device_slot();
    if (!attr_set[slot]) {
        CES_CUDA(cudaFuncSetAttribute(gemm_dmma_kernel<AM, BM_, ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
        attr_set[slot] = true;
    }
    gemm_dmma_kernel<AM, BM_, ROWS><<<grid, GEMM_THREADS, GEMM_SMEM_BYTES, st>>>(ma, mb, a);
    CES_LAUNCHED(1);
    return CES_OK;
}
template <int ROWS>
static int launch_modes(cudaStream_t st, const GemmCall& c, const CUtensorMap& ma, const CUtensorMap& mb, const GemmArgs& a, dim3 grid) {
    if (c.a_mode == A_MK && c.b_mode == B_KN) return launch_one<0, 0, ROWS>(st, ma, mb, a, grid);
    if (c.a_mode == A_KM && c.b_mode == B_KN) return launch_one<1, 0, ROWS>(st, ma, mb, a, grid);
    if (c.a_mode == A_MK && c.b_mode == B_NK) return launch_one<0, 1, ROWS>(st, ma, mb, a, grid);
    return launch_one<1, 1, ROWS>(st, ma, mb, a, grid);
}

int gemm_tiles(int M, int N) { return (int)(ceil_div(M, GEMM_BM) * ceil_div(N, GEMM_BN)); }

int64_t gemm_trap_tiles(int M, int N) {
    const int64_t tm = ceil_div(M, GEMM_BM), tn = ceil_div(N, GEMM_BN);
    return tm * tn - tn * (tn - 1) / 2;
}

int64_t gemm_trap_entries(int M, int N) {
    int64_t e = 0;
    for (int64_t n0 = 0; n0 < N; n0 += GEMM_BN) e += (N - n0 < GEMM_BN ? N - n0 : GEMM_BN) * (M - n0);
    return e;
}

// 32 x 32 blocks through shared memory (coalesced on both sides); a block lies inside one 128 x 128 tile
__global__ void __launch_bounds__(256) mirror_lower_tiles_kernel(double* __restrict__ C, long long ldc, int n) {
    __shared__ double blk[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;          // destination block (upper tile)
    if (r0 / GEMM_BM >= c0 / GEMM_BN) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int y = ty; y < 32; y += 8)
        if (c0 + y < n && r0 + tx < n) blk[y][tx] = C[(size_t)(c0 + y) * ldc + r0 + tx];
    __syncthreads();
    for (int y = ty; y < 32; y += 8)
        if (r0 + y < n && c0 + tx < n) C[(size_t)(r0 + y) * ldc + c0 + tx] = blk[tx][y];
}

int mirror_lower_tiles(cudaStream_t st, double* C, int64_t ldc, int64_t n) {
    if (n <= GEMM_BN) return CES_OK;
    const unsigned b = (unsigned)ceil_div(n, 32);
    mirror_lower_tiles_kernel<<<dim3(b, b), 256, 0, st>>>(C, ldc, (int)n);
    CES_LAUNCHED(1);
    return CES_OK;
}

int gemm_sm_count() {
    static int sms_of[kMaxDevices] = {};
    int& sms = sms_of[device_slot()];
    if (!sms) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1)
            sms = 148;
    }
    return sms;
}

int gemm(cudaStream_t st, const GemmCall& c) {
    // every argument check runs before the tensor maps are built (those need the driver), so a rejected call does no
    // device work at all
    if (c.M < 1 || c.N < 1 || c.K < 1 || !c.A || !c.B || !c.C) return fail(CES_ERR_INVALID, "gemm: bad shape or null operand%s", "");
    const int64_t nb = c.batch > 1 ? c.batch : 1;
    // a batch either writes one C per problem (c_batch_elems) or, with a workspace, is summed into a single C
    // (one plane per batch, reduced like split-K); it cannot be combined with split-K itself
    if (nb > 1 && c.splits > 1) return fail(CES_ERR_INVALID, "gemm: batching excludes split-K%s", "");
    const int kb_total = (int)ceil_div(c.K, GEMM_BK);
    int splits = c.splits > 1 ? c.splits : 1;
    if (splits > kb_total) splits = kb_total;
    // With a workspace the kernel writes raw partial products and the reduce kernel applies
    // alpha / beta / diag_add and mirrors symmetric results (also used with a single split).
    const bool via_ws = c.splitk_ws != nullptr;
    if (splits > 1 && !via_ws) return fail(CES_ERR_INVALID, "gemm: split-K needs a workspace%s", "");
    if (via_ws && c.ssq_partials) return fail(CES_ERR_INVALID, "gemm: workspace path cannot produce sum-of-squares partials%s", "");
    if (!via_ws && c.diag_add != 0.0) return fail(CES_ERR_INVALID, "gemm: diag_add needs the workspace path%s", "");
    if (c.row_vec && via_ws) return fail(CES_ERR_INVALID, "gemm: row_vec needs the direct epilogue%s", "");
    if (c.flags & GEMM_C_LOWER_TRAP) {
        if (c.M < c.N) return fail(CES_ERR_INVALID, "gemm: GEMM_C_LOWER_TRAP needs M >= N%s", "");
        if (via_ws || nb > 1 || (c.flags & GEMM_C_LOWER_ONLY))
            return fail(CES_ERR_INVALID, "gemm: GEMM_C_LOWER_TRAP excludes the workspace, batching and GEMM_C_LOWER_ONLY%s", "");
    }
    if (c.flags & GEMM_C_LOWER_ONLY) {
        if (c.M != c.N) return fail(CES_ERR_INVALID, "gemm: GEMM_C_LOWER_ONLY needs a square C%s", "");
        // the skipped tiles would leave their partial slots unwritten
        if (c.ssq_partials) return fail(CES_ERR_INVALID, "gemm: GEMM_C_LOWER_ONLY cannot produce sum-of-squares partials%s", "");
    }
    // The last contraction box of batch z reads rows K .. round_up(K, 16) of a row-batched operand, which are batch z+1's.
    // That is harmless only where the other operand is zero-filled there (A_MK / B_NK, or a shared operand).
    if (nb > 1 && c.a_mode == A_KM && c.b_mode == B_KN && c.a_batch_rows != 0 && c.b_batch_rows != 0 && c.K % GEMM_BK != 0)
        return fail(CES_ERR_INVALID, "gemm: A_KM x B_KN with both operands batched needs K %% 16 == 0%s", "");
    if (c.wave_ctas < 0 || c.serpentine < -1 || c.serpentine > 1) return fail(CES_ERR_INVALID, "gemm: bad wave_ctas or serpentine%s", "");

    CUtensorMap ma, mb;
    // tensor-map row extents cover every batch of a batched operand
    const int64_t a_rows = (c.a_mode == A_MK ? c.M : c.K) + (nb - 1) * c.a_batch_rows;
    const int64_t b_rows = (c.b_mode == B_NK ? c.N : c.K) + (nb - 1) * c.b_batch_rows;
    // problems with at most 64 rows run the 64-row tile variant (half the A tile, no DMMA wasted on zero rows)
    const int bm = (c.M <= 64 && nb == 1) ? 64 : GEMM_BM;
    if (c.a_mode == A_MK) CES_TRY(make_map_2d(&ma, c.A, c.K, a_rows, c.lda, 16, bm));
    else                  CES_TRY(make_map_2d(&ma, c.A, c.M, a_rows, c.lda, 16, 16));
    if (c.b_mode == B_NK) CES_TRY(make_map_2d(&mb, c.B, c.K, b_rows, c.ldb, 16, 128));
    else                  CES_TRY(make_map_2d(&mb, c.B, c.N, b_rows, c.ldb, 16, 16));

    GemmArgs a;
    a.M = c.M; a.N = c.N; a.K = c.K;
    a.C = c.C; a.ldc = c.ldc;
    a.alpha = c.alpha; a.beta = c.beta; a.alpha_dev = c.alpha_dev;
    a.ssq_partials = c.ssq_partials;
    a.tiles_m = (int)ceil_div(c.M, bm);
    a.tiles_n = (int)ceil_div(c.N, GEMM_BN);
    static const int env_group = []() { const char* e = std::getenv("CES_GEMM_GROUP_M"); return e ? atoi(e) : 0; }();
    a.group_m = c.group_m > 0 ? c.group_m : (env_group > 0 ? env_group : 16);
    a.flags = c.flags;
    {
        a.wave_ctas = c.wave_ctas > 0 ? c.wave_ctas : gemm_sm_count();
        static const int env_serp = []() { const char* e = std::getenv("CES_GEMM_SERPENTINE"); return e ? atoi(e) : -1; }();
        // default on: -23 % DRAM reads on the D GEMM (profiles/r01_gemm_raster_sweep.csv); CES_GEMM_SERPENTINE=0 disables
        const bool serp = c.serpentine >= 0 ? c.serpentine == 1 : env_serp != 0;
        if (serp) a.flags |= GEMM_SERPENTINE_K;
        else      a.flags &= ~GEMM_SERPENTINE_K;
    }
    a.a_batch_rows = (int)c.a_batch_rows; a.b_batch_rows = (int)c.b_batch_rows; a.c_batch_elems = c.c_batch_elems;
    a.kblocks_per_split = (int)ceil_div(kb_total, splits);
    a.splits = (int)ceil_div(kb_total, a.kblocks_per_split);
    a.splitk_ws = c.splitk_ws;
    a.row_vec = c.row_vec;
    const int64_t ctas = (c.flags & GEMM_C_LOWER_TRAP) ? (int64_t)a.tiles_m * a.tiles_n - (int64_t)a.tiles_n * (a.tiles_n - 1) / 2
                                                       : (int64_t)a.tiles_m * a.tiles_n;
    dim3 grid((unsigned)ctas, (unsigned)nb, (unsigned)a.splits);
    CES_TRY(bm == 64 ? launch_modes<64>(st, c, ma, mb, a, grid) : launch_modes<128>(st, c, ma, mb, a, grid));
    if (via_ws) {
        const long long total = (long long)c.M * c.N;
        const int threads = 256;
        splitk_reduce_kernel<<<(unsigned)ceil_div(total, threads), threads, 0, st>>>(
            c.splitk_ws, nb > 1 ? (int)nb : a.splits, c.M, c.N, c.C, c.ldc, c.alpha, c.alpha_dev, c.beta, c.diag_add,
            (c.flags & GEMM_C_LOWER_ONLY) ? 1 : 0);
        CES_LAUNCHED(1);
    }
    return CES_OK;
}

}  // namespace ces
