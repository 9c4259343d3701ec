// FP64 tensor-core GEMM family for the ensemble Kalman update (sm_100a).
//
//   C[M,N] = alpha * sum_kk A(m,kk) B(kk,n)  (+ beta * C)
//
// Operands are row-major in HBM and may have either axis contiguous:
//   A_MK : A(m,kk) = A[m*lda + kk]   (contraction axis contiguous;  U~, Gamma^-1, L, C^uu ...)
//   A_KM : A(m,kk) = A[kk*lda + m]   (row axis contiguous;          E in D = E^T W)
//   B_KN : B(kk,n) = B[kk*ldb + n]   (column axis contiguous;       W, D, xi, Z)
//   B_NK : B(kk,n) = B[n*ldb + kk]   (contraction axis contiguous;  U~^T in C^uu = U~ U~^T)
//
// Design (one CTA per 128x128 output tile, BK = 16 doubles = one 128-byte swizzle span):
//   * warp 8 is the TMA producer: per stage it arms an mbarrier with the stage's byte count and
//     issues cp.async.bulk.tensor.2d loads (SWIZZLE_128B) for a 128x16 A tile and a 16x128 B tile;
//     out-of-range rows/columns/contraction indices are zero-filled by the TMA unit, so ragged
//     shapes need no special casing in the math loop;
//   * warps 0..7 are consumers on a 2x4 grid, 64x32 outputs each = 8x4 DMMA.8x8x4 accumulators
//     (128 registers), fed by conflict-free 64-bit LDS from the swizzled tiles.  To get one
//     wavefront per half-warp out of the 128-byte swizzle the fragments use permuted rows /
//     columns of the tile (the permutation is undone in the epilogue):
//        contraction-contiguous tile : fragment row g of 8x8 block b  -> tile row 16*grp + 2g + b
//        row/col-contiguous tile     : fragment row g of block b      -> 16*grp + 4b + 2(g>>2) + (g&1) + 8((g>>1)&1)
//     and contraction index kk = 4*step + t for lane t = lane & 3 in both;
//   * full/empty mbarrier ring of STAGES slots; consumers release a slot with one arrive per warp.
#pragma once
#include "tma.cuh"
#include "kernels.h"

namespace ces {

constexpr int GEMM_STAGES = 5;
constexpr int GEMM_CONSUMER_WARPS = 8;
constexpr int GEMM_THREADS = (GEMM_CONSUMER_WARPS + 4) * 32;   // 2 consumer warpgroups + 1 producer warpgroup
constexpr int GEMM_REGS_CONSUMER = 232, GEMM_REGS_PRODUCER = 40;   // setmaxnreg split of 384 x 168
constexpr int GEMM_TILE_BYTES = GEMM_BM * GEMM_BK * 8;           // 16 KB per operand per stage
constexpr int GEMM_STAGE_BYTES = 2 * GEMM_TILE_BYTES;            // 32 KB
constexpr int GEMM_SMEM_BYTES = GEMM_STAGES * GEMM_STAGE_BYTES + 1024;

struct GemmArgs {
    int M, N, K;
    double* C;
    long long ldc;
    double alpha, beta;
    const double* alpha_dev;   // optional device scalar multiplied into alpha
    double* ssq_partials;      // optional: [tiles] per-CTA sum of squares of the stored outputs (alpha*acc + beta*C), in range
    double* splitk_ws;         // when set: raw partial products go to [split][M][N] (ld = N) for the reduce kernel
    int tiles_m, tiles_n, group_m;
    int kblocks_per_split, splits;
    int flags;
    // batching over blockIdx.y: batch z uses operand rows shifted by z*{a,b}_batch_rows (0 = shared operand)
    // and writes C + z*c_batch_elems.  When K % 16 != 0 the last k-box of problem z also reads stored rows K .. round_up(K, 16)
    // of a batched A_KM / B_KN operand, which belong to problem z+1 (or to the padding between problems): those rows must be
    // finite and meet a zero-filled operand (A_MK / B_NK, or a shared operand).  gemm() refuses A_KM x B_KN with both batched.
    int a_batch_rows, b_batch_rows;
    long long c_batch_elems;
    int wave_ctas;             // CTAs resident at once (SM count); used by GEMM_SERPENTINE_K
    const double* row_vec;     // optional [M]: stored value alpha * (acc - row_vec[m]) (+ beta * C)
};

// GEMM_C_LOWER_TRAP: linear CTA index -> tile (tm, tn) of the lower trapezoid tn <= tm (tiles_m >= tiles_n), launched
// compactly.  Same grouped rasterisation as the full grid with the tiles above the diagonal left out: in a group of gs
// row tiles starting at f, columns tn < f have all gs rows, columns f <= tn < f + gs the rows tn .. f + gs - 1.
__device__ __forceinline__ void trap_tile(int L, int tiles_m, int tiles_n, int group_m, int& tm, int& tn) {
    for (int f = 0; f < tiles_m; f += group_m) {
        const int gs = min(tiles_m - f, group_m);
        const int full = min(f, tiles_n);
        const int nd = max(min(f + gs, tiles_n) - f, 0);      // columns crossing the group's diagonal
        const int cnt = full * gs + nd * gs - nd * (nd - 1) / 2;
        if (L < cnt) {
            if (L < full * gs) { tm = f + L % gs; tn = L / gs; return; }
            L -= full * gs;
            for (int c = f;; ++c) {
                const int rows = f + gs - c;
                if (L < rows) { tn = c; tm = c + L; return; }
                L -= rows;
            }
        }
        L -= cnt;
    }
    tm = tn = 0;   // not reached for L < the trapezoid's tile count
}

// Byte offset of element (row r, contraction index kk) in a contraction-contiguous 128x16 tile.
__device__ __forceinline__ uint32_t off_kc(int r, int kk) {
    return (uint32_t)(r * 128 + ((((kk >> 1) ^ (r & 7)) << 4) | ((kk & 1) << 3)));
}
// Byte offset of element (index mn, contraction index kk) in a row/col-contiguous 16x128 tile
// (stored as 8 sub-tiles of 16(kk) x 16(mn), 2 KB each).
__device__ __forceinline__ uint32_t off_mc(int mn, int kk) {
    const int in = mn & 15;
    return (uint32_t)((mn >> 4) * 2048 + kk * 128 + ((((in >> 1) ^ (kk & 7)) << 4) | ((in & 1) << 3)));
}
// Fragment-row permutations (see header).
__device__ __forceinline__ int perm_kc(int blk, int g) { return 16 * (blk >> 1) + 2 * g + (blk & 1); }
__device__ __forceinline__ int perm_mc(int blk, int g) {
    return 16 * (blk >> 1) + 4 * (blk & 1) + 2 * (g >> 2) + (g & 1) + 8 * ((g >> 1) & 1);
}

template <int IMM>
__device__ __forceinline__ double lds64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1+%2];" : "=d"(v) : "r"(addr), "n"(IMM));
    return v;
}

// BM = 128: the 8 consumer warps form a 2 x 4 grid of 64 x 32 outputs.  BM = 64 (problems with at most 64 rows: V = U~ D,
// C Z, L xi at d <= 64 would waste half of every DMMA on zero rows): a 1 x 8 grid of 64 x 16 outputs, half the A tile.
template <int A_MODE /*0=MK,1=KM*/, int B_MODE /*0=KN,1=NK*/, int BM /*128 or 64*/>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_dmma_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const GemmArgs args) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[GEMM_STAGES];
    __shared__ __align__(8) uint64_t bar_empty[GEMM_STAGES];
    __shared__ double ssq_warp[GEMM_CONSUMER_WARPS];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // ---- tile coordinates (grouped rasterisation: consecutive CTAs share B panels and a few A panels)
    int tm, tn;
    if (args.flags & GEMM_C_LOWER_TRAP) {
        trap_tile(blockIdx.x, args.tiles_m, args.tiles_n, args.group_m, tm, tn);
    } else {
        const int L = blockIdx.x;
        const int per_group = args.group_m * args.tiles_n;
        const int gid = L / per_group;
        const int first_m = gid * args.group_m;
        const int gsize = min(args.tiles_m - first_m, args.group_m);
        const int r = L - gid * per_group;
        tm = first_m + r % gsize;
        tn = r / gsize;
    }
    if ((args.flags & GEMM_C_LOWER_ONLY) && tn > tm) return;

    // ---- contraction range of this CTA
    int kb_total = (args.K + GEMM_BK - 1) / GEMM_BK;
    if (args.flags & GEMM_A_LOWER_TRI) kb_total = min(kb_total, ((tm + 1) * BM + GEMM_BK - 1) / GEMM_BK);
    if (args.flags & GEMM_B_UPPER_TRI) kb_total = min(kb_total, ((tn + 1) * GEMM_BN + GEMM_BK - 1) / GEMM_BK);
    int kb_begin = 0, kb_end = kb_total;
    if (args.splits > 1) {
        kb_begin = blockIdx.z * args.kblocks_per_split;
        kb_end = min(kb_total, kb_begin + args.kblocks_per_split);
    }
    const int nkb = max(kb_end - kb_begin, 0);
    // Alternate waves of CTAs walk the contraction axis in opposite directions: when a wave ends the L2 holds the
    // high-k part of its panels, which is exactly where the next wave (sharing the group's A panels) then starts.
    const bool reverse_k = (args.flags & GEMM_SERPENTINE_K) && (((int)blockIdx.x / args.wave_ctas) & 1);

    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t full0 = smem_u32(bar_full), empty0 = smem_u32(bar_empty);

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < GEMM_STAGES; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, GEMM_CONSUMER_WARPS);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp >= GEMM_CONSUMER_WARPS) {
        // ================================ TMA producer warpgroup ================================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(GEMM_REGS_PRODUCER));
        if (warp == GEMM_CONSUMER_WARPS && lane == 0) {
            tma_prefetch_desc(&mapA);
            tma_prefetch_desc(&mapB);
            const int m0 = tm * BM, n0 = tn * GEMM_BN;
            constexpr uint32_t stage_tx = (uint32_t)(BM * GEMM_BK * 8 + GEMM_TILE_BYTES);
            for (int it = 0; it < nkb; ++it) {
                const int s = it % GEMM_STAGES;
                const uint32_t ph = (uint32_t)(it / GEMM_STAGES) & 1u;
                mbar_wait(empty0 + 8 * s, ph ^ 1u);
                const uint32_t fb = full0 + 8 * s;
                mbar_expect_tx(fb, stage_tx);
                const uint32_t a_dst = smem_base + s * GEMM_STAGE_BYTES;
                const uint32_t b_dst = a_dst + GEMM_TILE_BYTES;
                const int k0 = (reverse_k ? (kb_end - 1 - it) : (kb_begin + it)) * GEMM_BK;
                const int az = (int)blockIdx.y * args.a_batch_rows, bz = (int)blockIdx.y * args.b_batch_rows;
                if (A_MODE == 0) {
                    tma_load_2d(a_dst, &mapA, fb, k0, m0 + az);
                } else {
#pragma unroll
                    for (int o = 0; o < BM / 16; ++o) tma_load_2d(a_dst + o * 2048, &mapA, fb, m0 + 16 * o, k0 + az);
                }
                if (B_MODE == 1) {
                    tma_load_2d(b_dst, &mapB, fb, k0, n0 + bz);
                } else {
#pragma unroll
                    for (int o = 0; o < 8; ++o) tma_load_2d(b_dst + o * 2048, &mapB, fb, n0 + 16 * o, k0 + bz);
                }
            }
        }
        return;
    }

    // ================================ DMMA consumers ================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(GEMM_REGS_CONSUMER));
    constexpr int NJ = BM == 128 ? 4 : 2;                               // 8-column blocks per warp
    const int wm = BM == 128 ? warp >> 2 : 0, wn = BM == 128 ? (warp & 3) : warp;
    const int g = lane >> 2, t = lane & 3;

    double acc[8][NJ][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // Per-lane byte offsets of the step-0 fragments of 8x8 blocks 0 and 1 inside a stage.  Block i
    // sits 2048*(i>>1) bytes further in both tile layouts (an LDS immediate), and step `st` changes
    // the offset by XOR / add constants (below), so four registers address all 48 fragment loads.
    uint32_t a_par[2], b_par[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        a_par[q] = (A_MODE == 0) ? off_kc(wm * 64 + perm_kc(q, g), t) : off_mc(wm * 64 + perm_mc(q, g), t);
        b_par[q] = GEMM_TILE_BYTES + ((B_MODE == 1) ? off_kc(wn * (8 * NJ) + perm_kc(q, g), t) : off_mc(wn * (8 * NJ) + perm_mc(q, g), t));
    }

    for (int it = 0; it < nkb; ++it) {
        const int s = it % GEMM_STAGES;
        const uint32_t ph = (uint32_t)(it / GEMM_STAGES) & 1u;
        mbar_wait(full0 + 8 * s, ph);
        const uint32_t sb = smem_base + s * GEMM_STAGE_BYTES;
#pragma unroll
        for (int st = 0; st < 4; ++st) {
            // kk = 4*st + t.  Contraction-contiguous: 16-byte chunk index (kk>>1) changes by XOR 2*st.
            // Row/col-contiguous: row kk adds st*512 bytes and the chunk XOR flips bit 2 when st is odd.
            uint32_t pa[2], pb[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                pa[q] = sb + ((A_MODE == 0) ? (a_par[q] ^ (uint32_t)(st << 5))
                                            : ((a_par[q] ^ (uint32_t)((st & 1) << 6)) + (uint32_t)(st * 512)));
                pb[q] = sb + ((B_MODE == 1) ? (b_par[q] ^ (uint32_t)(st << 5))
                                            : ((b_par[q] ^ (uint32_t)((st & 1) << 6)) + (uint32_t)(st * 512)));
            }
            double a[8], b[NJ];
            a[0] = lds64<0>(pa[0]);    a[1] = lds64<0>(pa[1]);
            a[2] = lds64<2048>(pa[0]); a[3] = lds64<2048>(pa[1]);
            a[4] = lds64<4096>(pa[0]); a[5] = lds64<4096>(pa[1]);
            a[6] = lds64<6144>(pa[0]); a[7] = lds64<6144>(pa[1]);
            b[0] = lds64<0>(pb[0]);    b[1] = lds64<0>(pb[1]);
            if (NJ == 4) { b[NJ - 2] = lds64<2048>(pb[0]); b[NJ - 1] = lds64<2048>(pb[1]); }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < NJ; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * s);
    }

    // ================================ epilogue ================================
    double alpha = args.alpha;
    if (args.alpha_dev) alpha *= *args.alpha_dev;
    const double beta = args.beta;
    const int m_base = tm * BM + wm * 64, n_base = tn * GEMM_BN + wn * (8 * NJ);
    double ssq = 0.0;
    const bool to_ws = args.splitk_ws != nullptr;
    // workspace planes: one per split (blockIdx.z) or, for a batch reduced into one C, one per batch (blockIdx.y)
    double* out = to_ws ? args.splitk_ws + (size_t)(blockIdx.z + blockIdx.y) * (size_t)args.M * (size_t)args.N
                        : args.C + (size_t)blockIdx.y * (size_t)args.c_batch_elems;
    const long long ldo = to_ws ? (long long)args.N : args.ldc;
    // The sum of squares is that of alpha * acc (+ beta * C), before the row term is taken off.  A trapezoid tile below
    // the diagonal also stands for its mirror (row and column indices swapped), whose row term is row_vec[n].
    const bool mirror = (args.flags & GEMM_C_LOWER_TRAP) && tm != tn;
    double shift_n[NJ][2];
#pragma unroll
    for (int j = 0; j < NJ; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int n = n_base + ((B_MODE == 1) ? perm_kc(j, 2 * t + e) : perm_mc(j, 2 * t + e));
            shift_n[j][e] = (mirror && args.row_vec && n < args.N) ? alpha * args.row_vec[n] : 0.0;
        }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m_base + ((A_MODE == 0) ? perm_kc(i, g) : perm_mc(i, g));
        if (m >= args.M) continue;
        double* row = out + (size_t)m * ldo;
        const double rv = args.row_vec ? args.row_vec[m] : 0.0;
        // beta != 0: all of this row's old values are loaded before the first store (independent loads in flight;
        // interleaved with the stores they would serialise on possible aliasing -- the epilogue is exposed, one CTA per SM)
        double old[NJ][2];
        if (!to_ws && beta != 0.0) {
#pragma unroll
            for (int j = 0; j < NJ; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int n = n_base + ((B_MODE == 1) ? perm_kc(j, 2 * t + e) : perm_mc(j, 2 * t + e));
                    old[j][e] = n < args.N ? __ldcs(row + n) : 0.0;
                }
        }
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int n = n_base + ((B_MODE == 1) ? perm_kc(j, 2 * t + e) : perm_mc(j, 2 * t + e));
                if (n >= args.N) continue;
                if (to_ws) {
                    row[n] = acc[i][j][e];
                } else {
                    double v = alpha * (acc[i][j][e] - rv);
                    if (beta != 0.0) v += beta * old[j][e];
                    // of the value stored (plus the row term): a contraction accumulated in chunks (beta = 1) sums the final D
                    const double d = v + alpha * rv;
                    ssq += d * d;
                    if (mirror) {
                        const double dt = v + shift_n[j][e];
                        ssq += dt * dt;
                    }
                    row[n] = v;
                }
            }
        }
    }
    if (args.ssq_partials) {
        ssq = warp_sum(ssq);
        if (lane == 0) ssq_warp[warp] = ssq;
        // consumers only: named barrier 1 over the 8 consumer warps
        asm volatile("bar.sync 1, %0;" ::"n"(GEMM_CONSUMER_WARPS * 32));
        if (threadIdx.x == 0) {
            double tot = 0.0;
#pragma unroll
            for (int w = 0; w < GEMM_CONSUMER_WARPS; ++w) tot += ssq_warp[w];
            args.ssq_partials[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = tot;
        }
    }
}

// Deterministic split-K reduction: C = alpha * sum_z ws[z] (+ beta * C) (+ diag_add on the diagonal).
// With `symmetric` the lower triangle of the sum is mirrored (only tiles tn <= tm were computed).
__global__ void splitk_reduce_kernel(const double* __restrict__ ws, int splits, int M, int N, double* __restrict__ C,
                                     long long ldc, double alpha, const double* alpha_dev, double beta, double diag_add,
                                     int symmetric) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)M * N) return;
    const int m = (int)(idx / N), n = (int)(idx % N);
    int sm = m, sn = n;
    if (symmetric && n > m) { sm = n; sn = m; }
    const size_t plane = (size_t)M * (size_t)N;
    double s = 0.0;
    for (int z = 0; z < splits; ++z) s += ws[z * plane + (size_t)sm * N + sn];
    double a = alpha;
    if (alpha_dev) a *= *alpha_dev;
    double v = a * s;
    if (beta != 0.0) v += beta * C[(size_t)m * ldc + n];
    if (m == n) v += diag_add;
    C[(size_t)m * ldc + n] = v;
}

}  // namespace ces
