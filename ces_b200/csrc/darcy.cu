// Batched 2-D Darcy forward solve, one thread-block cluster per ensemble member.
//
// Reference arithmetic: ces/darcy.py:20-38,84-98,129-138 -> utilities/mfiles/gaussrnd_coarse.m:6-23 (KL field by
// inverse 2-D DCT) and utilities/mfiles/solve_gwf.m:4-39 (spline to the K x K nodes, 5-point finite differences with
// arithmetic-mean face coefficients scaled by (K-1)^2, right-hand side 1, zero Dirichlet boundary, spline back to the
// cell centres), one MATLAB-engine round trip per particle in the reference.
//
// Here, per chunk of members (all buffers member-major, a member's K x K field contiguous):
//   Theta = U^T Phi^T                       DMMA GEMM (A_KM x B_KN)
//   a     = exp(Theta)                      elementwise
//   T1    = a S^T ; c_z = S T1_z            two DMMA GEMMs (stacked, then batched with the shared operand S)
//   solve sum_faces w (p_i - p_nb) = h^2    darcy_pcg_tile_kernel: two-level preconditioned CG, the member's vectors live in
//                                           registers + shared memory of a cluster of CTAs (row strips; halo rows and
//                                           partial dot products travel through distributed shared memory)
//   T2 = p S2^T ; P_z = S2 T2_z             spline back to the centres (two more GEMMs)
//   G[o, member] = P_z[obs_index[o]]        gather (or the transposed full field)
#include <cooperative_groups.h>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>
#include "kernels.h"
#include "tma.cuh"

namespace cg = cooperative_groups;

namespace ces {

// ------------------------------------------------------------------------------------------------------------------
// Conjugate-gradient solver.  Preconditioned CG (Jacobi scaling + an aggregation coarse level, see CoarseGeom below), laid
// out so that one SM carries 4 032 nodes (everything but the search direction in registers) and a cluster-wide reduction
// costs one DSMEM round trip instead of a cluster barrier:
//
//  * symmetric Jacobi scaling: with s = diag(A)^(-1/2) the solver runs plain CG on A^ = S A S (unit diagonal), which is
//    Jacobi-preconditioned CG on A in exact arithmetic (same iterates, r^.r^ = r.M^-1 r, so the stopping rule
//    r.M^-1 r <= tol^2 r0.M^-1 r0 is unchanged).  No z vector, no 1/diag array, 9 FP64 operations per node and iteration.
//  * every thread owns a 4 x 2 tile of nodes: x, r, p and the 14 scaled weights of the faces inside / above / below the
//    tile stay in registers; only p (for the neighbours) and the weights of the faces between horizontally adjacent tiles
//    live in shared memory, stored as separate even-column / odd-column planes so every access is a conflict-free,
//    fully coalesced 64-bit access.
//  * cluster-wide sums and halo rows travel as st.async stores that complete a transaction count on the receiver's
//    mbarrier (one DSMEM latency, no barrier.cluster, no L1 flush); the two barriers alternate (r.r / p.Ap), so a peer can
//    run at most one synchronisation point ahead and single-buffered slots are race free.
//  * a strip's halo needs no p exchange: a CTA receives the neighbour's residual row and updates its own copy of
//    the neighbour's p row with the same p = r + beta p, bit-identical to the owner's.
struct __align__(16) TileShared {
    double red[2][8];                   // [which][cluster rank] block partials of r.r (0) and p.Ap (1)
    double wsum[2][16];                 // [which][warp] warp partials
    unsigned long long bar[2];          // mbarriers of the two synchronisation points
};

__device__ __forceinline__ uint32_t cluster_map(uint32_t local_smem_addr, uint32_t rank) {
    uint32_t out;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(out) : "r"(local_smem_addr), "r"(rank));
    return out;
}
__device__ __forceinline__ void st_async_f64(uint32_t remote_addr, double v, uint32_t remote_bar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(remote_addr),
                 "l"(__double_as_longlong(v)), "r"(remote_bar)
                 : "memory");
}
__device__ __forceinline__ void st_async_f64x2(uint32_t remote_addr, double a, double b, uint32_t remote_bar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v2.b64 [%0], {%1, %2}, [%3];" ::"r"(remote_addr),
                 "l"(__double_as_longlong(a)), "l"(__double_as_longlong(b)), "r"(remote_bar)
                 : "memory");
}

constexpr int TILE_THREADS = 512;

// Warp-wide sum on the FP64 tensor pipe: two dependent DMMA.8x8x4 and one add instead of five shuffle rounds (ten SHFL
// and five adds) -- about half the latency, and latency is what the CG iteration is made of.  With A = 1 and B = v the
// first product leaves in lane (g, t) the sums of lane groups 2t and 2t+1; their sum s(t) as A against B = 1 gives every
// lane the total.  Fixed hardware summation order: identical in every warp, CTA and run.
__device__ __forceinline__ double warp_sum_mma(double v) {
    double c0 = 0.0, c1 = 0.0;
    dmma884(c0, c1, 1.0, v);
    const double s = c0 + c1;
    double d0 = 0.0, d1 = 0.0;
    dmma884(d0, d1, s, 1.0);
    return d0;
}

// 1/x to (almost) full precision: MUFU.RCP64H seed + two Newton steps, 5 dependent operations instead of the ~20 of an
// IEEE division.  Not correctly rounded (<= 2 ulp), which CG does not care about; what matters is that every thread of
// the cluster executes the same instructions on the same bits and so gets the same alpha and beta.
__device__ __forceinline__ double fast_rcp(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    y = fma(y, e, y);
    e = fma(-x, y, 1.0);
    return fma(y, e, y);
}

// Two-level preconditioner (COARSE): M^-1 = I + P Ac^-1 P^T on the scaled system, P = piecewise constants on aggregates of
// H x H nodes (H = 16 at K = 128, 8 at K = 64: at most 8 x 8 = 64 aggregates, aligned with the thread tiles and the CTA
// strips), Ac = P^T A^ P assembled from the face weights at start-up and inverted in shared memory by every CTA (in-place
// Gauss-Jordan, 64 x 64).  Per iteration the restriction P^T r rides on the r.r exchange (one extra double per aggregate),
// every CTA applies the dense 64 x 64 inverse redundantly, and r.M^-1 r = r.r + rc.ec needs no further exchange -- the
// number of DSMEM round trips per iteration stays two while the iteration count drops by ~2.7 (610 -> 225 at 128^2).
// Between the two sits a third, purely local level: aggregates of 4 x 4 nodes (the tiles of two adjacent lanes) with a
// diagonal solve, M^-1 = I + P1 diag(P1^T A^ P1)^-1 P1^T + P Ac^-1 P^T (additive multilevel).  It costs one shuffle and a
// handful of flops per iteration -- its term of r.M^-1 r is added to the thread's partial before the exchange, and the
// halo rows are pushed as r + P1 e1 so the neighbour's copy of the search direction stays exact -- and takes another
// third off the iteration count (225 -> 150 at 128^2).
// Members with a negative diagonal (see below) and shapes whose aggregates do not align run plain Jacobi scaling.
struct CoarseGeom {
    int H, HQ, HG, NCR, NCC, NA;
};
__host__ __device__ constexpr CoarseGeom coarse_geom(int K) {
    // smallest aggregate side in {4, 8, 16} that leaves at most 8 x 8 aggregates; H/2 is a power of two (segmented shuffles)
    const int H = K <= 32 ? 4 : (K <= 64 ? 8 : 16);
    return CoarseGeom{H, H / 2, H / 4, (K - 3) / H + 1, (K - 2) / H + 1, ((K - 3) / H + 1) * ((K - 2) / H + 1)};
}
constexpr int COARSE_SMEM_DOUBLES = 4096 + 64 + 64 + 128 + 320 + 256;
// Threads per row of the 64 x 64 coarse solve, fixed by the default launch shape of each grid size (compile-time so the
// short loops over a row unroll): 128 threads at K = 32, 288 at K = 48, 512 at K = 64 (256 with a 2-CTA cluster) and K = 128.
__host__ __device__ constexpr int coarse_parts(int KH, bool cluster) {
    return KH == 16 ? 2 : KH == 24 ? 4 : KH == 32 ? (cluster ? 4 : 8) : KH == 64 ? 8 : (KH == 40 || KH == 48 || KH == 56) ? 4 : 0;
}

// One cluster of C CTAs per member; CTA `crank` owns the interior rows 1 + crank*4G ... (4G rows, G row groups of 4);
// thread (g, q) owns rows 4g..4g+3 of the strip and the columns 2q, 2q+1.  blockDim.x = round_up(G * KH, 32), KH = K/2
// is a template parameter so every shared-memory access is one base register plus an immediate offset.
// The template grid K = 2 KH (a multiple of 16) may be larger than the member's grid: `Kact` x `Kact` nodes stored with row
// pitch `ldk`; rows / columns from Kact - 1 on are padding (s = 0: inert, like boundary nodes), so any Nmesh <= 128 runs.
template <int KH, bool CLUSTER, bool COARSE>
__global__ void __launch_bounds__(TILE_THREADS, 1)
darcy_pcg_tile_kernel(const double* __restrict__ cn, double* __restrict__ pn, int G, double tol2, int max_iter,
                      int* __restrict__ iters_out, int Kact, int ldk) {
    constexpr int K = 2 * KH;
    cg::cluster_group cluster = cg::this_cluster();
    const int C = CLUSTER ? (int)cluster.num_blocks() : 1;        // CLUSTER == false: one CTA per member, no DSMEM traffic
    const int crank = CLUSTER ? (int)cluster.block_rank() : 0;
    const long long member = blockIdx.x / C;
    const int R = 4 * G;
    extern __shared__ double smem[];
    const int plane = (R + 2) * KH;
    double* pe = smem;                  // (R+2) x KH  search direction, even columns, rows r0-1 .. r0+R
    double* po = pe + plane;            //             odd columns
    double* se = po + plane;            // (R+2) x KH  s = |diag|^(-1/2), even / odd columns (0 on boundary nodes)
    double* so = se + plane;
    double* we = so + plane;            // R x (KH+1)  entry q+1: -s_i s_j w of the face between columns 2q+1 and 2q+2; entry 0: 0
    double* zh = we + R * (KH + 1);           // 2 x K       residual rows of the neighbouring strips: [0,K) above, [K,2K) below
    // coarse level (COARSE only)
    constexpr CoarseGeom CG = coarse_geom(K);
    double* Ainv = zh + 2 * K;          // 64 x 64 inverse of Ac, element (i, j) at (j % JP) * 64 * PARTS + i * PARTS + j / JP
    double* rcv = Ainv + 4096;          // 64  coarse residual P^T r (gathered from all CTAs)
    double* ec = rcv + 64;              // 64  coarse correction Ac^-1 rc
    double* stage = ec + 64;            // G x NCC  per row group partial restriction
    double* cgath = stage + 128;        // 5 x 64   coarse matrix entries (diag, N, S, W, E) of every aggregate
    double* prow = cgath + 320;         // 2 x 64 + 2 x 64  pivot rows / pivot columns of the inversion (double-buffered)
    __shared__ TileShared sh;
    __shared__ int sflag[8];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int g = tid / KH, q = tid - g * KH;
    const bool active = g < G;
    const int r0 = 1 + crank * R;
    const int i0 = r0 + 4 * g;
    const int lr = 4 * g + 1;           // local row of the tile's first row in the (R+2)-row planes
    const double* cfield = cn + (size_t)member * Kact * ldk;

    for (int idx = tid; idx < 4 * plane + R * (KH + 1); idx += blockDim.x) pe[idx] = 0.0;      // pe, po, se, so, we
    for (int idx = tid; idx < 2 * K + (COARSE ? COARSE_SMEM_DOUBLES : 0); idx += blockDim.x) zh[idx] = 0.0;
    for (int idx = tid; idx < 48; idx += blockDim.x) (&sh.red[0][0])[idx] = 0.0;    // red + wsum
    if (tid == 0) {
        mbar_init(smem_u32(&sh.bar[0]), 1);
        mbar_init(smem_u32(&sh.bar[1]), 1);
        mbar_fence_init();
    }
    if (CLUSTER) cluster.sync(); else __syncthreads();

    // ---- face weights from the nodal coefficients (solve_gwf.m:16-30): w = (c_i + c_j) / 2
    unsigned negmask = 0, okmask = 0;
    int nvalid = 0;
    double wv[5][2], wi[4], wr[4], s[4][2];       // wr and s are dead once the loop starts
    {
        double cl[6][4], wl[4];
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            const int row = min(max(i0 - 1 + a, 0), Kact - 1);
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int col = min(max(2 * q - 1 + b, 0), Kact - 1);
                cl[a][b] = active ? __ldg(cfield + (size_t)row * ldk + col) : 0.0;
            }
        }
#pragma unroll
        for (int a = 0; a < 5; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) wv[a][b] = 0.5 * (cl[a][b + 1] + cl[a + 1][b + 1]);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            wl[a] = 0.5 * (cl[a + 1][0] + cl[a + 1][1]);
            wi[a] = 0.5 * (cl[a + 1][1] + cl[a + 1][2]);
            wr[a] = 0.5 * (cl[a + 1][2] + cl[a + 1][3]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                const int row = i0 + a, col = 2 * q + b;
                const bool ok = active && row <= Kact - 2 && col >= 1 && col <= Kact - 2;
                const double d = ((wv[a][b] + wv[a + 1][b]) + (b == 0 ? wl[a] : wi[a])) + (b == 0 ? wi[a] : wr[a]);
                if (ok && d < 0.0) negmask |= 1u << (2 * a + b);
                nvalid += ok ? 1 : 0;
                if (ok) okmask |= 1u << (2 * a + b);
                s[a][b] = ok ? 1.0 / sqrt(fabs(d)) : 0.0;
            }
        if (active) {
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                se[(lr + a) * KH + q] = s[a][0];
                so[(lr + a) * KH + q] = s[a][1];
            }
            // s of the rows next to a strip boundary is needed by the neighbouring CTA for the shared faces
            if (g == 0 && crank > 0) {
                cluster.map_shared_rank(se, crank - 1)[(R + 1) * KH + q] = s[0][0];
                cluster.map_shared_rank(so, crank - 1)[(R + 1) * KH + q] = s[0][1];
            }
            if (g == G - 1 && crank < C - 1) {
                cluster.map_shared_rank(se, crank + 1)[q] = s[3][0];
                cluster.map_shared_rank(so, crank + 1)[q] = s[3][1];
            }
        }
    }
    if (CLUSTER) cluster.sync(); else __syncthreads();

    // ---- scaled, negated weights: nw = -(s_i s_j) w, identical on both sides of a face (the product s_i s_j commutes).
    // s = 0 on boundary / padding nodes, so every face of such a node has weight 0: its A^p is exactly 0, its r and p stay
    // 0 for ever, and no masking is needed inside the loop.
    const int qw = q > 0 ? q - 1 : q, qe = q < KH - 1 ? q + 1 : q;
    if (active) {
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const double* sp = b == 0 ? se : so;
            wv[0][b] *= -(sp[(lr - 1) * KH + q] * s[0][b]);
#pragma unroll
            for (int a = 1; a < 4; ++a) wv[a][b] *= -(s[a - 1][b] * s[a][b]);
            wv[4][b] *= -(s[3][b] * sp[(lr + 4) * KH + q]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            wi[a] *= -(s[a][0] * s[a][1]);
            we[(4 * g + a) * (KH + 1) + q + 1] = wr[a] * -(s[a][1] * se[(lr + a) * KH + qe]);
        }
    } else {
#pragma unroll
        for (int a = 0; a < 5; ++a) wv[a][0] = wv[a][1] = 0.0;
#pragma unroll
        for (int a = 0; a < 4; ++a) wi[a] = 0.0;
    }
    // x = 0, r = b^ = s h^2, p = 0
    double x[4][2], r[4][2], p[4][2];
    const double h2 = 1.0 / ((double)(Kact - 1) * (double)(Kact - 1));
    double part = 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            x[a][b] = 0.0;
            p[a][b] = 0.0;
            r[a][b] = s[a][b] * h2;         // s = 0 on boundary nodes
            if ((negmask >> (2 * a + b)) & 1u) r[a][b] = -r[a][b];
            part += ((negmask >> (2 * a + b)) & 1u) ? -(r[a][b] * r[a][b]) : r[a][b] * r[a][b];
        }
    // A spline of exp(theta) can undershoot below zero (the reference's own example does: all 256 modes at prior scale
    // 10), and then diag(A) has negative entries.  The reference hands the matrix to a direct solver; here the CG
    // recurrence with M = diag(A) is run regardless, exactly as written for the unscaled system: with s = |d|^(-1/2), sigma = sign(d) the scaled
    // operator has diagonal sigma, the register `r` holds t = sigma r^ (so p = t + beta p), and r.M^-1 r = sum sigma t^2.
    // The sign flips are integer operations compiled only into the variant a CTA with a negative diagonal runs.
    const bool cta_signed = __syncthreads_or(negmask != 0) != 0;       // also: `we` is complete
    const double* const we_t = we + 4 * g * (KH + 1) + q;   // [0]: west face of the tile, [1]: east face

    // ---- coarse level: assemble Ac = P^T A^ P and invert it (identically in every CTA of the cluster)
    constexpr int PARTS_RAW = coarse_parts(KH, CLUSTER);  // threads per coarse row (0: this shape has no coarse level)
    constexpr int PARTS = PARTS_RAW > 0 ? PARTS_RAW : 1;
    constexpr int JP = 64 / PARTS;
    const int ARL = CLUSTER ? R / CG.H : CG.NCR;          // aggregate rows owned by this CTA
    const int a_own = ((crank * R + 4 * g) / CG.H) * CG.NCC + (2 * q) / CG.H;      // aggregate of this thread's tile
    // coarse vectors (rcv, ec, the pivot row of the inversion) are stored permuted, entry j at (j % JP) * PARTS + j / JP: the
    // PARTS threads of a coarse row then read consecutive words (no bank conflicts); dot products do not care about order
    auto cpos = [&](int j) -> int { return (j % JP) * PARTS + j / JP; };
    bool use_coarse = false;
    double inv_d1 = 0.0;                                  // 1 / diagonal entry of this tile pair on the intermediate level
    if (COARSE) {
        bool any_signed = cta_signed;
        if (CLUSTER) {
            if (tid < C) *cluster.map_shared_rank(&sflag[crank], tid) = cta_signed ? 1 : 0;
            cluster.sync();
            any_signed = false;
            for (int c = 0; c < C; ++c) any_signed = any_signed || sflag[c] != 0;
        }
        use_coarse = !any_signed && PARTS_RAW >= 2 && (int)blockDim.x >= 64 * PARTS && (!CLUSTER || R % CG.H == 0);
        if (use_coarse) {
            // contributions of this tile: unit diagonal of the valid nodes, faces inside the tile twice, faces to a tile
            // of the same aggregate once (the other side adds its own), faces to another aggregate as off-diagonal entries
            const int NT = (int)blockDim.x;
            double cd = 0.0, cN = 0.0, cS = 0.0, cW = 0.0, cE = 0.0;
            double own_int = 0.0, shared_faces = 0.0;
            if (active) {
                double inner = ((wi[0] + wi[1]) + (wi[2] + wi[3])) + (((wv[1][0] + wv[1][1]) + (wv[2][0] + wv[2][1])) + (wv[3][0] + wv[3][1]));
                cd = (double)nvalid + 2.0 * inner;
                own_int = cd;
                const double north = wv[0][0] + wv[0][1], south = wv[4][0] + wv[4][1];
                const double west = (we_t[0] + we_t[KH + 1]) + (we_t[2 * (KH + 1)] + we_t[3 * (KH + 1)]);
                const double east = (we_t[1] + we_t[KH + 2]) + (we_t[2 * (KH + 1) + 1] + we_t[3 * (KH + 1) + 1]);
                shared_faces = (q & 1) ? west : east;           // the faces between the two tiles of a pair
                if ((i0 - 1) % CG.H != 0) cd += north; else cN = north;
                if ((i0 + 3) % CG.H != 0) cd += south; else cS = south;
                if ((2 * q) % CG.H != 0) cd += west; else cW = west;
                if ((2 * q + 2) % CG.H != 0) cd += east; else cE = east;
            }
            // intermediate level: aggregates of 4 x 4 nodes = the tiles of lanes (2m, 2m+1); only its diagonal is used
            {
                const double pair_d = (own_int + __shfl_xor_sync(0xffffffffu, own_int, 1)) + 2.0 * shared_faces;
                // (at Nmesh = 32 the coarse aggregates are these very 4 x 4 blocks: a second copy would over-correct)
                inv_d1 = (CG.H > 4 && pair_d > 0.0) ? 1.0 / pair_d : 0.0;
            }
            double* st5 = Ainv;                         // staging: 5 x NT (the inverse is built afterwards)
            st5[tid] = cd; st5[NT + tid] = cN; st5[2 * NT + tid] = cS; st5[3 * NT + tid] = cW; st5[4 * NT + tid] = cE;
            __syncthreads();
            if (tid < ARL * CG.NCC) {
                const int arl = tid / CG.NCC, ac = tid - arl * CG.NCC;
                const int ar = crank * ARL + arl;
                if (ar < CG.NCR) {
                    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
                    for (int gg = 0; gg < CG.HG; ++gg) {
                        const int gl = arl * CG.HG + gg;
                        if (gl >= G) break;
                        for (int qq = 0; qq < CG.HQ; ++qq) {
                            const int ql = ac * CG.HQ + qq;
                            if (ql >= KH) break;
                            const int tt = gl * KH + ql;
#pragma unroll
                            for (int v = 0; v < 5; ++v) acc[v] += st5[v * NT + tt];
                        }
                    }
                    const int ag = ar * CG.NCC + ac;
                    for (int c = 0; c < C; ++c) {
                        double* dst = CLUSTER ? cluster.map_shared_rank(cgath, c) : cgath;
#pragma unroll
                        for (int v = 0; v < 5; ++v) dst[v * 64 + ag] = acc[v];
                    }
                }
            }
            if (CLUSTER) cluster.sync(); else __syncthreads();
            for (int idx = tid; idx < 4096; idx += NT) Ainv[idx] = 0.0;
            __syncthreads();
            auto at = [&](int i, int j) -> double& { return Ainv[(j % JP) * (64 * PARTS) + i * PARTS + j / JP]; };
            if (tid < 64) {
                const int a = tid, ar = a / CG.NCC, ac = a - ar * CG.NCC;
                if (a < CG.NA && cgath[a] != 0.0) {          // (an aggregate made of padding only has no entries)
                    at(a, a) = cgath[a];
                    if (ar > 0) at(a, a - CG.NCC) = cgath[64 + a];
                    if (ar < CG.NCR - 1) at(a, a + CG.NCC) = cgath[128 + a];
                    if (ac > 0) at(a, a - 1) = cgath[192 + a];
                    if (ac < CG.NCC - 1) at(a, a + 1) = cgath[256 + a];
                } else {
                    at(a, a) = 1.0;
                }
            }
            __syncthreads();
            // in-place Gauss-Jordan without pivoting (Ac is symmetric positive definite, condition number O(30)).  Every
            // thread keeps its JP elements of one row in registers; the pivot row and pivot column of the next step are
            // published through double-buffered shared memory, so a step costs one barrier.  A step is one uniform
            // rank-one update e -= f * (row_k[j] / piv): publishing piv + 1 as the pivot row's own diagonal entry and
            // using f = piv - 1 for the pivot row itself produces 1/piv, row_k/piv and -col_k/piv in the right places
            // without any per-element case distinction.
            double* prowB = prow;                       // [2][64], permuted like rcv
            double* fcolB = prow + 128;                 // [2][64]
            const bool worker = tid < 64 * PARTS;
            const int gi = tid / PARTS, gp = tid - gi * PARTS;
            double el[JP];
#pragma unroll
            for (int jj = 0; jj < JP; ++jj) el[jj] = worker ? Ainv[jj * (64 * PARTS) + tid] : 0.0;
            auto pick = [&](int idx) -> double {         // el[idx] for a warp-uniform run-time index
                double v = el[0];
#pragma unroll
                for (int jj = 1; jj < JP; ++jj) v = (jj == idx) ? el[jj] : v;
                return v;
            };
            if (worker) {
                if (gi == 0) {
#pragma unroll
                    for (int jj = 0; jj < JP; ++jj) prowB[jj * PARTS + gp] = el[jj] + ((gp == 0 && jj == 0) ? 1.0 : 0.0);
                }
                if (gp == 0) fcolB[gi] = el[0];
            }
            __syncthreads();
            bool ok_inv = true;
            for (int k = 0; k < 64; ++k) {
                const double* pr = prowB + (k & 1) * 64;
                const double* fc = fcolB + (k & 1) * 64;
                const double piv = fc[k];
                if (!(piv > 1e-300)) { ok_inv = false; break; }           // uniform: every thread reads the same pivot
                const double ipiv = fast_rcp(piv);
                const int nq = (k + 1) / JP, nr = (k + 1) - nq * JP;      // column k+1 is element nr of the threads with gp == nq
                if (worker) {
                    const double f = (gi == k) ? piv - 1.0 : fc[gi];
#pragma unroll
                    for (int jj = 0; jj < JP; ++jj) el[jj] = fma(-f, pr[jj * PARTS + gp] * ipiv, el[jj]);
                    if (k + 1 < 64) {
                        double* prn = prowB + ((k + 1) & 1) * 64;
                        const double nextcol = pick(nr);
                        if (gi == k + 1) {
#pragma unroll
                            for (int jj = 0; jj < JP; ++jj) prn[jj * PARTS + gp] = el[jj];
                            if (gp == nq) prn[nr * PARTS + gp] = nextcol + 1.0;
                        }
                        if (gp == nq) fcolB[((k + 1) & 1) * 64 + gi] = nextcol;
                    }
                }
                __syncthreads();
            }
            if (worker) {
#pragma unroll
                for (int jj = 0; jj < JP; ++jj) Ainv[jj * (64 * PARTS) + tid] = el[jj];
            }
            __syncthreads();
            use_coarse = ok_inv;
        }
    }

    // ---- synchronisation machinery
    const uint32_t bar0 = smem_u32(&sh.bar[0]);         // bar[1] is bar0 + 8
    const bool first_group = active && g == 0 && crank > 0, last_group = active && g == G - 1 && crank < C - 1;
    uint32_t push_n_addr = 0, push_s_addr = 0;
    if (first_group) push_n_addr = cluster_map(smem_u32(zh + K + 2 * q), (uint32_t)(crank > 0 ? crank - 1 : 0));    // our first row = its row below
    if (last_group) push_s_addr = cluster_map(smem_u32(zh + 2 * q), crank + 1);         // our last row = its row above
    const uint32_t push_n_bar = cluster_map(bar0, crank > 0 ? crank - 1 : 0), push_s_bar = cluster_map(bar0, crank < C - 1 ? crank + 1 : 0);
    // bytes this CTA receives at each synchronisation point
    const uint32_t expect0 = (uint32_t)((C - 1) * 8 + ((crank > 0) + (crank < C - 1)) * K * 8 + (use_coarse ? CG.NA * 8 : 0)),
                   expect1 = (uint32_t)((C - 1) * 8);
    uint32_t phase = 0;                                 // bit w = parity to wait for on bar[w]
    // lane l (1 <= l < C) of warp 0 sends this CTA's partial to the peer (crank + l) % C
    uint32_t peer_slot0 = 0, peer_bar0 = 0;
    if (wid == 0 && lane >= 1 && lane < C) {
        const uint32_t peer = (uint32_t)((crank + lane) % C);
        peer_slot0 = cluster_map(smem_u32(&sh.red[0][crank]), peer);        // red[1][crank] is 64 bytes further
        peer_bar0 = cluster_map(bar0, peer);
    }
    // broadcast loads of 16 doubles + a depth-4 tree: shorter than a shuffle tree, same order in every thread
    auto sum16 = [&](const double* w) -> double {
        const double2* w2 = reinterpret_cast<const double2*>(w);
        double t[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { const double2 v = w2[i]; t[i] = v.x + v.y; }
        return ((t[0] + t[1]) + (t[2] + t[3])) + ((t[4] + t[5]) + (t[6] + t[7]));
    };
    // boundary rows of the strip for the neighbour's copy of p: r plus the correction of the intermediate level (e1 = 0
    // without it), which the neighbour cannot know; it adds the coarse correction itself
    const bool colok0 = 2 * q >= 1 && 2 * q <= Kact - 2, colok1 = 2 * q + 1 <= Kact - 2;    // interior columns of this thread
    auto push_rows = [&](double e1 = 0.0) {
        const double e1a = colok0 ? e1 : 0.0, e1b = colok1 ? e1 : 0.0;          // boundary / padding columns carry no correction
        if (first_group) st_async_f64x2(push_n_addr, r[0][0] + e1a, r[0][1] + e1b, push_n_bar);
        if (last_group) st_async_f64x2(push_s_addr, r[3][0] + e1a, r[3][1] + e1b, push_s_bar);
    };
    // part -> warp sum -> block sum -> every CTA of the cluster.  Every stage is a fixed xor-shuffle tree, identical in
    // every warp of every CTA, so all threads of the cluster see bit-identical sums and take identical decisions.
    // Restriction P^T r of the coarse level, riding on the r.r exchange: tile sum -> segment of HQ lanes (the tiles of one
    // aggregate in this row group) -> `stage`; after the barrier one thread per owned aggregate adds its HG row groups
    // and delivers the entry to every CTA (st.async also to itself, so the mbarrier orders all of it).
    auto restrict_stage = [&](double ts) {
#pragma unroll
        for (int o = 1; o < CG.HQ; o <<= 1) ts += __shfl_xor_sync(0xffffffffu, ts, o);
        if (active && (q % CG.HQ) == 0) stage[g * CG.NCC + (2 * q) / CG.H] = ts;
    };
    auto restrict_send = [&]() {
        const int rt = tid - 32;                         // warps 1.. : warp 0 is busy with the r.r partial
        if (rt >= 0 && rt < ARL * CG.NCC) {
            const int arl = rt / CG.NCC, ac = rt - arl * CG.NCC, ar = crank * ARL + arl;
            if (ar < CG.NCR) {
                double v = 0.0;
#pragma unroll
                for (int gg = 0; gg < CG.HG; ++gg) {
                    const int gl = arl * CG.HG + gg;
                    if (gl < G) v += stage[gl * CG.NCC + ac];
                }
                const int ag = ar * CG.NCC + ac;
                if (CLUSTER) {
                    const uint32_t dst = smem_u32(rcv + cpos(ag));
                    for (int c = 0; c < C; ++c) st_async_f64(cluster_map(dst, (uint32_t)c), v, cluster_map(bar0, (uint32_t)c));
                } else {
                    rcv[cpos(ag)] = v;
                }
            }
        }
    };
    auto reduce_send = [&](double v, int which, bool coarse = false, double ts = 0.0) {
        v = warp_sum_mma(v);
        if (lane == 0) sh.wsum[which][wid] = v;
        if (COARSE && coarse) restrict_stage(ts);
        __syncthreads();
        if (COARSE && coarse) restrict_send();
        if (CLUSTER) {
            if (wid == 0) {
                const double b = sum16(sh.wsum[which]);
                if (lane == 0) {
                    sh.red[which][crank] = b;
                    mbar_expect_tx(bar0 + 8 * which, which == 0 ? expect0 : expect1);
                } else if (lane < C) {
                    st_async_f64(peer_slot0 + 64 * which, b, peer_bar0 + 8 * which);
                }
            }
        }
    };
    auto reduce_wait = [&](int which) -> double {
        if (CLUSTER) {
            mbar_wait(bar0 + 8 * which, (phase >> which) & 1u);
            phase ^= 1u << which;
            const double2* rr2 = reinterpret_cast<const double2*>(sh.red[which]);      // unused slots stay zero
            const double2 a = rr2[0], b = rr2[1];
            if (C <= 4) return (a.x + a.y) + (b.x + b.y);
            const double2 c = rr2[2], d = rr2[3];
            return ((a.x + a.y) + (b.x + b.y)) + ((c.x + c.y) + (d.x + d.y));
        }
        return sum16(sh.wsum[which]);
    };

    // thread-constant shared-memory bases: everything in the loop is base + immediate
    double* const pe_t = pe + lr * KH + q;              // own tile, row a: pe_t[a * KH]
    double* const po_t = po + lr * KH + q;
    const int dqw = qw - q, dqe = qe - q;               // -1 / +1, or 0 at the domain boundary (the face weight is 0 there)

    // ec = Ac^-1 rc by every CTA; returns rc.ec and leaves this tile's (and the halo rows') corrections in ect / ecn / ecs
    double ect = 0.0, ecn = 0.0, ecs = 0.0;
    auto coarse_apply = [&]() -> double {
        if (!CLUSTER) __syncthreads();                   // rcv was written with plain stores
        if (tid < 64 * PARTS) {
            const int part_ = tid % PARTS;
            double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
            for (int jj = 0; jj < JP; jj += 2) {
                acc0 = fma(Ainv[jj * (64 * PARTS) + tid], rcv[jj * PARTS + part_], acc0);
                acc1 = fma(Ainv[(jj + 1) * (64 * PARTS) + tid], rcv[(jj + 1) * PARTS + part_], acc1);
            }
            double acc = acc0 + acc1;
#pragma unroll
            for (int o = 1; o < PARTS; o <<= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (part_ == 0) ec[cpos(tid / PARTS)] = acc;
        }
        __syncthreads();
        const double qv = fma(rcv[lane], ec[lane], rcv[lane + 32] * ec[lane + 32]);
        ect = active ? ec[cpos(a_own)] : 0.0;
        ecn = first_group ? ec[cpos(a_own - CG.NCC)] : 0.0;
        ecs = last_group ? ec[cpos(a_own + CG.NCC)] : 0.0;
        return warp_sum_mma(qv);
    };
    auto tile_sum = [&]() -> double {
        return ((r[0][0] + r[0][1]) + (r[1][0] + r[1][1])) + ((r[2][0] + r[2][1]) + (r[3][0] + r[3][1]));
    };

    // intermediate level: r1 = sum of r over the tile pair, e1 = r1 / d1, and r1 e1 (half from each lane) joins r.r
    double e1 = 0.0, ts0 = 0.0;
    auto pair_level = [&](double& acc) {
        ts0 = tile_sum();
        const double r1 = ts0 + __shfl_xor_sync(0xffffffffu, ts0, 1);
        e1 = r1 * inv_d1;
        acc = fma(0.5 * r1, e1, acc);
    };
    if (COARSE && use_coarse) pair_level(part);
    push_rows(e1);
    reduce_send(part, 0, use_coarse, ts0);
    double rr = reduce_wait(0);
    if (COARSE && use_coarse) rr += coarse_apply();
    const double rr0 = rr;
    double beta = 0.0;
    int it = 0;
    auto flip = [&](double v, int node) -> double {          // sigma_node * v
        return __hiloint2double(__double2hiint(v) ^ (int)(((negmask >> node) & 1u) << 31), __double2loint(v));
    };
    auto iterate = [&](auto tag) {
        constexpr bool SIGNED = decltype(tag)::value;
        constexpr bool CO = COARSE && !SIGNED;           // the coarse correction is never combined with the sign handling
        double nwl[4] = {0.0, 0.0, 0.0, 0.0}, nwr[4] = {0.0, 0.0, 0.0, 0.0};
        if (active) {
#pragma unroll
            for (int a = 0; a < 4; ++a) { nwl[a] = we_t[a * (KH + 1)]; nwr[a] = we_t[a * (KH + 1) + 1]; }
        }
        for (it = 0; it < max_iter; ++it) {
            // ---- p = r + beta p (own tile and this CTA's copies of the neighbouring rows)
            if (active) {
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    // z = r + P ec; P has no entries on boundary / padding nodes (their r, p stay exactly 0)
                    p[a][0] = fma(beta, p[a][0], CO ? r[a][0] + (((okmask >> (2 * a)) & 1u) ? ect + e1 : 0.0) : r[a][0]);
                    p[a][1] = fma(beta, p[a][1], CO ? r[a][1] + (((okmask >> (2 * a + 1)) & 1u) ? ect + e1 : 0.0) : r[a][1]);
                    pe_t[a * KH] = p[a][0];
                    po_t[a * KH] = p[a][1];
                }
                if (first_group) {
                    const double2 z = *reinterpret_cast<const double2*>(zh + 2 * q);
                    pe[q] = fma(beta, pe[q], CO ? z.x + (colok0 ? ecn : 0.0) : z.x);
                    po[q] = fma(beta, po[q], CO ? z.y + (colok1 ? ecn : 0.0) : z.y);
                }
                if (last_group) {
                    const double2 z = *reinterpret_cast<const double2*>(zh + K + 2 * q);
                    pe_t[4 * KH] = fma(beta, pe_t[4 * KH], CO ? z.x + (colok0 ? ecs : 0.0) : z.x);
                    po_t[4 * KH] = fma(beta, po_t[4 * KH], CO ? z.y + (colok1 ? ecs : 0.0) : z.y);
                }
            }
            __syncthreads();
            // ---- ap = A^ p = sigma p + sum nw p_neighbour ; two accumulators for p.Ap
            double ap[4][2];
            double part0 = 0.0, part1 = 0.0, part2 = 0.0, part3 = 0.0;
            if (active) {
                const double n0 = pe_t[-KH], n1 = po_t[-KH];
                const double s0 = pe_t[4 * KH], s1 = po_t[4 * KH];
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const double pw = po_t[a * KH + dqw];
                    const double pE = pe_t[a * KH + dqe];
                    const double up0 = a == 0 ? n0 : p[a - 1][0], up1 = a == 0 ? n1 : p[a - 1][1];
                    const double dn0 = a == 3 ? s0 : p[a + 1][0], dn1 = a == 3 ? s1 : p[a + 1][1];
                    double v0 = fma(wv[a][0], up0, SIGNED ? flip(p[a][0], 2 * a) : p[a][0]);
                    double v1 = fma(wv[a][1], up1, SIGNED ? flip(p[a][1], 2 * a + 1) : p[a][1]);
                    v0 = fma(wv[a + 1][0], dn0, v0);
                    v1 = fma(wv[a + 1][1], dn1, v1);
                    v0 = fma(nwl[a], pw, v0);
                    v1 = fma(wi[a], p[a][0], v1);
                    v0 = fma(wi[a], p[a][1], v0);
                    v1 = fma(nwr[a], pE, v1);
                    ap[a][0] = v0;
                    ap[a][1] = v1;
                    if (a & 1) {
                        part2 = fma(p[a][0], v0, part2);
                        part3 = fma(p[a][1], v1, part3);
                    } else {
                        part0 = fma(p[a][0], v0, part0);
                        part1 = fma(p[a][1], v1, part1);
                    }
                }
            } else {
#pragma unroll
                for (int a = 0; a < 4; ++a) ap[a][0] = ap[a][1] = 0.0;
            }
            reduce_send((part0 + part1) + (part2 + part3), 1);
            const double inv_rr = fast_rcp(rr);                 // for beta; off the critical path (overlaps the round trip)
            const double pap = reduce_wait(1);
            const double alpha = rr * fast_rcp(pap);
            part0 = part1 = part2 = part3 = 0.0;
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                r[a][0] = fma(-alpha, SIGNED ? flip(ap[a][0], 2 * a) : ap[a][0], r[a][0]);
                r[a][1] = fma(-alpha, SIGNED ? flip(ap[a][1], 2 * a + 1) : ap[a][1], r[a][1]);
                if (a & 1) {
                    part2 = fma(SIGNED ? flip(r[a][0], 2 * a) : r[a][0], r[a][0], part2);
                    part3 = fma(SIGNED ? flip(r[a][1], 2 * a + 1) : r[a][1], r[a][1], part3);
                } else {
                    part0 = fma(SIGNED ? flip(r[a][0], 2 * a) : r[a][0], r[a][0], part0);
                    part1 = fma(SIGNED ? flip(r[a][1], 2 * a + 1) : r[a][1], r[a][1], part1);
                }
            }
            if (CO && use_coarse) pair_level(part0);
            push_rows(CO ? e1 : 0.0);
            reduce_send((part0 + part1) + (part2 + part3), 0, CO && use_coarse, CO ? ts0 : 0.0);
            if (active) {           // next iteration's outer face weights: `ap` is dead, so this costs no registers
#pragma unroll
                for (int a = 0; a < 4; ++a) { nwl[a] = we_t[a * (KH + 1)]; nwr[a] = we_t[a * (KH + 1) + 1]; }
            }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 2; ++b) x[a][b] = fma(alpha, p[a][b], x[a][b]);     // overlaps the round trip
            double rr_new = reduce_wait(0);
            if (CO && use_coarse) rr_new += coarse_apply();         // r.M^-1 r = r.r + rc.ec
            if (rr_new <= tol2 * rr0) { ++it; break; }
            beta = rr_new * inv_rr;
            rr = rr_new;
        }
    };
    if (rr0 > 0.0) {
        if (cta_signed) iterate(std::true_type{});
        else iterate(std::false_type{});
    }
    // ---- nodal pressure = s * x^ (boundary stays zero: the buffer is cleared beforehand)
    if (active) {
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            const int row = i0 + a;
            if (row <= Kact - 2 && 2 * q < Kact) {
                double* out = pn + (size_t)member * Kact * ldk + (size_t)row * ldk + 2 * q;     // ldk is even: 16-byte aligned
                const double v0 = se[(lr + a) * KH + q] * x[a][0], v1 = so[(lr + a) * KH + q] * x[a][1];
                if (2 * q + 1 < Kact) *reinterpret_cast<double2*>(out) = make_double2(v0, v1);
                else out[0] = v0;
            }
        }
    }
    if (tid == 0 && crank == 0) {
        atomicMax(iters_out, it);
        atomicAdd(iters_out + 1, it);           // total over the batch (statistics)
    }
    if (CLUSTER) cluster.sync();              // no CTA may exit while a neighbour can still touch its shared memory
}

// G[o, col0 + m] = P[m, obs[o]]  (n_obs rows) -- or, with obs == nullptr, the full transposed field.
// (fields are N x N with row pitch ldn, `cells` = N * ldn doubles per member; cell indices are row-major over N x N)
__global__ void __launch_bounds__(256) darcy_gather_kernel(const double* __restrict__ P, long long cells, int members,
                                                           const long long* __restrict__ obs, int rows,
                                                           double* __restrict__ G, long long ldg, int N, int ldn) {
    const int m = blockIdx.x * 256 + threadIdx.x;
    const int o = blockIdx.y;
    if (m >= members) return;
    const long long cell = obs ? obs[o] : o;
    const long long r = cell / N, c = cell - r * N;
    G[(size_t)o * ldg + m] = P[(size_t)m * cells + r * ldn + c];
}

struct DarcyModel {
    int N = 0, p = 0, n_obs = 0;
    int Kt = 0;                     // template grid of the solver: 2 * round_up(ceil(N / 2), 8) >= N
    int ldn = 0;                    // row pitch of every N x N field: round_up(N, 2) (TMA operands need an even pitch)
    int tile_C = 1, tile_G = 0;     // solver: cluster size and row groups (of 4 rows) per CTA
    bool coarse = false;            // two-level preconditioner (aggregates aligned with tiles and strips)
    int64_t chunk = 0;
    cudaStream_t st = nullptr;
    double *PhiT = nullptr, *S = nullptr, *S2 = nullptr, *B0 = nullptr, *B1 = nullptr, *B2 = nullptr, *Upad = nullptr;
    long long* obs = nullptr;
    int* iters = nullptr;           // [0] largest, [1] summed CG iteration count of the last forward call
    std::vector<cudaEvent_t> ev;    // start/stop pairs around the solver launches of the last forward call
    int ev_used = 0;
    long long last_members = 0;
    int64_t upad_cols = 0;
};

static int pcg_tile_launch(DarcyModel* m, const double* cn, double* pn, int members, double tol, int max_iter) {
    const int K = m->Kt, KH = K / 2, R = 4 * m->tile_G;
    const size_t smem = ((size_t)4 * (R + 2) * KH + (size_t)R * (KH + 1) + 2 * K + (m->coarse ? COARSE_SMEM_DOUBLES : 0)) * sizeof(double);
    typedef void (*TileKernel)(const double*, double*, int, double, int, int*, int, int);
#define CES_TILE_ROW(CL, CO)                                                                                              \
    darcy_pcg_tile_kernel<8, CL, CO>, darcy_pcg_tile_kernel<16, CL, CO>, darcy_pcg_tile_kernel<24, CL, CO>,               \
        darcy_pcg_tile_kernel<32, CL, CO>, darcy_pcg_tile_kernel<40, CL, CO>, darcy_pcg_tile_kernel<48, CL, CO>,          \
        darcy_pcg_tile_kernel<56, CL, CO>, darcy_pcg_tile_kernel<64, CL, CO>
    static const TileKernel table[32] = {CES_TILE_ROW(false, false), CES_TILE_ROW(true, false), CES_TILE_ROW(false, true),
                                         CES_TILE_ROW(true, true)};
#undef CES_TILE_ROW
    static size_t configured[kMaxDevices][32] = {};
    const int slot = K / 16 - 1 + (m->tile_C > 1 ? 8 : 0) + (m->coarse ? 16 : 0);
    const TileKernel kernel = table[slot];
    size_t& conf = configured[device_slot()][slot];
    if (smem > conf) {
        CES_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        conf = smem;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(members * m->tile_C));
    cfg.blockDim = dim3((unsigned)round_up((int64_t)m->tile_G * KH, 32));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = m->st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)m->tile_C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CES_CUDA(cudaLaunchKernelEx(&cfg, kernel, cn, pn, m->tile_G, tol * tol, max_iter, m->iters, m->N, m->ldn));
    CES_LAUNCHED(1);
    return CES_OK;
}

}  // namespace ces

using namespace ces;

extern "C" {

int ces_darcy_create(int64_t N, int64_t p, const double* PhiT_host, const double* S_host, const double* S2_host,
                     const int64_t* obs_host, int64_t n_obs, void* stream, void** out) {
    if (!out) return fail(CES_ERR_INVALID, "ces_darcy_create: null output%s", "");
    *out = nullptr;
    if (N < 4 || N > 128 || p < 1 || p > N * N || !PhiT_host || !S_host || !S2_host || n_obs < 0 || (n_obs > 0 && !obs_host))
        return fail(CES_ERR_INVALID, "ces_darcy_create: needs 4 <= N <= 128 and 1 <= p <= N^2%s", "");
    for (int64_t o = 0; o < n_obs; ++o)
        if (obs_host[o] < 0 || obs_host[o] >= N * N) return fail(CES_ERR_INVALID, "ces_darcy_create: obs_index out of range%s", "");
    DarcyModel* m = new DarcyModel();
    m->N = (int)N; m->p = (int)p; m->n_obs = (int)n_obs;
    m->ldn = (int)round_up(N, 2);
    m->Kt = 2 * (int)round_up((N + 1) / 2, 8);             // the solver is instantiated for grids that are multiples of 16
    m->st = static_cast<cudaStream_t>(stream);
    {   // NG row groups of 4 interior rows over C CTAs, G per CTA, G * Kt/2 threads <= TILE_THREADS.  The coarse level
        // needs strips that end on aggregate boundaries (G a multiple of H/4 in a cluster) and >= 64 * parts threads for
        // the 64 x 64 coarse solve: the smallest cluster that can have it is taken, else the smallest cluster at all.
        const int NG = (int)((N - 2 + 3) / 4), KH = m->Kt / 2;
        const CoarseGeom cgm = coarse_geom(m->Kt);
        const bool pow2 = (cgm.HQ & (cgm.HQ - 1)) == 0;
        bool want_coarse = true;
        if (const char* e = getenv("CES_DARCY_COARSE")) want_coarse = atoi(e) != 0;      // experiments: 0 disables
        int forced = 0;
        if (const char* e = getenv("CES_DARCY_CLUSTER")) forced = atoi(e);              // experiments: a given cluster size
        int tc_plain = 0, g_plain = 0;
        m->tile_C = 0;
        for (int tc = 1; tc <= 8 && m->tile_C == 0; ++tc) {
            if (forced >= 1 && forced <= 8 && tc != forced) continue;
            const int g0 = (NG + tc - 1) / tc;
            if (g0 * KH > TILE_THREADS) continue;
            if (!tc_plain) { tc_plain = tc; g_plain = g0; }
            const int parts = coarse_parts(KH, tc > 1);
            const int gc = tc > 1 ? (int)round_up(g0, cgm.HG) : g0;
            const int threads = (int)round_up((int64_t)gc * KH, 32);
            if (want_coarse && pow2 && parts >= 2 && gc * KH <= TILE_THREADS && threads >= 64 * parts) {
                m->tile_G = gc;
                m->tile_C = (NG + gc - 1) / gc;            // rounding G up may leave the last CTA without rows: drop it
                m->coarse = true;
            }
        }
        if (m->tile_C == 0) {
            if (!tc_plain) { delete m; return fail(CES_ERR_INVALID, "ces_darcy_create: no launch shape for this grid%s", ""); }
            m->tile_C = tc_plain; m->tile_G = g_plain; m->coarse = false;
        }
    }
    const int64_t cells = N * m->ldn;              // doubles per stored field (row pitch ldn)
    m->chunk = (1ll << 29) / (cells * 8);          // 512 MiB per field buffer
    if (m->chunk > 32768) m->chunk = 32768;
    if (m->chunk < 64) m->chunk = 64;
    // constant operators, re-packed to the even row pitch (zero padding): Phi^T p x (N x ldn), S and S2 N x ldn
    auto up2d = [&](double** dst, const double* src, int64_t rows, int64_t width, int64_t pitch) -> int {
        CES_CUDA(cudaMalloc(dst, rows * pitch * sizeof(double)));
        CES_CUDA(cudaMemsetAsync(*dst, 0, rows * pitch * sizeof(double), m->st));
        CES_CUDA(cudaMemcpy2DAsync(*dst, pitch * sizeof(double), src, width * sizeof(double), width * sizeof(double), rows,
                                   cudaMemcpyHostToDevice, m->st));
        return CES_OK;
    };
    int s = up2d(&m->PhiT, PhiT_host, p * N, N, m->ldn);
    if (s == CES_OK) s = up2d(&m->S, S_host, N, N, m->ldn);
    if (s == CES_OK) s = up2d(&m->S2, S2_host, N, N, m->ldn);

    if (s == CES_OK && n_obs > 0) {
        if (cudaMalloc(&m->obs, n_obs * sizeof(long long)) != cudaSuccess) s = fail(CES_ERR_NOMEM, "cudaMalloc failed%s", "");
        else if (cudaMemcpyAsync(m->obs, obs_host, n_obs * sizeof(long long), cudaMemcpyHostToDevice, m->st) != cudaSuccess)
            s = fail(CES_ERR_CUDA, "obs upload failed%s", "");
    }
    if (s == CES_OK && cudaMalloc(&m->iters, 2 * sizeof(int)) != cudaSuccess) s = fail(CES_ERR_NOMEM, "cudaMalloc failed%s", "");
    if (s == CES_OK && cudaStreamSynchronize(m->st) != cudaSuccess) s = fail(CES_ERR_CUDA, "ces_darcy_create: upload failed%s", "");
    if (s != CES_OK) { ces_darcy_destroy(m); return s; }
    *out = m;
    return CES_OK;
}

int ces_darcy_destroy(void* handle) {
    DarcyModel* m = static_cast<DarcyModel*>(handle);
    if (!m) return CES_OK;
    cudaStreamSynchronize(m->st);
    cudaFree(m->PhiT); cudaFree(m->S); cudaFree(m->S2); cudaFree(m->B0); cudaFree(m->B1); cudaFree(m->B2);
    cudaFree(m->Upad); cudaFree(m->obs); cudaFree(m->iters);
    for (cudaEvent_t e : m->ev) cudaEventDestroy(e);
    delete m;
    cudaGetLastError();
    return CES_OK;
}

}  // extern "C"

namespace ces {

int darcy_max_iter(const DarcyModel* m, int max_iter) { return max_iter > 0 ? max_iter : 40 * m->N; }

DarcyShape darcy_shape(const DarcyModel* m) { return DarcyShape{m->N, m->p, m->n_obs, m->st, m->iters}; }

// The pipeline of ces_darcy_forward without its final synchronisation; the chains of darcy_mh.cu call it once per step.
int darcy_forward_async(DarcyModel* m, const double* U, int64_t ldu, int64_t cols, double* G, int64_t ldg, int full_solution,
                        double tol, int max_iter) {
    if (cols == 0) return CES_OK;
    const int N = m->N, p = m->p, ldn = m->ldn;
    const int64_t cells = (int64_t)N * ldn;        // doubles per stored field
    cudaStream_t st = m->st;
    if (tol <= 0.0) tol = 1e-13;
    max_iter = darcy_max_iter(m, max_iter);
    const int64_t chunk = cols < m->chunk ? cols : m->chunk;
    if (!m->B0) {
        const size_t bytes = (size_t)m->chunk * cells * sizeof(double);
        if (cudaMalloc(&m->B0, bytes) != cudaSuccess || cudaMalloc(&m->B1, bytes) != cudaSuccess ||
            cudaMalloc(&m->B2, bytes) != cudaSuccess) {
            cudaGetLastError();
            return fail(CES_ERR_NOMEM, "ces_darcy_forward: workspace allocation failed%s", "");
        }
    }
    // the KL GEMM reads U^T through TMA: 16-byte aligned base and even pitch, else re-pack once
    const double* Uuse = U;
    int64_t ldu_use = ldu;
    if ((reinterpret_cast<uintptr_t>(U) & 15) != 0 || (ldu & 1)) {
        const int64_t ldp = padded_ld(cols);
        if (m->upad_cols < ldp) {
            cudaFree(m->Upad);
            m->Upad = nullptr;
            if (cudaMalloc(&m->Upad, (size_t)p * ldp * sizeof(double)) != cudaSuccess) return fail(CES_ERR_NOMEM, "cudaMalloc failed%s", "");
            m->upad_cols = ldp;
        }
        CES_TRY(pad_copy(st, U, ldu, p, cols, m->Upad, ldp));
        Uuse = m->Upad; ldu_use = ldp;
    }
    CES_CUDA(cudaMemsetAsync(m->iters, 0, 2 * sizeof(int), st));
    m->ev_used = 0;
    m->last_members = cols;
    for (int64_t c0 = 0; c0 < cols; c0 += chunk) {
        const int64_t mc = (cols - c0) < chunk ? (cols - c0) : chunk;
        if (c0 % 2 != 0) return fail(CES_ERR_ALIGN, "ces_darcy_forward: odd chunk offset%s", "");
        // 1. Theta = U^T Phi^T  (mc x cells)
        GemmCall g;
        g.a_mode = A_KM; g.b_mode = B_KN;
        g.M = (int)mc; g.N = (int)cells; g.K = p;
        g.A = Uuse + c0; g.lda = ldu_use; g.B = m->PhiT; g.ldb = cells; g.C = m->B0; g.ldc = cells;
        CES_TRY(gemm(st, g));
        // 2. a = exp(Theta)
        CES_TRY(exp_map(st, m->B0, cells, mc, cells, m->B0, cells));
        // 3. T1 = a S^T (stacked rows), c_z = S T1_z
        GemmCall t1;
        t1.a_mode = A_MK; t1.b_mode = B_NK;
        t1.M = (int)(mc * N); t1.N = N; t1.K = N;
        t1.A = m->B0; t1.lda = ldn; t1.B = m->S; t1.ldb = ldn; t1.C = m->B1; t1.ldc = ldn;
        CES_TRY(gemm(st, t1));
        GemmCall cz;
        cz.a_mode = A_MK; cz.b_mode = B_KN;
        cz.M = N; cz.N = N; cz.K = N;
        cz.A = m->S; cz.lda = ldn; cz.B = m->B1; cz.ldb = ldn; cz.C = m->B2; cz.ldc = ldn;
        cz.batch = mc; cz.b_batch_rows = N; cz.c_batch_elems = cells;
        CES_TRY(gemm(st, cz));
        // 4. solve; nodal pressure into B0 (cleared: boundary nodes stay zero)
        CES_CUDA(cudaMemsetAsync(m->B0, 0, (size_t)mc * cells * sizeof(double), st));
        while ((int)m->ev.size() < m->ev_used + 2) {
            cudaEvent_t e;
            CES_CUDA(cudaEventCreate(&e));
            m->ev.push_back(e);
        }
        CES_CUDA(cudaEventRecord(m->ev[m->ev_used], st));
        CES_TRY(pcg_tile_launch(m, m->B2, m->B0, (int)mc, tol, max_iter));
        CES_CUDA(cudaEventRecord(m->ev[m->ev_used + 1], st));
        m->ev_used += 2;
        // 5. back to the cell centres: T2 = p S2^T, P_z = S2 T2_z
        GemmCall t2 = t1;
        t2.A = m->B0; t2.B = m->S2; t2.C = m->B1;
        CES_TRY(gemm(st, t2));
        GemmCall pz = cz;
        pz.A = m->S2; pz.B = m->B1; pz.C = m->B2;
        CES_TRY(gemm(st, pz));
        // 6. observations (or the whole field), particle index contiguous
        const int rows = full_solution ? N * N : m->n_obs;
        dim3 grid((unsigned)ceil_div(mc, 256), (unsigned)rows);
        darcy_gather_kernel<<<grid, 256, 0, st>>>(m->B2, cells, (int)mc, full_solution ? nullptr : m->obs, rows, G + c0, ldg, N, ldn);
        CES_LAUNCHED(1);
    }
    return CES_OK;
}

}  // namespace ces

extern "C" {

int ces_darcy_forward(void* handle, const double* U, int64_t ldu, int64_t cols, double* G, int64_t ldg, int full_solution,
                      double tol, int max_iter, int* iters_host) {
    DarcyModel* m = static_cast<DarcyModel*>(handle);
    if (!m || !U || !G || cols < 0 || ldu < cols || ldg < cols) return fail(CES_ERR_INVALID, "ces_darcy_forward: bad argument%s", "");
    if (!full_solution && m->n_obs == 0) return fail(CES_ERR_STATE, "ces_darcy_forward: no obs_index was given%s", "");
    if (cols == 0) return CES_OK;
    CES_TRY(darcy_forward_async(m, U, ldu, cols, G, ldg, full_solution, tol, max_iter));
    max_iter = darcy_max_iter(m, max_iter);
    cudaStream_t st = m->st;
    int iters = 0;
    CES_CUDA(cudaMemcpyAsync(&iters, m->iters, sizeof(int), cudaMemcpyDeviceToHost, st));
    CES_CUDA(cudaStreamSynchronize(st));
    if (iters_host) *iters_host = iters;
    if (iters >= max_iter) return fail(CES_ERR_STATE, "ces_darcy_forward: CG did not converge in %s%lld iterations", "", max_iter);
    return CES_OK;
}

int ces_darcy_last_stats(void* handle, int64_t* members, int64_t* total_iterations, double* solver_ms) {
    DarcyModel* m = static_cast<DarcyModel*>(handle);
    if (!m) return fail(CES_ERR_INVALID, "ces_darcy_last_stats: null model%s", "");
    int it[2] = {0, 0};
    CES_CUDA(cudaStreamSynchronize(m->st));
    CES_CUDA(cudaMemcpy(it, m->iters, 2 * sizeof(int), cudaMemcpyDeviceToHost));
    double ms = 0.0;
    for (int i = 0; i + 1 < m->ev_used; i += 2) {
        float t = 0.f;
        CES_CUDA(cudaEventElapsedTime(&t, m->ev[i], m->ev[i + 1]));
        ms += t;
    }
    if (members) *members = m->last_members;
    if (total_iterations) *total_iterations = it[1];
    if (solver_ms) *solver_ms = ms;
    return CES_OK;
}

}  // extern "C"
