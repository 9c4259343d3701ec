"""Exact-arithmetic contract of the FP64 DMMA GEMM family (ces_gemm_ex) and of the blocked Cholesky, solve and inverse
built on it.

GEMM cases use small integer operands ({-4..4}) and alpha, beta in {1, 2, -1/2}: every product and partial sum is then
exactly representable, so the device result must EQUAL the numpy int64 reference whatever the summation order, split or
walk direction -- a wrong row, column, k-block, batch offset or mirror is a nonzero difference, not something a tolerance
absorbs.  Operands sit inside wider buffers poisoned with NaN (rows above and below, columns left and right); C sits inside
a sentinel bit pattern that must survive bit for bit.  Shapes cross the 64 / 128-row tiles, the 128-column tiles, the
16-wide k-blocks and the 5-stage ring (80 = 5 x 16)."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ces_b200 import _lib  # noqa: E402

U64 = 2.0 ** -53
SENTINEL = 0x7FFCDEAD0000BEEF          # a quiet NaN with a payload no kernel produces
A_MK, A_KM, B_KN, B_NK = 0, 1, 0, 1
LOWER_A, LOWER_C, UPPER_B = 1, 2, 4
LAYOUTS = [(A_MK, B_KN), (A_KM, B_KN), (A_MK, B_NK), (A_KM, B_NK)]
NAN = float("nan")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _ints(rng, shape, lo=-4, hi=4):
    return rng.integers(lo, hi + 1, size=shape).astype(np.float64)


class Buf:
    """`vals` (rows x cols) inside a wider device buffer: `top` rows above, `bottom` below, `left` columns to the left and
    at least one to the right (pitch even, base 16-byte aligned), all holding `fill` (a float, or the sentinel bits)."""

    def __init__(self, vals, fill=NAN, top=2, bottom=3, left=2):
        vals = np.asarray(vals, dtype=np.float64)
        rows, cols = vals.shape
        ld = left + cols + 1
        ld += ld % 2
        shape = (top + rows + bottom, ld)
        host = np.full(shape, fill, dtype=np.int64).view(np.float64) if isinstance(fill, int) else np.full(shape, fill)
        host[top:top + rows, left:left + cols] = vals
        self.host0 = host.copy()
        self.buf = torch.from_numpy(host).cuda()
        self.view = self.buf[top:top + rows, left:left + cols]
        self.ld, self.rows, self.cols = ld, rows, cols
        self.inside = np.zeros(host.shape, dtype=bool)
        self.inside[top:top + rows, left:left + cols] = True
        assert self.ptr % 16 == 0

    @property
    def ptr(self):
        return self.view.data_ptr()

    def get(self):
        return self.view.cpu().numpy()

    def outside_intact(self):
        now = self.buf.cpu().numpy().view(np.int64)
        return np.array_equal(now[~self.inside], self.host0.view(np.int64)[~self.inside])


def gemm(am, bm, M, N, K, A, B, C, alpha=1.0, beta=0.0, **kw):
    """ces_gemm_ex on Buf operands (or raw (ptr, ld) pairs); returns the status."""
    ptr = lambda x: (x.ptr, x.ld) if isinstance(x, Buf) else x
    (pa, lda), (pb, ldb), (pc, ldc) = ptr(A), ptr(B), ptr(C)
    d = _lib.GemmDesc(a_mode=am, b_mode=bm, M=M, N=N, K=K, A=pa, lda=lda, B=pb, ldb=ldb, C=pc, ldc=ldc, alpha=alpha,
                      beta=beta, **kw)
    return _lib.load().ces_gemm_ex(_stream(), ctypes.byref(d))


def stored(op, mode, transposed_mode):
    """The stored form of a logical operand: its transpose when `mode` is the transposed layout."""
    return np.ascontiguousarray(op.T) if mode == transposed_mode else op


def explain(got, ref, A, B, alpha, bm=128, limit=6):
    """(tile row, tile column, k-block candidates) of the first differing entries: the k-blocks whose contribution
    equals the error (dropped: -1, doubled: +1)."""
    bad = np.argwhere(~(got == ref))
    out = []
    for m, n in bad[:limit]:
        err = got[m, n] - ref[m, n]
        K = A.shape[1]
        parts = [alpha * float(A[m, k0:k0 + 16] @ B[k0:k0 + 16, n]) for k0 in range(0, K, 16)]
        kbs = [(b, s) for b, p in enumerate(parts) for s in (1, -1) if p != 0 and err == s * p]
        out.append(dict(tile=(int(m) // bm, int(n) // 128), entry=(int(m), int(n)), got=float(got[m, n]),
                        ref=float(ref[m, n]), kblocks=kbs))
    return "%d differing entries, e.g. %s" % (len(bad), out)


def check_exact(tag, got, ref, A, B, alpha, failures, bm=128):
    if not np.array_equal(got, ref):
        failures.append("%s: %s" % (tag, explain(got, ref, A, B, alpha, bm)))


def run_exact(rng, am, bm, M, N, K, alpha, beta, Aop=None, Bop=None, C0=None, tag="", failures=None, AB=None, scale=1.0,
              **kw):
    """One exact GEMM on poisoned operands; appends a message to `failures` on any mismatch.  AB: the int64 product of
    Aop and Bop when the caller has it already; scale: the value behind alpha_dev."""
    Aop = _ints(rng, (M, K)) if Aop is None else Aop
    Bop = _ints(rng, (K, N)) if Bop is None else Bop
    C0 = _ints(rng, (M, N)) if C0 is None else C0
    Ab = Buf(stored(Aop, am, A_KM))
    Bb = Buf(stored(Bop, bm, B_NK))
    Cb = Buf(C0 if beta != 0 else np.full((M, N), NAN), fill=SENTINEL)
    s = gemm(am, bm, M, N, K, Ab, Bb, Cb, alpha, beta, **kw)
    if s != 0:
        failures.append("%s: status %d %s" % (tag, s, _lib.load().ces_last_error()))
        return
    AB = Aop.astype(np.int64) @ Bop.astype(np.int64) if AB is None else AB
    ref = alpha * scale * AB.astype(np.float64)
    if beta != 0:
        ref = ref + beta * C0
    check_exact(tag, Cb.get(), ref, Aop, Bop, alpha * scale, failures, 64 if M <= 64 and kw.get("batch", 1) == 1 else 128)
    if not Cb.outside_intact():
        failures.append("%s: C's surroundings changed" % tag)
    if not (Ab.outside_intact() and Bb.outside_intact()):
        failures.append("%s: an operand buffer changed" % tag)


ALPHA_BETA = [(1.0, 0.0), (2.0, 1.0), (-0.5, 2.0), (1.0, -0.5), (-0.5, 0.0)]


# ------------------------------------------------------------------------------------------------------------ layouts
@pytest.mark.parametrize("K", [1, 15, 16, 17, 80, 81, 1000])
def test_all_layouts_at_tile_fragment_and_ring_edges_are_exact(K):
    """M x N over {1, 17, 64, 65, 128, 129, 300} x {1, 16, 127, 128, 129, 257} in all four layouts: both tile variants
    (M <= 64 runs the 64-row tiles), ragged fragments, partial k-blocks, the exact 5-stage ring (K = 80) and its wrap."""
    rng = np.random.default_rng(K)
    failures = []
    i = 0
    for M in (1, 17, 64, 65, 128, 129, 300):
        Aop = _ints(rng, (M, K))
        for N in (1, 16, 127, 128, 129, 257):
            Bop, C0 = _ints(rng, (K, N)), _ints(rng, (M, N))
            prod = Aop.astype(np.int64) @ Bop.astype(np.int64)
            for am, bm in LAYOUTS:
                alpha, beta = ALPHA_BETA[i % len(ALPHA_BETA)]
                i += 1
                run_exact(rng, am, bm, M, N, K, alpha, beta, Aop, Bop, C0, "M=%d N=%d K=%d modes=%d%d a=%g b=%g"
                          % (M, N, K, am, bm, alpha, beta), failures, AB=prod)
    torch.cuda.synchronize()
    assert not failures, "\n".join(failures)


# ------------------------------------------------------------------------------------------------- raster and the walk
def test_group_m_and_serpentine_walks_are_exact_and_deterministic():
    """group_m in {1, 3, 16, > tiles_m}, serpentine on / off with waves of 1, 2 and SM-count CTAs (wave_ctas = 1 makes every
    odd CTA walk the contraction backwards), with and without split-K: bit-identical on integers; on random data every
    configuration repeated gives bit-identical results."""
    rng = np.random.default_rng(11)
    failures = []
    configs = [dict(group_m=g, serpentine=s, wave_ctas=w) for g in (1, 3, 16, 40) for s in (0, 1) for w in (1, 2, _sms())]
    for (M, N, K) in [(700, 520, 300), (40, 700, 161)]:
        Aop, Bop, C0 = _ints(rng, (M, K)), _ints(rng, (K, N)), _ints(rng, (M, N))
        prod = Aop.astype(np.int64) @ Bop.astype(np.int64)
        for am, bm in LAYOUTS:
            for cfg in configs:
                run_exact(rng, am, bm, M, N, K, 2.0, 1.0, Aop, Bop, C0, "M=%d N=%d K=%d modes=%d%d %s"
                          % (M, N, K, am, bm, cfg), failures, AB=prod, **cfg)
        for splits in (2, 3):
            ws = torch.full((splits * M * N,), NAN, dtype=torch.float64, device="cuda")
            for cfg in configs[::5]:
                run_exact(rng, A_KM, B_KN, M, N, K, -0.5, 2.0, Aop, Bop, C0, "split %d %s" % (splits, cfg), failures,
                          AB=prod, splits=splits, splitk_ws=ws.data_ptr(), splitk_ws_elems=ws.numel(), **cfg)
    # random data: a repeated call is bit-identical in every configuration
    M, N, K = 300, 260, 333
    A = Buf(rng.standard_normal((M, K)))
    B = Buf(rng.standard_normal((K, N)))
    for cfg in configs[::2]:
        outs = []
        for _ in range(2):
            C = Buf(np.full((M, N), NAN), fill=SENTINEL)
            assert gemm(A_MK, B_KN, M, N, K, A, B, C, 0.7, 0.0, **cfg) == 0
            outs.append(C.get().view(np.int64))
        if not np.array_equal(outs[0], outs[1]):
            failures.append("random data not reproducible under %s" % cfg)
    assert not failures, "\n".join(failures)


# ------------------------------------------------------------------------------------------------ triangular operands
def _tri_stored(op, read_limit, lower, mode, transposed_mode):
    """Stored form of a triangular operand whose ignored triangle is zero where the kernel reads it and NaN beyond.
    lower: op is M x K lower triangular, row tile rows [r0, r1) reads kk < read_limit(r); else op is K x N upper."""
    poisoned = op.copy()
    if lower:
        for m in range(op.shape[0]):
            poisoned[m, read_limit(m):] = NAN
    else:
        for n in range(op.shape[1]):
            poisoned[read_limit(n):, n] = NAN
    return stored(poisoned, mode, transposed_mode)


def _tri(rng, shape, lower):
    """Nonzero entries everywhere on and inside the triangle (so over-truncation is caught), zeros outside."""
    v = rng.integers(1, 5, size=shape) * rng.choice([-1, 1], size=shape)
    return (np.tril(v) if lower else np.triu(v)).astype(np.float64)


@pytest.mark.parametrize("splits", [1, 2, 3, 7])
def test_triangular_operand_flags_truncate_exactly(splits):
    """GEMM_A_LOWER_TRI / GEMM_B_UPPER_TRI read every k-block up to the end of the tile's diagonal block and none after:
    the triangle is nonzero right up to the diagonal, every entry beyond the read range is NaN, and the zeros above the
    diagonal inside the last read block stay zeros.  With split-K the later splits of the upper tiles get no k-blocks."""
    rng = np.random.default_rng(splits)
    failures = []
    for (M, N, K) in [(40, 37, 40), (64, 300, 64), (100, 37, 100), (129, 260, 129), (300, 129, 300), (515, 40, 515),
                      (100, 50, 300), (300, 70, 100)]:
        bmr = 64 if M <= 64 else 128
        lim_a = lambda m: min(K, (m // bmr + 1) * bmr)
        lim_b = lambda n: min(K, (n // 128 + 1) * 128)
        ws = torch.full((max(splits, 1) * M * N,), NAN, dtype=torch.float64, device="cuda")
        wkw = dict(splits=splits, splitk_ws=ws.data_ptr(), splitk_ws_elems=ws.numel()) if splits > 1 else {}
        for am, bm in LAYOUTS:
            La, Ub = _tri(rng, (M, K), True), _tri(rng, (K, N), False)
            Bf, Af = _ints(rng, (K, N)), _ints(rng, (M, K))
            Ap, Bp = Buf(_tri_stored(La, lim_a, True, am, A_KM)), Buf(_tri_stored(Ub, lim_b, False, bm, B_NK))
            # both flags: a CTA reads the intersection of the two ranges
            cases = [("A lower", LOWER_A, La, Bf, Ap, Buf(stored(Bf, bm, B_NK))),
                     ("B upper", UPPER_B, Af, Ub, Buf(stored(Af, am, A_KM)), Bp),
                     ("both", LOWER_A | UPPER_B, La, Ub, Ap, Bp)]
            for name, flags, Aop, Bop, Ab, Bb in cases:
                C0 = _ints(rng, (M, N))
                Cb = Buf(C0, fill=SENTINEL)
                s = gemm(am, bm, M, N, K, Ab, Bb, Cb, -0.5, 1.0, flags=flags, **wkw)
                tag = "%s M=%d N=%d K=%d modes=%d%d splits=%d" % (name, M, N, K, am, bm, splits)
                if s != 0:
                    failures.append("%s: status %d" % (tag, s))
                    continue
                ref = -0.5 * (Aop.astype(np.int64) @ Bop.astype(np.int64)) + C0
                check_exact(tag, Cb.get(), ref, Aop, Bop, -0.5, failures, bmr)
                if not Cb.outside_intact():
                    failures.append("%s: C's surroundings changed" % tag)
    assert not failures, "\n".join(failures)


# --------------------------------------------------------------------------------------------------- lower-only C
def test_lower_only_without_workspace_leaves_the_upper_tiles_alone():
    """GEMM_C_LOWER_ONLY: tiles with tn <= tm are complete (the diagonal tiles on both sides of the diagonal), every
    other tile keeps its bits."""
    rng = np.random.default_rng(3)
    failures = []
    for n, K in [(40, 33), (64, 64), (129, 17), (300, 200), (515, 81)]:
        bmr = 64 if n <= 64 else 128
        for beta in (0.0, 1.0):
            A = _ints(rng, (n, K))
            C0 = _ints(rng, (n, n))
            init = C0 if beta else np.full((n, n), SENTINEL, dtype=np.int64).view(np.float64)
            Cb = Buf(init, fill=SENTINEL)
            Ab = Buf(A)
            assert gemm(A_MK, B_NK, n, n, K, Ab, Ab, Cb, 2.0, beta, flags=LOWER_C) == 0
            got = Cb.get()
            ref = 2.0 * (A.astype(np.int64) @ A.T.astype(np.int64)) + beta * C0
            tm = np.arange(n)[:, None] // bmr
            tn = np.arange(n)[None, :] // 128
            comp = tn <= tm
            if not np.array_equal(got[comp], ref[comp]):
                failures.append("n=%d K=%d beta=%g: computed tiles wrong (%d entries)" % (n, K, beta, int((got[comp] != ref[comp]).sum())))
            if not np.array_equal(got.view(np.int64)[~comp], init.view(np.int64)[~comp]):
                failures.append("n=%d K=%d beta=%g: an upper tile was written" % (n, K, beta))
            if not Cb.outside_intact():
                failures.append("n=%d: C's surroundings changed" % n)
    assert not failures, "\n".join(failures)


def test_lower_only_with_workspace_is_the_mirrored_symmetric_result_plus_diag_add():
    """The SYRK form of C^uu / C^pp: lower tiles into the workspace, summed, mirrored, alpha / beta / diag_add applied,
    for splits in {1, 2, 3, 7, more than the k-blocks}.  The workspace starts NaN: the reduce must never read a plane
    entry of a skipped tile."""
    rng = np.random.default_rng(4)
    failures = []
    for n, K in [(40, 100), (129, 97), (300, 81)]:
        kb = -(-K // 16)
        A = _ints(rng, (n, K))
        AAt = (A.astype(np.int64) @ A.T.astype(np.int64)).astype(np.float64)
        for splits in (1, 2, 3, 7, kb + 3):
            for alpha, beta, diag in ((1.0, 0.0, 0.5), (-0.5, 2.0, 3.0), (2.0, 1.0, 0.0)):
                ws = torch.full((min(splits, kb) * n * n,), NAN, dtype=torch.float64, device="cuda")
                C0 = _ints(rng, (n, n))
                Cb = Buf(C0 if beta else np.full((n, n), NAN), fill=SENTINEL)
                Ab = Buf(A)
                s = gemm(A_MK, B_NK, n, n, K, Ab, Ab, Cb, alpha, beta, flags=LOWER_C, splits=splits, splitk_ws=ws.data_ptr(),
                         splitk_ws_elems=ws.numel(), diag_add=diag)
                tag = "n=%d K=%d splits=%d a=%g b=%g diag=%g" % (n, K, splits, alpha, beta, diag)
                if s != 0:
                    failures.append("%s: status %d" % (tag, s))
                    continue
                ref = alpha * AAt + diag * np.eye(n) + (beta * C0 if beta else 0.0)
                check_exact(tag, Cb.get(), ref, A, A.T, alpha, failures)
                if not Cb.outside_intact():
                    failures.append("%s: C's surroundings changed" % tag)
    assert not failures, "\n".join(failures)


# ------------------------------------------------------------------------------------------------------ alpha_dev
def test_alpha_dev_scales_both_epilogues():
    rng = np.random.default_rng(5)
    failures = []
    dev = torch.tensor([-0.5], dtype=torch.float64, device="cuda")
    for M, N, K in [(40, 129, 33), (300, 257, 81)]:
        ws = torch.full((3 * M * N,), NAN, dtype=torch.float64, device="cuda")
        for am, bm in LAYOUTS:
            run_exact(rng, am, bm, M, N, K, 2.0, 1.0, tag="alpha_dev direct M=%d" % M, failures=failures, scale=-0.5,
                      alpha_dev=dev.data_ptr())
            run_exact(rng, am, bm, M, N, K, 2.0, 1.0, tag="alpha_dev reduce M=%d" % M, failures=failures, scale=-0.5,
                      alpha_dev=dev.data_ptr(), splits=3, splitk_ws=ws.data_ptr(), splitk_ws_elems=ws.numel())
    assert not failures, "\n".join(failures)


# ---------------------------------------------------------------------------------------------- sum-of-squares partials
def raster(M, N, bm, group_m):
    """Linear CTA index -> (tile row, tile column) of the grouped rasterisation."""
    tiles_m, tiles_n = -(-M // bm), -(-N // 128)
    out = []
    for L in range(tiles_m * tiles_n):
        per = group_m * tiles_n
        gid = L // per
        first = gid * group_m
        gsize = min(tiles_m - first, group_m)
        r = L - gid * per
        out.append((first + r % gsize, r // gsize))
    return out


def test_sum_of_squares_partials_are_exact_per_tile_and_slot():
    """One partial per CTA and problem, at slot z * tiles + (linear CTA index): each equals the exact sum of squares of
    the values that CTA stored (beta = 1 accumulation included), every slot up to gemm_tiles(M, N) * batch is written,
    the slots after it keep their bits.  Entries in {-2..2}, K <= 256: every square and sum is exact."""
    rng = np.random.default_rng(6)
    failures = []
    for (M, N, K, batch, group_m) in [(40, 300, 200, 1, 0), (64, 129, 256, 1, 0), (300, 257, 81, 1, 0), (700, 300, 33, 1, 3),
                                      (300, 257, 100, 3, 0), (129, 200, 17, 2, 1)]:
        bmr = 64 if (M <= 64 and batch == 1) else 128
        tiles = -(-M // 128) * -(-N // 128)
        for beta in (0.0, 1.0):
            A = _ints(rng, (batch * M, K), -2, 2)
            B = _ints(rng, (K, N), -2, 2)
            C0 = _ints(rng, (batch * M, N), -2, 2)
            part = torch.full((tiles * batch + 5,), NAN, dtype=torch.float64, device="cuda")
            part0 = part.clone()
            Ab, Bb = Buf(A), Buf(B)
            Cb = Buf(C0 if beta else np.full(C0.shape, NAN), fill=SENTINEL)
            s = gemm(A_MK, B_KN, M, N, K, Ab, Bb, Cb, 1.0, beta, group_m=group_m, batch=batch, a_batch_rows=M,
                     c_batch_elems=M * Cb.ld, ssq_partials=part.data_ptr(), ssq_partials_elems=tiles * batch)
            tag = "M=%d N=%d K=%d batch=%d beta=%g" % (M, N, K, batch, beta)
            if s != 0:
                failures.append("%s: status %d" % (tag, s))
                continue
            got = part.cpu().numpy()
            ref = (A.astype(np.int64).reshape(batch, M, K) @ B.astype(np.int64)) + beta * C0.reshape(batch, M, N)
            if not np.array_equal(Cb.get(), ref.reshape(batch * M, N)):
                failures.append("%s: C wrong" % tag)
            want = np.empty(tiles * batch)
            for z in range(batch):
                for L, (tm, tn) in enumerate(raster(M, N, bmr, group_m or 16)):
                    blk = ref[z, tm * bmr:(tm + 1) * bmr, tn * 128:(tn + 1) * 128]
                    want[z * tiles + L] = float((blk.astype(np.int64) ** 2).sum())
            if not np.array_equal(got[:tiles * batch], want):
                failures.append("%s: partials %s != %s" % (tag, got[:tiles * batch][:8], want[:8]))
            if got[:tiles * batch].sum() != float((ref.astype(np.int64) ** 2).sum()):
                failures.append("%s: partials do not sum to ||C||^2" % tag)
            if not torch.equal(part.view(torch.int64)[tiles * batch:], part0.view(torch.int64)[tiles * batch:]):
                failures.append("%s: a slot past gemm_tiles * batch was written" % tag)
    assert not failures, "\n".join(failures)


# ------------------------------------------------------------------------------------------------------ batched forms
def _stack(blocks, stride_rows, gap_fill):
    """Blocks stacked every `stride_rows` rows; the gap rows hold `gap_fill`."""
    rows, cols = blocks[0].shape
    out = np.full((stride_rows * (len(blocks) - 1) + rows, cols), gap_fill)
    for z, b in enumerate(blocks):
        out[z * stride_rows:z * stride_rows + rows] = b
    return out


def test_batched_forms_one_c_per_problem_and_summed():
    """batch problems with each operand shared or batched, in every layout.  Gap rows between batches are NaN where they
    can only feed discarded outputs (rows of A_MK, B_NK), and finite junk where the last k-box reads them against the
    other operand's zero fill (rows K .. round_up(K, 16) of A_KM, B_KN)."""
    rng = np.random.default_rng(7)
    failures = []
    nb = 3
    for (M, N, K) in [(70, 200, 45), (129, 130, 64), (17, 257, 81)]:
        for am, bm in LAYOUTS:
            for a_b, b_b in ((True, False), (False, True), (True, True)):
                if am == A_KM and bm == B_KN and a_b and b_b and K % 16:
                    continue                                       # the refused hazard, below
                As = [_ints(rng, (M, K)) for _ in range(nb if a_b else 1)]
                Bs = [_ints(rng, (K, N)) for _ in range(nb if b_b else 1)]
                gap = 7
                sa = [stored(a, am, A_KM) for a in As]
                sb = [stored(b, bm, B_NK) for b in Bs]
                ra, rb = sa[0].shape[0] + gap, sb[0].shape[0] + gap
                fa = 3.0 if am == A_KM else NAN
                fb = 3.0 if bm == B_KN else NAN
                Ab, Bb = Buf(_stack(sa, ra, fa)), Buf(_stack(sb, rb, fb))
                Aop = lambda z: As[z if a_b else 0]
                Bop = lambda z: Bs[z if b_b else 0]
                ref = [(Aop(z).astype(np.int64) @ Bop(z).astype(np.int64)).astype(np.float64) for z in range(nb)]
                kw = dict(batch=nb, a_batch_rows=ra if a_b else 0, b_batch_rows=rb if b_b else 0)
                tag = "M=%d N=%d K=%d modes=%d%d batched=%s%s" % (M, N, K, am, bm, a_b, b_b)
                # one C per problem, problem z at C + z * (M + 3) rows
                C0 = _ints(rng, (nb * (M + 3), N))
                Cb = Buf(C0, fill=SENTINEL)
                s = gemm(am, bm, M, N, K, Ab, Bb, Cb, 2.0, -0.5, c_batch_elems=(M + 3) * Cb.ld, **kw)
                if s != 0:
                    failures.append("%s: status %d %s" % (tag, s, _lib.load().ces_last_error()))
                    continue
                want = C0.copy()                                   # the 3 rows after each problem stay as they were
                for z in range(nb):
                    want[z * (M + 3):z * (M + 3) + M] = 2.0 * ref[z] - 0.5 * C0[z * (M + 3):z * (M + 3) + M]
                if not np.array_equal(Cb.get(), want):
                    failures.append("%s: per-problem C wrong at rows %s" % (tag, np.unique(np.argwhere(Cb.get() != want)[:, 0])[:10]))
                # summed into one C through the workspace, with beta
                ws = torch.full((nb * M * N,), NAN, dtype=torch.float64, device="cuda")
                C1 = _ints(rng, (M, N))
                Cs = Buf(C1, fill=SENTINEL)
                s = gemm(am, bm, M, N, K, Ab, Bb, Cs, -0.5, 2.0, splitk_ws=ws.data_ptr(), splitk_ws_elems=ws.numel(), **kw)
                if s != 0 or not np.array_equal(Cs.get(), -0.5 * sum(ref) + 2.0 * C1):
                    failures.append("%s: summed C wrong (status %d)" % (tag, s))
                if not (Cb.outside_intact() and Cs.outside_intact()):
                    failures.append("%s: C's surroundings changed" % tag)
    assert not failures, "\n".join(failures)


def test_batched_hazard_of_two_contraction_row_operands_is_refused():
    """A_KM x B_KN with both operands batched and K % 16 != 0: the last k-box of problem z reads rows K .. round_up(K, 16)
    of BOTH operands from problem z + 1, and nothing zero-fills either.  The call is refused; with K % 16 == 0 it is
    exact."""
    rng = np.random.default_rng(8)
    M, N, nb = 40, 70, 3
    for K in (45, 48):
        As = [_ints(rng, (K, M)) for _ in range(nb)]
        Bs = [_ints(rng, (K, N)) for _ in range(nb)]
        Ab, Bb = Buf(np.concatenate(As)), Buf(np.concatenate(Bs))
        Cb = Buf(np.full((nb * M, N), NAN), fill=SENTINEL)
        s = gemm(A_KM, B_KN, M, N, K, Ab, Bb, Cb, batch=nb, a_batch_rows=K, b_batch_rows=K, c_batch_elems=M * Cb.ld)
        ref = np.concatenate([As[z].T.astype(np.int64) @ Bs[z].astype(np.int64) for z in range(nb)]).astype(np.float64)
        if K % 16:
            got = Cb.get()
            assert s == _lib.CES_ERR_INVALID, "accepted; exact: %s, max error %g" % (
                np.array_equal(got, ref), float(np.nanmax(np.abs(got - ref))))
            assert b"K % 16" in _lib.load().ces_last_error()
            assert Cb.outside_intact() and np.isnan(Cb.get()).all()       # no device work
        else:
            assert s == 0 and np.array_equal(Cb.get(), ref)


def test_library_gemm_configurations_restated_exactly():
    """The batched calls of the library, each with its own geometry:
    D GEMM (api.cu): D_z = (1/J) E_z^T W, A_KM with a_batch_rows = k (k % 16 != 0), W shared, the contraction in two
      chunks (k_lo > 0 accumulates with beta = 1 and leaves the sum-of-squares partials of the final D);
    multi-rank V: V = sum_z U~_z D_z (+ beta V), A_MK x B_KN both batched, summed through the workspace;
    GP prediction (emulate.cu): V_i = L_i^-1 K*_i, A lower triangular, npad-row blocks, K = n;
    Darcy c_z = S T1_z (darcy.cu): S shared, T1 batched every N rows, ld = round_up(N, 2)."""
    rng = np.random.default_rng(9)
    # --- D GEMM: E blocks (k x Jl) stacked every k rows, W (k x nc) shared, two chunks [0, 16), [16, k)
    k, Jl, nc, run = 50, 300, 257, 3
    E = _ints(rng, (run * k, Jl), -2, 2)
    W = _ints(rng, (k, nc), -2, 2)
    Eb, Wb = Buf(E), Buf(W)
    ldD = nc + 7 + (nc + 7) % 2
    D = torch.full((run * Jl * ldD,), NAN, dtype=torch.float64, device="cuda")
    tiles = -(-Jl // 128) * -(-nc // 128)
    part = torch.full((tiles * run + 3,), NAN, dtype=torch.float64, device="cuda")
    for k_lo, k_hi in ((0, 16), (16, k)):
        kw = dict(batch=run, a_batch_rows=k, c_batch_elems=Jl * ldD)
        if k_lo:
            kw.update(ssq_partials=part.data_ptr(), ssq_partials_elems=tiles * run)
        s = gemm(A_KM, B_KN, Jl, nc, k_hi - k_lo, (Eb.ptr + k_lo * Eb.ld * 8, Eb.ld), (Wb.ptr + k_lo * Wb.ld * 8, Wb.ld),
                 (D.data_ptr(), ldD), 2.0, 1.0 if k_lo else 0.0, **kw)
        assert s == 0, _lib.load().ces_last_error()
    Dh = D.view(run, Jl, ldD).cpu().numpy()
    refD = [2.0 * (E[z * k:(z + 1) * k].T.astype(np.int64) @ W.astype(np.int64)) for z in range(run)]
    for z in range(run):
        assert np.array_equal(Dh[z, :, :nc], refD[z]), "D GEMM, block %d" % z
        assert np.isnan(Dh[z, :, nc:]).all()
    assert part.cpu().numpy()[:tiles * run].sum() == sum(float((r.astype(np.int64) ** 2).sum()) for r in refD)
    # --- multi-rank V: U~ blocks (p x Jl) every p rows, D blocks (Jl x nc) every Jl rows, summed (+ V)
    p = 70
    Ut = _ints(rng, (run * p, Jl))
    Dd = _ints(rng, (run * Jl, nc))
    V0 = _ints(rng, (p, nc))
    Vb = Buf(V0, fill=SENTINEL)
    ws = torch.full((run * p * nc,), NAN, dtype=torch.float64, device="cuda")
    s = gemm(A_MK, B_KN, p, nc, Jl, Buf(Ut), Buf(Dd), Vb, 1.0, 1.0, batch=run, a_batch_rows=p, b_batch_rows=Jl,
             splitk_ws=ws.data_ptr(), splitk_ws_elems=ws.numel())
    assert s == 0
    refV = V0 + sum(Ut[z * p:(z + 1) * p].astype(np.int64) @ Dd[z * Jl:(z + 1) * Jl].astype(np.int64) for z in range(run))
    assert np.array_equal(Vb.get(), refV) and Vb.outside_intact()
    # --- GP prediction: L_i^-1 (n x n in npad x npad blocks), K*_i (n x m in npad-row blocks), one V_i per output
    n, npad, m, outs = 100, 128, 77, 3
    LI = np.full((outs * npad, npad), NAN)
    KS = np.full((outs * npad, m), NAN)
    Ls, Ks = [], []
    for i in range(outs):
        L = _tri(rng, (n, n), True)
        Kx = _ints(rng, (n, m))
        LI[i * npad:i * npad + n, :n] = L
        LI[i * npad:i * npad + n, n:] = NAN                         # columns past K: outside the map
        KS[i * npad:i * npad + n] = Kx
        KS[i * npad + n:i * npad + 112] = 5.0                       # rows K .. round_up(K, 16): read against zero fill
        Ls.append(L)
        Ks.append(Kx)
    LIb, KSb = Buf(LI), Buf(KS)
    Vg = torch.full((outs, npad, KSb.ld), NAN, dtype=torch.float64, device="cuda")
    s = gemm(A_MK, B_KN, n, m, n, LIb, KSb, (Vg.data_ptr(), KSb.ld), flags=LOWER_A, batch=outs, a_batch_rows=npad,
             b_batch_rows=npad, c_batch_elems=npad * KSb.ld)
    assert s == 0
    Vh = Vg.cpu().numpy()
    for i in range(outs):
        assert np.array_equal(Vh[i, :n, :m], Ls[i].astype(np.int64) @ Ks[i].astype(np.int64)), "GP output %d" % i
    # --- Darcy c_z = S T1_z
    N, mc = 30, 5
    ldn = N + N % 2
    S = _ints(rng, (N, N))
    T1 = [_ints(rng, (N, N)) for _ in range(mc)]
    Sd = torch.zeros((N, ldn), dtype=torch.float64, device="cuda")
    Sd[:, :N] = torch.from_numpy(S)
    T1d = torch.zeros((mc * N, ldn), dtype=torch.float64, device="cuda")
    T1d[:, :N] = torch.from_numpy(np.concatenate(T1))
    B2 = torch.full((mc * N, ldn), NAN, dtype=torch.float64, device="cuda")
    s = gemm(A_MK, B_KN, N, N, N, (Sd.data_ptr(), ldn), (T1d.data_ptr(), ldn), (B2.data_ptr(), ldn), batch=mc,
             b_batch_rows=N, c_batch_elems=N * ldn)
    assert s == 0
    B2h = B2.cpu().numpy()
    for z in range(mc):
        assert np.array_equal(B2h[z * N:(z + 1) * N, :N], S.astype(np.int64) @ T1[z].astype(np.int64)), "Darcy %d" % z


# ----------------------------------------------------------------------------------------------------- in place
def test_in_place_products_as_the_blocked_cholesky_uses_them():
    """trsm_lower's diagonal multiply writes C = B (M <= 64 or one 128-row tile, many column tiles) and potrf_lower's
    panel writes C = A (N <= 64, one column tile); every CTA reads its whole contraction before it stores.  K up to 64
    and 96 (past the 5-stage ring)."""
    rng = np.random.default_rng(10)
    failures = []
    for nb in (17, 64, 96):
        for am in (A_MK, A_KM):
            X = _tri(rng, (nb, nb), True)
            Bi = _ints(rng, (nb, 700))
            Bb = Buf(Bi)
            s = gemm(am, B_KN, nb, 700, nb, Buf(stored(X, am, A_KM)), Bb, Bb)
            want = (X.astype(np.int64) @ Bi.astype(np.int64)).astype(np.float64)
            if s != 0 or not np.array_equal(Bb.get(), want) or not Bb.outside_intact():
                failures.append("diagonal multiply nb=%d a_mode=%d" % (nb, am))
        A21 = _ints(rng, (600, nb))
        Li = _tri(rng, (nb, nb), True)
        Ab = Buf(A21)
        s = gemm(A_MK, B_NK, 600, nb, nb, Ab, Buf(Li), Ab)          # A21 Linv^T, Linv stored as given (N x K)
        want = (A21.astype(np.int64) @ Li.T.astype(np.int64)).astype(np.float64)
        if s != 0 or not np.array_equal(Ab.get(), want) or not Ab.outside_intact():
            failures.append("panel nb=%d" % nb)
    assert not failures, "\n".join(failures)


# --------------------------------------------------------------------------------------------- rounding, random data
def _mixed(rng, shape):
    return rng.standard_normal(shape) * 10.0 ** rng.uniform(-6, 6, size=shape)


@pytest.mark.parametrize("M,N,K", [(300, 257, 1000), (40, 129, 333), (129, 64, 4096)])
def test_rounding_is_componentwise_bounded_on_mixed_magnitudes(M, N, K):
    """|C - ref| <= 2 K u (|alpha| |A| |B| + |beta| |C0|) entry by entry, ref in long double, on operands whose entries
    span twelve decades and whose products cancel heavily (the second half of B's rows is the negated first half plus a
    small perturbation, so most of every sum cancels)."""
    rng = np.random.default_rng(M + N + K)
    failures = []
    A = _mixed(rng, (M, K))
    B = _mixed(rng, (K, N))
    h = K // 2
    A[:, h:2 * h] = A[:, :h]
    B[h:2 * h] = -B[:h] * (1 + 1e-9 * rng.standard_normal((h, N)))
    C0 = _mixed(rng, (M, N))
    alpha, beta = 0.7, -1.3
    ref = (np.longdouble(alpha) * (A.astype(np.longdouble) @ B.astype(np.longdouble)) + np.longdouble(beta) * C0)
    bound = 2 * K * U64 * (abs(alpha) * (np.abs(A) @ np.abs(B)) + abs(beta) * np.abs(C0))
    for am, bm in LAYOUTS:
        for kw in (dict(), dict(splits=3)):
            ws = torch.full((3 * M * N,), NAN, dtype=torch.float64, device="cuda")
            if kw:
                kw.update(splitk_ws=ws.data_ptr(), splitk_ws_elems=ws.numel())
            Cb = Buf(C0, fill=SENTINEL)
            assert gemm(am, bm, M, N, K, Buf(stored(A, am, A_KM)), Buf(stored(B, bm, B_NK)), Cb, alpha, beta, **kw) == 0
            err = np.abs(Cb.get().astype(np.longdouble) - ref).astype(np.float64)
            if not (err <= bound).all():
                r = err / np.maximum(bound, 1e-300)
                failures.append("modes=%d%d %s: %d entries over the bound, worst ratio %.3g" % (am, bm, bool(kw), int((err > bound).sum()), r.max()))
    assert not failures, "\n".join(failures)


# ------------------------------------------------------------------------------------------ Cholesky, solve, inverse
CHOL_N = [1, 2, 31, 32, 33, 63, 64, 65, 96, 127, 128, 129, 192, 193, 257, 1025]


def _spd(rng, n, cond):
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.logspace(0, -np.log10(cond), n) if n > 1 else np.ones(1)
    A = (Q * lam) @ Q.T
    return (A + A.T) / 2


def _rows_for_residual(n):
    """All rows, or for n = 1025 (a long double product of that size takes minutes) the first rows, the rows on both sides
    of the 512 block boundary and the last rows."""
    if n <= 257:
        return np.arange(n)
    return np.r_[0:33, 480:545, n - 33:n]


def _potrf(A, upper_fill=None):
    n = A.shape[0]
    host = A.copy()
    if upper_fill is not None:
        host[np.triu_indices(n, 1)] = upper_fill
    b = Buf(host)
    s = _lib.load().ces_potrf(_stream(), ctypes.c_void_p(b.ptr), b.ld, n)
    return s, b


@pytest.mark.parametrize("cond", [10.0, 1e12])
def test_cholesky_backward_error_and_the_uplo_l_contract(cond):
    """||A - L L^T|| / ||A|| <= 4 n u (long double residual), the upper triangle of the result exactly 0, and the strict
    upper triangle of the input never read: NaN there gives a bit-identical L."""
    failures = []
    for n in CHOL_N:
        rng = np.random.default_rng(n)
        A = _spd(rng, n, cond)
        s, b = _potrf(A)
        s2, b2 = _potrf(A, NAN)
        if s != 0 or s2 != 0:
            failures.append("n=%d: status %d / %d" % (n, s, s2))
            continue
        L = b.get()
        if not (L[np.triu_indices(n, 1)] == 0).all():
            failures.append("n=%d: upper triangle not zero" % n)
        if not np.array_equal(L.view(np.int64), b2.get().view(np.int64)):
            failures.append("n=%d: NaN in the upper triangle changed L" % n)
        if not (b.outside_intact() and b2.outside_intact()):
            failures.append("n=%d: the factor's surroundings changed" % n)
        rows = _rows_for_residual(n)
        Ll = L.astype(np.longdouble)
        R = (A[rows].astype(np.longdouble) - Ll[rows] @ Ll.T).astype(np.float64)
        berr = np.linalg.norm(R) / np.linalg.norm(A)
        if not berr <= 4 * n * U64:
            failures.append("n=%d cond=%g: backward error %.3g > 4 n u" % (n, cond, berr))
    assert not failures, "\n".join(failures)


def test_cholesky_reports_the_first_failing_pivot():
    """LAPACK's info: the 1-based index q of the first non-positive pivot, named in the message as `pivot q`, for a
    negative diagonal entry and for the 2 x 2 block [[1, 2], [2, 1]] at rows q-2, q-1 (Schur complement -3), which for
    q = 33 straddles the 32-column halves of a diagonal block and for q = 65, 129 a 64-block boundary, so the failure
    arises only after a GEMM trailing update."""
    lib = _lib.load()
    failures = []
    n = 200
    for q in (1, 17, 32, 33, 64, 65, 129, n):
        for kind in ("negative", "pair"):
            if kind == "pair" and q < 2:
                continue
            A = np.eye(n) * 2.0
            if kind == "negative":
                A[q - 1, q - 1] = -1.0
            else:
                A[q - 2:q, q - 2:q] = [[1.0, 2.0], [2.0, 1.0]]
            s, _ = _potrf(A)
            msg = lib.ces_last_error().decode()
            if s != _lib.CES_ERR_NOT_SPD or ("pivot %d)" % q) not in msg:
                failures.append("q=%d %s: status %d, %r" % (q, kind, s, msg))
    assert not failures, "\n".join(failures)


def test_posv_residual_and_padding():
    """||A X - B|| <= 8 n u ||A|| ||X|| (long double residual) for nrhs in {1, 16, 17, 128, 129, 300}; NaN in B's padding
    columns stays there and never reaches X."""
    lib = _lib.load()
    failures = []
    for n in (65, 193):
        rng = np.random.default_rng(n)
        A = _spd(rng, n, 1e6)
        for nrhs in (1, 16, 17, 128, 129, 300):
            B = rng.standard_normal((n, nrhs))
            Ab, Bb = Buf(A), Buf(B)
            s = lib.ces_posv(_stream(), ctypes.c_void_p(Ab.ptr), Ab.ld, n, ctypes.c_void_p(Bb.ptr), Bb.ld, nrhs)
            X = Bb.get()
            if s != 0 or not np.isfinite(X).all() or not Bb.outside_intact():
                failures.append("n=%d nrhs=%d: status %d, finite %s" % (n, nrhs, s, np.isfinite(X).all()))
                continue
            R = (A.astype(np.longdouble) @ X.astype(np.longdouble) - B).astype(np.float64)
            bound = 8 * n * U64 * np.linalg.norm(A) * np.linalg.norm(X)
            if not np.linalg.norm(R) <= bound:
                failures.append("n=%d nrhs=%d: residual %.3g > %.3g" % (n, nrhs, np.linalg.norm(R), bound))
    assert not failures, "\n".join(failures)


def test_potri_inverse_residual():
    """ces_potri: ||A A^-1 - I|| <= 8 n u ||A|| ||A^-1|| (long double), A^-1 symmetric to rounding, NaN around it kept."""
    lib = _lib.load()
    failures = []
    for n in CHOL_N:
        rng = np.random.default_rng(n + 1)
        A = _spd(rng, n, 1e6)
        Ab = Buf(A)
        Xb = Buf(np.full((n, n), NAN), fill=SENTINEL)
        s = lib.ces_potri(_stream(), ctypes.c_void_p(Ab.ptr), Ab.ld, n, ctypes.c_void_p(Xb.ptr), Xb.ld)
        X = Xb.get()
        if s != 0 or not np.isfinite(X).all() or not Xb.outside_intact():
            failures.append("n=%d: status %d" % (n, s))
            continue
        rows = _rows_for_residual(n)
        R = (A[rows].astype(np.longdouble) @ X.astype(np.longdouble)).astype(np.float64) - np.eye(n)[rows]
        bound = 8 * n * U64 * np.linalg.norm(A) * np.linalg.norm(X)
        if not np.linalg.norm(R) <= bound:
            failures.append("n=%d: residual %.3g > %.3g" % (n, np.linalg.norm(R), bound))
    Ab, Xb = Buf(-np.eye(8)), Buf(np.eye(8))
    s = lib.ces_potri(_stream(), ctypes.c_void_p(Ab.ptr), Ab.ld, 8, ctypes.c_void_p(Xb.ptr), Xb.ld)
    if s != _lib.CES_ERR_NOT_SPD or b"pivot 1)" not in lib.ces_last_error():
        failures.append("not-SPD input: status %d" % s)
    assert not failures, "\n".join(failures)


# --------------------------------------------------------------------------------------------- strided step tensors
@pytest.mark.parametrize("rule", ["aldi", "eks", "aldi_constant"])
def test_step_with_nan_neighbours_and_a_sliced_output(rule):
    """Engine.step on column slices of wider buffers whose neighbour columns are NaN on both sides, at an aligned (2) and
    an odd (3) column offset -- the odd one re-packs the noise operand --, with `out` a slice whose neighbours hold a
    sentinel: the oracle's update at 1e-10 and the sentinel bitwise unchanged."""
    from ces_b200.engine import Engine
    from oracle import eks_oracle as eo

    d, k, J = 20, 12, 101
    pr = eo.linear_gaussian_problem(d, k, J)
    o = eo.step(rule, pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], pr["xi"])
    eng = Engine(d, k, J)
    try:
        eng.set_problem(pr["y"], pr["Gamma"], pr["Sigma0"], pr["mu"], pr["ustar"])
        for off in (2, 3):
            wide = lambda a: torch.from_numpy(np.concatenate([np.full((a.shape[0], off), NAN), a,
                                                              np.full((a.shape[0], 5), NAN)], axis=1)).cuda()
            Uw, Gw, Xw = wide(pr["U0"]), wide(pr["G"]), wide(pr["xi"])
            U, G, xi = (w[:, off:off + J] for w in (Uw, Gw, Xw))
            ow = torch.from_numpy(np.full((d, off + J + 5), SENTINEL, dtype=np.int64).view(np.float64)).cuda()
            out = ow[:, off:off + J]
            res, hk, _ = eng.step(rule, U, G, xi, out=out)
            torch.cuda.synchronize()
            assert res.data_ptr() == out.data_ptr()
            got = out.cpu().numpy()
            assert float(np.abs(got - o["Uk"]).max() / np.abs(o["Uk"]).max()) < 1e-10, (rule, off)
            assert abs(hk - o["hk"]) <= 1e-10 * o["hk"], (rule, off)
            bits = ow.view(torch.int64).cpu().numpy()
            assert (bits[:, :off] == SENTINEL).all() and (bits[:, off + J:] == SENTINEL).all(), (rule, off)
            assert torch.equal(U.cpu(), torch.from_numpy(pr["U0"]))
    finally:
        eng.close()
