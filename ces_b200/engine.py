"""Per-GPU engine: owns one ``ces_handle_t`` and drives the phases of an update.

Torch is plumbing only: device buffers (``torch.Tensor`` as allocations), the
current CUDA stream and ``torch.distributed`` for the collectives between phases
when the ensemble is sharded by particle columns over several GPUs
(SURVEY.md section 8e).  All arithmetic happens in libces_b200.so.
"""
import contextlib
import ctypes
import os

import numpy as np

from . import _lib

_METRIC_KEYS = ("self-bias", "bias", "self-bias-data", "bias-data")


def shard_width(J, nranks):
    """Common (padded) shard width: every rank holds ceil(J / nranks) columns, the
    trailing ranks possibly fewer true ones."""
    return -(-J // nranks)


def shard_range(J, rank, nranks):
    w = shard_width(J, nranks)
    lo = min(J, rank * w)
    return lo, min(J, lo + w)


def run_phases(phases, buffer, comm, p, k, rule, resolve=None, formulation="interaction"):
    """One update as phases with the collectives of a column-sharded ensemble in between
    (include/ces_b200.h).  ``comm`` is None on a single GPU, else ``(dist, group, rank)``:

        sums      -> all-reduce(sum)  "sums"  (k + p doubles)            means of G and U
        centre    -> all-reduce(sum)  "cuu"   (p x ldp)                  C^uu from the local U~ U~^T
                     all-gather       "e_all", "ut_all" (rank-major)     every rank needs all of E and U~
        interact  -> all-reduce(sum)  "scalars"[0:5]                     ||D||_F^2 and the four diagnostics
        [peek -> cpp -> all-reduce(sum) "cpp" (k x ldk) -> resolve]      non-default time_step only (K11)
        drift     -> all-reduce(max)  "scalars"[5:6]                     aldi_constant only
        update

    ``formulation``: "interaction" forms D = (1/J) E^T W in panels (the reference's formulation, the default);
    "factored" computes the same V = U~ D as (1/J)(U~ E^T) W and ||D||_F through two k x k Gram matrices, with
    all-reduces of "p1", "gram_e", "gram_w" instead of the all-gathers (opt-in, see DESIGN.md).

    ``resolve``: None (default step size rule), "always" ('constant': D is formed once, with
    hk C^pp + Gamma), ``(t_last, threshold)`` ('mix': re-solve when t_last + hk > threshold,
    ces/calibrate.py:470-473), or "spectral" (hk = 1 / lambda_max(D), :249-251: the "spectral" phase sets the
    step size from the all-reduced C^pp and the update is called with the marker "spectral").  ``phases`` maps the names to callables, ``buffer(name)`` returns the torch
    tensor a collective runs on.  The engine passes the ctypes calls; tests/test_multirank_gloo.py passes a
    numpy stand-in to exercise this orchestration over gloo without a GPU."""
    if comm is not None:
        dist, group, rank = comm

        def allreduce(t, op=None):
            dist.all_reduce(t, group=group) if op is None else dist.all_reduce(t, op=op, group=group)

        def allreduce_slice(t, lo, hi, op=None):
            allreduce(t[0, lo:hi], op)        # a contiguous view: reduced in place, no staging copies
    else:
        rank = 0

        def allreduce(t, op=None):
            return None

        def allreduce_slice(t, lo, hi, op=None):
            return None

    mark = phases.get("mark", lambda name: None)      # per-phase timeline (Engine.timeline), no-op by default
    phases["sums"]()
    allreduce(buffer("sums") if comm is not None else None)
    mark("allreduce:sums:done")
    phases["centre"]()
    if formulation == "factored":
        if resolve is not None:
            raise NotImplementedError("the factored formulation supports the default step-size rule only")
        if comm is not None:
            allreduce(buffer("cuu"))
        phases["products"]()
        if comm is not None:
            for name in ("p1", "gram_e", "gram_w"):
                allreduce(buffer(name))
        phases["finish_factored"]()
    else:
        overlapped = False
        if comm is not None:
            allreduce(buffer("cuu"))
            mark("allreduce:cuu:done")
            e_all, ut_all = buffer("e_all"), buffer("ut_all")
            e_own, ut_own = e_all[rank * k:(rank + 1) * k], ut_all[rank * p:(rank + 1) * p]
            if "peer_gather" in phases and resolve != "always" and "interact_own" in phases:
                # the other ranks' blocks are pulled by copy engines over NVLink (ces_peer_gather: peers mapped through
                # CUDA IPC) while the D / V GEMMs of this rank's own block run with every SM; the all-reduce of C^uu
                # just queued is the cross-rank ordering the pulls need
                phases["peer_gather"]()
                phases["interact_own"]()
                phases["peer_wait"]()
                mark("peer_gather:waited")
                phases["interact_rest"]()
                overlapped = True
            elif dist.get_backend(group) == "nccl" and resolve != "always" and "interact_own" in phases:
                # NCCL: in-place all-gathers started asynchronously; the D / V GEMMs of this rank's own block (already
                # in place after the centring phase) run while the other ranks' blocks arrive over NVLink
                works = [dist.all_gather_into_tensor(e_all, e_own, group=group, async_op=True),
                         dist.all_gather_into_tensor(ut_all, ut_own, group=group, async_op=True)]
                phases["interact_own"]()
                for wk in works:
                    wk.wait()
                mark("allgather:e,ut:waited")
                phases["interact_rest"]()
                overlapped = True
            elif "peer_gather" in phases:
                phases["peer_gather"]()
                phases["peer_wait"]()
            else:
                dist.all_gather_into_tensor(e_all, e_own.clone(), group=group)
                dist.all_gather_into_tensor(ut_all, ut_own.clone(), group=group)
        if not overlapped:
            phases["interact"](resolve == "always")
    if comm is not None:
        allreduce_slice(buffer("scalars"), 0, 5)
        mark("allreduce:scalars:done")
    keep = False
    if resolve == "spectral":
        # hk = 1 / lambda_max(D) (ces/calibrate.py:249-251); lambda_max(D) = lambda_max(Gamma^-1 C^pp), see csrc/eig.cu
        phases["cpp"]()
        if comm is not None:
            allreduce(buffer("cpp"))
        phases["spectral"]()
        phases["update"]("spectral")
        return
    if resolve is not None:
        hk = phases["peek"]()
        if resolve == "always" or resolve[0] + hk > resolve[1]:
            phases["cpp"]()
            if comm is not None:
                allreduce(buffer("cpp"))
            phases["resolve"]()
        keep = True
    if rule == "aldi_constant":
        phases["drift"]()
        if comm is not None:
            allreduce_slice(buffer("scalars"), 5, 6, dist.ReduceOp.MAX)
    phases["update"](keep)


def run_host_phases(phases, buffer, comm, p, k, rule, bounds):
    """The pipelined HOST step of a column shard (include/ces_b200.h: "the host step in pieces") with this rank's
    collectives in between.  ``bounds`` = the row chunks of the G upload (``ces_host_chunk_schedule``: identical on every
    rank -- the means are all-reduced slice by slice, so every rank must cut the same chunks):

        for chunk c:  sums_g(c) -> all-reduce(sum) "sums"[bounds[c]:bounds[c+1]] -> centre_g(c) [+ interact_chunk(c)]
        sums_u        -> all-reduce(sum) "sums"[k:k+p]
        centre_u      -> all-reduce(sum) "cuu";  gathers of "e_all" / "ut_all" started (peer pulls, or all-gathers)
        interact_chunk(last), interact_own   (run while the other ranks' blocks arrive)
        interact_rest -> all-reduce(sum) "scalars"[0:5]
        [drift        -> all-reduce(max) "scalars"[5:6]]          aldi_constant only
        update

    The last chunk's share of the own block's D panel is deferred until the gathers have been started, so they run under
    it.  ``phases`` maps the names to callables (the engine passes the ctypes calls of the library;
    tests/test_multirank_gloo.py passes a numpy stand-in and runs this over gloo without a GPU)."""
    dist, group, rank = comm
    mark = phases.get("mark", lambda name: None)
    sums = buffer("sums")
    nchunks = len(bounds) - 1
    last = nchunks - 1
    for c in range(nchunks):
        phases["sums_g"](c)
        dist.all_reduce(sums[0, bounds[c]:bounds[c + 1]], group=group)
        phases["centre_g"](c, c != last)
    phases["sums_u"]()
    dist.all_reduce(sums[0, k:k + p], group=group)
    phases["centre_u"]()
    dist.all_reduce(buffer("cuu"), group=group)
    mark("allreduce:cuu:done")
    e_all, ut_all = buffer("e_all"), buffer("ut_all")
    e_own, ut_own = e_all[rank * k:(rank + 1) * k], ut_all[rank * p:(rank + 1) * p]
    if "peer_gather" in phases:
        phases["peer_gather"]()
        phases["interact_chunk"](last)
        phases["interact_own"]()
        phases["peer_wait"]()
    elif dist.get_backend(group) == "nccl":
        works = [dist.all_gather_into_tensor(e_all, e_own, group=group, async_op=True),
                 dist.all_gather_into_tensor(ut_all, ut_own, group=group, async_op=True)]
        phases["interact_chunk"](last)
        phases["interact_own"]()
        for wk in works:
            wk.wait()
    else:
        dist.all_gather_into_tensor(e_all, e_own.clone(), group=group)
        dist.all_gather_into_tensor(ut_all, ut_own.clone(), group=group)
        phases["interact_chunk"](last)
        phases["interact_own"]()
    mark("gather:e,ut:waited")
    phases["interact_rest"]()
    scal = buffer("scalars")
    dist.all_reduce(scal[0, 0:5], group=group)
    mark("allreduce:scalars:done")
    if rule == "aldi_constant":
        phases["drift"]()
        dist.all_reduce(scal[0, 5:6], op=dist.ReduceOp.MAX, group=group)
    phases["update"]()


@contextlib.contextmanager
def stream_guard(torch, lib_stream):
    """A library handle launches on the stream that was current when it was created.  Torch work issued around it
    (collectives, copies, noise) must be ordered with those launches: when the caller has since switched streams
    (``with torch.cuda.stream(s): eks.run(...)``), the library stream first waits for the caller's stream, becomes the
    current stream for the duration of the call, and the caller's stream waits for it afterwards."""
    cur = torch.cuda.current_stream()
    if cur.cuda_stream == lib_stream.cuda_stream:
        yield
        return
    lib_stream.wait_stream(cur)
    with torch.cuda.stream(lib_stream):
        yield
    cur.wait_stream(lib_stream)


class _DeviceView(object):
    """Zero-copy torch view of a library-owned device buffer (``__cuda_array_interface__``)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {
            "shape": tuple(int(s) for s in shape), "typestr": "<f8", "data": (int(ptr), False),
            "version": 2, "strides": None,
        }


class Engine(object):
    """One sampler's device state on the current CUDA device.

    p, k      parameter / observation dimensions (``enka.__init__``, ces/calibrate.py:14-22)
    J         global ensemble size
    group     torch.distributed process group when the ensemble is column-sharded
              (None: single GPU).  Rank r owns columns ``shard_range(J, r, nranks)``.
    """

    def __init__(self, p, k, J, group=None, d_panel_bytes=0):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("ces_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = torch
        self.lib = _lib.load()
        self.p, self.k, self.J = int(p), int(k), int(J)
        self.group = group
        if group is not None:
            import torch.distributed as dist

            self.dist = dist
            self.rank, self.nranks = dist.get_rank(group), dist.get_world_size(group)
        else:
            self.dist = None
            self.rank, self.nranks = 0, 1
        self.Jl = shard_width(self.J, self.nranks)
        lo, hi = shard_range(self.J, self.rank, self.nranks)
        self.col_lo, self.col_hi = lo, hi
        self.cols = hi - lo
        self.stream = torch.cuda.current_stream()
        h = ctypes.c_void_p()
        _lib.check(self.lib.ces_create(self.p, self.k, self.Jl, self.J, self.rank, self.nranks, self.cols,
                                       ctypes.c_void_p(self.stream.cuda_stream), int(d_panel_bytes), ctypes.byref(h)))
        self.h = h
        self._views = {}
        self._hk = ctypes.c_double()
        self._met = (ctypes.c_double * 4)()
        self.peer_gather = False
        if (self.nranks > 1 and int(d_panel_bytes) >= 0 and os.environ.get("CES_PEER_GATHER", "1") != "0"
                and self.dist.get_backend(group) == "nccl"):
            self.peer_gather = self._setup_peer_gather()

    def _setup_peer_gather(self):
        """Map every peer's E / U~ buffers through CUDA IPC (ces_ipc_*), so the per-step gathers run as copy-engine
        copies over NVLink instead of an NCCL all-gather.  All ranks must agree: if the mapping fails anywhere (ranks on
        different nodes, IPC unavailable) everybody keeps the NCCL path."""
        torch, dist = self.torch, self.dist
        ok = 1
        try:
            he, hu = ctypes.create_string_buffer(64), ctypes.create_string_buffer(64)
            _lib.check(self.lib.ces_ipc_export(self.h, he, hu))
            mine = (self.rank, he.raw, hu.raw)
        except Exception:
            ok, mine = 0, (self.rank, None, None)
        everyone = [None] * self.nranks
        dist.all_gather_object(everyone, mine, group=self.group)
        if ok:
            try:
                for rank, e_raw, u_raw in everyone:
                    if rank == self.rank:
                        continue
                    if e_raw is None:
                        raise RuntimeError("peer %d exported nothing" % rank)
                    _lib.check(self.lib.ces_ipc_import(self.h, int(rank), e_raw, u_raw))
            except Exception:
                ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        return bool(flag.item())

    def on_stream(self):
        return stream_guard(self.torch, self.stream)

    def close(self):
        if getattr(self, "h", None):
            self.lib.ces_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ problem data
    def set_problem(self, y_obs, Gamma, sigma, mu, ustar):
        y = np.ascontiguousarray(np.asarray(y_obs, dtype=np.float64).reshape(self.k))
        Gam = np.ascontiguousarray(np.asarray(Gamma, dtype=np.float64).reshape(self.k, self.k))
        Sig = np.ascontiguousarray(np.asarray(sigma, dtype=np.float64).reshape(self.p, self.p))
        m = np.ascontiguousarray(np.asarray(mu, dtype=np.float64).reshape(self.p))
        us = np.ascontiguousarray(np.asarray(ustar, dtype=np.float64).reshape(self.p))
        _lib.check(self.lib.ces_set_problem(self.h, _lib.host_ptr(y), _lib.host_ptr(Gam), _lib.host_ptr(Sig),
                                            _lib.host_ptr(m), _lib.host_ptr(us)))

    # ------------------------------------------------------------------ buffers
    def buffer(self, name):
        """Torch view (rows x ld) of a named library buffer (see ces_buffer in the header)."""
        if name not in self._views:
            ptr, rows, cols, ld = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
            _lib.check(self.lib.ces_buffer(self.h, name.encode(), ctypes.byref(ptr), ctypes.byref(rows),
                                           ctypes.byref(cols), ctypes.byref(ld)))
            view = _DeviceView(ptr.value, (rows.value, ld.value))
            self._views[name] = self.torch.as_tensor(view, device="cuda")
        return self._views[name]

    def profile(self, on=True):
        """Bracket every D = E^T W launch with CUDA events (see ces_profile_enable)."""
        _lib.check(self.lib.ces_profile_enable(self.h, 1 if on else 0))

    def profile_read(self):
        """(summed ms, launches, algorithmic flops) of the D GEMM since the previous read."""
        ms, n, fl = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
        _lib.check(self.lib.ces_profile_read(self.h, ctypes.byref(ms), ctypes.byref(n), ctypes.byref(fl)))
        return ms.value, n.value, fl.value

    def timeline(self, on=True):
        """Record named CUDA events per phase (ces_timeline_*); ``timeline_read`` returns [(name, ms), ...]."""
        _lib.check(self.lib.ces_timeline_enable(self.h, 1 if on else 0))
        self._timeline_on = bool(on)

    def mark(self, name):
        if getattr(self, "_timeline_on", False):
            _lib.check(self.lib.ces_timeline_mark(self.h, name.encode()))

    def timeline_read(self):
        cap = 4096
        names = ctypes.create_string_buffer(64 * cap)
        ms = (ctypes.c_double * cap)()
        n = ctypes.c_int64()
        _lib.check(self.lib.ces_timeline_read(self.h, names, 64 * cap, ms, cap, ctypes.byref(n)))
        labels = names.value.decode().split("\n")
        return [(labels[i] if i < len(labels) else "?", float(ms[i])) for i in range(n.value)]

    def normal_noise(self, rows, seed, step, out=None):
        """(rows, cols) standard normal noise for this rank's columns, generated on the device (ces_fill_normal);
        identical to the corresponding columns of a single-GPU draw with the same (seed, step)."""
        torch = self.torch
        if out is None:
            out = torch.empty(rows, self.cols, dtype=torch.float64, device="cuda")
        if self.cols:
          with self.on_stream():
            _lib.check(self.lib.ces_fill_normal(ctypes.c_void_p(self.stream.cuda_stream), int(seed), int(step),
                                                ctypes.c_void_p(out.data_ptr()), int(out.stride(0)), int(rows),
                                                int(self.cols), int(self.col_lo)))
        return out

    def set_noise(self, kind, seed=0, step=0, xi=None):
        """Noise term of the following steps (ces_set_noise): "cholesky" (the reference's sqrt(2h) chol(C^uu) xi with the
        (p, cols) xi given to each step) or "ensemble" (sqrt(2h / n_C) (U - ubar) xi with a J x J xi: from the device's
        Philox stream at (seed, step) when ``xi`` is None, else ``xi``, a (J, cols) float64 CUDA tensor holding this rank's
        columns, kept alive here until the next call)."""
        if kind not in _lib.NOISES:
            raise ValueError("noise must be 'cholesky' or 'ensemble'")
        if kind == "ensemble" and xi is not None:
            if tuple(xi.shape) != (self.J, self.cols):
                raise ValueError("ensemble noise xi must be (J, cols) = (%d, %d), got %s" % (self.J, self.cols, tuple(xi.shape)))
            if xi.stride(1) != 1 or xi.stride(0) % 2 or xi.stride(0) < 1 or xi.data_ptr() % 16:
                # the GEMM reads xi through TMA: 16-byte aligned base, even leading dimension (odd J, narrow shards)
                padded = self.torch.zeros(self.J, -(-max(self.cols, 1) // 16) * 16, dtype=self.torch.float64, device="cuda")
                padded[:, :self.cols] = xi
                xi = padded[:, :self.cols]
            Xp, ldx = self._dev(xi)
        else:
            xi, Xp, ldx = None, None, 0
        _lib.check(self.lib.ces_set_noise(self.h, _lib.NOISES[kind], int(seed), int(step), Xp, ldx))
        self._noise_xi = xi

    def _apply_noise(self, noise):
        """``noise``: None (the reference's Cholesky form) or ("ensemble", seed, step, xi or None); a host xi is uploaded."""
        if noise is None:
            return self.set_noise("cholesky")
        kind, seed, step, xi = noise
        if xi is not None and not hasattr(xi, "is_cuda"):
            xi = self.torch.from_numpy(np.ascontiguousarray(xi, dtype=np.float64)).cuda()
        self.set_noise(kind, seed, step, xi)

    def launch_count(self):
        return int(self.lib.ces_launch_count(self.h))

    @staticmethod
    def _dev(t):
        assert t.is_cuda and t.dtype.is_floating_point and t.element_size() == 8 and t.stride(1) == 1, \
            "device ensembles must be float64 CUDA tensors with the particle axis contiguous"
        return ctypes.c_void_p(t.data_ptr()), int(t.stride(0))

    # ------------------------------------------------------------------ one update
    def step(self, rule, U, G, xi, out=None, fixed_h=None, switch=1.0, resolve=None, formulation="interaction", noise=None):
        with self.on_stream():
            return self._step(rule, U, G, xi, out, fixed_h, switch, resolve, formulation, noise)

    def _step(self, rule, U, G, xi, out, fixed_h, switch, resolve, formulation, noise=None):
        """One update on this rank's columns.  U (p, cols), G (k, cols), xi (p, cols) are float64 CUDA
        tensors; returns (U_next, hk, metrics dict).  ``fixed_h`` gives the step size ('constant', 'mix' after
        spin-up); ``resolve`` asks for the hk C^pp + Gamma re-solve of D (see ``run_phases``).  ``noise``: None for
        the reference's Cholesky noise, or ("ensemble", seed, step, xi_ens or None) (``set_noise``; xi is then
        ignored and may be None)."""
        torch = self.torch
        self._apply_noise(noise)
        r = _lib.RULES[rule]
        ts = _lib.TS_FIXED if fixed_h is not None else _lib.TS_FROBENIUS
        fh = float(fixed_h) if fixed_h is not None else 0.0
        if out is None:
            out = torch.empty_like(U)
        Up, ldu = self._dev(U)
        Gp, ldg = self._dev(G)
        Op, ldo = self._dev(out)
        if xi is not None:
            Xp, ldx = self._dev(xi)
        else:
            Xp, ldx = ctypes.c_void_p(0), 0
        lib, h = self.lib, self.h
        if formulation not in ("interaction", "factored"):
            raise ValueError("formulation must be 'interaction' or 'factored'")
        if self.nranks == 1 and resolve is None:
            _lib.check(lib.ces_step(h, r, ts, fh, float(switch), _lib.FORMULATIONS[formulation], Up, ldu, Gp, ldg, Xp, ldx,
                                    Op, ldo, ctypes.byref(self._hk), self._met))
        else:
            def peek():
                hk = ctypes.c_double()
                _lib.check(lib.ces_peek_step_size(h, ts, fh, ctypes.byref(hk)))
                return hk.value

            def spectral():
                lam, steps = ctypes.c_double(), ctypes.c_int()
                _lib.check(lib.ces_phase3d_spectral(h, ctypes.byref(lam), ctypes.byref(steps)))
                self.last_radspec, self.last_lanczos_steps = lam.value, abs(steps.value)
                if steps.value < 0:
                    import warnings

                    warnings.warn("time_step='spectral': Lanczos stopped after %d steps without converging; lambda_max "
                                  "(%.6e) is a lower bound, hk may be too large" % (-steps.value, lam.value), RuntimeWarning)
                return lam.value

            def update(keep):
                ev = getattr(self, "_xi_ready", None)
                if ev is not None:                  # sharded host step: the noise was uploaded on a side stream
                    torch.cuda.current_stream().wait_event(ev)
                    self._xi_ready = None
                if keep == "spectral":
                    kind, val = _lib.TS_FIXED, 1.0 / self.last_radspec
                else:
                    kind, val = (_lib.TS_KEEP if keep else ts), fh
                _lib.check(lib.ces_phase4_update(h, r, kind, val, Up, ldu, Xp, ldx, Op, ldo, ctypes.byref(self._hk),
                                                 self._met))

            phases = {
                "sums": lambda: _lib.check(lib.ces_phase1_sums(h, Up, ldu, Gp, ldg)),
                "centre": lambda: _lib.check(lib.ces_phase2_centre(h, r, Up, ldu, Gp, ldg)),
                "interact": lambda skip: _lib.check(lib.ces_phase3_interact(h, r, 1 if skip else 0)),
                "interact_own": lambda: _lib.check(lib.ces_phase3_blocks(h, r, 0, 1)),
                "interact_rest": lambda: _lib.check(lib.ces_phase3_blocks(h, r, 1, self.nranks - 1)),
                "peek": peek,
                "cpp": lambda: _lib.check(lib.ces_phase3b_cpp(h)),
                "resolve": lambda: _lib.check(lib.ces_phase3c_resolve(h, r)),
                "spectral": spectral,
                "products": lambda: _lib.check(lib.ces_phase3f_products(h, r)),
                "finish_factored": lambda: _lib.check(lib.ces_phase3f_finish(h, r)),
                "drift": lambda: _lib.check(lib.ces_phase4a_drift(h, float(switch))),
                "update": update,
                "mark": self.mark,
            }
            if self.peer_gather:
                phases["peer_gather"] = lambda: _lib.check(lib.ces_peer_gather(h))
                phases["peer_wait"] = lambda: _lib.check(lib.ces_peer_gather_wait(h))
            comm = (self.dist, self.group, self.rank) if self.nranks > 1 else None
            run_phases(phases, self.buffer, comm, self.p, self.k, rule, resolve, formulation)
        met = {key: float(self._met[i]) for i, key in enumerate(_METRIC_KEYS)}
        return out, float(self._hk.value), met

    def step_host(self, rule, U, G, xi, fixed_h=None, switch=1.0, resolve=None, formulation="interaction", noise=None):
        """The same update on host numpy arrays: the copies to and from the device are part of the call.  This is what
        ``sampling.eks_update*`` invoke.  Single GPU: (p, J) / (k, J) arrays through ``ces_step_host``.  Column-sharded
        (``nranks > 1``): this rank's (p, cols) / (k, cols) shards in, its (p, cols) shard of U_next out, the phases
        with their collectives in between (``_step_host_sharded``).  ``noise`` as in ``step`` (a host xi_ens is
        uploaded)."""
        if formulation not in _lib.FORMULATIONS:
            raise ValueError("formulation must be 'interaction' or 'factored'")
        if self.nranks != 1:
            return self._step_host_sharded(rule, U, G, xi, fixed_h, switch, resolve, formulation, noise)
        if resolve is not None:
            # non-default time_step: the phase-by-phase device path, with explicit copies around it
            torch = self.torch
            dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()
            out, hk, met = self.step(rule, dev(U), dev(G), dev(xi) if xi is not None else None, fixed_h=fixed_h,
                                     switch=switch, resolve=resolve, formulation=formulation, noise=noise)
            return out.cpu().numpy(), hk, met
        self._apply_noise(noise)
        r = _lib.RULES[rule]
        ts = _lib.TS_FIXED if fixed_h is not None else _lib.TS_FROBENIUS
        fh = float(fixed_h) if fixed_h is not None else 0.0
        U = np.ascontiguousarray(U, dtype=np.float64)
        G = np.ascontiguousarray(G, dtype=np.float64)
        assert U.shape == (self.p, self.J) and G.shape == (self.k, self.J), (U.shape, G.shape)
        # a fresh array per call like the reference (callers keep references in Uall), in page-locked memory
        # from torch's caching host allocator so the device->host copy runs at full PCIe rate
        if U.nbytes >= (1 << 20):
            out = self.torch.empty((self.p, self.J), dtype=self.torch.float64, pin_memory=True).numpy()
        else:
            out = np.empty_like(U)
        if xi is not None and noise is None:
            xi = np.ascontiguousarray(xi, dtype=np.float64)
            assert xi.shape == U.shape
            xp = _lib.host_ptr(xi)
        else:
            xp = None
        _lib.check(self.lib.ces_step_host(self.h, r, ts, fh, float(switch), _lib.FORMULATIONS[formulation],
                                          _lib.host_ptr(U), _lib.host_ptr(G), xp,
                                          _lib.host_ptr(out), ctypes.byref(self._hk), self._met))
        met = {key: float(self._met[i]) for i, key in enumerate(_METRIC_KEYS)}
        return out, float(self._hk.value), met

    def _pinned(self, name, shape):
        """Reusable page-locked staging array (numpy view of a torch pinned tensor)."""
        key = ("pin", name, tuple(shape))
        if key not in self._views:
            self._views[key] = self.torch.empty(tuple(shape), dtype=self.torch.float64, pin_memory=True)
        return self._views[key]

    def _step_host_sharded(self, rule, U, G, xi, fixed_h, switch, resolve, formulation, noise=None):
        """Column shard on host arrays.  Default rule set (no re-solve of D, interaction formulation): the pipelined
        pieces of the library's host step (include/ces_b200.h) with this rank's collectives in between -- G uploads in
        row chunks while the chunks already on the device are summed (all-reduce of that slice of the means), centred and
        contracted into the own block's first D panel; U and xi follow behind; U_next comes back in overlapped column
        chunks.  Other modes: plain uploads, then the device-pointer phases."""
        torch, lib, h, dist, group = self.torch, self.lib, self.h, self.dist, self.group
        U = np.ascontiguousarray(U, dtype=np.float64)
        G = np.ascontiguousarray(G, dtype=np.float64)
        assert U.shape == (self.p, self.cols) and G.shape == (self.k, self.cols), (U.shape, G.shape, self.cols)
        if noise is not None:
            xi = None                               # ensemble noise: the J x J xi replaces the (p, cols) one
        if xi is not None:
            xi = np.ascontiguousarray(xi, dtype=np.float64)
            assert xi.shape == U.shape
        host = torch.empty((self.p, self.cols), dtype=torch.float64, pin_memory=self.p * self.cols * 8 >= (1 << 20))
        ptr = lambda a: (_lib.host_ptr(a) if a is not None and a.size else None)
        with self.on_stream():
            if resolve is None and formulation == "interaction":
                self._apply_noise(noise)
                r = _lib.RULES[rule]
                ts = _lib.TS_FIXED if fixed_h is not None else _lib.TS_FROBENIUS
                nch, bounds = ctypes.c_int(), (ctypes.c_int64 * 9)()
                _lib.check(lib.ces_host_begin(h, r, 0, ptr(U), ptr(G), ptr(xi), ctypes.byref(nch), bounds))
                fh = float(fixed_h) if fixed_h is not None else 0.0
                out_ptr = host.data_ptr() if self.cols else None
                phases = {
                    "sums_g": lambda c: _lib.check(lib.ces_host_sums_g(h, c)),
                    "centre_g": lambda c, interact: _lib.check(lib.ces_host_centre_g(h, c, 1 if interact else 0)),
                    "interact_chunk": lambda c: _lib.check(lib.ces_host_interact_chunk(h, c)),
                    "sums_u": lambda: _lib.check(lib.ces_host_sums_u(h)),
                    "centre_u": lambda: _lib.check(lib.ces_host_centre_u(h)),
                    "interact_own": lambda: _lib.check(lib.ces_host_interact_own(h)),
                    "interact_rest": lambda: _lib.check(lib.ces_phase3_blocks(h, r, 1, self.nranks - 1)),
                    "drift": lambda: _lib.check(lib.ces_phase4a_drift(h, float(switch))),
                    "update": lambda: _lib.check(lib.ces_host_update(h, ts, fh, out_ptr, ctypes.byref(self._hk), self._met)),
                    "mark": self.mark,
                }
                if self.peer_gather:
                    phases["peer_gather"] = lambda: _lib.check(lib.ces_peer_gather(h))
                    phases["peer_wait"] = lambda: _lib.check(lib.ces_peer_gather_wait(h))
                run_host_phases(phases, self.buffer, (dist, group, self.rank), self.p, self.k, rule,
                                [int(bounds[i]) for i in range(nch.value + 1)])
                met = {key: float(self._met[i]) for i, key in enumerate(_METRIC_KEYS)}
                return host.numpy(), float(self._hk.value), met
            # ---- non-default modes: plain uploads (xi on a side stream: only the last phase needs it), device phases
            if "h2d" not in self._views:
                self._views["h2d"] = torch.cuda.Stream()
                for name, rows in (("U", self.p), ("G", self.k), ("xi", self.p), ("out", self.p)):
                    self._views["dev_" + name] = torch.empty(rows, max(self.cols, 1), dtype=torch.float64, device="cuda")
            copy_st = self._views["h2d"]
            Ud, Gd, Xd, Od = (self._views["dev_" + n] for n in ("U", "G", "xi", "out"))
            main = torch.cuda.current_stream()
            copy_st.wait_stream(main)               # the previous step's readers of the staging buffers
            Ud.copy_(torch.from_numpy(U), non_blocking=True)
            Gd.copy_(torch.from_numpy(G), non_blocking=True)
            xi_ready = None
            if xi is not None:
                with torch.cuda.stream(copy_st):
                    Xd.copy_(torch.from_numpy(xi), non_blocking=True)
                    xi_ready = torch.cuda.Event()
                    xi_ready.record(copy_st)
            self._xi_ready = xi_ready
            # the last phase downloads U_next itself, in column chunks overlapped with their assembly
            _lib.check(lib.ces_set_pending_output(h, host.data_ptr() if self.cols else None))
            try:
                out, hk, met = self._step(rule, Ud, Gd, Xd if xi is not None else None, Od, fixed_h, switch, resolve, formulation,
                                          noise)
            finally:
                lib.ces_set_pending_output(h, None)
            main.synchronize()
            return host.numpy(), hk, met

    def gather_columns_host(self, local):
        """Full (rows, J) host array from every rank's (rows, cols) host shard (all ranks receive it)."""
        torch = self.torch
        local = np.ascontiguousarray(local, dtype=np.float64)
        rows = local.shape[0]
        pad = torch.zeros(rows, self.Jl, dtype=torch.float64, device="cuda")
        pad[:, :self.cols] = torch.from_numpy(local).cuda()
        full = torch.empty(self.nranks, rows, self.Jl, dtype=torch.float64, device="cuda")
        self.dist.all_gather_into_tensor(full.view(-1), pad.view(-1), group=self.group)
        return full.permute(1, 0, 2).reshape(rows, self.nranks * self.Jl)[:, :self.J].cpu().numpy()

    # ------------------------------------------------------------------ forward maps
    def forward_map(self, kind, U, G, A=None, lda=0, b=None, params=None):
        """G[:, j] = model(U[:, j]) on the device for the ces.utils maps (enka.G_ens)."""
        with self.on_stream():
            return self._forward_map(kind, U, G, A, lda, b, params)

    def _forward_map(self, kind, U, G, A, lda, b, params):
        Up, ldu = self._dev(U)
        Gp, ldg = self._dev(G)
        Ap = ctypes.c_void_p(A.data_ptr()) if A is not None else None
        bp = ctypes.c_void_p(b.data_ptr()) if b is not None else None
        if params is not None:
            pr = np.ascontiguousarray(params, dtype=np.float64)
            pp = _lib.host_ptr(pr)
        else:
            pp = None
        _lib.check(self.lib.ces_forward_map(self.h, _lib.MAPS[kind], Ap, int(lda), bp, pp, Up, ldu, Gp, ldg))
        return G
