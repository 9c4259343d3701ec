"""Order of the library calls and collectives of one column-sharded update (ces_b200.engine.run_phases and
run_host_phases), world_size 2 over gloo on CPU.  The phases are the numpy stand-in (tests/_numpy_phases.py) wrapped
so that every call is logged with its arguments; the collectives go through a proxy of torch.distributed that logs
each one as (kind, buffer, element range, reduce op) before running it.  The device time of a sharded step depends on
this order -- which GEMMs run while the other ranks' blocks are in flight -- and no CPU test of the arithmetic sees it.

Both ways E / U~ reach the other ranks are covered: peer pulls (``peer_gather`` / ``peer_wait``) and in-place
asynchronous all-gathers.  The sequence must not depend on the process-group backend: the proxy reports "nccl" and
"gloo" in turn and both must give the same calls.  Timeline marks are not part of the sequence."""
import inspect
import os
import sys

import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

P, K, J = 5, 40, 37                 # diagonal Gamma (the pipelined host step's case); a ragged last shard
DEVICE_MODES = {                    # case -> (rule, resolve, formulation)
    "default": ("aldi", None, "interaction"),
    "aldi_constant": ("aldi_constant", None, "interaction"),
    "always": ("aldi", "always", "interaction"),
    "mix": ("aldi", (1.5, 1.0), "interaction"),
    "spectral": ("aldi", "spectral", "interaction"),
    "factored": ("aldi", None, "factored"),
}
HOST_MODES = {                      # case -> (rule, row chunks of the G upload)
    "host-1chunk": ("aldi", [0, K]),
    "host-3chunks": ("aldi_constant", [0, 16, 32, K]),
}


class _DistProxy(object):
    """torch.distributed for the orchestration: logs every collective, then runs it on the real (gloo) group."""

    ReduceOp = dist.ReduceOp

    def __init__(self, ph, log, backend):
        self.ph, self.log, self.backend = ph, log, backend

    def get_backend(self, group=None):
        return self.backend

    def _where(self, t):
        for name, b in self.ph.buf.items():
            if t.untyped_storage().data_ptr() == b.untyped_storage().data_ptr():
                lo = t.storage_offset() - b.storage_offset()
                return name if (lo, t.numel()) == (0, b.numel()) else "%s[%d:%d]" % (name, lo, lo + t.numel())
        raise AssertionError("a collective on a tensor that is no named buffer")

    def all_reduce(self, t, op=dist.ReduceOp.SUM, group=None, async_op=False):
        self.log.append("all_reduce %s %s" % (self._where(t), "max" if op == dist.ReduceOp.MAX else "sum"))
        return dist.all_reduce(t, op=op, group=group, async_op=async_op)

    def all_gather_into_tensor(self, out, inp, group=None, async_op=False):
        name = self._where(out)
        self.log.append("all_gather %s%s" % (name, " async" if async_op else ""))
        work = dist.all_gather_into_tensor(out, inp, group=group, async_op=async_op)
        return _LoggedWork(work, self.log, "wait %s" % name) if async_op else work


class _LoggedWork(object):
    def __init__(self, work, log, entry):
        self.work, self.log, self.entry = work, log, entry

    def wait(self):
        self.log.append(self.entry)
        return self.work.wait()


def _logged(phases, log):
    """The phases, each call logged as name(arguments with defaults applied)."""
    def wrap(name, fn):
        sig = inspect.signature(fn)

        def call(*a, **kw):
            b = sig.bind(*a, **kw)
            b.apply_defaults()
            log.append("%s(%s)" % (name, ", ".join(repr(v) for v in b.arguments.values())))
            return fn(*a, **kw)
        return call
    return {name: wrap(name, fn) for name, fn in phases.items()}


def _record(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from _numpy_phases import NumpyPhases
        from ces_b200.engine import run_host_phases, run_phases
        from oracle import eks_oracle as eo

        pr = eo.linear_gaussian_problem(P, K, J)
        seqs = {}
        for strategy, backends in (("peer", ("nccl",)), ("all_gather", ("nccl", "gloo"))):
            for backend in backends:
                for case in list(DEVICE_MODES) + list(HOST_MODES):
                    ph = NumpyPhases(P, K, J, rank, world, pr["y"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"])
                    sl = slice(ph.lo, ph.hi)
                    args = (pr["U0"][:, sl], pr["G"][:, sl], pr["xi"][:, sl])
                    log = []
                    comm = (_DistProxy(ph, log, backend), None, rank)
                    if case in DEVICE_MODES:
                        rule, resolve, formulation = DEVICE_MODES[case]
                        phases = ph.bind(rule, *args, peer=strategy == "peer")
                        run_phases(_logged(phases, log), ph.buffer, comm, P, K, rule, resolve, formulation)
                    else:
                        rule, bounds = HOST_MODES[case]
                        phases = ph.bind_host(rule, *args, bounds, peer=strategy == "peer")
                        run_host_phases(_logged(phases, log), ph.buffer, comm, P, K, rule, bounds)
                    seqs[(strategy, backend, case)] = log
        q.put((rank, seqs))
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def recorded():
    """{(strategy, backend, case): [call, ...]} of both ranks, recorded in one world-2 process group."""
    import socket

    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_record, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=240) for _ in procs)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    return got


# Recorded from the orchestration before the two gather paths were merged into one (peer pulls, or in-place asynchronous
# all-gathers behind an NCCL group).  One sequence differs on purpose: with resolve "always" the all-gathers used to be
# blocking and are now started asynchronously and waited for at once, before interact(True).  A gloo group used to take
# the blocking all-gathers and interact(False) in every mode; it now takes the same calls as NCCL.
EXPECTED = {
    ("peer", "default"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "peer_gather()", "interact_own()",
        "peer_wait()", "interact_rest()", "all_reduce scalars[0:5] sum", "update(False)",
    ],
    ("peer", "aldi_constant"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "peer_gather()", "interact_own()",
        "peer_wait()", "interact_rest()", "all_reduce scalars[0:5] sum", "drift()", "all_reduce scalars[5:6] max",
        "update(False)",
    ],
    ("peer", "always"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "peer_gather()", "peer_wait()",
        "interact(True)", "all_reduce scalars[0:5] sum", "peek()", "cpp()", "all_reduce cpp sum", "resolve()",
        "update(True)",
    ],
    ("peer", "mix"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "peer_gather()", "interact_own()",
        "peer_wait()", "interact_rest()", "all_reduce scalars[0:5] sum", "peek()", "cpp()", "all_reduce cpp sum",
        "resolve()", "update(True)",
    ],
    ("peer", "spectral"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "peer_gather()", "interact_own()",
        "peer_wait()", "interact_rest()", "all_reduce scalars[0:5] sum", "cpp()", "all_reduce cpp sum", "spectral()",
        "update('spectral')",
    ],
    ("peer", "factored"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "products()", "all_reduce p1 sum",
        "all_reduce gram_e sum", "all_reduce gram_w sum", "finish_factored()", "all_reduce scalars[0:5] sum",
        "update(False)",
    ],
    ("peer", "host-1chunk"): [
        "sums_g(0)", "all_reduce sums[0:40] sum", "centre_g(0, False)", "sums_u()", "all_reduce sums[40:45] sum",
        "centre_u()", "all_reduce cuu sum", "peer_gather()", "interact_chunk(0)", "interact_own()", "peer_wait()",
        "interact_rest()", "all_reduce scalars[0:5] sum", "update(False)",
    ],
    ("peer", "host-3chunks"): [
        "sums_g(0)", "all_reduce sums[0:16] sum", "centre_g(0, True)", "sums_g(1)", "all_reduce sums[16:32] sum",
        "centre_g(1, True)", "sums_g(2)", "all_reduce sums[32:40] sum", "centre_g(2, False)", "sums_u()",
        "all_reduce sums[40:45] sum", "centre_u()", "all_reduce cuu sum", "peer_gather()", "interact_chunk(2)",
        "interact_own()", "peer_wait()", "interact_rest()", "all_reduce scalars[0:5] sum", "drift()",
        "all_reduce scalars[5:6] max", "update(False)",
    ],
    ("all_gather", "default"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "all_gather e_all async",
        "all_gather ut_all async", "interact_own()", "wait e_all", "wait ut_all", "interact_rest()",
        "all_reduce scalars[0:5] sum", "update(False)",
    ],
    ("all_gather", "aldi_constant"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "all_gather e_all async",
        "all_gather ut_all async", "interact_own()", "wait e_all", "wait ut_all", "interact_rest()",
        "all_reduce scalars[0:5] sum", "drift()", "all_reduce scalars[5:6] max", "update(False)",
    ],
    ("all_gather", "always"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "all_gather e_all async",
        "all_gather ut_all async", "wait e_all", "wait ut_all", "interact(True)", "all_reduce scalars[0:5] sum",
        "peek()", "cpp()", "all_reduce cpp sum", "resolve()", "update(True)",
    ],
    ("all_gather", "mix"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "all_gather e_all async",
        "all_gather ut_all async", "interact_own()", "wait e_all", "wait ut_all", "interact_rest()",
        "all_reduce scalars[0:5] sum", "peek()", "cpp()", "all_reduce cpp sum", "resolve()", "update(True)",
    ],
    ("all_gather", "spectral"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "all_gather e_all async",
        "all_gather ut_all async", "interact_own()", "wait e_all", "wait ut_all", "interact_rest()",
        "all_reduce scalars[0:5] sum", "cpp()", "all_reduce cpp sum", "spectral()", "update('spectral')",
    ],
    ("all_gather", "factored"): [
        "sums()", "all_reduce sums sum", "centre()", "all_reduce cuu sum", "products()", "all_reduce p1 sum",
        "all_reduce gram_e sum", "all_reduce gram_w sum", "finish_factored()", "all_reduce scalars[0:5] sum",
        "update(False)",
    ],
    ("all_gather", "host-1chunk"): [
        "sums_g(0)", "all_reduce sums[0:40] sum", "centre_g(0, False)", "sums_u()", "all_reduce sums[40:45] sum",
        "centre_u()", "all_reduce cuu sum", "all_gather e_all async", "all_gather ut_all async", "interact_chunk(0)",
        "interact_own()", "wait e_all", "wait ut_all", "interact_rest()", "all_reduce scalars[0:5] sum", "update(False)",
    ],
    ("all_gather", "host-3chunks"): [
        "sums_g(0)", "all_reduce sums[0:16] sum", "centre_g(0, True)", "sums_g(1)", "all_reduce sums[16:32] sum",
        "centre_g(1, True)", "sums_g(2)", "all_reduce sums[32:40] sum", "centre_g(2, False)", "sums_u()",
        "all_reduce sums[40:45] sum", "centre_u()", "all_reduce cuu sum", "all_gather e_all async",
        "all_gather ut_all async", "interact_chunk(2)", "interact_own()", "wait e_all", "wait ut_all", "interact_rest()",
        "all_reduce scalars[0:5] sum", "drift()", "all_reduce scalars[5:6] max", "update(False)",
    ],
}


@pytest.mark.parametrize("strategy,backend", [("peer", "nccl"), ("all_gather", "nccl"), ("all_gather", "gloo")])
@pytest.mark.parametrize("case", list(DEVICE_MODES) + list(HOST_MODES))
def test_phase_and_collective_order(recorded, strategy, backend, case):
    for rank in (0, 1):
        assert recorded[rank][(strategy, backend, case)] == EXPECTED[(strategy, case)], rank
