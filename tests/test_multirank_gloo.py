"""world_size-2 (and 3) gloo test of the column-sharded orchestration (ces_b200.engine.run_phases and
run_host_phases) on CPU: the collectives between the phases, the rank-major gather layout and the zero-padded
ragged last shard must reproduce the single-process oracle step, with E / U~ gathered by the asynchronous in-place
all-gathers and by the peer pulls (an in-place all-gather stands in for them).  The per-rank arithmetic is a numpy
stand-in (tests/_numpy_phases.py); on the GPU the same orchestration drives libces_b200.so."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    import socket

    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]
ROOT = os.path.dirname(HERE)


def _worker(rank, world, port, rule, d, k, J, q, ts=None, t_last=None, formulation="interaction", peer=False):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from _numpy_phases import NumpyPhases
        from ces_b200.engine import run_phases
        from oracle import eks_oracle as eo

        pr = eo.linear_gaussian_problem(d, k, J, dense_gamma=True)
        fixed, resolve = None, None
        if ts == "constant":
            fixed, resolve = 0.02, "always"
        elif ts == "mix":
            fixed, resolve = (0.02 if t_last >= 4.0 else None), (t_last, 1.0)
        elif ts == "spectral":
            resolve = "spectral"
        ph = NumpyPhases(d, k, J, rank, world, pr["y"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"])
        sl = slice(ph.lo, ph.hi)
        phases = ph.bind(rule, pr["U0"][:, sl], pr["G"][:, sl], pr["xi"][:, sl], fixed_h=fixed, peer=peer)
        run_phases(phases, ph.buffer, (dist, None, rank), d, k, rule, resolve, formulation)
        ref = eo.step(rule, pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], pr["xi"],
                      time_step=ts, delta_t=0.02, t_last=t_last)
        err = np.abs(ph.out - ref["Uk"][:, sl]).max() / np.abs(ref["Uk"]).max() if ph.cols else 0.0
        herr = abs(ph.hk - ref["hk"]) / ref["hk"]
        merr = max(abs(ph.metrics[m] - ref["metrics"][m]) / abs(ref["metrics"][m]) for m in ph.metrics)
        q.put((rank, float(err), float(herr), float(merr)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("peer", [False, True], ids=["allgather", "peer"])
@pytest.mark.parametrize("world,rule,J,ts,t_last", [
    (2, "aldi", 37, None, None), (2, "aldi_constant", 40, None, None), (2, "eks", 33, None, None),
    (3, "aldi", 16, None, None), (2, "eki", 21, None, None),
    (2, "aldi", 29, "constant", 0.3), (2, "eks", 26, "constant", None), (2, "aldi", 31, "mix", 1.5),
    (2, "aldi", 31, "mix", 5.0), (2, "aldi", 35, "factored", None), (3, "eks", 22, "factored", None),
    (2, "aldi_constant", 27, "factored", None), (2, "aldi", 30, "spectral", None), (3, "eks", 19, "spectral", None)])
def test_sharded_orchestration_matches_single_process(world, rule, J, ts, t_last, peer):
    formulation = "interaction"
    if ts == "factored":
        ts, formulation = None, "factored"
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, rule, 5, 7, J, q, ts, t_last, formulation, peer))
             for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    got = sorted(q.get(timeout=10) for _ in range(world))
    for rank, err, herr, merr in got:
        assert err < 1e-12 and herr < 1e-12 and merr < 1e-12, (rank, err, herr, merr)


def _host_worker(rank, world, port, rule, d, k, J, bounds, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from _numpy_phases import NumpyPhases
        from ces_b200.engine import run_host_phases
        from oracle import eks_oracle as eo

        pr = eo.linear_gaussian_problem(d, k, J)                       # diagonal Gamma (the pipelined host step's case)
        ref = eo.step(rule, pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], pr["xi"])
        for peer in (False, True):
            ph = NumpyPhases(d, k, J, rank, world, pr["y"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"])
            sl = slice(ph.lo, ph.hi)
            if bounds == "library":
                # the chunks the library itself would cut for this shape (a pure host function: needs no GPU)
                import ctypes

                from ces_b200 import _lib

                b = (ctypes.c_int64 * 9)()
                n = _lib.load().ces_host_chunk_schedule(k, ph.Jl, ph.ldJ, world, 0.0, b)
                bounds = [int(b[i]) for i in range(n + 1)]
            phases = ph.bind_host(rule, pr["U0"][:, sl], pr["G"][:, sl], pr["xi"][:, sl], bounds, peer=peer)
            run_host_phases(phases, ph.buffer, (dist, None, rank), d, k, rule, bounds)
            err = np.abs(ph.out - ref["Uk"][:, sl]).max() / np.abs(ref["Uk"]).max() if ph.cols else 0.0
            herr = abs(ph.hk - ref["hk"]) / ref["hk"]
            merr = max(abs(ph.metrics[m] - ref["metrics"][m]) / abs(ref["metrics"][m]) for m in ph.metrics)
            # the last chunk's share of the own block is deferred until after the all-reduce of cuu (gathers started first)
            last = len(bounds) - 2
            order = [c for c in ph.calls if c[0] != "sums_g"]
            ok_order = ("centre_g", last, False) in order and order.index(("interact_chunk", last)) > order.index(("centre_g", last, False))
            q.put((rank, peer, float(err), float(herr), float(merr), len(bounds) - 1, bool(ok_order)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,rule,d,k,J,bounds", [
    (2, "aldi", 5, 40, 37, [0, 16, 40]), (3, "aldi_constant", 4, 48, 29, [0, 16, 32, 48]), (2, "eks", 5, 33, 26, [0, 33]),
    (2, "eki", 3, 64, 21, [0, 16, 24, 32, 40, 48, 56, 60, 64]), (3, "aldi", 4, 20, 2, [0, 16, 20]),
    (2, "aldi", 3, 272, 4300, "library")])
def test_sharded_host_step_orchestration_matches_single_process(world, rule, d, k, J, bounds):
    """ces_b200.engine.run_host_phases -- the pipelined host step of a column shard: the means all-reduced chunk by chunk, the
    own block's D panel accumulated over the chunks with the last chunk deferred behind the start of the gathers -- over
    gloo with a numpy stand-in for the library pieces: same update as the single-process oracle for 1, 2, 3 and 8 chunks,
    ragged shards and a rank without particles (J = 2 on 3 ranks), with and without the peer pulls; the last case cuts the
    chunks with the library's own ces_host_chunk_schedule."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_host_worker, args=(r, world, port, rule, d, k, J, bounds, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(240)
        assert p.exitcode == 0
    got = sorted(q.get(timeout=10) for _ in range(2 * world))
    assert len(set(g[5] for g in got)) == 1                      # every rank cut the same number of chunks
    for rank, peer, err, herr, merr, nchunks, ok_order in got:
        assert err < 1e-12 and herr < 1e-12 and merr < 1e-12, (rank, peer, err, herr, merr)
        assert ok_order
    if bounds == "library":
        assert got[0][5] > 1
