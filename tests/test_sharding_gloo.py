"""World-size-2 gloo tests (CPU) of the multi-GPU host logic: batch partition, result gather, statistics reduction and the closed loop sharded by scenario
(safe-autonomous-driving-mpc_b200/sharding.py).  The per-shard "solve" is the solver source compiled for the host
(tests/hostbuild) -- the product itself has no CPU path; what is under test here is that a sharded run returns
bit-identical results to an unsharded one and that the reductions are right."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _host_solver():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    sys.path.insert(0, ROOT)
    import host_solver_check as H
    from oracle import tracker_port as P
    tab = P.RefTable.from_npz(os.path.join(ROOT, "data", "trajectory3.npz"))

    def solve(x0, obs, n):
        U, st, it, obj = H.host_solve(tab, x0, obs, n)
        return dict(U=U, status=st, obj=obj, iters=it)
    return P, tab, solve


def _worker(rank, world, port, B, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sys.path.insert(0, ROOT)
        from safe_autonomous_driving_mpc_b200 import sharding as S
        P, tab, solve = _host_solver()
        x0, obs, n = P.monte_carlo_problems(tab, B)
        full, (lo, hi) = S.solve_sharded(solve, x0, obs, n, gather=True)
        stats = S.reduce_stats(full["status"][lo:hi], full["iters"][lo:hi], ms=10.0 + rank)
        # the tensor-level gather bench.py's strong-scaling block uses (NCCL there, gloo here): ragged and equal shards
        import torch
        for Bg in (B, B - 1):
            l2, h2 = S.shard_bounds(Bg, rank, world)
            Ug, sg = S.gather_device(torch.from_numpy(full["U"][l2:h2].copy()), torch.from_numpy(full["status"][l2:h2].copy()), Bg)
            assert np.array_equal(Ug.numpy(), full["U"][:Bg]) and np.array_equal(sg.numpy(), full["status"][:Bg])
        # closed loop sharded by scenario (the simulation object is a stand-in here: the device loop has no CPU form)
        class FakeSim:
            def __init__(self, lo, hi):
                self.lo, self.hi = lo, hi
            def run(self, max_steps, check_every):
                return 64 * (1 + self.lo // 10)
            def state(self):
                idx = np.arange(self.lo, self.hi)
                return np.outer(idx, np.ones(5)) + 0.25, (idx * 3).astype(np.int32), (idx % 2).astype(np.int32)
        r = S.simulate_sharded(FakeSim, 33)
        idx = np.arange(33)
        assert np.array_equal(r["x"], np.outer(idx, np.ones(5)) + 0.25) and np.array_equal(r["steps"], idx * 3)
        assert np.array_equal(r["unsolved"], idx % 2) and r["enqueued"] == 64 * (1 + 16 // 10) and r["shard"] == S.shard_bounds(33, rank, world)
        q.put((rank, lo, hi, full["U"], full["status"], full["obj"], stats))
    finally:
        dist.destroy_process_group()


def test_shard_bounds_partition():
    sys.path.insert(0, ROOT)
    from safe_autonomous_driving_mpc_b200 import sharding as S
    for B in (0, 1, 7, 8, 65536, 65537):
        for G in (1, 2, 3, 4, 8):
            b = [S.shard_bounds(B, g, G) for g in range(G)]
            assert b[0][0] == 0 and b[-1][1] == B
            assert all(b[g][1] == b[g + 1][0] for g in range(G - 1))
            sizes = [h - l for l, h in b]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        S.shard_bounds(10, 2, 2)


def test_sharded_equals_unsharded_world2():
    import torch.multiprocessing as mp
    B, world = 301, 2                      # odd size: ragged shards
    # compiles tests/hostbuild once, here, so that the two workers do not both write the library on a fresh checkout
    P, tab, solve = _host_solver()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, B, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    x0, obs, n = P.monte_carlo_problems(tab, B)
    ref = solve(x0, obs, n)
    got.sort(key=lambda t: t[0])
    assert (got[0][1], got[0][2]) == (0, 150) and (got[1][1], got[1][2]) == (150, 301)
    for rank, lo, hi, U, st, obj, stats in got:
        assert np.array_equal(U.reshape(B, 10), ref["U"])          # bitwise: problems are independent
        assert np.array_equal(st, ref["status"]) and np.array_equal(obj, ref["obj"])
        hist = np.bincount(ref["status"], minlength=3)
        assert (stats["solved"], stats["maxiter"], stats["infeasible"]) == tuple(int(v) for v in hist[:3])
        assert stats["problems"] == B and stats["iters"] == int(ref["iters"][:, 1].sum())
        assert stats["ms_max"] == 11.0                              # MAX over ranks
