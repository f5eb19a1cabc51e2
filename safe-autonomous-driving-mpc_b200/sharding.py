"""Batch sharding across the GPUs of one box (SURVEY.md 8e).

Problems are independent, so the solve path has no collective: rank g of G solves the contiguous shard
``[g*B//G, (g+1)*B//G)`` of the batch on its own GPU.  ``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests) is
used only afterwards, to gather results and to reduce statistics:

    shard_bounds      the partition
    solve_sharded     scatter-free sharded solve + optional gather of (U, status, obj) to every rank
    gather_device     all-gather of the shards' device-resident U / status (NCCL), no host round trip
    reduce_stats      status histogram / iteration sums (SUM) and timings (MAX) over ranks
"""
import numpy as np


def shard_bounds(B, rank, world):
    """Contiguous shard [lo, hi) of a batch of B problems owned by `rank` of `world` (sizes differ by at most 1)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    return (B * rank) // world, (B * (rank + 1)) // world


def _dist():
    import torch.distributed as dist
    return dist


def reduce_stats(status, iters, ms, group=None, device=None):
    """status [b] int, iters [b,2] int, ms: float (this rank's time).  Returns dict with the whole-job status
    histogram (SUM), summed rounds / iterations (SUM), problem count (SUM) and the slowest rank's time (MAX)."""
    import torch
    dist = _dist()
    status = np.asarray(status)
    iters = np.asarray(iters).reshape(-1, 2)
    hist = np.bincount(status, minlength=3)[:3]
    sums = torch.tensor([hist[0], hist[1], hist[2], iters[:, 0].sum(), iters[:, 1].sum(), len(status)],
                        dtype=torch.int64, device=device)
    tmax = torch.tensor([float(ms)], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX, group=group)
    s = [int(v) for v in sums.cpu()]
    return dict(solved=s[0], maxiter=s[1], infeasible=s[2], rounds=s[3], iters=s[4], problems=s[5],
                ms_max=float(tmax.cpu()[0]))


def solve_sharded(solve_fn, x0, obs_sv, n_obs, group=None, gather=True, device=None):
    """Every rank holds the whole batch description (x0 [B,5], obs_sv [B,2,2], n_obs [B], numpy) and solves only its
    shard with ``solve_fn(x0_shard, obs_shard, n_shard) -> dict(U [b,5,2], status [b], obj [b], iters [b,2])``.
    With ``gather`` the per-shard U / status / obj are all-gathered so that every rank returns the full arrays;
    otherwise each rank returns its shard only.  Returns (result dict, (lo, hi))."""
    import torch
    dist = _dist()
    on = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if on else 1
    rank = dist.get_rank(group) if on else 0
    B = len(n_obs)
    lo, hi = shard_bounds(B, rank, world)
    r = solve_fn(x0[lo:hi], obs_sv[lo:hi], n_obs[lo:hi])
    out = dict(U=np.asarray(r["U"]).reshape(hi - lo, 5, 2), status=np.asarray(r["status"]).astype(np.int32),
               obj=np.asarray(r["obj"], dtype=np.float64), iters=np.asarray(r["iters"]).reshape(hi - lo, 2))
    if not gather or world == 1:
        return out, (lo, hi)
    full = {}
    sizes = [shard_bounds(B, g, world) for g in range(world)]
    pad = max(h - l for l, h in sizes)
    for key, width, dt in (("U", 10, torch.float64), ("status", 1, torch.int32), ("obj", 1, torch.float64),
                           ("iters", 2, torch.int32)):
        mine = torch.zeros((pad, width), dtype=dt, device=device)
        mine[: hi - lo] = torch.from_numpy(np.ascontiguousarray(out[key]).reshape(hi - lo, width)).to(device=device, dtype=dt)
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine, group=group)                # results only: never on the solve path
        cat = torch.cat([p[: h - l] for p, (l, h) in zip(parts, sizes)]).cpu().numpy()
        full[key] = cat
    return dict(U=full["U"].reshape(B, 5, 2), status=full["status"].reshape(B), obj=full["obj"].reshape(B),
                iters=full["iters"].reshape(B, 2)), (lo, hi)


def gather_device(U_shard, status_shard, B, group=None):
    """All-gather of device-resident shard results after a sharded solve: ``U_shard`` [b,5,2] f64 and ``status_shard``
    [b] i32 of this rank's contiguous shard of a batch of B -> (U [B,5,2], status [B]) on every rank, in batch order.
    One collective per array (``all_gather_into_tensor`` when the shards are equal, padded ``all_gather`` otherwise);
    never on the solve path."""
    import torch
    dist = _dist()
    on = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if on else 1
    if world == 1:
        return U_shard, status_shard
    sizes = [shard_bounds(B, g, world) for g in range(world)]
    b = U_shard.shape[0]
    if all(h - l == b for l, h in sizes):
        U = torch.empty((B, 5, 2), dtype=U_shard.dtype, device=U_shard.device)
        st = torch.empty((B,), dtype=status_shard.dtype, device=status_shard.device)
        dist.all_gather_into_tensor(U, U_shard.contiguous(), group=group)
        dist.all_gather_into_tensor(st, status_shard.contiguous(), group=group)
        return U, st
    pad = max(h - l for l, h in sizes)
    outs = []
    for a in (U_shard.reshape(b, -1), status_shard.reshape(b, 1)):
        mine = torch.zeros((pad, a.shape[1]), dtype=a.dtype, device=a.device)
        mine[:b] = a
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine, group=group)
        outs.append(torch.cat([p[: h - l] for p, (l, h) in zip(parts, sizes)]))
    return outs[0].reshape(B, 5, 2), outs[1].reshape(B)


def simulate_sharded(make_sim, B, max_steps=200000, check_every=64, group=None, device=None):
    """Closed-loop Monte-Carlo sharded by scenario (SURVEY 8e: "shards the same way by scenario"): rank g drives the
    vehicles [g*B//G, (g+1)*B//G) to their destination on its own GPU -- ``make_sim(lo, hi)`` returns the
    ``BatchedSimulation`` of that shard (its scenarios, its start states; with ``noise=dict(..., first_id=lo)`` it draws
    the unsharded fleet's disturbances) -- with no exchange between ranks while the
    vehicles drive (run_simulation's loop, trajectory_tracking.py:395-410, is per vehicle).  Afterwards the final states
    [B,5], step counts [B] and unsolved-step counts [B] are all-gathered, so every rank returns the whole fleet's
    result; the slowest rank's number of enqueued steps comes back with it (MAX).  Returns a dict."""
    import torch
    dist = _dist()
    on = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if on else 1
    rank = dist.get_rank(group) if on else 0
    lo, hi = shard_bounds(B, rank, world)
    sim = make_sim(lo, hi)
    enq = sim.run(max_steps=max_steps, check_every=check_every) if hi > lo else 0
    x, steps, unsolved = sim.state() if hi > lo else (np.zeros((0, 5)), np.zeros(0, np.int32), np.zeros(0, np.int32))
    out = dict(x=np.asarray(x, dtype=np.float64).reshape(hi - lo, 5), steps=np.asarray(steps, dtype=np.int32),
               unsolved=np.asarray(unsolved, dtype=np.int32), enqueued=int(enq), shard=(lo, hi), sim=sim)
    if world == 1:
        return out
    sizes = [shard_bounds(B, g, world) for g in range(world)]
    pad = max(h - l for l, h in sizes)
    full = {}
    for key, width, dt in (("x", 5, torch.float64), ("steps", 1, torch.int32), ("unsolved", 1, torch.int32)):
        mine = torch.zeros((pad, width), dtype=dt, device=device)
        mine[: hi - lo] = torch.from_numpy(np.ascontiguousarray(out[key]).reshape(hi - lo, width)).to(device=device, dtype=dt)
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine, group=group)
        full[key] = torch.cat([p[: h - l] for p, (l, h) in zip(parts, sizes)]).cpu().numpy()
    e = torch.tensor([out["enqueued"]], dtype=torch.int64, device=device)
    dist.all_reduce(e, op=dist.ReduceOp.MAX, group=group)
    out.update(x=full["x"].reshape(B, 5), steps=full["steps"].reshape(B), unsolved=full["unsolved"].reshape(B),
               enqueued=int(e.cpu()[0]))
    return out
