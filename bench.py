#!/usr/bin/env python
"""Benchmark of the batched tracking-MPC solve path (BASELINE.json metric: tracking-MPC solves/s + p99 latency).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]

A "step" is one pass of the hot path (mpcb_solve_batch: warm start -> linearise -> ADMM QP rounds -> outputs) over
one batch of BASELINE config 4: the seeded Monte-Carlo set of 65,536 perturbed states / obstacle scenarios on
trajectory3 (SURVEY.md 8d).  Weak scaling: every rank solves its own 65,536 problems (seed + rank); there is no
collective on the solve path, NCCL only reduces the timing and the statistics.

value     whole-job solves/s with the inputs resident in HBM: K steps enqueued back to back on two handles / streams
          (the robust pass of one batch overlaps the first pass of the next), CUDA events around the K steps, max over
          ranks; `single_call` is one call alone on an idle GPU, `strong` one batch sharded over the ranks + NCCL gather
e2e       the same through the public host API (BatchedTracker.solve_batch_host_async / wait ->
          mpcb_solve_batch_host_async): pinned host buffers in, pinned host buffers out, H2D + kernels + D2H of every
          step inside the timed region, three batches in flight
roofline  neither HBM nor tensor cores bound this path (SURVEY 8d): it is reported against the FP64 FMA pipe,
          algorithmic flops per SURVEY 8d's formula, peak measured in-process by a register-resident DFMA loop
--impl reference   the reference's CPU algorithm (oracle port of trajectory_tracking.py solve(): SLSQP ftol=1e-3,
          maxiter=15, finite differences) on all host cores, bounded sample per step
--dump-outputs DIR   after the timed steps, the outputs of the last timed step of the device-resident arm (what
          mpcb_solve_batch hands its caller) as DIR/<name>.npy in float64, rank 0 only: U, Xpred, obj, status, iters,
          cmin, and the 64-bit active-set mask as its low and high 32-bit halves.  The inputs are seeded, so two builds
          run with the same arguments can be compared output for output.  Above 64 MB a fixed seeded sample of problems
          is written, with its indices in sample_index.npy
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tracking_mpc_qp_solves_per_sec"
UNIT = "solves/s"
BATCH = 65536
TRAJ = os.path.join(ROOT, "data", "trajectory3.npz")
WORKLOAD = "BASELINE config 4: Monte-Carlo 65,536 perturbed states/obstacle scenarios on trajectory3 (seed 20261018)"


# ------------------------------------------------------------------------------------------------
def _cpu_worker_init():
    global _TAB
    from oracle import tracker_port as P
    _TAB = P.RefTable.from_npz(TRAJ)


def _cpu_worker(args):
    from oracle import tracker_port as P
    x0, obs, n = args
    t0 = time.perf_counter()
    P.solve_as_shipped(_TAB, x0, [tuple(o) for o in obs[:n]])
    return time.perf_counter() - t0


def cpu_reference_rate(x0, obs, n, cores):
    """Solves/s of the reference's CPU algorithm (oracle port, as-shipped SLSQP settings) on `cores` processes."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    work = [(x0[i], obs[i], int(n[i])) for i in range(len(n))]
    with ctx.Pool(cores, initializer=_cpu_worker_init) as pool:
        pool.map(_cpu_worker, work[: cores])        # spin-up, untimed
        t0 = time.perf_counter()
        lat = pool.map(_cpu_worker, work, chunksize=max(1, len(work) // (cores * 4)))
        dt = time.perf_counter() - t0
    return len(work) / dt, float(np.mean(lat) * 1e3), float(np.quantile(lat, 0.99) * 1e3)


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU every 100 ms while running."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4,
                 "hw_power_brake_slowdown": 0x80}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------
def algorithmic_flops(iters, n_obs):
    """SURVEY.md 8(d): F_alg = R*F_asm(m) + K_tot*F_it(m), m = 5(7 + 2 n_obs) linearised rows."""
    m = 5.0 * (7.0 + 2.0 * n_obs)
    R = iters[:, 0].astype(np.float64)
    K = iters[:, 1].astype(np.float64)
    return float(np.sum(R * (3900.0 + 110.0 * m) + K * (200.0 + 53.0 * m)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import tracker_port as P
    tab = P.RefTable.from_npz(TRAJ)
    x0, obs, n = P.monte_carlo_problems(tab, BATCH)
    cores = host_cores()
    per_step = max(64, 16 * cores)
    _cpu_worker_init()
    times = []
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_worker_init) as pool:
        for step in range(args.warmup + args.steps):
            lo = (step * per_step) % (BATCH - per_step)
            work = [(x0[i], obs[i], int(n[i])) for i in range(lo, lo + per_step)]
            t0 = time.perf_counter()
            pool.map(_cpu_worker, work, chunksize=max(1, per_step // (cores * 4)))
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
    ms = float(np.mean(times) * 1e3)
    val = per_step / (ms * 1e-3)
    sample = f"{per_step} consecutive problems of the seeded 65,536 set per step, oracle port of solve() as shipped"
    line = {"metric": METRIC, "value": val, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample_per_step": per_step, "solver": "scipy SLSQP ftol=1e-3 maxiter=15"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=_OUT, flush=True)
    return 0


N_HANDLES = 2      # device-resident arm: batches in flight (one handle + one stream each); measured on B200: 1 handle
                   # 0.556 ms per batch, 2: 0.396, 3: 0.410, 4: 0.444 (tools/gpu_pipeline.py)
N_HANDLES_E2E = 3  # host arm (tools/gpu_e2e_pipe.py): every output 1 / 2 / 3 / 4 handles 1.06 / 0.92 / 0.55 / 0.59 ms per batch,
                   # closed-loop form 0.71 / 0.51 / 0.44 / 0.44
N_SETS = 8         # distinct seeded 65,536-problem sets the steps rotate over: 8 x 28 MB of inputs + outputs > 126 MB L2
DUMP_LIMIT = 64 << 20   # bytes --dump-outputs may write (at the default batch every output fits: 24 MB)


def dump_outputs(out, dirname):
    """Write the device outputs of one solve_batch call as dirname/<name>.npy, float64 (exact for every field; the
    active-set mask is split into its low and high 32-bit halves).  Returns the number of bytes written."""
    arrs = {k: v.cpu().numpy() for k, v in out.items()}
    act = arrs["active"].view(np.uint64)
    arrs["active"] = np.stack([act & np.uint64(0xFFFFFFFF), act >> np.uint64(32)], axis=1)
    arrs = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrs.items()}
    B = len(arrs["obj"])
    row = sum(a.nbytes for a in arrs.values()) // max(B, 1)
    slack = 4096                                              # .npy headers
    if B * row + slack > DUMP_LIMIT:
        m = (DUMP_LIMIT - slack) // (row + 8)                  # + 8: the index of each sampled problem
        idx = np.sort(np.random.default_rng(0).choice(B, m, replace=False))
        arrs = {k: v[idx] for k, v in arrs.items()}
        arrs["sample_index"] = idx.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, v in arrs.items():
        np.save(os.path.join(dirname, k + ".npy"), v)
    return sum(a.nbytes for a in arrs.values())


def traffic_from_profile():
    """dram bytes per step of the two solve launches, from the committed ncu --set full capture of this workload."""
    f = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(f):
        return None, None
    t = json.load(open(f))
    return float(t["first_pass_dram_bytes"]) + float(t["second_pass_dram_bytes"]), t.get("source")


def config_extras(M, P, dev, torch):
    """BASELINE configs 1-3 (closed loops through the reference-shaped B = 1 call, and as a device loop of 4,096
    vehicles) and config 5 (planner Hermite-Simpson evaluation, x64 tile, with its own HBM roofline)."""
    from safe_autonomous_driving_mpc_b200 import environment as E
    out = {}
    for i in (1, 2, 3):
        traj = os.path.join(ROOT, "data", f"trajectory{i}.npz")
        L = M.TrajectoryLoader(traj)
        T = M.BatchedTracker(L, device=dev.index)
        sc = {1: None, 2: E.SCENARIO_TRAJECTORY2, 3: E.SCENARIO_TRAJECTORY3}[i]
        fsm = M.ObstaclesFSM(i > 1, i > 1, scenario=sc)
        flags = []
        t0 = time.perf_counter()
        hx, hu, ht, *_ = M.run_simulation(T, fsm, L, record_flags=flags)
        wall = time.perf_counter() - t0
        ht = np.array(ht[5:]) * 1e3
        st = np.array([f[0] for f in flags])
        scen = M.make_scenario(2, dynamic_obstacle=0, traffic_light=0) if i == 1 else M.make_scenario(i)
        nveh = 4096
        sim = M.BatchedSimulation(T, scen, B=nveh)
        sim.step(8)
        torch.cuda.synchronize()
        sim = M.BatchedSimulation(T, scen, B=nveh)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sim.run(max_steps=len(hu) + 64, check_every=128)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        _, steps, _ = sim.state()
        sim = M.BatchedSimulation(T, scen, B=nveh, hot_start=True)      # previous plan, advanced one step, as the start
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sim.run(max_steps=len(hu) + 64, check_every=128)
        torch.cuda.synchronize()
        dt_hot = time.perf_counter() - t0
        _, steps_hot, _ = sim.state()
        out[f"config{i + 0}_trajectory{i}_closed_loop"] = {
            "steps": int(len(hu)), "status_hist": np.bincount(st, minlength=3).tolist(), "wall_s": wall,
            "solve_ms_p50": float(np.median(ht)), "solve_ms_p99": float(np.quantile(ht, 0.99)),
            "device_loop_vehicles": nveh, "device_loop_vehicle_steps_per_s": float(steps.sum() / dt),
            "device_loop_hot_start_vehicle_steps_per_s": float(steps_hot.sum() / dt_hot),
            "device_loop_hot_start_steps": int(steps_hot[0]),
            "reference": "trajectory_tracking.py:377-443"}
        del sim, T
    traj3 = os.path.join(ROOT, "data", "trajectory3.npz")
    L = M.TrajectoryLoader(traj3)
    T = M.BatchedTracker(L, device=dev.index)
    z3 = np.load(traj3)
    N = len(z3["U"])
    Ev = M.PlannerEvaluator(T, N=N, simpson_sign=+1)
    z = Ev.pack(z3["X"], z3["U"], z3["S"])
    tiles = 64
    zt = torch.from_numpy(np.tile(z, (tiles, 1))).to(dev)
    lam = torch.from_numpy(np.random.default_rng(7).normal(size=(tiles, N, 5))).to(dev)
    o = Ev.eval_defects(zt, lam=lam, want_jac=True, want_hess=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ms = []
    for _ in range(12):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        Ev.eval_defects(zt, lam=lam, want_jac=True, want_hess=True, out=o)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms = float(np.median(ms[2:]))
    n_int = tiles * N
    byt = n_int * (5 + 60 + 144 + 5) * 8 + tiles * (8 * N + 5) * 8      # defects + Jacobian + Hessian blocks out, lam + z in
    mp_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak = json.load(open(mp_file))["hbm_gbs"] if os.path.exists(mp_file) else 6650.0
    out["config5_planner_hs_eval_x64"] = {
        "intervals": n_int, "ms": ms, "intervals_per_s": n_int / ms * 1e3,
        "roofline": {"bound": "hbm", "achieved": byt / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
                     "frac": byt / ms / 1e6 / hbm_peak, "bytes_per_interval": byt / n_int},
        "reference": "trajectory_planning.py:183-208"}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        # CPU baseline first, before this process owns a CUDA context (the worker pool forks)
        from oracle import tracker_port as P0
        tab0 = P0.RefTable.from_npz(TRAJ)
        cx0, cobs, cn = P0.monte_carlo_problems(tab0, BATCH)
        cores = host_cores()
        ns = 2048                                              # SURVEY 8(d): "oracle/CPU timing on the first 2,048 problems"
        v, mean_ms, p99_ms = cpu_reference_rate(cx0[:ns], cobs[:ns], cn[:ns], cores)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {ns} problems of the same seeded set, oracle port of the reference solve() as "
                         f"shipped (SLSQP ftol=1e-3, maxiter=15, FD gradients); mean {mean_ms:.1f} ms, p99 "
                         f"{p99_ms:.1f} ms per solve"}
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import safe_autonomous_driving_mpc_b200 as M
    from oracle import tracker_port as P        # problem generator + cpu_baseline leg only
    B = args.batch
    loader = M.TrajectoryLoader(TRAJ)
    trackers = [M.BatchedTracker(loader, device=local) for _ in range(max(N_HANDLES, N_HANDLES_E2E))]
    tracker = trackers[0]
    tab = P.RefTable.from_npz(TRAJ)
    # weak scaling: every rank its own N_SETS seeded sets (set 0 of rank 0 is THE BASELINE config-4 set)
    host_sets = [P.monte_carlo_problems(tab, B, seed=P.MC_SEED + rank * N_SETS + k) for k in range(N_SETS)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: N_HANDLES batches in flight on as many streams ----------------------------
    dsets = [[torch.from_numpy(a).to(dev) for a in hs] for hs in host_sets]
    outs = [tracker.solve_batch(*ds) for ds in dsets]
    torch.cuda.synchronize()
    peak_tf, _ = tracker.measure_fp64_peak()
    flops_set = [algorithmic_flops(o["iters"].cpu().numpy(), hs[2].astype(np.float64)) for o, hs in zip(outs, host_sets)]
    streams = [torch.cuda.Stream(dev) for _ in range(N_HANDLES)]
    main = torch.cuda.current_stream(dev)

    def pipelined(nsteps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for s_ in streams:
            s_.wait_event(e0)
        for i in range(nsteps):
            k = i % N_SETS
            trackers[i % N_HANDLES].solve_batch(*dsets[k], out=outs[k], stream=streams[i % N_HANDLES].cuda_stream)
        for s_ in streams:
            ev = torch.cuda.Event()
            ev.record(s_)
            main.wait_event(ev)
        e1.record(main)
        return e0, e1

    pipelined(max(args.warmup, 3))        # warm-up steps (every input set has been solved once before, too)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = sum(t.launch_count() for t in trackers)
    barrier()
    t_wall0 = time.perf_counter()
    e0, e1 = pipelined(args.steps)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms_dev = e0.elapsed_time(e1) / args.steps
    launches = sum(t.launch_count() for t in trackers) - launches0
    flops_step = float(np.mean([flops_set[i % N_SETS] for i in range(args.steps)]))
    if args.dump_outputs and rank == 0:
        # the last timed step solved set (steps - 1) % N_SETS into its output buffers; later blocks reuse outs[0]
        k_last = (args.steps - 1) % N_SETS
        nbytes = dump_outputs(outs[k_last], args.dump_outputs)
        print(f"bench.py: outputs of timed step {args.steps - 1} (input set {k_last}) written to {args.dump_outputs} "
              f"({nbytes / 1e6:.1f} MB)", file=sys.stderr)

    # ---- one call alone (latency of a whole batch, per-pass times), L2 flushed between calls ---------------
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    single = []
    for it in range(3 + 10):
        flush.zero_()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        tracker.solve_batch(*dsets[0], out=outs[0])
        a1.record()
        torch.cuda.synchronize()
        if it >= 3:
            single.append(a0.elapsed_time(a1))
    pass_ms = tracker.last_pass_ms()
    ms_single = float(np.mean(single))

    # ---- strong scaling: ONE 65,536-problem batch (rank 0's set 0) sharded over the ranks, results all-gathered ----
    x0s, obss, ns_ = P.monte_carlo_problems(tab, B, seed=P.MC_SEED)
    lo, hi = M.sharding.shard_bounds(B, rank, world)
    sx0, sobs, sn = (torch.from_numpy(np.ascontiguousarray(a[lo:hi])).to(dev) for a in (x0s, obss, ns_))
    sout = tracker.solve_batch(sx0, sobs, sn)
    strong_solve, strong_gather = [], []
    for it in range(3 + 10):
        flush.zero_()
        barrier()
        a0, a1, a2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a0.record()
        tracker.solve_batch(sx0, sobs, sn, out=sout)
        a1.record()
        full = M.sharding.gather_device(sout["U"], sout["status"], B)        # NCCL all_gather, after the solve
        a2.record()
        torch.cuda.synchronize()
        if it >= 3:
            strong_solve.append(a0.elapsed_time(a1))
            strong_gather.append(a1.elapsed_time(a2))
    sp = tracker.last_pass_ms()
    strong_ms = float(np.mean(strong_solve)) + float(np.mean(strong_gather))
    del full

    # ---- closed loop sharded by scenario: every rank drives its own 4,096 vehicles down trajectory3 (config 3's scenario)
    # without leaving the GPU; no exchange while they drive (SURVEY 8e) -------------------------------------------------
    nveh = 4096
    scen3 = M.make_scenario(3)
    sim = M.BatchedSimulation(tracker, scen3, B=nveh)
    sim.step(8)
    torch.cuda.synchronize()
    sim = M.BatchedSimulation(tracker, scen3, B=nveh)
    barrier()
    t0 = time.perf_counter()
    sim.run(max_steps=2294 + 64, check_every=128)
    torch.cuda.synchronize()
    fleet_s = time.perf_counter() - t0
    _, fsteps, _ = sim.state()
    fleet_steps = int(fsteps.sum())
    del sim

    # ---- end-to-end arm: public host API (asynchronous form, N_HANDLES_E2E batches in flight), pinned host buffers,
    # H2D + kernels + D2H inside the timed region; full outputs, and the closed-loop form (U*[0] + status) beside it ----
    PB = M.tracker.PinnedBuffer
    keep = []

    def pinned(a):
        b_ = PB(a.shape, a.dtype)
        b_.array[...] = a
        keep.append(b_)
        return b_.array

    def pinned_out(spec):
        o_ = {}
        for k_, (shp, dt_) in spec.items():
            b_ = PB(shp, dt_)
            keep.append(b_)
            o_[k_] = b_.array
        return o_

    FULL = dict(U=((B, 5, 2), np.float64), Xpred=((B, 6, 5), np.float64), obj=((B,), np.float64),
                status=((B,), np.int32), iters=((B, 2), np.int32), cmin=((B,), np.float64), active=((B,), np.uint64))
    U0 = dict(u0=((B, 2), np.float64), status=((B,), np.int32))
    nh = N_HANDLES_E2E
    pins = [[pinned(a) for a in host_sets[k]] for k in range(nh)]

    def e2e_run(spec_outs, nsteps):
        t0 = time.perf_counter()
        for i in range(nsteps):
            k = i % nh
            if i >= nh:
                trackers[k].wait()
            trackers[k].solve_batch_host_async(*pins[k], spec_outs[k])
        for k in range(nh):
            trackers[k].wait()
        return (time.perf_counter() - t0) / nsteps * 1e3

    e2e_ms = {}
    for name, spec in (("full", FULL), ("closed_loop", U0)):
        po = [pinned_out(spec) for _ in range(nh)]
        e2e_run(po, 3 * nh)
        barrier()
        e2e_ms[name] = e2e_run(po, args.steps)
        barrier()
        if name == "full":
            res = po[0]
    clocks = sampler.stop()
    h2d = B * (40 + 32 + 4)
    d2h = B * (80 + 240 + 8 + 4 + 8 + 8 + 8)

    status = res["status"].copy()
    iters = res["iters"].copy()
    # NCCL is used only here, after the timed regions: MAX of the times, SUM of the statistics (no collective on the
    # solve path, SURVEY 8e)
    red = {k: M.sharding.reduce_stats(status, iters, v, device=dev)
           for k, v in (("dev", ms_dev), ("single", ms_single), ("e2e", e2e_ms["full"]), ("e2e_cl", e2e_ms["closed_loop"]),
                        ("strong", strong_ms), ("strong_first_max", sp[0]), ("strong_second_max", sp[1]),
                        ("strong_first_min", -sp[0]), ("strong_second_min", -sp[1]), ("fleet", fleet_s * 1e3))}
    tot = red["dev"]
    ms_dev_max = tot["ms_max"]
    hist = [tot["solved"], tot["maxiter"], tot["infeasible"]]

    if rank == 0:
        # single-solve latency through the reference-shaped call (B = 1, host API, includes launch + copies)
        x0, obs, n = host_sets[0]
        lat = []
        for i in range(320):
            o = [{"s": float(obs[i, k, 0]), "v": float(obs[i, k, 1]), "type": "car"} for k in range(int(n[i]))]
            t0 = time.perf_counter()
            tracker.solve(x0[i], o)
            lat.append((time.perf_counter() - t0) * 1e3)
        lat = np.array(lat[20:])
        achieved = flops_step / (ms_dev * 1e-3) / 1e12
        hbm_bytes = B * 416.0
        mp_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak = json.load(open(mp_file))["hbm_gbs"] if os.path.exists(mp_file) else 6650.0
        traffic, traffic_src = traffic_from_profile()
        iters0 = outs[0]["iters"].cpu().numpy()
        roofline = {"bound": "fp64", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": achieved / peak_tf,
                    # dram__bytes_read.sum + dram__bytes_write.sum of the two solve launches of one step, read from the
                    # committed ncu --set full capture of this workload; algorithmic bytes are 416 B/solve = 27.3 MB
                    "traffic": traffic, "traffic_source": traffic_src,
                    "note": "path is bound by the FP64 FMA pipe, not HBM or tensor cores (SURVEY 8d); peak = DFMA "
                            "loop measured in this run (mpcb_measure_fp64_peak); flops per SURVEY 8d formula with "
                            "the kernel's own per-problem round/iteration counts, over the step time of the timed "
                            "region (batches in flight overlap, so no kernel is timed alone there)",
                    "dominant_kernel": {"name": "mpcb_solve_cls_kernel (first pass, thread per problem, one instantiation per obstacle count)",
                                        "ms_alone": pass_ms[0],
                                        "achieved_alone": algorithmic_flops(iters0, host_sets[0][2].astype(np.float64))
                                        / ((pass_ms[0] + pass_ms[1]) * 1e-3) / 1e12},
                    "mean_rounds": float(iters0[:, 0].mean()), "mean_admm_iters": float(iters0[:, 1].mean()),
                    "hbm": {"achieved": hbm_bytes / (ms_dev * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": hbm_bytes / (ms_dev * 1e-3) / 1e9 / hbm_peak,
                            "peak_source": "measured" if os.path.exists(mp_file) else "fallback"}}
        line = {"metric": METRIC, "value": B * world / (ms_dev_max * 1e-3), "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev_max,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "batch_per_gpu": B, "horizon": 5, "n_var": 10,
                           "l2": f"inputs larger than L2: the steps rotate over {N_SETS} seeded sets per GPU "
                                 f"({N_SETS} x {B * 416 / 1e6:.0f} MB of inputs and outputs against 126 MB of L2)",
                           "in_flight": f"{N_HANDLES} batches (one handle and stream each): the robust pass of one batch "
                                        "overlaps the first pass of the next",
                           "parallelism": f"batch-sharded x{world}"},
                # headline: the closed-loop form of the host call -- U*[0] and status, what run_simulation consumes from
                # solve() (trajectory_tracking.py:401-406); the call that also brings back U*, predict(x0, U*), objective,
                # iteration counts, cmin and the active set is timed beside it
                "e2e": {"value": B * world / (red["e2e_cl"]["ms_max"] * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": B * 20, "ms_per_step": red["e2e_cl"]["ms_max"], "copies_declared": True,
                        "api": f"BatchedTracker.solve_batch_host_async(out = u0, status) / wait, {nh} batches in flight",
                        "every_output": {"value": B * world / (red["e2e"]["ms_max"] * 1e-3), "unit": UNIT,
                                         "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                         "ms_per_step": red["e2e"]["ms_max"],
                                         "note": "U*, predict(x0, U*), objective, status, iteration counts, cmin, active "
                                                 "set: 356 B per solve over the one device-to-host engine"}},
                "gpu_launches": int(launches) * world,
                "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
                "single_call": {"ms": red["single"]["ms_max"], "solves_per_s": B * world / (red["single"]["ms_max"] * 1e-3),
                                "first_ms": pass_ms[0], "second_ms": pass_ms[1], "second_pass_problems": pass_ms[2],
                                "note": "one mpcb_solve_batch call alone on an idle GPU, L2 flushed before it (256 MiB "
                                        "write): the robust pass's latency tail is exposed"},
                "strong": {"problems": B, "ms": red["strong"]["ms_max"], "solves_per_s": B / (red["strong"]["ms_max"] * 1e-3),
                           "gather_ms": float(np.mean(strong_gather)),
                           "first_ms_max": red["strong_first_max"]["ms_max"], "first_ms_min": -red["strong_first_min"]["ms_max"],
                           "second_ms_max": red["strong_second_max"]["ms_max"],
                           "second_ms_min": -red["strong_second_min"]["ms_max"],
                           "note": "ONE 65,536-problem batch, shard [g*B/G, (g+1)*B/G) per GPU, U and status all-gathered "
                                   "with NCCL after the solve (gather_ms: rank 0)"},
                "closed_loop_fleet": {"vehicles": nveh * world, "vehicle_steps": fleet_steps * world,
                                      "seconds": red["fleet"]["ms_max"] * 1e-3,
                                      "vehicle_steps_per_s": fleet_steps * world / (red["fleet"]["ms_max"] * 1e-3),
                                      "note": "trajectory3 with its car and red light, 4,096 vehicles per GPU driven to the "
                                              "destination on the device (FSM -> solve -> plant step), sharded by scenario: "
                                              "no exchange between ranks; slowest rank's wall time"},
                "latency": {"B": 1, "p50_ms": float(np.median(lat)), "p99_ms": float(np.quantile(lat, 0.99)),
                            "n": int(len(lat)), "path": "BatchedTracker.solve (host API, includes copies + launch)"},
                "status_hist": {"solved": hist[0], "maxiter": hist[1], "infeasible": hist[2]},
                "wall_s_timed_region": t_wall}
        if not args.no_extras:
            line["configs"] = config_extras(M, P, dev, torch)
        print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def _quiet_stdout():
    """Libraries (NCCL's version banner, for one) write to fd 1; the contract is ONE JSON line on stdout.  Point fd 1 at
    stderr for the duration of the run and return a writer on the real stdout for the final line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the closed-loop / planner lines of configs 1-3 and 5")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    global _OUT
    _OUT = _quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
