"""Cost of following (mpcb_sim_set_follow) in the device closed loop: the staggered trajectory3 fleets of
tools/gpu_sim_fleet.py at 4,096 and 65,536 vehicles with FLEET_SOLVER_CAPS, following off and on, alternated in one run.
Prints the card, its power limit, vehicle-steps/s of each run (CUDA events around 400 steps after 8 warm-up steps) and,
from a separate torch.profiler pass over 20 steps of the fleet with following on, the device time per step of the key
kernel, the two radix sorts and the leader kernel against the whole step.
    python tools/gpu_sim_follow.py [follow_range=30] [out=PATH.json]"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import safe_autonomous_driving_mpc_b200 as M

args = dict(a.split("=") for a in sys.argv[1:])
RANGE = float(args.get("follow_range", 30.0))
OUT = args.get("out")
STEPS, WARM, ROUNDS, PROF_STEPS = 400, 8, 2, 20

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print("card:", card, "| follow_range", RANGE, "m", flush=True)
L = M.TrajectoryLoader(f"{ROOT}/data/trajectory3.npz")
T = M.BatchedTracker(L, **M.FLEET_SOLVER_CAPS)


def fleet(B):
    """tools/gpu_sim_fleet.py's fleet of B vehicles (same seed and draws)."""
    rng = np.random.default_rng(11)
    if B == 65536:                                      # gpu_sim_fleet.py draws the 4,096 fleet first
        fleet_draws(rng, 4096)
    return fleet_draws(rng, B)


def fleet_draws(rng, B):
    s0 = rng.uniform(0.0, L.s_max - 400.0, B)
    xi = np.array([L.get_state(s) for s in s0])
    xi[:, 4] = np.clip(xi[:, 4], 0.5, None)
    scen = [M.make_scenario(3, tl_pos=float(s + rng.uniform(150, 350)), obs_trigger_s=float(s + 5),
                            obs_start_s=float(s + 60), obs_end_s=float(s + 300)) for s in s0]
    return xi, scen


def timed(B, xi, scen, follow):
    sim = M.BatchedSimulation(T, scen, x_init=xi, follow_range=RANGE if follow else None)
    sim.step(WARM)
    torch.cuda.synchronize()
    _x, st0, _u = sim.state()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(torch.cuda.default_stream())             # the simulation runs on the legacy default stream
    sim.step(STEPS)
    e1.record(torch.cuda.default_stream())
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    _x, st, uns = sim.state()
    vs = int(st.sum() - st0.sum())
    return dict(ms_per_step=ms / STEPS, vehicle_steps_per_s=vs / (ms * 1e-3), alive=sim.alive(), unsolved=int(uns.sum()))


def kernel_split(xi, scen):
    """Device time per step of the following kernels against all kernels of the step (torch.profiler, CUDA)."""
    from torch.profiler import profile, ProfilerActivity
    sim = M.BatchedSimulation(T, scen, x_init=xi, follow_range=RANGE)
    sim.step(WARM)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sim.step(PROF_STEPS)
        torch.cuda.synchronize()
    split = dict(key=0.0, sort=0.0, leader=0.0, all=0.0)
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if us <= 0:
            continue
        name = ev.key
        split["all"] += us
        if "mpcb_follow_key_kernel" in name:
            split["key"] += us
        elif "mpcb_follow_leader_kernel" in name:
            split["leader"] += us
        elif "DeviceRadixSort" in name or "Onesweep" in name or "RadixSort" in name:
            split["sort"] += us
    return {k: v / PROF_STEPS for k, v in split.items()}       # microseconds per step


res = dict(card=card, follow_range=RANGE, steps=STEPS, runs={})
for B in (4096, 65536):
    xi, scen = fleet(B)
    runs = {"off": [], "on": []}
    for _ in range(ROUNDS):
        for mode in ("off", "on"):
            r = timed(B, xi, scen, mode == "on")
            runs[mode].append(r)
            print(f"fleet {B:6d} following {mode:3s}: {r['ms_per_step']:.3f} ms/step, "
                  f"{r['vehicle_steps_per_s'] / 1e6:.2f} M vehicle-steps/s, unsolved vehicle-steps {r['unsolved']}",
                  flush=True)
    sp = kernel_split(xi, scen)
    print(f"fleet {B:6d} following on, device time per step (torch.profiler, {PROF_STEPS} steps): key "
          f"{sp['key']:.1f} us, sorts {sp['sort']:.1f} us, leader {sp['leader']:.1f} us; together "
          f"{sp['key'] + sp['sort'] + sp['leader']:.1f} us of {sp['all']:.1f} us of kernels "
          f"({100 * (sp['key'] + sp['sort'] + sp['leader']) / sp['all']:.2f} %)", flush=True)
    off_ms = float(np.median([r["ms_per_step"] for r in runs["off"]]))
    print(f"fleet {B:6d}: following kernels = {100 * (sp['key'] + sp['sort'] + sp['leader']) * 1e-3 / off_ms:.2f} % "
          f"of a step with following off ({off_ms:.3f} ms)", flush=True)
    res["runs"][B] = dict(runs=runs, kernels_us_per_step=sp)
if OUT:
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        json.dump(res, f, indent=1)
