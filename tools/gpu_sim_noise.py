"""Cost and use of seeded disturbances (mpcb_sim_set_noise) in the device closed loop: the staggered trajectory3 fleets
of tools/gpu_sim_fleet.py at 4,096 and 65,536 vehicles with FLEET_SOLVER_CAPS, noise off and on (all three channels at
the base level below), alternated in one run.  Prints the card, its power limit and maximum SM clock, vehicle-steps/s
of each run (CUDA events around 400 steps after 8 warm-up steps) and, from separate torch.profiler passes over 20 steps
with noise off and on, the device time per step of the FSM and plant kernels (the two kernels noise changes) against
all kernels of the step.  Then the pass rate of every check item (mpcb_sim_check) of the 4,096-vehicle fleet driven to
its destination with the noise at 0, 0.5, 1 and 2 times the base level.
    python tools/gpu_sim_noise.py [out=PATH.json]"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import safe_autonomous_driving_mpc_b200 as M

args = dict(a.split("=") for a in sys.argv[1:])
OUT = args.get("out")
STEPS, WARM, ROUNDS, PROF_STEPS, SWEEP_MAX = 400, 8, 2, 20, 3000
SEED = 7
# base level, per component: measurement of (s, d, o, k, v), actuation of (u1, u2), process noise per 0.2 s step
BASE = dict(meas=[0.05, 0.02, 0.005, 0.001, 0.05], act=[0.02, 0.1], proc=[0.01, 0.005, 0.002, 0.0005, 0.02])
SCALES = (0.0, 0.5, 1.0, 2.0)

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print("card:", card, "| base noise", BASE, flush=True)
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


def noise(scale):
    return None if scale == 0.0 else dict(seed=SEED, **{k: [scale * v for v in vs] for k, vs in BASE.items()})


def timed(xi, scen, on):
    sim = M.BatchedSimulation(T, scen, x_init=xi, noise=noise(1.0 if on else 0.0))
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


def kernel_split(xi, scen, on):
    """Device time per step of the FSM and plant kernels against all kernels of the step (torch.profiler, CUDA)."""
    from torch.profiler import profile, ProfilerActivity
    sim = M.BatchedSimulation(T, scen, x_init=xi, noise=noise(1.0 if on else 0.0))
    sim.step(WARM)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sim.step(PROF_STEPS)
        torch.cuda.synchronize()
    split = dict(fsm=0.0, plant=0.0, all=0.0)
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if us <= 0:
            continue
        split["all"] += us
        if "mpcb_fsm_kernel" in ev.key:
            split["fsm"] += us
        elif "mpcb_plant_kernel" in ev.key:
            split["plant"] += us
    return {k: v / PROF_STEPS for k, v in split.items()}       # microseconds per step


def sweep(xi, scen):
    """Pass rate of every check item with the fleet driven to its destination, noise at each scale of BASE."""
    out = {}
    for scale in SCALES:
        sim = M.BatchedSimulation(T, scen, x_init=xi, history_steps=SWEEP_MAX, noise=noise(scale))
        n = sim.run(max_steps=SWEEP_MAX, check_every=100)
        v = sim.check()
        _x, _st, uns = sim.state()
        rates = {k: float(np.mean(v[k])) for k in M.BatchedSimulation.CHECKS + ("passed",)}
        out[scale] = dict(steps=n, unsolved_per_vehicle_step=float(uns.sum() / v["steps"].sum()), pass_rate=rates)
        print(f"sweep sigma x {scale:3.1f}: {n} steps, " + ", ".join(f"{k} {100 * r:.2f} %" for k, r in rates.items()) +
              f"; unsolved {100 * out[scale]['unsolved_per_vehicle_step']:.3f} % of vehicle-steps", flush=True)
        del sim
    return out


res = dict(card=card, base=BASE, seed=SEED, steps=STEPS, runs={})
for B in (4096, 65536):
    xi, scen = fleet(B)
    runs = {"off": [], "on": []}
    for _ in range(ROUNDS):
        for mode in ("off", "on"):
            r = timed(xi, scen, mode == "on")
            runs[mode].append(r)
            print(f"fleet {B:6d} noise {mode:3s}: {r['ms_per_step']:.3f} ms/step, "
                  f"{r['vehicle_steps_per_s'] / 1e6:.2f} M vehicle-steps/s, unsolved vehicle-steps {r['unsolved']}",
                  flush=True)
    sp = {mode: kernel_split(xi, scen, mode == "on") for mode in ("off", "on")}
    for mode in ("off", "on"):
        print(f"fleet {B:6d} noise {mode:3s}, device time per step (torch.profiler, {PROF_STEPS} steps): fsm "
              f"{sp[mode]['fsm']:.1f} us, plant {sp[mode]['plant']:.1f} us, together "
              f"{sp[mode]['fsm'] + sp[mode]['plant']:.1f} us of {sp[mode]['all']:.1f} us of kernels", flush=True)
    extra = sp["on"]["fsm"] + sp["on"]["plant"] - sp["off"]["fsm"] - sp["off"]["plant"]
    print(f"fleet {B:6d}: noise adds {extra:.1f} us per step to the fsm and plant kernels", flush=True)
    res["runs"][B] = dict(runs=runs, kernels_us_per_step=sp, fsm_plant_extra_us=extra)
res["sweep_4096"] = sweep(*fleet(4096))
if OUT:
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        json.dump(res, f, indent=1)
