"""Cost of worlds (mpcb_sim_set_worlds, mpcb_sim_branch_worlds) and the near-miss splitting estimator
(rare_events.near_miss_probability) against crude Monte-Carlo.

  1. following's device time per step (torch.profiler, 20 steps after 8) at 65,536 vehicles on the trajectory3 fleet of
     tools/gpu_sim_fleet.py with FLEET_SOLVER_CAPS, follow_range 30 m: the global path (key kernel, two radix sorts,
     leader kernel) against the world kernel at M = 8, 64 and 1024;
  2. the whole step (CUDA events around 200 steps after 8) and vehicle-steps/s of the same fleet: following off, global,
     and worlds of 8, 64, 1024, alternated over two rounds;
  3. one branch_worlds at 65,536 vehicles (M = 8 and 1024, no histories; host clock around the call and a synchronise,
     median of 20);
  4. near misses of the tight noisy platoons of tests/test_gpu_sim_worlds.py: crude on 65,536 worlds against REPS
     splitting estimates on 8,192 worlds at two lam, with the vehicle-steps each spends and the work-normalised
     variance se^2 x vehicle-steps;
  5. bench.py's headline and closed_loop_fleet lines of this tree and of the tree at PARENT (a checkout of the parent
     commit with its library built), alternated.
Prints the card, its power limit and maximum SM clock beside the numbers.
    python tools/gpu_sim_worlds.py parent=build/parent out=profiles/r05_sim_worlds.json"""
import json, os, statistics, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import safe_autonomous_driving_mpc_b200 as M
from safe_autonomous_driving_mpc_b200.rare_events import near_miss_probability

args = dict(a.split("=", 1) for a in sys.argv[1:])
RANGE, B, WARM, PROF_STEPS, STEPS, ROUNDS, REPS = 30.0, 65536, 8, 20, 200, 2, 8
WORLDS = (8, 64, 1024)


def save():
    if args.get("out"):
        os.makedirs(os.path.dirname(os.path.abspath(args["out"])), exist_ok=True)
        with open(args["out"], "w") as f:
            json.dump(res, f, indent=1)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print("card:", card, flush=True)
res = dict(card=card, follow_range=RANGE, vehicles=B)
L3 = M.TrajectoryLoader(f"{ROOT}/data/trajectory3.npz")
T3 = M.BatchedTracker(L3, **M.FLEET_SOLVER_CAPS)


def fleet_draws(rng, n):
    s0 = rng.uniform(0.0, L3.s_max - 400.0, n)
    xi = np.array([L3.get_state(s) for s in s0])
    xi[:, 4] = np.clip(xi[:, 4], 0.5, None)
    scen = [M.make_scenario(3, tl_pos=float(s + rng.uniform(150, 350)), obs_trigger_s=float(s + 5),
                            obs_start_s=float(s + 60), obs_end_s=float(s + 300)) for s in s0]
    return xi, scen


rng = np.random.default_rng(11)                         # tools/gpu_sim_fleet.py draws the 4,096 fleet first
fleet_draws(rng, 4096)
XI, SCEN = fleet_draws(rng, B)
MODES = {"off": (None, None), "global": (RANGE, None), **{f"world{m}": (RANGE, m) for m in WORLDS}}


def make(mode):
    rng_, ws = MODES[mode]
    return M.BatchedSimulation(T3, SCEN, x_init=XI, follow_range=rng_, world_size=ws)


def follow_us(mode):
    """Device time per step of following's kernels and of all kernels (microseconds)."""
    from torch.profiler import profile, ProfilerActivity
    sim = make(mode)
    sim.step(WARM)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sim.step(PROF_STEPS)
        torch.cuda.synchronize()
    split = dict(follow=0.0, all=0.0)
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if us <= 0:
            continue
        split["all"] += us
        if any(k in ev.key for k in ("mpcb_follow_key_kernel", "mpcb_follow_leader_kernel", "mpcb_follow_world_kernel",
                                     "RadixSort", "Onesweep")):
            split["follow"] += us
    return {k: v / PROF_STEPS for k, v in split.items()}


res["follow_us"] = {}
for mode in MODES:
    if mode == "off":
        continue
    sp = follow_us(mode)
    res["follow_us"][mode] = sp
    print(f"{mode:9s}: following {sp['follow']:.2f} us per step of {sp['all']:.1f} us of kernels", flush=True)
save()


def timed(mode):
    sim = make(mode)
    sim.step(WARM)
    torch.cuda.synchronize()
    st0 = sim.state()[1]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(torch.cuda.default_stream())             # the simulation runs on the legacy default stream
    sim.step(STEPS)
    e1.record(torch.cuda.default_stream())
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    vs = int(sim.state()[1].sum() - st0.sum())
    return dict(ms_per_step=ms / STEPS, vehicle_steps_per_s=vs / (ms * 1e-3))


res["step"] = {m: [] for m in MODES}
for _ in range(ROUNDS):
    for mode in MODES:
        r = timed(mode)
        res["step"][mode].append(r)
        print(f"{mode:9s}: {r['ms_per_step']:.3f} ms per step, {r['vehicle_steps_per_s'] / 1e6:.2f} M vehicle-steps/s",
              flush=True)
save()

res["branch_worlds_ms"] = {}
for m in (8, 1024):
    sim = M.BatchedSimulation(T3, SCEN, x_init=XI, follow_range=RANGE, world_size=m)
    sim.step(1)
    prng = np.random.default_rng(3)
    ts = []
    for _ in range(21):
        p = prng.integers(0, sim.W, sim.W)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sim.branch_worlds(p)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    res["branch_worlds_ms"][m] = statistics.median(ts[1:])
    print(f"branch_worlds, {B} vehicles in worlds of {m}, no histories: {res['branch_worlds_ms'][m]:.3f} ms", flush=True)
    del sim
save()

# 4. near misses of the tight noisy platoons
from test_gpu_sim_worlds import (NEAR_CAP, NEAR_STEPS, PLATOON_RANGE, near_noise,  # noqa: E402
                                 tight_platoons)
L2 = M.TrajectoryLoader(f"{ROOT}/data/trajectory2.npz")
T2 = M.BatchedTracker(L2)
m8, x8, s8 = tight_platoons(L2, 1)


def platoon_sim(W, seed):
    return M.BatchedSimulation(T2, s8 * W, x_init=np.tile(x8, (W, 1)), follow_range=PLATOON_RANGE,
                               noise=near_noise(seed), world_size=m8)


t0 = time.perf_counter()
crude = platoon_sim(65536, 91)
crude.step(NEAR_STEPS)
fail = ~crude.running_follow_check()["ok"].reshape(65536, m8).all(axis=1)
p = float(fail.mean())
vs = int(crude.state()[1].sum())
res["near_miss"] = dict(crude=dict(p=p, se=float(np.sqrt(p * (1 - p) / fail.size)), failures=int(fail.sum()),
                                   vehicle_steps=vs, seconds=time.perf_counter() - t0))
c = res["near_miss"]["crude"]
print(f"near miss, crude on 65,536 worlds: p = {p:.3e} +- {c['se']:.1e} ({c['failures']} worlds, {vs:.3e} "
      f"vehicle-steps, se^2 x vehicle-steps {c['se'] ** 2 * vs:.3e})", flush=True)
del crude
for lam, every in ((2.0, 50), (4.0, 50)):
    ps, vs, t0 = [], 0, time.perf_counter()
    for rep in range(REPS):
        r = near_miss_probability(platoon_sim(8192, 100 + rep), lam, every, seed=rep, gap_cap=NEAR_CAP,
                                  max_steps=NEAR_STEPS)
        ps.append(r["p"])
        vs += r["vehicle_steps"]
    mean, se = float(np.mean(ps)), float(np.std(ps, ddof=1) / np.sqrt(REPS))
    res["near_miss"][f"lam{lam:g}"] = dict(p=ps, mean=mean, se=se, vehicle_steps=vs, every=every,
                                           seconds=time.perf_counter() - t0)
    print(f"near miss, splitting lam {lam:g} every {every}, {REPS} x 8,192 worlds: p = {mean:.3e} +- {se:.1e} "
          f"({vs:.3e} vehicle-steps, se^2 x vehicle-steps {se ** 2 * vs:.3e}): {['%.2e' % q for q in ps]}", flush=True)
save()


def sub(cmd, cwd):
    r = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{cmd} in {cwd} failed:\n{r.stdout[-2000:]}\n{r.stderr[-3000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


PARENT = os.path.abspath(args.get("parent", os.path.join(ROOT, "build", "parent")))
res["bench"] = {}
for _ in range(ROUNDS):
    for name, root in (("parent", PARENT), ("new", ROOT)):
        line = sub([sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "5"], root)
        res["bench"].setdefault(name, []).append(line)
        fl = line.get("closed_loop_fleet", {})
        print(f"bench {name:6s}: {line.get('metric')} {line.get('value'):.4g} {line.get('unit')}; closed_loop_fleet "
              f"{fl.get('vehicle_steps_per_s', float('nan')) / 1e6:.2f} M vehicle-steps/s", flush=True)
save()
