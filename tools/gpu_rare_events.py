"""Cost of the running verdicts and of branching, and the splitting estimator (rare_events.offroad_probability) against
crude Monte-Carlo, on the trajectory3 fleets of tools/gpu_sim_noise.py with FLEET_SOLVER_CAPS and its base noise level.

  1. FSM + plant kernel time per step (torch.profiler, 20 steps after 8, noise on at the base level) of this tree against
     the tree at PARENT (a checkout of the parent commit with its library built), alternated in one run, at 4,096 and
     65,536 vehicles; and bench.py's headline and closed_loop_fleet lines of both trees, alternated;
  2. the time of one mpcb_sim_branch (random parents; host clock around the call and a synchronise, median of 20) at
     4,096 and 65,536 vehicles without histories, and with 100 and 200 recorded rows;
  3. at twice the base noise (crude sees 10^-3 - 10^-2 on_road failures) and at the base level: a crude estimate on
     65,536 drives (16 noise draws of the 4,096 starts) against REPS splitting estimates on 4,096 vehicles, with the
     vehicle-steps each spends.  Every drive is cut at MAX_DRIVE steps.
Prints the card, its power limit and maximum SM clock beside the numbers.
    python tools/gpu_rare_events.py parent=build/parent out=profiles/r04_rare_events.json"""
import json, os, statistics, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

args = dict(a.split("=", 1) for a in sys.argv[1:])
PROF_STEPS, WARM, ROUNDS, MAX_DRIVE, REPS, EVERY = 20, 8, 2, 4000, 8, 500
BASE = dict(meas=[0.05, 0.02, 0.005, 0.001, 0.05], act=[0.02, 0.1], proc=[0.01, 0.005, 0.002, 0.0005, 0.02])


def noise(scale, seed=7):
    return dict(seed=seed, **{k: [scale * v for v in vs] for k, vs in BASE.items()})


def setup(root):
    sys.path.insert(0, root)
    import numpy as np
    import safe_autonomous_driving_mpc_b200 as M
    L = M.TrajectoryLoader(f"{root}/data/trajectory3.npz")
    T = M.BatchedTracker(L, **M.FLEET_SOLVER_CAPS)

    def fleet(B):
        """tools/gpu_sim_fleet.py's fleet of B vehicles (same seed and draws)."""
        rng = np.random.default_rng(11)
        if B == 65536:
            draws(rng, 4096)
        return draws(rng, B)

    def draws(rng, B):
        s0 = rng.uniform(0.0, L.s_max - 400.0, B)
        xi = np.array([L.get_state(s) for s in s0])
        xi[:, 4] = np.clip(xi[:, 4], 0.5, None)
        scen = [M.make_scenario(3, tl_pos=float(s + rng.uniform(150, 350)), obs_trigger_s=float(s + 5),
                                obs_start_s=float(s + 60), obs_end_s=float(s + 300)) for s in s0]
        return xi, scen
    return np, M, T, fleet


def worker_kernels(root, B):
    """Device time per step of the FSM and plant kernels and of all kernels (microseconds), in the tree at root."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    np, M, T, fleet = setup(root)
    xi, scen = fleet(B)
    sim = M.BatchedSimulation(T, scen, x_init=xi, noise=noise(1.0))
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
    print(json.dumps({k: v / PROF_STEPS for k, v in split.items()}))


def sub(cmd, cwd):
    r = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{cmd} in {cwd} failed:\n{r.stdout[-2000:]}\n{r.stderr[-3000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def branch_costs(np, M, T, fleet):
    import torch
    out = {}
    for B in (4096, 65536):
        xi, scen = fleet(B)
        rng = np.random.default_rng(3)
        for rows in (0, 100, 200):
            sim = M.BatchedSimulation(T, scen, x_init=xi, history_steps=rows, noise=noise(1.0))
            sim.step(max(rows, 1))
            ts = []
            for _ in range(21):
                p = rng.integers(0, B, B)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                sim.branch(p)
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            out[f"{B}_{rows}"] = statistics.median(ts[1:])
            print(f"branch {B:6d} vehicles, {rows:3d} recorded rows (noise history on): {out[f'{B}_{rows}']:.3f} ms",
                  flush=True)
            del sim
        print(f"branch {B:6d}: +{(out[f'{B}_200'] - out[f'{B}_0']) / 2:.3f} ms per 100 recorded rows", flush=True)
    return out


def estimates(np, M, T, fleet):
    from safe_autonomous_driving_mpc_b200.rare_events import offroad_probability
    xi, scen = fleet(4096)
    out = {}
    for scale, lam in ((2.0, 4.0), (1.0, 4.0), (1.0, 12.0)):
        key = f"x{scale:g}"
        if key not in out:
            t0 = time.perf_counter()
            crude = M.BatchedSimulation(T, scen * 16, x_init=np.tile(xi, (16, 1)), noise=noise(scale, 91))
            n = crude.run(max_steps=MAX_DRIVE, check_every=100)
            r = crude.running_check()
            fail = ~r["on_road"]
            p = float(fail.mean())
            out[key] = dict(crude=dict(p=p, se=float(np.sqrt(p * (1 - p) / fail.size)), failures=int(fail.sum()),
                                       vehicle_steps=int(r["steps"].sum()), steps=n, alive=crude.alive(),
                                       seconds=time.perf_counter() - t0))
            del crude
            print(f"noise x{scale:g}: crude on 65,536 drives p = {p:.3e} +- {out[key]['crude']['se']:.1e} "
                  f"({int(fail.sum())} failures, {out[key]['crude']['vehicle_steps']:.3e} vehicle-steps)", flush=True)
        ps, vs, t0 = [], 0, time.perf_counter()
        for rep in range(REPS):
            sim = M.BatchedSimulation(T, scen, x_init=xi, noise=noise(scale, 100 + rep))
            res = offroad_probability(sim, lam, EVERY, seed=rep, max_steps=MAX_DRIVE)
            ps.append(res["p"])
            vs += res["vehicle_steps"]
            del sim
        m, se = float(np.mean(ps)), float(np.std(ps, ddof=1) / np.sqrt(REPS))
        out[key][f"lam{lam:g}"] = dict(p=ps, mean=m, se=se, vehicle_steps=vs, seconds=time.perf_counter() - t0)
        print(f"noise x{scale:g}: splitting lam {lam:g} every {EVERY}, {REPS} x 4,096 vehicles, p = {m:.3e} +- {se:.1e} "
              f"({vs:.3e} vehicle-steps): {['%.2e' % q for q in ps]}", flush=True)
    return out


def save():
    if args.get("out"):
        os.makedirs(os.path.dirname(os.path.abspath(args["out"])), exist_ok=True)
        with open(args["out"], "w") as f:
            json.dump(res, f, indent=1)


if args.get("mode") == "kernels":
    worker_kernels(args["root"], int(args["B"]))
    sys.exit(0)

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print("card:", card, "| base noise", BASE, flush=True)
PARENT = os.path.abspath(args.get("parent", os.path.join(ROOT, "build", "parent")))
trees = {"parent": PARENT, "new": ROOT}
res = dict(card=card, base=BASE, kernels={}, bench={})
for B in (4096, 65536):
    got = {k: [] for k in trees}
    for _ in range(ROUNDS):
        for name, root in trees.items():
            got[name].append(sub([sys.executable, os.path.abspath(__file__), "mode=kernels", f"root={root}", f"B={B}"], ROOT))
    for name in trees:
        fp = [g["fsm"] + g["plant"] for g in got[name]]
        print(f"fleet {B:6d} {name:6s}: fsm + plant {', '.join('%.2f' % f for f in fp)} us per step "
              f"(of {got[name][-1]['all']:.1f} us of kernels)", flush=True)
    d = statistics.mean(g["fsm"] + g["plant"] for g in got["new"]) - statistics.mean(
        g["fsm"] + g["plant"] for g in got["parent"])
    print(f"fleet {B:6d}: running verdicts add {d:.2f} us per step to the fsm and plant kernels", flush=True)
    res["kernels"][B] = dict(runs=got, extra_us=d)
np, M, T, fleet = setup(ROOT)
res["branch_ms"] = branch_costs(np, M, T, fleet)
save()
res["estimates"] = estimates(np, M, T, fleet)
save()
for _ in range(ROUNDS):
    for name, root in trees.items():
        line = sub([sys.executable, "bench.py", "--gpus", "1", "--steps", "20", "--warmup", "5"], root)
        res["bench"].setdefault(name, []).append(line)
        fl = line.get("closed_loop_fleet", {})
        print(f"bench {name:6s}: {line.get('metric')} {line.get('value'):.4g} {line.get('unit')}; closed_loop_fleet "
              f"{json.dumps(fl)[:300]}", flush=True)
save()
