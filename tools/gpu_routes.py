"""Several routes on one handle against one handle per route (DESIGN.md 4, "Several routes on one handle").

  solve  65,536 Monte-Carlo problems mixed over trajectories 1-3: one call on a routed handle, against the same problems
         as three single-route calls on one stream, and as three handles on three streams.  Device time per call (CUDA
         events), and the first- and robust-pass times of each call.
  fleet  3 x 4,096 vehicles (trajectories 1-3, staggered starts, per-vehicle scenarios, FLEET_SOLVER_CAPS): one routed
         simulation, three simulations stepped in turn on one stream, three simulations on three streams; vehicle-steps/s.

    python tools/gpu_routes.py [out.json]"""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import safe_autonomous_driving_mpc_b200 as M
from oracle import tracker_port as P

assert torch.cuda.is_available(), "needs a GPU"
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()[0]
dev = torch.device("cuda:0")
Ls = [M.TrajectoryLoader(f"{ROOT}/data/trajectory{i}.npz") for i in (1, 2, 3)]
tabs = [P.RefTable.from_npz(f"{ROOT}/data/trajectory{i}.npz") for i in (1, 2, 3)]
res = {"gpu": gpu}


def ev():
    return torch.cuda.Event(enable_timing=True)


# ---- solve -----------------------------------------------------------------------------------------------------------
B = 65536
route = np.random.default_rng(5).integers(0, 3, B).astype(np.int32)
rows = np.arange(B)
sets = [P.monte_carlo_problems(t, B) for t in tabs]
mixed = [np.ascontiguousarray(np.stack([s[k] for s in sets])[route, rows]) for k in range(3)]
d_mixed = [torch.from_numpy(a).to(dev) for a in mixed] + [torch.from_numpy(route).to(dev)]
d_parts = [[torch.from_numpy(np.ascontiguousarray(a[route == r])).to(dev) for a in mixed] for r in range(3)]
TR = M.BatchedTracker(Ls)
TS = [M.BatchedTracker(L) for L in Ls]
streams = [torch.cuda.Stream() for _ in range(3)]
main = torch.cuda.current_stream()
out_r = TR.solve_batch(*d_mixed[:3], route=d_mixed[3])
out_s = [TS[r].solve_batch(*d_parts[r]) for r in range(3)]
torch.cuda.synchronize()
reps = 30
arms = {"routed": [], "three_calls_one_stream": [], "three_handles_three_streams": []}
for it in range(reps + 3):
    e0, e1 = ev(), ev()
    e0.record(); TR.solve_batch(*d_mixed[:3], route=d_mixed[3], out=out_r); e1.record(); torch.cuda.synchronize()
    f, s, n2 = TR.last_pass_ms()
    arms["routed"].append((e0.elapsed_time(e1), f, s, n2))
    e0, e1 = ev(), ev()
    passes = []
    e0.record()
    for r in range(3):
        TS[r].solve_batch(*d_parts[r], out=out_s[r])
    e1.record(); torch.cuda.synchronize()
    for r in range(3):
        passes.append(TS[r].last_pass_ms())
    arms["three_calls_one_stream"].append((e0.elapsed_time(e1), sum(p[0] for p in passes), sum(p[1] for p in passes),
                                           sum(p[2] for p in passes)))
    e0, e1 = ev(), ev()
    e0.record()
    for r in range(3):
        streams[r].wait_stream(main)
        TS[r].solve_batch(*d_parts[r], out=out_s[r], stream=streams[r].cuda_stream)
    for r in range(3):
        main.wait_stream(streams[r])
    e1.record(); torch.cuda.synchronize()
    arms["three_handles_three_streams"].append((e0.elapsed_time(e1), float("nan"), float("nan"), 0))
solve = {}
for k, v in arms.items():
    a = np.array(v[3:], dtype=np.float64)
    solve[k] = {"call_ms_median": float(np.median(a[:, 0])), "call_ms_min": float(a[:, 0].min()),
                "first_pass_ms_median": float(np.median(a[:, 1])), "robust_pass_ms_median": float(np.median(a[:, 2])),
                "robust_pass_problems": int(a[-1, 3])}
    print(k, json.dumps(solve[k]), flush=True)
res["solve_65536_three_routes"] = solve

# ---- fleet -----------------------------------------------------------------------------------------------------------
per = 4096
rng = np.random.default_rng(21)
fleet = []
for r, L in enumerate(Ls):
    s0 = rng.uniform(0.0, max(L.s_max - 150.0, 1.0), per)
    xi = np.array([L.get_state(s) for s in s0])
    xi[:, 4] = np.clip(xi[:, 4], 0.5, None)
    if r == 0:
        sc = [M.make_scenario(2, dynamic_obstacle=0, traffic_light=0) for _ in s0]
    else:
        sc = [M.make_scenario(2, tl_pos=float(s + rng.uniform(120, 300)), obs_trigger_s=float(s + 5),
                              obs_start_s=float(s + 50), obs_end_s=float(s + 250), tl_stop_duration=4.0) for s in s0]
    fleet.append((xi, sc))
n_warm, n_steps = 20, 300
TRf = M.BatchedTracker(Ls, **M.FLEET_SOLVER_CAPS)
TSf = [M.BatchedTracker(L, **M.FLEET_SOLVER_CAPS) for L in Ls]


def driven(sims):
    return sum(int(s.state()[1].sum()) for s in sims)


def run_fleet(kind):
    if kind == "routed":
        sims = [M.BatchedSimulation(TRf, sum((f[1] for f in fleet), []), x_init=np.vstack([f[0] for f in fleet]),
                                    route=np.repeat(np.arange(3), per))]
    else:
        sims = [M.BatchedSimulation(TSf[r], fleet[r][1], x_init=fleet[r][0]) for r in range(3)]
    st = [streams[r].cuda_stream for r in range(3)] if kind == "three_streams" else [main.cuda_stream] * 3

    def step(n):
        for k in range(0, n, 10):
            for i, s in enumerate(sims):
                s.step(min(10, n - k), stream=st[i])

    step(n_warm)
    torch.cuda.synchronize()
    v0 = driven(sims)
    t0 = time.perf_counter()
    step(n_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    v = driven(sims) - v0
    return {"vehicle_steps": v, "seconds": dt, "vehicle_steps_per_s": v / dt}


fl = {}
for rep in range(2):
    for kind in ("routed", "three_sims_one_stream", "three_streams"):
        r = run_fleet(kind)
        fl.setdefault(kind, []).append(r)
        print(kind, json.dumps(r), flush=True)
res["fleet_3x4096"] = {k: {"vehicle_steps_per_s": [r["vehicle_steps_per_s"] for r in v], "vehicle_steps": v[-1]["vehicle_steps"]}
                       for k, v in fl.items()}
res["fleet_3x4096"]["steps_timed"] = n_steps
print(json.dumps(res))
if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        json.dump(res, f, indent=1)
