"""Step-by-step replay of device closed loops (mpcb_sim_*) against the oracle, vehicle by vehicle.

A device loop step is three kernels: the obstacle FSM, the solve over the list of vehicles still driving, the plant
step.  The recorded history (BatchedSimulation.history: the state before each step, the applied U*[0], the status, the
car position, the light colour) lets every step of every vehicle be replayed on its own:

  1. the FSM kernel against oracle.tracker_port.ObstacleFSMPort driven with the vehicle's own scenario constants and its
     recorded (s, v): car positions bit for bit, light colours, and the frozen rows after arrival;
  2. the plant kernel against x + DT * dynamics(x, u, k_ref(s)) (trajectory_tracking.py:404-406) to 1e-12, step counts
     and unsolved counts;
  3. (cold loops) every in-loop solve against the plain solve of the same problem -- recorded state, obstacles from the
     oracle FSM -- in a batch of the loop's size, so that it takes the loop's execution shape: bitwise;
  4. (hot-started loops) every in-loop solve against the cold plain solve of the same problem: same flags and the same
     control to the tolerance used between execution shapes.

Four staggered fleets on trajectory2, each vehicle with its own start and scenario constants, car and light switched on
and off independently: 3,500 vehicles (more than coop_max_batch = 3,072: thread-per-problem first pass, class kernels
fed from the list of vehicles still driving) and 600 vehicles (warp-per-problem first pass), each cold and hot-started.
The replay helpers (closed_loop_oracle) are checked without a GPU against the reference's own closed-loop logs (tests/golden/closed_loop_*),
so that a failure on the GPU cannot come from the replay itself."""
import numpy as np
import pytest

from closed_loop_oracle import fsm_replay, k_ref, plant_step
from conftest import golden
from oracle import tracker_port as P

# name: (vehicles, hot start, seed of the fleet)
FLEETS = {"bulk_cold": (3500, False, 31), "bulk_hot": (3500, True, 31),
          "small_cold": (600, False, 32), "small_hot": (600, True, 32)}
MAX_STEPS = 1200      # the longest drive of these fleets is well below; 1,200 x 3,500 recorded steps are ~300 MB
CHUNK = 100           # steps enqueued between looks at the fleet


# --------------------------------------------------------------------------------------------------------------------
# 5. the helpers against the reference's own closed-loop logs (no GPU)
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("i", [2, 3])
def test_fsm_replay_reproduces_reference_logs(i):
    """fsm_replay driven by the reference's state history gives its obstacle sets, car positions and colours exactly."""
    z = golden(f"closed_loop_traj{i}")
    cfg = {2: P.FSM_TRAJ2, 3: P.FSM_TRAJ3}[i]
    k = len(z["hist_u"])
    obs_sv, n_obs, car, green = fsm_replay(P.ObstacleFSMPort(True, True, **cfg), z["hist_x"][:k, 0], z["hist_x"][:k, 4])
    assert np.array_equal(n_obs, z["n_obs"])
    assert np.array_equal(obs_sv, z["obs_sv"])
    assert np.array_equal(car, z["hist_obs_s"], equal_nan=True)
    assert np.array_equal(green, z["hist_tl"] == "GREEN")
    assert (n_obs > 0).any() and (n_obs == 0).any()


@pytest.mark.parametrize("i", [1, 2, 3])
def test_plant_replay_reproduces_reference_logs(i, port_tables):
    """plant_step reproduces the reference's next state bit for bit, and its k_ref is RefTable.get_state's, also past
    the end of the table."""
    tab = port_tables[i]
    z = golden(f"closed_loop_traj{i}")
    hx, hu = z["hist_x"], z["hist_u"]
    assert np.array_equal(plant_step(tab, hx[:-1], hu), hx[1:])
    s = np.concatenate([np.linspace(-3.0, tab.s_max + 3.0, 4001), tab.s, [tab.s_max, np.nextafter(tab.s_max, np.inf)],
                        hx[:, 0]])
    assert np.array_equal(k_ref(tab, s), [tab.get_state(q)[3] for q in s])


# --------------------------------------------------------------------------------------------------------------------
# fleets on the GPU
# --------------------------------------------------------------------------------------------------------------------
def _fleet_constants(s_max, B, seed):
    """Per-vehicle start and scenario constants; car and light on or off independently, all four combinations."""
    rng = np.random.default_rng(seed)
    s0 = rng.uniform(0.0, s_max - 150.0, B)
    trig = s0 + rng.uniform(0.0, 60.0, B)
    start = trig + rng.uniform(20.0, 120.0, B)
    consts = dict(obs_trigger_s=trig, obs_start_s=start, obs_v=rng.uniform(4.0, 8.0, B),
                  obs_end_s=start + rng.uniform(60.0, 250.0, B), tl_pos=s0 + rng.uniform(40.0, 400.0, B),
                  tl_trigger_s=rng.uniform(60.0, 120.0, B), tl_stop_duration=rng.uniform(2.0, 8.0, B))
    combo = rng.permutation(np.arange(B) % 4)
    return s0, [{k: float(a[b]) for k, a in consts.items()} for b in range(B)], combo & 1, combo >> 1


@pytest.fixture(scope="module")
def fleet(request, gpu_trackers, port_tables):
    """Runs one fleet to the end with every step recorded and replays its FSM with the oracle for every vehicle."""
    import safe_autonomous_driving_mpc_b200 as M
    name = request.param
    B, hot, seed = FLEETS[name]
    L, T = gpu_trackers[2]
    assert (B > T.params.coop_max_batch) == name.startswith("bulk"), "each fleet size must keep its execution shape"
    s0, consts, dyn, tl = _fleet_constants(L.s_max, B, seed)
    x_init = np.array([L.get_state(s) for s in s0])
    x_init[:, 4] = np.maximum(x_init[:, 4], 0.5)
    scen = [M.make_scenario(2, dynamic_obstacle=int(dyn[b]), traffic_light=int(tl[b]), **consts[b]) for b in range(B)]
    sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=MAX_STEPS, hot_start=hot)
    n_run = 0
    while n_run < MAX_STEPS:
        sim.step(CHUNK)
        n_run += CHUNK
        assert T.last_call_used_coop() == (B <= T.params.coop_max_batch), "execution shape of the loop's solve"
        if sim.alive() == 0:
            break
    x_final, steps, n_unsolved = sim.state()
    h = sim.history()
    del sim
    assert h["x"].shape[0] == n_run
    # oracle FSM of every vehicle over the steps it drove
    obs_sv = np.zeros((n_run, B, 2, 2))
    n_obs = np.zeros((n_run, B), np.int32)
    car = np.full((n_run, B), np.nan)
    green = np.zeros((n_run, B), np.int32)
    for b in range(B):
        k = int(steps[b])
        fsm = P.ObstacleFSMPort(bool(dyn[b]), bool(tl[b]), **consts[b])
        obs_sv[:k, b], n_obs[:k, b], car[:k, b], green[:k, b] = fsm_replay(fsm, h["x"][:k, b, 0], h["x"][:k, b, 4])
    return dict(name=name, B=B, hot=hot, T=T, L=L, tab=port_tables[2], dyn=dyn, tl=tl, n_run=n_run, hist=h,
                x_final=x_final, steps=steps, n_unsolved=n_unsolved, obs_sv=obs_sv, n_obs=n_obs, car=car, green=green)


def _replay_solves(F):
    """Plain solves of every recorded problem, step by step: the vehicles still driving at step t with their recorded
    states and the oracle FSM's obstacles, tiled to the fleet's size so that the call takes the loop's execution shape.
    Yields (t, live vehicles, U[:, 0] and status of the whole tiled batch)."""
    h, B, T = F["hist"], F["B"], F["T"]
    for t in range(F["n_run"]):
        live = np.flatnonzero(F["steps"] > t)
        if live.size == 0:
            break
        rep = np.resize(live, B)
        r = T.solve_batch_host(h["x"][t, rep], F["obs_sv"][t, rep], F["n_obs"][t, rep])
        assert T.last_call_used_coop() == (B <= T.params.coop_max_batch)
        yield t, live, r["U"][:, 0].copy(), r["status"].copy()


@pytest.mark.gpu
@pytest.mark.parametrize("fleet", list(FLEETS), indirect=True)
def test_fsm_kernel_matches_oracle(fleet):
    """1. Car position bit for bit (NaN exactly where there is no car) and light colour of every vehicle at every step
    against the oracle FSM with the vehicle's own constants; after arrival the rows are frozen: tl = status = -1, x, u
    and the car NaN."""
    F = fleet
    h, steps, n = F["hist"], F["steps"], F["n_run"]
    live = np.arange(n)[:, None] < steps[None, :]
    assert steps.min() >= 1
    bad = ~((h["obs_s"] == F["car"]) | (np.isnan(h["obs_s"]) & np.isnan(F["car"])))
    bad |= live & (h["tl"] != F["green"])
    t_bad, b_bad = np.nonzero(bad)
    assert t_bad.size == 0, ("FSM differs from the oracle at (step, vehicle)", list(zip(t_bad[:10], b_bad[:10])),
                             h["obs_s"][t_bad[:5], b_bad[:5]], F["car"][t_bad[:5], b_bad[:5]])
    dead = ~live
    assert np.all(h["tl"][dead] == -1) and np.all(h["status"][dead] == -1)
    assert np.all(np.isnan(h["x"][dead])) and np.all(np.isnan(h["u"][dead])) and np.all(np.isnan(h["obs_s"][dead]))
    assert np.all(np.isin(h["status"][live], (0, 1, 2)))
    # the fleet exercises what it is meant to: every combination of car and light, cars present, lights turning green
    assert set(zip(F["dyn"].tolist(), F["tl"].tolist())) == {(0, 0), (0, 1), (1, 0), (1, 1)}
    had_car = (~np.isnan(F["car"])).any(axis=0)
    had_green = (F["green"] == 1).any(axis=0)
    assert had_car[F["dyn"] == 1].mean() > 0.25 and not had_car[F["dyn"] == 0].any()
    assert had_green[F["tl"] == 1].mean() > 0.25 and not had_green[F["tl"] == 0].any()
    assert (F["n_obs"] == 2).any()


@pytest.mark.gpu
@pytest.mark.parametrize("fleet", list(FLEETS), indirect=True)
def test_plant_kernel_matches_oracle(fleet):
    """2. Every recorded step of every vehicle: hist_x[t+1] (the final state after the last step) is the oracle's plant
    step of (hist_x[t], hist_u[t]) to 1e-12 relative -- the device interpolates the table with FMA, nothing else differs;
    steps[b] is the first step that crosses s_max - 1; n_unsolved[b] counts the recorded non-zero statuses."""
    F = fleet
    h, steps, n, B = F["hist"], F["steps"], F["n_run"], F["B"]
    s_stop = F["L"].s_max - 1.0
    assert F["tab"].s_max == F["L"].s_max
    target = np.concatenate([h["x"][1:], np.full((1, B, 5), np.nan)])
    target[steps - 1, np.arange(B)] = F["x_final"]
    worst = 0.0
    for a in range(0, n, CHUNK):
        sl = slice(a, min(a + CHUNK, n))
        live = np.arange(sl.start, sl.stop)[:, None] < steps[None, :]
        got = plant_step(F["tab"], h["x"][sl], h["u"][sl])[live]
        want = target[sl][live]
        assert np.all(np.isfinite(want))
        err = np.abs(got - want) / np.maximum(1.0, np.abs(want))
        if err.size:
            worst = max(worst, float(err.max()))
    assert worst <= 1e-12, worst
    # step counts: every recorded state was still driving, the state after the last step has arrived (or the run ended)
    live = np.arange(n)[:, None] < steps[None, :]
    assert np.all(h["x"][:, :, 0][live] <= s_stop)
    arrived = F["x_final"][:, 0] > s_stop
    assert np.all(arrived | (steps == n)) and np.all(steps <= n)
    # a vehicle whose random stop line fell where the reference trajectory leaves the lane margin may stay at the
    # formulation's standstill fixed point (test_gpu_sim.py::test_stop_line_inside_the_tight_bend_is_a_fixed_point)
    assert (~arrived).sum() <= B // 200, (~arrived).sum()
    assert np.array_equal(F["n_unsolved"], ((h["status"] != 0) & live).sum(axis=0))


@pytest.mark.gpu
@pytest.mark.parametrize("fleet", list(FLEETS), indirect=True)
def test_in_loop_solves_against_plain_solves(fleet):
    """3. Cold fleets: every in-loop solve is bitwise the plain solve of the same problem in a batch of the same size --
    the execution shape is decided by the size of the whole batch, and a problem's answer does not depend on its batch,
    its part of the batch or its slot in the list of vehicles still driving.  Tiled copies agree with each other.

    4. Hot-started fleets (first pass from the previous plan advanced by one step, rows on their bounds active): against
    the cold plain solve of the same recorded problem, flags agree on >= 99.9 % of the vehicle-steps (borderline flags
    may flip between solver paths, as between execution shapes), and where both are SOLVED, U*[0] agrees to 1e-6 (the
    tolerance between execution shapes) on all but at most 0.1 % -- the allowance the parity tests make for problems
    with two local optima.  Those tests re-check each such point with the oracle's SLSQP; that needs the whole plan,
    which the closed loop does not expose (only U*[0] is recorded), so here the exceptions are counted and listed."""
    F = fleet
    h = F["hist"]
    n_steps = n_agree = n_both = 0
    diff, far = [], []
    for t, live, u0, st in _replay_solves(F):
        m = live.size
        rec_u, rec_s = h["u"][t, live], h["status"][t, live]
        if not F["hot"]:
            for j in np.flatnonzero(np.any(rec_u != u0[:m], axis=1) | (rec_s != st[:m]))[:3]:
                diff.append((t, int(live[j]), rec_u[j].tolist(), u0[j].tolist(), int(rec_s[j]), int(st[j])))
            ref = np.arange(F["B"]) % m
            assert np.array_equal(u0, u0[ref]) and np.array_equal(st, st[ref]), f"step {t}: tiled copies disagree"
        agree = rec_s == st[:m]
        both = agree & (st[:m] == 0)
        du = np.abs(rec_u - u0[:m]).max(axis=1)
        far += [(t, int(live[j]), float(du[j])) for j in np.flatnonzero(both & (du > 1e-6))]
        n_steps += m
        n_agree += int(agree.sum())
        n_both += int(both.sum())
    big = sorted(far, key=lambda e: -e[2])
    print(f"\n{F['name']}: {n_steps} vehicle-steps, flags differ on {n_steps - n_agree}, |du0| > 1e-6 on {len(far)} "
          f"of {n_both} solved by both (> 1e-5: {sum(e[2] > 1e-5 for e in far)}, > 1e-4: "
          f"{sum(e[2] > 1e-4 for e in far)}; largest {big[:3]})")
    assert n_steps == int(F["steps"].sum())
    if not F["hot"]:
        assert not diff, f"in-loop solves that differ from the plain solve (step, vehicle, loop u0, plain u0, loop " \
                         f"status, plain status), up to 3 per step: {diff[:8]}"
        return
    assert n_agree >= 0.999 * n_steps, (n_steps - n_agree, n_steps)
    assert len(far) <= max(1, n_both // 1000), f"{len(far)} of {n_both} (step, vehicle, |du0|): {far[:20]}"
