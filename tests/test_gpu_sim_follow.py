"""Following in the device closed loop (mpcb_sim_set_follow): the nearest vehicle ahead on the same route is a moving
obstacle.

  1. leader replay: from the recorded states, a numpy reference of the leader rule (per route, order (s, index), next
     vehicle within follow_range, arrived vehicles excluded) gives the recorded leaders and their (s, v) bit for bit;
  2. obstacle sets and in-loop solves: the oracle FSM plus the merge rule (nearer of scripted car and leader in the car
     slot, tie to the scripted car, light after it) fed to plain routed solves of the loop's batch size gives every cold
     in-loop U*[0] and status bit for bit; the plant step matches to 1e-12;
  3. a platoon driven by a host loop (solve_batch_host + the numpy leader rule + the numpy plant step) against the device
     loop; without following the vehicles drive through each other, with it every follower keeps a gap of at least
     1 m, also through the steps its solver leaves unsolved while the platoon queues at the light;
  4. following off (never switched on, or switched on and off before the first step) is today's loop bit for bit, with
     the same launch count; switched on halfway, the loop is the off loop up to that step;
  5. argument checks.
The leader and merge rules (closed_loop_oracle) are checked without a GPU on hand-made cases."""
import ctypes as C

import numpy as np
import pytest

from closed_loop_oracle import fsm_replay, leaders, merge, plant_step
from conftest import traj_path
from oracle import tracker_port as P


# --------------------------------------------------------------------------------------------------------------------
# the helpers on hand-made cases (no GPU)
# --------------------------------------------------------------------------------------------------------------------
def test_leader_rule_on_hand_made_cases():
    """Order by (s, index), ties to the higher index, the range filter, routes apart, arrived vehicles nobody's
    leader and without one."""
    s = np.array([10.0, 10.0, 12.0, 40.0, 11.0, 5.0, 13.0, 10.0])
    x = np.zeros((8, 5))
    x[:, 0] = s
    x[:, 4] = np.arange(8) + 0.5
    route = np.array([0, 0, 0, 0, 1, 1, 0, 0])
    live = np.array([True, True, True, True, True, True, False, True])
    lead, sv = leaders(x, live, route, 20.0)
    # route 0, live, by (s, b): 0 (10), 1 (10), 7 (10), 2 (12), 3 (40); vehicle 6 (13) has arrived
    assert lead.tolist() == [1, 7, -1, -1, -1, 4, -1, 2]
    assert np.array_equal(sv[0], [10.0, 1.5]) and np.array_equal(sv[5], [11.0, 4.5]) and np.isnan(sv[2]).all()
    lead, _ = leaders(x, live, route, 28.0)
    assert lead[2] == 3                                   # 40 - 12 = 28 <= range
    lead, _ = leaders(x, live, route, np.nextafter(28.0, 0.0))
    assert lead[2] == -1


def test_merge_rule_on_hand_made_cases():
    """Nearer wins, the scripted car on a tie, the light behind the car slot, nothing changes without a leader."""
    L = (300.0, 0.0)
    # (FSM obstacles, n, car) x leader -> expected
    cases = [
        ([(100.0, 4.0), L], 2, 100.0, (90.0, 7.0), [(90.0, 7.0), L], 2),     # leader nearer
        ([(100.0, 4.0), L], 2, 100.0, (110.0, 7.0), [(100.0, 4.0), L], 2),   # car nearer
        ([(100.0, 4.0), L], 2, 100.0, (100.0, 7.0), [(100.0, 4.0), L], 2),   # tie: the scripted car
        ([L, (0.0, 0.0)], 1, np.nan, (50.0, 3.0), [(50.0, 3.0), L], 2),       # light only: leader in front of it
        ([(0.0, 0.0), (0.0, 0.0)], 0, np.nan, (50.0, 3.0), [(50.0, 3.0), (0.0, 0.0)], 1),
        ([(100.0, 4.0), (0.0, 0.0)], 1, 100.0, (np.nan, np.nan), [(100.0, 4.0), (0.0, 0.0)], 1),
        ([L, (0.0, 0.0)], 1, np.nan, (np.nan, np.nan), [L, (0.0, 0.0)], 1),
    ]
    for obs, n, car, ld, want, n_want in cases:
        o, m = merge(np.array(obs), np.array(n), np.array(car), np.array(ld))
        assert np.array_equal(o, want) and m == n_want, (obs, ld, o, m)
    # vectorised over leading axes the same as case by case
    obs = np.array([c[0] for c in cases])
    o, m = merge(obs, np.array([c[1] for c in cases]), np.array([c[2] for c in cases]), np.array([c[3] for c in cases]))
    assert np.array_equal(o, np.array([c[4] for c in cases])) and m.tolist() == [c[5] for c in cases]


# --------------------------------------------------------------------------------------------------------------------
# routed fleets on the GPU
# --------------------------------------------------------------------------------------------------------------------
RANGE = 10.0
N_STEPS = 300
# name: (vehicles, hot start); 3,500 > coop_max_batch: thread-per-problem first pass; 600: warp-per-problem
FLEETS = {"bulk_cold": (3500, False), "small_cold": (600, False), "small_hot": (600, True)}
EQUAL_PAIRS = [(10, 12), (21, 23), (40, 42), (51, 53), (100, 102)]   # same route (same parity), same start


@pytest.fixture(scope="module")
def routed():
    import safe_autonomous_driving_mpc_b200 as M
    Ls = [M.TrajectoryLoader(traj_path(i)) for i in (2, 3)]
    return Ls, [P.RefTable.from_npz(traj_path(i)) for i in (2, 3)]


def _fleet_setup(Ls, B, seed):
    import safe_autonomous_driving_mpc_b200 as M
    rng = np.random.default_rng(seed)
    route = (np.arange(B) % 2).astype(np.int32)
    s_max = np.array([L.s_max for L in Ls])[route]
    s0 = rng.uniform(0.0, s_max - 150.0)
    for a, b in EQUAL_PAIRS:
        s0[b] = s0[a]
    x_init = np.array([Ls[route[b]].get_state(s0[b]) for b in range(B)])
    x_init[:, 4] = np.maximum(x_init[:, 4], 0.5)
    trig = s0 + rng.uniform(0.0, 60.0, B)
    start = trig + rng.uniform(20.0, 120.0, B)
    consts = dict(obs_trigger_s=trig, obs_start_s=start, obs_v=rng.uniform(4.0, 8.0, B),
                  obs_end_s=start + rng.uniform(60.0, 250.0, B), tl_pos=s0 + rng.uniform(40.0, 400.0, B),
                  tl_trigger_s=rng.uniform(60.0, 120.0, B), tl_stop_duration=rng.uniform(2.0, 8.0, B))
    combo = rng.permutation(np.arange(B) % 4)
    dyn, tl = combo & 1, combo >> 1
    consts = [{k: float(a[b]) for k, a in consts.items()} for b in range(B)]
    scen = [M.make_scenario(2, dynamic_obstacle=int(dyn[b]), traffic_light=int(tl[b]), **consts[b]) for b in range(B)]
    return route, x_init, scen, consts, dyn, tl


@pytest.fixture(scope="module")
def fleet(request, routed):
    """One routed fleet driven N_STEPS steps with following on and every step recorded."""
    import safe_autonomous_driving_mpc_b200 as M
    name = request.param
    B, hot = FLEETS[name]
    Ls, tabs = routed
    T = M.BatchedTracker(Ls)
    assert (B > T.params.coop_max_batch) == name.startswith("bulk")
    route, x_init, scen, consts, dyn, tl = _fleet_setup(Ls, B, 41)
    sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=N_STEPS, hot_start=hot, route=route,
                              follow_range=RANGE)
    sim.step(N_STEPS)
    assert T.last_call_used_coop() == (B <= T.params.coop_max_batch)
    x_final, steps, n_unsolved = sim.state()
    F = dict(name=name, B=B, hot=hot, T=T, tabs=tabs, route=route, consts=consts, dyn=dyn, tl=tl, hist=sim.history(),
             lead=sim.follow_history(), x_final=x_final, steps=steps, n_unsolved=n_unsolved, check=sim.follow_check())
    del sim
    return F


@pytest.mark.gpu
@pytest.mark.parametrize("fleet", list(FLEETS), indirect=True)
def test_recorded_leaders_match_the_numpy_rule(fleet):
    """1. At every step, the numpy leader rule on the recorded states gives hist_lead_idx and hist_lead_sv bit for bit;
    the fleet exercises what it should: equal starts, leaders out of range, arrivals, both routes."""
    F = fleet
    h, ld, B = F["hist"], F["lead"], F["B"]
    assert ld["lead"].shape == (N_STEPS, B)
    n_lead = n_arrived = n_out = 0
    for t in range(N_STEPS):
        x = h["x"][t]
        live = F["steps"] > t
        assert np.array_equal(live, ~np.isnan(x[:, 0]))
        lead, sv = leaders(np.where(live[:, None], x, 0.0), live, F["route"], RANGE)
        assert np.array_equal(ld["lead"][t], lead), (t, np.flatnonzero(ld["lead"][t] != lead)[:8])
        assert np.array_equal(ld["lead_s"][t], sv[:, 0], equal_nan=True), t
        assert np.array_equal(ld["lead_v"][t], sv[:, 1], equal_nan=True), t
        n_lead += int((lead >= 0).sum())
        n_out += int(((leaders(np.where(live[:, None], x, 0.0), live, F["route"], np.inf)[0] >= 0) & (lead < 0)).sum())
        n_arrived += int((~live).sum())
    assert n_lead > 0 and n_arrived > 0
    a, b = EQUAL_PAIRS[0]
    assert ld["lead"][0, a] == b and ld["lead_s"][0, a] == h["x"][0, a, 0]
    assert n_out > 0                                      # next vehicle of the route beyond the range
    assert set(F["route"][ld["lead"][0] >= 0].tolist()) == {0, 1}
    # the follow check on the recorded leaders
    gap = np.where(ld["lead"] >= 0, ld["lead_s"] - h["x"][..., 0], np.inf).min(axis=0)
    want = np.where(np.isinf(gap), 1e30, gap)
    assert np.array_equal(F["check"]["min_gap"], want) and np.array_equal(F["check"]["ok"], ~(want < 1.0))


@pytest.mark.gpu
@pytest.mark.parametrize("fleet", ["bulk_cold", "small_cold"], indirect=True)
def test_in_loop_solves_see_the_merged_obstacles(fleet):
    """2. The oracle FSM of every vehicle plus the merge rule on the recorded leaders, fed to plain routed solves of
    the loop's batch size, gives every in-loop U*[0] and status bit for bit; the scripted car's recorded position is the
    oracle's; the plant step matches to 1e-12."""
    import torch
    F = fleet
    h, B, T, route = F["hist"], F["B"], F["T"], F["route"]
    ld = F["lead"]
    obs_sv = np.zeros((N_STEPS, B, 2, 2))
    n_obs = np.zeros((N_STEPS, B), np.int32)
    car = np.full((N_STEPS, B), np.nan)
    for b in range(B):
        k = int(min(F["steps"][b], N_STEPS))
        fsm = P.ObstacleFSMPort(bool(F["dyn"][b]), bool(F["tl"][b]), **F["consts"][b])
        obs_sv[:k, b], n_obs[:k, b], car[:k, b], _green = fsm_replay(fsm, h["x"][:k, b, 0], h["x"][:k, b, 4])
    assert np.array_equal(h["obs_s"], car, equal_nan=True)
    lead_sv = np.stack([ld["lead_s"], ld["lead_v"]], axis=-1)
    obs_m, n_m = merge(obs_sv, n_obs, car, lead_sv)
    took = ~np.isnan(ld["lead_s"]) & ~(car <= ld["lead_s"])
    assert took.any()
    dev = torch.device("cuda", 0)
    diff = []
    for t in range(N_STEPS):
        live = np.flatnonzero(F["steps"] > t)
        if live.size == 0:
            break
        rep = np.resize(live, B)
        args = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (h["x"][t, rep], obs_m[t, rep], n_m[t, rep],
                                                                              route[rep])]
        r = T.solve_batch(*args[:3], route=args[3])
        torch.cuda.synchronize()
        assert T.last_call_used_coop() == (B <= T.params.coop_max_batch)
        u0 = r["U"][:, 0].cpu().numpy()[: live.size]
        st = r["status"].cpu().numpy()[: live.size]
        bad = np.any(h["u"][t, live] != u0, axis=1) | (h["status"][t, live] != st)
        diff += [(t, int(live[j])) for j in np.flatnonzero(bad)[:3]]
    assert not diff, diff[:10]
    assert (n_m == 2).any() and (h["status"] == 2).any() and (h["status"] == 0).any()
    # plant step, each vehicle on its route's table
    steps, worst = F["steps"], 0.0
    target = np.concatenate([h["x"][1:], np.full((1, B, 5), np.nan)])
    fin = steps <= N_STEPS
    target[steps[fin] - 1, np.flatnonzero(fin)] = F["x_final"][fin]
    for r in (0, 1):
        sel = route == r
        live = np.arange(N_STEPS)[:, None] < steps[None, sel]
        got = plant_step(F["tabs"][r], h["x"][:, sel], h["u"][:, sel])[live]
        want = target[:, sel][live]
        ok = np.isfinite(want).all(axis=1)                   # the state after the last recorded step is x_final
        worst = max(worst, float((np.abs(got[ok] - want[ok]) / np.maximum(1.0, np.abs(want[ok]))).max()))
    assert worst <= 1e-12, worst


# --------------------------------------------------------------------------------------------------------------------
# a platoon: host loop against device loop
# --------------------------------------------------------------------------------------------------------------------
def _platoon(L):
    import safe_autonomous_driving_mpc_b200 as M
    B = 8
    s0 = 300.0 - 15.0 * np.arange(B)                     # vehicle 0 in front, 15 m apart
    x_init = np.array([L.get_state(s) for s in s0])
    x_init[:, 4] = 4.0 + 0.5 * np.arange(B)              # the rear ones faster
    consts = [dict(traffic_light=int(b == 0), dynamic_obstacle=0) for b in range(B)]
    scen = [M.make_scenario(2, **c) for c in consts]
    return B, x_init, scen, consts


@pytest.mark.gpu
def test_platoon_host_loop_equals_device_loop(gpu_trackers, port_tables):
    """3. Eight vehicles on trajectory2, the front one stopping at the light: a host loop (solve_batch_host, numpy leader
    rule, oracle FSM, numpy plant step) and the device loop with following take the same steps and the same leaders,
    statuses equal, states to 1e-7 (the device interpolates the plant step's curvature with FMA, numpy does not).
    Without following the vehicles drive through each other; with it every follower keeps >= 1 m to its leader."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    tab = port_tables[2]
    B, x_init, scen, consts = _platoon(L)
    RNG, MAXS = 40.0, 1200
    sc0 = P.FSM_TRAJ2
    fsms = [P.ObstacleFSMPort(False, c["traffic_light"] == 1, **sc0) for c in consts]
    x = x_init.copy()
    route = np.zeros(B, np.int32)
    hx, hl, hs = [], [], []
    for t in range(MAXS):
        live = x[:, 0] <= tab.s_max - 1.0
        if not live.any():
            break
        lead, lsv = leaders(x, live, route, RNG)
        obs = np.zeros((B, 2, 2))
        n = np.zeros(B, np.int32)
        car = np.full(B, np.nan)
        for b in np.flatnonzero(live):
            o, m, c, _green = fsm_replay(fsms[b], x[b:b + 1, 0], x[b:b + 1, 4])
            obs[b], n[b], car[b] = o[0], m[0], c[0]
        obs, n = merge(obs, n, car, lsv)
        r = T.solve_batch_host(x, obs, n)
        hx.append(np.where(live[:, None], x, np.nan))
        hl.append(lead)
        hs.append(np.where(live, r["status"], -1))
        x = np.where(live[:, None], plant_step(tab, x, r["U"][:, 0]), x)
    n_host = len(hx)
    assert n_host < MAXS
    hx, hl, hs = np.array(hx), np.array(hl), np.array(hs)

    def device(follow):
        sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=MAXS, follow_range=RNG if follow else None)
        sim.run(max_steps=MAXS, check_every=100)
        return sim.state(), sim.history(), sim.follow_history(), sim.follow_check()

    (xf, steps, uns), h, ld, chk = device(True)
    k = int(steps.max())
    assert k == n_host, (k, n_host)
    assert np.array_equal(ld["lead"][:k], hl)
    assert np.array_equal(h["status"][:k], hs)
    assert np.nanmax(np.abs(h["x"][:k] - hx)) <= 1e-7 and np.array_equal(np.isnan(h["x"][:k]), np.isnan(hx))
    assert (hl[:, 1:] == np.arange(B - 1)[None, :]).any(axis=0).all()   # every rear vehicle followed the one ahead
    print(f"\nplatoon: {k} steps, unsolved steps per vehicle {uns.tolist()}, min gaps {chk['min_gap'].round(2).tolist()}")
    # the front vehicle has no leader; every other one keeps more than 1 m, also through its unsolved steps at the light
    assert chk["min_gap"][0] == 1e30 and (chk["min_gap"][1:] >= 1.0).all() and chk["ok"].all()
    live = h["status"][:k] >= 0
    assert (h["status"][:k] == 0).sum() >= 0.8 * live.sum()
    # without following they drive through each other
    (_x, st_off, _u), h_off, ld_off, chk_off = device(False)
    assert (ld_off["lead"] == -1).all() and (chk_off["min_gap"] == 1e30).all()
    s = h_off["x"][..., 0]
    gap = s[:, :-1] - s[:, 1:]                           # vehicle b - 1 is ahead of vehicle b at the start
    assert np.nanmin(gap) < 0.0


# --------------------------------------------------------------------------------------------------------------------
# following off
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_following_off_is_todays_loop(gpu_trackers):
    """4. follow_range=None, and on-then-off before the first step, give today's histories, verdicts and launch count
    bit for bit; switched on halfway, the loop equals the off loop up to that step and records leaders from it on."""
    import safe_autonomous_driving_mpc_b200 as M
    Ls = [gpu_trackers[2][0]]
    B, n, half = 600, 240, 120
    route, x_init, scen, _c, _d, _t = _fleet_setup(Ls * 2, B, 7)

    def run(mode):
        T = M.BatchedTracker(Ls[0])
        kw = {} if mode == "base" else dict(follow_range=None)
        sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=n, **kw)
        if mode == "on_off":
            sim.set_follow(25.0)
            sim.set_follow(None)
        l0 = T.launch_count()
        if mode == "half":
            sim.step(half)
            sim.set_follow(25.0)
            sim.step(n - half)
        else:
            sim.step(n)
        return sim.state(), sim.history(), sim.check(), T.launch_count() - l0, sim.follow_history()

    ref, off, on_off, half_ = run("base"), run("off"), run("on_off"), run("half")
    for got in (off, on_off):
        for a, b in zip(got[0], ref[0]):
            assert np.array_equal(a, b)
        for key in ref[1]:
            assert np.array_equal(got[1][key], ref[1][key], equal_nan=True), key
        for key in ref[2]:
            assert np.array_equal(got[2][key], ref[2][key], equal_nan=True), key
        assert got[3] == ref[3]
        assert (got[4]["lead"] == -1).all() and np.isnan(got[4]["lead_s"]).all()
    for key in ref[1]:
        assert np.array_equal(half_[1][key][:half], ref[1][key][:half], equal_nan=True), key
    assert (half_[4]["lead"][:half] == -1).all() and (half_[4]["lead"][half:] >= 0).any()
    assert not np.array_equal(half_[1]["u"][half:], ref[1]["u"][half:], equal_nan=True)


@pytest.mark.gpu
def test_follow_check_needs_histories(gpu_trackers):
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    sim = M.BatchedSimulation(T, M.make_scenario(2), B=4, follow_range=10.0)
    with pytest.raises(M._lib.MpcbError):
        sim.follow_check()
    assert T._lib.mpcb_sim_follow_check(sim._h, None, None, None) == -1


# --------------------------------------------------------------------------------------------------------------------
# 5. argument checks without a GPU
# --------------------------------------------------------------------------------------------------------------------
def test_follow_arguments_are_checked_without_a_device():
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import _lib
    lib = _lib.load()
    ok, gap, n = np.zeros(4, np.int32), np.zeros(4), C.c_int()
    assert lib.mpcb_sim_set_follow(None, 1, 10.0) == -1
    assert lib.mpcb_sim_set_follow(None, 0, 0.0) == -1
    assert lib.mpcb_sim_follow_history(None, C.byref(n), None, None, None) == -1
    assert lib.mpcb_sim_follow_check(None, ok.ctypes.data_as(C.c_void_p), gap.ctypes.data_as(C.c_void_p), None) == -1
    T = M.BatchedTracker(None)                           # attributes only: the checks come before any device call
    sc = M.make_scenario(2)
    for bad in (0.0, -1.0, -0.0, float("nan"), float("inf"), -float("inf")):
        with pytest.raises(ValueError):
            M.BatchedSimulation(T, sc, B=8, follow_range=bad)
