"""GPU tests of the batched closed loop on the device (mpcb_sim_*, SURVEY 8(f1))."""
import numpy as np
import pytest

from conftest import golden

pytestmark = pytest.mark.gpu


def _scenario(M, i):
    if i == 1:
        return M.make_scenario(2, dynamic_obstacle=0, traffic_light=0)
    return M.make_scenario(i)


@pytest.mark.parametrize("i", [1, 2, 3])
def test_device_loop_matches_host_driven_loop(i, gpu_trackers):
    """The device loop (FSM kernel -> solve -> plant kernel) against the reference-shaped host loop that calls the same
    solver once per step (environment.run_simulation): same step count, same obstacle log, states equal to rounding."""
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import environment as E
    L, T = gpu_trackers[i]
    sc = {1: None, 2: E.SCENARIO_TRAJECTORY2, 3: E.SCENARIO_TRAJECTORY3}[i]
    fsm = M.ObstaclesFSM(dynamic_obstacle=i > 1, traffic_light=i > 1, scenario=sc)
    flags = []
    hx, hu, ht, hp, hobs, htl, _ = M.run_simulation(T, fsm, L, record_flags=flags)
    sim = M.BatchedSimulation(T, _scenario(M, i), B=1, history_steps=len(hu) + 64)
    n = sim.run(max_steps=len(hu) + 64, check_every=32)
    x, steps, unsolved = sim.state()
    assert steps[0] == len(hu), (steps[0], len(hu))
    assert n >= steps[0] and sim.alive() == 0
    h = sim.history()
    k = steps[0]
    assert np.all(h["status"][k:, 0] == -1)                                   # frozen after arrival
    assert np.abs(h["x"][:k, 0] - hx[:-1]).max() <= 1e-7
    assert np.abs(x[0] - hx[-1]).max() <= 1e-7
    assert np.abs(h["u"][:k, 0] - hu).max() <= 1e-6
    obs_ref = np.array(hobs, dtype=np.float64)
    assert np.array_equal(np.isnan(h["obs_s"][:k, 0]), np.isnan(obs_ref))
    assert np.nanmax(np.abs(h["obs_s"][:k, 0] - obs_ref), initial=0.0) <= 1e-9
    assert [("GREEN" if t else "RED") for t in h["tl"][:k, 0]] == list(htl)
    assert unsolved[0] == sum(1 for f in flags if f[0] != 0)
    # vectorised sanity checks == the reference's verdicts on its own run (all items pass, sanity_checks.py:79-184)
    c = sim.check()
    assert c["passed"][0] and c["history_complete"][0] and c["steps"][0] == k
    assert abs(c["max_dev"][0] - np.abs(np.vstack([h["x"][:k, 0], x[:1]])[:, 1]).max()) == 0.0
    # same step count as the unmodified reference's own run (172 / 985 / 2294)
    z = golden(f"closed_loop_traj{i}")
    assert k == len(z["hist_u"])


def test_many_vehicles_monte_carlo(gpu_trackers):
    """256 vehicles on trajectory2 with perturbed starts and per-vehicle scenario constants: copies of the same vehicle
    are bitwise identical, every vehicle arrives, nobody collides with the car or runs the red light."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    rng = np.random.default_rng(11)
    B = 256
    x_init = np.tile([0.0, 0.0, 0.0, 0.0, 0.5], (B, 1))
    x_init[8:, 1] += rng.normal(0, 0.05, B - 8)
    x_init[8:, 4] += rng.uniform(0, 3.0, B - 8)
    scen = []
    for b in range(B):
        if b < 8:
            scen.append(M.make_scenario(2))
        else:
            scen.append(M.make_scenario(2, obs_v=float(rng.uniform(3.0, 6.0)), tl_pos=float(rng.uniform(450.0, 650.0)),
                                        tl_stop_duration=float(rng.uniform(5.0, 25.0))))
    sim = M.BatchedSimulation(T, scen, B=B, x_init=x_init, history_steps=3000)
    sim.run(max_steps=3000, check_every=100)
    assert sim.alive() == 0
    x, steps, unsolved = sim.state()
    h = sim.history()
    assert np.all(x[:, 0] > L.s_max - 1.0) and np.all(np.isfinite(x))
    for b in range(1, 8):
        assert steps[b] == steps[0]
        assert np.array_equal(h["x"][:, b], h["x"][:, 0], equal_nan=True)
    # safety verdicts per vehicle (sanity_checks.py:141-176): gap to the car >= 1 m, red light not run
    for b in range(B):
        k = steps[b]
        gap = h["obs_s"][:k, b] - h["x"][:k, b, 0]
        assert np.nanmin(np.where(gap > -50.0, gap, np.nan), initial=np.inf) >= 1.0
        red = h["tl"][:k, b] == 0
        tl_pos = scen[b].tl_pos
        assert np.all(h["x"][:k, b, 0][red] <= tl_pos + 1e-9)
    assert (unsolved / np.maximum(steps, 1)).mean() < 0.1
    # the device check against a numpy restatement of sanity_checks.py:79-184 on the same histories
    c = sim.check()
    for b in range(B):
        k = steps[b]
        hx = np.vstack([h["x"][:k, b], x[b:b + 1]])
        hu = h["u"][:k, b]
        ref = dict(destination=not (hx[-1, 0] < L.s_max - 1.0), on_road=not (np.abs(hx[:, 1]).max() > 1.5),
                   steering=not (hu[:, 0].min() < -0.6 - 0.1 or hu[:, 0].max() > 0.6 + 0.1),
                   acceleration=not (hu[:, 1].min() < -5.0 - 0.1 or hu[:, 1].max() > 4.0 + 0.1))
        os_ = h["obs_s"][:k, b]
        m = ~np.isnan(os_)
        ref["obstacle"] = not (m.any() and (os_[m] - hx[:k, 0][m]).min() < 1.0)
        idx = np.where(hx[:, 0] > scen[b].tl_pos)[0]
        ref["light"] = not (len(idx) > 0 and idx[0] < k and h["tl"][idx[0], b] == 0)
        for name, val in ref.items():
            assert bool(c[name][b]) == val, (b, name)
    assert c["passed"].all() and c["history_complete"].all()


def test_device_checks_against_the_reference_function(gpu_trackers):
    """mpcb_check_histories (the kernel behind BatchedSimulation.check) against the UNMODIFIED reference's
    trajectory_tracking_check (sanity_checks.py:79-184) on recorded drives that pass and on variants that FAIL an item:
    stopped short, |d| > 1.5, a control past its limit +- 0.1 (and exactly on it), the car within 1 m (and exactly 1 m,
    and behind), a run red light, items switched off in the scenario, several at once.  Fixture:
    tests/golden/sanity_cases.npz from tools/make_golden_sanity.py (verdict per item parsed from the reference's
    output, overall verdict = its return value)."""
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import simulation as S
    z = golden("sanity_cases")
    _, T = gpu_trackers[2]
    names = [str(x) for x in z["item_names"]]
    assert (~z["ref_passed"]).sum() >= 10 and z["ref_passed"].sum() >= 5
    for s_total in np.unique(z["s_total"]):
        sel = np.where(z["s_total"] == s_total)[0]
        scen = [M.make_scenario(2, dynamic_obstacle=int(z["dynamic_obstacle"][b]), traffic_light=int(z["traffic_light"][b]),
                                tl_pos=float(z["tl_pos"][b])) for b in sel]
        c = S.check_histories(T, float(s_total), scen, z["x_final"][sel], z["steps"][sel], z["hist_x"][:, sel],
                              z["hist_u"][:, sel], z["hist_obs"][:, sel], z["hist_tl"][:, sel])
        for k, b in enumerate(sel):
            for j, name in enumerate(names):
                assert bool(c[name][k]) == bool(z["ref_items"][b, j]), (str(z["names"][b]), name)
            assert bool(c["passed"][k]) == bool(z["ref_passed"][b]), str(z["names"][b])
            assert c["steps"][k] == z["steps"][b] and c["history_complete"][k]


def test_stop_line_inside_the_tight_bend_is_a_fixed_point(gpu_trackers):
    """Known limitation (DESIGN.md 4, K-sim): a red light placed INSIDE the tight bend of trajectory3 (s ~ 720-728 m),
    where the committed reference trajectory itself leaves the lane margin, makes the tracking MPC as formulated a
    fixed point at standstill -- the optimum of the reference formulation is 'stay put'.  This test pins that behaviour
    (the vehicle stops before the line, never runs the light, never leaves the road, never collides) instead of leaving
    it undocumented; nothing on the three committed scenarios comes near this state."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[3]
    scen = M.make_scenario(3, dynamic_obstacle=0, tl_pos=726.0, tl_stop_duration=6.0)
    x_init = np.tile(L.get_state(600.0), (1, 1))
    x_init[0, 4] = 6.0
    sim = M.BatchedSimulation(T, scen, B=1, x_init=x_init, history_steps=1500)
    sim.step(1500)
    x, steps, unsolved = sim.state()
    h = sim.history()
    k = int(steps[0])
    red = h["tl"][:k, 0] == 0
    assert np.all(h["x"][:k, 0, 0][red] <= 726.0 + 1e-9), "ran the red light"
    assert np.abs(h["x"][:k, 0, 1]).max() <= 1.5 and np.all(np.isfinite(x))
    # reversing at a red light is a property of the formulation (SURVEY 4.3: the reference solved to convergence reaches
    # -0.96 m/s on trajectory2's red-light approach, -1.6 m/s as shipped); measured here on B200: -0.37 m/s
    assert h["x"][:k, 0, 4].min() >= -0.96
    # it reaches the stop line region and comes to rest there
    assert h["x"][:k, 0, 0].max() > 700.0
    if x[0, 0] <= 726.0:                                      # stuck at the fixed point: at rest, same answer every step
        assert abs(x[0, 4]) < 0.05 and np.abs(np.diff(h["x"][k - 50:k, 0, 0])).max() < 1e-3


def test_fleet_caps_drive_a_staggered_fleet_like_the_defaults(gpu_trackers):
    """FLEET_SOLVER_CAPS (three active-set updates per linearisation in the thread-per-problem first pass) only move
    problems from the robust pass into the first pass: a staggered fleet of 4,000 vehicles on trajectory2 (> 3,072, so the
    bulk kernel drives it) with per-vehicle scenarios arrives with the same verdicts and, vehicle by vehicle, within a
    few steps of the default caps' run."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    B = 4000
    rng = np.random.default_rng(21)
    s0 = rng.uniform(0.0, L.s_max - 500.0, B)
    xi = np.array([L.get_state(s) for s in s0])
    xi[:, 4] = np.clip(xi[:, 4], 0.5, None)
    scen = [M.make_scenario(2, tl_pos=float(s + rng.uniform(120, 300)), obs_trigger_s=float(s + 5), obs_start_s=float(s + 50),
                            obs_end_s=float(s + 250), tl_stop_duration=4.0) for s in s0]
    runs = []
    for T_ in (T, M.BatchedTracker(L, **M.FLEET_SOLVER_CAPS)):
        sim = M.BatchedSimulation(T_, scen, x_init=xi, history_steps=2600)
        sim.run(max_steps=2600, check_every=200)
        # a few vehicles whose random stop line fell where the reference trajectory itself leaves the lane margin stay at
        # the formulation's standstill fixed point (DESIGN.md 4, K-sim; test_stop_line_inside_the_tight_bend...)
        assert sim.alive() <= B // 200
        runs.append((sim.state(), sim.check()))
    (xa, sa, ua), ca = runs[0]
    (xb, sb, ub), cb = runs[1]
    both = ca["destination"] & cb["destination"]
    assert both.mean() > 0.99
    for name in M.BatchedSimulation.CHECKS:
        assert np.mean(ca[name] == cb[name]) > 0.995, name
    assert ca["passed"].mean() > 0.97 and cb["passed"].mean() > 0.97
    d = np.abs(sa - sb)[both]
    assert np.quantile(d, 0.99) <= 3 and d.max() <= 0.05 * sa.max(), (np.quantile(d, [0.5, 0.99]), d.max())


@pytest.mark.parametrize("i", [1, 2, 3])
def test_hot_start_drives_the_same_closed_loop(i, gpu_trackers):
    """mpcb_sim_set_hot_start: from its second step on a vehicle's first pass starts from its previous plan advanced by one
    step, rows on their bounds taken as active.  The problem and its converged answer are the same: the device loop takes
    the reference's step counts (172 / 985 / 2294), passes the same checks and follows the default loop's states -- up to
    the last 10 m of the route, where the horizon runs off the end of the table and the optimum is no longer unique
    (DESIGN.md 5, envelope test)."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[i]
    scen = M.make_scenario(2, dynamic_obstacle=0, traffic_light=0) if i == 1 else M.make_scenario(i)
    want = {1: 172, 2: 985, 3: 2294}[i]
    out = []
    for hot in (False, True):
        sim = M.BatchedSimulation(T, scen, B=4, history_steps=want + 8, hot_start=hot)
        sim.run(max_steps=want + 8, check_every=64)
        x, steps, uns = sim.state()
        c = sim.check()
        assert np.all(steps == want) and c["passed"].all() and c["history_complete"].all()
        out.append((sim.history(), uns))
    (ha, ua), (hb, ub) = out
    assert np.abs(ua - ub).max() <= 3
    far = ha["x"][:want, 0, 0] < L.s_max - 10.0
    dx = np.abs(ha["x"][:want, 0] - hb["x"][:want, 0])[far]
    # trajectory1 / 3: 1e-6 .. 1e-5.  trajectory2: 0.075 m / 1.2e-4 m / 0.027 m/s -- its red-light approach is infeasible
    # for 70 steps in a row, and what an infeasible problem returns depends on the path the solver took (SURVEY 4.4-4:
    # flags only there); the two loops rejoin behind the light
    assert dx[:, 1].max() <= 5e-4 and dx[:, 2].max() <= 5e-4 and dx[:, 4].max() <= 0.05 and dx[:, 0].max() <= 0.1, dx.max(axis=0)


def test_failed_create_and_destroy_leave_no_device_memory_behind(gpu_trackers):
    """A simulation whose histories cannot be allocated (100,000 vehicles x 10^7 recorded steps, some 70 TB) is refused
    with MPCB_ERR_NOMEM (-3) and holds no device memory; a created, following, stepped and destroyed simulation gives all
    of its device memory back; a simulation created afterwards steps as usual.  The driver keeps freed pages of small
    allocations for reuse and returns them when an allocation fails, so every reading of free memory is taken right
    after a refused create, with the garbage collector off."""
    import ctypes as C
    import gc
    import torch
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    sc = M.make_scenario(2)
    x_init = np.array([L.get_state(s) for s in (100.0, 104.0, 300.0, 303.0)])
    x_init[:, 4] = np.maximum(x_init[:, 4], 0.5)

    def following_run():
        sim = M.BatchedSimulation(T, sc, x_init=x_init, history_steps=16, follow_range=10.0)
        sim.step(8)
        lead = sim.follow_history()["lead"]
        del sim
        return lead

    def free_after_refused_create():
        h = C.c_void_p()
        rc = T._lib.mpcb_sim_create_routes(C.byref(h), T._need(), 100_000, (M._lib.Scenario * 1)(sc), 1, None, None,
                                           10_000_000)
        assert rc == -3 and not h.value
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info()[0]

    # once before measuring: the handle's solve workspace and the modules of the kernels are loaded on first use
    assert (following_run() >= 0).any()
    gc.collect()
    gc.disable()
    try:
        free0 = free_after_refused_create()
        assert free_after_refused_create() == free0
        assert (following_run() >= 0).any()
        assert free_after_refused_create() == free0
    finally:
        gc.enable()
    sim = M.BatchedSimulation(T, sc, x_init=x_init, history_steps=8)
    sim.step(8)
    x, steps, _ = sim.state()
    assert np.all(steps == 8) and np.all(np.isfinite(x)) and np.all(x[:, 0] > x_init[:, 0])
