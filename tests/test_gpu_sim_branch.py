"""Running verdicts (mpcb_sim_running_check), branching (mpcb_sim_branch) and the splitting estimator built on them
(rare_events.offroad_probability).

  1. argument checks of both entry points, in the ABI and in Python, before any device call;
  2. the estimator's arithmetic on a numpy stand-in (Gaussian random walks, V = running max |X|): unbiased against a
     10^7-sample crude estimate of a ~10^-3 event, the crude fraction itself at lam = 0, the plain indicator for
     noiseless walkers that all start alike;
  3. (GPU) running verdicts equal mpcb_sim_check bit for bit on the staggered trajectory2 fleets of
     test_gpu_closed_loop_replay.py driven to the end with full histories: noise off and on, hot start, following,
     two routes; and without histories;
  4. (GPU) an identity branch changes nothing; a branch with duplicates and drops gives every vehicle its parent's
     future, bit for bit, cold and hot-started; with noise on, the copies draw their own slot's noise and the plant
     replay holds; histories longer than the gather window; refusals leave the simulation alone;
  5. (GPU) the estimator on the device: the crude fraction at lam = 0, and agreement with a crude 65,536-drive estimate
     at twice the base noise level of tools/gpu_sim_noise.py on trajectory3.

The GPU half takes about a minute on one B200 (1,000 W power limit)."""
import ctypes as C
import math

import numpy as np
import pytest

from closed_loop_oracle import plant_step
from conftest import traj_path
from noise_oracle import sim_normals
from test_gpu_closed_loop_replay import _fleet_constants

SIGMA = dict(meas=[2.0 ** -6, 2.0 ** -8, 2.0 ** -9, 2.0 ** -11, 2.0 ** -6], act=[2.0 ** -8, 2.0 ** -6],
             proc=[2.0 ** -8, 2.0 ** -9, 2.0 ** -10, 2.0 ** -12, 2.0 ** -7])
SIGMA12 = np.concatenate([SIGMA["meas"], SIGMA["act"], SIGMA["proc"]])
VERDICT_KEYS = ("destination", "on_road", "steering", "acceleration", "obstacle", "light", "passed", "max_dev",
                "min_gap", "s_final", "steps")
HIST_ROW_BYTES = 188            # every history a vehicle can record (include/mpcb200.h, mpcb_sim_branch)


def _w12(nh):
    return np.concatenate([nh["meas"], nh["act"], nh["proc"]], axis=-1)


def branch_launches(B, cap, n_rec):
    """Kernels mpcb_sim_branch launches (include/mpcb200.h)."""
    w = min(cap, max(1, 2 ** 26 // (HIST_ROW_BYTES * B))) if cap > 0 else 1
    return 2 + 2 * (-(-min(n_rec, cap) // w))


# --------------------------------------------------------------------------------------------------------------------
# 1. argument checks (no GPU)
# --------------------------------------------------------------------------------------------------------------------
def test_branch_and_running_check_arguments_are_checked_without_a_device():
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import _lib
    lib = _lib.load()
    v, m, p = np.zeros(4, np.int32), np.zeros((4, 4)), np.zeros(4, np.int32)
    dp = lambda a: a.ctypes.data_as(C.c_void_p)
    assert lib.mpcb_sim_branch(None, dp(p), None) == -1
    assert lib.mpcb_sim_branch(None, None, None) == -1
    assert lib.mpcb_sim_running_check(None, dp(v), dp(m), None) == -1
    assert lib.mpcb_sim_running_check(None, None, None, None) == -1

    class NoDevice(M.BatchedSimulation):                   # attributes only: a device call would fail on _h
        def __init__(self, B):
            self.B, self._lib, self._h = B, None, None

    sim = NoDevice(4)
    for bad in ([0, 1, 2], [0, 1, 2, 3, 0], [[0, 1, 2, 3]], np.zeros(4), [0, 1, 2, 4], [0, -1, 2, 3],
                np.array([0, 1, 2, 2 ** 40]), np.array([True] * 4), ["a"] * 4):
        with pytest.raises(ValueError):
            sim.branch(bad)


# --------------------------------------------------------------------------------------------------------------------
# 2. the estimator on a stand-in (no GPU)
# --------------------------------------------------------------------------------------------------------------------
class WalkFleet:
    """B walkers of n steps, X += drift + sigma z (a fresh draw per slot and step, like the device's slot-keyed noise);
    max_dev = running max |X|, on_road = max_dev <= 1.5, as the device's running verdicts."""

    def __init__(self, B, n, sigma, seed, drift=0.0, x0=0.0):
        self.B, self.n, self.sigma, self.drift = B, n, sigma, drift
        self.rng = np.random.default_rng(seed)
        self.x = np.full(B, float(x0))
        self.v = np.abs(self.x)
        self.st = np.zeros(B, np.int64)
        self.t = 0
        self.branches = 0

    def step(self, k):
        for _ in range(min(k, self.n - self.t)):
            self.x = self.x + self.drift + self.sigma * self.rng.standard_normal(self.B)
            self.v = np.maximum(self.v, np.abs(self.x))
            self.st += 1
            self.t += 1

    def alive(self):
        return self.B if self.t < self.n else 0

    def running_check(self):
        return dict(max_dev=self.v.copy(), on_road=~(self.v > 1.5), steps=self.st.copy())

    def branch(self, parent):
        self.x, self.v, self.st = self.x[parent], self.v[parent], self.st[parent]
        self.branches += 1


N_WALK, SIGMA_WALK = 16, 0.11


def crude_walk_probability(n_samples=10 ** 7, chunk=10 ** 6, seed=1):
    rng = np.random.default_rng(seed)
    hits = 0
    for _ in range(n_samples // chunk):
        X = np.cumsum(SIGMA_WALK * rng.standard_normal((N_WALK, chunk)), axis=0)
        hits += int((np.abs(X).max(axis=0) > 1.5).sum())
    p = hits / n_samples
    return p, math.sqrt(p * (1.0 - p) / n_samples)


def test_estimator_is_unbiased_on_random_walks():
    """Means over 60 repetitions of 1,000 walkers, at three lam, within 4 combined standard errors of a 10^7-sample
    crude estimate (~1.1e-3); lam = 0 is the crude fraction exactly, with no branch; effort is B x n per repetition."""
    from safe_autonomous_driving_mpc_b200.rare_events import offroad_probability
    p_ref, se_ref = crude_walk_probability()
    assert 5e-4 < p_ref < 3e-3, p_ref
    for lam in (4.0, 8.0, 12.0):
        ps = []
        for r in range(60):
            f = WalkFleet(1000, N_WALK, SIGMA_WALK, seed=1000 + r)
            res = offroad_probability(f, lam, 2, seed=r)
            assert res["resamplings"] == f.branches == N_WALK // 2 - 1 and len(res["log_w"]) == res["resamplings"]
            assert res["vehicle_steps"] == 1000 * N_WALK and res["alive"] == 0
            assert all(w >= 0.0 for w in res["log_w"])             # G >= 1: V never decreases
            ps.append(res["p"])
        se = np.std(ps, ddof=1) / math.sqrt(len(ps))
        assert abs(np.mean(ps) - p_ref) <= 4.0 * math.hypot(se, se_ref), (lam, np.mean(ps), se, p_ref, se_ref)
    f = WalkFleet(1000, N_WALK, SIGMA_WALK, seed=7)
    res = offroad_probability(f, 0.0, 3, seed=0)
    g = WalkFleet(1000, N_WALK, SIGMA_WALK, seed=7)
    g.step(N_WALK)
    assert f.branches == 0 and res["resamplings"] == 0 and res["p"] == float(np.mean(g.v > 1.5))


@pytest.mark.parametrize("drift, fails", [(0.05, False), (0.2, True)])
def test_estimator_gives_the_indicator_for_identical_noiseless_walkers(drift, fails):
    from safe_autonomous_driving_mpc_b200.rare_events import offroad_probability
    for lam in (0.0, 0.5, 5.0, 50.0):
        res = offroad_probability(WalkFleet(64, 20, 0.0, seed=0, drift=drift), lam, 3, seed=1)
        assert res["p"] == pytest.approx(1.0 if fails else 0.0, rel=1e-12, abs=0.0), (lam, res)


def test_estimator_checks_its_arguments():
    from safe_autonomous_driving_mpc_b200.rare_events import offroad_probability
    f = WalkFleet(8, 4, 0.1, seed=0)
    for kw in (dict(lam=-1.0), dict(lam=float("nan")), dict(every=0), dict(every=1.5), dict(seed=-1)):
        with pytest.raises(ValueError):
            offroad_probability(f, **dict(dict(lam=1.0, every=1, seed=0), **kw))
    assert f.t == 0


# --------------------------------------------------------------------------------------------------------------------
# fleets on the GPU
# --------------------------------------------------------------------------------------------------------------------
MAX_STEPS, CHUNK = 1200, 100


def _fleet(L, B, seed, route_of=None):
    """Staggered trajectory2 fleet of test_gpu_closed_loop_replay.py (per-vehicle start and scenario constants)."""
    import safe_autonomous_driving_mpc_b200 as M
    s0, consts, dyn, tl = _fleet_constants(L.s_max, B, seed)
    x_init = np.array([L.get_state(s) for s in s0])
    x_init[:, 4] = np.maximum(x_init[:, 4], 0.5)
    scen = [M.make_scenario(2, dynamic_obstacle=int(dyn[b]), traffic_light=int(tl[b]), **consts[b]) for b in range(B)]
    return x_init, scen


def _drive(sim, max_steps=MAX_STEPS):
    n = 0
    while n < max_steps:
        sim.step(CHUNK)
        n += CHUNK
        if sim.alive() == 0:
            break
    return n


def _equal_verdicts(a, b, keys=VERDICT_KEYS):
    return [k for k in keys if not np.array_equal(a[k], b[k], equal_nan=True)]


RUNNING = {"cold": dict(), "noise": dict(noise=dict(seed=7, **SIGMA)), "hot": dict(hot_start=True),
           "follow": dict(follow_range=10.0), "two_routes": dict()}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(RUNNING))
def test_running_check_equals_check(gpu_trackers, case):
    """600 vehicles driven to the end (or MAX_STEPS) with every step recorded: bits 0-5 and all four metrics bit for bit, bit 6 set;
    the same fleet without histories gives the same running verdicts."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    B = 600
    x_init, scen = _fleet(L, B, 32)
    kw = dict(RUNNING[case])
    if case == "two_routes":
        L1 = gpu_trackers[1][0]
        T = M.BatchedTracker([L, L1])
        route = np.arange(B) % 2
        x1, scen1 = _fleet(L1, B, 33)
        x_init = np.where(route[:, None] == 1, x1, x_init)
        scen = [scen1[b] if route[b] else scen[b] for b in range(B)]
        kw["route"] = route
    sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=MAX_STEPS, **kw)
    _drive(sim)                                            # with following a few vehicles stall: every step recorded
    ref, got = sim.check(), sim.running_check()
    assert ref["history_complete"].all() and got["history_complete"].all()
    assert not _equal_verdicts(got, ref), _equal_verdicts(got, ref)
    # the fleets exercise the items: cars and lights met, a spread of gaps and deviations
    assert (ref["min_gap"] < 1e29).any() and (ref["min_gap"] == 1e30).any() and np.isfinite(ref["max_dev"]).all()
    bare = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=0, **kw)
    _drive(bare)
    assert not _equal_verdicts(bare.running_check(), got), _equal_verdicts(bare.running_check(), got)
    with pytest.raises(M._lib.MpcbError):
        bare.check()


def _everything(sim):
    x, st, uns = sim.state()
    return dict(x=x, steps=st, uns=uns, hist=sim.history(), w=_w12(sim.noise_history()), run=sim.running_check())


def _assert_same(a, b, sel=slice(None), what=""):
    assert np.array_equal(a["x"], b["x"][sel]), what
    assert np.array_equal(a["steps"], b["steps"][sel]) and np.array_equal(a["uns"], b["uns"][sel]), what
    for k in a["hist"]:
        assert np.array_equal(a["hist"][k], b["hist"][k][:, sel], equal_nan=True), (what, k)
    assert np.array_equal(a["w"], b["w"][:, sel], equal_nan=True), what
    bad = _equal_verdicts(a["run"], {k: v[sel] for k, v in b["run"].items()})
    assert not bad, (what, bad)


@pytest.mark.gpu
def test_identity_branch_changes_nothing(gpu_trackers):
    """Noisy hot-started fleet of 600, identity branch at step 37: states, every history, the noise history and the
    running verdicts bit for bit; launch count = the unbranched run's + the documented branch kernels."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    B, k, n = 600, 37, 300
    x_init, scen = _fleet(L, B, 41)

    def run(identity):
        sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=n, hot_start=True, noise=dict(seed=3, **SIGMA))
        l0 = T.launch_count()
        sim.step(k)
        if identity:
            sim.branch(np.arange(B))
        sim.step(n - k)
        return _everything(sim), T.launch_count() - l0

    ref, l_ref = run(False)
    got, l_got = run(True)
    _assert_same(got, ref, what="identity")
    assert l_got == l_ref + branch_launches(B, n, k) == l_ref + 4


@pytest.mark.gpu
@pytest.mark.parametrize("hot", [False, True])
def test_branch_with_duplicates_and_drops(gpu_trackers, hot):
    """Noise off, routed fleet of 600 (two routes, per-vehicle scenarios, one execution shape): branched at step 60
    with a random parent map, every output of vehicle b to the end of the drive is the unbranched run's vehicle
    parent[b], bit for bit."""
    import safe_autonomous_driving_mpc_b200 as M
    L, _T = gpu_trackers[2]
    L1 = gpu_trackers[1][0]
    T = M.BatchedTracker([L, L1])
    B, k = 600, 60
    assert B <= T.params.coop_max_batch
    route = (np.arange(B) % 3 == 2).astype(np.int64)
    x_init, scen = _fleet(L, B, 42)
    x1, scen1 = _fleet(L1, B, 43)
    x_init = np.where(route[:, None] == 1, x1, x_init)
    scen = [scen1[b] if route[b] else scen[b] for b in range(B)]
    parent = np.random.default_rng(5).integers(0, B, B)
    assert len(np.unique(parent)) < B

    def run(p):
        sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=MAX_STEPS, hot_start=hot, route=route)
        sim.step(k)
        if p is not None:
            sim.branch(p)
        sim.step(MAX_STEPS - k)                            # the same steps in both runs, stalled vehicles or not
        return _everything(sim)

    ref = run(None)
    assert (ref["steps"] > k).sum() > B // 2
    _assert_same(run(parent), ref, sel=parent, what=f"hot={hot}")


@pytest.mark.gpu
def test_branch_with_noise_draws_the_copies_own_noise(gpu_trackers, port_tables):
    """Noise on, 600 vehicles, branched at step 40: recorded rows before 40 are the parent's; rows from 40 on are
    sigma z of sim_normals for the copy's own id (first_id + b); the plant replay with the recorded disturbances holds
    to 1e-12; the running verdicts equal mpcb_sim_check on the gathered histories."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    B, k, seed, first_id = 600, 40, 11, 1000
    x_init, scen = _fleet(L, B, 44)
    parent = np.random.default_rng(6).integers(0, B, B)
    nz = dict(seed=seed, first_id=first_id, **SIGMA)
    ref = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=k, noise=nz)
    ref.step(k)
    w_ref = _w12(ref.noise_history())
    sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=MAX_STEPS, noise=nz)
    sim.step(k)
    sim.branch(parent)
    n = k + _drive(sim, MAX_STEPS - k)
    assert sim.alive() == 0
    F = _everything(sim)
    h, w, steps = F["hist"], F["w"], F["steps"]
    assert np.array_equal(w[:k], w_ref[:, parent], equal_nan=True)
    t = np.arange(k, n)
    live = t[:, None] < steps[None, :]
    z = sim_normals(seed, first_id + np.arange(B)[None, :], t[:, None])
    assert live.any() and np.abs(w[k:n][live] / SIGMA12 - z[live]).max() <= 1e-12
    assert np.isnan(w[k:n][~live]).all()
    target = np.concatenate([h["x"][1:n], np.full((1, B, 5), np.nan)])
    target[steps - 1, np.arange(B)] = F["x"]
    live = np.arange(n)[:, None] < steps[None, :]
    got = (plant_step(port_tables[2], h["x"][:n], h["u"][:n] + w[:n, :, 5:7]) + w[:n, :, 7:])[live]
    want = target[live]
    assert np.isfinite(want).all()
    assert (np.abs(got - want) / np.maximum(1.0, np.abs(want))).max() <= 1e-12
    assert not _equal_verdicts(F["run"], sim.check())


@pytest.mark.gpu
def test_history_longer_than_the_window_and_refusals(gpu_trackers):
    """4,096 vehicles (87 history rows per window) with following on for the first 20 steps and noise throughout,
    branched at step 200: every recorded row of every history is the parent's (three windows); the launch count is
    the documented one.  Following on, or a parent out of range through the ABI, is refused and changes nothing."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    B, k = 4096, 200
    x_init, scen = _fleet(L, B, 45)
    sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=400, follow_range=10.0, noise=dict(seed=2, **SIGMA))
    sim.step(20)
    parent = np.random.default_rng(7).integers(0, B, B)
    before = _everything(sim)
    with pytest.raises(M._lib.MpcbError):                  # following on
        sim.branch(parent)
    sim.set_follow(None)
    bad = parent.astype(np.int32)
    bad[-1] = B
    assert sim._lib.mpcb_sim_branch(sim._h, bad.ctypes.data_as(C.c_void_p), None) == -1
    _assert_same(_everything(sim), before, what="refused")
    sim.step(k - 20)
    before, lead = _everything(sim), sim.follow_history()
    assert (lead["lead"][:20] >= 0).any() and (lead["lead"][20:] == -1).all()
    l0 = T.launch_count()
    sim.branch(parent)
    assert T.launch_count() - l0 == branch_launches(B, 400, k) == 2 + 2 * 3
    after = _everything(sim)
    _assert_same(after, before, sel=parent, what="windows")
    got = sim.follow_history()
    for q in lead:
        assert np.array_equal(got[q], lead[q][:, parent], equal_nan=True), q


# --------------------------------------------------------------------------------------------------------------------
# 5. the estimator on the device
# --------------------------------------------------------------------------------------------------------------------
# tools/gpu_sim_noise.py's base noise level and trajectory3 fleet (4,096 vehicles of tools/gpu_sim_fleet.py's draws)
BASE = dict(meas=[0.05, 0.02, 0.005, 0.001, 0.05], act=[0.02, 0.1], proc=[0.01, 0.005, 0.002, 0.0005, 0.02])


def trajectory3_fleet(L, B=4096):
    import safe_autonomous_driving_mpc_b200 as M
    rng = np.random.default_rng(11)
    s0 = rng.uniform(0.0, L.s_max - 400.0, B)
    xi = np.array([L.get_state(s) for s in s0])
    xi[:, 4] = np.clip(xi[:, 4], 0.5, None)
    scen = [M.make_scenario(3, tl_pos=float(s + rng.uniform(150, 350)), obs_trigger_s=float(s + 5),
                            obs_start_s=float(s + 60), obs_end_s=float(s + 300)) for s in s0]
    return xi, scen


MAX_DRIVE = 4000


def noise_at(scale, seed):
    return dict(seed=seed, **{k: [scale * v for v in vs] for k, vs in BASE.items()})


@pytest.mark.gpu
def test_estimator_on_the_device():
    """lam = 0 is the crude on_road failure fraction of the running verdicts, bit for bit.  At twice the base noise
    (crude Monte-Carlo sees ~0.27 % on_road failures, tools/gpu_sim_noise.py), the mean of 8 splitting estimates on
    4,096 vehicles (lam = 4, resampling every 500 steps) agrees with a crude estimate on 65,536 drives (16 noise draws of
    the same 4,096 starts) within 4 combined standard errors.  Both are cut at MAX_DRIVE steps: under noise a few
    vehicles stall before their destination, and a failure is counted within the same horizon by both."""
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200.rare_events import offroad_probability
    L = M.TrajectoryLoader(traj_path(3))
    T = M.BatchedTracker(L, **M.FLEET_SOLVER_CAPS)
    xi, scen = trajectory3_fleet(L)
    B = len(xi)
    sim = M.BatchedSimulation(T, scen, x_init=xi, noise=noise_at(2.0, 90))
    res = offroad_probability(sim, 0.0, 100, seed=0, max_steps=MAX_DRIVE)
    assert res["resamplings"] == 0
    assert res["p"] == float(np.mean(~sim.running_check()["on_road"]))
    crude = M.BatchedSimulation(T, scen * 16, x_init=np.tile(xi, (16, 1)), noise=noise_at(2.0, 91))
    crude.run(max_steps=MAX_DRIVE, check_every=100)
    fail = ~crude.running_check()["on_road"]
    p_crude, se_crude = fail.mean(), math.sqrt(fail.mean() * (1.0 - fail.mean()) / fail.size)
    assert 1e-3 <= p_crude <= 1e-2, p_crude
    ps = []
    for r in range(8):
        sim = M.BatchedSimulation(T, scen, x_init=xi, noise=noise_at(2.0, 100 + r))
        res = offroad_probability(sim, 4.0, 500, seed=r, max_steps=MAX_DRIVE)
        assert res["resamplings"] >= 3
        ps.append(res["p"])
    se = np.std(ps, ddof=1) / math.sqrt(len(ps))
    print(f"\ncrude {p_crude:.3e} +- {se_crude:.1e}, splitting {np.mean(ps):.3e} +- {se:.1e}: {ps}")
    assert abs(np.mean(ps) - p_crude) <= 4.0 * math.hypot(se, se_crude), (ps, p_crude, se_crude)
