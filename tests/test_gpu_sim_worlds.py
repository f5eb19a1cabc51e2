"""Worlds in one closed-loop fleet (mpcb_sim_set_worlds), the running follower gap (mpcb_sim_running_follow_check),
world branching (mpcb_sim_branch_worlds) and the near-miss splitting estimate built on them
(rare_events.near_miss_probability).

  1. argument checks of the three entry points, in the ABI and in Python, before any device call;
  2. the per-world leader rule in numpy (lexsort by world, route key, s key, index) on hand-made cases: equal positions,
     -0.0, arrived vehicles, M = 1, and one world equal to the rule of test_gpu_sim_follow.py;
  3. the estimator's arithmetic on a numpy stand-in (worlds of followers whose gaps are random walks) against a
     10^7-sample crude estimate, and the crude fraction itself at lam = 0;
  4. (GPU) recorded leaders equal the numpy rule bit for bit on two-route fleets with equal starts, M = 1, 8, 64, 1024,
     cold and hot;
  5. (GPU) set_worlds(B) equals following without worlds bit for bit (the world kernel against the radix-sort path),
     with one kernel fewer per step; the running follower gap equals follow_check on both paths, noise off and on, cold
     and hot, and without histories;
  6. (GPU) identical 8-car platoons in W worlds (one execution shape) drive alike and as a standalone platoon, and with
     noise world w drives as a standalone platoon with first_id = w M;
  7. (GPU) branch_worlds: the identity changes nothing; duplicates and drops with following on give every copy its
     parent world's state, histories (leaders translated) and future; noisy copies draw their own slots' normals;
     refusals;
  8. (GPU) the estimator on the device: the crude fraction at lam = 0, and agreement with crude Monte-Carlo on a
     tight, noisy platoon setting.

The GPU half takes about 10 s on one B200 (1,000 W power limit)."""
import ctypes as C
import math

import numpy as np
import pytest

from closed_loop_oracle import leaders
from conftest import traj_path
from noise_oracle import sim_normals
from test_gpu_sim_follow import EQUAL_PAIRS, _fleet_setup, _platoon

SIGMA = dict(meas=[2.0 ** -6, 2.0 ** -8, 2.0 ** -9, 2.0 ** -11, 2.0 ** -6], act=[2.0 ** -8, 2.0 ** -6],
             proc=[2.0 ** -8, 2.0 ** -9, 2.0 ** -10, 2.0 ** -12, 2.0 ** -7])
SIGMA12 = np.concatenate([SIGMA["meas"], SIGMA["act"], SIGMA["proc"]])
HIST_ROW_BYTES = 188            # every history a vehicle can record (include/mpcb200.h, mpcb_sim_branch)
VERDICT_KEYS = ("destination", "on_road", "steering", "acceleration", "obstacle", "light", "passed", "max_dev",
                "min_gap", "s_final", "steps")


def branch_launches(B, cap, n_rec):
    """Kernels mpcb_sim_branch and mpcb_sim_branch_worlds launch (include/mpcb200.h)."""
    w = min(cap, max(1, 2 ** 26 // (HIST_ROW_BYTES * B))) if cap > 0 else 1
    return 2 + 2 * (-(-min(n_rec, cap) // w))


# --------------------------------------------------------------------------------------------------------------------
# 1. argument checks (no GPU)
# --------------------------------------------------------------------------------------------------------------------
def test_world_arguments_are_checked_without_a_device():
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import _lib
    lib = _lib.load()
    ok, g, p = np.zeros(8, np.int32), np.zeros(8), np.zeros(2, np.int32)
    dp = lambda a: a.ctypes.data_as(C.c_void_p)
    for m in (0, 4, -1, 2048):
        assert lib.mpcb_sim_set_worlds(None, m) == -1
    assert lib.mpcb_sim_running_follow_check(None, dp(ok), dp(g), None) == -1
    assert lib.mpcb_sim_running_follow_check(None, None, None, None) == -1
    assert lib.mpcb_sim_branch_worlds(None, dp(p), None) == -1
    assert lib.mpcb_sim_branch_worlds(None, None, None) == -1

    T = M.BatchedTracker(None)                           # attributes only: the checks come before any device call
    sc = M.make_scenario(2)
    for bad in (3, 1025, 2048, -1, -8, 1.0, 8.0, True, "8", np.float64(4.0)):
        with pytest.raises(ValueError):
            M.BatchedSimulation(T, sc, B=2048 if bad == 2048 else 8, world_size=bad)

    class NoDevice(M.BatchedSimulation):                   # attributes only: a device call would fail on _h
        def __init__(self, B, world_size=None):
            self.B, self._lib, self._h = B, None, None
            self.world_size, self.W = (world_size, B // world_size) if world_size else (None, 1)

    sim = NoDevice(24)
    for bad in (5, 7, 48, 1025, -2, -24, 2.0, False):
        with pytest.raises(ValueError):
            sim.set_worlds(bad)
    with pytest.raises(ValueError):                        # no worlds
        sim.branch_worlds([0])
    sim = NoDevice(24, world_size=8)
    for bad in ([0, 1], [0, 1, 2, 0], [[0, 1, 2]], np.zeros(3), [0, 1, 3], [0, -1, 2], np.array([0, 1, 2 ** 40]),
                np.array([True] * 3), ["a"] * 3, list(range(24))):
        with pytest.raises(ValueError):
            sim.branch_worlds(bad)


# --------------------------------------------------------------------------------------------------------------------
# 2. the per-world leader rule (no GPU)
# --------------------------------------------------------------------------------------------------------------------
def s_keys(s):
    """The device's order-preserving 64-bit key of s + 0.0 (-0.0 folded onto +0.0)."""
    u = (np.asarray(s, np.float64) + 0.0).view(np.uint64)
    return np.where((u >> np.uint64(63)) == 1, ~u, u | np.uint64(1 << 63))


def world_leaders(x, live, route, M, follow_range):
    """mpcb_sim_set_worlds' leader rule for one step: x [B,5] states at the start of the step, live [B] still driving,
    route [B], world size M.  The live vehicles ordered by (world, route, s key, index); the leader of b is the next one
    when it is in b's world and on b's route and s_leader - s_b <= follow_range.  Returns lead [B] (-1: none) and
    lead_sv [B,2] (NaN: none)."""
    B = len(x)
    idx = np.flatnonzero(live)
    order = idx[np.lexsort((idx, s_keys(x[idx, 0]), route[idx], idx // M))]
    a, b = order[:-1], order[1:]
    near = (a // M == b // M) & (route[a] == route[b]) & (x[b, 0] - x[a, 0] <= follow_range)
    lead = np.full(B, -1, np.int64)
    lead[a[near]] = b[near]
    sv = np.full((B, 2), np.nan)
    has = lead >= 0
    sv[has] = x[lead[has]][:, [0, 4]]
    return lead, sv


def test_world_leader_rule_on_hand_made_cases():
    """Equal positions ordered by index, -0.0 equal to +0.0, routes and worlds apart, arrived vehicles nobody's leader
    and without one, the range filter, M = 1 without leaders, one world equal to the global rule."""
    s = np.array([10.0, 10.0, -0.0, 0.0, 5.0, 12.0, 11.0, 5.0])
    x = np.zeros((8, 5))
    x[:, 0] = s
    x[:, 4] = np.arange(8) + 0.5
    route = np.array([0, 0, 0, 0, 0, 1, 0, 0])
    live = np.array([True] * 7 + [False])
    # world 0 by (s key, b): 2 (-0.0), 3 (0.0), 0, 1; world 1, route 0: 4 (5), 6 (11); 5 alone on route 1; 7 arrived
    lead, sv = world_leaders(x, live, route, 4, 20.0)
    assert lead.tolist() == [1, -1, 3, 0, 6, -1, -1, -1]
    assert np.array_equal(sv[2], [0.0, 3.5]) and np.array_equal(sv[4], [11.0, 6.5]) and np.isnan(sv[1]).all()
    lead, _ = world_leaders(x, live, route, 4, 6.0)
    assert lead.tolist() == [1, -1, 3, -1, 6, -1, -1, -1]            # 10 - 0 > 6; 11 - 5 = 6 <= 6
    lead, _ = world_leaders(x, live, route, 4, np.nextafter(6.0, 0.0))
    assert lead[4] == -1
    # -0.0 without the fold would come first: its bit pattern is smaller as a signed-magnitude key
    assert s_keys([-0.0])[0] == s_keys([0.0])[0]
    # one world: 2, 3, 4, 0, 1, 6 on route 0
    lead, _ = world_leaders(x, live, route, 8, 20.0)
    assert lead.tolist() == [1, 6, 3, 4, 0, -1, -1, -1]
    assert np.array_equal(lead, leaders(x, live, route, 20.0)[0])
    lead, sv = world_leaders(x, live, route, 1, 1e9)
    assert (lead == -1).all() and np.isnan(sv).all()
    # random fleets with ties: each world is the global rule on its slice; one world is the global rule
    rng = np.random.default_rng(0)
    for M in (1, 2, 8, 64):
        B = 256
        x = np.zeros((B, 5))
        x[:, 0] = rng.integers(-3, 40, B) * 0.5
        x[:, 0][rng.random(B) < 0.1] = -0.0
        x[:, 4] = rng.random(B)
        route = rng.integers(0, 3, B)
        live = rng.random(B) < 0.9
        lead, sv = world_leaders(x, live, route, M, 4.0)
        for w in range(B // M):
            sl = slice(w * M, (w + 1) * M)
            ref, rsv = leaders(x[sl], live[sl], route[sl], 4.0)
            assert np.array_equal(lead[sl], np.where(ref >= 0, ref + w * M, -1))
            assert np.array_equal(sv[sl], rsv, equal_nan=True)
    assert np.array_equal(world_leaders(x, live, route, B, 4.0)[0], leaders(x, live, route, 4.0)[0])


# --------------------------------------------------------------------------------------------------------------------
# 3. the estimator on a stand-in (no GPU)
# --------------------------------------------------------------------------------------------------------------------
class GapWorlds:
    """W worlds of M vehicles: vehicle 0 of a world leads (no leader: 1e30), the gap of each follower is g0 plus a random
    walk (a fresh draw per slot and step, like the device's slot-keyed noise); min_gap = running least gap, ok =
    min_gap >= 1, as the device's running follow check."""

    def __init__(self, W, M, n, sigma, seed, g0=2.5):
        self.W, self.M, self.B, self.n, self.sigma = W, M, W * M, n, sigma
        self.rng = np.random.default_rng(seed)
        self.gap = np.full((W, M - 1), float(g0))
        self.min_gap = np.full(self.B, 1e30)
        self.st = np.zeros(self.B, np.int64)
        self.t = 0
        self.branches = 0

    def step(self, k):
        for _ in range(min(k, self.n - self.t)):
            self.gap = self.gap + self.sigma * self.rng.standard_normal(self.gap.shape)
            g = self.min_gap.reshape(self.W, self.M)
            g[:, 1:] = np.minimum(g[:, 1:], self.gap)
            self.st += 1
            self.t += 1

    def alive(self):
        return self.B if self.t < self.n else 0

    def running_check(self):
        return dict(steps=self.st.copy())

    def running_follow_check(self):
        return dict(ok=~(self.min_gap < 1.0), min_gap=self.min_gap.copy())

    def branch_worlds(self, parent):
        W, M = self.W, self.M
        self.gap = self.gap[parent]
        self.min_gap = self.min_gap.reshape(W, M)[parent].reshape(-1)
        self.st = self.st.reshape(W, M)[parent].reshape(-1)
        self.branches += 1


N_GAP, M_GAP, SIGMA_GAP, GAP_CAP = 16, 3, 0.11, 2.5


def crude_gap_probability(n_samples=10 ** 7, chunk=10 ** 6, seed=1):
    rng = np.random.default_rng(seed)
    hits = 0
    for _ in range(n_samples // chunk):
        G = 2.5 + np.cumsum(SIGMA_GAP * rng.standard_normal((N_GAP, M_GAP - 1, chunk), dtype=np.float32), axis=0)
        hits += int((G.min(axis=(0, 1)) < 1.0).sum())
    p = hits / n_samples
    return p, math.sqrt(p * (1.0 - p) / n_samples)


def test_near_miss_estimator_is_unbiased_on_random_walks():
    """Means over 60 repetitions of 1,000 worlds of 3, at three lam, within 4 combined standard errors of a
    10^7-sample crude estimate (~1e-3); lam = 0 is the crude fraction of worlds exactly, with no branch."""
    from safe_autonomous_driving_mpc_b200.rare_events import near_miss_probability
    p_ref, se_ref = crude_gap_probability()
    assert 3e-4 < p_ref < 3e-3, p_ref
    for lam in (4.0, 8.0, 12.0):
        ps = []
        for r in range(60):
            f = GapWorlds(1000, M_GAP, N_GAP, SIGMA_GAP, seed=1000 + r)
            res = near_miss_probability(f, lam, 2, seed=r, gap_cap=GAP_CAP)
            assert res["resamplings"] == f.branches == N_GAP // 2 - 1 and len(res["log_w"]) == res["resamplings"]
            assert res["vehicle_steps"] == 1000 * M_GAP * N_GAP and res["alive"] == 0
            assert all(w >= 0.0 for w in res["log_w"])             # G >= 1: V never decreases
            ps.append(res["p"])
        se = np.std(ps, ddof=1) / math.sqrt(len(ps))
        assert abs(np.mean(ps) - p_ref) <= 4.0 * math.hypot(se, se_ref), (lam, np.mean(ps), se, p_ref, se_ref)
    f = GapWorlds(1000, M_GAP, N_GAP, SIGMA_GAP, seed=7)
    res = near_miss_probability(f, 0.0, 3, seed=0, gap_cap=GAP_CAP)
    g = GapWorlds(1000, M_GAP, N_GAP, SIGMA_GAP, seed=7)
    g.step(N_GAP)
    assert f.branches == 0 and res["resamplings"] == 0
    assert res["p"] == float(np.mean((g.min_gap.reshape(1000, M_GAP) < 1.0).any(axis=1)))


def test_near_miss_estimator_checks_its_arguments():
    from safe_autonomous_driving_mpc_b200.rare_events import near_miss_probability
    f = GapWorlds(8, 3, 4, 0.1, seed=0)
    for kw in (dict(lam=-1.0), dict(lam=float("nan")), dict(every=0), dict(every=1.5), dict(seed=-1),
               dict(gap_cap=1.0), dict(gap_cap=0.5), dict(gap_cap=float("inf")), dict(gap_cap=float("nan"))):
        with pytest.raises(ValueError):
            near_miss_probability(f, **dict(dict(lam=1.0, every=1, seed=0, gap_cap=2.0), **kw))
    assert f.t == 0


# --------------------------------------------------------------------------------------------------------------------
# fleets on the GPU
# --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def routed2():
    """A two-route tracker (trajectory2, trajectory3) and its loaders."""
    import safe_autonomous_driving_mpc_b200 as M
    Ls = [M.TrajectoryLoader(traj_path(i)) for i in (2, 3)]
    return Ls, M.BatchedTracker(Ls)


@pytest.fixture(scope="module")
def bulk2():
    """trajectory2 with one execution shape for every batch size (thread-per-problem first pass), so that a world's
    solves do not depend on how many other worlds share the batch."""
    import safe_autonomous_driving_mpc_b200 as M
    L = M.TrajectoryLoader(traj_path(2))
    return L, M.BatchedTracker(L, coop_max_batch=0)


def _w12(nh):
    return np.concatenate([nh["meas"], nh["act"], nh["proc"]], axis=-1)


def _everything(sim):
    x, st, uns = sim.state()
    return dict(x=x, steps=st, uns=uns, hist=sim.history(), w=_w12(sim.noise_history()), lead=sim.follow_history(),
                run=sim.running_check(), gap=sim.running_follow_check())


def _translated(lead, shift):
    """Leader indices moved by shift [B] (broadcast over rows), -1 kept."""
    return np.where(lead >= 0, lead + shift, lead)


def _assert_same(a, b, sel=slice(None), shift=0, what=""):
    """a equals b's vehicles sel (every output), a's recorded leaders equal b's moved by shift."""
    assert np.array_equal(a["x"], b["x"][sel]), what
    assert np.array_equal(a["steps"], b["steps"][sel]) and np.array_equal(a["uns"], b["uns"][sel]), what
    for k in a["hist"]:
        assert np.array_equal(a["hist"][k], b["hist"][k][:, sel], equal_nan=True), (what, k)
    assert np.array_equal(a["w"], b["w"][:, sel], equal_nan=True), what
    assert np.array_equal(a["lead"]["lead"], _translated(b["lead"]["lead"][:, sel], shift)), what
    for k in ("lead_s", "lead_v"):
        assert np.array_equal(a["lead"][k], b["lead"][k][:, sel], equal_nan=True), (what, k)
    for k in VERDICT_KEYS:
        assert np.array_equal(a["run"][k], b["run"][k][sel], equal_nan=True), (what, k)
    for k in ("ok", "min_gap"):
        assert np.array_equal(a["gap"][k], b["gap"][k][sel]), (what, k)


# --------------------------------------------------------------------------------------------------------------------
# 4. the leader rule on the device
# --------------------------------------------------------------------------------------------------------------------
WORLD_RANGE = 150.0


@pytest.mark.gpu
@pytest.mark.parametrize("hot", [False, True])
def test_recorded_leaders_follow_the_world_rule(routed2, hot):
    """2,048 vehicles on two routes with equal starting pairs, 120 steps recorded, for M = 1, 8, 64, 1024: at every step
    the numpy world rule on the recorded states gives hist_lead_idx and hist_lead_sv bit for bit."""
    import safe_autonomous_driving_mpc_b200 as M
    Ls, T = routed2
    B, n = 2048, 120
    route, x_init, scen, *_ = _fleet_setup(Ls, B, 51)
    for m in (1, 8, 64, 1024):
        sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=n, hot_start=hot, route=route,
                                  follow_range=WORLD_RANGE, world_size=m)
        assert sim.W == B // m and sim.world_size == m
        sim.step(n)
        h, ld, steps = sim.history(), sim.follow_history(), sim.state()[1]
        n_lead = 0
        for t in range(n):
            live = steps > t
            x = np.where(live[:, None], h["x"][t], 0.0)
            lead, sv = world_leaders(x, live, route, m, WORLD_RANGE)
            assert np.array_equal(ld["lead"][t], lead), (m, t, np.flatnonzero(ld["lead"][t] != lead)[:8])
            assert np.array_equal(ld["lead_s"][t], sv[:, 0], equal_nan=True), (m, t)
            assert np.array_equal(ld["lead_v"][t], sv[:, 1], equal_nan=True), (m, t)
            n_lead += int((lead >= 0).sum())
        if m == 1:
            assert n_lead == 0
        else:
            assert n_lead > 0, m
            a, b = EQUAL_PAIRS[0]
            assert ld["lead"][0, a] == b                    # equal starts in one world: the higher index leads


# --------------------------------------------------------------------------------------------------------------------
# 5. one world of B against the radix-sort path; the running follower gap
# --------------------------------------------------------------------------------------------------------------------
CROSS = {"cold": dict(), "hot": dict(hot_start=True), "noise": dict(noise=dict(seed=5, **SIGMA)),
         "noise_hot": dict(hot_start=True, noise=dict(seed=6, **SIGMA))}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CROSS))
def test_one_world_equals_following_without_worlds(routed2, case):
    """600 vehicles on two routes, 300 steps recorded, following within 10 m: set_worlds(600) gives every output of
    following without worlds bit for bit (states, statuses, histories, leaders, verdicts, follow checks) with one
    kernel fewer per step; on both paths the running follower gap equals follow_check bit for bit, and a world-path
    run without histories gives the same running gap."""
    import safe_autonomous_driving_mpc_b200 as M
    Ls, T = routed2
    B, n = 600, 300
    route, x_init, scen, *_ = _fleet_setup(Ls, B, 41)
    kw = dict(x_init=x_init, route=route, follow_range=10.0, **CROSS[case])

    def run(world_size, hist=n):
        sim = M.BatchedSimulation(T, scen, history_steps=hist, world_size=world_size, **kw)
        l0 = T.launch_count()
        sim.step(n)
        return sim, T.launch_count() - l0

    ref, l_ref = run(None)
    got, l_got = run(B)
    a, b = _everything(got), _everything(ref)
    _assert_same(a, b, what=case)
    for k, v in ref.check().items():
        assert np.array_equal(got.check()[k], v, equal_nan=True), k
    fc_ref, fc_got = ref.follow_check(), got.follow_check()
    for k in ("ok", "min_gap"):
        assert np.array_equal(fc_got[k], fc_ref[k]), k
        assert np.array_equal(b["gap"][k], fc_ref[k]), k       # running gap = follow_check, radix-sort path
        assert np.array_equal(a["gap"][k], fc_got[k]), k       # and world path
    assert (fc_ref["min_gap"] < 1e29).any() and (fc_ref["min_gap"] == 1e30).any()
    assert l_ref - l_got == n
    bare, _ = run(B, hist=0)
    g = bare.running_follow_check()
    assert np.array_equal(g["min_gap"], fc_ref["min_gap"]) and np.array_equal(g["ok"], fc_ref["ok"])


@pytest.mark.gpu
def test_running_follow_check_without_following_and_worlds_without_following(gpu_trackers):
    """Following never on: 1e30 and ok, before and after steps.  Worlds set with following off: the same launches and
    states as without worlds."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = gpu_trackers[2]
    B, x_init, scen, _c = _platoon(L)
    out = []
    for ws in (None, 4):
        sim = M.BatchedSimulation(T, scen, x_init=x_init, world_size=ws)
        g = sim.running_follow_check()
        assert (g["min_gap"] == 1e30).all() and g["ok"].all()
        l0 = T.launch_count()
        sim.step(50)
        out.append((sim.state(), T.launch_count() - l0))
        g = sim.running_follow_check()
        assert (g["min_gap"] == 1e30).all() and g["ok"].all()
    for a, b in zip(out[0][0], out[1][0]):
        assert np.array_equal(a, b)
    assert out[0][1] == out[1][1]


# --------------------------------------------------------------------------------------------------------------------
# 6. worlds are independent
# --------------------------------------------------------------------------------------------------------------------
PLATOON_RANGE = 40.0


def platoons(L, W, seed=None):
    """W platoons of test_gpu_sim_follow.py's 8 cars on trajectory2 (the front one stops at the light), world w =
    vehicles [8 w, 8 w + 8).  seed: each platoon shifted along the route and spaced and paced differently (else W
    identical platoons)."""
    m, x0, scen, _c = _platoon(L)
    if seed is None:
        return m, np.tile(x0, (W, 1)), scen * W
    rng = np.random.default_rng(seed)
    s = (rng.uniform(200.0, 320.0, W)[:, None] - rng.uniform(8.0, 20.0, W)[:, None] * np.arange(m)).reshape(-1)
    x = np.array([L.get_state(v) for v in s])
    x[:, 4] = np.tile(x0[:, 4], W) + rng.uniform(-1.0, 1.0, W * m)
    return m, x, scen * W


@pytest.mark.gpu
def test_identical_platoons_drive_alike(bulk2):
    """64 identical platoons, 400 steps recorded: without noise every world's drive equals world 0's and a standalone
    platoon's bit for bit (leaders moved by 8 w); with noise, worlds 0, 1, 37 and 63 each equal a standalone platoon
    with first_id = 8 w."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = bulk2
    W, n = 64, 400
    m, x, scen = platoons(L, W)
    B = W * m

    def drive(xi, sc, **kw):
        sim = M.BatchedSimulation(T, sc, x_init=xi, history_steps=n, follow_range=PLATOON_RANGE, **kw)
        sim.step(n)
        return _everything(sim)

    world = drive(x, scen, world_size=m)
    alone = drive(x[:m], scen[:m])
    assert (world["lead"]["lead"] >= 0).any() and (world["steps"] > 0).all()
    for w in range(W):
        sel = slice(w * m, (w + 1) * m)
        _assert_same(_slice(world, sel), alone, shift=w * m, what=f"world {w}")
    world = drive(x, scen, world_size=m, noise=dict(seed=9, **SIGMA))
    for w in (0, 1, 37, 63):
        alone = drive(x[:m], scen[:m], noise=dict(seed=9, first_id=w * m, **SIGMA))
        _assert_same(_slice(world, slice(w * m, (w + 1) * m)), alone, shift=w * m, what=f"noisy world {w}")
    assert not np.array_equal(world["x"][:m], world["x"][m:2 * m])


def _slice(F, sel):
    """The outputs of vehicles sel only."""
    return dict(x=F["x"][sel], steps=F["steps"][sel], uns=F["uns"][sel],
                hist={k: v[:, sel] for k, v in F["hist"].items()}, w=F["w"][:, sel],
                lead={k: v[:, sel] for k, v in F["lead"].items()},
                run={k: v[sel] for k, v in F["run"].items()}, gap={k: v[sel] for k, v in F["gap"].items()})


# --------------------------------------------------------------------------------------------------------------------
# 7. branch_worlds
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_identity_world_branch_changes_nothing(bulk2):
    """64 different platoons, noise, hot start, following on, identity branch at step 37: every output bit for bit;
    launch count = the unbranched run's + the documented branch kernels."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = bulk2
    W, k, n = 64, 37, 300
    m, x, scen = platoons(L, W, seed=1)

    def run(identity):
        sim = M.BatchedSimulation(T, scen, x_init=x, history_steps=n, hot_start=True, follow_range=PLATOON_RANGE,
                                  noise=dict(seed=3, **SIGMA), world_size=m)
        l0 = T.launch_count()
        sim.step(k)
        if identity:
            sim.branch_worlds(np.arange(W))
        sim.step(n - k)
        return _everything(sim), T.launch_count() - l0

    ref, l_ref = run(False)
    got, l_got = run(True)
    _assert_same(got, ref, what="identity")
    assert l_got == l_ref + branch_launches(W * m, n, k) == l_ref + 4


@pytest.mark.gpu
def test_world_branch_with_duplicates_and_drops(bulk2):
    """64 different platoons, following on, noise off, 360 steps recorded, branched at step 60 with a random parent map
    of worlds: right after the branch every vehicle's state, accumulators and histories are its parent's with recorded
    leaders moved into its world, and at the end of the run every output still is."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = bulk2
    W, k, n = 64, 60, 360
    m, x, scen = platoons(L, W, seed=2)
    B = W * m
    pw = np.random.default_rng(5).integers(0, W, W)
    assert len(np.unique(pw)) < W and (pw != np.arange(W)).any()
    parent = (pw[:, None] * m + np.arange(m)).reshape(-1)
    shift = np.arange(B) - parent

    def sim():
        return M.BatchedSimulation(T, scen, x_init=x, history_steps=n, follow_range=PLATOON_RANGE, world_size=m)

    ref = sim()
    ref.step(k)
    ref_k = _everything(ref)
    ref.step(n - k)
    ref_n = _everything(ref)
    assert (ref_k["lead"]["lead"] >= 0).any() and (ref_k["gap"]["min_gap"] < 1e29).any()
    got = sim()
    got.step(k)
    got.branch_worlds(pw)
    _assert_same(_everything(got), ref_k, sel=parent, shift=shift, what="after the branch")
    got.step(n - k)
    _assert_same(_everything(got), ref_n, sel=parent, shift=shift, what="at the end")


@pytest.mark.gpu
def test_world_branch_with_noise_draws_the_copies_own_noise(bulk2):
    """Noise on, branched at step 40: rows before 40 are the parent's; rows from 40 on are sigma z of sim_normals for the
    copy's own id (first_id + b)."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = bulk2
    W, k, n, seed, first_id = 32, 40, 160, 11, 1000
    m, x, scen = platoons(L, W, seed=3)
    B = W * m
    pw = np.random.default_rng(6).integers(0, W, W)
    parent = (pw[:, None] * m + np.arange(m)).reshape(-1)
    kw = dict(x_init=x, follow_range=PLATOON_RANGE, world_size=m, noise=dict(seed=seed, first_id=first_id, **SIGMA))
    ref = M.BatchedSimulation(T, scen, history_steps=k, **kw)
    ref.step(k)
    sim = M.BatchedSimulation(T, scen, history_steps=n, **kw)
    sim.step(k)
    sim.branch_worlds(pw)
    sim.step(n - k)
    w, steps = _w12(sim.noise_history()), sim.state()[1]
    assert np.array_equal(w[:k], _w12(ref.noise_history())[:, parent], equal_nan=True)
    t = np.arange(k, n)
    live = t[:, None] < steps[None, :]
    z = sim_normals(seed, first_id + np.arange(B)[None, :], t[:, None])
    assert live.any() and np.abs(w[k:n][live] / SIGMA12 - z[live]).max() <= 1e-12
    assert np.isnan(w[k:n][~live]).all()


@pytest.mark.gpu
def test_world_branch_refusals_change_nothing(bulk2):
    """branch_worlds without worlds (Python and ABI), a parent out of range and bad world sizes through the ABI, and
    mpcb_sim_branch with following on are refused and leave the simulation as it was."""
    import safe_autonomous_driving_mpc_b200 as M
    L, T = bulk2
    W = 8
    m, x, scen = platoons(L, W, seed=4)
    sim = M.BatchedSimulation(T, scen, x_init=x, history_steps=40, follow_range=PLATOON_RANGE)
    sim.step(20)
    before = _everything(sim)
    dp = lambda a: a.ctypes.data_as(C.c_void_p)
    pw = np.arange(W, dtype=np.int32)[::-1].copy()
    with pytest.raises(ValueError):
        sim.branch_worlds(pw)
    assert sim._lib.mpcb_sim_branch_worlds(sim._h, dp(pw), None) == -1
    for bad in (3, 5, 1025, -1, 128):
        assert sim._lib.mpcb_sim_set_worlds(sim._h, bad) == -1
    sim.set_worlds(m)
    bad = pw.copy()
    bad[-1] = W
    assert sim._lib.mpcb_sim_branch_worlds(sim._h, dp(bad), None) == -1
    bad[-1] = -1
    assert sim._lib.mpcb_sim_branch_worlds(sim._h, dp(bad), None) == -1
    with pytest.raises(M._lib.MpcbError):                  # vehicle branching with following on, worlds or not
        sim.branch(np.arange(W * m))
    _assert_same(_everything(sim), before, what="refused")
    sim.set_worlds(None)
    assert sim.W == 1 and sim.world_size is None


# --------------------------------------------------------------------------------------------------------------------
# 8. the estimator on the device
# --------------------------------------------------------------------------------------------------------------------
# Tight noisy platoons: 8 cars on trajectory2, NEAR_SPACING m apart, the front one stopping at the light, noise at
# NEAR_SCALE x the base level of tools/gpu_sim_noise.py; drives cut at NEAR_STEPS steps.
BASE = dict(meas=[0.05, 0.02, 0.005, 0.001, 0.05], act=[0.02, 0.1], proc=[0.01, 0.005, 0.002, 0.0005, 0.02])
# (at twice the base level crude sees ~0.5 % of worlds near-miss within 400 steps, at 4x half of them)
NEAR_SPACING, NEAR_SCALE, NEAR_STEPS, NEAR_CAP, NEAR_LAM = 7.0, 2.0, 400, 4.0, 2.0


def tight_platoons(L, W):
    m, x0, scen, _c = _platoon(L)
    s = 300.0 - NEAR_SPACING * np.arange(m)
    x = np.array([L.get_state(v) for v in s])
    x[:, 4] = x0[:, 4]
    return m, np.tile(x, (W, 1)), scen * W


def near_noise(seed, scale=NEAR_SCALE):
    return dict(seed=seed, **{k: [scale * v for v in vs] for k, vs in BASE.items()})


@pytest.mark.gpu
def test_near_miss_estimator_on_the_device(gpu_trackers):
    """lam = 0 is the crude fraction of worlds with a near miss, bit for bit.  On the tight noisy platoons (crude sees
    1e-3 .. 1e-2 of worlds), the mean of 8 splitting estimates on 1,024 worlds agrees with a crude estimate on 8,192
    worlds within 4 combined standard errors."""
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200.rare_events import near_miss_probability
    L, T = gpu_trackers[2]
    m, x, scen = tight_platoons(L, 1024)

    def sim(W, seed):
        return M.BatchedSimulation(T, scen[:m] * W, x_init=np.tile(x[:m], (W, 1)), follow_range=PLATOON_RANGE,
                                   noise=near_noise(seed), world_size=m)

    s = sim(1024, 90)
    res = near_miss_probability(s, 0.0, 100, seed=0, gap_cap=NEAR_CAP, max_steps=NEAR_STEPS)
    assert res["resamplings"] == 0 and res["steps"] == NEAR_STEPS
    assert res["p"] == float(np.mean(~s.running_follow_check()["ok"].reshape(1024, m).all(axis=1)))
    crude = sim(8192, 91)
    crude.step(NEAR_STEPS)
    fail = ~crude.running_follow_check()["ok"].reshape(8192, m).all(axis=1)
    p_crude, se_crude = fail.mean(), math.sqrt(fail.mean() * (1.0 - fail.mean()) / fail.size)
    assert 1e-3 <= p_crude <= 1e-2, p_crude
    ps = []
    for r in range(8):
        res = near_miss_probability(sim(1024, 100 + r), NEAR_LAM, 50, seed=r, gap_cap=NEAR_CAP, max_steps=NEAR_STEPS)
        assert res["resamplings"] >= 3
        ps.append(res["p"])
    se = np.std(ps, ddof=1) / math.sqrt(len(ps))
    print(f"\ncrude {p_crude:.3e} +- {se_crude:.1e}, splitting {np.mean(ps):.3e} +- {se:.1e}: {ps}")
    assert abs(np.mean(ps) - p_crude) <= 4.0 * math.hypot(se, se_crude), (ps, p_crude, se_crude)
