"""The device's reference-table lookups on routes other than the three committed ones.

The committed routes (data/trajectory{1,2,3}.npz) have at most 0.31 knots per lookup bucket, no repaired knots, start
at s = 0 and define their controls on K - 1 knots, so the bucket index of the cold lookups never has to walk, the hinted
walk never gives up, and Ku = K, Ku < K - 1 and two- or three-knot tables never reach the device.  The table families
below do.  Each is built by a deterministic numpy generator from a committed route (or from nothing, for the minimal
tables) and checked:

  * without a GPU: the generators yield what they claim (knot counts, control knots, smallest gap, knots per bucket
    as the device's bucket index sees them), the same-function families are the base route's functions, and the
    injected-position rollout used below equals the oracle's predict / cost bit for bit;
  * function level: BatchedTracker.eval_batch (warm start, rollout, cost, constraint rows, linearisation) against the
    oracle, on Monte-Carlo problems and on knot probes (positions on, just beside and between knots and bucket edges);
  * metamorphic: a refined, clustered or shifted copy of a route gives the base route's answers, in every execution
    shape, below and above one wave of the first pass;
  * solves judged by the oracle's rows and a KKT certificate (tests/kkt.py);
  * the planner evaluator against the oracle and against the base route;
  * closed-loop fleets replayed against the oracle's plant step;
  * sixteen routes on one handle, bit for bit against single-route handles, and a following fleet over them.

Positions propagated through the rollout differ from the oracle's by an ulp (the device contracts s + h v into an FMA);
on a table whose slopes reach 1e4 that ulp becomes a visible difference in the looked-up value.  So rolled-out values
are compared with an oracle rollout that looks up at the device's own positions (``rollout_at``); the positions
themselves are compared with the oracle's to a few ulp."""
import functools

import numpy as np
import pytest

from closed_loop_oracle import DT, leaders, plant_step
from conftest import VARIANTS, golden, traj_path
from oracle import planner_port as Q
from oracle import sqp_admm_model as A
from oracle import tracker_port as P

FN_TOL = 1e-12
LUT_N = 4096                       # buckets of the device's cold-lookup index (upload_table, mpcb_api.cu)
WAVE = 148 * 2 * 128               # problems of one wave of the first pass on a B200 (148 SMs x 2 CTAs x 128)
SHIFT_UP, SHIFT_DOWN = 10000.0, -700.0


# --------------------------------------------------------------------------------------------------------------------
# table families (numpy only)
# --------------------------------------------------------------------------------------------------------------------
def _base(i):
    z = np.load(traj_path(i))
    return np.ascontiguousarray(z["X"], dtype=np.float64), np.ascontiguousarray(z["U"], dtype=np.float64)


def control_fn(tab, s):
    """The base route's control function at s, linear extrapolation included and WITHOUT the s >= s_max -> 0 rule of
    get_control: what a refined table must store at its last knot so that it interpolates the same function."""
    s = np.asarray(s, dtype=np.float64)
    su = tab.s[: tab.Ku]
    i = np.clip(np.searchsorted(su, s, side="left"), 1, tab.Ku - 1)
    lo = i - 1
    x_lo, x_hi = su[lo], su[i]
    wl = (s - x_lo) / (x_hi - x_lo)
    wr = (x_hi - s) / (x_hi - x_lo)
    Y = tab.U[: tab.Ku]
    return wl[..., None] * Y[i] + wr[..., None] * Y[lo]


def _same_function(base_i, s_new):
    """Table on the knots s_new (a superset of the base route's knots) carrying the base route's state and control
    functions: rows from the base interpolator, a control row at every knot (Ku = K)."""
    X0, U0 = _base(base_i)
    tab = P.RefTable(X0, U0)
    assert np.all(np.isin(tab.s, s_new))
    X = np.empty((len(s_new), 5))
    X[:, 0] = s_new
    X[:, 1:] = A.lookup(tab, s_new)[0]
    return X, control_fn(tab, s_new)


def _split(s, pieces):
    """Every segment [s[i-1], s[i]] split evenly into pieces[i-1] parts."""
    out = [s[:1]]
    for a, b, n in zip(s[:-1], s[1:], pieces):
        t = np.arange(1, n + 1) / n
        seg = a + (b - a) * t
        seg[-1] = b
        out.append(seg)
    return np.concatenate(out)


def _refined():
    s = P.RefTable(*_base(3)).s
    return _same_function(3, _split(s, np.full(len(s) - 1, 4)))


def _dense(base_i=3):
    s = P.RefTable(*_base(base_i)).s
    return _same_function(base_i, _split(s, np.ceil(np.diff(s) / 0.03).astype(int)))


def _clustered():
    """20 bursts of 200 knots within 0.3 m (about one bucket) on trajectory2: ten inside segments, ten across bucket
    edges, each clear of the base knots by 5 mm."""
    s = P.RefTable(*_base(2)).s
    scale = LUT_N / (s[-1] - s[0])
    rng = np.random.default_rng(3)
    width, margin = 0.3, 5e-3
    bursts = []

    def clear(lo, hi):
        return not np.any((s > lo - margin) & (s < hi + margin)) and all(hi < a - margin or lo > b + margin
                                                                          for a, b in bursts)
    while len(bursts) < 10:                            # inside segments
        i = int(rng.integers(1, len(s)))
        if s[i] - s[i - 1] < 4 * width:
            continue
        lo = s[i - 1] + rng.uniform(margin + 0.01, s[i] - s[i - 1] - width - margin - 0.01)
        if clear(lo, lo + width):
            bursts.append((lo, lo + width))
    while len(bursts) < 20:                            # straddling a bucket edge s0 + b / scale
        b = int(rng.integers(1, LUT_N))
        edge = s[0] + b / scale
        lo = edge - width * rng.uniform(0.2, 0.8)
        if clear(lo, lo + width):
            bursts.append((lo, lo + width))
    new = np.concatenate([lo + (hi - lo) * np.arange(200) / 199 for lo, hi in bursts])
    return _same_function(2, np.union1d(s, new))


def _ku_short():
    X, U = _base(1)
    return X, U[: len(X) - 20]


def _shifted(off):
    X, U = _base(2)
    X = X.copy()
    X[:, 0] += off
    return X, U


REPAIR_SEED = 11


def _repaired(steep):
    """trajectory2 with 30 knots repeated 1-5 times and one run of decreasing s: mpcb_table_create and the reference's
    loader spread them 1e-5 m apart.  steep: the repeated rows step by (0.05, 0.02, 0.01, 0.5) in (d, o, k, v)."""
    X, U = _base(2)
    rng = np.random.default_rng(REPAIR_SEED)
    K = len(X)
    at = np.sort(rng.choice(np.arange(5, K - 5), 31, replace=False))
    reps = rng.integers(1, 6, 31)
    step = np.array([0.0, 0.05, 0.02, 0.01, 0.5]) if steep else np.zeros(5)
    rows, urows = [], []
    for i in range(K):
        rows.append(X[i])
        if i < K - 1:
            urows.append(U[i])
        if i in at:
            j = int(np.searchsorted(at, i))
            for m in range(1, int(reps[j]) + 1):
                r = X[i] + m * step
                if j == 0:                                # the run of decreasing s
                    r = r.copy()
                    r[0] = X[i, 0] - 0.25 * m
                rows.append(r)
                urows.append(U[min(i, K - 2)])
    X2 = np.array(rows)
    return X2, np.array(urows[: len(X2) - 1])


def _straight(nu):
    X = np.array([[0.0, 0.0, 0.0, 0.0, 8.0], [400.0, 0.0, 0.0, 0.0, 8.0]])
    U = np.array([[0.01, 0.5], [-0.02, -0.3], [0.03, 1.0], [0.0, 0.2], [0.01, -0.1]])[:nu]
    return X, U


def _arc(nu):
    X = np.array([[0.0, 0.0, 0.0, 0.02, 8.0], [150.0, 0.0, 0.0, 0.02, 8.0], [300.0, 0.0, 0.0, 0.02, 8.0]])
    U = np.array([[0.01, 0.5], [-0.02, -0.3], [0.03, 1.0], [0.0, 0.2], [0.01, -0.1]])[:nu]
    return X, U


class Family:
    def __init__(self, name, make, base=None, off=0.0, same=False, steep=False, K=None, Ku=None, gap=None):
        self.name, self.make, self.base, self.off, self.same, self.steep = name, make, base, off, same, steep
        self.want = dict(K=K, Ku=Ku, gap=gap)

    @functools.cached_property
    def XU(self):
        return self.make()

    @functools.cached_property
    def tab(self):
        return P.RefTable(*self.XU)

    @functools.cached_property
    def base_tab(self):
        return P.RefTable(*_base(self.base)) if self.base else None


# same: the state and control functions are the base route's (shifted by `off`)
FAMILIES = {f.name: f for f in [
    Family("refined", _refined, base=3, same=True, K=4 * 1258 + 1, Ku=4 * 1258 + 1),
    Family("dense", _dense, base=3, same=True, K=115895, Ku=115895),
    Family("clustered", _clustered, base=2, same=True, K=481 + 20 * 200, Ku=481 + 20 * 200),
    Family("ku_short", _ku_short, base=1, K=115, Ku=95),
    Family("shifted_up", lambda: _shifted(SHIFT_UP), base=2, off=SHIFT_UP, same=True, K=481, Ku=480),
    Family("shifted_down", lambda: _shifted(SHIFT_DOWN), base=2, off=SHIFT_DOWN, same=True, K=481, Ku=480),
    Family("repaired_equal", lambda: _repaired(False), base=2, gap=1e-5),
    Family("repaired_steep", lambda: _repaired(True), base=2, steep=True, gap=1e-5),
    Family("straight_k2", lambda: _straight(2), K=2, Ku=2),
    Family("arc_k3_u2", lambda: _arc(2), K=3, Ku=2),
    Family("arc_k3_u3", lambda: _arc(3), K=3, Ku=3),
    Family("arc_k3_u5", lambda: _arc(5), K=3, Ku=3),
]}
SAME = [n for n, f in FAMILIES.items() if f.same]
NOT_STEEP = [n for n, f in FAMILIES.items() if not f.steep]


def lut_of(s):
    """The bucket index exactly as upload_table builds it: lut[b] = searchsorted-left of the bucket's left edge, clipped
    to [1, K - 1]; also the edges and the scale."""
    K = len(s)
    span = s[-1] - s[0]
    scale = LUT_N / span if span > 0 else 0.0
    edges = s[0] + (np.arange(LUT_N) / scale if scale > 0 else np.zeros(LUT_N))
    lut = np.clip(np.searchsorted(s, edges, side="left"), 1, K - 1)
    return lut, edges, scale


def knots_per_bucket(s):
    lut, _, _ = lut_of(s)
    return int(np.max(np.diff(np.append(lut, len(s) - 1))))


def knot_probes(f, max_own=6000):
    """Positions where segment choices go wrong: the knots where the slope changes (the base route's, shifted; a small
    table's own), their neighbours one ulp up and down, before the first knot, at and around s_max, and a sample of
    the bucket edges as upload_table computes them."""
    s = f.tab.s
    if f.same and f.base:
        pick = f.base_tab.s + f.off
    else:
        pick = s if len(s) <= max_own else s[:: len(s) // max_own + 1]
    _, edges, _ = lut_of(s)
    ends = [s[0] - 1.0, f.tab.s_max, np.nextafter(f.tab.s_max, -np.inf), f.tab.s_max + 1.0]
    pts = np.concatenate([pick, np.nextafter(pick, np.inf), np.nextafter(pick, -np.inf), ends, edges[::8], edges[-3:]])
    return np.unique(pts)


def probe_problems(f):
    """x0 = (s, d, o, k, 0) with U = 0: all six lookups of a rollout (and the warm start's five) happen at exactly s."""
    s = knot_probes(f)
    B = len(s)
    x0 = np.zeros((B, 5))
    x0[:, 0] = s
    x0[:, 1], x0[:, 2], x0[:, 3] = 0.05, -0.01, 0.004
    return x0, np.zeros((B, 2, 2)), np.zeros(B, np.int32), np.zeros((B, 10))


def mc_problems(f, B, seed=P.MC_SEED):
    """Monte-Carlo problems (oracle generator; for a shifted route drawn on the base route and offset) and controls
    around the clipped warm start."""
    tab = f.base_tab if f.off else f.tab
    x0, obs, n = P.monte_carlo_problems(tab, B, seed)
    x0 = x0.copy()
    obs = obs.copy()
    x0[:, 0] += f.off
    for k in range(2):
        obs[:, k, 0] = np.where(n > k, obs[:, k, 0] + f.off, obs[:, k, 0])
    rng = np.random.default_rng(seed + 1)
    U = A.warm_start(f.tab, x0, obs, n) + rng.normal(0.0, 0.2, (B, 10))
    return x0, obs, n, U


# --------------------------------------------------------------------------------------------------------------------
# oracle rollout at given positions
# --------------------------------------------------------------------------------------------------------------------
def rollout_at(tab, x0, U, spos):
    """predict / cost / constraints_wrapper (trajectory_tracking.py:87-209) for a batch, in the reference's operation
    order, except that the positions are spos [B,6] instead of s + DT v: every table lookup of step j happens at
    spos[:, j].  With the oracle's own positions this IS the oracle (checked bit for bit below).
    Returns X [B,6,5], cost [B], cons [B,45] (NaN-padded like the device's)."""
    B = len(x0)
    Um = np.asarray(U).reshape(B, 5, 2)
    X = np.zeros((B, 6, 5))
    X[:, 0] = x0
    X[:, 0, 0] = spos[:, 0]
    for j in range(5):
        d, o, k, v = X[:, j, 1], X[:, j, 2], X[:, j, 3], X[:, j, 4]
        kap = A.lookup(tab, spos[:, j])[0][:, 2]
        X[:, j + 1, 0] = spos[:, j + 1]
        X[:, j + 1, 1] = d + DT * (v * o)
        X[:, j + 1, 2] = o + DT * (v * (k - kap))
        X[:, j + 1, 3] = k + DT * Um[:, j, 0]
        X[:, j + 1, 4] = v + DT * Um[:, j, 1]
    cost = np.zeros(B)
    for j in range(1, 6):
        r = A.lookup(tab, spos[:, j])[0]
        cost += P.W_D * (X[:, j, 1] - r[:, 0]) ** 2
        cost += P.W_O * (X[:, j, 2] - r[:, 1]) ** 2
        cost += P.W_V * (X[:, j, 4] - r[:, 3]) ** 2
    for j in range(5):
        cost += P.W_U1 * Um[:, j, 0] ** 2
        cost += P.W_U2 * Um[:, j, 1] ** 2
    return X, cost


def cons_of(X, obs, n):
    """constraints_wrapper rows (trajectory_tracking.py:164-209) from a rollout, NaN-padded to 45."""
    B = len(X)
    c = np.full((B, 45), np.nan)
    row = np.zeros(B, np.int64)
    ar = np.arange(B)
    sld = P.LANE_WIDTH / 2.0 - P.VEHICLE_RADIUS - P.SAFE_LANE_MARGIN
    for j in range(1, 6):
        s, d, o, v = X[:, j, 0], X[:, j, 1], X[:, j, 2], X[:, j, 4]
        for al in (0.0, P.WHEELBASE / 2.0, P.WHEELBASE):
            val = d if al == 0.0 else d + al * o
            c[ar, row] = sld - val
            c[ar, row + 1] = val + sld
            row = row + 2
        for k in range(2):
            on = n > k
            gap = (obs[:, k, 0] + obs[:, k, 1] * (j * DT)) - s
            c[ar[on], row[on]] = (gap - np.maximum(P.OBS_SAFETY_DIST, v * P.MAX_TIME_2_OBS))[on]
            row = row + on
        c[ar, row] = v
        row = row + 1
    return c


def cons_tol(f):
    """Obstacle rows are differences of positions (s_obs + v t - s): beside FN_TOL, a few ulp of the largest position
    on a route far from s = 0 (at 1e4 m one ulp is 1.8e-12)."""
    return FN_TOL + (4.0 * np.spacing(max(abs(f.tab.s[0]), abs(f.tab.s_max))) if f.off else 0.0)


def shift_tol(f):
    """A shifted route equals its base route only to the rounding of the offset: its knots and the positions looked up
    on it each move by up to a few ulp of the offset (1.8e-12 at 1e4 m), and the table's slopes (up to 6.7 per metre on
    trajectory2) and the cost weights magnify that.  The same bound as the oracle-level check of the same-function
    families; FN_TOL on every route that is not shifted."""
    return FN_TOL * max(1.0, abs(f.off))


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    m = ~(np.isnan(a) & np.isnan(b))
    return float(np.max(np.abs(a[m] - b[m]) / np.maximum(1.0, np.abs(b[m])), initial=0.0))


# --------------------------------------------------------------------------------------------------------------------
# 8. CPU: the generators and the rollout helper
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(FAMILIES))
def test_generator_yields_what_it_claims(name):
    import safe_autonomous_driving_mpc_b200 as M
    f = FAMILIES[name]
    tab = f.tab
    L = M.TrajectoryLoader(*f.XU)
    assert L.s_max == tab.s_max
    if f.want["K"] is not None:
        assert tab.K == f.want["K"] and tab.Ku == f.want["Ku"], (tab.K, tab.Ku)
    gap = np.diff(tab.s).min()
    assert gap > 0.0
    if f.same:
        assert gap >= 1e-3, gap
    if f.want["gap"] is not None:
        assert gap == pytest.approx(f.want["gap"], rel=1e-6)
        assert len(f.XU[0]) - 481 >= 30 + 30                           # 30 repeated knots (and one decreasing run)
        assert np.any(np.diff(f.XU[0][:, 0]) < 0)
    kpb = knots_per_bucket(tab.s)
    # most knots between two bucket edges: beyond 6 the cold lookup's walk gives up and searches (dense, clustered)
    claims = dict(refined=(7, 16), dense=(25, 35), clustered=(190, 210), repaired_equal=(5, 6), repaired_steep=(5, 6))
    assert claims.get(name, (0, 3))[0] <= kpb <= claims.get(name, (0, 3))[1], kpb
    if name == "clustered":                                           # beside near-empty buckets
        assert np.sum(np.diff(lut_of(tab.s)[0]) == 0) > LUT_N // 2
    # the host interpolators of the library agree with the oracle on the family (positions at and around the probes)
    for q in knot_probes(f)[:: max(1, len(knot_probes(f)) // 200)]:
        np.testing.assert_allclose(L.get_state(q), tab.get_state(q), rtol=0, atol=1e-12 * max(1.0, abs(q)))
        np.testing.assert_allclose(L.get_control(q), tab.get_control(q), rtol=0, atol=1e-11)


@pytest.mark.parametrize("name", SAME)
def test_same_function_families_are_the_base_functions(name):
    """Oracle get_state / get_control on the family equal the base route's at 10^4 random points and at every probe, to
    1e-12.  A shifted family is looked up at s + offset and the base route at (s + offset) - offset: the rounding of
    the offset moves the point by up to an ulp of the offset, which the bound allows for."""
    f = FAMILIES[name]
    b = f.base_tab
    rng = np.random.default_rng(2)
    s = np.concatenate([rng.uniform(b.s[0] - 5.0, b.s_max + 5.0, 10000) + f.off, knot_probes(f)])
    tol = shift_tol(f)
    s = s[(s < f.tab.s_max) == (s - f.off < b.s_max)]      # both on the same side of the s >= s_max rule
    assert np.max(np.abs(A.lookup(f.tab, s)[0] - A.lookup(b, s - f.off)[0])) <= tol
    assert np.max(np.abs(A.lookup_control(f.tab, s) - A.lookup_control(b, s - f.off))) <= tol
    if not f.off:
        # a control row at every knot; the last one is the base function's extrapolated value (get_control gives 0)
        assert f.tab.Ku == f.tab.K
        assert np.array_equal(f.tab.U[-1], control_fn(b, f.tab.s[-1]))


@pytest.mark.parametrize("i", [1, 2, 3])
def test_rollout_helper_is_the_oracle_at_its_own_positions(i, port_tables):
    tab = port_tables[i]
    x0, obs, n = P.monte_carlo_problems(tab, 64)
    U = np.random.default_rng(i).uniform(-1.0, 1.0, (64, 10))
    want = np.array([P.predict(tab, x0[b], U[b]) for b in range(64)])
    X, cost = rollout_at(tab, x0, U, want[:, :, 0])
    assert np.array_equal(X, want)
    assert np.array_equal(cost, [P.cost(tab, U[b], x0[b]) for b in range(64)])
    c = cons_of(X, obs, n)
    for b in range(64):
        cb = P.constraint_values(tab, U[b], x0[b], [tuple(o) for o in obs[b, : n[b]]])
        assert np.array_equal(c[b, : len(cb)], cb) and np.all(np.isnan(c[b, len(cb):]))


# --------------------------------------------------------------------------------------------------------------------
# GPU fixtures
# --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def loaders():
    import safe_autonomous_driving_mpc_b200 as M
    out = {n: M.TrajectoryLoader(*f.XU) for n, f in FAMILIES.items()}
    out["dense_traj2"] = M.TrajectoryLoader(*_dense(2))
    for i in (1, 2, 3):
        out[f"traj{i}"] = M.TrajectoryLoader(traj_path(i))
    return out


@pytest.fixture(scope="module")
def trackers(loaders):
    """Lazily built trackers: trackers(name, variant)."""
    import safe_autonomous_driving_mpc_b200 as M
    cache = {}

    def get(name, variant="default"):
        key = (name, variant)
        if key not in cache:
            kw = dict(VARIANTS, fast0=dict(fast_pass=0))[variant]
            cache[key] = M.BatchedTracker(loaders[name], **kw)
        return cache[key]
    return get


def _base_name(f):
    return f"traj{f.base}"


# --------------------------------------------------------------------------------------------------------------------
# 2. function level against the oracle
# --------------------------------------------------------------------------------------------------------------------
def _lin_ref(tab, x0, U, obs, n):
    asm = A.assemble(tab, x0, U)
    qp = A.build_qp(asm, x0, U, obs, n)
    il, jl = np.tril_indices(10)                          # row-major lower triangle: (0,0), (1,0), (1,1), ...
    H = np.asarray(qp["P"])[:, il, jl]
    return asm, H, np.asarray(qp["q"])


def _check_lin(r, tab, x0, U, obs, n, what):
    asm, H, q = _lin_ref(tab, x0, U, obs, n)
    lin = r["lin"]
    assert np.max(np.abs(lin[:, :55] - H)) <= 1e-9 * max(1.0, np.abs(H).max()), what
    assert np.max(np.abs(lin[:, 55:65] - q)) <= 1e-9 * max(1.0, np.abs(q).max()), what
    D, O = asm["dX"][:, 2:6, 1], asm["dX"][:, 2:6, 2]
    assert np.max(np.abs(lin[:, 65:105].reshape(-1, 4, 10) - D)) <= 1e-9 * max(1.0, np.abs(D).max()), what
    assert np.max(np.abs(lin[:, 105:145].reshape(-1, 4, 10) - O)) <= 1e-9 * max(1.0, np.abs(O).max()), what


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FAMILIES))
def test_eval_batch_against_the_oracle(name, trackers):
    f = FAMILIES[name]
    tab = f.tab
    T = trackers(name)
    sets = dict(mc=mc_problems(f, 4096), probes=probe_problems(f))
    for what, (x0, obs, n, U) in sets.items():
        r = T.eval_batch(x0, U, obs, n)
        # warm start: the reference's (unclipped)
        warm = np.array([P.warm_start(tab, x0[b], [tuple(o) for o in obs[b, : n[b]]]) for b in range(len(x0))])
        bad = np.abs(r["warm"] - warm).max(axis=1) > FN_TOL
        assert not bad.any(), (what, np.flatnonzero(bad)[:5], x0[bad][:3, 0])
        # positions: the oracle's to a few ulp (FMA contraction of s + h v)
        Xo, cost_o = rollout_at(tab, x0, U, A.assemble(tab, x0, U)["X"][:, :, 0])
        sp = r["Xpred"][:, :, 0]
        assert np.all(np.abs(sp - Xo[:, :, 0]) <= 1e-14 * np.maximum(1.0, np.abs(Xo[:, :, 0]))), what
        # everything else: the oracle at the device's own positions
        Xd, cost_d = rollout_at(tab, x0, U, sp)
        assert rel(r["Xpred"], Xd) <= FN_TOL, (what, rel(r["Xpred"], Xd))
        assert rel(r["cost"], cost_d) <= FN_TOL, (what, rel(r["cost"], cost_d))
        cd = cons_of(Xd, obs, n)
        assert np.array_equal(np.isnan(r["cons"]), np.isnan(cd))
        assert rel(r["cons"], cd) <= cons_tol(f), what
        if not f.steep:                                    # and the oracle itself
            assert rel(r["Xpred"], Xo) <= FN_TOL and rel(r["cost"], cost_o) <= FN_TOL, what
            assert rel(r["cons"], cons_of(Xo, obs, n)) <= cons_tol(f), what
        if not f.steep or what == "probes":
            _check_lin(r, tab, x0, U, obs, n, what)


# --------------------------------------------------------------------------------------------------------------------
# 3. metamorphic: the same function gives the same answers
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", SAME)
def test_eval_batch_equals_the_base_route(name, trackers):
    f = FAMILIES[name]
    x0, obs, n, U = mc_problems(f, 4096)
    got = trackers(name).eval_batch(x0, U, obs, n)
    xb, ob = x0.copy(), obs.copy()
    xb[:, 0] -= f.off
    for k in range(2):
        ob[:, k, 0] = np.where(n > k, obs[:, k, 0] - f.off, obs[:, k, 0])
    want = trackers(_base_name(f)).eval_batch(xb, U, ob, n)
    gx = got["Xpred"].copy()
    gx[:, :, 0] -= f.off
    assert np.all(np.abs(got["Xpred"][:, :, 0] - f.off - want["Xpred"][:, :, 0])
                  <= FN_TOL * np.maximum(1.0, np.abs(got["Xpred"][:, :, 0])))
    assert rel(gx[:, :, 1:], want["Xpred"][:, :, 1:]) <= shift_tol(f), rel(gx[:, :, 1:], want["Xpred"][:, :, 1:])
    for k in ("cost", "cons", "warm"):
        assert rel(got[k], want[k]) <= shift_tol(f), (k, rel(got[k], want[k]))
    assert np.max(np.abs(got["lin"] - want["lin"])) <= 1e-9 * max(1.0, np.abs(want["lin"]).max())


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS) + ["fast0"])
@pytest.mark.parametrize("B", [2000, 65536])
@pytest.mark.parametrize("name", SAME)
def test_solves_equal_the_base_route(name, B, variant, trackers):
    f = FAMILIES[name]
    if B == 65536:
        assert B > WAVE
    x0, obs, n, _ = mc_problems(f, B)
    got = {k: v.copy() for k, v in trackers(name, variant).solve_batch_host(x0, obs, n, pinned_out=False).items()}
    xb, ob = x0.copy(), obs.copy()
    xb[:, 0] -= f.off
    for k in range(2):
        ob[:, k, 0] = np.where(n > k, obs[:, k, 0] - f.off, obs[:, k, 0])
    want = trackers(_base_name(f), variant).solve_batch_host(xb, ob, n, pinned_out=False)
    agree = got["status"] == want["status"]
    assert agree.mean() >= 0.999, agree.mean()
    ok = agree & (want["status"] == 0)
    assert ok.mean() > 0.8
    assert np.abs(got["U"] - want["U"])[ok].max() <= 1e-6


# --------------------------------------------------------------------------------------------------------------------
# 4. solves judged by the oracle only
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["default", "bulk"])
@pytest.mark.parametrize("name", [n for n in FAMILIES if not FAMILIES[n].steep])
def test_solves_judged_by_the_oracle(name, variant, trackers):
    import kkt
    f = FAMILIES[name]
    tab = f.tab
    B = 8192
    x0, obs, n, _ = mc_problems(f, B)
    r = {k: v.copy() for k, v in trackers(name, variant).solve_batch_host(x0, obs, n, pinned_out=False).items()}
    U = r["U"].reshape(B, 10)
    c, G, asm, G2, kink = kkt.reference_rows(tab, x0, U, obs, n, with_kinks=True)
    cmin = np.nanmin(c, axis=1)
    ok = r["status"] == 0
    assert ok.mean() > 0.5
    assert cmin[ok].min() >= -1e-6, f"a SOLVED problem violates a reference row by {cmin[ok].min():.3e}"
    assert np.all(U >= np.tile(P.U_MIN, 5) - 1e-12) and np.all(U <= np.tile(P.U_MAX, 5) + 1e-12)
    bad = r["status"] == 2
    assert np.all(cmin[bad] < -1e-6), "an INFEASIBLE flag on a point that satisfies every reference row"
    assert np.max(np.abs(U[ok, 8])) < 1e-6
    assert np.max(np.abs(asm["cost"] - r["obj"]) / np.maximum(1.0, np.abs(asm["cost"]))) < 1e-12
    assert np.max(np.abs(cmin - r["cmin"]) / np.maximum(1.0, np.abs(cmin))) < 1e-10
    bits = ((r["active"][:, None] >> np.arange(45, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(bool)
    valid = ~np.isnan(c)
    assert np.all(bits[valid & (c <= 1e-6 - 1e-9)]) and not np.any(bits[valid & (c > 1e-6 + 1e-9)])
    assert not np.any(bits[~valid])
    g = kkt.cost_gradient(asm, U)
    res, nact = kkt.kkt_residual(c[ok], G[ok], g[ok], U[ok], G2=G2[ok], kink=kink[ok])
    assert res.max() <= 1e-5, f"KKT residual {res.max():.3e} at solved problem {np.where(ok)[0][np.argmax(res)]}"


# --------------------------------------------------------------------------------------------------------------------
# 5. planner evaluator
# --------------------------------------------------------------------------------------------------------------------
def _probe_windows(f, N=16):
    """Windows whose nodes sit on the knot probes (sorted, N + 1 nodes per window)."""
    s = knot_probes(f)
    s = s[: (len(s) // (N + 1)) * (N + 1)].reshape(-1, N + 1)
    W = len(s)
    X = np.zeros((W, N + 1, 5))
    X[..., 0] = s
    X[..., 1], X[..., 2], X[..., 3], X[..., 4] = 0.05, -0.01, 0.004, 5.0
    Uw = np.tile([0.01, 0.3], (W, N, 1))
    return np.concatenate([X.reshape(W, -1), Uw.reshape(W, -1), np.zeros((W, N))], axis=1), N


def _golden_windows(f):
    g = golden(f"planner_traj{f.base}")
    z = g["z"].copy()
    N = int(g["N"])
    z[:, 0: 5 * (N + 1): 5] += f.off
    return z, N


@pytest.mark.gpu
@pytest.mark.parametrize("name", NOT_STEEP)
def test_planner_evaluator_against_the_oracle(name, trackers):
    import safe_autonomous_driving_mpc_b200 as M
    f = FAMILIES[name]
    tab = f.tab
    sets = [_probe_windows(f)] + ([_golden_windows(f)] if f.base else [])
    rng = np.random.default_rng(4)
    for z, N in sets:
        E = M.PlannerEvaluator(trackers(name), N=N)
        r = E.evaluate_host(z, want_jac=True)
        d_ref = np.array([Q.defects(tab, w, N) for w in z])
        assert rel(r["defect"], d_ref) <= FN_TOL, rel(r["defect"], d_ref)
        for w in rng.choice(len(z), min(len(z), 24), replace=False):
            X, Uw, _ = Q.unpack(z[w], N)
            for k in rng.choice(N, min(N, 4), replace=False):
                J = Q.hs_defect_jac(tab, X[k], X[k + 1], Uw[k])
                assert np.all(np.abs(r["jac"][w, k] - J) <= 1e-11 * np.maximum(1.0, np.abs(J))), (w, k)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["refined", "dense", "clustered"])
def test_planner_whole_route_equals_the_base_route(name, trackers):
    """The whole base trajectory as one window (sign +1), on the refined table and on the base route: defects to 1e-12,
    Jacobian and Lagrangian-Hessian blocks to 1e-9 relative."""
    import safe_autonomous_driving_mpc_b200 as M
    f = FAMILIES[name]
    z0 = np.load(traj_path(f.base))
    N = len(z0["U"])
    lam = np.random.default_rng(7).normal(size=(1, N, 5))
    out = []
    for T in (trackers(name), trackers(_base_name(f))):
        E = M.PlannerEvaluator(T, N=N, simpson_sign=+1)
        out.append(E.evaluate_host(E.pack(z0["X"], z0["U"], z0["S"]), lam=lam, want_jac=True, want_hess=True))
    got, want = out
    assert rel(got["defect"], want["defect"]) <= FN_TOL
    for k in ("jac", "hess"):
        assert np.all(np.abs(got[k] - want[k]) <= 1e-9 * np.maximum(1.0, np.abs(want[k]))), k


# --------------------------------------------------------------------------------------------------------------------
# 6. closed loop on routes that are not committed
# --------------------------------------------------------------------------------------------------------------------
CL_FLEETS = {"dense_traj2": (3500, 51), "repaired_equal": (600, 52)}
CL_MAX_STEPS = 1200


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CL_FLEETS))
def test_closed_loop_plant_steps_match_the_oracle(name, loaders):
    import safe_autonomous_driving_mpc_b200 as M
    B, seed = CL_FLEETS[name]
    L = loaders[name]
    tab = P.RefTable(L.X_ref, L.U_ref)
    T = M.BatchedTracker(L)
    assert (B > T.params.coop_max_batch) == (B == 3500)
    rng = np.random.default_rng(seed)
    s0 = rng.uniform(0.0, L.s_max - 150.0, B)
    trig = s0 + rng.uniform(0.0, 60.0, B)
    start = trig + rng.uniform(20.0, 120.0, B)
    combo = rng.permutation(np.arange(B) % 4)
    scen = [M.make_scenario(2, dynamic_obstacle=int(combo[b] & 1), traffic_light=int(combo[b] >> 1),
                            obs_trigger_s=float(trig[b]), obs_start_s=float(start[b]), obs_v=float(rng.uniform(4, 8)),
                            obs_end_s=float(start[b] + 150.0), tl_pos=float(s0[b] + rng.uniform(40.0, 400.0)),
                            tl_trigger_s=100.0, tl_stop_duration=float(rng.uniform(2.0, 8.0))) for b in range(B)]
    x_init = np.array([L.get_state(s) for s in s0])
    x_init[:, 4] = np.maximum(x_init[:, 4], 0.5)
    sim = M.BatchedSimulation(T, scen, x_init=x_init, history_steps=CL_MAX_STEPS)
    n_run = 0
    while n_run < CL_MAX_STEPS:
        sim.step(100)
        n_run += 100
        assert T.last_call_used_coop() == (B <= T.params.coop_max_batch)
        if sim.alive() == 0:
            break
    x_final, steps, n_unsolved = sim.state()
    h = sim.history()
    del sim
    target = np.concatenate([h["x"][1:], np.full((1, B, 5), np.nan)])
    target[steps - 1, np.arange(B)] = x_final
    worst = 0.0
    for a in range(0, n_run, 100):
        sl = slice(a, min(a + 100, n_run))
        live = np.arange(sl.start, sl.stop)[:, None] < steps[None, :]
        got = plant_step(tab, h["x"][sl], h["u"][sl])[live]
        want = target[sl][live]
        assert np.all(np.isfinite(want))
        worst = max(worst, rel(got, want))
    assert worst <= FN_TOL, worst
    s_stop = L.s_max - 1.0
    live = np.arange(n_run)[:, None] < steps[None, :]
    assert np.all(h["x"][:, :, 0][live] <= s_stop)
    arrived = x_final[:, 0] > s_stop
    assert np.all(arrived | (steps == n_run)) and steps.min() >= 1
    assert (~arrived).sum() <= B // 200, (~arrived).sum()
    assert np.array_equal(n_unsolved, ((h["status"] != 0) & live).sum(axis=0))


# --------------------------------------------------------------------------------------------------------------------
# 7. sixteen routes on one handle
# --------------------------------------------------------------------------------------------------------------------
ROUTES16 = list(FAMILIES)[:8] + ["dense_traj2", "traj1", "traj2", "traj3", "arc_k3_u2", "arc_k3_u3", "arc_k3_u5",
                                  "straight_k2"]


def _family_of(name):
    if name in FAMILIES:
        return FAMILIES[name]
    if name == "dense_traj2":
        return Family(name, lambda: _dense(2), base=2)
    i = int(name[-1])
    return Family(name, lambda: _base(i), base=None)


def _mixed16(B, seed=5):
    sets = [mc_problems(_family_of(n), B)[:3] for n in ROUTES16]
    route = np.random.default_rng(seed).integers(0, 16, B).astype(np.int32)
    rows = np.arange(B)
    x0 = np.stack([s[0] for s in sets])[route, rows]
    obs = np.stack([s[1] for s in sets])[route, rows]
    n = np.stack([s[2] for s in sets])[route, rows].astype(np.int32)
    return x0, obs, n, route


@pytest.fixture(scope="module")
def routed16(loaders):
    import safe_autonomous_driving_mpc_b200 as M
    Ls = [loaders[n] for n in ROUTES16]
    assert len(Ls) == M.BatchedTracker.MAX_ROUTES == 16
    return Ls


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS) + ["fast0"])
@pytest.mark.parametrize("B", [2000, 65536])
def test_sixteen_routes_equal_single_route_solves(B, variant, routed16, trackers):
    import safe_autonomous_driving_mpc_b200 as M
    from test_gpu_routes import _solve, _equal_rows
    kw = dict(VARIANTS, fast0=dict(fast_pass=0))[variant]
    TR = M.BatchedTracker(routed16, **kw)
    assert TR.n_routes == 16
    x0, obs, n, route = _mixed16(B)
    assert np.any(route == 15)
    got = _solve(TR, x0, obs, n, route)
    for r, name in enumerate(ROUTES16):
        ref = _solve(trackers(name, variant), x0, obs, n)
        _equal_rows(got, ref, route == r)
    assert np.all(got["status"] != 3)


@pytest.mark.gpu
def test_sixteen_route_fleet_follows_the_numpy_leader_rule(routed16):
    """A following fleet over all sixteen routes, with vehicles on route 15 (the last slot) and vehicles that arrive:
    the recorded leaders equal the numpy rule at every step."""
    import safe_autonomous_driving_mpc_b200 as M
    TR = M.BatchedTracker(routed16)
    B, n_steps, rng_range = 640, 150, 10.0
    route = (np.arange(B) % 16).astype(np.int32)
    rng = np.random.default_rng(8)
    x_init = np.empty((B, 5))
    for b in range(B):
        L = routed16[route[b]]
        s_lo = float(L.X_ref[0, 0])
        near_end = b % 5 == 0                           # these arrive within the run
        s0 = L.s_max - rng.uniform(2.0, 40.0) if near_end else s_lo + rng.uniform(0.0, max(L.s_max - s_lo - 60.0, 1.0))
        if b >= 16 and b % 7 == 0:
            s0 = min(x_init[b - 16, 0] + rng.uniform(0.5, 8.0), L.s_max - 2.0)   # close to a vehicle of its route
        x_init[b] = L.get_state(s0)
        x_init[b, 0] = s0
        x_init[b, 4] = max(x_init[b, 4], 0.5)
    scen = M.make_scenario(2, dynamic_obstacle=0, traffic_light=0)
    sim = M.BatchedSimulation(TR, [scen] * B, x_init=x_init, history_steps=n_steps, route=route,
                              follow_range=rng_range)
    sim.step(n_steps)
    _, steps, _ = sim.state()
    h, ld = sim.history(), sim.follow_history()
    del sim
    n_lead = 0
    for t in range(n_steps):
        live = steps > t
        x = h["x"][t]
        assert np.array_equal(live, ~np.isnan(x[:, 0]))
        lead, sv = leaders(np.where(live[:, None], x, 0.0), live, route, rng_range)
        assert np.array_equal(ld["lead"][t], lead), (t, np.flatnonzero(ld["lead"][t] != lead)[:8])
        assert np.array_equal(ld["lead_s"][t], sv[:, 0], equal_nan=True), t
        assert np.array_equal(ld["lead_v"][t], sv[:, 1], equal_nan=True), t
        n_lead += int((lead >= 0).sum())
    assert n_lead > 0
    arrived = steps < n_steps
    assert arrived[route == 15].any() and not arrived.all()
    assert (ld["lead"][0][route == 15] >= 0).any()
