"""Several routes on one handle (mpcb_create_routes, mpcb_solve_batch_routes, mpcb_sim_create_routes).

A problem's answer on a routed handle depends only on its own inputs and its route's table: each routed result must
equal, bit for bit, the same problem solved by a single-route tracker of that route in the same execution shape.  A
route outside the handle's tables is reported per problem and never read as a table index."""
import ctypes as C

import numpy as np
import pytest

from conftest import VARIANTS, traj_path

SOLVE_THREADS, SOLVE_CTAS = 128, 2          # problems per CTA and CTAs per SM of the first pass (mpcb_api.cu)
ROUTE_VARIANTS = dict(VARIANTS, fast0=dict(fast_pass=0))
KEYS = ("U", "Xpred", "obj", "status", "iters", "cmin", "active")
BAD_ROUTE = 3


def _loaders():
    import safe_autonomous_driving_mpc_b200 as M
    return [M.TrajectoryLoader(traj_path(i)) for i in (1, 2, 3)]


@pytest.fixture(scope="module")
def route_trackers():
    """Per variant: the tracker over routes 1-3 and the three single-route trackers."""
    import safe_autonomous_driving_mpc_b200 as M
    Ls = _loaders()
    return {name: (M.BatchedTracker(Ls, **kw), [M.BatchedTracker(L, **kw) for L in Ls])
            for name, kw in ROUTE_VARIANTS.items()}


def _mixed_batch(port_tables, B, seed=5):
    from oracle import tracker_port as P
    sets = [P.monte_carlo_problems(port_tables[i], B) for i in (1, 2, 3)]
    route = np.random.default_rng(seed).integers(0, 3, B).astype(np.int32)
    rows = np.arange(B)
    x0 = np.stack([s[0] for s in sets])[route, rows]
    obs = np.stack([s[1] for s in sets])[route, rows]
    n = np.stack([s[2] for s in sets])[route, rows].astype(np.int32)
    return x0, obs, n, route


def _solve(T, x0, obs, n, route=None):
    import torch
    dev = torch.device("cuda:0")
    d = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (x0, obs, n)]
    r = T.solve_batch(*d, route=None if route is None else torch.from_numpy(route).to(dev))
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in r.items()}


def _equal_rows(a, b, rows):
    for k in KEYS:
        assert np.array_equal(a[k][rows], b[k][rows], equal_nan=True), k


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(ROUTE_VARIANTS))
@pytest.mark.parametrize("B", [2000, 24000, 65536])
def test_routed_solve_equals_single_route_solves(B, variant, route_trackers, port_tables):
    import torch
    TR, singles = route_trackers[variant]
    assert TR.n_routes == 3
    wave = torch.cuda.get_device_properties(0).multi_processor_count * SOLVE_CTAS * SOLVE_THREADS
    if B == 24000:
        assert B <= wave, "one wave: the first pass runs every round in the class kernel"
    if B == 65536:
        assert B > wave, "more than one wave: the first pass compacts its survivors"
    x0, obs, n, route = _mixed_batch(port_tables, B)
    for r in range(3):
        for k in range(3):
            assert np.any((route == r) & (n == k)), (r, k)
    got = _solve(TR, x0, obs, n, route)
    if variant == "default":
        assert TR.last_call_used_coop() == (B <= 3072)
    for r in range(3):
        ref = _solve(singles[r], x0, obs, n)          # same B rows: same execution shape
        _equal_rows(got, ref, route == r)
    assert (got["status"] == 0).mean() > 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("B", [2000, 24000])
def test_route_zero_and_existing_entry_points_on_a_routed_handle(B, route_trackers, port_tables):
    """route=None, all-zero routes, and the entry points without a route argument: route 0, bit for bit."""
    TR, singles = route_trackers["default"]
    T1 = singles[0]
    from oracle import tracker_port as P
    x0, obs, n = P.monte_carlo_problems(port_tables[1], B)
    ref = _solve(T1, x0, obs, n)
    l0 = T1.launch_count()
    _solve(T1, x0, obs, n)
    launches_single = T1.launch_count() - l0
    l0 = TR.launch_count()
    got = _solve(TR, x0, obs, n)
    assert TR.launch_count() - l0 == launches_single
    _equal_rows(got, ref, slice(None))
    _equal_rows(_solve(TR, x0, obs, n, np.zeros(B, np.int32)), ref, slice(None))
    host_ref = T1.solve_batch_host(x0, obs, n, pinned_out=False)
    host_got = TR.solve_batch_host(x0, obs, n, pinned_out=False)
    _equal_rows(host_got, host_ref, slice(None))
    u0_ref = T1.solve_batch_host_u0(x0, obs, n, want_obj=True, pinned_out=False)
    u0_got = TR.solve_batch_host_u0(x0, obs, n, want_obj=True, pinned_out=False)
    for k in u0_ref:
        assert np.array_equal(u0_got[k], u0_ref[k], equal_nan=True), k


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(ROUTE_VARIANTS))
@pytest.mark.parametrize("B", [2000, 24000])
def test_out_of_range_routes_are_reported_per_problem(B, variant, route_trackers, port_tables):
    TR, _ = route_trackers[variant]
    x0, obs, n, route = _mixed_batch(port_tables, B, seed=9)
    bad = np.array([0, 1, 37, B // 2, B - 1])
    good = np.setdiff1d(np.arange(B), bad)
    route_bad = route.copy()
    route_bad[bad] = [-1, TR.n_routes, 1 << 20, -(1 << 30), TR.n_routes + 1]
    route_ok = route.copy()
    route_ok[bad] = 0
    got = _solve(TR, x0, obs, n, route_bad)
    ref = _solve(TR, x0, obs, n, route_ok)
    _equal_rows(got, ref, good)
    assert np.all(got["status"][bad] == BAD_ROUTE)
    for k in ("U", "Xpred", "obj", "cmin"):
        assert np.all(np.isnan(got[k][bad])), k
    assert np.all(got["iters"][bad] == 0) and np.all(got["active"][bad] == 0)
    assert np.all(got["status"][good] != BAD_ROUTE)


def _scenario(M, i):
    if i == 1:
        return M.make_scenario(2, dynamic_obstacle=0, traffic_light=0)
    return M.make_scenario(i)


@pytest.mark.gpu
@pytest.mark.parametrize("coop_max_batch", [0, 4096], ids=["thread", "warp"])
@pytest.mark.parametrize("hot", [False, True], ids=["cold", "hot"])
def test_routed_fleet_equals_single_route_fleets(coop_max_batch, hot):
    """One simulation over three routes (vehicle b on route b % 3, per-vehicle scenarios, staggered starts) against the
    three single-route simulations of the same vehicles, in the same execution shape and for the same number of steps."""
    import safe_autonomous_driving_mpc_b200 as M
    Ls = _loaders()
    per, n_steps = 200, 2400
    B = 3 * per
    route = np.arange(B, dtype=np.int32) % 3
    rng = np.random.default_rng(17)
    x_init = np.empty((B, 5))
    scen = []
    for b in range(B):
        r, L = route[b], Ls[route[b]]
        base = _scenario(M, r + 1)
        if b < 3:                                   # vehicle 0 of each route: the reference's start and scenario
            x_init[b] = [0.0, 0.0, 0.0, 0.0, 0.5]
            scen.append(base)
            continue
        s0 = rng.uniform(0.0, max(L.s_max - 150.0, 1.0))
        x_init[b] = L.get_state(s0)
        x_init[b, 4] = max(x_init[b, 4], 0.5)
        kw = {f: getattr(base, f) for f, _ in base._fields_}
        kw.update(obs_v=float(rng.uniform(3.0, 6.0)), tl_stop_duration=float(rng.uniform(4.0, 20.0)))
        if r > 0:
            kw.update(tl_pos=float(s0 + rng.uniform(120.0, 300.0)), obs_trigger_s=float(s0 + 5.0),
                      obs_start_s=float(s0 + 50.0), obs_end_s=float(s0 + 250.0))
        scen.append(M.make_scenario(2, **kw))

    def run(T, sel, rt):
        sim = M.BatchedSimulation(T, [scen[b] for b in sel], x_init=x_init[sel], history_steps=n_steps,
                                  hot_start=hot, route=rt)
        sim.step(n_steps)
        return sim.state(), sim.history(), sim.check()

    TR = M.BatchedTracker(Ls, coop_max_batch=coop_max_batch)
    (x, steps, uns), hist, chk = run(TR, np.arange(B), route)
    assert steps[0] == 172 and steps[1] == 985 and steps[2] == 2294
    for r in range(3):
        sel = np.where(route == r)[0]
        (xr, sr, ur), hr, cr = run(M.BatchedTracker(Ls[r], coop_max_batch=coop_max_batch), sel, None)
        assert np.array_equal(x[sel], xr) and np.array_equal(steps[sel], sr) and np.array_equal(uns[sel], ur), r
        for k in hr:
            assert np.array_equal(hist[k][:, sel], hr[k], equal_nan=True), (r, k)
        for k in cr:
            assert np.array_equal(chk[k][sel], cr[k], equal_nan=True), (r, k)
    assert chk["passed"][:3].all() and chk["history_complete"].all()


# ---- CPU: argument checks -----------------------------------------------------------------------------------------

def test_create_routes_rejects_bad_counts_and_null_tables_without_a_device():
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import _lib
    lib = _lib.load()
    p = _lib.Params()
    assert lib.mpcb_default_params(C.byref(p)) == 0
    L = M.TrajectoryLoader(traj_path(1))
    h = C.c_void_p()
    for n in (0, 17, -1):
        tabs = (C.c_void_p * max(n, 1))(*([L._h] * max(n, 1)))
        assert lib.mpcb_create_routes(C.byref(h), C.byref(p), tabs, n, 0) == -1, n
    tabs = (C.c_void_p * 2)(L._h, None)
    assert lib.mpcb_create_routes(C.byref(h), C.byref(p), tabs, 2, 0) == -1
    assert lib.mpcb_create_routes(C.byref(h), C.byref(p), None, 1, 0) == -1
    assert lib.mpcb_n_routes(None) == -1
    with pytest.raises(ValueError):
        M.BatchedTracker([])
    with pytest.raises(ValueError):
        M.BatchedTracker([L] * 17)


def test_wrappers_reject_route_arrays_of_the_wrong_shape_or_dtype():
    import torch
    import safe_autonomous_driving_mpc_b200 as M
    T = M.BatchedTracker(None)                       # attributes only: the checks come before any device call
    B = 8
    x0, obs, n = torch.zeros((B, 5), dtype=torch.float64), torch.zeros((B, 2, 2), dtype=torch.float64), torch.zeros(B, dtype=torch.int32)
    for bad in (torch.zeros(B + 1, dtype=torch.int32), torch.zeros(B, dtype=torch.int64), torch.zeros((B, 1), dtype=torch.int32),
                np.zeros(B, np.int32)):
        with pytest.raises(ValueError):
            T.solve_batch(x0, obs, n, route=bad)
    sc = M.make_scenario(2)
    for bad in (np.zeros(B - 1, np.int32), np.zeros(B, np.float64), np.zeros((B, 2), np.int32), 1.0):
        with pytest.raises(ValueError):
            M.BatchedSimulation(T, sc, B=B, route=bad)
