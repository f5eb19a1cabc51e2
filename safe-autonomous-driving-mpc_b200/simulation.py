"""Batched closed loop on the GPU (SURVEY.md 8(f1)): host mirror of ``run_simulation`` (trajectory_tracking.py:377-443)
for B vehicles at once.  The loop body -- ObstaclesFSM.update, solve, Euler plant step, stop test -- runs as device
kernels behind ``mpcb_sim_*``; the host only decides how many steps to enqueue and when to look."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import Scenario, check


def _dp(a):
    return a.ctypes.data_as(C.c_void_p)


def make_scenario(which=2, **over):
    """Scenario constants: which=2 as committed (:294-308), which=3 the commented trajectory3 block (:313-327)."""
    s = Scenario()
    check(_lib.load().mpcb_scenario_default(C.byref(s), int(which)))
    for k, v in over.items():
        if not hasattr(s, k):
            raise TypeError(f"unknown scenario field {k!r}")
        setattr(s, k, v)
    return s


# Solver caps for a large fleet whose vehicles are in different phases of their drives.  The defaults are tuned for a
# Monte-Carlo batch of perturbed states, where 1.4 % of the problems are left to the robust pass; in a closed loop a
# quarter of the vehicles is at any time braking for, waiting at or leaving a stop line, the two-level first pass with
# ONE active-set update per linearisation gives most of those up, and the robust pass (one warp per problem) becomes the
# step.  Three updates per linearisation keep them in the first pass.  Measured on B200, 65,536 vehicles on trajectory3
# with staggered starts and per-vehicle scenarios (tools/gpu_sim_fleet.py): 16.0 -> 41.8 M vehicle-steps/s; the same caps
# cost a Monte-Carlo batch 0.31 -> 0.42+ ms in its first pass, which is why they are not the default.
#     T = BatchedTracker(loader, **FLEET_SOLVER_CAPS);  sim = BatchedSimulation(T, scenarios, x_init=...)
FLEET_SOLVER_CAPS = dict(thread_max_segments=3)

CHECKS = ("destination", "on_road", "steering", "acceleration", "obstacle", "light", "history_complete")


def _verdict_dict(v, m):
    out = {name: ((v >> k) & 1).astype(bool) for k, name in enumerate(CHECKS)}
    out["passed"] = (v & 63) == 63
    out.update(max_dev=m[:, 0], min_gap=m[:, 1], s_final=m[:, 2], steps=m[:, 3].astype(np.int64))
    return out


def check_histories(tracker, s_total, scenarios, x_final, steps, hist_x, hist_u, hist_obs, hist_tl):
    """trajectory_tracking_check (sanity_checks.py:79-184) on the GPU for B recorded drives supplied by the caller:
    hist_x [T,B,5] (state before each step), hist_u [T,B,2], hist_obs [T,B] (NaN: no car), hist_tl [T,B] (0 red,
    1 green), x_final [B,5], steps [B].  Returns the same dict as ``BatchedSimulation.check``."""
    lib = tracker._lib
    hist_x = np.ascontiguousarray(hist_x, dtype=np.float64)
    T, B = hist_x.shape[:2]
    hist_u = np.ascontiguousarray(hist_u, dtype=np.float64).reshape(T, B, 2)
    hist_obs = np.ascontiguousarray(hist_obs, dtype=np.float64).reshape(T, B)
    hist_tl = np.ascontiguousarray(hist_tl, dtype=np.int32).reshape(T, B)
    x_final = np.ascontiguousarray(x_final, dtype=np.float64).reshape(B, 5)
    steps = np.ascontiguousarray(steps, dtype=np.int32).reshape(B)
    scen = list(scenarios)
    assert len(scen) == B
    arr = (Scenario * B)(*scen)
    v = np.empty(B, np.int32)
    m = np.empty((B, 4))
    check(lib.mpcb_check_histories(tracker._need(), B, T, float(s_total), arr, _dp(x_final), _dp(steps), _dp(hist_x),
                                   _dp(hist_u), _dp(hist_obs), _dp(hist_tl), _dp(v), _dp(m)), "mpcb_check_histories")
    return _verdict_dict(v, m)


def _follow_range(r):
    r = float(r)
    if not (np.isfinite(r) and r > 0.0):
        raise ValueError(f"follow_range must be positive and finite, got {r!r}")
    return r


class BatchedSimulation:
    def __init__(self, tracker, scenarios, B=None, x_init=None, history_steps=0, hot_start=False, route=None,
                 follow_range=None):
        """tracker: BatchedTracker; scenarios: one Scenario (shared) or a list of B; x_init: [B,5] or None for the
        reference's start state.  hot_start: from its second step on a vehicle's solve starts from its previous plan
        advanced by one step (mpcb_sim_set_hot_start) instead of the reference's table-based warm start.
        route: one int or an int array [B], vehicle b driving ``tracker.routes[route[b]]`` (None: route 0).
        follow_range: None (off) or a positive distance: the nearest vehicle ahead on the same route within that
        distance is a moving obstacle (``set_follow``)."""
        self._lib = tracker._lib
        self._t = tracker
        if follow_range is not None:
            follow_range = _follow_range(follow_range)
        scen = list(scenarios) if isinstance(scenarios, (list, tuple)) else [scenarios]
        if B is None:
            B = len(scen) if len(scen) > 1 else (len(x_init) if x_init is not None else 1)
        arr = (Scenario * len(scen))(*scen)
        xi = None
        if x_init is not None:
            xi = np.ascontiguousarray(x_init, dtype=np.float64).reshape(B, 5)
        rt = None
        if route is not None:
            rt = np.asarray(route)
            if rt.ndim == 0:
                rt = np.full(B, rt)
            if not np.issubdtype(rt.dtype, np.integer) or rt.shape != (B,):
                raise ValueError(f"route must be one int or an int array of shape ({B},)")
            rt = np.ascontiguousarray(rt, dtype=np.int32)
        h = C.c_void_p()
        check(self._lib.mpcb_sim_create_routes(C.byref(h), tracker._need(), int(B), arr, len(scen),
                                               _dp(rt) if rt is not None else None,
                                               _dp(xi) if xi is not None else None, int(history_steps)),
              "mpcb_sim_create_routes")
        self._h = h
        self.B = int(B)
        self.history_steps = int(history_steps)
        if hot_start:
            check(self._lib.mpcb_sim_set_hot_start(h, 1), "mpcb_sim_set_hot_start")
        if follow_range is not None:
            self.set_follow(follow_range)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.mpcb_sim_destroy(h)
            self._h = None

    def step(self, n=1, stream=None):
        check(self._lib.mpcb_sim_step(self._h, int(n), C.c_void_p(stream or 0)), "mpcb_sim_step")

    def alive(self):
        n = C.c_int()
        check(self._lib.mpcb_sim_alive(self._h, C.byref(n), None))
        return n.value

    def state(self):
        x = np.empty((self.B, 5)); st = np.empty(self.B, np.int32); nu = np.empty(self.B, np.int32)
        check(self._lib.mpcb_sim_state(self._h, _dp(x), _dp(st), _dp(nu), None))
        return x, st, nu

    def history(self):
        n = C.c_int()
        check(self._lib.mpcb_sim_history(self._h, C.byref(n), None, None, None, None, None, None))
        T, B = n.value, self.B
        hx = np.empty((T, B, 5)); hu = np.empty((T, B, 2)); ho = np.empty((T, B))
        hs = np.empty((T, B), np.int32); ht = np.empty((T, B), np.int32)
        check(self._lib.mpcb_sim_history(self._h, C.byref(n), _dp(hx), _dp(hu), _dp(ho), _dp(hs), _dp(ht), None))
        return dict(x=hx, u=hu, obs_s=ho, status=hs, tl=ht)

    def set_follow(self, follow_range):
        """Following from the next step on (mpcb_sim_set_follow): at the start of every step the nearest vehicle still
        driving ahead on the same route, ordered by (s, index), is vehicle b's leader when it is at most
        ``follow_range`` metres ahead; the nearer of the leader and the scripted car takes the car slot of b's obstacle
        set.  None switches following off."""
        if follow_range is None:
            check(self._lib.mpcb_sim_set_follow(self._h, 0, 0.0), "mpcb_sim_set_follow")
            return
        check(self._lib.mpcb_sim_set_follow(self._h, 1, _follow_range(follow_range)), "mpcb_sim_set_follow")

    def follow_history(self):
        """Leaders of the recorded steps: lead [T,B] (vehicle index, -1: none, arrived, or following off), lead_s and
        lead_v [T,B] (the leader's s and v at the start of the step, NaN where lead is -1)."""
        n = C.c_int()
        check(self._lib.mpcb_sim_follow_history(self._h, C.byref(n), None, None, None), "mpcb_sim_follow_history")
        T, B = n.value, self.B
        li = np.empty((T, B), np.int32)
        sv = np.empty((T, B, 2))
        check(self._lib.mpcb_sim_follow_history(self._h, C.byref(n), _dp(li), _dp(sv), None), "mpcb_sim_follow_history")
        return dict(lead=li, lead_s=sv[..., 0], lead_v=sv[..., 1])

    def follow_check(self):
        """Gap to the leader over the recorded steps: min_gap [B] (1e30 if never had a leader) and ok [B] = gap >= 1 m,
        the reference's moving-obstacle safety distance (sanity_checks.py:142-164)."""
        ok = np.empty(self.B, np.int32)
        g = np.empty(self.B)
        check(self._lib.mpcb_sim_follow_check(self._h, _dp(ok), _dp(g), None), "mpcb_sim_follow_check")
        return dict(ok=ok.astype(bool), min_gap=g)

    CHECKS = CHECKS

    def check(self):
        """trajectory_tracking_check (sanity_checks.py:79-184) per vehicle: dict of bool arrays [B] plus metrics."""
        v = np.empty(self.B, np.int32)
        m = np.empty((self.B, 4))
        check(self._lib.mpcb_sim_check(self._h, _dp(v), _dp(m), None), "mpcb_sim_check")
        return _verdict_dict(v, m)

    def run(self, max_steps=200000, check_every=64):
        """Drive until every vehicle has passed s_max - 1 (or max_steps).  Returns the number of steps enqueued."""
        done = 0
        while done < max_steps:
            k = min(check_every, max_steps - done)
            self.step(k)
            done += k
            if self.alive() == 0:
                break
        return done
