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


WORLD_MAX = 1024       # largest world of mpcb_sim_set_worlds


def _world_size(B, m):
    """Checked world size of mpcb_sim_set_worlds: 0 (one world) for None or 0, else an integer in [1, 1024] that divides
    B; ValueError otherwise."""
    if m is None:
        return 0
    if isinstance(m, bool) or not isinstance(m, (int, np.integer)) or not 0 <= int(m) <= WORLD_MAX or (m and B % int(m)):
        raise ValueError(f"world_size must be an integer in [1, {WORLD_MAX}] that divides B = {B} (or None / 0 for "
                         f"one world), got {m!r}")
    return int(m)


NOISE_CHANNELS = (("meas", 5), ("act", 2), ("proc", 5))


def _noise_args(B, seed, meas, act, proc, first_id):
    """Checked arguments of mpcb_sim_set_noise: (seed, first_id, three float64 arrays or None); ValueError otherwise."""
    if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)) or not 0 <= int(seed) < 2 ** 64:
        raise ValueError(f"seed must be an integer in [0, 2^64), got {seed!r}")
    if isinstance(first_id, bool) or not isinstance(first_id, (int, np.integer)) or not 0 <= int(first_id) <= 2 ** 31 - B:
        raise ValueError(f"first_id must be an integer in [0, 2^31 - B] (B = {B}), got {first_id!r}")
    sig = []
    for (name, n), v in zip(NOISE_CHANNELS, (meas, act, proc)):
        if v is None:
            sig.append(None)
            continue
        a = np.array(np.broadcast_to(np.asarray(v, dtype=np.float64), (n,)))
        if not (np.all(np.isfinite(a)) and np.all(a >= 0.0)):
            raise ValueError(f"{name} sigmas must be finite and >= 0, got {v!r}")
        sig.append(a)
    return int(seed), int(first_id), sig


class BatchedSimulation:
    def __init__(self, tracker, scenarios, B=None, x_init=None, history_steps=0, hot_start=False, route=None,
                 follow_range=None, noise=None, world_size=None):
        """tracker: BatchedTracker; scenarios: one Scenario (shared) or a list of B; x_init: [B,5] or None for the
        reference's start state.  hot_start: from its second step on a vehicle's solve starts from its previous plan
        advanced by one step (mpcb_sim_set_hot_start) instead of the reference's table-based warm start.
        route: one int or an int array [B], vehicle b driving ``tracker.routes[route[b]]`` (None: route 0).
        follow_range: None (off) or a positive distance: the nearest vehicle ahead on the same route within that
        distance is a moving obstacle (``set_follow``).
        noise: None (off) or a dict of ``set_noise``'s arguments (seed, meas, act, proc, first_id).
        world_size: None (one world) or M: vehicles [w M, (w + 1) M) form world w and follow only each other
        (``set_worlds``)."""
        self._lib = tracker._lib
        self._t = tracker
        if follow_range is not None:
            follow_range = _follow_range(follow_range)
        scen = list(scenarios) if isinstance(scenarios, (list, tuple)) else [scenarios]
        if B is None:
            B = len(scen) if len(scen) > 1 else (len(x_init) if x_init is not None else 1)
        if noise is not None:
            noise = dict(noise)
            unknown = set(noise) - {"seed", "meas", "act", "proc", "first_id"}
            if unknown or "seed" not in noise:
                raise ValueError(f"noise takes seed, meas, act, proc and first_id, got {sorted(noise)}")
            nz = _noise_args(int(B), noise["seed"], noise.get("meas"), noise.get("act"), noise.get("proc"),
                             noise.get("first_id", 0))
        world_size = _world_size(int(B), world_size)
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
        self.world_size, self.W = None, 1
        if hot_start:
            check(self._lib.mpcb_sim_set_hot_start(h, 1), "mpcb_sim_set_hot_start")
        if follow_range is not None:
            self.set_follow(follow_range)
        if noise is not None:
            self._set_noise(*nz)
        if world_size:
            self.set_worlds(world_size)

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

    def set_worlds(self, world_size):
        """Worlds from the next step on (mpcb_sim_set_worlds; include/mpcb200.h has the rules): world w is vehicles
        [w M, (w + 1) M) for M = world_size, and a vehicle's leader is searched for only inside its own world.  M must
        be in [1, 1024] and divide B, else ValueError before any device call; None or 0 returns to one world.  Sets
        ``world_size`` (None: one world) and ``W`` (the number of worlds)."""
        m = _world_size(self.B, world_size)
        check(self._lib.mpcb_sim_set_worlds(self._h, m), "mpcb_sim_set_worlds")
        self.world_size, self.W = (m, self.B // m) if m else (None, 1)

    def set_noise(self, seed, meas=None, act=None, proc=None, first_id=0):
        """Seeded Gaussian disturbances from the next step on (mpcb_sim_set_noise; include/mpcb200.h has the rules):
        meas [5] sigmas of the state the solve sees, act [2] of the applied control, proc [5] added to the state after
        each step; a scalar stands for every component, None for zeros.  Vehicle b draws as vehicle first_id + b, so a
        shard [lo, hi) of a fleet with first_id=lo draws the whole fleet's noise.  No sigma > 0: noise off."""
        self._set_noise(*_noise_args(self.B, seed, meas, act, proc, first_id))

    def _set_noise(self, seed, first_id, sig):
        check(self._lib.mpcb_sim_set_noise(self._h, seed, first_id, *(None if a is None else _dp(a) for a in sig)),
              "mpcb_sim_set_noise")

    def noise_history(self):
        """The disturbances added in the recorded steps, sigma * z (0.0 where sigma is 0): meas [T,B,5], act [T,B,2],
        proc [T,B,5]; NaN where the vehicle had arrived or noise was off."""
        n = C.c_int()
        check(self._lib.mpcb_sim_noise_history(self._h, C.byref(n), None, None), "mpcb_sim_noise_history")
        w = np.empty((n.value, self.B, 12))
        check(self._lib.mpcb_sim_noise_history(self._h, C.byref(n), _dp(w), None), "mpcb_sim_noise_history")
        return dict(meas=w[..., :5], act=w[..., 5:7], proc=w[..., 7:])

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

    def running_follow_check(self):
        """The same dict as ``follow_check``, from the least gap to the leader the loop keeps per vehicle
        (mpcb_sim_running_follow_check): needs no history.  Equal to ``follow_check`` bit for bit when the history
        covers every drive; min_gap 1e30 and ok True if following was never on."""
        ok = np.empty(self.B, np.int32)
        g = np.empty(self.B)
        check(self._lib.mpcb_sim_running_follow_check(self._h, _dp(ok), _dp(g), None), "mpcb_sim_running_follow_check")
        return dict(ok=ok.astype(bool), min_gap=g)

    CHECKS = CHECKS

    def check(self):
        """trajectory_tracking_check (sanity_checks.py:79-184) per vehicle: dict of bool arrays [B] plus metrics."""
        v = np.empty(self.B, np.int32)
        m = np.empty((self.B, 4))
        check(self._lib.mpcb_sim_check(self._h, _dp(v), _dp(m), None), "mpcb_sim_check")
        return _verdict_dict(v, m)

    def running_check(self):
        """The same dict as ``check``, from the accumulators the loop keeps per vehicle (mpcb_sim_running_check): needs
        no history, and history_complete is always True.  Equal to ``check`` bit for bit when the history covers every
        drive; max_dev includes the current state, so it never decreases while a vehicle drives."""
        v = np.empty(self.B, np.int32)
        m = np.empty((self.B, 4))
        check(self._lib.mpcb_sim_running_check(self._h, _dp(v), _dp(m), None), "mpcb_sim_running_check")
        return _verdict_dict(v, m)

    def branch(self, parent, stream=None):
        """Vehicle b takes over the whole state of vehicle parent[b], histories and running verdicts included
        (mpcb_sim_branch; include/mpcb200.h has the rules).  parent: integer array [B] with values in [0, B), else
        ValueError before any device call.  Vehicle b keeps drawing noise as vehicle first_id + b, so copies of one
        parent draw independent futures.  Refused (MpcbError) while following is on."""
        p = np.asarray(parent)
        if p.shape != (self.B,) or not np.issubdtype(p.dtype, np.integer):
            raise ValueError(f"parent must be an int array of shape ({self.B},), got {p.dtype} {p.shape}")
        if p.size and (p.min() < 0 or p.max() >= self.B):
            raise ValueError(f"parent values must be in [0, {self.B})")
        p = np.ascontiguousarray(p, dtype=np.int32)
        check(self._lib.mpcb_sim_branch(self._h, _dp(p), C.c_void_p(stream or 0)), "mpcb_sim_branch")

    def branch_worlds(self, parent_world, stream=None):
        """World w takes over the whole state of world parent_world[w], vehicle by vehicle, histories and running
        verdicts included; recorded leaders are moved into the copy's world (mpcb_sim_branch_worlds; include/mpcb200.h
        has the rules).  Needs worlds (``set_worlds``); parent_world: integer array [W] with values in [0, W), else
        ValueError before any device call.  Following may be on."""
        if not self.world_size:
            raise ValueError("branch_worlds needs worlds: set_worlds(M) or BatchedSimulation(world_size=M)")
        p = np.asarray(parent_world)
        if p.shape != (self.W,) or not np.issubdtype(p.dtype, np.integer):
            raise ValueError(f"parent_world must be an int array of shape ({self.W},), got {p.dtype} {p.shape}")
        if p.min() < 0 or p.max() >= self.W:
            raise ValueError(f"parent_world values must be in [0, {self.W})")
        p = np.ascontiguousarray(p, dtype=np.int32)
        check(self._lib.mpcb_sim_branch_worlds(self._h, _dp(p), C.c_void_p(stream or 0)), "mpcb_sim_branch_worlds")

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
