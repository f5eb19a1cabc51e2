"""Test helper: the closed loop's callers either side of the solve path, modelled with numpy and the oracle only.

``fsm_replay`` drives an oracle obstacle FSM over recorded states, ``plant_step`` is the reference's plant step,
``leaders`` and ``merge`` are the rules of following (the nearest vehicle ahead on the same route as a moving
obstacle).  The device closed loop (mpcb_sim_*) is checked against these; they are themselves checked without a GPU
against the reference's closed-loop logs and hand-made cases (test_gpu_closed_loop_replay.py, test_gpu_sim_follow.py)."""
import numpy as np

from oracle import sqp_admm_model as A
from oracle import tracker_port as P

DT = P.DT


def fsm_replay(fsm, s, v):
    """Drive an oracle FSM over recorded states (s[t], v[t]): the obstacle set the solver of step t sees (obs_sv [k,2,2],
    unused slots 0, car first; n_obs [k]), the position of the moving car (NaN when there is none) and the light colour
    (1 green, 0 red), as ObstacleFSMPort.update returns them."""
    k = len(s)
    obs_sv = np.zeros((k, 2, 2))
    n_obs = np.zeros(k, np.int32)
    car = np.full(k, np.nan)
    green = np.zeros(k, np.int32)
    for t, (st, vt) in enumerate(zip(np.asarray(s).tolist(), np.asarray(v).tolist())):
        act, colour = fsm.update(DT, st, vt)
        for j, o in enumerate(act):
            obs_sv[t, j] = (o["s"], o["v"])
            if o["type"] == "car":
                car[t] = o["s"]
        n_obs[t] = len(act)
        green[t] = colour == "GREEN"
    return obs_sv, n_obs, car, green


def k_ref(tab, s):
    """get_state(s)[3] (trajectory_loader.py:86-93), vectorised; s >= s_max gives the last knot's curvature."""
    return A.lookup(tab, s)[0][..., 2]


def plant_step(tab, x, u):
    """x + DT * dynamics(x, u, k_ref(s)) (trajectory_tracking.py:50-67, :404-406) over leading axes, in the reference's
    operation order."""
    s, o, k, v = x[..., 0], x[..., 2], x[..., 3], x[..., 4]
    f = np.stack([v, v * o, v * (k - k_ref(tab, s)), u[..., 0], u[..., 1]], axis=-1)
    return x + DT * f


def leaders(x, live, route, follow_range):
    """The leader rule for one step: x [B,5] states at the start of the step, live [B] still driving, route [B].
    Returns lead [B] (-1: none) and lead_sv [B,2] (NaN: none)."""
    B = len(x)
    s = x[:, 0]
    lead = np.full(B, -1, np.int64)
    for r in np.unique(route[live]):
        idx = np.flatnonzero(live & (route == r))
        order = idx[np.lexsort((idx, s[idx]))]           # by s, then by index
        a, b = order[:-1], order[1:]
        near = s[b] - s[a] <= follow_range
        lead[a[near]] = b[near]
    sv = np.full((B, 2), np.nan)
    has = lead >= 0
    sv[has] = x[lead[has]][:, [0, 4]]
    return lead, sv


def merge(obs_sv, n_obs, car, lead_sv):
    """The FSM's obstacle set (car first when present, then the light; unused slots 0) with the leader merged into the
    car slot: the nearer of scripted car and leader, the scripted car on a tie.  Leading axes are arbitrary."""
    obs_sv, n_obs = obs_sv.copy(), n_obs.copy()
    ls = lead_sv[..., 0]
    has_car = ~np.isnan(car)
    take = ~np.isnan(ls) & ~(has_car & (car <= ls))
    shift = take & ~has_car                              # no car: the light (if any) moves behind the leader
    obs_sv[..., 1, :] = np.where(shift[..., None], obs_sv[..., 0, :], obs_sv[..., 1, :])
    obs_sv[..., 0, :] = np.where(take[..., None], lead_sv, obs_sv[..., 0, :])
    n_obs = n_obs + shift
    return obs_sv, n_obs.astype(np.int32)
