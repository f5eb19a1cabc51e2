"""Rare failures of noisy closed-loop fleets: splitting estimates of the probability that a vehicle leaves the road
(``offroad_probability``) and that a follower comes within 1 m of the vehicle ahead (``near_miss_probability``).

Crude Monte-Carlo needs about 10^7 whole drives to resolve a failure rate of 10^-6 to +-30 %.  ``offroad_probability``
instead runs a fixed-effort interacting particle system (Del Moral & Garnier, "Genealogical particle analysis of rare
events", Ann. Appl. Probab. 15(4), 2005) on a noisy ``BatchedSimulation``: every ``every`` steps it weighs each vehicle
by how much closer to the road's edge it has come since the last resampling, draws B parents in proportion to those
weights, and lets ``branch`` copy the chosen vehicles over the others.  The copies draw fresh noise (the generator is
keyed by vehicle slot), so the fleet's effort goes to the drives that are heading off the road.

With V_b = min(running max |d| of vehicle b, 1.5) (``running_check()["max_dev"]``, capped at the off-road level; it
never decreases and is copied with the vehicle) and G_b = exp(lam (V_b - V_b^prev)) at each resampling k, where V^prev is the lineage's V at the previous
resampling (at the start for the first):

    p = prod_k mean(G^(k)) * mean_b[ fail_b * exp(-lam (V_b^last - V_b^0)) ]

with fail_b the cleared on_road bit (max |d| > 1.5) once no vehicle is driving (or at max_steps), V^last the lineage's V at the last
resampling and V^0 its start.  The cap matters: a vehicle that has left the road may keep diverging, and an uncapped
score would hand the whole population to one runaway lineage.  The potentials telescope along each lineage, so p is unbiased for any lam >= 0; lam
trades how hard the fleet is pushed toward the edge against the spread of the final weights.  lam = 0 never branches
and returns the crude fraction.  Repetitions (a new seed for the noise and for the resampling each) and their standard
error are the caller's.

``sim`` is anything with ``B``, ``step(n)``, ``alive()``, ``running_check()`` (a dict with ``max_dev``, ``on_road`` and
``steps`` arrays [B]) and ``branch(parent)``; the tests plug a numpy stand-in in here to check the arithmetic without a
GPU.

``near_miss_probability`` runs the same particle system with whole worlds as the particles (``world_size``,
``branch_worlds``): V_w = -min(max(g_w, 1), gap_cap) with g_w the least running follower gap of world w
(``running_follow_check()["min_gap"]``), never decreasing and capped at the 1 m failure level for the same reason, and
fail_w = some vehicle of world w not ok.  There ``sim`` also needs ``W`` and ``running_follow_check()`` (a dict with
``ok`` and ``min_gap`` arrays [B]), and ``branch_worlds(parent_world)`` in place of ``branch``."""
import math

import numpy as np

OFFROAD = 1.5          # lateral deviation of trajectory_tracking_check's on_road item, and the cap of the score
SAFETY = 1.0           # gap to the leader of the follow check's ok, and the cap of the near-miss score


def _score(r):
    return np.minimum(np.asarray(r["max_dev"], dtype=np.float64), OFFROAD)


def _check(lam, every, seed):
    lam = float(lam)
    if not (math.isfinite(lam) and lam >= 0.0):
        raise ValueError(f"lam must be finite and >= 0, got {lam!r}")
    if isinstance(every, bool) or not isinstance(every, (int, np.integer)) or every < 1:
        raise ValueError(f"every must be a positive integer, got {every!r}")
    if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)) or seed < 0:
        raise ValueError(f"seed must be a non-negative integer, got {seed!r}")
    return lam


def _splitting(sim, n, lam, every, seed, max_steps, observe, branch):
    """The particle system over n particles: observe() -> (V [n], fail [n], steps driven [n]) after every epoch,
    branch(parent [n]) copies particles.  Returns the dict of offroad_probability."""
    v0, _fail, st_prev = observe()                         # V^0 of each lineage
    v_prev = v0.copy()                                     # V of each lineage at its last resampling
    log_w = []
    done = vehicle_steps = epoch = 0
    alive = sim.B
    while done < max_steps:
        k = min(int(every), max_steps - done)
        sim.step(k)
        done += k
        alive = sim.alive()
        v, fail, st = observe()
        vehicle_steps += int((st - st_prev).sum())
        st_prev = st
        if alive == 0 or done >= max_steps:               # fail is the final verdicts
            break
        if lam > 0.0:
            a = lam * (v - v_prev)                         # log G, >= 0
            top = a.max()
            g = np.exp(a - top)
            log_w.append(float(top + math.log(g.mean())))
            parent = np.random.default_rng((int(seed), epoch)).choice(n, size=n, p=g / g.sum())
            branch(parent)
            v_prev, v0, st_prev = v[parent], v0[parent], st[parent]
        epoch += 1
    if lam == 0.0:
        p = float(fail.mean())
    else:
        tail = float(np.mean(np.where(fail, np.exp(-lam * (v_prev - v0)), 0.0)))
        p = math.exp(sum(log_w)) * tail if tail > 0.0 else 0.0
    return dict(p=p, log10_p=math.log10(p) if p > 0.0 else -math.inf, log_w=log_w, resamplings=len(log_w),
                vehicle_steps=vehicle_steps, steps=done, alive=int(alive))


def offroad_probability(sim, lam, every, seed, max_steps=200000):
    """Splitting estimate of P(a vehicle leaves the road) on ``sim``, driven from its current state until no vehicle
    is driving (or ``max_steps``).  Returns a dict: ``p``, ``log10_p`` (-inf when p = 0), ``log_w`` (log W_k = log mean
    G of each resampling), ``resamplings``, ``vehicle_steps`` (steps driven by all vehicles, copies included), ``steps``
    (loop steps enqueued) and ``alive`` (vehicles still driving at the end; 0 unless ``max_steps`` cut the drives)."""
    lam = _check(lam, every, seed)

    def observe():
        r = sim.running_check()
        return _score(r), ~np.asarray(r["on_road"], dtype=bool), np.asarray(r["steps"], dtype=np.int64)

    return _splitting(sim, int(sim.B), lam, every, seed, max_steps, observe, sim.branch)


def near_miss_probability(sim, lam, every, seed, gap_cap, max_steps=200000):
    """Splitting estimate of P(some follower of a world comes within 1 m of its leader) on ``sim``, a simulation with
    worlds and following on, driven from its current state until no vehicle is driving (or ``max_steps``); the
    particles are its W worlds.  gap_cap > 1: the gap from which the score starts to rise (a smaller gap counts as
    closer to failing).  Returns the dict of ``offroad_probability``, ``vehicle_steps`` counting every vehicle of every
    world."""
    lam = _check(lam, every, seed)
    gap_cap = float(gap_cap)
    if not (math.isfinite(gap_cap) and gap_cap > SAFETY):
        raise ValueError(f"gap_cap must be finite and > {SAFETY}, got {gap_cap!r}")
    W = int(sim.W)
    M = int(sim.B) // W

    def observe():
        steps = np.asarray(sim.running_check()["steps"], dtype=np.int64).reshape(W, M).sum(axis=1)
        f = sim.running_follow_check()
        g = np.asarray(f["min_gap"], dtype=np.float64).reshape(W, M).min(axis=1)
        fail = ~np.asarray(f["ok"], dtype=bool).reshape(W, M).all(axis=1)
        return -np.minimum(np.maximum(g, SAFETY), gap_cap), fail, steps

    return _splitting(sim, W, lam, every, seed, max_steps, observe, sim.branch_worlds)
