"""Planner host driver (safe-autonomous-driving-mpc_b200/planner_driver.py, SURVEY 8(f3)).
CPU tests drive it with the oracle evaluator; the GPU test plugs the CUDA evaluator in and must reproduce both."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, golden, traj_path


def _driver():
    import importlib
    return importlib.import_module("safe_autonomous_driving_mpc_b200.planner_driver")


# At the reference's ftol = 1e-4, where SLSQP stops on this chunk moves by up to ~4e-3 in U when the last bits of a BLAS
# sum change (the objective agrees to 1e-8 either way), and OpenBLAS sums differently with its thread count and with the
# kernels it picks for the host CPU.  The chunk is therefore solved in a child process with OpenBLAS on one thread and
# its generic x86-64 kernels: one floating-point path on every host, so the comparison below means the same everywhere.
PINNED_BLAS = {"OPENBLAS_NUM_THREADS": "1", "OPENBLAS_CORETYPE": "Prescott"}

_CHUNK_SOLVE = """
import importlib, os, sys
import numpy as np
root, out = sys.argv[1], sys.argv[2]
sys.path.insert(0, root)
from oracle import planner_port as Q, tracker_port as P
D = importlib.import_module("safe_autonomous_driving_mpc_b200.planner_driver")
g = np.load(os.path.join(root, "tests", "golden", "planner_chunk_traj1.npz"))
tab = P.RefTable.from_npz(os.path.join(root, "data", "trajectory1.npz"))
ev = Q.OracleEvaluator(tab, int(g["N"]), simpson_sign=-1, s_total=float(g["s_total"]), v_max=float(g["v_max"]))
X, U, S, sol, n_eval = D.optimize_chunk(ev, g["x0"], float(g["s_target"]), False)
np.savez(out, X=X, U=U, S=S, x=sol.x, fun=sol.fun, status=sol.status, n_eval=n_eval)
"""


def test_chunk_matches_reference_optimize(port_tables, tmp_path):
    """One chunk of the reference NLP (committed Simpson sign) against the UNMODIFIED reference optimizer
    (TrajectoryOptimizer.optimize, SLSQP + finite differences; tools/make_golden_planner.py --chunk):
    same objective to 1e-6 relative, same solution to 1e-3, in a comparable number of SLSQP iterations but ~40
    batched evaluations instead of 1,857 cost + ~15,000 closure calls per Jacobian."""
    from oracle import planner_port as Q
    g = golden("planner_chunk_traj1")
    N = int(g["N"])
    out = str(tmp_path / "chunk.npz")
    r = subprocess.run([sys.executable, "-c", _CHUNK_SOLVE, ROOT, out], env=dict(os.environ, **PINNED_BLAS),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    c = np.load(out)
    X, U, S = c["X"], c["U"], c["S"]
    assert int(c["status"]) == 0
    assert abs(float(c["fun"]) - float(g["cost"])) <= 1e-6 * abs(float(g["cost"]))
    assert np.abs(X - g["X"]).max() <= 1e-3 and np.abs(U - g["U"]).max() <= 1e-3 and np.abs(S - g["S"]).max() <= 1e-3
    assert int(c["n_eval"]) < 100
    assert np.abs(Q.defects(port_tables[1], c["x"], N, simpson_sign=-1)).max() < 1e-6


def test_constraint_jacobians_against_finite_differences(port_tables):
    from oracle import planner_port as Q
    D = _driver()
    N = 6
    ev = Q.OracleEvaluator(port_tables[1], N, simpson_sign=+1, s_total=300.0, v_max=12.0)
    prob = D.ChunkProblem(ev, np.array([3.0, 0.0, 0.0, 0.0, 2.0]), 23.0, False)
    rng = np.random.default_rng(3)
    z = D.initial_guess(N, prob.x0, 23.0, False) + rng.normal(0, 0.05, 8 * N + 5)
    for fun, jac in ((prob.eq, prob.eq_jac), (prob.ineq, prob.ineq_jac), (lambda y: np.array([prob.cost(y)]),
                                                                              lambda y: prob.cost_grad(y)[None])):
        J = jac(z)
        Jn = np.zeros_like(J)
        for j in range(len(z)):
            e = np.zeros_like(z)
            e[j] = 1e-6
            Jn[:, j] = (fun(z + e) - fun(z - e)) / 2e-6
        assert np.abs(J - Jn).max() <= 2e-6 * max(1.0, np.abs(Jn).max())


def test_full_short_route_physical_sign(port_tables):
    """Receding-horizon loop (trajectory_planning.py:491-554) over the first 70 m of trajectory1's curvature profile
    with the physical Simpson sign: arrives, stops, passes the reference's own trajectory checks."""
    from oracle import planner_port as Q
    D = _driver()
    tab = port_tables[1]
    s_total, v_max = 70.0, 8.0
    X, U, S, log = D.optimize_full_trajectory(lambda N, st: Q.OracleEvaluator(tab, N, simpson_sign=+1, s_total=st, v_max=v_max),
                                              s_total, v_max)
    assert len(log) >= 2 and log[-1]["final"] and all(c["status"] == 0 for c in log)
    v = D.reference_trajectory_verdicts(X, U, S, s_total)
    assert all(v.values()), v
    assert len(X) == len(U) + 1 == len(S) + 1
    assert np.all(np.diff(X[:, 0]) > -1e-2)          # the final approach may creep back by < 1 cm (v >= -0.1 tolerance)


def ev_pack(X, U, S):
    return np.concatenate([np.ravel(X), np.ravel(U), np.ravel(S)])


@pytest.mark.gpu
def test_gpu_evaluator_drives_the_same_solution(gpu_trackers, port_tables):
    """The CUDA evaluator behind the driver: the reference's chunk (objective as above) and the physical short route
    (passes the reference's checks; the evaluator agrees with the CPU oracle at every point of the plan)."""
    import safe_autonomous_driving_mpc_b200 as M
    from oracle import planner_port as Q
    D = _driver()
    L, T = gpu_trackers[1]
    g = golden("planner_chunk_traj1")
    N = int(g["N"])
    ev = M.PlannerEvaluator(T, N=N, simpson_sign=-1, s_total=float(g["s_total"]), v_max=float(g["v_max"]))
    X, U, S, sol, n_eval = D.optimize_chunk(ev, g["x0"], float(g["s_target"]), False)
    assert sol.status == 0 and abs(sol.fun - float(g["cost"])) <= 1e-6 * abs(float(g["cost"]))
    assert np.abs(X - g["X"]).max() <= 1e-3
    s_total, v_max = 70.0, 8.0
    Xg, Ug, Sg, logg = D.optimize_full_trajectory(
        lambda n, st: M.PlannerEvaluator(T, N=n, simpson_sign=+1, s_total=st, v_max=v_max), s_total, v_max)
    assert all(D.reference_trajectory_verdicts(Xg, Ug, Sg, s_total).values())
    assert abs(Xg[-1, 0] - s_total) <= 1e-3 and abs(Xg[-1, 4]) <= 1e-3 and all(c["status"] == 0 for c in logg)
    # The same route planned with the CPU oracle as the evaluator takes a different SLSQP path (ftol = 1e-4, the reference's
    # setting: rounding-level differences between the evaluators move the accepted iterates, and on some host CPUs one of
    # the two runs ends in a different local solution of a chunk), so the two PLANS are not compared.  What must agree is
    # what the evaluators return at the same points -- here along the GPU-driven plan, window by window.
    N = 12
    for k0 in range(0, len(Ug) - N, N):
        z = ev_pack(Xg[k0:k0 + N + 1], Ug[k0:k0 + N], Sg[k0:k0 + N])
        eg = M.PlannerEvaluator(T, N=N, simpson_sign=+1, s_total=s_total, v_max=v_max).evaluate_host(z, want_jac=True)
        ec = Q.OracleEvaluator(port_tables[1], N, simpson_sign=+1, s_total=s_total, v_max=v_max).evaluate_host(z, want_jac=True)
        for key in ("defect", "jac", "node_rows", "ctrl_rows", "cost", "cost_grad"):
            a, b = np.asarray(eg[key]), np.asarray(ec[key])
            assert np.abs(a - b).max() <= 1e-9 * max(1.0, np.abs(b).max()), (key, k0)
