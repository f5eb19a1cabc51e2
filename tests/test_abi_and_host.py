"""CPU-side checks of the product: the C-ABI library loads and exports every declared symbol, the host table
reproduces the reference's lookups bit-for-bit, the FSM/closed-loop host logic matches the reference's log, and the
compute entry points fail loudly without a GPU (no fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, golden, traj_path


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "mpcb200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(mpcb_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    from safe_autonomous_driving_mpc_b200 import _lib
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/mpcb200.h but not exported"
        assert n in _lib.SYMBOLS, f"{n} has no ctypes signature"
    assert lib.mpcb_abi_version() == 7
    assert lib.mpcb_strerror(-1) == b"invalid argument"


def test_params_struct_mirrors_reference_constants():
    from safe_autonomous_driving_mpc_b200 import _lib
    p = _lib.Params()
    assert _lib.load().mpcb_default_params(C.byref(p)) == 0
    assert (p.dt, p.N) == (0.2, 5)
    assert list(p.u_min) == [-0.6, -5.0] and list(p.u_max) == [0.6, 4.0]
    assert (p.w_d, p.w_o, p.w_v, p.w_u1, p.w_u2) == (10.0, 10.0, 5.0, 0.5, 0.5)
    assert (p.obstacle_safety_distance, p.max_time_2_obs, p.wheelbase, p.lane_width) == (5.0, 1.5, 2.8, 3.0)
    assert (p.vehicle_radius, p.safe_lane_margin) == (1.0, 0.1)
    # sizeof must match the C struct (catches field drift between header and ctypes)
    # sizeof must match the C struct (catches field drift between header and ctypes)
    assert C.sizeof(p) == _lib.load().mpcb_sizeof_params()
    assert C.sizeof(_lib.PlannerParams()) == _lib.load().mpcb_sizeof_planner_params()
    

@pytest.mark.parametrize("i", [1, 2, 3])
def test_host_table_bit_exact(i):
    import safe_autonomous_driving_mpc_b200 as M
    z = golden(f"fn_traj{i}")
    L = M.TrajectoryLoader(traj_path(i))
    gs = np.array([L.get_state(s) for s in z["s_query"]])
    gc = np.array([L.get_control(s) for s in z["s_query"]])
    assert np.array_equal(gs, z["get_state"]) and np.array_equal(gc, z["get_control"])


def test_table_monotone_repair_and_edge_cases():
    import safe_autonomous_driving_mpc_b200 as M
    from oracle import tracker_port as P
    X = np.array([[0, 0, 0, 0, 1.0], [1, .1, 0, 0, 2], [1, .2, 0, 0, 3], [0.5, .3, 0, 0, 4], [2, .4, .1, .2, 0]], float)
    U = np.array([[.1, .2], [.2, .3], [.3, .4], [.4, .5]])
    L = M.TrajectoryLoader(X, U)
    tab = P.RefTable(X, U)
    assert L.s_max == tab.s_max == 2.0
    for s in (-1.0, 0.0, 0.5, 1.0, 1.000005, 1.00001, 1.5, 1.99, 2.0, 3.0):
        assert np.array_equal(L.get_state(s), tab.get_state(s))
        assert np.array_equal(L.get_control(s), tab.get_control(s))
    with pytest.raises(ValueError):
        M.TrajectoryLoader(np.zeros((3, 4)), np.zeros((2, 2)))
    with pytest.raises(FileNotFoundError):
        M.TrajectoryLoader("/nonexistent/file.json")


def test_loader_reads_reference_json_format(tmp_path):
    import json
    import safe_autonomous_driving_mpc_b200 as M
    z = np.load(traj_path(1))
    p = tmp_path / "t.json"
    p.write_text(json.dumps({"X": z["X"].tolist(), "U": z["U"].tolist(), "S": z["S"].tolist()}))
    L = M.TrajectoryLoader(str(p))
    assert np.array_equal(L.X_ref, z["X"]) and np.array_equal(L.U_ref, z["U"])


def test_fsm_matches_reference_log():
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import environment as E
    for i, sc in ((2, E.SCENARIO_TRAJECTORY2), (3, E.SCENARIO_TRAJECTORY3)):
        z = golden(f"closed_loop_traj{i}")
        fsm = M.ObstaclesFSM(True, True, scenario=sc)
        for t in range(len(z["hist_u"])):
            obs, tl = fsm.update(0.2, z["hist_x"][t, 0], z["hist_x"][t, 4])
            assert len(obs) == z["n_obs"][t]
            for k, o in enumerate(obs):
                assert (o["s"], o["v"]) == (z["obs_sv"][t, k, 0], z["obs_sv"][t, k, 1])
            assert tl == str(z["hist_tl"][t])


def test_no_cpu_fallback_without_gpu():
    """Without a GPU the solver context must refuse to exist.  Runs in a child process with every device hidden
    (CUDA_VISIBLE_DEVICES=""), so that it means the same on a machine with a GPU."""
    import subprocess
    import sys
    code = ("import sys\n"
            "sys.path.insert(0, sys.argv[1])\n"
            "import safe_autonomous_driving_mpc_b200 as M\n"
            "L = M.TrajectoryLoader(sys.argv[2])\n"
            "try:\n"
            "    M.BatchedTracker(L)\n"
            "except M._lib.MpcbError as e:\n"
            "    print('refused:', e)\n"
            "    sys.exit(0)\n"
            "sys.exit('a solver context was created without a visible GPU')\n")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", code, ROOT, traj_path(1)], env=env, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "refused:" in r.stdout, r.stdout + r.stderr


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "safe-autonomous-driving-mpc_b200")
    for dirpath, _d, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("converged-oracle", ""), f"{f} mentions oracle/"


def test_integration_stub_struct_matches_library():
    """the ctypes mirror printed in INTEGRATION.md must stay in step with struct mpcb_params"""
    import re
    from safe_autonomous_driving_mpc_b200 import _lib
    src = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    m = re.search(r"class Params\(C\.Structure\):.*?\n\n", src, re.S)
    ns = {"C": C}
    exec(m.group(0), ns)
    assert C.sizeof(ns["Params"]) == _lib.load().mpcb_sizeof_params()
    assert [f[0] for f in ns["Params"]._fields_] == [f[0] for f in _lib.Params._fields_]


def test_table_binary_cache_roundtrip(tmp_path):
    """JSON/npz -> table -> .mpct -> table: bit-identical inputs and lookups; a damaged file is rejected."""
    import safe_autonomous_driving_mpc_b200 as M
    from safe_autonomous_driving_mpc_b200 import _lib
    L = M.TrajectoryLoader(traj_path(2))
    p = str(tmp_path / "t2.mpct")
    L.save_binary(p)
    L2 = M.TrajectoryLoader(p)
    assert np.array_equal(L2.X_ref, L.X_ref) and np.array_equal(L2.U_ref, L.U_ref) and L2.s_max == L.s_max
    for s in (-3.0, 0.0, 17.3, 640.123, L.s_max - 1e-9, L.s_max, L.s_max + 5):
        assert np.array_equal(L2.get_state(s), L.get_state(s)) and np.array_equal(L2.get_control(s), L.get_control(s))
    raw = bytearray(open(p, "rb").read())
    raw[0] ^= 0xFF
    bad = str(tmp_path / "bad.mpct")
    open(bad, "wb").write(raw)
    with pytest.raises(_lib.MpcbError):
        M.TrajectoryLoader(bad)
    open(bad, "wb").write(open(p, "rb").read()[:-8])          # truncated
    with pytest.raises(_lib.MpcbError):
        M.TrajectoryLoader(bad)
