"""Development: problems entering each round kernel of the first pass, per obstacle class, read back from the device
(library built with -DMPCB_ROUND_STATS, MPCB_LIB set), on the benchmark's seeded 65,536-problem set.
    python tools/gpu_round_counts.py build     (cross-compiles build/libmpcb200_rounds.so)
    python tools/gpu_round_counts.py           (on the GPU box)"""
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
LIB = os.path.join(ROOT, "build", "libmpcb200_rounds.so")
if len(sys.argv) > 1 and sys.argv[1] == "build":
    import importlib
    b = importlib.import_module("safe_autonomous_driving_mpc_b200._build")
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    print(b.build(defines=["MPCB_ROUND_STATS"], out=LIB))
    sys.exit(0)
if os.environ.get("MPCB_LIB") != LIB:
    sys.exit(subprocess.run([sys.executable, __file__], env=dict(os.environ, MPCB_LIB=LIB)).returncode)
import numpy as np
import torch
import safe_autonomous_driving_mpc_b200 as M
from oracle import tracker_port as P

lib = M._lib.load(build_if_missing=False)
traj = os.path.join(ROOT, "data", "trajectory3.npz")
T = M.BatchedTracker(M.TrajectoryLoader(traj))
x0, obs, n = P.monte_carlo_problems(P.RefTable.from_npz(traj), 65536)
d = [torch.from_numpy(a).cuda() for a in (x0, obs, n)]
out = T.solve_batch(*d)
torch.cuda.synchronize()
cnt = (C.c_ulonglong * 48)()
lib.mpcb_debug_round_counts(cnt, 1)
T.solve_batch(*d, out=out)
torch.cuda.synchronize()
lib.mpcb_debug_round_counts(cnt, 0)
c = np.array(cnt[:], dtype=np.int64).reshape(16, 3)
print("problems per class", np.bincount(n, minlength=3).tolist(), "robust pass", T.last_pass_ms()[2])
for r in range(16):
    if c[r].sum():
        print(f"entering round {r + 1}: {int(c[r].sum())} (class 0/1/2: {c[r].tolist()})")
