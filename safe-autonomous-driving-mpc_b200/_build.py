"""Build libmpcb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("MPCB_LIB") or os.path.join(HERE, "libmpcb200.so")   # MPCB_LIB: development variants
SOURCES = ["mpcb_api.cu", "mpcb_planner.cu", "mpcb_sim.cu"]
HEADERS = ["mpcb_device.cuh", "mpcb_solver.cuh", "mpcb_planner.cuh", "mpcb_internal.h", "mpcb_coop.cuh", "mpcb_params.h",
           "mpcb_philox.cuh"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libmpcb200.so cannot be built")


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(ROOT, "include", "mpcb200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """Compile csrc/*.cu -> libmpcb200.so.  Returns the library path."""
    if out is None and not force and not stale():
        return LIB
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-Xptxas", "-v", "-I", os.path.join(ROOT, "include"), "-I", CSRC, "-shared", "-Xcompiler", "-fPIC",
           "-o", out or LIB] + ["-D" + d for d in defines] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libmpcb200.so")
    if out is None:
        with open(os.path.join(HERE, "build_ptxas.log"), "w") as f:
            f.write(res.stderr)
    return out or LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
