"""Development: build kernel-configuration variants of libmpcb200.so (build/variants/, git-ignored) and time them.
    python tools/variants.py build            (here, no GPU)
    python tools/variants.py run              (on the GPU box: one subprocess per variant)"""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "build", "variants")
VARIANTS = {
    "T96_C3_M5": ["MPCB_SOLVE_THREADS=96", "MPCB_SOLVE_CTAS=3", "MPCB_STORE_MASK=5"],
    "T96_C3_M3": ["MPCB_SOLVE_THREADS=96", "MPCB_SOLVE_CTAS=3", "MPCB_STORE_MASK=3"],
    "T64_C4_M5": ["MPCB_SOLVE_THREADS=64", "MPCB_SOLVE_CTAS=4", "MPCB_STORE_MASK=5"],
    "T32_C8_M7": ["MPCB_SOLVE_THREADS=32", "MPCB_SOLVE_CTAS=8", "MPCB_STORE_MASK=7"],
    "T32_C9_M5": ["MPCB_SOLVE_THREADS=32", "MPCB_SOLVE_CTAS=9", "MPCB_STORE_MASK=5"],
    "T128_C1_M189": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=1", "MPCB_STORE_MASK=189"],
    "T64_C2_M189": ["MPCB_SOLVE_THREADS=64", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=189"],
    "T96_C1_M191": ["MPCB_SOLVE_THREADS=96", "MPCB_SOLVE_CTAS=1", "MPCB_STORE_MASK=191"],
    "T64_C2_M191": ["MPCB_SOLVE_THREADS=64", "MPCB_SOLVE_CTAS=1", "MPCB_STORE_MASK=255"],
    "T128_C1_M29": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=1", "MPCB_STORE_MASK=29"],
    "T192_C1_M21": ["MPCB_SOLVE_THREADS=192", "MPCB_SOLVE_CTAS=1", "MPCB_STORE_MASK=21"],
    "T128_C2_M13": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=13"],
    "T128_C2_M9": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=9"],
    "T128_C2_M37": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=37"],
    "T128_C2_M133": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=133"],
    "T64_C4_M7": ["MPCB_SOLVE_THREADS=64", "MPCB_SOLVE_CTAS=4", "MPCB_STORE_MASK=7"],
    "T128_C2_M3": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=3"],
    "T128_C2_M5": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=5"],
    "T128_C2_M135": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=135"],
    "T256_C1_M7": ["MPCB_SOLVE_THREADS=256", "MPCB_SOLVE_CTAS=1", "MPCB_STORE_MASK=7"],
    "T96_C3_M1": ["MPCB_SOLVE_THREADS=96", "MPCB_SOLVE_CTAS=3", "MPCB_STORE_MASK=1"],
    "COOP2": ["MPCB_COOP_CTAS=2"],
    "COOP3": ["MPCB_COOP_CTAS=3"],
    "COOP4": ["MPCB_COOP_CTAS=4"],
    "T128_C2_M7": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=7"],
    "T128_C2_M7_W": ["MPCB_SOLVE_THREADS=128", "MPCB_SOLVE_CTAS=2", "MPCB_STORE_MASK=7", "MPCB_WARP_UNIFORM=1"],
    "T64_C4_M7_W": ["MPCB_SOLVE_THREADS=64", "MPCB_SOLVE_CTAS=4", "MPCB_STORE_MASK=7", "MPCB_WARP_UNIFORM=1"],
    "T32_C8_M7_W": ["MPCB_SOLVE_THREADS=32", "MPCB_SOLVE_CTAS=8", "MPCB_STORE_MASK=7", "MPCB_WARP_UNIFORM=1"],
    "T256_C1_M7_W": ["MPCB_SOLVE_THREADS=256", "MPCB_SOLVE_CTAS=1", "MPCB_STORE_MASK=7", "MPCB_WARP_UNIFORM=1"],
}
if sys.argv[1] == "build":
    import importlib
    b = importlib.import_module("safe_autonomous_driving_mpc_b200._build")
    os.makedirs(OUT, exist_ok=True)
    names = sys.argv[2:] or list(VARIANTS)
    for n in names:
        lib = os.path.join(OUT, n + ".so")
        res = subprocess.run([b.nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
                              "-Xptxas", "-v", "-I", os.path.join(ROOT, "include"), "-I", b.CSRC, "-shared", "-Xcompiler",
                              "-fPIC", "-o", lib] + ["-D" + d for d in VARIANTS[n]] +
                             [os.path.join(b.CSRC, s) for s in b.SOURCES], capture_output=True, text=True)
        info = [l for l in res.stderr.splitlines() if "_kernel" in l or "stack frame" in l or "Used" in l]
        sel = []
        for i, l in enumerate(info):
            if ("solve_kernel" in l or "coop_kernel" in l) and "Function properties" in l:
                sel += [info[i + 1].strip(), info[i + 2].strip()]
        print(n, res.returncode, " | ".join(sel))
        if res.returncode != 0:
            print(res.stderr[-2000:])
else:
    for n in (sys.argv[2:] or list(VARIANTS)):
        env = dict(os.environ, MPCB_LIB=os.path.join(OUT, n + ".so"))
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", os.environ.get("VTOOL", "gpu_quick.py"))], env=env, capture_output=True, text=True)
        lines = r.stdout.strip().splitlines()
        print(n, " || ".join(l for l in lines if l.startswith("B=")) if os.environ.get("VTOOL") else (lines[-1] if lines else r.stderr[-500:]))
