"""Host-side mirror of the reference's tracker interface on top of the C ABI.

``TrajectoryLoader``  mirrors trajectory_loader.py:13-30, :64-102 (table part only; the global-pose
                      reconstruction :32-62 is animation-only and out of scope).
``BatchedTracker``    mirrors TrajectoryTracker (trajectory_tracking.py:8-263): same constructor argument, same
                      attributes, ``solve(x0, obstacles)`` with the same return tuple, plus ``solve_batch``.

numpy is used for host arrays; torch (optional) only to hand device tensors / streams to the library.
"""
import ctypes as C
import json
import time

import numpy as np

from . import _lib
from ._lib import Params as TrackerParams, check


def _dp(a):
    return a.ctypes.data_as(C.c_void_p)


class TrajectoryLoader:
    """Reference-signal table.  Accepts the reference's JSON format ({'X','U','S'}), an .npz with the same
    keys, or arrays."""

    def __init__(self, source, U=None):
        if isinstance(source, str) and source.endswith(".mpct"):      # binary cache written by save_binary
            lib = _lib.load()
            h = C.c_void_p()
            check(lib.mpcb_table_load(C.byref(h), source.encode()), "mpcb_table_load")
            K, KU = lib.mpcb_table_knots(h), lib.mpcb_table_control_knots(h)
            self.X_ref = np.empty((K, 5))
            self.U_ref = np.empty((KU, 2))
            check(lib.mpcb_table_raw(h, _dp(self.X_ref), _dp(self.U_ref)))
            self._h, self._lib = h, lib
            self.s_max = float(lib.mpcb_table_s_max(h))
            return
        if isinstance(source, str):
            if source.endswith(".npz"):
                z = np.load(source)
                X, U = z["X"], z["U"]
            else:
                try:
                    with open(source, "r") as f:
                        data = json.load(f)
                except FileNotFoundError:
                    raise FileNotFoundError(f"File not found : {source}.")
                X, U = np.array(data["X"]), np.array(data["U"])
        else:
            X = source
        self.X_ref = np.ascontiguousarray(X, dtype=np.float64)
        self.U_ref = np.ascontiguousarray(U, dtype=np.float64)
        if self.X_ref.ndim != 2 or self.X_ref.shape[1] != 5 or self.U_ref.ndim != 2 or self.U_ref.shape[1] != 2:
            raise ValueError("X must be (K,5) and U (K-1,2)")
        lib = _lib.load()
        h = C.c_void_p()
        check(lib.mpcb_table_create(C.byref(h), self.X_ref.ctypes.data_as(_lib.c_double_p), self.X_ref.shape[0],
                                    self.U_ref.ctypes.data_as(_lib.c_double_p), self.U_ref.shape[0]),
              "mpcb_table_create")
        self._h = h
        self._lib = lib
        self.s_max = float(lib.mpcb_table_s_max(h))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.mpcb_table_destroy(h)
            self._h = None

    def save_binary(self, path):
        """Write the packed table cache (``.mpct``); ``TrajectoryLoader(path)`` reads it back."""
        check(self._lib.mpcb_table_save(self._h, str(path).encode()), "mpcb_table_save")

    def get_state(self, s):
        out = (C.c_double * 5)()
        check(self._lib.mpcb_table_get_state(self._h, float(s), out))
        return np.array(out[:])

    def get_control(self, s):
        out = (C.c_double * 2)()
        check(self._lib.mpcb_table_get_control(self._h, float(s), out))
        return np.array(out[:])


class PinnedBuffer:
    """numpy view over page-locked host memory from mpcb_host_alloc."""

    def __init__(self, shape, dtype):
        lib = _lib.load()
        self._lib = lib
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        check(lib.mpcb_host_alloc(C.byref(p), max(nbytes, 1)), "mpcb_host_alloc")
        self._p = p
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        p = getattr(self, "_p", None)
        if p:
            self._lib.mpcb_host_free(p)
            self._p = None


class BatchedTracker:
    """Drop-in for the reference's TrajectoryTracker, running on one B200.

    Same attributes as trajectory_tracking.py:12-47; ``solve`` has the reference's signature and return
    tuple so the object can be passed to the reference's own ``run_simulation``.

    ``X_ref`` may also be a sequence of up to ``MAX_ROUTES`` loaders: the tracker then holds one route per loader
    (``routes``, ``n_routes``), ``solve_batch(..., route=)`` and ``BatchedSimulation(..., route=)`` pick a route per
    problem or vehicle, and every other call runs on route 0.  ``X_ref`` is then the first loader."""

    STATUS_SOLVED, STATUS_MAXITER, STATUS_INFEASIBLE, STATUS_BAD_ROUTE = 0, 1, 2, 3
    MAX_ROUTES = 16

    def __init__(self, X_ref=None, device=0, **solver_overrides):
        routes = tuple(X_ref) if isinstance(X_ref, (list, tuple)) else ((X_ref,) if X_ref is not None else ())
        if isinstance(X_ref, (list, tuple)) and not 1 <= len(routes) <= self.MAX_ROUTES:
            raise ValueError(f"a tracker holds 1 to {self.MAX_ROUTES} routes, got {len(routes)}")
        X_ref = routes[0] if routes else None
        lib = _lib.load()
        self._lib = lib
        p = TrackerParams()
        check(lib.mpcb_default_params(C.byref(p)))
        for k, v in solver_overrides.items():
            if not hasattr(p, k):
                raise TypeError(f"unknown parameter {k!r}")
            setattr(p, k, v)
        self.params = p
        self.X_ref = X_ref
        self.routes = routes
        self.n_routes = len(routes)
        # attributes of the reference object (read by run_simulation, sanity checks, plots)
        self.dt = p.dt
        self.N = p.N
        self.u_min = np.array(p.u_min[:])
        self.u_max = np.array(p.u_max[:])
        self.vehicle_radius = p.vehicle_radius
        self.w_d, self.w_o, self.w_v, self.w_u1, self.w_u2 = p.w_d, p.w_o, p.w_v, p.w_u1, p.w_u2
        self.obstacle_safety_distance = p.obstacle_safety_distance
        self.max_time_2_obs = p.max_time_2_obs
        self.wheelbase = p.wheelbase
        self.lane_width = p.lane_width
        self.safe_lane_margin = p.safe_lane_margin
        self.device = device
        self._h = None
        if len(routes) == 1:
            h = C.c_void_p()
            check(lib.mpcb_create(C.byref(h), C.byref(p), X_ref._h, int(device)), "mpcb_create")
            self._h = h
        elif routes:
            h = C.c_void_p()
            tabs = (C.c_void_p * len(routes))(*[L._h for L in routes])
            check(lib.mpcb_create_routes(C.byref(h), C.byref(p), tabs, len(routes), int(device)), "mpcb_create_routes")
            self._h = h
        self._pin = {}
        self.last_status = None
        self.last_iters = None

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.mpcb_destroy(h)
            self._h = None

    # ---- reference API ---------------------------------------------------------------------------
    def dynamics(self, x, u, k_ref):
        """trajectory_tracking.py:50-67 (host-side plant model used by run_simulation's Euler step)."""
        s, d, o, k, v = x
        return np.array([v, v * o, v * (k - k_ref), u[0], u[1]])

    def unpack(self, U_flat):
        return np.asarray(U_flat).reshape(self.N, 2)

    @staticmethod
    def pack(U):
        return np.asarray(U).ravel()

    def _need(self):
        if self._h is None:
            raise _lib.MpcbError("tracker was built without a reference table (X_ref=None): attributes only")
        return self._h

    def solve(self, x0, obstacles):
        """Same contract as TrajectoryTracker.solve (trajectory_tracking.py:213-263): returns
        (U*[0] (2,), predict(x0, U*) (6,5), seconds).  Solver flags are left in ``last_status`` /
        ``last_iters``."""
        x0a = np.ascontiguousarray(x0, dtype=np.float64).reshape(1, 5)
        obs = np.zeros((1, 2, 2))
        n = min(len(obstacles), 2)
        for k in range(n):
            o = obstacles[k]
            obs[0, k] = (o["s"], o["v"]) if isinstance(o, dict) else (o[0], o[1])
        t0 = time.time()
        r = self.solve_batch_host(x0a, obs, np.array([n], dtype=np.int32))
        sec = time.time() - t0
        self.last_status = int(r["status"][0])
        self.last_iters = r["iters"][0].copy()
        return r["U"][0, 0].copy(), r["Xpred"][0].copy(), sec

    # ---- batched API -----------------------------------------------------------------------------
    def _pinned(self, key, shape, dtype):
        cur = self._pin.get(key)
        if cur is None or cur.array.shape != tuple(shape):
            cur = PinnedBuffer(tuple(shape), dtype)
            self._pin[key] = cur
        return cur.array

    def solve_batch_host(self, x0, obs_sv, n_obs, pinned_out=True):
        """Host arrays in, host arrays out (copies included).  Returns dict of numpy arrays."""
        h = self._need()
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        B = x0.shape[0]
        obs_sv = np.ascontiguousarray(obs_sv, dtype=np.float64).reshape(B, 2, 2)
        n_obs = np.ascontiguousarray(n_obs, dtype=np.int32).reshape(B)
        mk = (lambda k, s, d: self._pinned(k, s, d)) if pinned_out else (lambda k, s, d: np.empty(s, d))
        out = dict(U=mk("U", (B, 5, 2), np.float64), Xpred=mk("X", (B, 6, 5), np.float64),
                   obj=mk("obj", (B,), np.float64), status=mk("st", (B,), np.int32),
                   iters=mk("it", (B, 2), np.int32), cmin=mk("cm", (B,), np.float64),
                   active=mk("ac", (B,), np.uint64))
        check(self._lib.mpcb_solve_batch_host(h, B, _dp(x0), _dp(obs_sv), _dp(n_obs), _dp(out["U"]), _dp(out["Xpred"]),
                                              _dp(out["obj"]), _dp(out["status"]), _dp(out["iters"]),
                                              _dp(out["cmin"]), _dp(out["active"])), "mpcb_solve_batch_host")
        return out

    def solve_batch_host_u0(self, x0, obs_sv, n_obs, want_obj=False, pinned_out=True):
        """Closed-loop form: host arrays in, only ``U*[0]`` [B,2], ``status`` [B] (and ``obj`` [B]) out -- what
        run_simulation consumes (trajectory_tracking.py:401-406) -- 20-28 bytes per solve over PCIe instead of 356."""
        h = self._need()
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        B = x0.shape[0]
        obs_sv = np.ascontiguousarray(obs_sv, dtype=np.float64).reshape(B, 2, 2)
        n_obs = np.ascontiguousarray(n_obs, dtype=np.int32).reshape(B)
        mk = (lambda k, s, d: self._pinned(k, s, d)) if pinned_out else (lambda k, s, d: np.empty(s, d))
        out = dict(u0=mk("u0", (B, 2), np.float64), status=mk("st0", (B,), np.int32))
        if want_obj:
            out["obj"] = mk("obj0", (B,), np.float64)
        check(self._lib.mpcb_solve_batch_host_u0(h, B, _dp(x0), _dp(obs_sv), _dp(n_obs), _dp(out["u0"]),
                                                 _dp(out["status"]), _dp(out["obj"]) if want_obj else None),
              "mpcb_solve_batch_host_u0")
        return out

    def solve_batch_host_async(self, x0, obs_sv, n_obs, out):
        """Asynchronous host call (mpcb_solve_batch_host_async): ``x0`` [B,5] f64, ``obs_sv`` [B,2,2] f64, ``n_obs`` [B] i32
        and the arrays of ``out`` (any of U, Xpred, obj, status, iters, cmin, active, u0; U or u0 required) must be
        C-contiguous page-locked arrays (``PinnedBuffer``) and stay untouched until ``wait()``.  One batch in flight per
        tracker; use several trackers to overlap copies and kernels of consecutive batches."""
        h = self._need()
        B = x0.shape[0]
        for a in (x0, obs_sv, n_obs, *out.values()):
            assert a.flags["C_CONTIGUOUS"]
        assert x0.dtype == np.float64 and obs_sv.dtype == np.float64 and n_obs.dtype == np.int32
        g = lambda k: _dp(out[k]) if k in out else None   # noqa: E731
        check(self._lib.mpcb_solve_batch_host_async(h, B, _dp(x0), _dp(obs_sv), _dp(n_obs), g("U"), g("Xpred"), g("obj"),
                                                    g("status"), g("iters"), g("cmin"), g("active"), g("u0")),
              "mpcb_solve_batch_host_async")
        return out

    def wait(self):
        check(self._lib.mpcb_wait(self._need()), "mpcb_wait")

    def solve_batch(self, x0, obs_sv, n_obs, out=None, stream=None, route=None):
        """Device tensors in, device tensors out (torch used only for memory + stream hand-off).
        Asynchronous on ``stream`` (default: torch's current stream).  ``route``: device int32 tensor [B], problem b on
        ``routes[route[b]]`` (None: route 0); a problem whose route is out of range gets ``STATUS_BAD_ROUTE`` and NaN."""
        import torch
        B = x0.shape[0]
        if route is not None and not (isinstance(route, torch.Tensor) and route.dtype == torch.int32
                                      and tuple(route.shape) == (B,) and route.is_contiguous()):
            raise ValueError(f"route must be a contiguous int32 tensor of shape ({B},)")
        h = self._need()
        dev = x0.device
        assert x0.dtype == torch.float64 and obs_sv.dtype == torch.float64 and n_obs.dtype == torch.int32
        assert x0.is_contiguous() and obs_sv.is_contiguous() and n_obs.is_contiguous()
        if out is None:
            out = dict(U=torch.empty((B, 5, 2), dtype=torch.float64, device=dev),
                       Xpred=torch.empty((B, 6, 5), dtype=torch.float64, device=dev),
                       obj=torch.empty((B,), dtype=torch.float64, device=dev),
                       status=torch.empty((B,), dtype=torch.int32, device=dev),
                       iters=torch.empty((B, 2), dtype=torch.int32, device=dev),
                       cmin=torch.empty((B,), dtype=torch.float64, device=dev),
                       active=torch.empty((B,), dtype=torch.int64, device=dev))
        st = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        check(self._lib.mpcb_solve_batch_routes(h, B, x0.data_ptr(), obs_sv.data_ptr(), n_obs.data_ptr(),
                                                route.data_ptr() if route is not None else None,
                                                out["U"].data_ptr(), out["Xpred"].data_ptr(), out["obj"].data_ptr(),
                                                out["status"].data_ptr(), out["iters"].data_ptr(), out["cmin"].data_ptr(),
                                                out["active"].data_ptr(), C.c_void_p(st)), "mpcb_solve_batch_routes")
        return out

    def eval_batch(self, x0, U, obs_sv, n_obs):
        """predict / cost / constraints / linearisation / warm start on the GPU for host arrays (tests)."""
        h = self._need()
        lib = self._lib
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        B = x0.shape[0]
        U = np.ascontiguousarray(U, dtype=np.float64).reshape(B, 10)
        obs_sv = np.ascontiguousarray(obs_sv, dtype=np.float64).reshape(B, 2, 2)
        n_obs = np.ascontiguousarray(n_obs, dtype=np.int32).reshape(B)
        host_in = [x0, U, obs_sv, n_obs]
        host_out = dict(Xpred=np.empty((B, 6, 5)), cost=np.empty(B), cons=np.empty((B, 45)), lin=np.empty((B, 150)),
                        warm=np.empty((B, 10)))
        dptr = []
        try:
            for a in host_in + list(host_out.values()):
                p = C.c_void_p()
                check(lib.mpcb_device_alloc(h, C.byref(p), a.nbytes), "mpcb_device_alloc")
                dptr.append(p)
            for a, p in zip(host_in, dptr):
                check(lib.mpcb_memcpy_h2d(h, p, _dp(a), a.nbytes))
            check(lib.mpcb_eval_batch(h, B, *dptr, None), "mpcb_eval_batch")
            for a, p in zip(host_out.values(), dptr[4:]):
                check(lib.mpcb_memcpy_d2h(h, _dp(a), p, a.nbytes))   # cudaMemcpy synchronises the null stream
        finally:
            for p in dptr:
                lib.mpcb_device_free(h, p)
        return host_out

    def last_kernel_ms(self):
        ms = C.c_float()
        check(self._lib.mpcb_last_kernel_ms(self._need(), C.byref(ms)))
        return ms.value

    def last_pass_ms(self):
        """(first-pass ms, second-pass ms, problems handled by the second pass) of the last solve."""
        a, b, n = C.c_float(), C.c_float(), C.c_int()
        check(self._lib.mpcb_last_pass_ms(self._need(), C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def last_call_used_coop(self):
        """True when the first pass of the last solve ran one warp per problem (small batches)."""
        return self._lib.mpcb_last_first_pass_shape(self._need()) == 1

    def launch_count(self):
        return int(self._lib.mpcb_launch_count(self._need()))

    def measure_fp64_peak(self):
        tf, ms = C.c_double(), C.c_float()
        check(self._lib.mpcb_measure_fp64_peak(self._need(), C.byref(tf), C.byref(ms)), "mpcb_measure_fp64_peak")
        return tf.value, ms.value
