// mpcb_device.cuh -- device-side model of the tracking MPC (one thread = one problem).
//
// What is computed follows the reference formulation exactly:
//   rollout      trajectory_tracking.py:87-114   (explicit Euler, k_ref looked up at the predicted s)
//   cost         trajectory_tracking.py:116-152
//   constraints  trajectory_tracking.py:155-211  (row order kept for the outputs)
//   warm start   trajectory_tracking.py:223-246
//   table lookup trajectory_loader.py:86-102 + scipy interp1d linear rule (SURVEY.md A.2)
// How it is computed is new: exact forward sensitivities instead of finite differences, a Gauss-Newton
// linearise->QP loop instead of SLSQP, and an OSQP-style ADMM (sigma = 0, single-vector state, per-row
// step-size ladder) for the QP.  Everything is fp64.
#pragma once
#include <math.h>
#ifdef __CUDACC__
#include <cuda_runtime.h>
#define MPCB_HD __host__ __device__ __forceinline__
#define MPCB_D __device__ __forceinline__
#else
// host build: test infrastructure only (tests/hostbuild compiles these headers with g++ to validate the
// algorithm on the CPU; the product library is nvcc-built and has no CPU path)
#define MPCB_HD inline
#define MPCB_D inline
#define __host__
#define __device__
#endif
#if defined(__CUDA_ARCH__)
#define MPCB_LDG(p) __ldg(p)
#else
#define MPCB_LDG(p) (*(p))
#endif

// Checked build (-DMPCB_CHECKED, tools/gpu_checked.py): bounds of every table segment, work-list slot and class-list
// slot are asserted on the device.  compute-sanitizer is closed on the GPU pool this was developed on, so these asserts,
// small cases and the parity tests are the memory-safety evidence (profiles/README.md).
#if defined(MPCB_CHECKED)
#include <assert.h>
#define MPCB_ASSERT(c) assert(c)
#else
#define MPCB_ASSERT(c) ((void)0)
#endif

namespace mpcb {

constexpr int NH = 5;     // horizon
constexpr int NV = 10;    // decision variables
constexpr int NTRI = 55;  // packed lower triangle of a 10x10 symmetric matrix
constexpr int MAXRUNG = 8;
constexpr double BIG = 1e30;

__host__ __device__ constexpr int tri(int i, int j) { return i * (i + 1) / 2 + j; }  // i >= j

struct DevTable {
  const double* s;   // [K]   strictly increasing knots
  const double* y;   // [K][4] d,o,k,v
  const double* u;   // [Ku][2] u1,u2 (defined on the first Ku knots)
  int K, Ku;
  double s_max;
  double last[4];    // X_ref[-1][1:5], returned for s >= s_max
  // optional bucket index over [s[0], s[K-1]]: lut[b] = segment of the left edge of bucket b (nullptr: binary search)
  const int* lut;
  int lut_n;
  double lut_s0, lut_scale;
  // optional 1 / (s[i] - s[i-1]) per segment (IEEE division done once when the table is built): the device lookups of
  // the tracking path multiply by it instead of dividing three times per lookup (weights differ by at most one ulp
  // from the reference's quotient form; the host build and the planner keep the divisions)
  const double* sinv;
};

#ifndef MPCB_MAX_ROUTES
#define MPCB_MAX_ROUTES 16   // include/mpcb200.h
#endif
// The tables of a handle, handed to the kernels as one grid-constant parameter: a problem on route r runs on t[r].
struct DevTables {
  DevTable t[MPCB_MAX_ROUTES];
  int n;
};
static_assert(sizeof(DevTables) <= 2048, "DevTables must stay well inside the 4 KB a kernel's parameters may take");

// Route of problem b: route[b] (route == nullptr: 0 for every problem), or -1 when route[b] is outside [0, n).  Every
// kernel that reads a caller's route array goes through here, so no route from outside the library becomes a table index.
MPCB_HD int problem_route(const int* __restrict__ route, int b, int n) {
  if (!route) return 0;
  const int r = route[b];
  return (r >= 0 && r < n) ? r : -1;
}

#ifdef __CUDACC__
// Slot of this thread in a list (warp-aggregated append to counter; every lane of the warp calls it), -1 if !pred.
__device__ __forceinline__ int warp_append(bool pred, int* counter) {
  const unsigned m = __ballot_sync(0xffffffffu, pred);
  if (m == 0u) return -1;
  const unsigned lane = threadIdx.x & 31u;
  const int leader = __ffs(m) - 1;
  int base = 0;
  if ((int)lane == leader) base = atomicAdd(counter, __popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  return pred ? base + __popc(m & ((1u << lane) - 1u)) : -1;
}
#endif

// Step-size policy of the ADMM machinery (mpcb_solver.cuh).
struct Policy {
  double lad[MAXRUNG];        // step-size ladder
  double lad_ratio[MAXRUNG];  // lad[k-1]/lad[k] (k>=1): rescale of (v - z) when a row moves up one rung
  double relax;               // ADMM over-relaxation alpha
  int n_rung, e_init;
  int hysteresis;             // a row changes rung only after two consecutive segments of the same activity
  int drop_all;               // inactive rows fall to rung 0 at once
  int max_segments, segment_iters;
};

struct DevParams {
  double h;
  double umin[2], umax[2];
  double wd, wo, wv, wu[2];
  double obs_safe, tgap;
  double sld;          // lane_width/2 - vehicle_radius - safe_lane_margin
  double alpha_lane[3];// 0, wheelbase/2, wheelbase
  double brake_lookahead, brake_guess;
  int max_rounds, fast_max_rounds;
  int thread_max_rounds, thread_max_segments;   // two-level policy caps inside the thread-per-problem kernel
  int max_fail_rounds; // robust pass: give up after this many rounds whose QP did not close
  int fast_fail_rounds;// first pass (thread kernel): rounds whose QP did not close that are tolerated (the ADMM state
                       // carries over, so the active-set search simply continues on the next linearisation)
  Policy pol[2];       // [0] robust ladder, [1] two-level (first pass)
  double eps_p, eps_d, eps_inf, step_tol, feas_tol;
  double qp_forcing, qp_eps_loose;   // robust pass: QP tolerance of a round = clamp(forcing * previous SQP step, eps, loose)
  double inrm_v[NH], inrm_r1[NH], inrm_r2[NH];  // 1/max(|a|^2, floor) of the constant-coefficient rows
};

// ------------------------------------------------------------------------------------------------
// Reference-signal table.  searchsorted(side='left') clipped to [1, K-1], then the two-term formula.
// ------------------------------------------------------------------------------------------------
MPCB_HD int seg_index(const double* __restrict__ s, int K, double x) {
  int lo = 0, hi = K;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (MPCB_LDG(s + mid) < x) lo = mid + 1; else hi = mid;
  }
  return (lo < 1) ? 1 : ((lo > K - 1) ? K - 1 : lo);
}

// get_state(s)[1:5] and the slope of each column on the bracketing segment
MPCB_HD void lookup_state(const DevTable& T, double s, double (&val)[4], double (&slope)[4]) {
  if (s >= T.s_max) {
#pragma unroll
    for (int c = 0; c < 4; ++c) { val[c] = T.last[c]; slope[c] = 0.0; }
    return;
  }
  const int i = seg_index(T.s, T.K, s);
  const double x_lo = MPCB_LDG(T.s + i - 1), x_hi = MPCB_LDG(T.s + i);
  const double inv = 1.0 / (x_hi - x_lo);
  const double wl = (s - x_lo) / (x_hi - x_lo), wr = (x_hi - s) / (x_hi - x_lo);
  double ylo[4], yhi[4];
#if defined(__CUDA_ARCH__)
  {
    const double2* yl = reinterpret_cast<const double2*>(T.y + 4 * (i - 1));
    const double2 l0 = __ldg(yl), l1 = __ldg(yl + 1), h0 = __ldg(yl + 2), h1 = __ldg(yl + 3);
    ylo[0] = l0.x; ylo[1] = l0.y; ylo[2] = l1.x; ylo[3] = l1.y;
    yhi[0] = h0.x; yhi[1] = h0.y; yhi[2] = h1.x; yhi[3] = h1.y;
  }
#else
  for (int c = 0; c < 4; ++c) { ylo[c] = T.y[4 * (i - 1) + c]; yhi[c] = T.y[4 * i + c]; }
#endif
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    val[c] = wl * yhi[c] + wr * ylo[c];
    slope[c] = (yhi[c] - ylo[c]) * inv;
  }
}

// Same as lookup_state, with the table segment remembered between calls: consecutive predicted positions (and the
// same step in the next linearisation round) land in the same or a neighbouring segment, so a short walk from the
// previous index replaces the binary search.  `hint` is updated.
MPCB_HD int seg_index_hint(const double* __restrict__ sa, int K, double x, int& hint) {
  int i = hint < 1 ? 1 : (hint > K - 1 ? K - 1 : hint);
  bool found = false;
  for (int t = 0; t < 6 && !found; ++t) {
    if (i < K - 1 && MPCB_LDG(sa + i) < x) ++i;
    else if (i > 1 && MPCB_LDG(sa + i - 1) >= x) --i;
    else found = true;
  }
  if (!found) i = seg_index(sa, K, x);
  hint = i;
  return i;
}

// The knots and rows of the hinted segment are loaded speculatively, all at once; when the hint is right (the usual
// case) the lookup is ONE memory round trip instead of a chain of three (walk, knots, rows).
// seg_index without a previous segment to walk from: the bucket index gives a first guess that is at most a knot or
// two off, the walk of seg_index_hint does the rest (13 dependent loads of the binary search -> 2 or 3).
MPCB_HD int seg_index_cold(const DevTable& T, int K, double x) {
  if (!T.lut) return seg_index(T.s, K, x);
  double t = (x - T.lut_s0) * T.lut_scale;
  t = t > 0.0 ? t : 0.0;                                // also catches NaN
  t = t < (double)(T.lut_n - 1) ? t : (double)(T.lut_n - 1);
  MPCB_ASSERT((int)t >= 0 && (int)t < T.lut_n);
  int hint = MPCB_LDG(T.lut + (int)t);
  return seg_index_hint(T.s, K, x, hint);
}

MPCB_HD void lookup_state_hint(const DevTable& T, double s, double (&val)[4], double (&slope)[4], int& hint) {
  if (s >= T.s_max) {
#pragma unroll
    for (int c = 0; c < 4; ++c) { val[c] = T.last[c]; slope[c] = 0.0; }
    return;
  }
  int i = hint < 1 ? 1 : (hint > T.K - 1 ? T.K - 1 : hint);
  MPCB_ASSERT(i >= 1 && i <= T.K - 1);
  double x_lo = MPCB_LDG(T.s + i - 1), x_hi = MPCB_LDG(T.s + i);
  double ylo[4], yhi[4];
#if defined(__CUDA_ARCH__)
  double inv = __ldg(T.sinv + i);             // speculative like the rest: no load waits for the hint check
#endif
  auto load_rows = [&](int ii) {
#if defined(__CUDA_ARCH__)
    const double2* yl = reinterpret_cast<const double2*>(T.y + 4 * (ii - 1));
    const double2 l0 = __ldg(yl), l1 = __ldg(yl + 1), h0 = __ldg(yl + 2), h1 = __ldg(yl + 3);
    ylo[0] = l0.x; ylo[1] = l0.y; ylo[2] = l1.x; ylo[3] = l1.y;
    yhi[0] = h0.x; yhi[1] = h0.y; yhi[2] = h1.x; yhi[3] = h1.y;
#else
    for (int c = 0; c < 4; ++c) { ylo[c] = T.y[4 * (ii - 1) + c]; yhi[c] = T.y[4 * ii + c]; }
#endif
  };
  load_rows(i);
  if (!((i == T.K - 1 || x_hi >= s) && (i == 1 || x_lo < s))) {   // hint off: walk / search, then load again
    i = seg_index_hint(T.s, T.K, s, hint);
    MPCB_ASSERT(i >= 1 && i <= T.K - 1);
    x_lo = MPCB_LDG(T.s + i - 1);
    x_hi = MPCB_LDG(T.s + i);
#if defined(__CUDA_ARCH__)
    inv = __ldg(T.sinv + i);
#endif
    load_rows(i);
  }
  hint = i;
#if defined(__CUDA_ARCH__)
  const double wl = (s - x_lo) * inv, wr = (x_hi - s) * inv;
#else
  const double inv = 1.0 / (x_hi - x_lo);
  const double wl = (s - x_lo) / (x_hi - x_lo), wr = (x_hi - s) / (x_hi - x_lo);
#endif
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    val[c] = wl * yhi[c] + wr * ylo[c];
    slope[c] = (yhi[c] - ylo[c]) * inv;
  }
}

MPCB_HD void lookup_control(const DevTable& T, double s, double (&u)[2], int& hint) {
  if (s >= T.s_max) { u[0] = 0.0; u[1] = 0.0; return; }
  const int i = (hint > 0) ? seg_index_hint(T.s, T.Ku, s, hint) : (hint = seg_index_cold(T, T.Ku, s));
  MPCB_ASSERT(i >= 1 && i <= T.Ku - 1);
  const double x_lo = MPCB_LDG(T.s + i - 1), x_hi = MPCB_LDG(T.s + i);
#if defined(__CUDA_ARCH__)
  const double inv = __ldg(T.sinv + i);
  const double wl = (s - x_lo) * inv, wr = (x_hi - s) * inv;
#else
  const double wl = (s - x_lo) / (x_hi - x_lo), wr = (x_hi - s) / (x_hi - x_lo);
#endif
  const double ul0 = MPCB_LDG(T.u + 2 * (i - 1)), ul1 = MPCB_LDG(T.u + 2 * (i - 1) + 1);
  const double uh0 = MPCB_LDG(T.u + 2 * i), uh1 = MPCB_LDG(T.u + 2 * i + 1);
  u[0] = wl * uh0 + wr * ul0;
  u[1] = wl * uh1 + wr * ul1;
}

// warm start, trajectory_tracking.py:223-246 (unclipped)
// hints[j] (optional) receives the table segment of the j-th probe position s0 + j h v0, a good first guess for the
// lookups of the rollout.
MPCB_HD void warm_start(const DevTable& T, const DevParams& P, const double (&x0)[5],
                                           const double (&obs)[2][2], int n_obs, double (&U)[NV], int* hints = nullptr) {
  int hint = 0;          // 0: first probe uses the binary search, the following ones walk from it
  double s_cur = x0[0];
  const double v_cur = x0[4];
  bool brake = false;
#pragma unroll
  for (int j = 0; j < NH; ++j) {
#pragma unroll
    for (int k = 0; k < 2; ++k)
      if (k < n_obs && (obs[k][0] - s_cur) < P.brake_lookahead) brake = true;
    double ur[2];
    lookup_control(T, s_cur, ur, hint);
    if (hints) hints[j] = hint;
    U[2 * j] = ur[0];
    U[2 * j + 1] = brake ? P.brake_guess : ur[1];
    s_cur += v_cur * P.h;
  }
}

// the same from reference controls looked up beforehand: ur[j] = get_control(s0 + j h v0) (warp-per-problem kernel,
// where five lanes do the five lookups at once)
MPCB_HD void warm_fill(const DevParams& P, const double (&x0)[5], const double (&obs)[2][2], int n_obs,
                       const double (*ur)[2], double (&U)[NV]) {
  double s_cur = x0[0];
  const double v_cur = x0[4];
  bool brake = false;
#pragma unroll
  for (int j = 0; j < NH; ++j) {
#pragma unroll
    for (int k = 0; k < 2; ++k)
      if (k < n_obs && (obs[k][0] - s_cur) < P.brake_lookahead) brake = true;
    U[2 * j] = ur[j][0];
    U[2 * j + 1] = brake ? P.brake_guess : ur[j][1];
    s_cur += v_cur * P.h;
  }
}

// ------------------------------------------------------------------------------------------------
// Values-only rollout: X[6][5], cost, and constraint rows in the reference's order.
// ------------------------------------------------------------------------------------------------
MPCB_HD void rollout_values(const DevTable& T, const DevParams& P, const double (&x0)[5],
                                               const double (&U)[NV], double (&X)[NH + 1][5], double& cost,
                                               const int* hints = nullptr) {
  int hloc[NH + 1];
#pragma unroll
  for (int j = 0; j <= NH; ++j) hloc[j] = hints ? hints[j] : 1;
#pragma unroll
  for (int c = 0; c < 5; ++c) X[0][c] = x0[c];
  double val[4], slope[4];
  double c_acc = 0.0;
#pragma unroll
  for (int j = 0; j < NH; ++j) {
    const double s = X[j][0], d = X[j][1], o = X[j][2], k = X[j][3], v = X[j][4];
    lookup_state_hint(T, s, val, slope, hloc[j]);
    if (j > 0) {  // tracking terms of step j use the lookup at s_j
      const double rd = d - val[0], ro = o - val[1], rv = v - val[3];
      c_acc += P.wd * (rd * rd);
      c_acc += P.wo * (ro * ro);
      c_acc += P.wv * (rv * rv);
    }
    X[j + 1][0] = s + P.h * v;
    X[j + 1][1] = d + P.h * (v * o);
    X[j + 1][2] = o + P.h * (v * (k - val[2]));
    X[j + 1][3] = k + P.h * U[2 * j];
    X[j + 1][4] = v + P.h * U[2 * j + 1];
  }
  {
    lookup_state_hint(T, X[NH][0], val, slope, hloc[NH]);
    const double rd = X[NH][1] - val[0], ro = X[NH][2] - val[1], rv = X[NH][4] - val[3];
    c_acc += P.wd * (rd * rd);
    c_acc += P.wo * (ro * ro);
    c_acc += P.wv * (rv * rv);
  }
#pragma unroll
  for (int j = 0; j < NH; ++j) {
    c_acc += P.wu[0] * (U[2 * j] * U[2 * j]);
    c_acc += P.wu[1] * (U[2 * j + 1] * U[2 * j + 1]);
  }
  cost = c_acc;
}

// constraint rows of constraints_wrapper (trajectory_tracking.py:171-207) for step j (1-based), written to
// out[0 .. 6+n_obs]; returns the number of rows.
MPCB_HD int constraint_rows(const DevParams& P, const double (&Xj)[5], int j,
                                               const double (&obs)[2][2], int n_obs, double* out) {
  const double s = Xj[0], d = Xj[1], o = Xj[2], v = Xj[4];
  int r = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double val = d + P.alpha_lane[a] * o;
    out[r++] = P.sld - val;
    out[r++] = val + P.sld;
  }
  for (int k = 0; k < n_obs; ++k) {
    const double s_obs = obs[k][0] + obs[k][1] * (j * P.h);
    const double safe = fmax(P.obs_safe, v * P.tgap);
    out[r++] = (s_obs - s) - safe;
  }
  out[r++] = v;
  return r;
}

}  // namespace mpcb
