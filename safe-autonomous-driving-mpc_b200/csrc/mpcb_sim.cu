// mpcb_sim.cu -- batched closed loop on the device (SURVEY.md 8(f1)): the callers either side of the solve path.
//
//   obstacle-set producer   ObstaclesFSM.update            trajectory_tracking.py:330-374
//   plant step              x += dt * dynamics(x, u0, k_ref(s))   trajectory_tracking.py:404-406 (dynamics :50-67)
//   loop condition          while current_s <= s_max - 1.0         trajectory_tracking.py:395
//
// One simulation object holds B vehicles (each with its own scenario constants and FSM state).  A step is three
// launches on one stream -- FSM kernel -> mpcb_solve_batch -> plant kernel -- with no host round trip, so a
// Monte-Carlo of whole drives never leaves the GPU; histories are recorded into device buffers when asked for.  With
// following on (mpcb_sim_set_follow), a key kernel, two radix sorts and a leader kernel come first.
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include <new>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "mpcb200.h"
#include "mpcb_internal.h"

namespace mpcb {

struct DevScenario {          // per vehicle, mirrors ObstaclesFSM.__init__ (:285-308)
  double obs_trigger_s, obs_start_s, obs_v, obs_end_s;
  double tl_pos, tl_trigger_s, tl_stop_duration;
  int dynamic_obstacle, traffic_light;
};

enum { F_OBS_ACTIVE = 1, F_OBS_TRIGGERED = 2, F_TL_GREEN = 4, F_TL_WAITING = 8 };

// Table of vehicle b's route (route == nullptr: route 0).  The routes of a simulation are checked when it is created.
__device__ __forceinline__ const DevTable& vehicle_table(const DevTables& Ts, const int* __restrict__ route, int b) {
  const int r = problem_route(route, b, Ts.n);
  MPCB_ASSERT(r >= 0 && r < Ts.n);
  return Ts.t[r < 0 ? 0 : r];
}

// loop condition (:395): still driving while s <= s_max - 1 of the vehicle's route
__device__ __forceinline__ double stop_s(const DevTables& Ts, const int* __restrict__ route, int b) {
  return vehicle_table(Ts, route, b).s_max - 1.0;
}

// ---- following (mpcb_sim_set_follow): the nearest vehicle ahead on the same route is a moving obstacle ---------------
// Each step, before the FSM kernel and from the states the loop condition is evaluated on, the vehicles are ordered by
// (driving, route, s, b): the key kernel writes an order-preserving 64-bit key of s and a 32-bit tag (route key << 27 | b,
// route key MPCB_MAX_ROUTES for a vehicle that is not driving), a stable radix sort by the s key carries the tags, and a
// stable sort of the tags by their route bits groups them by route.  Both sorts are stable and the input is in index
// order, so equal positions are ordered by index.  The leader of b is the next tag of its route segment, if it is within
// follow_range.
constexpr int FOLLOW_IDX_BITS = 27;                     // vehicles of a following simulation: < 2^27
constexpr unsigned FOLLOW_IDX_MASK = (1u << FOLLOW_IDX_BITS) - 1u;
constexpr int FOLLOW_ROUTE_BITS = 5;                    // route keys 0 .. MPCB_MAX_ROUTES (= not driving)
static_assert(MPCB_MAX_ROUTES < (1 << FOLLOW_ROUTE_BITS), "route key does not fit its bits");
static_assert(FOLLOW_IDX_BITS + FOLLOW_ROUTE_BITS == 32, "tag layout");

__global__ void __launch_bounds__(128)
mpcb_follow_key_kernel(const __grid_constant__ DevTables Ts, const int* __restrict__ route, int B,
                       const double* __restrict__ x, unsigned long long* __restrict__ key, unsigned* __restrict__ tag) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double s = x[(size_t)b * 5] + 0.0;              // -0.0 -> +0.0: equal positions get equal keys
  const bool live = s <= stop_s(Ts, route, b);          // loop condition (:395), as the FSM kernel evaluates it
  const unsigned long long u = (unsigned long long)__double_as_longlong(s);
  key[b] = (u >> 63) ? ~u : (u | (1ull << 63));         // order-preserving: unsigned order of keys = order of s
  const unsigned r = live ? (unsigned)problem_route(route, b, Ts.n) : (unsigned)MPCB_MAX_ROUTES;
  MPCB_ASSERT(r <= (unsigned)MPCB_MAX_ROUTES);
  tag[b] = (r << FOLLOW_IDX_BITS) | (unsigned)b;
}

// over the sorted tags: lead_idx[b] (-1: none) and lead_sv[b] = (s, v) of the leader (NaN: none)
__global__ void __launch_bounds__(128)
mpcb_follow_leader_kernel(int B, double range, const double* __restrict__ x, const unsigned* __restrict__ sorted,
                          int* __restrict__ lead_idx, double* __restrict__ lead_sv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const unsigned t = sorted[i];
  const int b = (int)(t & FOLLOW_IDX_MASK);
  const unsigned r = t >> FOLLOW_IDX_BITS;
  MPCB_ASSERT(b < B && r <= (unsigned)MPCB_MAX_ROUTES);
  int lead = -1;
  double ls = nan(""), lv = nan("");
  if (r < (unsigned)MPCB_MAX_ROUTES && i + 1 < B) {
    const unsigned tn = sorted[i + 1];
    if ((tn >> FOLLOW_IDX_BITS) == r) {
      const int j = (int)(tn & FOLLOW_IDX_MASK);
      MPCB_ASSERT(j < B && j != b);
      const double sj = x[(size_t)j * 5];
      if (sj - x[(size_t)b * 5] <= range) { lead = j; ls = sj; lv = x[(size_t)j * 5 + 4]; }
    }
  }
  lead_idx[b] = lead;
  lead_sv[2 * b] = ls;
  lead_sv[2 * b + 1] = lv;
}

// ObstaclesFSM.update for every vehicle that is still driving (:330-374); car first, then light (:349, :362).
// lead_sv != nullptr (following on): the car slot takes the nearer of the scripted car and the leader (lead_idx /
// lead_sv of mpcb_follow_leader_kernel), which is recorded into hist_lead_idx / hist_lead_sv.
__global__ void __launch_bounds__(128)
mpcb_fsm_kernel(const __grid_constant__ DevTables Ts, const int* __restrict__ route, int B, double dt,
                const double* __restrict__ x, const DevScenario* __restrict__ scen,
                double* __restrict__ fsm_f, int* __restrict__ fsm_i, int* __restrict__ alive,
                double* __restrict__ obs_sv, int* __restrict__ n_obs, int rec_t, double* __restrict__ hist_obs,
                int* __restrict__ hist_tl, int* __restrict__ alive_idx, int* __restrict__ alive_cnt,
                int* __restrict__ next_cnt, const int* __restrict__ lead_idx, const double* __restrict__ lead_sv,
                int* __restrict__ hist_lead_idx, double* __restrict__ hist_lead_sv) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) *next_cnt = 0;                                 // the other counter of the pair: next step's list length
  const bool in = b < B;
  const double s = in ? x[(size_t)b * 5] : 0.0, v = in ? x[(size_t)b * 5 + 4] : 0.0;
  const int live = (in && s <= stop_s(Ts, route, b)) ? 1 : 0;   // loop condition (:395), evaluated before the step
  // list of the vehicles still driving: the solve of this step runs over the list, not over all B (one atomic per warp;
  // the order of the list does not matter, every problem is solved on its own and written to its own slot)
  const int slot = warp_append(live, alive_cnt);
  if (live) alive_idx[slot] = b;
  if (!in) return;
  alive[b] = live;
  int n = 0;
  double o[4] = {0.0, 0.0, 0.0, 0.0};
  double car_s = nan("");
  int f = fsm_i[b];
  if (live) {
    const DevScenario sc = scen[b];
    double obs_s = fsm_f[2 * b], timer = fsm_f[2 * b + 1];
    if (sc.dynamic_obstacle) {
      if (s >= sc.obs_trigger_s && !(f & F_OBS_TRIGGERED)) f |= F_OBS_TRIGGERED | F_OBS_ACTIVE;
      if (f & F_OBS_ACTIVE) {
        // no FMA contraction: the car advances by the rounded product, as in the reference, so the obstacle the
        // solver sees is the reference's to the bit (the rounding difference otherwise grows with every step)
        obs_s = __dadd_rn(obs_s, __dmul_rn(sc.obs_v, dt));
        if (obs_s > sc.obs_end_s) f &= ~F_OBS_ACTIVE;
        else { o[0] = obs_s; o[1] = sc.obs_v; n = 1; car_s = obs_s; }
      }
    }
    if (lead_sv) {
      // the car slot holds the nearer of the scripted car and the leader (tie: the scripted car).  On a single-lane
      // route the farther car is behind the nearer one, and the nearer car is itself constrained by it, so keeping
      // clear of the nearer one is enough; one car slot keeps n_obs <= MPCB_MAX_OBS with the light after it.
      const double ls = lead_sv[2 * b];
      if (!isnan(ls) && !(n == 1 && o[0] <= ls)) { o[0] = ls; o[1] = lead_sv[2 * b + 1]; n = 1; }
    }
    if (sc.traffic_light && !(f & F_TL_GREEN)) {
      const double gap = sc.tl_pos - s;
      if (0.0 < gap && gap < sc.tl_trigger_s) {
        o[2 * n] = sc.tl_pos; o[2 * n + 1] = 0.0; ++n;
        if (v < 0.1 && gap < 10.0) f |= F_TL_WAITING;
      }
      if (f & F_TL_WAITING) {
        timer += dt;
        if (timer >= sc.tl_stop_duration) { f |= F_TL_GREEN; f &= ~F_TL_WAITING; }
      }
    }
    fsm_f[2 * b] = obs_s;
    fsm_f[2 * b + 1] = timer;
    fsm_i[b] = f;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) obs_sv[(size_t)b * 4 + k] = o[k];
  n_obs[b] = n;
  if (hist_obs && rec_t >= 0) {
    hist_obs[(size_t)rec_t * B + b] = car_s;                 // position of the moving car, NaN when absent
    hist_tl[(size_t)rec_t * B + b] = live ? ((f & F_TL_GREEN) ? 1 : 0) : -1;   // light colour returned by update()
  }
  if (lead_sv && hist_lead_idx && rec_t >= 0) {             // leader of this step; -1 / NaN: none or arrived
    const size_t i = (size_t)rec_t * B + b;
    const int lead = live ? lead_idx[b] : -1;
    MPCB_ASSERT(lead >= -1 && lead < B);
    hist_lead_idx[i] = lead;
    hist_lead_sv[2 * i] = lead >= 0 ? lead_sv[2 * b] : nan("");
    hist_lead_sv[2 * i + 1] = lead >= 0 ? lead_sv[2 * b + 1] : nan("");
  }
}

// plant step (:404-406) for the vehicles that were alive at the start of the step
__global__ void __launch_bounds__(128)
mpcb_plant_kernel(const __grid_constant__ DevTables Ts, const int* __restrict__ route, int B, double dt, double* __restrict__ x,
                  const double* __restrict__ U, const int* __restrict__ status, const int* __restrict__ alive,
                  int* __restrict__ steps, int* __restrict__ n_unsolved, int rec_t, double* __restrict__ hist_x,
                  double* __restrict__ hist_u, int* __restrict__ hist_status) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int live = alive[b];
  double xs[5];
#pragma unroll
  for (int c = 0; c < 5; ++c) xs[c] = x[(size_t)b * 5 + c];
  const double u1 = U[(size_t)b * NV], u2 = U[(size_t)b * NV + 1];
  if (hist_x && rec_t >= 0) {                                // state and control of THIS step (before the update)
#pragma unroll
    for (int c = 0; c < 5; ++c) hist_x[((size_t)rec_t * B + b) * 5 + c] = live ? xs[c] : nan("");
    hist_u[((size_t)rec_t * B + b) * 2] = live ? u1 : nan("");
    hist_u[((size_t)rec_t * B + b) * 2 + 1] = live ? u2 : nan("");
    hist_status[(size_t)rec_t * B + b] = live ? status[b] : -1;
  }
  if (!live) return;
  double val[4], slope[4];
  lookup_state(vehicle_table(Ts, route, b), xs[0], val, slope);   // k_ref = get_state(current_s)[3]  (:404)
  const double kref = val[2];
  const double s = xs[0], o = xs[2], k = xs[3], v = xs[4];
  // x + dt * [v, v o, v (k - k_ref), u1, u2]   (:50-67, :406); no FMA contraction: same rounding as numpy
  x[(size_t)b * 5 + 0] = __dadd_rn(s, __dmul_rn(dt, v));
  x[(size_t)b * 5 + 1] = __dadd_rn(xs[1], __dmul_rn(dt, __dmul_rn(v, o)));
  x[(size_t)b * 5 + 2] = __dadd_rn(o, __dmul_rn(dt, __dmul_rn(v, __dadd_rn(k, -kref))));
  x[(size_t)b * 5 + 3] = __dadd_rn(k, __dmul_rn(dt, u1));
  x[(size_t)b * 5 + 4] = __dadd_rn(v, __dmul_rn(dt, u2));
  steps[b] += 1;
  if (status[b] != MPCB_SOLVED) n_unsolved[b] += 1;
}

__global__ void mpcb_count_alive_kernel(const __grid_constant__ DevTables Ts, const int* __restrict__ route, int B,
                                        const double* __restrict__ x, int* __restrict__ count) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int live = (b < B && x[(size_t)b * 5] <= stop_s(Ts, route, b)) ? 1 : 0;
  const unsigned m = __ballot_sync(0xffffffffu, live);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, __popc(m));
}

// trajectory_tracking_check (sanity_checks.py:79-184) for every vehicle at once, on the recorded histories; one thread
// per vehicle, coalesced over vehicles.  Verdict bits (1 = passed): 0 destination reached (:98-103), 1 stayed on road
// (:106-111), 2 steering within limits +-0.1 (:121-125), 3 acceleration within limits (:127-131), 4 moving obstacle
// avoided, gap >= 1 m (:142-164), 5 red light respected (:167-181), 6 history covers the whole drive.  route == nullptr:
// every vehicle's route is s_total long; else vehicle b's route's s_max.
// (The reference's CPU-time item :134-139 is a property of the host, not of the trajectory; it is not evaluated here.)
__global__ void __launch_bounds__(128)
mpcb_sim_check_kernel(const __grid_constant__ DevTables Ts, const int* __restrict__ route, int B, int n_rec,
                      double s_total, double u1_min, double u1_max, double u2_min, double u2_max,
                      const double* __restrict__ x_final, const int* __restrict__ steps,
                      const DevScenario* __restrict__ scen, const double* __restrict__ hist_x,
                      const double* __restrict__ hist_u, const double* __restrict__ hist_obs,
                      const int* __restrict__ hist_tl, int* __restrict__ verdict, double* __restrict__ metrics) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const DevScenario sc = scen[b];
  const int n = min(steps[b], n_rec);
  const double tol = 0.1, lateral = 1.5, safety = 1.0;
  double max_dev = fabs(x_final[(size_t)b * 5 + 1]);
  double u1lo = BIG, u1hi = -BIG, u2lo = BIG, u2hi = -BIG, min_gap = BIG;
  int first_pass = -1;
  for (int t = 0; t < n; ++t) {
    const size_t i = (size_t)t * B + b;
    const double s = hist_x[i * 5], d = hist_x[i * 5 + 1];
    max_dev = fmax(max_dev, fabs(d));
    const double a = hist_u[i * 2], c = hist_u[i * 2 + 1];
    u1lo = fmin(u1lo, a); u1hi = fmax(u1hi, a); u2lo = fmin(u2lo, c); u2hi = fmax(u2hi, c);
    const double os = hist_obs[i];
    if (!isnan(os)) min_gap = fmin(min_gap, os - s);
    if (first_pass < 0 && s > sc.tl_pos) first_pass = t;
  }
  const double s_final = x_final[(size_t)b * 5];
  int v = 0;
  const double s_end = route ? vehicle_table(Ts, route, b).s_max : s_total;
  if (!(s_final < s_end - 1.0)) v |= 1;
  if (!(max_dev > lateral)) v |= 2;
  if (!(u1lo < u1_min - tol || u1hi > u1_max + tol)) v |= 4;
  if (!(u2lo < u2_min - tol || u2hi > u2_max + tol)) v |= 8;
  if (!(sc.dynamic_obstacle && min_gap < safety)) v |= 16;
  const bool ran_red = sc.traffic_light && first_pass >= 0 && hist_tl[(size_t)first_pass * B + b] == 0;
  if (!ran_red) v |= 32;
  if (steps[b] <= n_rec) v |= 64;
  verdict[b] = v;
  metrics[(size_t)b * 4 + 0] = max_dev;
  metrics[(size_t)b * 4 + 1] = min_gap;
  metrics[(size_t)b * 4 + 2] = s_final;
  metrics[(size_t)b * 4 + 3] = (double)steps[b];
}

// the check of item 4 (gap >= 1 m, sanity_checks.py:142-164) against the recorded leaders: min over the recorded steps
// of s_leader - s (BIG if never had a leader) and ok = that gap >= 1 m
__global__ void __launch_bounds__(128)
mpcb_follow_check_kernel(int B, int n_rec, const int* __restrict__ steps, const double* __restrict__ hist_x,
                         const double* __restrict__ hist_lead_sv, int* __restrict__ ok, double* __restrict__ min_gap) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int n = min(steps[b], n_rec);
  const double safety = 1.0;
  double g = BIG;
  for (int t = 0; t < n; ++t) {
    const size_t i = (size_t)t * B + b;
    const double ls = hist_lead_sv[2 * i];
    if (!isnan(ls)) g = fmin(g, ls - hist_x[i * 5]);
  }
  ok[b] = g < safety ? 0 : 1;
  min_gap[b] = g;
}

}  // namespace mpcb

using namespace mpcb;

struct mpcb_sim {
  mpcb_handle h;
  int B, cap, t;              // vehicles, history capacity (steps), steps recorded so far
  int hot_start = 0;          // first pass of step t > 0 starts from step t - 1's plans advanced by one step (mpcb_sim_set_hot_start)
  double dt;
  int* route = nullptr;       // route of each vehicle (device); nullptr: all on route 0
  DevScenario* scen = nullptr;
  double *x = nullptr, *fsm_f = nullptr, *obs_sv = nullptr, *U = nullptr;
  int *fsm_i = nullptr, *alive = nullptr, *n_obs = nullptr, *status = nullptr, *steps = nullptr, *n_unsolved = nullptr,
      *count = nullptr;
  int *alive_idx = nullptr, *alive_cnt = nullptr;   // list of the vehicles still driving; its length, double-buffered
  int* d_verdict = nullptr;                         // outputs of mpcb_sim_check (allocated with the histories)
  double* d_metrics = nullptr;
  double *hist_x = nullptr, *hist_u = nullptr, *hist_obs = nullptr;
  int *hist_status = nullptr, *hist_tl = nullptr;
  // following (mpcb_sim_set_follow); the buffers are allocated the first time it is switched on
  int follow = 0;
  double follow_range = 0.0;
  unsigned long long* f_key = nullptr;   // [2][B]: s keys, then sorted
  unsigned* f_tag = nullptr;             // [3][B]: tags, sorted by s, then by route
  void* f_temp = nullptr;                // radix-sort workspace, sized for B
  size_t f_temp_bytes = 0;
  int* lead_idx = nullptr;               // [B] leader of this step (-1: none)
  double* lead_sv = nullptr;             // [B][2] its (s, v) (NaN: none)
  int* hist_lead_idx = nullptr;          // [cap][B], -1 where not recorded
  double* hist_lead_sv = nullptr;        // [cap][B][2], NaN where not recorded
  int* d_follow_ok = nullptr;            // outputs of mpcb_sim_follow_check
  double* d_min_gap = nullptr;
};

extern "C" {

int mpcb_scenario_default(mpcb_scenario* s, int which) {
  if (!s) return MPCB_ERR_INVALID;
  memset(s, 0, sizeof(*s));
  if (which == 3) {            // trajectory3 constants, the commented block trajectory_tracking.py:313-327
    s->obs_trigger_s = 5.0; s->obs_start_s = 150.0; s->obs_v = 4.0; s->obs_end_s = 850.0;
    s->tl_pos = 2000.0; s->tl_trigger_s = 100.0; s->tl_stop_duration = 20.0;
  } else {                     // trajectory2 constants as committed, :294-308
    s->obs_trigger_s = 710.0; s->obs_start_s = 780.0; s->obs_v = 4.0; s->obs_end_s = 1050.0;
    s->tl_pos = 550.0; s->tl_trigger_s = 100.0; s->tl_stop_duration = 20.0;
  }
  s->dynamic_obstacle = 1; s->traffic_light = 1;
  return MPCB_OK;
}

int mpcb_sim_destroy(mpcb_sim_handle s) {
  if (!s) return MPCB_ERR_INVALID;
  cudaSetDevice(s->h->device);
  void* ptrs[] = {s->route, s->scen, s->x, s->fsm_f, s->obs_sv, s->U, s->fsm_i, s->alive, s->n_obs, s->status, s->steps,
                  s->n_unsolved, s->count, s->hist_x, s->hist_u, s->hist_obs, s->hist_status, s->hist_tl, s->alive_idx,
                  s->alive_cnt, s->d_verdict, s->d_metrics, s->f_key, s->f_tag, s->f_temp, s->lead_idx, s->lead_sv,
                  s->hist_lead_idx, s->hist_lead_sv, s->d_follow_ok, s->d_min_gap};
  for (void* p : ptrs) if (p) cudaFree(p);
  delete s;
  return MPCB_OK;
}

int mpcb_sim_create(mpcb_sim_handle* out, mpcb_handle h, int B, const mpcb_scenario* scen, int n_scen,
                    const double* x_init, int history_steps) {
  return mpcb_sim_create_routes(out, h, B, scen, n_scen, nullptr, x_init, history_steps);
}

int mpcb_sim_create_routes(mpcb_sim_handle* out, mpcb_handle h, int B, const mpcb_scenario* scen, int n_scen,
                           const int* route, const double* x_init, int history_steps) {
  if (!out || !h || B < 1 || !scen || (n_scen != 1 && n_scen != B) || history_steps < 0) return MPCB_ERR_INVALID;
  if (route)
    for (int b = 0; b < B; ++b)
      if (route[b] < 0 || route[b] >= h->dt.n) return MPCB_ERR_INVALID;
  *out = nullptr;
  CK(cudaSetDevice(h->device));
  mpcb_sim* s = new (std::nothrow) mpcb_sim();
  if (!s) return MPCB_ERR_NOMEM;
  s->h = h; s->B = B; s->cap = history_steps; s->t = 0;
  s->dt = h->params.dt;
  auto fail = [&](int code) { mpcb_sim_destroy(s); return code; };
  const size_t nb = (size_t)B;
#define SIM_ALLOC(ptr, bytes) if (cudaMalloc((void**)&(ptr), (bytes)) != cudaSuccess) { cudaGetLastError(); return fail(MPCB_ERR_NOMEM); }
  SIM_ALLOC(s->scen, nb * sizeof(DevScenario));
  SIM_ALLOC(s->x, nb * 40); SIM_ALLOC(s->fsm_f, nb * 16); SIM_ALLOC(s->obs_sv, nb * 32); SIM_ALLOC(s->U, nb * 80);
  SIM_ALLOC(s->fsm_i, nb * 4); SIM_ALLOC(s->alive, nb * 4); SIM_ALLOC(s->n_obs, nb * 4); SIM_ALLOC(s->status, nb * 4);
  SIM_ALLOC(s->steps, nb * 4); SIM_ALLOC(s->n_unsolved, nb * 4); SIM_ALLOC(s->count, 4);
  SIM_ALLOC(s->alive_idx, nb * 4); SIM_ALLOC(s->alive_cnt, 8);
  if (route) SIM_ALLOC(s->route, nb * 4);
  if (history_steps > 0) {
    SIM_ALLOC(s->d_verdict, nb * 4); SIM_ALLOC(s->d_metrics, nb * 32);
    const size_t nt = (size_t)history_steps * nb;
    SIM_ALLOC(s->hist_x, nt * 40); SIM_ALLOC(s->hist_u, nt * 16); SIM_ALLOC(s->hist_obs, nt * 8);
    SIM_ALLOC(s->hist_status, nt * 4); SIM_ALLOC(s->hist_tl, nt * 4);
  }
#undef SIM_ALLOC
  std::vector<DevScenario> hs(nb);
  std::vector<double> hx(nb * 5), hf(nb * 2);
  for (size_t b = 0; b < nb; ++b) {
    const mpcb_scenario& c = scen[n_scen == 1 ? 0 : b];
    hs[b] = DevScenario{c.obs_trigger_s, c.obs_start_s, c.obs_v, c.obs_end_s, c.tl_pos, c.tl_trigger_s,
                        c.tl_stop_duration, c.dynamic_obstacle, c.traffic_light};
    if (x_init) for (int k = 0; k < 5; ++k) hx[b * 5 + k] = x_init[b * 5 + k];
    else { hx[b * 5] = hx[b * 5 + 1] = hx[b * 5 + 2] = hx[b * 5 + 3] = 0.0; hx[b * 5 + 4] = 0.5; }   // :382
    hf[b * 2] = c.obs_start_s;                                          // obs_s = obs_start_s (:297)
    hf[b * 2 + 1] = 0.0;
  }
  cudaError_t e;
  if (route && (e = cudaMemcpy(s->route, route, nb * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemcpy"));
  if ((e = cudaMemcpy(s->scen, hs.data(), nb * sizeof(DevScenario), cudaMemcpyHostToDevice)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemcpy"));
  if ((e = cudaMemcpy(s->x, hx.data(), nb * 40, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemcpy"));
  if ((e = cudaMemcpy(s->fsm_f, hf.data(), nb * 16, cudaMemcpyHostToDevice)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemcpy"));
  if ((e = cudaMemset(s->fsm_i, 0, nb * 4)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset"));
  if ((e = cudaMemset(s->steps, 0, nb * 4)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset"));
  if ((e = cudaMemset(s->n_unsolved, 0, nb * 4)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset"));
  if ((e = cudaMemset(s->alive_cnt, 0, 8)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset"));
  if ((e = cudaMemset(s->status, 0, nb * 4)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset"));
  if ((e = cudaMemset(s->U, 0, nb * 80)) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset"));
  *out = s;
  return MPCB_OK;
}

int mpcb_sim_step(mpcb_sim_handle s, int n_steps, void* cuda_stream) {
  if (!s || n_steps < 0) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int grid = (s->B + 127) / 128;
  for (int k = 0; k < n_steps; ++k) {
    const int rec = (s->t < s->cap) ? s->t : -1;
    int* cnt = s->alive_cnt + (s->t & 1);
    if (s->follow) {                                         // leaders of this step, from the states before it
      const size_t nb = (size_t)s->B;
      mpcb_follow_key_kernel<<<grid, 128, 0, st>>>(s->h->dt, s->route, s->B, s->x, s->f_key, s->f_tag);
      CK(cudaGetLastError());
      size_t tb = s->f_temp_bytes;
      CK(cub::DeviceRadixSort::SortPairs(s->f_temp, tb, s->f_key, s->f_key + nb, s->f_tag, s->f_tag + nb, s->B, 0, 64, st));
      tb = s->f_temp_bytes;
      CK(cub::DeviceRadixSort::SortKeys(s->f_temp, tb, s->f_tag + nb, s->f_tag + 2 * nb, s->B, FOLLOW_IDX_BITS, 32, st));
      mpcb_follow_leader_kernel<<<grid, 128, 0, st>>>(s->B, s->follow_range, s->x, s->f_tag + 2 * nb, s->lead_idx,
                                                      s->lead_sv);
      CK(cudaGetLastError());
      s->h->launches += 2;                                   // the radix sorts' own kernels are not counted
    }
    mpcb_fsm_kernel<<<grid, 128, 0, st>>>(s->h->dt, s->route, s->B, s->dt, s->x, s->scen, s->fsm_f, s->fsm_i, s->alive, s->obs_sv,
                                          s->n_obs, rec, s->hist_obs, s->hist_tl, s->alive_idx, cnt,
                                          s->alive_cnt + ((s->t + 1) & 1), s->lead_idx,
                                          s->follow ? s->lead_sv : nullptr, s->hist_lead_idx, s->hist_lead_sv);
    CK(cudaGetLastError());
    // the solve runs over the list of vehicles still driving (arrived vehicles are frozen and cost nothing)
    int rc = mpcb_solve_list_internal(s->h, s->B, s->alive_idx, cnt, s->x, s->obs_sv, s->n_obs, s->route, s->U, s->status,
                                      st, (s->hot_start && s->t > 0) ? s->U : nullptr);
    if (rc != MPCB_OK) return rc;
    mpcb_plant_kernel<<<grid, 128, 0, st>>>(s->h->dt, s->route, s->B, s->dt, s->x, s->U, s->status, s->alive, s->steps,
                                            s->n_unsolved, rec, s->hist_x, s->hist_u, s->hist_status);
    CK(cudaGetLastError());
    s->h->launches += 2;
    s->t += 1;
  }
  return MPCB_OK;
}

int mpcb_sim_set_hot_start(mpcb_sim_handle s, int on) {
  if (!s) return MPCB_ERR_INVALID;
  s->hot_start = on ? 1 : 0;
  return MPCB_OK;
}

int mpcb_sim_set_follow(mpcb_sim_handle s, int on, double follow_range) {
  if (!s) return MPCB_ERR_INVALID;
  if (!on) { s->follow = 0; return MPCB_OK; }
  if (!(follow_range > 0.0) || !isfinite(follow_range) || (unsigned)s->B > FOLLOW_IDX_MASK + 1u) return MPCB_ERR_INVALID;
  if (!s->f_key) {
    CK(cudaSetDevice(s->h->device));
    const size_t nb = (size_t)s->B;
    size_t t1 = 0, t2 = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, t1, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                       (unsigned*)nullptr, (unsigned*)nullptr, s->B, 0, 64));
    CK(cub::DeviceRadixSort::SortKeys(nullptr, t2, (unsigned*)nullptr, (unsigned*)nullptr, s->B, FOLLOW_IDX_BITS, 32));
    const size_t temp = t1 > t2 ? t1 : t2;
    const size_t nt = (size_t)s->cap * nb;
    bool ok = cudaMalloc((void**)&s->f_key, nb * 16) == cudaSuccess && cudaMalloc((void**)&s->f_tag, nb * 12) == cudaSuccess &&
              cudaMalloc(&s->f_temp, temp) == cudaSuccess && cudaMalloc((void**)&s->lead_idx, nb * 4) == cudaSuccess &&
              cudaMalloc((void**)&s->lead_sv, nb * 16) == cudaSuccess;
    if (ok && nt > 0)
      ok = cudaMalloc((void**)&s->hist_lead_idx, nt * 4) == cudaSuccess &&
           cudaMalloc((void**)&s->hist_lead_sv, nt * 16) == cudaSuccess &&
           cudaMalloc((void**)&s->d_follow_ok, nb * 4) == cudaSuccess && cudaMalloc((void**)&s->d_min_gap, nb * 8) == cudaSuccess;
    if (!ok) {
      cudaGetLastError();
      void* ptrs[] = {s->f_key, s->f_tag, s->f_temp, s->lead_idx, s->lead_sv, s->hist_lead_idx, s->hist_lead_sv,
                      s->d_follow_ok, s->d_min_gap};
      for (void* p : ptrs) if (p) cudaFree(p);
      s->f_key = nullptr; s->f_tag = nullptr; s->f_temp = nullptr; s->lead_idx = nullptr; s->lead_sv = nullptr;
      s->hist_lead_idx = nullptr; s->hist_lead_sv = nullptr; s->d_follow_ok = nullptr; s->d_min_gap = nullptr;
      return MPCB_ERR_NOMEM;
    }
    s->f_temp_bytes = temp;
    // rows of steps taken with following off stay -1 / NaN (all-ones bytes: int -1, a double NaN)
    if (nt > 0) {
      CK(cudaMemset(s->hist_lead_idx, 0xff, nt * 4));
      CK(cudaMemset(s->hist_lead_sv, 0xff, nt * 16));
      CK(cudaStreamSynchronize(0));
    }
  }
  s->follow = 1;
  s->follow_range = follow_range;
  return MPCB_OK;
}

int mpcb_sim_follow_history(mpcb_sim_handle s, int* n_recorded, int* hist_lead_idx, double* hist_lead_sv,
                            void* cuda_stream) {
  if (!s) return MPCB_ERR_INVALID;
  const int nt = s->t < s->cap ? s->t : s->cap;
  if (n_recorded) *n_recorded = nt;
  const size_t n = (size_t)nt * s->B;
  if (n == 0 || (!hist_lead_idx && !hist_lead_sv)) return MPCB_OK;
  if (!s->hist_lead_idx) {                                   // following never switched on: nothing recorded
    if (hist_lead_idx) for (size_t i = 0; i < n; ++i) hist_lead_idx[i] = -1;
    if (hist_lead_sv) for (size_t i = 0; i < 2 * n; ++i) hist_lead_sv[i] = nan("");
    return MPCB_OK;
  }
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (hist_lead_idx) CK(cudaMemcpyAsync(hist_lead_idx, s->hist_lead_idx, n * 4, cudaMemcpyDeviceToHost, st));
  if (hist_lead_sv) CK(cudaMemcpyAsync(hist_lead_sv, s->hist_lead_sv, n * 16, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

int mpcb_sim_follow_check(mpcb_sim_handle s, int* ok, double* min_gap, void* cuda_stream) {
  if (!s || !ok || s->cap < 1) return MPCB_ERR_INVALID;
  const size_t nb = (size_t)s->B;
  if (!s->hist_lead_sv) {                                    // following never switched on: no leader, ever
    for (size_t b = 0; b < nb; ++b) { ok[b] = 1; if (min_gap) min_gap[b] = BIG; }
    return MPCB_OK;
  }
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int nt = s->t < s->cap ? s->t : s->cap;
  mpcb_follow_check_kernel<<<(s->B + 127) / 128, 128, 0, st>>>(s->B, nt, s->steps, s->hist_x, s->hist_lead_sv,
                                                               s->d_follow_ok, s->d_min_gap);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ok, s->d_follow_ok, nb * 4, cudaMemcpyDeviceToHost, st));
  if (min_gap) CK(cudaMemcpyAsync(min_gap, s->d_min_gap, nb * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  s->h->launches += 1;
  return MPCB_OK;
}

int mpcb_sim_alive(mpcb_sim_handle s, int* n_alive, void* cuda_stream) {
  if (!s || !n_alive) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  CK(cudaMemsetAsync(s->count, 0, 4, st));
  mpcb_count_alive_kernel<<<(s->B + 127) / 128, 128, 0, st>>>(s->h->dt, s->route, s->B, s->x, s->count);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(n_alive, s->count, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

int mpcb_sim_state(mpcb_sim_handle s, double* x, int* steps, int* n_unsolved, void* cuda_stream) {
  if (!s) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const size_t nb = (size_t)s->B;
  if (x) CK(cudaMemcpyAsync(x, s->x, nb * 40, cudaMemcpyDeviceToHost, st));
  if (steps) CK(cudaMemcpyAsync(steps, s->steps, nb * 4, cudaMemcpyDeviceToHost, st));
  if (n_unsolved) CK(cudaMemcpyAsync(n_unsolved, s->n_unsolved, nb * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

int mpcb_sim_check(mpcb_sim_handle s, int* verdict, double* metrics, void* cuda_stream) {
  if (!s || !verdict || s->cap < 1) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const size_t nb = (size_t)s->B;
  const mpcb_params& p = s->h->params;
  const int nt = s->t < s->cap ? s->t : s->cap;
  mpcb_sim_check_kernel<<<(s->B + 127) / 128, 128, 0, st>>>(s->h->dt, s->route, s->B, nt, s->h->dt.t[0].s_max, p.u_min[0], p.u_max[0], p.u_min[1],
                                                           p.u_max[1], s->x, s->steps, s->scen, s->hist_x, s->hist_u,
                                                           s->hist_obs, s->hist_tl, s->d_verdict, s->d_metrics);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(verdict, s->d_verdict, nb * 4, cudaMemcpyDeviceToHost, st));
  if (metrics) CK(cudaMemcpyAsync(metrics, s->d_metrics, nb * 32, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  s->h->launches += 1;
  return MPCB_OK;
}

// The same checks on histories the CALLER supplies (host arrays, laid out like mpcb_sim_history returns them).  This is
// the entry the parity tests use to compare the device checker with the reference's trajectory_tracking_check on
// histories that FAIL an item (tests/golden/sanity_cases.npz).
int mpcb_check_histories(mpcb_handle h, int B, int T, double s_total, const mpcb_scenario* scen, const double* x_final,
                         const int* steps, const double* hist_x, const double* hist_u, const double* hist_obs,
                         const int* hist_tl, int* verdict, double* metrics) {
  if (!h || B < 1 || T < 1 || !scen || !x_final || !steps || !hist_x || !hist_u || !hist_obs || !hist_tl || !verdict)
    return MPCB_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  const size_t nb = (size_t)B, nt = (size_t)T * nb;
  std::vector<DevScenario> hs(nb);
  for (size_t b = 0; b < nb; ++b) {
    const mpcb_scenario& c = scen[b];
    hs[b] = DevScenario{c.obs_trigger_s, c.obs_start_s, c.obs_v, c.obs_end_s, c.tl_pos, c.tl_trigger_s,
                        c.tl_stop_duration, c.dynamic_obstacle, c.traffic_light};
  }
  // one allocation: the seven inputs, then the verdicts and the metrics
  const size_t sz[9] = {nb * sizeof(DevScenario), nb * 40, nb * 4, nt * 40, nt * 16, nt * 8, nt * 4, nb * 4, nb * 32};
  const void* src[7] = {hs.data(), x_final, steps, hist_x, hist_u, hist_obs, hist_tl};
  size_t off[10];
  region_offsets(sz, 9, off);
  char* d = nullptr;
  if (cudaMalloc((void**)&d, off[9]) != cudaSuccess) { cudaGetLastError(); return MPCB_ERR_NOMEM; }
  cudaStream_t st = h->stream;
  cudaError_t e = cudaSuccess;
  for (int k = 0; k < 7 && e == cudaSuccess; ++k) e = cudaMemcpyAsync(d + off[k], src[k], sz[k], cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    const mpcb_params& p = h->params;
    int* d_v = (int*)(d + off[7]);
    double* d_m = (double*)(d + off[8]);
    mpcb_sim_check_kernel<<<(B + 127) / 128, 128, 0, st>>>(h->dt, nullptr, B, T, s_total, p.u_min[0], p.u_max[0], p.u_min[1], p.u_max[1],
                                                          (const double*)(d + off[1]), (const int*)(d + off[2]),
                                                          (const DevScenario*)(d + off[0]), (const double*)(d + off[3]),
                                                          (const double*)(d + off[4]), (const double*)(d + off[5]),
                                                          (const int*)(d + off[6]), d_v, d_m);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(verdict, d_v, nb * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && metrics) e = cudaMemcpyAsync(metrics, d_m, nb * 32, cudaMemcpyDeviceToHost, st);
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d);
  if (e != cudaSuccess) return cuda_fail(e, "mpcb_check_histories");
  h->launches += 1;
  return MPCB_OK;
}

int mpcb_sim_history(mpcb_sim_handle s, int* n_recorded, double* hist_x, double* hist_u, double* hist_obs,
                     int* hist_status, int* hist_tl, void* cuda_stream) {
  if (!s) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int nt = s->t < s->cap ? s->t : s->cap;
  if (n_recorded) *n_recorded = nt;
  const size_t n = (size_t)nt * s->B;
  if (n > 0) {
    if (hist_x) CK(cudaMemcpyAsync(hist_x, s->hist_x, n * 40, cudaMemcpyDeviceToHost, st));
    if (hist_u) CK(cudaMemcpyAsync(hist_u, s->hist_u, n * 16, cudaMemcpyDeviceToHost, st));
    if (hist_obs) CK(cudaMemcpyAsync(hist_obs, s->hist_obs, n * 8, cudaMemcpyDeviceToHost, st));
    if (hist_status) CK(cudaMemcpyAsync(hist_status, s->hist_status, n * 4, cudaMemcpyDeviceToHost, st));
    if (hist_tl) CK(cudaMemcpyAsync(hist_tl, s->hist_tl, n * 4, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

}  // extern "C"
