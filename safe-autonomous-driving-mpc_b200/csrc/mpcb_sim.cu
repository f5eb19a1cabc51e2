// mpcb_sim.cu -- batched closed loop on the device (SURVEY.md 8(f1)): the callers either side of the solve path.
//
//   obstacle-set producer   ObstaclesFSM.update            trajectory_tracking.py:330-374
//   plant step              x += dt * dynamics(x, u0, k_ref(s))   trajectory_tracking.py:404-406 (dynamics :50-67)
//   loop condition          while current_s <= s_max - 1.0         trajectory_tracking.py:395
//
// One simulation object holds B vehicles (each with its own scenario constants and FSM state).  A step is three
// launches on one stream -- FSM kernel -> mpcb_solve_batch -> plant kernel -- with no host round trip, so a
// Monte-Carlo of whole drives never leaves the GPU; histories are recorded into device buffers when asked for.  With
// following on (mpcb_sim_set_follow), a key kernel, two radix sorts and a leader kernel come first, or one world kernel
// when the fleet is split into worlds (mpcb_sim_set_worlds).  With noise on
// (mpcb_sim_set_noise), the FSM kernel also writes the measured state the solve reads and the plant kernel disturbs the
// control it applies and the state it produces; the step keeps its launches.  The FSM and plant kernels also keep each
// vehicle's trajectory_tracking_check accumulators up to date (mpcb_sim_running_check), and mpcb_sim_branch copies
// whole vehicles (mpcb_sim_branch_worlds: whole worlds) onto others for splitting estimators of rare failures.
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include <new>
#include <type_traits>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "mpcb200.h"
#include "mpcb_internal.h"
#include "mpcb_philox.cuh"

namespace mpcb {

struct DevScenario {          // per vehicle, mirrors ObstaclesFSM.__init__ (:285-308)
  double obs_trigger_s, obs_start_s, obs_v, obs_end_s;
  double tl_pos, tl_trigger_s, tl_stop_duration;
  int dynamic_obstacle, traffic_light;
};

// The accumulators of trajectory_tracking_check (mpcb_sim_check_kernel) that the FSM and plant kernels keep per vehicle
// while it drives (R_RUN, [B][RUN_W] doubles), so that a verdict needs no history: max |d| over the states before each
// step (NaN before the first; the check folds in the final state), the commanded control's extremes, the least gap to
// the scripted car, and the light colour at the first step past tl_pos (-1: not passed yet).
enum { RUN_DEV, RUN_U1LO, RUN_U1HI, RUN_U2LO, RUN_U2HI, RUN_GAP, RUN_TL, RUN_W };

// The device arrays of a simulation, in five groups: the loop state and the histories are one block made at create,
// following and its histories one block made by the first mpcb_sim_set_follow(on), the measured states and the noise
// history one block made by the first mpcb_sim_set_noise that switches noise on.  The layout of a block, every copy and
// every fill, and what mpcb_sim_branch gathers, is derived from SIM_BYTES.
enum SimRegion {
  R_SCEN, R_X, R_FSM_F, R_OBS_SV, R_U, R_FSM_I, R_ALIVE, R_N_OBS, R_STATUS, R_STEPS, R_N_UNSOLVED, R_ALIVE_IDX,
  R_ALIVE_CNT, R_COUNT, R_RUN, R_RUN_VERDICT, R_RUN_METRICS, R_ROUTE,                     // loop state
  R_HIST_X, R_HIST_U, R_HIST_OBS, R_HIST_STATUS, R_HIST_TL, R_VERDICT, R_METRICS,         // histories
  R_F_KEY, R_F_TAG, R_F_TEMP, R_LEAD_IDX, R_LEAD_SV, R_RUN_FOLLOW,                        // following
  R_HIST_LEAD_IDX, R_HIST_LEAD_SV, R_FOLLOW_OK, R_MIN_GAP,                                // following histories
  R_X_MEAS, R_HIST_NOISE,                                                                 // noise
  N_SIM
};
typedef unsigned long long SimMask;                                 // bit r selects region r
constexpr SimMask sim_bit(int r) { return 1ull << r; }
constexpr SimMask sim_span(int lo, int hi) { return (sim_bit(hi) - 1ull) & ~(sim_bit(lo) - 1ull); }   // regions lo .. hi-1
constexpr SimMask SIM_LOOP = sim_span(R_SCEN, R_ROUTE);          // R_ROUTE only on a routed simulation
constexpr SimMask SIM_HIST = sim_span(R_HIST_X, R_F_KEY);
constexpr SimMask SIM_FOLLOW = sim_span(R_F_KEY, R_HIST_LEAD_IDX);
constexpr SimMask SIM_FOLLOW_HIST = sim_span(R_HIST_LEAD_IDX, R_X_MEAS);
static_assert(N_SIM < 64, "regions are selected by the bits of a SimMask");

enum SimPer { PER_VEHICLE, PER_STEP, FIXED };   // bytes per vehicle, per vehicle and recorded step, or in all
// What mpcb_sim_branch does with a region: STATE, per vehicle, and HIST, [row][B][w], are gathered by the parent index of
// every vehicle; SCRATCH is rebuilt before it is next read (by the next step, or by the call that returns it).
enum SimBranch { STATE, HIST, SCRATCH };
struct SimBytes { SimPer per; size_t bytes; SimBranch branch; };
static constexpr SimBytes SIM_BYTES[N_SIM] = {
  /* scen          */ {PER_VEHICLE, sizeof(DevScenario), STATE},
  /* x             */ {PER_VEHICLE, 5 * 8, STATE},
  /* fsm_f         */ {PER_VEHICLE, 2 * 8, STATE},      // car position, light timer
  /* obs_sv        */ {PER_VEHICLE, 4 * 8, STATE},
  /* U             */ {PER_VEHICLE, NV * 8, STATE},     // this step's plans; the next one's hot start
  /* fsm_i         */ {PER_VEHICLE, 4, STATE},
  /* alive         */ {PER_VEHICLE, 4, STATE},
  /* n_obs         */ {PER_VEHICLE, 4, STATE},
  /* status        */ {PER_VEHICLE, 4, STATE},
  /* steps         */ {PER_VEHICLE, 4, STATE},
  /* n_unsolved    */ {PER_VEHICLE, 4, STATE},
  /* alive_idx     */ {PER_VEHICLE, 4, SCRATCH},        // list of the vehicles still driving
  /* alive_cnt     */ {FIXED, 2 * 4, SCRATCH},          // its length, double-buffered
  /* count         */ {FIXED, 4, SCRATCH},              // mpcb_sim_alive
  /* run           */ {PER_VEHICLE, RUN_W * 8, STATE},  // running verdict accumulators (RunAcc)
  /* run_verdict   */ {PER_VEHICLE, 4, SCRATCH},        // mpcb_sim_running_check
  /* run_metrics   */ {PER_VEHICLE, 4 * 8, SCRATCH},
  /* route         */ {PER_VEHICLE, 4, STATE},
  /* hist_x        */ {PER_STEP, 5 * 8, HIST},          // [cap][B][5]
  /* hist_u        */ {PER_STEP, 2 * 8, HIST},
  /* hist_obs      */ {PER_STEP, 8, HIST},
  /* hist_status   */ {PER_STEP, 4, HIST},
  /* hist_tl       */ {PER_STEP, 4, HIST},
  /* verdict       */ {PER_VEHICLE, 4, SCRATCH},        // mpcb_sim_check
  /* metrics       */ {PER_VEHICLE, 4 * 8, SCRATCH},
  /* f_key         */ {PER_VEHICLE, 2 * 8, SCRATCH},    // [2][B]: s keys, then sorted
  /* f_tag         */ {PER_VEHICLE, 3 * 4, SCRATCH},    // [3][B]: tags, sorted by s, then by route
  /* f_temp        */ {FIXED, 0, SCRATCH},              // radix-sort workspace: its size query's bytes (sim_layout)
  /* lead_idx      */ {PER_VEHICLE, 4, SCRATCH},        // leader of this step (-1: none)
  /* lead_sv       */ {PER_VEHICLE, 2 * 8, SCRATCH},    // its (s, v) (NaN: none)
  /* run_follow    */ {PER_VEHICLE, 8, STATE},          // least gap to the leader so far (mpcb_sim_running_follow_check)
  /* hist_lead_idx */ {PER_STEP, 4, HIST},              // -1 where not recorded
  /* hist_lead_sv  */ {PER_STEP, 2 * 8, HIST},          // NaN where not recorded
  /* follow_ok     */ {PER_VEHICLE, 4, SCRATCH},        // mpcb_sim_follow_check
  /* min_gap       */ {PER_VEHICLE, 8, SCRATCH},
  /* x_meas        */ {PER_VEHICLE, 5 * 8, SCRATCH},    // the state the solve sees
  /* hist_noise    */ {PER_STEP, 12 * 8, HIST},         // [cap][B][12]: measurement 5, actuation 2, process 5; NaN where not recorded
};
// A gathered region is copied in 4-byte words, vehicle-major (STATE) or [row][B][w] (HIST).
constexpr bool sim_branch_classes_hold(int r = 0) {
  return r == N_SIM || ((SIM_BYTES[r].branch == HIST) == (SIM_BYTES[r].per == PER_STEP) &&
                        (SIM_BYTES[r].branch != STATE || SIM_BYTES[r].per == PER_VEHICLE) &&
                        (SIM_BYTES[r].branch == SCRATCH || SIM_BYTES[r].bytes % 4 == 0) && sim_branch_classes_hold(r + 1));
}
static_assert(sim_branch_classes_hold(), "every recorded region is a history, every gathered one whole words");

// Bytes of region r for B vehicles and T recorded steps (R_F_TEMP: see sim_layout).
static size_t sim_bytes(int r, size_t B, size_t T) {
  const SimBytes& s = SIM_BYTES[r];
  return s.bytes * (s.per == PER_VEHICLE ? B : s.per == PER_STEP ? T * B : 1);
}

// Layout of the regions in mask of a simulation of B vehicles and T recorded steps, with a radix-sort workspace of temp
// bytes: region r at off[r] (no bytes when it is not in mask), off[N_SIM] bytes in all.  Each region starts on 256
// bytes, which also keeps U 16-byte aligned for the solve's 128-bit stores into it.
static void sim_layout(size_t B, size_t T, SimMask mask, size_t temp, size_t (&off)[N_SIM + 1]) {
  size_t bytes[N_SIM];
  for (int r = 0; r < N_SIM; ++r) bytes[r] = !((mask >> r) & 1ull) ? 0 : r == R_F_TEMP ? temp : sim_bytes(r, B, T);
  region_offsets(bytes, N_SIM, off);
}

// The device arrays of a simulation (nullptr: not allocated), handed to its kernels as one grid-constant parameter.  The
// kernels bind the arrays they use to __restrict__ locals (the qualifier is not honoured on struct members): the
// read-only ones then load through the non-coherent path.
struct SimArrays {
  DevScenario* scen; double* x; double* fsm_f; double* obs_sv; double* U;
  int* fsm_i; int* alive; int* n_obs; int* status; int* steps; int* n_unsolved; int* alive_idx; int* alive_cnt;
  int* count; double* run; int* run_verdict; double* run_metrics; int* route;
  double* hist_x; double* hist_u; double* hist_obs; int* hist_status; int* hist_tl; int* verdict; double* metrics;
  unsigned long long* f_key; unsigned* f_tag; void* f_temp; int* lead_idx; double* lead_sv; double* run_follow;
  int* hist_lead_idx; double* hist_lead_sv; int* follow_ok; double* min_gap;
  double* x_meas; double* hist_noise;
};

// One block holding the regions in mask, laid out by sim_layout; points their arrays in d (and, when given, their
// addresses in ptr) into it and leaves the others.  nullptr (and no error left pending) when it cannot be allocated.
static char* sim_alloc(SimArrays& d, size_t B, size_t T, SimMask mask, size_t temp, size_t (&off)[N_SIM + 1],
                       char** ptr = nullptr) {
  sim_layout(B, T, mask, temp, off);
  char* base = nullptr;
  if (cudaMalloc((void**)&base, off[N_SIM]) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (ptr)
    for (int r = 0; r < N_SIM; ++r)
      if ((mask >> r) & 1ull) ptr[r] = base + off[r];
  auto at = [&](auto*& p, int r) {
    if ((mask >> r) & 1ull) p = (std::remove_reference_t<decltype(p)>)(base + off[r]);
  };
  at(d.scen, R_SCEN); at(d.x, R_X); at(d.fsm_f, R_FSM_F); at(d.obs_sv, R_OBS_SV); at(d.U, R_U);
  at(d.fsm_i, R_FSM_I); at(d.alive, R_ALIVE); at(d.n_obs, R_N_OBS); at(d.status, R_STATUS); at(d.steps, R_STEPS);
  at(d.n_unsolved, R_N_UNSOLVED); at(d.alive_idx, R_ALIVE_IDX); at(d.alive_cnt, R_ALIVE_CNT); at(d.count, R_COUNT);
  at(d.run, R_RUN); at(d.run_verdict, R_RUN_VERDICT); at(d.run_metrics, R_RUN_METRICS); at(d.route, R_ROUTE);
  at(d.hist_x, R_HIST_X); at(d.hist_u, R_HIST_U); at(d.hist_obs, R_HIST_OBS); at(d.hist_status, R_HIST_STATUS);
  at(d.hist_tl, R_HIST_TL); at(d.verdict, R_VERDICT); at(d.metrics, R_METRICS);
  at(d.f_key, R_F_KEY); at(d.f_tag, R_F_TAG); at(d.f_temp, R_F_TEMP); at(d.lead_idx, R_LEAD_IDX);
  at(d.lead_sv, R_LEAD_SV); at(d.run_follow, R_RUN_FOLLOW);
  at(d.hist_lead_idx, R_HIST_LEAD_IDX); at(d.hist_lead_sv, R_HIST_LEAD_SV); at(d.follow_ok, R_FOLLOW_OK);
  at(d.min_gap, R_MIN_GAP);
  at(d.x_meas, R_X_MEAS); at(d.hist_noise, R_HIST_NOISE);
  return base;
}

// The read-only arrays of the fsm, plant and count kernels are read with __ldg: the compiler takes this non-coherent
// path by itself for __restrict__ kernel parameters, but in these three kernels not for the restrict-qualified locals.
__device__ __forceinline__ DevScenario ldg(const DevScenario* p) {
  return DevScenario{__ldg(&p->obs_trigger_s), __ldg(&p->obs_start_s), __ldg(&p->obs_v), __ldg(&p->obs_end_s),
                     __ldg(&p->tl_pos), __ldg(&p->tl_trigger_s), __ldg(&p->tl_stop_duration),
                     __ldg(&p->dynamic_obstacle), __ldg(&p->traffic_light)};
}

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

// ---- noise (mpcb_sim_set_noise): seeded Gaussian disturbances, a draw a function of (seed, id, t, j) only -------------
// sigma[0..4] measurement, [5..6] actuation, [7..11] process; a channel is on when one of its sigmas is > 0, and a
// component whose sigma is 0 is left untouched.  With every channel off the kernels compute what they computed without
// noise, bit for bit.
struct SimNoise {
  unsigned long long seed;
  int first_id;                 // id of vehicle b is first_id + b (first_id + B <= 2^31)
  int on, meas, act, proc;      // on = meas | act | proc
  double sigma[12];
};
constexpr int NOISE_W = 12;     // values recorded per vehicle and step: measurement 5, actuation 2, process 5
constexpr int NOISE_ACT = 5, NOISE_PROC = 7;

__device__ __forceinline__ unsigned vehicle_id(const SimNoise& nz, int b) {
  const long long id = (long long)nz.first_id + b;
  MPCB_ASSERT(nz.first_id >= 0 && b >= 0 && id <= 0x7fffffffLL);
  return (unsigned)id;
}

// w[i] = sigma[c0 + i] z_i for the n components of the channel whose first Philox call is j0 (component i is output
// i mod 2 of call j0 + i / 2), 0.0 where that sigma is 0.  Rounded product, no contraction into the addition that
// applies it, so that a replay adds the recorded w and gets the same bits.
template <int N>
__device__ __forceinline__ void draw_channel(const SimNoise& nz, unsigned id, unsigned t, unsigned j0, int c0,
                                             double (&w)[N]) {
#pragma unroll
  for (int i = 0; i < N; i += 2) {
    double z[2];
    sim_normal_pair(nz.seed, id, t, j0 + i / 2, z);
#pragma unroll
    for (int k = 0; k < 2 && i + k < N; ++k) {
      const double sg = nz.sigma[c0 + i + k];
      w[i + k] = sg > 0.0 ? __dmul_rn(sg, z[k]) : 0.0;
    }
  }
}

// v + w where sigma > 0, v untouched where it is 0
__device__ __forceinline__ double disturb(double v, double sigma, double w) { return sigma > 0.0 ? __dadd_rn(v, w) : v; }

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

// order-preserving key of s (pass s + 0.0: -0.0 -> +0.0, so that equal positions get equal keys): unsigned order of
// keys = order of s
__device__ __forceinline__ unsigned long long follow_key(double s) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(s);
  return (u >> 63) ? ~u : (u | (1ull << 63));
}

__global__ void __launch_bounds__(128)
mpcb_follow_key_kernel(const __grid_constant__ DevTables Ts, const __grid_constant__ SimArrays sim, int B) {
  const int* __restrict__ route = sim.route;
  const double* __restrict__ x = sim.x;
  unsigned long long* __restrict__ key = sim.f_key;
  unsigned* __restrict__ tag = sim.f_tag;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double s = x[(size_t)b * 5] + 0.0;              // -0.0 -> +0.0: equal positions get equal keys
  const bool live = s <= stop_s(Ts, route, b);          // loop condition (:395), as the FSM kernel evaluates it
  key[b] = follow_key(s);
  const unsigned r = live ? (unsigned)problem_route(route, b, Ts.n) : (unsigned)MPCB_MAX_ROUTES;
  MPCB_ASSERT(r <= (unsigned)MPCB_MAX_ROUTES);
  tag[b] = (r << FOLLOW_IDX_BITS) | (unsigned)b;
}

// over the sorted tags (f_tag + 2 B): lead_idx[b] (-1: none) and lead_sv[b] = (s, v) of the leader (NaN: none)
__global__ void __launch_bounds__(128)
mpcb_follow_leader_kernel(const __grid_constant__ SimArrays sim, int B, double range) {
  const double* __restrict__ x = sim.x;
  const unsigned* __restrict__ sorted = sim.f_tag + 2 * (size_t)B;
  int* __restrict__ lead_idx = sim.lead_idx;
  double* __restrict__ lead_sv = sim.lead_sv;
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

// ---- worlds (mpcb_sim_set_worlds): with world size M, a leader is searched for only among the vehicles [w M, (w+1) M)
// of b's world w.  One launch replaces the key kernel, the two sorts and the leader kernel.  A CTA holds whole worlds
// (blockDim.x a multiple of M): it stages the s keys and route keys of the key kernel in shared memory, and each thread
// scans its world for the successor of (s key, b) among the vehicles with its route key, which is the next tag of the
// sorted route segment.  No workspace; at most M shared-memory reads of each array per thread.
constexpr int WORLD_MAX = 1024;

__global__ void __launch_bounds__(WORLD_MAX)
mpcb_follow_world_kernel(const __grid_constant__ DevTables Ts, const __grid_constant__ SimArrays sim, int B, int M,
                         double range) {
  __shared__ unsigned long long skey[WORLD_MAX];
  __shared__ unsigned sroute[WORLD_MAX];
  const int* __restrict__ route = sim.route;
  const double* __restrict__ x = sim.x;
  int* __restrict__ lead_idx = sim.lead_idx;
  double* __restrict__ lead_sv = sim.lead_sv;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = b < B;                                 // a CTA past B holds whole worlds past B
  unsigned long long k = 0;
  unsigned r = (unsigned)MPCB_MAX_ROUTES;
  double s = 0.0;
  if (in) {
    s = x[(size_t)b * 5];
    const double s0 = s + 0.0;
    k = follow_key(s0);
    if (s0 <= stop_s(Ts, route, b)) r = (unsigned)problem_route(route, b, Ts.n);   // the key kernel's live test
  }
  skey[threadIdx.x] = k;
  sroute[threadIdx.x] = r;
  __syncthreads();
  if (!in) return;
  const int i = threadIdx.x % M, t0 = threadIdx.x - i;   // b's place in its world, the world's first slot in the CTA
  int best = -1;
  unsigned long long bk = 0;
  if (r < (unsigned)MPCB_MAX_ROUTES)
    for (int j = 0; j < M; ++j) {
      MPCB_ASSERT((b - i + j) / M == b / M && b - i + j < B);
      const unsigned long long kj = skey[t0 + j];
      // after (k, i) in the order of (s key, index), and before the best so far (j rises: equal keys keep the first)
      if (sroute[t0 + j] == r && (kj > k || (kj == k && j > i)) && (best < 0 || kj < bk)) { best = j; bk = kj; }
    }
  int lead = -1;
  double ls = nan(""), lv = nan("");
  if (best >= 0) {
    const int j = b - i + best;
    MPCB_ASSERT(j / M == b / M && j != b && j < B);
    const double sj = x[(size_t)j * 5];
    if (sj - s <= range) { lead = j; ls = sj; lv = x[(size_t)j * 5 + 4]; }
  }
  lead_idx[b] = lead;
  lead_sv[2 * b] = ls;
  lead_sv[2 * b + 1] = lv;
}

// CTA width of the world kernel: whole worlds, about 256 threads when worlds are small, one world of M when M >= 256
static int world_threads(int M) { return M >= 256 ? M : (256 / M) * M; }

// ObstaclesFSM.update for every vehicle that is still driving (:330-374); car first, then light (:349, :362).
// alive_cnt / next_cnt: this step's and the next step's counter of the pair sim.alive_cnt.  With following on, the car
// slot takes the nearer of the scripted car and the leader (lead_idx / lead_sv of mpcb_follow_leader_kernel or
// mpcb_follow_world_kernel), which is recorded into hist_lead_idx / hist_lead_sv, and the gap to the leader is folded
// into run_follow.  With measurement noise on, x_meas = x + w_meas is the state step t's solve
// sees; everything here uses the true x.  With noise on, w_meas is recorded into hist_noise.
__global__ void __launch_bounds__(128)
mpcb_fsm_kernel(const __grid_constant__ DevTables Ts, const __grid_constant__ SimArrays sim, int B, double dt, int rec_t,
                int* __restrict__ alive_cnt, int* __restrict__ next_cnt, int follow, const __grid_constant__ SimNoise nz,
                unsigned t) {
  const int* __restrict__ route = sim.route;
  const double* __restrict__ x = sim.x;
  const DevScenario* __restrict__ scen = sim.scen;
  double* __restrict__ fsm_f = sim.fsm_f;
  int* __restrict__ fsm_i = sim.fsm_i;
  int* __restrict__ alive = sim.alive;
  double* __restrict__ obs_sv = sim.obs_sv;
  int* __restrict__ n_obs = sim.n_obs;
  double* __restrict__ hist_obs = sim.hist_obs;
  int* __restrict__ hist_tl = sim.hist_tl;
  int* __restrict__ alive_idx = sim.alive_idx;
  const int* __restrict__ lead_idx = sim.lead_idx;
  const double* __restrict__ lead_sv = follow ? sim.lead_sv : nullptr;
  int* __restrict__ hist_lead_idx = sim.hist_lead_idx;
  double* __restrict__ hist_lead_sv = sim.hist_lead_sv;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) *next_cnt = 0;                                 // the other counter of the pair: next step's list length
  const bool in = b < B;
  const double s = in ? __ldg(x + (size_t)b * 5) : 0.0, v = in ? __ldg(x + (size_t)b * 5 + 4) : 0.0;
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
    const DevScenario sc = ldg(scen + b);
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
      const double ls = __ldg(lead_sv + 2 * b);
      if (!isnan(ls)) {
        // running follower gap, with mpcb_follow_check_kernel's expression (hist_lead_sv's s - hist_x's s)
        double* __restrict__ run_follow = sim.run_follow;
        run_follow[b] = fmin(run_follow[b], ls - s);
        if (!(n == 1 && o[0] <= ls)) { o[0] = ls; o[1] = __ldg(lead_sv + 2 * b + 1); n = 1; }
      }
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
    // running verdicts, with mpcb_sim_check_kernel's expressions: the gap to the scripted car (hist_obs - hist_x's s)
    // and the colour recorded into hist_tl at the first step past the light
    double* __restrict__ run = sim.run + (size_t)b * RUN_W;
    if (!isnan(car_s)) run[RUN_GAP] = fmin(run[RUN_GAP], car_s - s);
    if (s > sc.tl_pos && run[RUN_TL] < 0.0) run[RUN_TL] = (f & F_TL_GREEN) ? 1.0 : 0.0;
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
    const int lead = live ? __ldg(lead_idx + b) : -1;
    MPCB_ASSERT(lead >= -1 && lead < B);
    hist_lead_idx[i] = lead;
    hist_lead_sv[2 * i] = lead >= 0 ? __ldg(lead_sv + 2 * b) : nan("");
    hist_lead_sv[2 * i + 1] = lead >= 0 ? __ldg(lead_sv + 2 * b + 1) : nan("");
  }
  if (nz.on) {
    double w[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (live && nz.meas) {
      double* __restrict__ x_meas = sim.x_meas;
      draw_channel(nz, vehicle_id(nz, b), t, 0u, 0, w);
#pragma unroll
      for (int c = 0; c < 5; ++c) x_meas[(size_t)b * 5 + c] = disturb(__ldg(x + (size_t)b * 5 + c), nz.sigma[c], w[c]);
    }
    double* __restrict__ hist_noise = sim.hist_noise;
    if (hist_noise && rec_t >= 0) {
#pragma unroll
      for (int c = 0; c < 5; ++c) hist_noise[((size_t)rec_t * B + b) * NOISE_W + c] = live ? w[c] : nan("");
    }
  }
}

// plant step (:404-406) for the vehicles that were alive at the start of the step.  With noise on, the step applies
// U*[0] + w_act and adds w_proc to the state it produces (hist_u keeps the commanded U*[0]); both are recorded into
// hist_noise.
__global__ void __launch_bounds__(128)
mpcb_plant_kernel(const __grid_constant__ DevTables Ts, const __grid_constant__ SimArrays sim, int B, double dt,
                  int rec_t, const __grid_constant__ SimNoise nz, unsigned t) {
  const int* __restrict__ route = sim.route;
  double* __restrict__ x = sim.x;
  const double* __restrict__ U = sim.U;
  const int* __restrict__ status = sim.status;
  const int* __restrict__ alive = sim.alive;
  int* __restrict__ steps = sim.steps;
  int* __restrict__ n_unsolved = sim.n_unsolved;
  double* __restrict__ hist_x = sim.hist_x;
  double* __restrict__ hist_u = sim.hist_u;
  int* __restrict__ hist_status = sim.hist_status;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int live = __ldg(alive + b);
  double xs[5];
#pragma unroll
  for (int c = 0; c < 5; ++c) xs[c] = x[(size_t)b * 5 + c];
  const double u1 = __ldg(U + (size_t)b * NV), u2 = __ldg(U + (size_t)b * NV + 1);
  if (hist_x && rec_t >= 0) {                                // state and control of THIS step (before the update)
#pragma unroll
    for (int c = 0; c < 5; ++c) hist_x[((size_t)rec_t * B + b) * 5 + c] = live ? xs[c] : nan("");
    hist_u[((size_t)rec_t * B + b) * 2] = live ? u1 : nan("");
    hist_u[((size_t)rec_t * B + b) * 2 + 1] = live ? u2 : nan("");
    hist_status[(size_t)rec_t * B + b] = live ? __ldg(status + b) : -1;
  }
  double wa[2] = {0.0, 0.0}, wp[5] = {0.0, 0.0, 0.0, 0.0, 0.0};   // actuation and process noise added, 0 where sigma is 0
  if (nz.on) {
    if (live && (nz.act | nz.proc)) {
      const unsigned id = vehicle_id(nz, b);
      if (nz.act) draw_channel(nz, id, t, 3u, NOISE_ACT, wa);
      if (nz.proc) draw_channel(nz, id, t, 4u, NOISE_PROC, wp);
    }
    double* __restrict__ hist_noise = sim.hist_noise;
    if (hist_noise && rec_t >= 0) {
      double* __restrict__ h = hist_noise + ((size_t)rec_t * B + b) * NOISE_W;
#pragma unroll
      for (int c = 0; c < 2; ++c) h[NOISE_ACT + c] = live ? wa[c] : nan("");
#pragma unroll
      for (int c = 0; c < 5; ++c) h[NOISE_PROC + c] = live ? wp[c] : nan("");
    }
  }
  if (!live) return;
  // running verdicts, with mpcb_sim_check_kernel's expressions: |d| of the state before the step, the commanded control
  double* __restrict__ run = sim.run + (size_t)b * RUN_W;
  run[RUN_DEV] = fmax(run[RUN_DEV], fabs(xs[1]));
  run[RUN_U1LO] = fmin(run[RUN_U1LO], u1); run[RUN_U1HI] = fmax(run[RUN_U1HI], u1);
  run[RUN_U2LO] = fmin(run[RUN_U2LO], u2); run[RUN_U2HI] = fmax(run[RUN_U2HI], u2);
  double val[4], slope[4];
  lookup_state(vehicle_table(Ts, route, b), xs[0], val, slope);   // k_ref = get_state(current_s)[3]  (:404)
  const double kref = val[2];
  const double s = xs[0], o = xs[2], k = xs[3], v = xs[4];
  const double a1 = disturb(u1, nz.sigma[NOISE_ACT], wa[0]), a2 = disturb(u2, nz.sigma[NOISE_ACT + 1], wa[1]);
  // x + dt * [v, v o, v (k - k_ref), a1, a2]   (:50-67, :406); no FMA contraction: same rounding as numpy
  const double xn[5] = {__dadd_rn(s, __dmul_rn(dt, v)), __dadd_rn(xs[1], __dmul_rn(dt, __dmul_rn(v, o))),
                        __dadd_rn(o, __dmul_rn(dt, __dmul_rn(v, __dadd_rn(k, -kref)))), __dadd_rn(k, __dmul_rn(dt, a1)),
                        __dadd_rn(v, __dmul_rn(dt, a2))};
#pragma unroll
  for (int c = 0; c < 5; ++c) x[(size_t)b * 5 + c] = disturb(xn[c], nz.sigma[NOISE_PROC + c], wp[c]);
  steps[b] += 1;
  if (__ldg(status + b) != MPCB_SOLVED) n_unsolved[b] += 1;
}

__global__ void mpcb_count_alive_kernel(const __grid_constant__ DevTables Ts, const __grid_constant__ SimArrays sim,
                                        int B) {
  const int* __restrict__ route = sim.route;
  const double* __restrict__ x = sim.x;
  int* __restrict__ count = sim.count;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int live = (b < B && __ldg(x + (size_t)b * 5) <= stop_s(Ts, route, b)) ? 1 : 0;
  const unsigned m = __ballot_sync(0xffffffffu, live);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, __popc(m));
}

// trajectory_tracking_check (sanity_checks.py:79-184) for every vehicle at once, on the recorded histories; one thread
// per vehicle, coalesced over vehicles.  Verdict bits (1 = passed): 0 destination reached (:98-103), 1 stayed on road
// (:106-111), 2 steering within limits +-0.1 (:121-125), 3 acceleration within limits (:127-131), 4 moving obstacle
// avoided, gap >= 1 m (:142-164), 5 red light respected (:167-181), 6 history covers the whole drive.  route == nullptr:
// every vehicle's route is s_total long; else vehicle b's route's s_max.
// (The reference's CPU-time item :134-139 is a property of the host, not of the trajectory; it is not evaluated here.)
// Bits 0-5 from the accumulators, shared with mpcb_sim_running_check_kernel:
__device__ __forceinline__ int tracking_verdict(const DevScenario& sc, double s_final, double s_end, double max_dev,
                                                double u1lo, double u1hi, double u2lo, double u2hi, double min_gap,
                                                bool ran_red, double u1_min, double u1_max, double u2_min,
                                                double u2_max) {
  const double tol = 0.1, lateral = 1.5, safety = 1.0;
  int v = 0;
  if (!(s_final < s_end - 1.0)) v |= 1;
  if (!(max_dev > lateral)) v |= 2;
  if (!(u1lo < u1_min - tol || u1hi > u1_max + tol)) v |= 4;
  if (!(u2lo < u2_min - tol || u2hi > u2_max + tol)) v |= 8;
  if (!(sc.dynamic_obstacle && min_gap < safety)) v |= 16;
  if (!ran_red) v |= 32;
  return v;
}

__global__ void __launch_bounds__(128)
mpcb_sim_check_kernel(const __grid_constant__ DevTables Ts, const __grid_constant__ SimArrays sim, int B, int n_rec,
                      double s_total, double u1_min, double u1_max, double u2_min, double u2_max) {
  const int* __restrict__ route = sim.route;
  const double* __restrict__ x_final = sim.x;
  const int* __restrict__ steps = sim.steps;
  const DevScenario* __restrict__ scen = sim.scen;
  const double* __restrict__ hist_x = sim.hist_x;
  const double* __restrict__ hist_u = sim.hist_u;
  const double* __restrict__ hist_obs = sim.hist_obs;
  const int* __restrict__ hist_tl = sim.hist_tl;
  int* __restrict__ verdict = sim.verdict;
  double* __restrict__ metrics = sim.metrics;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const DevScenario sc = scen[b];
  const int n = min(steps[b], n_rec);
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
  const double s_end = route ? vehicle_table(Ts, route, b).s_max : s_total;
  const bool ran_red = sc.traffic_light && first_pass >= 0 && hist_tl[(size_t)first_pass * B + b] == 0;
  int v = tracking_verdict(sc, s_final, s_end, max_dev, u1lo, u1hi, u2lo, u2hi, min_gap, ran_red, u1_min, u1_max, u2_min,
                           u2_max);
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
mpcb_follow_check_kernel(const __grid_constant__ SimArrays sim, int B, int n_rec) {
  const int* __restrict__ steps = sim.steps;
  const double* __restrict__ hist_x = sim.hist_x;
  const double* __restrict__ hist_lead_sv = sim.hist_lead_sv;
  int* __restrict__ ok = sim.follow_ok;
  double* __restrict__ min_gap = sim.min_gap;
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

// trajectory_tracking_check from the accumulators the FSM and plant kernels keep (R_RUN), into run_verdict and
// run_metrics; bit 6 is always set.  max |d| folds in the current state as the check folds in the final one.
__global__ void __launch_bounds__(128)
mpcb_sim_running_check_kernel(const __grid_constant__ DevTables Ts, const __grid_constant__ SimArrays sim, int B,
                              double s_total, double u1_min, double u1_max, double u2_min, double u2_max) {
  const int* __restrict__ route = sim.route;
  const double* __restrict__ x = sim.x;
  const int* __restrict__ steps = sim.steps;
  const DevScenario* __restrict__ scen = sim.scen;
  const double* __restrict__ run = sim.run;
  int* __restrict__ verdict = sim.run_verdict;
  double* __restrict__ metrics = sim.run_metrics;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const DevScenario sc = scen[b];
  const double* r = run + (size_t)b * RUN_W;
  const double max_dev = fmax(fabs(x[(size_t)b * 5 + 1]), r[RUN_DEV]);
  const double s_final = x[(size_t)b * 5];
  const double s_end = route ? vehicle_table(Ts, route, b).s_max : s_total;
  const bool ran_red = sc.traffic_light && r[RUN_TL] == 0.0;
  verdict[b] = 64 | tracking_verdict(sc, s_final, s_end, max_dev, r[RUN_U1LO], r[RUN_U1HI], r[RUN_U2LO], r[RUN_U2HI],
                                     r[RUN_GAP], ran_red, u1_min, u1_max, u2_min, u2_max);
  metrics[(size_t)b * 4 + 0] = max_dev;
  metrics[(size_t)b * 4 + 1] = r[RUN_GAP];
  metrics[(size_t)b * 4 + 2] = s_final;
  metrics[(size_t)b * 4 + 3] = (double)steps[b];
}

// ---- branching (mpcb_sim_branch): vehicle b takes over the whole state of vehicle parent[b] -------------------------
// A pass copies up to N_SIM arrays of n 4-byte words, one per blockIdx.y.  With parent, a gather: dst is laid out
// [rows][B][w] (one row for the loop state) and word (r, b, k) comes from word (r, parent[b], k) of src; without it a
// straight copy.  Consecutive threads take consecutive words of dst and of a row of src: coalesced on both sides.
// leaders: the words are vehicle indices (-1: none), moved with their vehicle: j >= 0 becomes j + b - parent[b]
// (mpcb_sim_branch_worlds, where b - parent[b] is the distance between the two worlds).
struct BranchCopy { const unsigned* src; unsigned* dst; unsigned long long n; unsigned w, leaders; };
struct BranchPass { BranchCopy c[N_SIM]; };
constexpr int BRANCH_THREADS = 256;

__global__ void __launch_bounds__(BRANCH_THREADS)
mpcb_branch_gather_kernel(const __grid_constant__ BranchPass g, const int* __restrict__ parent, int B) {
  const BranchCopy& c = g.c[blockIdx.y];
  const unsigned* __restrict__ src = c.src;
  unsigned* __restrict__ dst = c.dst;
  const unsigned long long row = (unsigned long long)B * c.w;
  for (unsigned long long e = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; e < c.n;
       e += (unsigned long long)gridDim.x * blockDim.x) {
    if (!parent) { dst[e] = src[e]; continue; }
    const unsigned long long r = e / row, i = e - r * row, b = i / c.w;
    const int p = __ldg(parent + b);
    MPCB_ASSERT(p >= 0 && p < B);
    const unsigned v = src[r * row + (unsigned long long)p * c.w + (i - b * c.w)];
    dst[e] = (c.leaders && (int)v >= 0) ? (unsigned)((int)v + (int)b - p) : v;
  }
}

}  // namespace mpcb

using namespace mpcb;

struct mpcb_sim {
  mpcb_handle h;
  int B, cap, t;              // vehicles, history capacity (steps), steps recorded so far
  int hot_start = 0;          // first pass of step t > 0 starts from step t - 1's plans advanced by one step (mpcb_sim_set_hot_start)
  double dt;
  SimArrays d = {};           // the device arrays: loop state and histories in block[0] (made at create), following and
  char* block[3] = {};        // its histories in block[1] (made the first time following is switched on), the measured
                              // states and the noise history in block[2] (made the first time noise is switched on)
  // following (mpcb_sim_set_follow)
  int follow = 0;
  double follow_range = 0.0;
  size_t f_temp_bytes = 0;    // bytes of d.f_temp
  int world_size = 0;         // mpcb_sim_set_worlds; 0: one world
  SimNoise noise = {};        // mpcb_sim_set_noise; off: every sigma 0
  char* region[N_SIM] = {};   // address of every allocated region (nullptr: not allocated), for mpcb_sim_branch
  // branching (mpcb_sim_branch), made by its first call: the device workspace (the parent indices, then the gathered
  // loop state or one window of history rows), the pinned staging of the parent indices and the event of their copy
  char* branch_ws = nullptr;
  int* branch_parent = nullptr;
  cudaEvent_t branch_copied = nullptr;
  int branch_rows = 0;        // history rows per window
};

// Rows of the history window of mpcb_sim_branch: as many as fit BRANCH_WINDOW_BYTES with every history a simulation
// can have (following and noise may be switched on after the first branch), at least one, at most the capacity.
constexpr size_t BRANCH_WINDOW_BYTES = size_t(1) << 26;
static int branch_window_rows(size_t B, int cap) {
  size_t row = 0;
  for (int r = 0; r < N_SIM; ++r) if (SIM_BYTES[r].branch == HIST) row += SIM_BYTES[r].bytes;
  const size_t w = BRANCH_WINDOW_BYTES / (row * B);
  return (int)(w < 1 ? 1 : w > (size_t)cap ? (size_t)cap : w);
}

static SimMask sim_branch_mask(SimBranch k) {
  SimMask m = 0;
  for (int r = 0; r < N_SIM; ++r) if (SIM_BYTES[r].branch == k) m |= sim_bit(r);
  return m;
}

static DevScenario to_dev_scenario(const mpcb_scenario& c) {
  return DevScenario{c.obs_trigger_s, c.obs_start_s, c.obs_v, c.obs_end_s, c.tl_pos, c.tl_trigger_s,
                     c.tl_stop_duration, c.dynamic_obstacle, c.traffic_light};
}

// The checks on the first n_rec recorded steps of d, on stream st; the verdicts (and the metrics, when metrics is given)
// are copied to the caller's arrays.
static cudaError_t launch_check(mpcb_handle h, const SimArrays& d, int B, int n_rec, double s_total, int* verdict,
                                double* metrics, cudaStream_t st) {
  const mpcb_params& p = h->params;
  mpcb_sim_check_kernel<<<(B + 127) / 128, 128, 0, st>>>(h->dt, d, B, n_rec, s_total, p.u_min[0], p.u_max[0], p.u_min[1],
                                                        p.u_max[1]);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(verdict, d.verdict, sim_bytes(R_VERDICT, B, 0), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && metrics)
    e = cudaMemcpyAsync(metrics, d.metrics, sim_bytes(R_METRICS, B, 0), cudaMemcpyDeviceToHost, st);
  return e;
}

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
  for (char* p : s->block) if (p) cudaFree(p);
  if (s->branch_ws) cudaFree(s->branch_ws);
  if (s->branch_parent) cudaFreeHost(s->branch_parent);
  if (s->branch_copied) cudaEventDestroy(s->branch_copied);
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
  const size_t nb = (size_t)B;
  const SimMask mask = SIM_LOOP | (route ? sim_bit(R_ROUTE) : 0ull) | (history_steps > 0 ? SIM_HIST : 0ull);
  size_t off[N_SIM + 1];
  if (!(s->block[0] = sim_alloc(s->d, nb, (size_t)history_steps, mask, 0, off, s->region))) {
    delete s;
    return MPCB_ERR_NOMEM;
  }
  auto fail = [&](int code) { mpcb_sim_destroy(s); return code; };
  std::vector<DevScenario> hs(nb);
  std::vector<double> hx(nb * 5), hf(nb * 2), hr(nb * RUN_W);
  for (size_t b = 0; b < nb; ++b) {
    double* r = &hr[b * RUN_W];                                         // the check kernel's start values
    r[RUN_DEV] = nan(""); r[RUN_U1LO] = r[RUN_U2LO] = r[RUN_GAP] = BIG; r[RUN_U1HI] = r[RUN_U2HI] = -BIG; r[RUN_TL] = -1.0;
    const mpcb_scenario& c = scen[n_scen == 1 ? 0 : b];
    hs[b] = to_dev_scenario(c);
    if (x_init) for (int k = 0; k < 5; ++k) hx[b * 5 + k] = x_init[b * 5 + k];
    else { hx[b * 5] = hx[b * 5 + 1] = hx[b * 5 + 2] = hx[b * 5 + 3] = 0.0; hx[b * 5 + 4] = 0.5; }   // :382
    hf[b * 2] = c.obs_start_s;                                          // obs_s = obs_start_s (:297)
    hf[b * 2 + 1] = 0.0;
  }
  // start values, synchronous on the default stream: from the host, then zeros
  const struct { int r; const void* src; } start[] = {{R_ROUTE, route}, {R_SCEN, hs.data()}, {R_X, hx.data()},
                                                      {R_FSM_F, hf.data()}, {R_RUN, hr.data()}};
  char* base = s->block[0];
  cudaError_t e;
  for (const auto& c : start)
    if (c.src && (e = cudaMemcpy(base + off[c.r], c.src, sim_bytes(c.r, nb, 0), cudaMemcpyHostToDevice)) != cudaSuccess)
      return fail(cuda_fail(e, "cudaMemcpy"));
  for (int r : {R_FSM_I, R_STEPS, R_N_UNSOLVED, R_ALIVE_CNT, R_STATUS, R_U})
    if ((e = cudaMemset(base + off[r], 0, sim_bytes(r, nb, 0))) != cudaSuccess) return fail(cuda_fail(e, "cudaMemset"));
  *out = s;
  return MPCB_OK;
}

int mpcb_sim_step(mpcb_sim_handle s, int n_steps, void* cuda_stream) {
  if (!s || n_steps < 0) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const SimArrays& d = s->d;
  const int grid = (s->B + 127) / 128;
  for (int k = 0; k < n_steps; ++k) {
    const int rec = (s->t < s->cap) ? s->t : -1;
    int* cnt = d.alive_cnt + (s->t & 1);
    if (s->follow && s->world_size > 0) {                    // leaders of this step within each world
      const int wt = world_threads(s->world_size);
      mpcb_follow_world_kernel<<<(s->B + wt - 1) / wt, wt, 0, st>>>(s->h->dt, d, s->B, s->world_size, s->follow_range);
      CK(cudaGetLastError());
      s->h->launches += 1;
    } else if (s->follow) {                                  // leaders of this step, from the states before it
      const size_t nb = (size_t)s->B;
      mpcb_follow_key_kernel<<<grid, 128, 0, st>>>(s->h->dt, d, s->B);
      CK(cudaGetLastError());
      size_t tb = s->f_temp_bytes;
      CK(cub::DeviceRadixSort::SortPairs(d.f_temp, tb, d.f_key, d.f_key + nb, d.f_tag, d.f_tag + nb, s->B, 0, 64, st));
      tb = s->f_temp_bytes;
      CK(cub::DeviceRadixSort::SortKeys(d.f_temp, tb, d.f_tag + nb, d.f_tag + 2 * nb, s->B, FOLLOW_IDX_BITS, 32, st));
      mpcb_follow_leader_kernel<<<grid, 128, 0, st>>>(d, s->B, s->follow_range);
      CK(cudaGetLastError());
      s->h->launches += 2;                                   // the radix sorts' own kernels are not counted
    }
    mpcb_fsm_kernel<<<grid, 128, 0, st>>>(s->h->dt, d, s->B, s->dt, rec, cnt, d.alive_cnt + ((s->t + 1) & 1), s->follow,
                                          s->noise, (unsigned)s->t);
    CK(cudaGetLastError());
    // the solve runs over the list of vehicles still driving (arrived vehicles are frozen and cost nothing)
    int rc = mpcb_solve_list_internal(s->h, s->B, d.alive_idx, cnt, s->noise.meas ? d.x_meas : d.x, d.obs_sv, d.n_obs,
                                      d.route, d.U, d.status, st, (s->hot_start && s->t > 0) ? d.U : nullptr);
    if (rc != MPCB_OK) return rc;
    mpcb_plant_kernel<<<grid, 128, 0, st>>>(s->h->dt, d, s->B, s->dt, rec, s->noise, (unsigned)s->t);
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
  if (!s->block[1]) {
    CK(cudaSetDevice(s->h->device));
    const size_t nb = (size_t)s->B, T = (size_t)s->cap;
    size_t t1 = 0, t2 = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, t1, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                       (unsigned*)nullptr, (unsigned*)nullptr, s->B, 0, 64));
    CK(cub::DeviceRadixSort::SortKeys(nullptr, t2, (unsigned*)nullptr, (unsigned*)nullptr, s->B, FOLLOW_IDX_BITS, 32));
    const size_t temp = t1 > t2 ? t1 : t2;
    size_t off[N_SIM + 1];
    if (!(s->block[1] = sim_alloc(s->d, nb, T, SIM_FOLLOW | (T > 0 ? SIM_FOLLOW_HIST : 0ull), temp, off, s->region)))
      return MPCB_ERR_NOMEM;
    s->f_temp_bytes = temp;
    // the running gap starts at the check's 1e30; rows of steps taken with following off stay -1 / NaN (all-ones
    // bytes: int -1, a double NaN)
    const std::vector<double> big(nb, BIG);
    CK(cudaMemcpy(s->d.run_follow, big.data(), sim_bytes(R_RUN_FOLLOW, nb, 0), cudaMemcpyHostToDevice));
    if (T > 0) {
      CK(cudaMemset(s->d.hist_lead_idx, 0xff, sim_bytes(R_HIST_LEAD_IDX, nb, T)));
      CK(cudaMemset(s->d.hist_lead_sv, 0xff, sim_bytes(R_HIST_LEAD_SV, nb, T)));
      CK(cudaStreamSynchronize(0));
    }
  }
  s->follow = 1;
  s->follow_range = follow_range;
  return MPCB_OK;
}

int mpcb_sim_set_noise(mpcb_sim_handle s, unsigned long long seed, int first_id, const double* sigma_meas,
                       const double* sigma_act, const double* sigma_proc) {
  if (!s || first_id < 0 || (long long)first_id + s->B > (1ll << 31)) return MPCB_ERR_INVALID;
  SimNoise nz = {};
  nz.seed = seed;
  nz.first_id = first_id;
  const struct { const double* sigma; int n, c0; int* on; } ch[] = {
      {sigma_meas, 5, 0, &nz.meas}, {sigma_act, 2, NOISE_ACT, &nz.act}, {sigma_proc, 5, NOISE_PROC, &nz.proc}};
  for (const auto& c : ch)
    for (int i = 0; i < c.n; ++i) {
      const double v = c.sigma ? c.sigma[i] : 0.0;
      if (!(v >= 0.0) || !isfinite(v)) return MPCB_ERR_INVALID;
      nz.sigma[c.c0 + i] = v;
      if (v > 0.0) *c.on = 1;
    }
  nz.on = nz.meas | nz.act | nz.proc;
  if (nz.on && !s->block[2]) {
    CK(cudaSetDevice(s->h->device));
    const size_t nb = (size_t)s->B, T = (size_t)s->cap;
    SimArrays d = s->d;
    size_t off[N_SIM + 1];
    char* region[N_SIM] = {};
    char* base = sim_alloc(d, nb, T, sim_bit(R_X_MEAS) | (T > 0 ? sim_bit(R_HIST_NOISE) : 0ull), 0, off, region);
    if (!base) return MPCB_ERR_NOMEM;
    // rows of steps taken with noise off stay NaN (all-ones bytes)
    cudaError_t e = T > 0 ? cudaMemset(d.hist_noise, 0xff, sim_bytes(R_HIST_NOISE, nb, T)) : cudaSuccess;
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) { cudaFree(base); return cuda_fail(e, "mpcb_sim_set_noise"); }
    s->block[2] = base;
    s->d = d;
    for (int r = 0; r < N_SIM; ++r) if (region[r]) s->region[r] = region[r];
  }
  s->noise = nz;
  return MPCB_OK;
}

int mpcb_sim_noise_history(mpcb_sim_handle s, int* n_recorded, double* hist_w, void* cuda_stream) {
  if (!s) return MPCB_ERR_INVALID;
  const int nt = s->t < s->cap ? s->t : s->cap;
  if (n_recorded) *n_recorded = nt;
  const size_t n = (size_t)nt * s->B * NOISE_W;
  if (n == 0 || !hist_w) return MPCB_OK;
  if (!s->d.hist_noise) {                                    // noise never switched on: nothing recorded
    for (size_t i = 0; i < n; ++i) hist_w[i] = nan("");
    return MPCB_OK;
  }
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  CK(cudaMemcpyAsync(hist_w, s->d.hist_noise, sim_bytes(R_HIST_NOISE, s->B, nt), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

int mpcb_sim_follow_history(mpcb_sim_handle s, int* n_recorded, int* hist_lead_idx, double* hist_lead_sv,
                            void* cuda_stream) {
  if (!s) return MPCB_ERR_INVALID;
  const int nt = s->t < s->cap ? s->t : s->cap;
  if (n_recorded) *n_recorded = nt;
  const size_t n = (size_t)nt * s->B;
  if (n == 0 || (!hist_lead_idx && !hist_lead_sv)) return MPCB_OK;
  if (!s->d.hist_lead_idx) {                                 // following never switched on: nothing recorded
    if (hist_lead_idx) for (size_t i = 0; i < n; ++i) hist_lead_idx[i] = -1;
    if (hist_lead_sv) for (size_t i = 0; i < 2 * n; ++i) hist_lead_sv[i] = nan("");
    return MPCB_OK;
  }
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const auto D2H = cudaMemcpyDeviceToHost;
  if (hist_lead_idx) CK(cudaMemcpyAsync(hist_lead_idx, s->d.hist_lead_idx, sim_bytes(R_HIST_LEAD_IDX, s->B, nt), D2H, st));
  if (hist_lead_sv) CK(cudaMemcpyAsync(hist_lead_sv, s->d.hist_lead_sv, sim_bytes(R_HIST_LEAD_SV, s->B, nt), D2H, st));
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

int mpcb_sim_follow_check(mpcb_sim_handle s, int* ok, double* min_gap, void* cuda_stream) {
  if (!s || !ok || s->cap < 1) return MPCB_ERR_INVALID;
  const size_t nb = (size_t)s->B;
  if (!s->d.hist_lead_sv) {                                  // following never switched on: no leader, ever
    for (size_t b = 0; b < nb; ++b) { ok[b] = 1; if (min_gap) min_gap[b] = BIG; }
    return MPCB_OK;
  }
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int nt = s->t < s->cap ? s->t : s->cap;
  mpcb_follow_check_kernel<<<(s->B + 127) / 128, 128, 0, st>>>(s->d, s->B, nt);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ok, s->d.follow_ok, sim_bytes(R_FOLLOW_OK, nb, 0), cudaMemcpyDeviceToHost, st));
  if (min_gap) CK(cudaMemcpyAsync(min_gap, s->d.min_gap, sim_bytes(R_MIN_GAP, nb, 0), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  s->h->launches += 1;
  return MPCB_OK;
}

int mpcb_sim_alive(mpcb_sim_handle s, int* n_alive, void* cuda_stream) {
  if (!s || !n_alive) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  CK(cudaMemsetAsync(s->d.count, 0, sim_bytes(R_COUNT, 0, 0), st));
  mpcb_count_alive_kernel<<<(s->B + 127) / 128, 128, 0, st>>>(s->h->dt, s->d, s->B);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(n_alive, s->d.count, sim_bytes(R_COUNT, 0, 0), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

int mpcb_sim_state(mpcb_sim_handle s, double* x, int* steps, int* n_unsolved, void* cuda_stream) {
  if (!s) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const size_t nb = (size_t)s->B;
  const auto D2H = cudaMemcpyDeviceToHost;
  if (x) CK(cudaMemcpyAsync(x, s->d.x, sim_bytes(R_X, nb, 0), D2H, st));
  if (steps) CK(cudaMemcpyAsync(steps, s->d.steps, sim_bytes(R_STEPS, nb, 0), D2H, st));
  if (n_unsolved) CK(cudaMemcpyAsync(n_unsolved, s->d.n_unsolved, sim_bytes(R_N_UNSOLVED, nb, 0), D2H, st));
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

int mpcb_sim_check(mpcb_sim_handle s, int* verdict, double* metrics, void* cuda_stream) {
  if (!s || !verdict || s->cap < 1) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int nt = s->t < s->cap ? s->t : s->cap;
  CK(launch_check(s->h, s->d, s->B, nt, s->h->dt.t[0].s_max, verdict, metrics, st));
  CK(cudaStreamSynchronize(st));
  s->h->launches += 1;
  return MPCB_OK;
}

int mpcb_sim_running_check(mpcb_sim_handle s, int* verdict, double* metrics, void* cuda_stream) {
  if (!s || !verdict) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(s->h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const mpcb_params& p = s->h->params;
  const size_t nb = (size_t)s->B;
  mpcb_sim_running_check_kernel<<<(s->B + 127) / 128, 128, 0, st>>>(s->h->dt, s->d, s->B, s->h->dt.t[0].s_max, p.u_min[0],
                                                                    p.u_max[0], p.u_min[1], p.u_max[1]);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(verdict, s->d.run_verdict, sim_bytes(R_RUN_VERDICT, nb, 0), cudaMemcpyDeviceToHost, st));
  if (metrics) CK(cudaMemcpyAsync(metrics, s->d.run_metrics, sim_bytes(R_RUN_METRICS, nb, 0), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  s->h->launches += 1;
  return MPCB_OK;
}

}  // extern "C"

// mpcb_sim_branch and mpcb_sim_branch_worlds on checked parents: vehicle b takes over the whole state of parent[b];
// leaders: the recorded leader indices are moved with their vehicle (BranchCopy::leaders).
static int sim_gather(mpcb_sim* s, const int* parent, bool leaders, void* cuda_stream) {
  CK(cudaSetDevice(s->h->device));
  const size_t nb = (size_t)s->B;
  SimMask have = 0;
  for (int r = 0; r < N_SIM; ++r) if (s->region[r]) have |= sim_bit(r);
  // workspace: the parent indices, then room for the gathered loop state or one window of every history there can be
  // (following, whose block holds loop state too, may be switched on after the first call)
  const SimMask state = sim_branch_mask(STATE) & have, hist = sim_branch_mask(HIST);
  size_t soff[N_SIM + 1], hoff[N_SIM + 1];
  const size_t pbytes = (nb * sizeof(int) + 255) & ~(size_t)255;
  if (!s->branch_ws) {
    const int rows = s->cap > 0 ? branch_window_rows(nb, s->cap) : 0;
    sim_layout(nb, 0, sim_branch_mask(STATE), 0, soff);
    sim_layout(nb, (size_t)rows, rows > 0 ? hist : 0ull, 0, hoff);
    char* ws = nullptr;
    int* hp = nullptr;
    cudaEvent_t ev = nullptr;
    if (cudaMalloc((void**)&ws, pbytes + (soff[N_SIM] > hoff[N_SIM] ? soff[N_SIM] : hoff[N_SIM])) != cudaSuccess ||
        cudaMallocHost((void**)&hp, nb * sizeof(int)) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      if (ws) cudaFree(ws);
      if (hp) cudaFreeHost(hp);
      return MPCB_ERR_NOMEM;
    }
    s->branch_ws = ws; s->branch_parent = hp; s->branch_copied = ev; s->branch_rows = rows;
    CK(cudaStreamSynchronize(0));
  }
  sim_layout(nb, 0, state, 0, soff);
  sim_layout(nb, (size_t)s->branch_rows, s->branch_rows > 0 ? hist : 0ull, 0, hoff);
  cudaStream_t st = (cudaStream_t)cuda_stream;
  // the caller's parent is read here; the staging is reused once the previous call's copy has left it
  CK(cudaEventSynchronize(s->branch_copied));
  memcpy(s->branch_parent, parent, nb * sizeof(int));
  const int* dpar = (const int*)s->branch_ws;
  CK(cudaMemcpyAsync((void*)dpar, s->branch_parent, nb * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(s->branch_copied, st));
  char* ws = s->branch_ws + pbytes;
  // one pass: gather regions of mask (rows from row0 on) into the workspace at off, then copy them back
  auto pass = [&](SimMask mask, const size_t (&off)[N_SIM + 1], size_t row0, size_t rows) -> cudaError_t {
    BranchPass g = {}, back = {};
    int n = 0;
    unsigned long long most = 0;
    for (int r = 0; r < N_SIM; ++r) {
      if (!((mask >> r) & 1ull)) continue;
      const size_t bytes = SIM_BYTES[r].bytes, at = row0 * nb * bytes, words = rows * nb * bytes / 4;
      g.c[n] = BranchCopy{(const unsigned*)(s->region[r] + at), (unsigned*)(ws + off[r]), words, (unsigned)(bytes / 4),
                          leaders && r == R_HIST_LEAD_IDX ? 1u : 0u};
      back.c[n] = BranchCopy{(const unsigned*)(ws + off[r]), (unsigned*)(s->region[r] + at), words, g.c[n].w, 0u};
      if (words > most) most = words;
      ++n;
    }
    if (n == 0) return cudaSuccess;
    const unsigned long long blocks = (most + BRANCH_THREADS - 1) / BRANCH_THREADS;
    const dim3 grid((unsigned)(blocks < 2048 ? blocks : 2048), (unsigned)n);
    mpcb_branch_gather_kernel<<<grid, BRANCH_THREADS, 0, st>>>(g, dpar, s->B);
    mpcb_branch_gather_kernel<<<grid, BRANCH_THREADS, 0, st>>>(back, nullptr, s->B);
    s->h->launches += 2;
    return cudaGetLastError();
  };
  CK(pass(state, soff, 0, 1));
  const int nt = s->t < s->cap ? s->t : s->cap;
  for (int row0 = 0; row0 < nt; row0 += s->branch_rows)
    CK(pass(hist & have, hoff, (size_t)row0, (size_t)(nt - row0 < s->branch_rows ? nt - row0 : s->branch_rows)));
  return MPCB_OK;
}

extern "C" {

int mpcb_sim_branch(mpcb_sim_handle s, const int* parent, void* cuda_stream) {
  if (!s || !parent || s->follow) return MPCB_ERR_INVALID;   // a copy would follow its parent at gap 0
  for (int b = 0; b < s->B; ++b)
    if (parent[b] < 0 || parent[b] >= s->B) return MPCB_ERR_INVALID;
  return sim_gather(s, parent, false, cuda_stream);
}

int mpcb_sim_set_worlds(mpcb_sim_handle s, int world_size) {
  if (!s || world_size < 0 || world_size > WORLD_MAX || (world_size > 0 && s->B % world_size != 0))
    return MPCB_ERR_INVALID;
  s->world_size = world_size;
  return MPCB_OK;
}

int mpcb_sim_branch_worlds(mpcb_sim_handle s, const int* parent_world, void* cuda_stream) {
  if (!s || !parent_world || s->world_size < 1) return MPCB_ERR_INVALID;
  const int M = s->world_size, W = s->B / M;
  for (int w = 0; w < W; ++w)
    if (parent_world[w] < 0 || parent_world[w] >= W) return MPCB_ERR_INVALID;
  std::vector<int> parent((size_t)s->B);
  for (int w = 0; w < W; ++w)
    for (int i = 0; i < M; ++i) parent[(size_t)w * M + i] = parent_world[w] * M + i;
  return sim_gather(s, parent.data(), true, cuda_stream);
}

int mpcb_sim_running_follow_check(mpcb_sim_handle s, int* ok, double* min_gap, void* cuda_stream) {
  if (!s || !ok) return MPCB_ERR_INVALID;
  const size_t nb = (size_t)s->B;
  std::vector<double> own(min_gap ? 0 : nb);
  double* g = min_gap ? min_gap : own.data();
  if (!s->d.run_follow) {                                    // following never switched on: no leader, ever
    for (size_t b = 0; b < nb; ++b) g[b] = BIG;
  } else {
    CK(cudaSetDevice(s->h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    CK(cudaMemcpyAsync(g, s->d.run_follow, sim_bytes(R_RUN_FOLLOW, nb, 0), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  for (size_t b = 0; b < nb; ++b) ok[b] = g[b] < 1.0 ? 0 : 1;   // mpcb_follow_check_kernel's safety test
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
  const size_t nb = (size_t)B;
  std::vector<DevScenario> hs(nb);
  for (size_t b = 0; b < nb; ++b) hs[b] = to_dev_scenario(scen[b]);
  // one block laid out as a simulation's: the caller's arrays (x_final in x), the verdicts and the metrics
  const struct { int r; const void* src; } in[] = {{R_SCEN, hs.data()}, {R_X, x_final}, {R_STEPS, steps},
                                                   {R_HIST_X, hist_x}, {R_HIST_U, hist_u}, {R_HIST_OBS, hist_obs},
                                                   {R_HIST_TL, hist_tl}};
  SimMask mask = sim_bit(R_VERDICT) | sim_bit(R_METRICS);
  for (const auto& c : in) mask |= sim_bit(c.r);
  SimArrays d = {};
  size_t off[N_SIM + 1];
  char* base = sim_alloc(d, nb, (size_t)T, mask, 0, off);
  if (!base) return MPCB_ERR_NOMEM;
  cudaStream_t st = h->stream;
  cudaError_t e = cudaSuccess;
  for (const auto& c : in)
    if (e == cudaSuccess) e = cudaMemcpyAsync(base + off[c.r], c.src, sim_bytes(c.r, nb, T), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = launch_check(h, d, B, T, s_total, verdict, metrics, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(base);
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
  if (nt > 0) {
    const struct { int r; void* dst; const void* src; } out[] = {
        {R_HIST_X, hist_x, s->d.hist_x}, {R_HIST_U, hist_u, s->d.hist_u}, {R_HIST_OBS, hist_obs, s->d.hist_obs},
        {R_HIST_STATUS, hist_status, s->d.hist_status}, {R_HIST_TL, hist_tl, s->d.hist_tl}};
    for (const auto& c : out)
      if (c.dst) CK(cudaMemcpyAsync(c.dst, c.src, sim_bytes(c.r, s->B, nt), cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  return MPCB_OK;
}

}  // extern "C"
