/* mpcb200.h -- C ABI of libmpcb200.so: batched tracking-MPC solver for NVIDIA B200 (sm_100a).
 *
 * Drop-in boundary for ONE hot path of medinammartin3/Safe-Autonomous-Driving-MPC: the per-timestep
 * tracking MPC `TrajectoryTracker.solve(x0, obstacles)` (reference trajectory_tracking.py:213-263) together
 * with the functions it evaluates (predict :87-114, cost :116-152, constraints :155-211, warm start :223-246)
 * and the reference-signal table it queries (trajectory_loader.py:13-30, :64-102).
 *
 * The reference has no FFI of its own (it is pure Python); these entry points are what a ctypes binding on
 * the reference side would call -- see INTEGRATION.md for that stub.  Plain pointers and sizes only.
 * All functions return 0 on success and a negative mpcb_status on failure; nothing throws or aborts.
 * There is no CPU fallback: every compute entry point fails with MPCB_ERR_CUDA if no sm_100 device is usable.
 */
#ifndef MPCB200_H
#define MPCB200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MPCB_HORIZON 5      /* N, trajectory_tracking.py:18 */
#define MPCB_NU 10          /* 2N decision variables, row-major [u1_0,u2_0,...] (:69-85) */
#define MPCB_MAX_OBS 2      /* ObstaclesFSM emits at most {car, light} (:330-374) */
#define MPCB_MAX_CONS 45    /* 5*(7+MAX_OBS) rows of constraints_wrapper (:164-209) */

typedef enum mpcb_status {
  MPCB_OK = 0,
  MPCB_ERR_INVALID = -1,    /* bad argument (null pointer, K < 2, B < 0, ...) */
  MPCB_ERR_CUDA = -2,       /* CUDA runtime error; mpcb_last_cuda_error() has the text */
  MPCB_ERR_NOMEM = -3,
  MPCB_ERR_UNSUPPORTED = -4 /* parameter set outside what the kernel was compiled for (N != 5) */
} mpcb_status;

/* per-problem solver exit flags written to status_out */
#define MPCB_SOLVED 0       /* SQP step and QP residuals under tolerance, all constraints satisfied */
#define MPCB_MAXITER 1      /* iteration caps hit; returned point satisfies the constraints to feas_tol */
#define MPCB_INFEASIBLE 2   /* infeasibility certificate, or returned point violates a constraint > feas_tol */
#define MPCB_BAD_ROUTE 3    /* routed solve: the problem's route is outside [0, n_routes); not solved */

#define MPCB_MAX_ROUTES 16  /* reference-signal tables one handle can hold (mpcb_create_routes) */

/* Mirrors the attributes of TrajectoryTracker.__init__ (trajectory_tracking.py:12-47) one to one, followed by
 * the solver controls of this implementation.  Fill with mpcb_default_params() first. */
typedef struct mpcb_params {
  double dt;                       /* :17  0.2 */
  int N;                           /* :18  5 (only 5 is supported) */
  double u_min[2], u_max[2];       /* :31-32 */
  double vehicle_radius;           /* :33 */
  double w_d, w_o, w_v, w_u1, w_u2;/* :36-40 */
  double obstacle_safety_distance; /* :43 */
  double max_time_2_obs;           /* :44 */
  double wheelbase;                /* :45 */
  double lane_width;               /* :46 */
  double safe_lane_margin;         /* :47 */
  double brake_lookahead;          /* :233  40.0 (literal in solve) */
  double brake_guess;              /* :241  -2.0 (literal in solve) */
  /* solver controls (no counterpart in the reference, which uses SLSQP ftol=1e-3/maxiter=15) */
  int max_rounds;                  /* linearise->QP rounds, default 10 */
  int max_segments;                /* ADMM segments per round, default 12 */
  int segment_iters;               /* ADMM iterations per segment, default 10 */
  double rho_lo, rho_hi, rho_init; /* per-row step-size ladder, defaults 0.1, 1e4, 1.0 (x10 per rung) */
  double alpha;                    /* over-relaxation, default 1.6 */
  double eps_prim, eps_dual;       /* QP residual tolerances (inf-norm), defaults 1e-9, 1e-8 */
  double eps_infeas;               /* infeasibility-certificate tolerance, default 1e-4 */
  double step_tol;                 /* SQP termination on |dU|_inf, default 1e-5 (the accepted iterate is
                                      the NEXT one: its error is ~1e-2 of that, 3e-7 measured) */
  double feas_tol;                 /* constraint tolerance for flags / active set, default 1e-6 */
  /* two-pass scheme: a first pass with two-level step sizes (inactive rows ~0, active rows a large augmented-
   * Lagrangian weight: a primal-dual active-set iteration run on the ADMM machinery) solves the non-degenerate
   * problems in a few iterations; whatever it does not certify as solved is re-solved from scratch by the robust
   * ladder pass above.  fast_pass = 0 disables the first pass. */
  int fast_pass;                   /* default 1 */
  double fast_rho_off, fast_rho_on;/* defaults 1e-9, 1e6 */
  int fast_max_rounds;             /* default 6 */
  int fast_max_segments;           /* default 4 */
  int fast_segment_iters;          /* default 2 */
  int coop_pass2;                  /* robust pass executed by one warp per problem (latency), default 1 */
  int coop_max_batch;              /* batches up to this size run the first pass one warp per problem too, default 3072
                                      (measured crossover with the thread-per-problem first pass: ~3,700 problems) */
  /* tighter caps of the two-level policy inside the thread-per-problem kernel, where the slowest problem of a CTA
   * holds up the other 127: what these caps cut off goes to the second pass (one warp per problem, nobody waits)
   * like everything else the first pass does not certify */
  int thread_max_rounds;           /* default 5 */
  int thread_max_segments;         /* default 1: one active-set update (two ADMM iterations) per linearisation */
  int thread_fail_rounds;          /* rounds whose QP did not close within thread_max_segments that the first pass tolerates
                                      (the ADMM state carries over: the active-set search continues on the next
                                      linearisation; only a round with a closed QP and a small step certifies), default 3 */
} mpcb_params;

typedef struct mpcb_ctx* mpcb_handle;
typedef struct mpcb_table* mpcb_table_handle;

/* Fill *p with the reference's constants and the default solver controls. */
int mpcb_default_params(mpcb_params* p);

/* Reference-signal table (host object, no GPU needed).  Replaces TrajectoryLoader.__init__'s table part
 * (trajectory_loader.py:13-30, :64-77, :84).
 * ref_X: [K][5] rows [s,d,o,k,v]; ref_U: [KU][2] rows [u1,u2] (KU = K-1 in the reference's files).
 * Applies the strict-monotone repair of s (:27-30) and the "controls see the first min(K,KU) knots" rule (:73-77). */
int mpcb_table_create(mpcb_table_handle* out, const double* ref_X, int K, const double* ref_U, int KU);
int mpcb_table_destroy(mpcb_table_handle t);
/* Scalar queries; replace TrajectoryLoader.get_state / get_control (trajectory_loader.py:86-102) for callers such
 * as run_simulation's plant step (trajectory_tracking.py:404). */
int mpcb_table_get_state(mpcb_table_handle t, double s, double out5[5]);
int mpcb_table_get_control(mpcb_table_handle t, double s, double out2[2]);
/* Binary cache of a table (the wire format feeding every config, instead of re-parsing JSON per process): the inputs of
 * mpcb_table_create behind a 16-byte header; loading re-applies the repair rules of mpcb_table_create. */
int mpcb_table_save(mpcb_table_handle t, const char* path);
int mpcb_table_load(mpcb_table_handle* out, const char* path);
double mpcb_table_s_max(mpcb_table_handle t);
int mpcb_table_knots(mpcb_table_handle t);
int mpcb_table_control_knots(mpcb_table_handle t);                       /* KU as given */
int mpcb_table_raw(mpcb_table_handle t, double* ref_X, double* ref_U);   /* copies the inputs back out ([K][5], [KU][2]) */

/* Solver context on CUDA device `device`: uploads the table, derives the constants.
 * Replaces TrajectoryTracker.__init__ (trajectory_tracking.py:12-47).  The table may be destroyed afterwards. */
int mpcb_create(mpcb_handle* out, const mpcb_params* p, mpcb_table_handle t, int device);
int mpcb_destroy(mpcb_handle h);

/* Solver context over several routes: tables[0 .. n_routes-1] (1 <= n_routes <= MPCB_MAX_ROUTES, none NULL; checked
 * before any CUDA call).  Route r of a routed call (mpcb_solve_batch_routes, mpcb_sim_create_routes) is tables[r].
 * mpcb_create(out, p, t, device) is mpcb_create_routes(out, p, &t, 1, device).
 * Every entry point without a route argument -- mpcb_solve_batch, the host-buffer and asynchronous entry points,
 * mpcb_eval_batch, the planner evaluators (mpcb_hs_*), mpcb_sim_create, mpcb_check_histories -- behaves on a multi-route
 * handle exactly as on a single-route handle of tables[0]: every problem or vehicle is on route 0. */
int mpcb_create_routes(mpcb_handle* out, const mpcb_params* p, const mpcb_table_handle* tables, int n_routes, int device);
int mpcb_n_routes(mpcb_handle h);   /* number of routes of the handle (1 for mpcb_create) */

/* Solve B independent problems.  DEVICE pointers; asynchronous on `cuda_stream` (a cudaStream_t, may be 0).
 *   x0      [B][5]             current states [s,d,o,k,v]
 *   obs_sv  [B][MAX_OBS][2]    (s, v) per obstacle, first n_obs[b] entries used
 *   n_obs   [B]                0..2
 * outputs (any may be NULL except U_out):
 *   U_out   [B][5][2]   optimal controls           Xpred_out [B][6][5]  predict(x0, U*)  (:261)
 *   obj_out [B]         cost(U*)                   status_out [B]       MPCB_SOLVED / MAXITER / INFEASIBLE
 *   iters_out [B][2]    {linearisation rounds, total ADMM iterations}
 *   cmin_out [B]        min over constraints_wrapper(U*) rows (reference order and sign)
 *   active_out [B]      bit r (r < 5*(7+n_obs)) set when constraint row r <= feas_tol; bit 45+i set when
 *                       variable i sits on a bound (within feas_tol)
 * U_out and Xpred_out must be 16-byte aligned (any cudaMalloc / torch allocation is); MPCB_ERR_INVALID otherwise.
 * Replaces TrajectoryTracker.solve (trajectory_tracking.py:213-263) for a batch. */
int mpcb_solve_batch(mpcb_handle h, int B, const double* x0, const double* obs_sv, const int* n_obs,
                     double* U_out, double* Xpred_out, double* obj_out, int* status_out, int* iters_out,
                     double* cmin_out, unsigned long long* active_out, void* cuda_stream);

/* mpcb_solve_batch over several routes: problem b follows route[b] (DEVICE [B]; NULL: route 0 for every problem, bitwise
 * identical to mpcb_solve_batch).  A problem's answer depends only on its own inputs and route, not on the routes of
 * the other problems of the batch.  A problem whose route is outside [0, n_routes) is not solved and reads no table:
 * status MPCB_BAD_ROUTE, U, Xpred, obj and cmin NaN, iters and active 0. */
int mpcb_solve_batch_routes(mpcb_handle h, int B, const double* x0, const double* obs_sv, const int* n_obs,
                            const int* route, double* U_out, double* Xpred_out, double* obj_out, int* status_out,
                            int* iters_out, double* cmin_out, unsigned long long* active_out, void* cuda_stream);

/* Same, with HOST buffers: copies inputs to the device, solves, copies results back and synchronises.
 * Pinned buffers (mpcb_host_alloc) make the copies asynchronous DMA. */
int mpcb_solve_batch_host(mpcb_handle h, int B, const double* x0, const double* obs_sv, const int* n_obs,
                          double* U_out, double* Xpred_out, double* obj_out, int* status_out, int* iters_out,
                          double* cmin_out, unsigned long long* active_out);

/* Closed-loop form of the host entry point: only what run_simulation consumes comes back (trajectory_tracking.py:260,
 * :401-406) -- u0_out [B][2] = U*[0], status_out [B] (may be NULL), obj_out [B] (may be NULL): 20-28 bytes per solve over
 * PCIe instead of 356.  Same solve, same flags as mpcb_solve_batch_host. */
int mpcb_solve_batch_host_u0(mpcb_handle h, int B, const double* x0, const double* obs_sv, const int* n_obs,
                             double* u0_out, int* status_out, double* obj_out);

/* Asynchronous form of the two host entry points above, for callers that keep several batches in flight (one handle per
 * batch in flight): enqueues the host-to-device copies, the solve and the device-to-host copies on the handle's own
 * streams and returns; the results are in the caller's buffers after mpcb_wait(h).  Buffers must be page-locked
 * (mpcb_host_alloc) for the copies to run asynchronously and must stay untouched until mpcb_wait returns.  U_out may be
 * NULL when u0_out is given (closed-loop form); any other output may be NULL.  With three handles the copies of one
 * batch overlap the kernels of the next and the latency tail of the robust pass of the one before (measured on B200:
 * see DESIGN.md).  Batches of up to 2,048 problems go through the packed staging path and complete inside the call. */
int mpcb_solve_batch_host_async(mpcb_handle h, int B, const double* x0, const double* obs_sv, const int* n_obs,
                                double* U_out, double* Xpred_out, double* obj_out, int* status_out, int* iters_out,
                                double* cmin_out, unsigned long long* active_out, double* u0_out);
int mpcb_wait(mpcb_handle h);

/* Evaluate the model functions at given controls (no optimisation).  DEVICE pointers, async on stream.
 *   U [B][10] -> Xpred_out [B][6][5] (predict), cost_out [B] (cost), cons_out [B][45] (constraints_wrapper rows,
 *   first 5*(7+n_obs[b]) valid, rest NaN), lin_out [B][150] (the solver's linearisation at U, packed: Gauss-Newton
 *   Hessian lower triangle [0:55), q = g - H U [55:65), d(d_j)/dU rows j=2..5 [65:105), d(o_j)/dU rows [105:145),
 *   5 zeros), warm_out [B][10] (the warm start of :223-246, unclipped).  Any output may be NULL. */
int mpcb_eval_batch(mpcb_handle h, int B, const double* x0, const double* U, const double* obs_sv,
                    const int* n_obs, double* Xpred_out, double* cost_out, double* cons_out, double* lin_out,
                    double* warm_out, void* cuda_stream);

/* Pinned host memory helpers (cudaHostAlloc / cudaFreeHost). */
int mpcb_host_alloc(void** ptr, unsigned long long bytes);
int mpcb_host_free(void* ptr);
/* Device memory helpers so that hosts without a tensor library can hold device buffers. */
int mpcb_device_alloc(mpcb_handle h, void** ptr, unsigned long long bytes);
int mpcb_device_free(mpcb_handle h, void* ptr);
int mpcb_memcpy_h2d(mpcb_handle h, void* dst, const void* src, unsigned long long bytes);
int mpcb_memcpy_d2h(mpcb_handle h, void* dst, const void* src, unsigned long long bytes);

/* Device time in milliseconds of the kernel launched by the last mpcb_solve_batch* call on this handle
 * (CUDA events on the launching stream; synchronises that stream). */
int mpcb_last_kernel_ms(mpcb_handle h, float* ms);
/* Device time of the two passes of the last solve (first: two-level pass incl. the list reset; second: robust pass over
 * the problems the first did not certify) and how many problems the second pass handled. */
int mpcb_last_pass_ms(mpcb_handle h, float* first_ms, float* second_ms, int* n_second);
/* Execution shape of the first pass of the last solve call: 0 one thread per problem (large batches), 1 one warp per
 * problem (batches up to coop_max_batch).  Lets a test assert which kernel produced an answer. */
int mpcb_last_first_pass_shape(mpcb_handle h);
/* Number of kernels this library has launched on this handle since creation. */
unsigned long long mpcb_launch_count(mpcb_handle h);

/* FP64 FMA-pipe peak probe: runs a register-resident DFMA loop on the handle's device and returns
 * the measured TFLOP/s (2 flop per DFMA).  Used by bench.py as the roofline denominator. */
int mpcb_measure_fp64_peak(mpcb_handle h, double* tflops, float* ms);

/* ---------------------------------------------------------------------------------------------------------
 * Planner function evaluation (north_star item (c)): the offline Hermite-Simpson NLP of trajectory_planning.py.
 * The outer optimisation loop stays on the host; these entry points evaluate, for all collocation intervals of a
 * batch of chunks at once, what the reference evaluates closure by closure with finite differences.
 * k_ref(s) is the curvature column of the handle's reference-signal table with linear extrapolation
 * (TrajectoryLoader.interp_k, trajectory_loader.py:69) -- the GraphHopper spline is not in the repository.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct mpcb_planner_params {
  double dt;                       /* trajectory_planning.py:514  0.3 */
  double w_y, w_s, w_u, w_slack;   /* :14   10, 10, 0.1, 100 */
  double u_min[2], u_max[2];       /* :36-37 */
  double k_min, k_max;             /* :44-45 */
  double a_max;                    /* :48 */
  int simpson_sign;                /* -1: x_pred = x_k - dt/6(...) as committed (:198); +1: the form the committed
                                      trajectories satisfy (SURVEY.md C7) */
  double v_min, v_max;             /* constant speed limits used when no per-node arrays are passed (:465, :476) */
  double s_total;                  /* route length used by the progress cost (:156-158) */
} mpcb_planner_params;

int mpcb_planner_default_params(mpcb_planner_params* p);

/* Hermite-Simpson defects and their derivatives.  DEVICE pointers, async on `cuda_stream`.
 *   z      [C][8N+5]    decision vectors in the reference layout [X (N+1)x5 ; U Nx2 ; S N] (:91-126)
 *   lam    [C][N][5]    multipliers of the defect rows (required iff hess != NULL)
 *   defect [C][N][5]    value of closure dynamics_constraints(z, k) (:183-208)
 *   jac    [C][N][5][12]  d defect / d (x_k, x_{k+1}, u_k)                        (may be NULL)
 *   hess   [C][N][12][12] d^2 (lam . defect) / d (x_k, x_{k+1}, u_k)^2            (may be NULL)
 * Replaces the N `dynamics_constraints` closures and scipy's finite differences of them. */
int mpcb_hs_eval(mpcb_handle h, const mpcb_planner_params* p, int n_chunks, int N, const double* z,
                 const double* lam, double* defect, double* jac, double* hess, void* cuda_stream);

/* Node-wise rows, stage costs and the cost gradient.  DEVICE pointers, async on `cuda_stream`.
 *   s0         [C]            x0[0] of each chunk (normalisation of the progress cost, :156-157)
 *   vmin_nodes, vmax_nodes [C][N+1]  v_min_fun(s_k), v_max_fun(s_k) evaluated by the host (NULL: constants from p)
 *   node_rows  [C][N+1][6]    (v+slack)-v_min, v_max-(v+slack), a_max-k v^2, a_max+k v^2, k-k_min, k_max-k (:249-307)
 *   ctrl_rows  [C][N][5]      u1-u1_min, u1_max-u1, u2-u2_min, u2_max-u2, slack                        (:310-347)
 *   cost_terms [C][N]         stage costs; cost [C] = their sum in the reference's order               (:128-170)
 *   cost_grad  [C][8N+5]      d cost / d z
 * Any output may be NULL (cost needs cost_terms). */
int mpcb_hs_nodes(mpcb_handle h, const mpcb_planner_params* p, int n_chunks, int N, const double* z, const double* s0,
                  const double* vmin_nodes, const double* vmax_nodes, double* node_rows, double* ctrl_rows,
                  double* cost_terms, double* cost, double* cost_grad, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------------------
 * Batched closed loop on the device (the callers either side of the solve path): ObstaclesFSM.update
 * (trajectory_tracking.py:330-374) -> solve -> explicit-Euler plant step (:404-406), repeated while
 * s <= s_max - 1 (:395), for B vehicles at once without leaving the GPU.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct mpcb_scenario {      /* mirrors ObstaclesFSM.__init__, trajectory_tracking.py:285-308 */
  int dynamic_obstacle, traffic_light;
  double obs_trigger_s, obs_start_s, obs_v, obs_end_s;     /* :294-299 */
  double tl_pos, tl_trigger_s, tl_stop_duration;           /* :302-308 */
} mpcb_scenario;

typedef struct mpcb_sim* mpcb_sim_handle;

/* which = 2: constants as committed (:294-308); which = 3: the commented trajectory3 block (:313-327) */
int mpcb_scenario_default(mpcb_scenario* s, int which);
/* B vehicles on the solver context h.  scen: HOST array of n_scen = 1 (shared) or B scenarios.  x_init: HOST [B][5]
 * or NULL for the reference's start [0,0,0,0,0.5] (:382).  history_steps > 0 records that many steps on the device. */
int mpcb_sim_create(mpcb_sim_handle* out, mpcb_handle h, int B, const mpcb_scenario* scen, int n_scen,
                    const double* x_init, int history_steps);
/* Same, vehicle b driving route[b] (HOST [B], each in [0, mpcb_n_routes(h)), else MPCB_ERR_INVALID; NULL: route 0):
 * its reference signal, its end-of-route test s <= s_max - 1 and the s_max of its mpcb_sim_check verdict are its route's. */
int mpcb_sim_create_routes(mpcb_sim_handle* out, mpcb_handle h, int B, const mpcb_scenario* scen, int n_scen,
                           const int* route, const double* x_init, int history_steps);
int mpcb_sim_destroy(mpcb_sim_handle s);
/* n_steps closed-loop steps, asynchronous on cuda_stream (3 + the solver's launches per step, no host round trip; with
 * following on, 2 more plus the kernels of two radix sorts, or 1 more when worlds are set, mpcb_sim_set_worlds).
 * Vehicles that have passed s_max - 1 are frozen. */
int mpcb_sim_step(mpcb_sim_handle s, int n_steps, void* cuda_stream);
/* Hot start (off by default): from its second step on, a vehicle's first pass starts from its previous plan advanced by
 * one step instead of from the reference's table-based warm start (trajectory_tracking.py:223-246), with the rows that
 * sit on their bounds there taken as active.  The problem solved is the same and so is its converged answer; what changes
 * is how often the robust pass is needed (a vehicle waiting at a red light poses the same problem a hundred steps in a row). */
int mpcb_sim_set_hot_start(mpcb_sim_handle s, int on);
/* Following (off by default; on = 1 takes effect from the next step, on = 0 switches it off and ignores follow_range):
 * the vehicles see each other.  At the start of every step, from the states the loop condition is evaluated on:
 *   - a leader is a vehicle still driving on the same route (an arrived vehicle has left the route);
 *   - the vehicles of a route are ordered by (s, index); the leader of b is the next vehicle in that order when
 *     s_leader - s_b <= follow_range, else b has none;
 *   - the FSM runs per vehicle as before, lights included; the car slot of the obstacle set takes the nearer (smaller s)
 *     of the scripted car, when the FSM reports one, and the leader, at (s, v) of the leader at the start of the step;
 *     on a tie the scripted car.  The light stays after the car slot, so n_obs <= MPCB_MAX_OBS.
 * Hot start and routes work unchanged.  With following off, every entry point behaves as without this call.
 * follow_range must be positive and finite (else MPCB_ERR_INVALID before any CUDA call); B <= 2^27.  The first call with
 * on = 1 allocates the sort workspace and the leader histories (synchronises the device's default stream).
 * mpcb_launch_count counts the two kernels following adds per step, not the kernels of its two radix sorts. */
int mpcb_sim_set_follow(mpcb_sim_handle s, int on, double follow_range);
/* Leaders of the first history_steps steps, HOST outputs (any may be NULL): hist_lead_idx [n_recorded][B] (-1: none),
 * hist_lead_sv [n_recorded][B][2] its (s, v) at the start of the step (NaN: none).  -1 / NaN also mark steps where the
 * vehicle had arrived and steps taken with following off. */
int mpcb_sim_follow_history(mpcb_sim_handle s, int* n_recorded, int* hist_lead_idx, double* hist_lead_sv,
                            void* cuda_stream);
/* Gap to the leader over the recorded steps (needs history_steps > 0, else MPCB_ERR_INVALID): min_gap [B] HOST (may be
 * NULL) = min of s_leader - s (1e30 for a vehicle that never had a leader), ok [B] HOST = min_gap >= 1 m (the reference's
 * safety distance of its moving-obstacle check, sanity_checks.py:142-164). */
int mpcb_sim_follow_check(mpcb_sim_handle s, int* ok, double* min_gap, void* cuda_stream);
/* Seeded Gaussian disturbances (off by default), in three independent channels.  For vehicle b at step t (steps since
 * mpcb_sim_create, the counter the histories use), id = first_id + b, z standard normals:
 *   - measurement: the solve sees x_meas = x + sigma_meas * z_m (per component).  The FSM, the loop condition, following
 *     and the plant use the true x; obstacles are not perturbed;
 *   - actuation: the plant applies u = U*[0] + sigma_act * z_a, not clipped; the history keeps the commanded U*[0], so
 *     mpcb_sim_check's steering and acceleration items judge the controller;
 *   - process: x' = Euler step(x, u) + sigma_proc * z_p, added every step.  Vehicles that have arrived stay frozen.
 * A component whose sigma is 0 is left untouched (nothing is added).  With every sigma 0 noise is off and every entry
 * point behaves as without this call, bit for bit, with the same launches; with the measurement sigmas all 0 the solve
 * reads the true state.  Additions and products are rounded separately (no fused multiply-add), so that a replay of the
 * recorded values gives the same bits.
 * Generator: z depends only on (seed, id, t, channel, component), not on B, on how the steps are split between calls, on
 * the execution shape or on which other channels are on.  Philox4x32-10 with key (seed & 0xffffffff, seed >> 32) and
 * counter (t, id, j, 0), j = 0..2 measurement, 3 actuation, 4..6 process; component i of a channel is output i mod 2 of
 * call j_first + i / 2.  A call's words x, y, z, w give W1 = x << 32 | y and W2 = z << 32 | w, u = ((W >> 11) + 0.5) 2^-53
 * each, and Box-Muller: rho = sqrt(-2 ln u1), output 0 = rho cos(2 pi u2), output 1 = rho sin(2 pi u2).  first_id lets a
 * shard of a fleet (vehicles lo .. hi-1, first_id = lo) draw exactly the whole fleet's noise.
 * sigma_meas [5], sigma_act [2], sigma_proc [5]: HOST, NULL = zeros; each finite and >= 0.  first_id >= 0 and
 * first_id + B <= 2^31.  Anything else is MPCB_ERR_INVALID before any CUDA call.  Takes effect from the next step.  The
 * first call that switches noise on allocates the measured states and the noise history (synchronises the device's
 * default stream); MPCB_ERR_NOMEM if that fails, noise then stays off. */
int mpcb_sim_set_noise(mpcb_sim_handle s, unsigned long long seed, int first_id, const double* sigma_meas,
                       const double* sigma_act, const double* sigma_proc);
/* The disturbances added in the first history_steps steps, HOST hist_w [n_recorded][B][12] (may be NULL): measurement
 * 5, actuation 2, process 5, each the value added (sigma z; 0.0 for a component whose sigma is 0).  NaN for steps where
 * the vehicle had arrived or noise was off. */
int mpcb_sim_noise_history(mpcb_sim_handle s, int* n_recorded, double* hist_w, void* cuda_stream);
/* number of vehicles still driving (synchronises the stream) */
int mpcb_sim_alive(mpcb_sim_handle s, int* n_alive, void* cuda_stream);
/* HOST outputs (any may be NULL): current states [B][5], steps driven [B], steps whose solve was not MPCB_SOLVED [B] */
int mpcb_sim_state(mpcb_sim_handle s, double* x, int* steps, int* n_unsolved, void* cuda_stream);
/* recorded history, HOST outputs sized [n_recorded][B]...: state before each step [.][5], applied control [.][2],
 * position of the moving car (NaN when absent), solver status (-1 once frozen), light colour (0 red, 1 green) */
int mpcb_sim_history(mpcb_sim_handle s, int* n_recorded, double* hist_x, double* hist_u, double* hist_obs,
                     int* hist_status, int* hist_tl, void* cuda_stream);

/* trajectory_tracking_check (sanity_checks.py:79-184) for every vehicle on the recorded history (needs history_steps > 0).
 * verdict [B] HOST: bit 0 destination reached, 1 stayed on road (|d| <= 1.5), 2 steering within limits, 3 acceleration
 * within limits (+-0.1), 4 moving obstacle avoided (gap >= 1 m), 5 red light respected, 6 history covers the whole drive
 * (1 = passed).  metrics [B][4] HOST (may be NULL): max |d|, min gap to the car (1e30 if never present), final s, steps. */
int mpcb_sim_check(mpcb_sim_handle s, int* verdict, double* metrics, void* cuda_stream);
/* trajectory_tracking_check from the accumulators the loop keeps, without histories (history_steps may be 0).
 * verdict [B] and metrics [B][4] HOST, same layout as mpcb_sim_check; bit 6 is always set.  On a simulation whose
 * history covers every vehicle's whole drive, bits 0-5 and metrics equal mpcb_sim_check's bit for bit.  The FSM and
 * plant kernels update the accumulators of the vehicles still driving, with the check's own expressions, inside the
 * step's launches; metrics[b][0] (max |d| so far, the current state included) never decreases while b drives. */
int mpcb_sim_running_check(mpcb_sim_handle s, int* verdict, double* metrics, void* cuda_stream);
/* Vehicle b takes over the whole state of vehicle parent[b], for every b at once (a gather: a vehicle may be the parent
 * of several, and a vehicle nobody names is dropped).  parent: HOST [B], each in [0, B); anything else, or following
 * on, is MPCB_ERR_INVALID before any CUDA call.  Ordered on cuda_stream like mpcb_sim_step; parent may be reused when
 * the call returns.  Copied: state, scenario, route, FSM state, previous plan (hot start), steps, unsolved count,
 * running-verdict accumulators, running follower gap, and the recorded rows of every history (states, controls, car,
 * status, light, leaders, disturbances).  After the call vehicle b keeps drawing noise as id first_id + b.  An identity parent
 * changes nothing, bit for bit.  The first call allocates the workspace (synchronises the device's default stream;
 * MPCB_ERR_NOMEM leaves the simulation as it was): B ints, then the larger of the loop state and a window of
 * W = min(history_steps, max(1, floor(2^26 / (188 B)))) history rows (188 bytes: every history a vehicle can record).
 * mpcb_launch_count counts 2 kernels for the loop state and 2 per window of the n_recorded rows: 2 + 2 ceil(n_recorded / W). */
int mpcb_sim_branch(mpcb_sim_handle s, const int* parent, void* cuda_stream);
/* Worlds (off by default): with world_size M, world w is vehicles [w M, (w + 1) M), W = B / M worlds, and a vehicle's
 * leader is searched for only inside its own world: among the vehicles of b's world still driving on b's route, ordered
 * by (s, index) with -0.0 equal to +0.0, the leader of b is the next one if s_leader - s_b <= follow_range.  So W
 * independent platoons, or W copies of one traffic situation, share one simulation.  M = B is mpcb_sim_set_follow's
 * rule for the whole fleet, bit for bit.  1 <= M <= 1024 with B % M == 0, or 0 for one world (every entry point then
 * behaves and launches as without this call); anything else is MPCB_ERR_INVALID before any CUDA call.  Takes effect
 * from the next step and may be changed at any time.  With worlds set and following on, following adds 1 kernel per
 * step (one CTA holds whole worlds and finds their leaders in shared memory) instead of 2 plus two radix sorts. */
int mpcb_sim_set_worlds(mpcb_sim_handle s, int world_size);
/* mpcb_sim_follow_check without histories (history_steps may be 0): same layout, ok [B] HOST, min_gap [B] HOST (may be
 * NULL), from the least gap to the leader that the FSM kernel keeps per vehicle while following is on, with the check's
 * expression.  On a simulation whose history covers every vehicle's whole drive it equals mpcb_sim_follow_check bit for
 * bit; if following was never switched on, min_gap is 1e30 and ok 1.  The gap is copied with its vehicle by
 * mpcb_sim_branch and mpcb_sim_branch_worlds.  Synchronises the stream; launches no kernel. */
int mpcb_sim_running_follow_check(mpcb_sim_handle s, int* ok, double* min_gap, void* cuda_stream);
/* World w takes over the whole state of world parent_world[w]: vehicle w M + i takes over everything mpcb_sim_branch
 * copies from vehicle parent_world[w] M + i, running accumulators and histories included, and recorded leader indices
 * j >= 0 are moved into the copy's world (j + (w - parent_world[w]) M).  parent_world: HOST [W], each in [0, W); worlds
 * must be set (mpcb_sim_set_worlds); anything else is MPCB_ERR_INVALID before any CUDA call.  Following may be on: a
 * copy only sees the vehicles of its own world.  Ordered on cuda_stream like mpcb_sim_step; vehicle b keeps drawing
 * noise as id first_id + b.  Workspace and launch count are mpcb_sim_branch's (the two share it), with its window of
 * rows = min(history_steps, max(1, floor(2^26 / (188 B)))) history rows: 2 + 2 ceil(n_recorded / rows) kernels. */
int mpcb_sim_branch_worlds(mpcb_sim_handle s, const int* parent_world, void* cuda_stream);

/* The same checks on histories the caller supplies (HOST arrays laid out like mpcb_sim_history returns them: hist_x
 * [T][B][5] = state BEFORE each step, hist_u [T][B][2], hist_obs [T][B] (NaN: no car), hist_tl [T][B] (0 red, 1 green);
 * x_final [B][5] = state after the last step, steps [B] = steps driven (<= T), scen [B]).  s_total = s_max of the
 * trajectory.  Replaces trajectory_tracking_check (sanity_checks.py:79-184) for a batch of recorded drives. */
int mpcb_check_histories(mpcb_handle h, int B, int T, double s_total, const mpcb_scenario* scen, const double* x_final,
                         const int* steps, const double* hist_x, const double* hist_u, const double* hist_obs,
                         const int* hist_tl, int* verdict, double* metrics);

const char* mpcb_strerror(int code);
const char* mpcb_last_cuda_error(void);
int mpcb_abi_version(void);
/* sizeof(mpcb_params) / sizeof(mpcb_planner_params) as compiled into the library: lets a binding check its mirror. */
unsigned long long mpcb_sizeof_params(void);
unsigned long long mpcb_sizeof_planner_params(void);

#ifdef __cplusplus
}
#endif
#endif /* MPCB200_H */
