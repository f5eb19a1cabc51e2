// mpcb_planner.cu -- kernels and C ABI of the planner function evaluator (see include/mpcb200.h, mpcb_planner.cuh).
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include "mpcb200.h"
#include "mpcb_internal.h"
#include "mpcb_planner.cuh"

namespace mpcb {

constexpr int HS_THREADS = 64;                 // threads per CTA: two lanes per collocation interval (32 / 96 / 128: the same
                                               // 38.9 - 40.4 us on the x64 tile)
constexpr int HS_INTERVALS = HS_THREADS / 2;   // intervals per CTA
constexpr int HS_TRI = 55;                     // packed lower triangle of the 10 x 10 state block of a Hessian block
template <bool WANT_JAC, bool WANT_HESS> struct HsStage {
  // doubles staged per interval: defect, Jacobian block, Hessian triangle (strides odd: conflict-free LDS/STS.64)
  static constexpr int STRIDE = WANT_HESS ? 5 + 60 + HS_TRI + 1 : (WANT_JAC ? 65 : 5);
};

// Two lanes per collocation interval (chunk c, interval k): hs_interval_pair of mpcb_planner.cuh.  Results are staged per
// interval in shared memory -- of the symmetric 12 x 12 Hessian block only the 55 entries of its 10 x 10 lower triangle
// (121 doubles per interval) -- and written out one interval per warp: lane l writes entries l, l + 32, ... of the
// interval's contiguous output, the mirror image and the zero rows / columns of the controls filled in on the way (the
// offsets depend on the lane only and are computed once).
template <bool WANT_JAC, bool WANT_HESS>
__global__ void __launch_bounds__(HS_THREADS)
mpcb_hs_eval_kernel(const __grid_constant__ DevTable T, const __grid_constant__ PlanParams P, int n_int, int N,
                    const double* __restrict__ z, const double* __restrict__ lam, double* __restrict__ defect,
                    double* __restrict__ jac, double* __restrict__ hess) {
  constexpr int STRIDE = HsStage<WANT_JAC, WANT_HESS>::STRIDE;
  extern __shared__ double stage[];
  const int t = threadIdx.x;
  const int first = blockIdx.x * HS_INTERVALS;
  const int q0 = t >> 1, p = t & 1;
  const int i = first + q0;
  const int nb = min(HS_INTERVALS, n_int - first);
  const unsigned pair_mask = __ballot_sync(0xffffffffu, i < n_int);
  if (i < n_int) {
    const int c = i / N, k = i - c * N;
    const double* zc = z + (size_t)c * (8 * N + 5);
    double xk[5], xn[5], u[2];
#pragma unroll
    for (int q = 0; q < 5; ++q) { xk[q] = zc[5 * k + q]; xn[q] = zc[5 * (k + 1) + q]; }
    u[0] = zc[5 * (N + 1) + 2 * k];
    u[1] = zc[5 * (N + 1) + 2 * k + 1];
    hs_interval_pair<WANT_JAC, WANT_HESS>(T, P, xk, xn, u, WANT_HESS ? lam + (size_t)i * 5 : nullptr, p, pair_mask,
                                          stage + (size_t)q0 * STRIDE);
  }
  __syncthreads();
  const int lane = t & 31, w = t >> 5;
  constexpr int NW = HS_THREADS / 32;
  // defects: the CTA's nb * 5 doubles are contiguous
  for (int e = t; e < nb * 5; e += HS_THREADS) defect[(size_t)first * 5 + e] = stage[(e / 5) * STRIDE + e % 5];
  if (WANT_JAC && jac) {
    for (int q = w; q < nb; q += NW) {
      const double* src = stage + (size_t)q * STRIDE + 5;
      double* dst = jac + ((size_t)first + q) * 60;
      const double a = src[lane];
      const double b = (lane < 28) ? src[32 + lane] : 0.0;
      dst[lane] = a;
      if (lane < 28) dst[32 + lane] = b;
    }
  }
  if (WANT_HESS && hess) {
    // entry e = lane + 32 m of the 12 x 12 block: (r, c) = (e / 12, e % 12); source = packed triangle, or zero
    int off[5];
#pragma unroll
    for (int m = 0; m < 5; ++m) {
      const int e = lane + 32 * m, r = e / 12, c = e - 12 * r;
      const int hi = r > c ? r : c, lo = r > c ? c : r;
      off[m] = (e < 144 && hi < 10) ? hi * (hi + 1) / 2 + lo : -1;
    }
#pragma unroll 2
    for (int q = w; q < nb; q += NW) {
      const double* src = stage + (size_t)q * STRIDE + 65;
      double* dst = hess + ((size_t)first + q) * 144;
      double v[5];
#pragma unroll
      for (int m = 0; m < 5; ++m) v[m] = off[m] >= 0 ? src[off[m]] : 0.0;
#pragma unroll
      for (int m = 0; m < 5; ++m)
        if (lane + 32 * m < 144) dst[lane + 32 * m] = v[m];
    }
  }
}

// One thread per node (chunk c, node k = 0..N): inequality rows, stage cost and its gradient in z layout.
__global__ void __launch_bounds__(128)
mpcb_hs_nodes_kernel(const __grid_constant__ PlanParams P, int n_nodes, int N, const double* __restrict__ z,
                     const double* __restrict__ s0, const double* __restrict__ vmin_nodes,
                     const double* __restrict__ vmax_nodes, double* __restrict__ node_rows,
                     double* __restrict__ ctrl_rows, double* __restrict__ cost_terms, double* __restrict__ cost_grad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_nodes) return;
  const int c = i / (N + 1), k = i - c * (N + 1);
  const int nz = 8 * N + 5;
  const double* zc = z + (size_t)c * nz;
  double x[5];
#pragma unroll
  for (int q = 0; q < 5; ++q) x[q] = zc[5 * k + q];
  const bool inner = k < N;
  const double slack = inner ? zc[7 * N + 5 + k] : 0.0;                      // no slack on the final state (:256-259)
  const double vmin = vmin_nodes ? vmin_nodes[i] : P.v_min_c;
  const double vmax = vmax_nodes ? vmax_nodes[i] : P.v_max_c;
  if (node_rows) {
    double r[6];
    hs_node_rows(P, x, slack, vmin, vmax, r);
#pragma unroll
    for (int q = 0; q < 6; ++q) node_rows[(size_t)i * 6 + q] = r[q];
  }
  double g[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (inner) {
    const double u[2] = {zc[5 * (N + 1) + 2 * k], zc[5 * (N + 1) + 2 * k + 1]};
    if (ctrl_rows) {
      double r[5];
      hs_ctrl_rows(P, u, slack, r);
#pragma unroll
      for (int q = 0; q < 5; ++q) ctrl_rows[((size_t)c * N + k) * 5 + q] = r[q];
    }
    const double ct = hs_stage_cost(P, x, u, slack, s0[c], g);
    if (cost_terms) cost_terms[(size_t)c * N + k] = ct;
  }
  if (cost_grad) {
    double* gc = cost_grad + (size_t)c * nz;
    gc[5 * k + 0] = g[0]; gc[5 * k + 1] = g[1]; gc[5 * k + 2] = g[2]; gc[5 * k + 3] = 0.0; gc[5 * k + 4] = 0.0;
    if (inner) {
      gc[5 * (N + 1) + 2 * k] = g[3];
      gc[5 * (N + 1) + 2 * k + 1] = g[4];
      gc[7 * N + 5 + k] = g[5];
    }
  }
}

// cost = sum_k terms in the reference's order (sequential accumulation, :141-169), one thread per chunk
__global__ void mpcb_hs_cost_sum_kernel(int C, int N, const double* __restrict__ terms, double* __restrict__ cost) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double acc = 0.0;
  for (int k = 0; k < N; ++k) acc += terms[(size_t)c * N + k];
  cost[c] = acc;
}

}  // namespace mpcb

using namespace mpcb;

static int derive_plan(const mpcb_planner_params* p, PlanParams& d) {
  if (!p || !(p->dt > 0) || (p->simpson_sign != 1 && p->simpson_sign != -1)) return MPCB_ERR_INVALID;
  d.dt = p->dt;
  d.w_y = p->w_y; d.w_s = p->w_s; d.w_u = p->w_u; d.w_slack = p->w_slack;
  for (int i = 0; i < 2; ++i) { d.u_min[i] = p->u_min[i]; d.u_max[i] = p->u_max[i]; }
  d.k_min = p->k_min; d.k_max = p->k_max; d.a_max = p->a_max;
  d.sigma = (double)p->simpson_sign;
  d.v_min_c = p->v_min; d.v_max_c = p->v_max;
  d.s_total = p->s_total;
  return MPCB_OK;
}

extern "C" {

int mpcb_planner_default_params(mpcb_planner_params* p) {
  if (!p) return MPCB_ERR_INVALID;
  memset(p, 0, sizeof(*p));
  p->dt = 0.3;                                               // trajectory_planning.py:514
  p->w_y = 10.0; p->w_s = 10.0; p->w_u = 0.1; p->w_slack = 100.0;   // :14
  p->u_min[0] = -0.6; p->u_min[1] = -5.0; p->u_max[0] = 0.6; p->u_max[1] = 4.0;   // :36-37
  p->k_min = -0.8; p->k_max = 0.8;                           // :44-45
  p->a_max = 6.0;                                            // :48
  p->simpson_sign = -1;                                      // as committed (:198)
  p->v_min = 0.0; p->v_max = 1.0;                            // :476-477 / :465 (v_max_array default)
  p->s_total = 0.0;
  return MPCB_OK;
}

int mpcb_hs_eval(mpcb_handle h, const mpcb_planner_params* p, int n_chunks, int N, const double* z, const double* lam,
                 double* defect, double* jac, double* hess, void* cuda_stream) {
  if (!h || n_chunks < 0 || N < 1 || (n_chunks > 0 && (!z || !defect)) || (hess && !lam)) return MPCB_ERR_INVALID;
  PlanParams d;
  int rc = derive_plan(p, d);
  if (rc != MPCB_OK) return rc;
  if (n_chunks == 0) return MPCB_OK;
  const long long n_int_ll = (long long)n_chunks * N;
  if (n_int_ll > 0x7fffffffLL / 144) return MPCB_ERR_INVALID;
  const int n_int = (int)n_int_ll;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int grid = (n_int + HS_INTERVALS - 1) / HS_INTERVALS;
  auto launch = [&](auto kern, size_t smem) -> int {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   // per device
    kern<<<grid, HS_THREADS, smem, st>>>(h->dt.t[0], d, n_int, N, z, lam, defect, jac, hess);
    return MPCB_OK;
  };
  const size_t per = sizeof(double) * HS_INTERVALS;
  if (hess) rc = launch(mpcb_hs_eval_kernel<true, true>, per * HsStage<true, true>::STRIDE);   // hess implies the Jacobian intermediates
  else if (jac) rc = launch(mpcb_hs_eval_kernel<true, false>, per * HsStage<true, false>::STRIDE);
  else rc = launch(mpcb_hs_eval_kernel<false, false>, per * HsStage<false, false>::STRIDE);
  if (rc != MPCB_OK) return rc;
  CK(cudaGetLastError());
  h->launches++;
  return MPCB_OK;
}

int mpcb_hs_nodes(mpcb_handle h, const mpcb_planner_params* p, int n_chunks, int N, const double* z, const double* s0,
                  const double* vmin_nodes, const double* vmax_nodes, double* node_rows, double* ctrl_rows,
                  double* cost_terms, double* cost, double* cost_grad, void* cuda_stream) {
  if (!h || n_chunks < 0 || N < 1 || (n_chunks > 0 && (!z || !s0)) || (cost && !cost_terms)) return MPCB_ERR_INVALID;
  PlanParams d;
  int rc = derive_plan(p, d);
  if (rc != MPCB_OK) return rc;
  if (n_chunks == 0) return MPCB_OK;
  const long long nn = (long long)n_chunks * (N + 1);
  if (nn > 0x7fffffffLL / 8) return MPCB_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  mpcb_hs_nodes_kernel<<<(int)((nn + 127) / 128), 128, 0, st>>>(d, (int)nn, N, z, s0, vmin_nodes, vmax_nodes, node_rows,
                                                                ctrl_rows, cost_terms, cost_grad);
  CK(cudaGetLastError());
  h->launches++;
  if (cost) {
    mpcb_hs_cost_sum_kernel<<<(n_chunks + 127) / 128, 128, 0, st>>>(n_chunks, N, cost_terms, cost);
    CK(cudaGetLastError());
    h->launches++;
  }
  return MPCB_OK;
}

}  // extern "C"
