// mpcb_internal.h -- host-side context shared by the translation units of libmpcb200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>

#include "mpcb200.h"
#include "mpcb_device.cuh"

extern thread_local char g_cuda_err[512];
int cuda_fail(cudaError_t e, const char* where);

namespace mpcb { struct PartLists; }

#define CK(call)                                        \
  do {                                                  \
    cudaError_t e_ = (call);                            \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
  } while (0)

// Regions of bytes[0 .. n-1] bytes back to back in one allocation, each 256-byte aligned: region k at off[k], off[n]
// bytes in all.
inline void region_offsets(const size_t* bytes, int n, size_t* off) {
  off[0] = 0;
  for (int k = 0; k < n; ++k) off[k + 1] = off[k] + ((bytes[k] + 255) & ~(size_t)255);
}

struct mpcb_ctx {
  int device;
  int n_sm = 148;
  mpcb_params params;
  mpcb::DevParams dp;
  mpcb::DevTables dt = {};     // one table per route (mpcb_create_routes); dt.t[r]'s arrays are owned by the context
  // workspace for the host-buffer entry points
  void* ws = nullptr;
  size_t ws_bytes = 0;
  char* lists = nullptr;      // work lists of the solve passes and the state the first pass carries (ensure_lists)
  int lists_cap = 0;          // problems they hold
  cudaStream_t stream = nullptr;   // private stream of the *_host entry points
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_mid = nullptr;
  cudaStream_t xs[4] = {nullptr, nullptr, nullptr, nullptr};   // xs[0] == stream; one stream per part of a large host batch
  cudaEvent_t xe[4] = {nullptr, nullptr, nullptr, nullptr};
  void* pin = nullptr;             // pinned staging block of the packed small-batch path
  mpcb::PartLists* lists_last = nullptr;   // header of the last timed solve
  bool timed = false;
  bool pass_timed = false;
  int last_shape = 0;              // first pass of the last solve: 0 thread per problem, 1 warp per problem
  unsigned long long launches = 0;
  // CUDA graphs of the host-buffer entry point: the second call with the same batch size and the same buffers is
  // captured, later ones are one cudaGraphLaunch instead of ~50 enqueue calls.  [0] packed small-batch path, [1] chunked
  struct GraphSlot {
    bool valid = false, have_last = false;
    unsigned long long key[16] = {0}, last[16] = {0};
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    unsigned long long launches = 0;
  } gslot[2];
  cudaEvent_t ev_fork = nullptr;
};

// Solve the problems idx[0 .. *n_idx - 1] (device list) of a batch of B on stream st, problem b on route[b] (nullptr:
// route 0); used by the device closed loop.
extern "C" int mpcb_solve_list_internal(mpcb_handle h, int B, const int* idx, const int* n_idx, const double* x0,
                                        const double* obs_sv, const int* n_obs, const int* route, double* U_out,
                                        int* status_out, cudaStream_t st, const double* U_start);
