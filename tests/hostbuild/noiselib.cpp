// noiselib.cpp -- TEST INFRASTRUCTURE ONLY.  Compiles the closed loop's noise generator (mpcb_philox.cuh) with g++ so
// that the words and normals the device draws can be checked against a numpy restatement without a GPU
// (tests/test_gpu_sim_noise.py builds it).  Nothing in the product package loads this library.
#include <math.h>

#define __forceinline__ inline
#define __restrict__

#include "mpcb_philox.cuh"

using namespace mpcb;

extern "C" {

// n draws of the generator: call (seed[i], id[i], t[i], j[i]) -> its four Philox words words[4 i ..] and its two
// normals z[2 i ..]
int host_sim_normals(int n, const unsigned long long* seed, const unsigned* id, const unsigned* t, const unsigned* j,
                     unsigned* words, double* z) {
  for (int i = 0; i < n; ++i) {
    Philox4 w;
    sim_normal_pair(seed[i], id[i], t[i], j[i], z + 2 * i, &w);
    words[4 * i] = w.x; words[4 * i + 1] = w.y; words[4 * i + 2] = w.z; words[4 * i + 3] = w.w;
  }
  return 0;
}

}  // extern "C"
