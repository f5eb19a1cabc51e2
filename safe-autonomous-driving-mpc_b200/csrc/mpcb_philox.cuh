// mpcb_philox.cuh -- the counter-based generator of the closed loop's disturbances (mpcb_sim_set_noise), host and device.
//
// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011) with curand's round and key
// schedule, and a Box-Muller transform of its two 64-bit words.  A draw depends only on (seed, id, t, j): the same code
// compiles with g++ for the tests (tests/hostbuild), which hold it to a numpy restatement.
#pragma once
#include "mpcb_device.cuh"

namespace mpcb {

struct Philox4 { unsigned x, y, z, w; };

MPCB_HD unsigned philox_mulhilo(unsigned a, unsigned b, unsigned* hi) {
  const unsigned long long p = (unsigned long long)a * b;
  *hi = (unsigned)(p >> 32);
  return (unsigned)p;
}

// Philox4x32-10 of counter c under key (k0, k1)
MPCB_HD Philox4 philox4x32_10(Philox4 c, unsigned k0, unsigned k1) {
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    unsigned hi0, hi1;
    const unsigned lo0 = philox_mulhilo(0xD2511F53u, c.x, &hi0);
    const unsigned lo1 = philox_mulhilo(0xCD9E8D57u, c.z, &hi1);
    c = Philox4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
  }
  return c;
}

// (0, 1) from the top 53 bits of a 64-bit word: ((W >> 11) + 0.5) 2^-53, never 0 or 1
MPCB_HD double philox_unit(unsigned hi, unsigned lo) {
  const unsigned long long w = ((unsigned long long)hi << 32) | lo;
  return ((double)(w >> 11) + 0.5) * 0x1p-53;
}

// Two standard normals of call j at step t for vehicle id under seed: counter (t, id, j, 0), key (seed low, seed high);
// Box-Muller on u1 = unit(x, y), u2 = unit(z, w): z[0] = rho cos(2 pi u2), z[1] = rho sin(2 pi u2), rho = sqrt(-2 ln u1).
MPCB_HD void sim_normal_pair(unsigned long long seed, unsigned id, unsigned t, unsigned j, double z[2],
                             Philox4* words = nullptr) {
  const Philox4 r = philox4x32_10(Philox4{t, id, j, 0u}, (unsigned)seed, (unsigned)(seed >> 32));
  if (words) *words = r;
  const double u1 = philox_unit(r.x, r.y), u2 = philox_unit(r.z, r.w);
  const double rho = sqrt(-2.0 * log(u1));
  double s, c;
#if defined(__CUDA_ARCH__)
  sincospi(2.0 * u2, &s, &c);
#else
  s = sin(2.0 * M_PI * u2);
  c = cos(2.0 * M_PI * u2);
#endif
  z[0] = rho * c;
  z[1] = rho * s;
}

}  // namespace mpcb
