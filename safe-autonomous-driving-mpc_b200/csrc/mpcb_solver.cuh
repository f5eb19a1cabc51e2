// mpcb_solver.cuh -- per-thread Gauss-Newton SQP with an OSQP-style ADMM QP solver (one thread = one problem).
//
// QP of one linearisation round, in the absolute variable x = U+ (SURVEY.md A.1 for the formulation):
//     min 1/2 x'Hx + q'x   s.t.  lo <= A x <= hi ,   H = diag(2 w_u) + 2 J'WJ  (Gauss-Newton),  q = g - H U
// Rows of A (M = 41), never stored densely:
//     0..9    box      x_i in [u_min, u_max]                                         (trajectory_tracking.py:249)
//     10..17  lane     (D_j + alpha O_j) x, j = 2..5, alpha in {0, wheelbase}        (:171-189)
//                      -- step 1 does not depend on U; the alpha = wheelbase/2 row is implied by the two outer ones
//                         (|d + alpha o| is convex in alpha), so it is not a row of the QP
//     18..22  speed    v_j - v0 = h sum_{i<j} b_i >= -v0                             (:207)
//     23+9k.. obstacle k:  R1_j (j = 2..5): S_j <= base_j - safe ;  R2_j (j = 1..5): S_j + tgap (v_j - v0) <= base_j - tgap v0
//                      with S_j = s_j - s0 - j h v0: the max(.,.) of :201 split into two affine rows (SURVEY A.1)
// ADMM with sigma = 0 and relaxation alpha in single-vector form (v = z_relaxed + y/rho; z = clip(v), y = rho (v - z)):
//     x  = K^-1 (A' rho (2 clip(v) - v) - q),  K = H + A' diag(rho) A = L L' ;   v += alpha (A x - clip(v))
// rho_r = lad[e_r] / max(|a_r|^2, floor).  A segment = factorisation + a few iterations, the last of which also
// evaluates residuals, the active set, the step-size policy and (robust pass) OSQP's infeasibility certificate.
// Two policies run on this machinery (mpcb_params.h): the first pass uses two rungs {~0, large} -- inactive rows
// exert no force, active rows are near-equalities: a primal-dual active-set iteration with augmented-Lagrangian
// inner solves -- and hands whatever it cannot close to the robust pass, which walks a x10 ladder with hysteresis.
//
// In the thread-per-problem kernel the first pass runs ONE segment per Gauss-Newton round and tolerates a few rounds
// whose QP did not close (the ADMM state carries over: the active-set search continues on the next linearisation).
//
// Data placement: a compile-time mask (MPCB_STORE_MASK) says which per-thread arrays live in a strided store (shared
// memory on the GPU: element i of thread t at base[i * CTA + t], conflict free) -- by default the per-row vectors v,
// rho and the obstacle bounds -- and which stay thread-private (registers / local memory): D, O, the 10x10 factor, H,
// q and the iterate.  The one-segment first pass also puts the factor and D, O in tensor memory (TCol below).
#pragma once
#include <stdint.h>
#include <type_traits>

#include "mpcb200.h"
#include "mpcb_device.cuh"

// Loop control is uniform over the whole CTA (all threads reach every barrier): the CTA walks through the
// straight-line solver code together, so one instruction stream per CTA goes through the instruction caches.
#if defined(__CUDA_ARCH__) && defined(MPCB_WARP_UNIFORM)
#define MPCB_ALL(pred) (__all_sync(0xffffffffu, pred) != 0)
#elif defined(__CUDA_ARCH__)
#define MPCB_ALL(pred) (__syncthreads_and(pred) != 0)
#else
#define MPCB_ALL(pred) (pred)
#endif

namespace mpcb {

constexpr int N_LANE = 8;
constexpr int ROW_LANE = 10, ROW_V = 18, ROW_OBS = 23, N_OBSROW = 9, M_ROWS = 41;
constexpr int N_DO = 20;   // flat storage of d(d_j)/dU (resp. o_j), j = 2..5: supports 2, 4, 6, 8
constexpr double NRM2_FLOOR = 1e-2;

__host__ __device__ constexpr int doff(int jj) { return jj * (jj + 1); }               // 0, 2, 6, 12
__host__ __device__ constexpr int row_r1(int k, int j) { return ROW_OBS + N_OBSROW * k + (j - 2); }   // j = 2..5
__host__ __device__ constexpr int row_r2(int k, int j) { return ROW_OBS + N_OBSROW * k + 4 + (j - 1); }  // j = 1..5

// On the GPU the store is accessed through volatile pointers: every access is a real shared-memory load / store.
// (Without it the compiler promotes the whole store to registers across the iteration loop and then spills those
// registers to local memory -- i.e. through L1 to L2/DRAM -- which is exactly what the store is there to avoid.)
#if defined(__CUDA_ARCH__) && !defined(MPCB_STORE_PLAIN)
typedef volatile double store_t;
#else
typedef double store_t;
#endif
template <int S>
struct Col {           // strided, volatile on the GPU: shared memory
  store_t* p;
  MPCB_HD store_t& operator[](int i) const { return p[i * S]; }
};
struct LCol {          // thread-private, plain: registers / local memory, placement left to the compiler
  double* p;
  MPCB_HD double& operator[](int i) const { return p[i]; }
};
// Tensor memory (first-pass class and round kernels): a column kind with no references, because tcgen05.ld is
// asynchronous.  Shape 32x32b maps TMEM lane t of the warp's sub-partition to lane t of the warp, so the columns are
// thread-private; double i of a TCol sits in its columns 2i (low word) and 2i + 1 (high word).  Every access is a block
// load (tcgen05.ld, then tcgen05.wait::ld before the values are used) or a block store, and is .sync.aligned: the whole
// warp must execute it together (see solve_round's one-segment path).  a: TMEM address of this warp's lanes and of the
// array's first column.
struct TCol { uint32_t a; };
template <class C> struct IsTmem : std::false_type {};
template <> struct IsTmem<TCol> : std::true_type {};

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ void tmem_converged() {
  __syncwarp();
  MPCB_ASSERT(__activemask() == 0xffffffffu);
}
#define MPCB_TLD_ASM(N, REGS, ...)                                                                                     \
  asm volatile("{\n\ttcgen05.ld.sync.aligned.32x32b.x" #N ".b32 " REGS ", [%" #N "];\n\ttcgen05.wait::ld.sync.aligned;\n}" \
               : __VA_ARGS__ : "r"(a) : "memory")
template <int N> __device__ __forceinline__ void tmem_ld(uint32_t a, uint32_t (&r)[N]);
template <> __device__ __forceinline__ void tmem_ld<2>(uint32_t a, uint32_t (&r)[2]) {
  MPCB_TLD_ASM(2, "{%0, %1}", "=r"(r[0]), "=r"(r[1]));
}
template <> __device__ __forceinline__ void tmem_ld<4>(uint32_t a, uint32_t (&r)[4]) {
  MPCB_TLD_ASM(4, "{%0, %1, %2, %3}", "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]));
}
template <> __device__ __forceinline__ void tmem_ld<8>(uint32_t a, uint32_t (&r)[8]) {
  MPCB_TLD_ASM(8, "{%0, %1, %2, %3, %4, %5, %6, %7}", "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]),
               "=r"(r[5]), "=r"(r[6]), "=r"(r[7]));
}
template <> __device__ __forceinline__ void tmem_ld<16>(uint32_t a, uint32_t (&r)[16]) {
  MPCB_TLD_ASM(16, "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}", "=r"(r[0]), "=r"(r[1]),
               "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
               "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]));
}
#undef MPCB_TLD_ASM
__device__ __forceinline__ void tmem_st2(uint32_t a, double x) {   // one double; completed by tmem_wait_st
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};"
               :: "r"(a), "r"(__double2loint(x)), "r"(__double2hiint(x)) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// chunk of 2 * W columns at double i + k of c into x[k .. k + W)
template <int W, int NMAX>
__device__ __forceinline__ void tload_chunk(const TCol& c, int i, int k, double (&x)[NMAX]) {
  uint32_t r[2 * W];
  tmem_ld<2 * W>(c.a + 2 * (i + k), r);
#pragma unroll
  for (int m = 0; m < W; ++m)
    if (k + m < NMAX) x[k + m] = __hiloint2double((int)r[2 * m + 1], (int)r[2 * m]);
}
// x[0 .. n) = doubles i .. i + n of c (n <= NMAX <= 15, a compile-time constant once the caller's loops are unrolled)
template <int NMAX>
__device__ __forceinline__ void tload(const TCol& c, int i, int n, double (&x)[NMAX]) {
  static_assert(NMAX <= 15, "chunks of 8, 4, 2, 1 doubles");
  tmem_converged();
  int k = 0;
  if (n - k >= 8) { tload_chunk<8>(c, i, k, x); k += 8; }
  if (n - k >= 4) { tload_chunk<4>(c, i, k, x); k += 4; }
  if (n - k >= 2) { tload_chunk<2>(c, i, k, x); k += 2; }
  if (n - k >= 1) tload_chunk<1>(c, i, k, x);
}
// doubles i .. i + n of c = x[0 .. n); the caller ends its stores with tmem_wait_st before anything reads them
template <int NMAX>
__device__ __forceinline__ void tstore(const TCol& c, int i, int n, const double (&x)[NMAX]) {
  tmem_converged();
#pragma unroll
  for (int m = 0; m < NMAX; ++m)
    if (m < n) tmem_st2(c.a + 2 * (i + m), x[m]);
}
#else
// the host never places an array in tensor memory (ColSel below); these only keep the discarded branches well formed
template <int NMAX> inline void tload(const TCol&, int, int, double (&)[NMAX]) {}
template <int NMAX> inline void tstore(const TCol&, int, int, const double (&)[NMAX]) {}
inline void tmem_wait_st() {}
#endif

// placement of an array group: 0 thread-private, 1 shared, 2 tensor memory, 3 not stored
template <int KIND, int S> struct ColSel { typedef Col<S> type; };
template <int S> struct ColSel<0, S> { typedef LCol type; };
template <int S> struct ColSel<3, S> { typedef LCol type; };
#if defined(__CUDA_ARCH__)
template <int S> struct ColSel<2, S> { typedef TCol type; };
#else
template <int S> struct ColSel<2, S> { typedef LCol type; };
#endif

// Per-thread working set.  MASK says which array groups sit in the strided (shared-memory) part, TMASK which sit in
// tensor memory (device only), NONE which are not stored at all; the rest lives in a thread-private buffer of LOCAL
// doubles (registers / local memory, placement left to the compiler):
//   bit 0  v        [41] ADMM state                      bit 4  L, rdiag   [55+10] factor of K
//   bit 1  rho      [41] step sizes                      bit 5  q, lane_c  [10+8]
//   bit 2  hio      [18] obstacle-row bounds             bit 6  H          [55]
//   bit 3  D, O     [20+20] lane sensitivities           bit 7  lane_inrm, lov, blo, bhi  [8+5+5+5]
// In tensor memory, L holds the factor column by column: column j at fcol(j) is rdiag[j], then L[j+1..9][j] (55 doubles
// in all; rdiag is not a separate array there).  Only bits 3 and 4 can go to tensor memory, only bit 6 (H, which the
// one-segment first pass hands from linearise to factor in registers) can be left out.
// MASK = 0: host build, evaluation kernel, cooperative kernel (S must be 1).
// NOBS: how many obstacle slots the problems of this instantiation can have (0, 1 or 2).  The thread-per-problem first
// pass runs one instantiation per obstacle count (the batch is partitioned by n_obs first, mpcb_api.cu): a problem
// without obstacles walks 23 rows instead of 41 and keeps 46 instead of 100 doubles of row state, so more of its
// working set fits in shared memory.  Rows keep their numbers; the slots k >= NOBS simply do not exist.
__host__ __device__ constexpr int fcol(int j) { return j * NV - j * (j - 1) / 2; }
template <int S, unsigned MASK, int NOBS = 2, unsigned TMASK = 0u, unsigned NONE = 0u>
struct Store {
  static_assert((MASK & TMASK) == 0u && ((MASK | TMASK) & NONE) == 0u, "one placement per array group");
  static_assert((TMASK & ~(8u | 16u)) == 0u && (NONE & ~64u) == 0u, "only D, O, L, rdiag go to tensor memory, only H can be left out");
  static constexpr int KOBS = NOBS;
  static constexpr int MROWS = ROW_OBS + N_OBSROW * NOBS;
  MPCB_HD static constexpr int kind(int bit) {
    return ((NONE >> bit) & 1u) ? 3 : ((TMASK >> bit) & 1u) ? 2 : ((MASK >> bit) & 1u) ? 1 : 0;
  }
  template <int BIT> using G = typename ColSel<kind(BIT), S>::type;
  static constexpr int size_of(int bit) {
    return bit == 0 ? MROWS : bit == 1 ? MROWS : bit == 2 ? NOBS * N_OBSROW : bit == 3 ? 2 * N_DO : bit == 4 ? NTRI + NV
         : bit == 5 ? NV + N_LANE : bit == 6 ? NTRI : N_LANE + 3 * NH;
  }
  static constexpr int doubles_of(int k) {
    int n = 0;
    for (int b = 0; b < 8; ++b) if (kind(b) == k) n += (k == 2 && b == 4) ? NTRI : size_of(b);
    return n;
  }
  static constexpr int TOTAL = 2 * MROWS + NOBS * N_OBSROW + 2 * N_DO + NTRI + NV + NV + N_LANE + NTRI + N_LANE + 3 * NH;
  static constexpr int SHARED = doubles_of(1);
  static constexpr int TMEM_COLS = 2 * doubles_of(2);   // 32-bit columns
  static constexpr int LOCAL = doubles_of(0) > 0 ? doubles_of(0) : 1;
  G<0> v;
  G<1> rho;
  G<2> hio;         // upper bounds of the obstacle rows (BIG: row absent or dropped)
  G<3> D, O;
  G<4> L, rdiag;
  G<5> q, lane_c;   // lane_c: row value offset (d_j + alpha o_j)(U) - a.U
  G<6> H;
  G<7> lane_inrm, lov, blo, bhi;   // lov: lower bound of the speed rows; blo/bhi: per-problem box of the accelerations
  // sh: this thread's first element of the strided part; lo: thread-private buffer of LOCAL doubles; tm: TMEM address of
  // this warp's lanes and of the first column the store may use (TMEM_COLS of them)
  MPCB_HD Store(double* sh, double* lo, uint32_t tm = 0u) {
    auto take = [&](auto& c, int k, int n) {
      if constexpr (IsTmem<std::decay_t<decltype(c)>>::value) {
        c.a = tm; tm += 2 * n;
      } else {
        typedef decltype(c.p) P;
        if (k == 1) { c.p = (P)sh; sh += n * S; }
        else if (k == 3) c.p = nullptr;
        else { c.p = (P)lo; lo += n; }
      }
    };
    (void)tm;
    take(v, kind(0), MROWS); take(rho, kind(1), MROWS); take(hio, kind(2), NOBS * N_OBSROW);
    take(D, kind(3), N_DO); take(O, kind(3), N_DO);
    take(L, kind(4), NTRI); take(rdiag, kind(4), kind(4) == 2 ? 0 : NV);
    take(q, kind(5), NV); take(lane_c, kind(5), N_LANE);
    take(H, kind(6), NTRI);
    take(lane_inrm, kind(7), N_LANE); take(lov, kind(7), NH); take(blo, kind(7), NH); take(bhi, kind(7), NH);
  }
};

struct Rungs {  // 4-bit ladder index per row
  unsigned int w[6];
  MPCB_HD int get(int r) const { return (w[r >> 3] >> ((r & 7) * 4)) & 15; }
  MPCB_HD void set(int r, int e) { w[r >> 3] = (w[r >> 3] & ~(15u << ((r & 7) * 4))) | ((unsigned)e << ((r & 7) * 4)); }
};

struct Problem {
  // inputs
  double x0[5];
  double obs[2][2];
  int n_obs;
  // SQP state
  double U[NV];
  double x[NV];
  // policy state
  Rungs E;
  unsigned long long act_prev;
  int hint[NH + 1];           // table segment of s_j found by the previous lookup
};

MPCB_HD double clipd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }
MPCB_HD double dmax(double a, double b) { return a > b ? a : b; }
// rows by sidedness: 0 two-sided (box, lane), 1 lower bound only (speed), 2 upper bound only (obstacle); the absent side
// is +-BIG, which no row value reaches, so its comparison is dropped at compile time
template <int KIND> using RowKind = std::integral_constant<int, KIND>;
template <int KIND> MPCB_HD double clipk(double v, double lo, double hi) {
  if (KIND == 1) return v < lo ? lo : v;
  if (KIND == 2) return v > hi ? hi : v;
  return clipd(v, lo, hi);
}
template <int KIND> MPCB_HD bool outside(double v, double lo, double hi) {
  if (KIND == 1) return v < lo;
  if (KIND == 2) return v > hi;
  return (v < lo) || (v > hi);
}

// ------------------------------------------------------------------------------------------------
// Linearisation: rollout with forward sensitivities at pb.U; fills H, q, D, O, lane_c, lane_inrm.
// const_viol = worst violation among the lane rows of step 1 (they do not depend on U).
// ------------------------------------------------------------------------------------------------
template <int L>
MPCB_HD void rank1(double (&H)[NTRI], const double (&a)[NV], double w) {
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const double wa = w * a[i];
#pragma unroll
    for (int j = 0; j <= i; ++j) H[tri(i, j)] = fma(wa, a[j], H[tri(i, j)]);
  }
}

template <int J>  // residual rows of step J (1..5): accumulate H and g
MPCB_HD void accumulate_step(const DevParams& P, double (&H)[NTRI], double (&g)[NV], const double (&dD)[NV],
                             const double (&dO)[NV], const double (&Xj)[5], const double (&val)[4],
                             const double (&slope)[4]) {
  constexpr int L = 2 * (J - 1);  // support of dD, dO, ds_J
  const double h = P.h;
  double Jd[NV], Jo[NV], Jv[NV];
#pragma unroll
  for (int c = 0; c < NV; ++c) { Jd[c] = 0.0; Jo[c] = 0.0; Jv[c] = 0.0; }
#pragma unroll
  for (int i = 0; i < J; ++i) {
    const double ds = (i < J - 1) ? h * h * (double)(J - 1 - i) : 0.0;  // d s_J / d b_i
    Jv[2 * i + 1] = h - slope[3] * ds;
    if (i < J - 1) {
      Jd[2 * i] = dD[2 * i];
      Jo[2 * i] = dO[2 * i];
      Jd[2 * i + 1] = dD[2 * i + 1] - slope[0] * ds;
      Jo[2 * i + 1] = dO[2 * i + 1] - slope[1] * ds;
    }
  }
  const double rd = Xj[1] - val[0], ro = Xj[2] - val[1], rv = Xj[4] - val[3];
  if (L > 0) {
    rank1<L>(H, Jd, 2.0 * P.wd);
    rank1<L>(H, Jo, 2.0 * P.wo);
#pragma unroll
    for (int c = 0; c < L; ++c) g[c] += 2.0 * (P.wd * rd * Jd[c] + P.wo * ro * Jo[c]);
  }
  // Jv lives on the b entries only
#pragma unroll
  for (int i = 0; i < J; ++i) {
    const double wa = 2.0 * P.wv * Jv[2 * i + 1];
#pragma unroll
    for (int k = 0; k <= i; ++k) H[tri(2 * i + 1, 2 * k + 1)] = fma(wa, Jv[2 * k + 1], H[tri(2 * i + 1, 2 * k + 1)]);
    g[2 * i + 1] += 2.0 * P.wv * rv * Jv[2 * i + 1];
  }
}

template <int J, class ST>  // lane rows of step J (2..5)
MPCB_HD void lane_rows(const DevParams& P, Problem& pb, const ST& st, const double (&dD)[NV],
                       const double (&dO)[NV], const double (&Xj)[5]) {
  constexpr int L = 2 * (J - 1);
  constexpr int o = doff(J - 2);
  double dU = 0.0, oU = 0.0, dd = 0.0, dox = 0.0, oo = 0.0;
  if constexpr (IsTmem<decltype(st.D)>::value) { tstore(st.D, o, L, dD); tstore(st.O, o, L, dO); }
#pragma unroll
  for (int c = 0; c < L; ++c) {
    if constexpr (!IsTmem<decltype(st.D)>::value) {
      st.D[o + c] = dD[c];
      st.O[o + c] = dO[c];
    }
    dU = fma(dD[c], pb.U[c], dU);
    oU = fma(dO[c], pb.U[c], oU);
    dd = fma(dD[c], dD[c], dd);
    dox = fma(dD[c], dO[c], dox);
    oo = fma(dO[c], dO[c], oo);
  }
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    const double al = a ? P.alpha_lane[2] : 0.0;
    st.lane_c[2 * (J - 2) + a] = (Xj[1] + al * Xj[2]) - (dU + al * oU);
    const double n2 = dd + 2.0 * al * dox + al * al * oo;
    st.lane_inrm[2 * (J - 2) + a] = 1.0 / dmax(n2, NRM2_FLOOR);
  }
}

// H: the Gauss-Newton Hessian, left in the caller's registers (the one-segment first pass factors it straight away)
template <class ST>
MPCB_HD void linearise(const DevTable& T, const DevParams& P, Problem& pb, const ST& st, double& const_viol,
                       double (&H)[NTRI]) {
  const double h = P.h;
#pragma unroll
  for (int i = 0; i < NTRI; ++i) H[i] = 0.0;
#pragma unroll
  for (int i = 0; i < NV; ++i) H[tri(i, i)] = 2.0 * P.wu[i & 1];
  double g[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) g[i] = 2.0 * P.wu[i & 1] * pb.U[i];

  double X[5] = {pb.x0[0], pb.x0[1], pb.x0[2], pb.x0[3], pb.x0[4]};
  double dD[NV], dO[NV];
#pragma unroll
  for (int c = 0; c < NV; ++c) { dD[c] = 0.0; dO[c] = 0.0; }
  double val[4] = {0.0, 0.0, 0.0, 0.0}, slope[4] = {0.0, 0.0, 0.0, 0.0};
  double cv = 0.0;

  auto advance = [&](auto jtag) {
    constexpr int j = decltype(jtag)::value;  // step j -> j+1
    const double s = X[0], d = X[1], o = X[2], k = X[3], v = X[4];
    const double kk = k - val[2];
    double nD[NV], nO[NV];
#pragma unroll
    for (int c = 0; c < NV; ++c) { nD[c] = dD[c]; nO[c] = dO[c]; }
#pragma unroll
    for (int i = 0; i < j; ++i) {
      const double ds = (i < j - 1) ? h * h * (double)(j - 1 - i) : 0.0;
      // a_i :  dk_j = h, dv_j = 0
      nD[2 * i] = dD[2 * i] + h * (v * dO[2 * i]);
      nO[2 * i] = dO[2 * i] + h * (v * h);
      // b_i :  dv_j = h, ds_j = ds
      nD[2 * i + 1] = dD[2 * i + 1] + h * (h * o + v * dO[2 * i + 1]);
      nO[2 * i + 1] = dO[2 * i + 1] + h * (h * kk - v * (slope[2] * ds));
    }
#pragma unroll
    for (int c = 0; c < NV; ++c) { dD[c] = nD[c]; dO[c] = nO[c]; }
    X[0] = s + h * v;
    X[1] = d + h * (v * o);
    X[2] = o + h * (v * kk);
    X[3] = k + h * pb.U[2 * j];
    X[4] = v + h * pb.U[2 * j + 1];
  };

  lookup_state_hint(T, X[0], val, slope, pb.hint[0]);
  advance(std::integral_constant<int, 0>{});
  // step 1: rows constant in U
  lookup_state_hint(T, X[0], val, slope, pb.hint[1]);
  accumulate_step<1>(P, H, g, dD, dO, X, val, slope);
  cv = dmax(cv, fabs(X[1]) - P.sld);
  cv = dmax(cv, fabs(X[1] + P.alpha_lane[2] * X[2]) - P.sld);
  advance(std::integral_constant<int, 1>{});
  lookup_state_hint(T, X[0], val, slope, pb.hint[2]);
  accumulate_step<2>(P, H, g, dD, dO, X, val, slope);
  lane_rows<2>(P, pb, st, dD, dO, X);
  advance(std::integral_constant<int, 2>{});
  lookup_state_hint(T, X[0], val, slope, pb.hint[3]);
  accumulate_step<3>(P, H, g, dD, dO, X, val, slope);
  lane_rows<3>(P, pb, st, dD, dO, X);
  advance(std::integral_constant<int, 3>{});
  lookup_state_hint(T, X[0], val, slope, pb.hint[4]);
  accumulate_step<4>(P, H, g, dD, dO, X, val, slope);
  lane_rows<4>(P, pb, st, dD, dO, X);
  advance(std::integral_constant<int, 4>{});
  lookup_state_hint(T, X[0], val, slope, pb.hint[5]);
  accumulate_step<5>(P, H, g, dD, dO, X, val, slope);
  lane_rows<5>(P, pb, st, dD, dO, X);

  // q = g - H U
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    double acc = g[i];
#pragma unroll
    for (int j = 0; j < NV; ++j) acc = fma(-H[i >= j ? tri(i, j) : tri(j, i)], pb.U[j], acc);
    st.q[i] = acc;
  }
  if constexpr (IsTmem<decltype(st.D)>::value) tmem_wait_st();   // D, O complete before the first read
  const_viol = cv;
}

template <class ST>
MPCB_HD void linearise(const DevTable& T, const DevParams& P, Problem& pb, const ST& st, double& const_viol) {
  double H[NTRI];
  linearise(T, P, pb, st, const_viol, H);
#pragma unroll
  for (int i = 0; i < NTRI; ++i) st.H[i] = H[i];
}

// ------------------------------------------------------------------------------------------------
// Row walk.  f(r, zt_r, lo, hi) is called for every row in index order with the row value zt_r = (A x)_r.
// Absent obstacles keep their rows (bounds BIG, rho 0 by construction), so the walk has no data-dependent branch.
// ------------------------------------------------------------------------------------------------
template <class ST, class F>
MPCB_HD void for_rows(const DevParams& P, const Problem& pb, const ST& st, const double (&x)[NV], F&& f) {
  const double h = P.h;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if (i & 1) f(i, x[i], st.blo[i >> 1], st.bhi[i >> 1], RowKind<0>{});
    else f(i, x[i], P.umin[0], P.umax[0], RowKind<0>{});
  }
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    double dj = 0.0, oj = 0.0;
    if constexpr (IsTmem<decltype(st.D)>::value) {
      double Db[8], Ob[8];
      tload(st.D, doff(jj), 2 * (jj + 1), Db);
      tload(st.O, doff(jj), 2 * (jj + 1), Ob);
#pragma unroll
      for (int c = 0; c < 2 * (jj + 1); ++c) {
        dj = fma(Db[c], x[c], dj);
        oj = fma(Ob[c], x[c], oj);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 2 * (jj + 1); ++c) {
        dj = fma(st.D[doff(jj) + c], x[c], dj);
        oj = fma(st.O[doff(jj) + c], x[c], oj);
      }
    }
    f(ROW_LANE + 2 * jj, dj, -P.sld - st.lane_c[2 * jj], P.sld - st.lane_c[2 * jj], RowKind<0>{});
    f(ROW_LANE + 2 * jj + 1, fma(P.alpha_lane[2], oj, dj), -P.sld - st.lane_c[2 * jj + 1],
      P.sld - st.lane_c[2 * jj + 1], RowKind<0>{});
  }
  double cum = 0.0, Sj = 0.0;
#pragma unroll
  for (int j = 1; j <= NH; ++j) {
    // S_j = h sum_{m<j} (v_m - v0);  cum = v_j - v0
    if (j > 1) Sj = fma(h, cum, Sj);
    cum = fma(h, x[2 * (j - 1) + 1], cum);
    f(ROW_V + j - 1, cum, st.lov[j - 1], BIG, RowKind<1>{});
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k < ST::KOBS) {
        if (j > 1) f(row_r1(k, j), Sj, -BIG, st.hio[N_OBSROW * k + (j - 2)], RowKind<2>{});
        f(row_r2(k, j), fma(P.tgap, cum, Sj), -BIG, st.hio[N_OBSROW * k + 4 + (j - 1)], RowKind<2>{});
      }
    }
  }
}

// out += A' w, fed row by row in the order for_rows walks (no per-row array needs to be kept):
//   box rows add straight into out; a lane step's two rows are folded into (wD, wO) and applied when the second
//   one arrives; speed / obstacle rows are folded into per-step sums Tv, Ts and applied by finish().
template <class ST>
struct AtAcc {
  const DevParams& P;
  const ST& st;
  double (&out)[NV];
  double w0;
  double Tv[NH], Ts[NH];
  MPCB_HD AtAcc(const DevParams& P_, const ST& st_, double (&out_)[NV]) : P(P_), st(st_), out(out_), w0(0.0) {
#pragma unroll
    for (int j = 0; j < NH; ++j) { Tv[j] = 0.0; Ts[j] = 0.0; }
  }
  MPCB_HD void add(int r, double w) {     // r is a compile-time constant after unrolling
    if (r < ROW_LANE) {
      out[r] += w;
    } else if (r < ROW_V) {
      const int jj = (r - ROW_LANE) >> 1;
      if (((r - ROW_LANE) & 1) == 0) {
        w0 = w;
      } else {
        const double wD = w0 + w, wO = P.alpha_lane[2] * w;
        if constexpr (IsTmem<decltype(st.D)>::value) {
          double Db[8], Ob[8];
          tload(st.D, doff(jj), 2 * (jj + 1), Db);
          tload(st.O, doff(jj), 2 * (jj + 1), Ob);
#pragma unroll
          for (int c = 0; c < 8; ++c)
            if (c < 2 * (jj + 1)) out[c] = fma(Db[c], wD, fma(Ob[c], wO, out[c]));
        } else {
#pragma unroll
          for (int c = 0; c < NV; ++c)
            if (c < 2 * (jj + 1)) out[c] = fma(st.D[doff(jj) + c], wD, fma(st.O[doff(jj) + c], wO, out[c]));
        }
      }
    } else if (r < ROW_OBS) {
      Tv[r - ROW_V] += w;
    } else {
      const int q = (r - ROW_OBS) % N_OBSROW;
      if (q < 4) {
        Ts[q + 1] += w;                       // R1_j, j = q + 2
      } else {
        Tv[q - 4] = fma(P.tgap, w, Tv[q - 4]);   // R2_j, j = q - 3
        Ts[q - 4] += w;
      }
    }
  }
  MPCB_HD void finish() {
    // b_i += h sum_{j>i} Tv[j] + h^2 sum_{j>=i+2} (j-1-i) Ts[j]      (j is 1-based; arrays are j-1)
    const double h = P.h;
    double sv = 0.0, ps = 0.0, cs = 0.0;
#pragma unroll
    for (int i = NH - 1; i >= 0; --i) {
      sv += Tv[i];
      out[2 * i + 1] = fma(h, sv, fma(h * h, cs, out[2 * i + 1]));
      ps += Ts[i];
      cs += ps;
    }
  }
};

// ------------------------------------------------------------------------------------------------
// rho_r from the rungs, then K = H + A' diag(rho) A = L L'  (packed lower triangle, reciprocal diagonal kept)
// ------------------------------------------------------------------------------------------------
// TWO: the two-level policy (two rungs, no hysteresis, inactive rows drop at once).  Under it a row's rung after a
// check is simply "was active in that check", i.e. the rung vector IS the bit mask act_prev: no 4-bit rung fields to
// read, modify and write back, and the two step sizes are selected, not looked up.
// K: the Gauss-Newton Hessian H on entry (st.H is not read), overwritten.
template <bool TWO, class ST>
MPCB_HD void factor(const DevParams& P, const Policy& pl, Problem& pb, const ST& st, double (&K)[NTRI]) {
  const double h = P.h;
  // step sizes of this factorisation
  const double lad0 = pl.lad[0], lad1 = pl.lad[1];
  auto step_size = [&](int r) -> double {
    if (TWO) return ((pb.act_prev >> r) & 1ull) ? lad1 : lad0;
    return pl.lad[pb.E.get(r)];
  };
#pragma unroll
  for (int i = 0; i < NV; ++i) st.rho[i] = step_size(i);
#pragma unroll
  for (int r = 0; r < N_LANE; ++r) st.rho[ROW_LANE + r] = step_size(ROW_LANE + r) * st.lane_inrm[r];
#pragma unroll
  for (int j = 1; j <= NH; ++j) {
    st.rho[ROW_V + j - 1] = step_size(ROW_V + j - 1) * P.inrm_v[j - 1];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k < ST::KOBS) {
        const bool on = k < pb.n_obs;
        if (j > 1) st.rho[row_r1(k, j)] = on ? step_size(row_r1(k, j)) * P.inrm_r1[j - 1] : 0.0;
        st.rho[row_r2(k, j)] = on ? step_size(row_r2(k, j)) * P.inrm_r2[j - 1] : 0.0;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) K[tri(i, i)] += st.rho[i];
  // lane rows of step j:  rho0 D D' + rho1 (D + wb O)(D + wb O)' = D (r0 D + r1 O)' + O (r1 D + r2 O)'
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    const double rho0 = st.rho[ROW_LANE + 2 * jj], rho1 = st.rho[ROW_LANE + 2 * jj + 1];
    const double wb = P.alpha_lane[2];
    const double r0 = rho0 + rho1, r1 = rho1 * wb, r2 = rho1 * wb * wb;
    auto rank2 = [&](const auto& Dc, const auto& Oc) {
#pragma unroll
      for (int i = 0; i < 2 * (jj + 1); ++i) {
        const double Di = Dc[doff(jj) + i], Oi = Oc[doff(jj) + i];
        const double p = r0 * Di + r1 * Oi;
        const double t = r1 * Di + r2 * Oi;
#pragma unroll
        for (int j = 0; j <= i; ++j)
          K[tri(i, j)] = fma(p, Dc[doff(jj) + j], fma(t, Oc[doff(jj) + j], K[tri(i, j)]));
      }
    };
    if constexpr (IsTmem<decltype(st.D)>::value) {
      double Db[8], Ob[8];   // indexed from doff(jj) like the store
      tload(st.D, doff(jj), 2 * (jj + 1), Db);
      tload(st.O, doff(jj), 2 * (jj + 1), Ob);
      struct Block {
        const double* p; int o;
        MPCB_HD double operator[](int e) const { return p[e - o]; }
      };
      rank2(Block{Db, doff(jj)}, Block{Ob, doff(jj)});
    } else {
      rank2(st.D, st.O);
    }
  }
  // constant-coefficient rows act on the b entries only: Kb[i][k] += sum_r rho_r c_r[i] c_r[k]
#pragma unroll
  for (int j = 1; j <= NH; ++j) {
    const double rv = st.rho[ROW_V + j - 1];
    double r1 = 0.0, r2 = 0.0;   // summed over obstacles (same coefficient vectors)
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k < ST::KOBS) {
        if (j > 1) r1 += st.rho[row_r1(k, j)];
        r2 += st.rho[row_r2(k, j)];
      }
    }
#pragma unroll
    for (int i = 0; i < j; ++i) {
      const double cs_i = h * h * (double)(j - 1 - i);   // S_j coefficient
      const double c2_i = cs_i + P.tgap * h;              // R2 coefficient
#pragma unroll
      for (int k = 0; k <= i; ++k) {
        const double cs_k = h * h * (double)(j - 1 - k);
        const double c2_k = cs_k + P.tgap * h;
        K[tri(2 * i + 1, 2 * k + 1)] += rv * (h * h) + r1 * (cs_i * cs_k) + r2 * (c2_i * c2_k);
      }
    }
  }
  // Cholesky K = L L' in place (lower), keeping reciprocal diagonals
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    double d = K[tri(j, j)];
#pragma unroll
    for (int k = 0; k < j; ++k) d = fma(-K[tri(j, k)], K[tri(j, k)], d);
    const double rs = rsqrt(d);
    K[tri(j, j)] = d * rs;
    if constexpr (!IsTmem<decltype(st.L)>::value) st.rdiag[j] = rs;
#pragma unroll
    for (int i = j + 1; i < NV; ++i) {
      double s = K[tri(i, j)];
#pragma unroll
      for (int k = 0; k < j; ++k) s = fma(-K[tri(i, k)], K[tri(j, k)], s);
      K[tri(i, j)] = s * rs;
    }
    if constexpr (IsTmem<decltype(st.L)>::value) {   // column j as chol_solve reads it: rdiag[j], L[j+1..9][j]
      double col[NV];
      col[0] = rs;
#pragma unroll
      for (int i = j + 1; i < NV; ++i) col[i - j] = K[tri(i, j)];
      tstore(st.L, fcol(j), NV - j, col);
    }
  }
  if constexpr (IsTmem<decltype(st.L)>::value) {
    tmem_wait_st();
  } else {
#pragma unroll
    for (int i = 0; i < NTRI; ++i) st.L[i] = K[i];
  }
}

template <bool TWO, class ST>
MPCB_HD void factor(const DevParams& P, const Policy& pl, Problem& pb, const ST& st) {
  double K[NTRI];
#pragma unroll
  for (int i = 0; i < NTRI; ++i) K[i] = st.H[i];
  factor<TWO>(P, pl, pb, st, K);
}

// x = K^-1 r through the factor (column-oriented substitutions: independent updates after every pivot)
template <class ST>
MPCB_HD void chol_solve(const ST& st, double (&r)[NV], double (&x)[NV]) {
  if constexpr (IsTmem<decltype(st.L)>::value) {
    // one column block per pivot; the back substitution reads column i of L to finish x[i], which applies the same
    // updates to r[i] in the same order (j = 9 down to i + 1) as the row updates below
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      double c[NV];
      tload(st.L, fcol(j), NV - j, c);
      r[j] *= c[0];
#pragma unroll
      for (int i = j + 1; i < NV; ++i) r[i] = fma(-c[i - j], r[j], r[i]);
    }
#pragma unroll
    for (int i = NV - 1; i >= 0; --i) {
      double c[NV];
      tload(st.L, fcol(i), NV - i, c);
#pragma unroll
      for (int j = NV - 1; j > i; --j) r[i] = fma(-c[j - i], x[j], r[i]);
      x[i] = r[i] * c[0];
    }
  } else {
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      r[j] *= st.rdiag[j];
#pragma unroll
      for (int i = j + 1; i < NV; ++i) r[i] = fma(-st.L[tri(i, j)], r[j], r[i]);
    }
#pragma unroll
    for (int j = NV - 1; j >= 0; --j) {
      x[j] = r[j] * st.rdiag[j];
#pragma unroll
      for (int i = 0; i < j; ++i) r[i] = fma(-st.L[tri(j, i)], x[j], r[i]);
    }
  }
}

struct SegStats { double rp, rd, nd, atdy, sup, bad; };   // rp: 0 when every row's primal residual is within eps_p,
                                                          // BIG otherwise (the exact maximum only in trace builds)

// One ADMM iteration.
//   CHECK = false: v += alpha (A x - clip(v)), nothing else.
//   CHECK = true : additionally residuals, active set, step-size policy; CERT adds the infeasibility certificate.
template <bool CHECK, bool CERT, bool TWO, class ST>
MPCB_HD void admm_iter(const DevParams& P, const Policy& pl, Problem& pb, const ST& st, SegStats& stt,
                       double eps_p = 0.0) {
  const double relax = pl.relax;
  double rhs[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) rhs[i] = -st.q[i];
  // pass A: w_r = rho_r (2 clip(v_r) - v_r); the plain iteration folds "- alpha clip(v)" into v on the way
  {
    AtAcc<ST> acc(P, st, rhs);
    for_rows(P, pb, st, pb.x, [&](int r, double, double lo, double hi, auto kind) {
      const double v = st.v[r];
      const double z = clipk<decltype(kind)::value>(v, lo, hi);
      acc.add(r, st.rho[r] * fma(2.0, z, -v));
      if (!CHECK) st.v[r] = fma(-relax, z, v);
    });
    acc.finish();
  }
  chol_solve(st, rhs, pb.x);
  if (!CHECK) {
    for_rows(P, pb, st, pb.x, [&](int r, double zt, double, double, auto) { st.v[r] = fma(relax, zt, st.v[r]); });
    return;
  }
  double o1[NV], o2[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) { o1[i] = 0.0; o2[i] = 0.0; }
  AtAcc<ST> acc1(P, st, o1), acc2(P, st, o2);
  double rp = 0.0, nd = 0.0, sup = 0.0, bad = 0.0;
  unsigned long long act = 0ull;
  for_rows(P, pb, st, pb.x, [&](int r, double zt, double lo, double hi, auto kind) {
    constexpr int KIND = decltype(kind)::value;
    const double v = st.v[r];
    const double rho = st.rho[r];
    const double z = clipk<KIND>(v, lo, hi);
    const double vn = fma(relax, zt - z, v);
    const double zn = clipk<KIND>(vn, lo, hi);
#ifdef MPCB_TRACE
    rp = dmax(rp, fabs(zt - zn));
#else
    if (!(fabs(zt - zn) <= eps_p)) rp = BIG;        // only "all rows within tolerance" is ever asked of rp
#endif
    // dual residual of (x, y_new): A' rho ((2 - alpha) z + (alpha - 1) zt - zn)
    acc1.add(r, rho * (fma(2.0 - relax, z, (relax - 1.0) * zt) - zn));
    if (CERT) {
      const double dy = rho * ((vn - zn) - (v - z));
      nd = dmax(nd, fabs(dy));
      if (dy > 0.0) { if (hi < BIG) sup = fma(hi, dy, sup); else bad = dmax(bad, dy); }
      else if (dy < 0.0) { if (lo > -BIG) sup = fma(lo, dy, sup); else bad = dmax(bad, -dy); }
      acc2.add(r, dy);
    }
    // step-size policy
    const bool a_now = outside<KIND>(vn, lo, hi);
    const bool a_prev = (pb.act_prev >> r) & 1ull;
    double vnew = vn;
    if (TWO) {
      // rung = activity in the previous check; a row that turns active moves up: keep (z, y), v' = z + (rho/rho')(v - z)
      if (a_now && !a_prev) vnew = fma(pl.lad_ratio[1], vn - zn, zn);
      if (a_now) act |= (1ull << r);
      st.v[r] = vnew;
      return;
    }
    const int e = pb.E.get(r);
    if (a_now && (a_prev || !pl.hysteresis) && e < pl.n_rung - 1) {
      pb.E.set(r, e + 1);
      vnew = fma(pl.lad_ratio[e + 1], vn - zn, zn);   // keep (z, y): v' = z + (rho/rho') (v - z)
    } else if (!a_now && (!a_prev || !pl.hysteresis) && e > 0) {
      pb.E.set(r, pl.drop_all ? 0 : e - 1);           // inactive: v == z, nothing to rescale
    }
    if (a_now) act |= (1ull << r);
    st.v[r] = vnew;
  });
  pb.act_prev = act;
  acc1.finish();
  double rd = 0.0, atdy = 0.0;
#pragma unroll
  for (int i = 0; i < NV; ++i) rd = dmax(rd, fabs(o1[i]));
  if (CERT) {
    acc2.finish();
#pragma unroll
    for (int i = 0; i < NV; ++i) atdy = dmax(atdy, fabs(o2[i]));
  }
  stt.rp = rp; stt.rd = rd; stt.nd = nd; stt.atdy = atdy; stt.sup = sup; stt.bad = bad;
}

// ------------------------------------------------------------------------------------------------
// Whole solve for one problem.
// ------------------------------------------------------------------------------------------------
struct SolveOut { int status, rounds, iters; bool const_infeasible; };

// Bounds of the rows that are exactly affine in U (speed, obstacle), and a rigorous screen: such a row that
// cannot be met anywhere inside the control box makes the problem infeasible whatever the other rows do
// (all coefficients are >= 0, so the row's extreme over the box sits at b = u2_min resp. u2_max).  Such a row is
// replaced by what violates it least without fighting the other affine rows: the accelerations it involves are pinned,
// through their box, to the "stop as fast as possible and stay stopped" profile (what a controller should do when it
// can no longer keep the gap), and the problem is flagged infeasible at once instead of waiting for an ADMM certificate.  Also: table hints, warm start
// (trajectory_tracking.py:223-246) clipped to the bounds as scipy does (_slsqp_py.py:322).  Returns "screened".
template <class ST>
MPCB_HD bool prologue(const DevTable& T, const DevParams& P, Problem& pb, const ST& st,
                      const double (*ur)[2] = nullptr) {   // ur: reference controls already looked up (pb.hint set)
  bool screened = false;
  double blo[NH], bhi[NH], bstop[NH];
  {
    // "stop as fast as the box allows and stay stopped" (never asks for a negative speed, so it cannot fight the
    // v_j >= 0 rows): the acceleration profile that violates an unreachable obstacle row least
    double vr = pb.x0[4];
#pragma unroll
    for (int i = 0; i < NH; ++i) {
      blo[i] = P.umin[1]; bhi[i] = P.umax[1];
      const double b = clipd(-vr / P.h, P.umin[1], P.umax[1]);
      bstop[i] = b;
      vr = fma(P.h, b, vr);
    }
  }
  // Pinning tightens the box, which can put further rows out of reach: sweep until nothing changes (each sweep pins
  // at least one more step or stops; 3 sweeps cover the cascades seen, the robust pass catches anything left).
  bool dead_v[NH], dead_1[2][NH], dead_2[2][NH];
#pragma unroll
  for (int j = 0; j < NH; ++j) { dead_v[j] = false; dead_1[0][j] = dead_1[1][j] = dead_2[0][j] = dead_2[1][j] = false; }
  for (int sweep = 0; sweep < 3; ++sweep) {
    double cum_lo = 0.0, cum_hi = 0.0, s_lo = 0.0;     // extremes over the current box of v_j - v0 and of S_j
#pragma unroll
    for (int j = 1; j <= NH; ++j) {
      if (j > 1) s_lo = fma(P.h, cum_lo, s_lo);        // S_j = h sum_{m<j} (v_m - v0)
      cum_lo = fma(P.h, blo[j - 1], cum_lo);
      cum_hi = fma(P.h, bhi[j - 1], cum_hi);
      bool pin_to_j = false, pin_to_jm1 = false;
      if (cum_hi < -pb.x0[4] - P.feas_tol) { dead_v[j - 1] = true; pin_to_j = true; }   // v_j >= 0 out of reach
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (k < ST::KOBS && k < pb.n_obs) {
          const double base = (pb.obs[k][0] + pb.obs[k][1] * (j * P.h)) - pb.x0[0] - j * P.h * pb.x0[4];
          if (s_lo > base - P.obs_safe + P.feas_tol) { dead_1[k][j - 1] = true; pin_to_jm1 = true; }   // j = 1: constant row
          if (fma(P.tgap, cum_lo, s_lo) > base - P.tgap * pb.x0[4] + P.feas_tol) { dead_2[k][j - 1] = true; pin_to_j = true; }
        }
      }
#pragma unroll
      for (int i = 0; i < NH; ++i)
        if ((pin_to_j && i < j) || (pin_to_jm1 && i < j - 1)) { blo[i] = bstop[i]; bhi[i] = bstop[i]; }
    }
  }
#pragma unroll
  for (int j = 1; j <= NH; ++j) {
    st.lov[j - 1] = dead_v[j - 1] ? -BIG : -pb.x0[4];
    screened |= dead_v[j - 1];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k < ST::KOBS) {
        const double base = (pb.obs[k][0] + pb.obs[k][1] * (j * P.h)) - pb.x0[0] - j * P.h * pb.x0[4];
        const bool on = k < pb.n_obs;
        if (j > 1) st.hio[N_OBSROW * k + (j - 2)] = (!on || dead_1[k][j - 1]) ? BIG : base - P.obs_safe;
        st.hio[N_OBSROW * k + 4 + (j - 1)] = (!on || dead_2[k][j - 1]) ? BIG : base - P.tgap * pb.x0[4];
        screened |= on && (dead_1[k][j - 1] || dead_2[k][j - 1]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NH; ++i) { st.blo[i] = blo[i]; st.bhi[i] = bhi[i]; }
  if (ur) warm_fill(P, pb.x0, pb.obs, pb.n_obs, ur, pb.U);
  else warm_start(T, P, pb.x0, pb.obs, pb.n_obs, pb.U, pb.hint);
  pb.hint[NH] = pb.hint[NH - 1];
#pragma unroll
  for (int i = 0; i < NV; ++i) pb.U[i] = clipd(pb.U[i], P.umin[i & 1], P.umax[i & 1]);  // scipy clips x0 to the bounds
#pragma unroll
  for (int i = 0; i < NH; ++i) pb.U[2 * i + 1] = clipd(pb.U[2 * i + 1], blo[i], bhi[i]);
  return screened;
}

// FIRST_PASS = true : two-level policy only; a QP it cannot close ends the attempt (status MPCB_MAXITER = "not
//                      certified"), no infeasibility verdict other than the rigorous screens.
// FIRST_PASS = false: robust ladder with OSQP's infeasibility certificate; inexact Gauss-Newton: the QP of a round is
//                      solved only as accurately as the previous SQP step warrants (P.qp_forcing).
// U_start (optional): controls to start from instead of the reference's warm start (clipped to the box and to the
// screen's pins like any start).  First pass: a HOT start -- the plan of a neighbouring problem, in the closed loop the
// previous time step's solution shifted by one step; rows that sit on their bounds there start as active, so the first
// segment is already a KKT solve on that active set (a vehicle waiting at a red light poses the same problem at every
// step: certified in one or two rounds instead of being left to the robust pass every time).
// The solve is cut into three pieces so that a kernel can stop a problem between two Gauss-Newton rounds, park what
// crosses the round boundary (SolveState, pb.U / x / act_prev / hint, v and the prologue's bounds in the store) and go on
// in another CTA; solve_one is their composition, which the host build, the robust pass and the evaluation kernel run.
struct SolveState {
  SolveOut out;
  bool done, infeasible, first, hot;
  int fails;
  double step_prev;
};

// start: prologue (screens, warm start), hot start, loop scalars
template <bool FIRST_PASS, class ST>
MPCB_HD void solve_start(const DevTable& T, const DevParams& P, Problem& pb, const ST& st, bool live,
                         const double* U_start, SolveState& s) {
  s.out = SolveOut{MPCB_MAXITER, 0, 0, false};
  const bool screened = prologue(T, P, pb, st);
  s.hot = FIRST_PASS && U_start != nullptr;
  if (U_start) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const double u = clipd(U_start[i], P.umin[i & 1], P.umax[i & 1]);
      pb.U[i] = (i & 1) ? clipd(u, st.blo[i >> 1], st.bhi[i >> 1]) : u;
    }
  }
  s.done = !live;
  s.infeasible = screened;
  s.out.const_infeasible = screened;
  s.first = true;
  s.step_prev = 1e30;
  s.fails = 0;
}

// one Gauss-Newton round: linearise (cold ADMM start on the first), segments, step test.  Every thread of the CTA calls it
// (the segment votes are CTA-uniform); a thread whose problem is done only takes part in the votes.
// ONESEG (first pass at thread_max_segments = 1, the only path whose store may sit in tensor memory): the round is one
// segment, so linearise hands H to factor in registers, and every lane of a warp that has an unfinished problem runs
// the round's arithmetic -- warp-convergent, as tcgen05.ld / st require -- while only lanes with an unfinished problem
// keep what it yields in pb.U and s (a finished lane's pb.x, act_prev, hints and store are scratch from then on: what is
// written out depends on pb.U and s alone).  A warp whose problems are all done skips the round as a whole.
template <bool FIRST_PASS, bool ONESEG = false, class ST>
MPCB_HD void solve_round(const DevTable& T, const DevParams& P, Problem& pb, const ST& st, SolveState& s, int round) {
  static_assert(!ONESEG || FIRST_PASS, "the one-segment round is the first pass's");
  const Policy& pl = P.pol[FIRST_PASS ? 1 : 0];
  const int max_segments = FIRST_PASS ? P.thread_max_segments : pl.max_segments;
  const bool hot = s.hot;
  // cold ADMM state at x: z = clip(A x), y = 0  ->  v = z ; all rows on the initial rung of policy m
  auto cold_start = [&](const double (&xx)[NV]) {
#pragma unroll
    for (int i = 0; i < 6; ++i) pb.E.w[i] = 0x11111111u * (unsigned)pl.e_init;
    unsigned long long act0 = 0ull;
    for_rows(P, pb, st, xx, [&](int r, double zt, double lo, double hi, auto kind) {
      constexpr int KIND = decltype(kind)::value;
      st.v[r] = clipk<KIND>(zt, lo, hi);
      // hot start (the controls come from a solution of a neighbouring problem, e.g. the previous time step's plan): a row
      // that sits on its bound there starts as active, so the first segment is already a KKT solve on that active set
      if (hot) {
        const bool at_lo = (KIND != 2) && (zt <= lo + P.feas_tol), at_hi = (KIND != 1) && (zt >= hi - P.feas_tol);
        if (at_lo || at_hi) act0 |= (1ull << r);
      }
    });
    pb.act_prev = act0;
  };
  auto start_round = [&](double cviol) {
    if (s.first) {
      cold_start(pb.U);
#pragma unroll
      for (int i = 0; i < NV; ++i) pb.x[i] = pb.U[i];
      s.first = false;
    }
    if (!s.done) {
      if (cviol > P.feas_tol) { s.infeasible = true; s.out.const_infeasible = true; }
      s.out.rounds++;
    }
  };
  bool conv = false;                           // this round's QP closed
  bool cert = false;
  if constexpr (ONESEG) {
#if defined(__CUDA_ARCH__)
    const bool work = __any_sync(0xffffffffu, !s.done);   // warp-uniform
#else
    const bool work = !s.done;
#endif
    if (work) {
      double H[NTRI], cviol;
      linearise(T, P, pb, st, cviol, H);
      start_round(cviol);
      factor<true>(P, pl, pb, st, H);
      SegStats ss;
      for (int it = 0; it < pl.segment_iters - 1; ++it) admm_iter<false, false, true>(P, pl, pb, st, ss);
      admm_iter<true, false, true>(P, pl, pb, st, ss, P.eps_p);
      if (!s.done) {
        s.out.iters += pl.segment_iters;
        conv = ss.rp <= P.eps_p && ss.rd <= P.eps_d;
      }
    }
  } else {
    if (!s.done) {
      double cviol;
      linearise(T, P, pb, st, cviol);
      start_round(cviol);
    }
    // inexact Gauss-Newton: a round's QP is only solved as accurately as the previous SQP step warrants
    const double step_prev = s.step_prev;
    const double loosen = (FIRST_PASS || P.qp_forcing <= 0.0) ? 1.0
                          : dmax(1.0, (step_prev * P.qp_forcing < P.qp_eps_loose ? step_prev * P.qp_forcing : P.qp_eps_loose) / P.eps_p);
    const double eps_p = P.eps_p * loosen, eps_d = P.eps_d * loosen;
    bool qdone = s.done;                         // nothing more to do on this round's QP (closed, certified or caps hit)
    for (int seg = 0; seg < max_segments; ++seg) {
      if (MPCB_ALL(qdone)) break;
      if (!qdone) {
        factor<FIRST_PASS>(P, pl, pb, st);
        SegStats ss;
        for (int it = 0; it < pl.segment_iters - 1; ++it) admm_iter<false, false, FIRST_PASS>(P, pl, pb, st, ss);
        admm_iter<true, !FIRST_PASS, FIRST_PASS>(P, pl, pb, st, ss, eps_p);
        s.out.iters += pl.segment_iters;
#ifdef MPCB_TRACE
        if (getenv("MPCB_TRACE")) {
          printf("  r%d s%d pass %d rp %.2e rd %.2e nd %.2e act %011llx E", round, seg, FIRST_PASS ? 1 : 2, ss.rp, ss.rd, ss.nd, pb.act_prev);
          for (int r = 0; r < M_ROWS; ++r) printf("%d", pb.E.get(r));
          printf(" x");
          for (int i = 0; i < NV; ++i) printf(" %.4f", pb.x[i]);
          printf("\n");
        }
#endif
        if (ss.rp <= eps_p && ss.rd <= eps_d) { conv = true; qdone = true; }
        else if (!FIRST_PASS && ss.nd > 1e-9 && ss.atdy <= P.eps_inf * ss.nd && ss.sup < -P.eps_inf * ss.nd &&
                 ss.bad <= P.eps_inf * ss.nd) { conv = true; cert = true; qdone = true; }
      }
    }
  }
  (void)round;
  if (!s.done) {
    double step = 0.0;
#pragma unroll
    for (int i = 0; i < NV; ++i) { step = dmax(step, fabs(pb.x[i] - pb.U[i])); pb.U[i] = pb.x[i]; }
    s.step_prev = step;
    if (cert) { s.infeasible = true; s.done = true; }
    else if (conv && step < P.step_tol) { s.done = true; s.out.status = 0; }
    else if (!conv) {
      // first pass: a QP it cannot close goes to the robust pass (after fast_fail_rounds tolerated ones);
      // robust pass: QPs that never close end as status 1, or 2 through the final constraint check
      ++s.fails;
      if (FIRST_PASS ? s.fails > P.fast_fail_rounds : s.fails >= P.max_fail_rounds) s.done = true;
    }
  }
}

// end: the infeasibility verdict and the box clip of the returned controls
template <bool FIRST_PASS>
MPCB_HD SolveOut solve_end(const DevParams& P, Problem& pb, const SolveState& s) {
  SolveOut out = s.out;
  // an infeasibility verdict is final only on a point the pass actually converged to (or, in the robust pass, gave
  // up on): a first pass that could not close its QP hands the problem over whatever the screens said
  if (s.infeasible && (!FIRST_PASS || out.status == 0)) out.status = 2;
  // the returned controls always respect the box (a no-op for converged problems; non-converged or infeasible
  // ADMM iterates may sit slightly outside).  SLSQP treats the bounds as hard in the same way.
#pragma unroll
  for (int i = 0; i < NV; ++i) pb.U[i] = clipd(pb.U[i], P.umin[i & 1], P.umax[i & 1]);
  return out;
}

// FIRST_PASS = true : two-level policy only; a QP it cannot close ends the attempt (status MPCB_MAXITER = "not
//                      certified"), no infeasibility verdict other than the rigorous screens.
// FIRST_PASS = false: robust ladder with OSQP's infeasibility certificate; inexact Gauss-Newton: the QP of a round is
//                      solved only as accurately as the previous SQP step warrants (P.qp_forcing).
// U_start (optional): controls to start from instead of the reference's warm start (clipped to the box and to the
// screen's pins like any start).  First pass: a HOT start -- the plan of a neighbouring problem, in the closed loop the
// previous time step's solution shifted by one step; rows that sit on their bounds there start as active, so the first
// segment is already a KKT solve on that active set (a vehicle waiting at a red light poses the same problem at every
// step: certified in one or two rounds instead of being left to the robust pass every time).
template <bool FIRST_PASS, class ST>
MPCB_HD SolveOut solve_one(const DevTable& T, const DevParams& P, Problem& pb, const ST& st, bool live,
                           const double* U_start = nullptr) {
  SolveState s;
  solve_start<FIRST_PASS>(T, P, pb, st, live, U_start, s);
  const int max_rounds = FIRST_PASS ? P.thread_max_rounds : P.max_rounds;
  for (int round = 0; round < max_rounds; ++round) {
    if (MPCB_ALL(s.done)) break;
    solve_round<FIRST_PASS>(T, P, pb, st, s, round);
  }
  return solve_end<FIRST_PASS>(P, pb, s);
}

}  // namespace mpcb
