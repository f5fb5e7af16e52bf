// qlb_solve_quad.cuh - the fused pipeline with ONE LEG PER LANE (four lanes per QP, eight QPs per warp).
//
// Everything that belongs to a leg - forward kinematics, Jacobian, gravity torques, the leg's three
// force components and five constraint rows, its 3x3 block K of the KKT matrix - lives in the registers
// of one thread and is plain straight-line FP64 code.  The only coupling between the legs of a QP is the
// 6x6 "dual" system  N t = rhs,  N = S^-1 + sum_legs A_k K_k^-1 A_k'  (A_k = the leg's 6x3 block of the
// wrench map): every lane accumulates its leg's contribution (21 + 6 numbers), a two-step butterfly
// (__shfl_xor 1, 2) sums them over the quad, and each lane then factorises the 6x6 matrix itself.
// Compared with the first design (a half-warp per QP around a 12x12 system, see git history) there is no
// redundant kinematics, no cross-lane exchange inside the linear algebra, and four times as many QPs per
// issued instruction.
//
// Reference path: see qlb_solve.cuh (ContactForceDistribution.cpp:99-136,138-336,385-578,614-625;
// quadrupedkinematics.cpp:143-278,485-552; VirtualModelController.cpp:89-268).
#pragma once

#include "qlb_solve.cuh"

namespace qlb {

#ifndef QLB_POLISH_MU
#define QLB_POLISH_MU 1e-5f      // interior point: complementarity gap (relative to the force scale) at which the
#define QLB_POLISH_MIN_IT 2      // rows with lambda > s are tried as the active set, and the earliest iteration for it
#endif
#ifndef QLB_PDAS_ROUNDS
#define QLB_PDAS_ROUNDS 4    // active-set repair rounds before a state is handed to the interior point
#endif
#ifndef QLB_IPM_MIN_CTAS
#define QLB_IPM_MIN_CTAS 3   // interior-point pass (and the single-pass variant)
#endif
#ifndef QLB_QUAD_MIN_CTAS
#define QLB_QUAD_MIN_CTAS 3
#endif
#ifndef QLB_FIRST_MIN_CTAS
#define QLB_FIRST_MIN_CTAS 3
#endif
constexpr int kQuadThreads = 128;

__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(kFull, v, 1));
  return fmaxf(v, __shfl_xor_sync(kFull, v, 2));
}
// max(|a|, |b|, |c|, |d|) over the quad, for the scales of tolerances.  A double is rounded down to its high word
// (< 2^-20 relative): the high words of |x| order like the values, so the comparisons and the shuffles are 32-bit
// integer work, off the FP64 pipe.  Scaling the inputs by a power of two scales the result exactly.
__device__ __forceinline__ int abs_hi(const double x) { return __double2hiint(x) & 0x7fffffff; }
__device__ __forceinline__ double from_hi(const int h) { return __hiloint2double(h, 0); }
__device__ __forceinline__ float quad_max_abs(float a, float b, float c, float d = 0.f) {
  return quad_max(fmaxf(fmaxf(fabsf(a), fabsf(b)), fmaxf(fabsf(c), fabsf(d))));
}
__device__ __forceinline__ double quad_max_abs(double a, double b, double c, double d = 0.0) {
  int h = max(max(abs_hi(a), abs_hi(b)), max(abs_hi(c), abs_hi(d)));
  h = max(h, __shfl_xor_sync(kFull, h, 1));
  h = max(h, __shfl_xor_sync(kFull, h, 2));
  return from_hi(h);
}
// max(|a|, |b|, |c|) of this lane (a double to its high word, as above)
__device__ __forceinline__ float lane_max_abs(float a, float b, float c) { return fmaxf(fabsf(a), fmaxf(fabsf(b), fabsf(c))); }
__device__ __forceinline__ double lane_max_abs(double a, double b, double c) { return from_hi(max(abs_hi(a), max(abs_hi(b), abs_hi(c)))); }
__device__ __forceinline__ float quad_min(float v) {
  v = fminf(v, __shfl_xor_sync(kFull, v, 1));
  return fminf(v, __shfl_xor_sync(kFull, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(kFull, v, 1);
  return v + __shfl_xor_sync(kFull, v, 2);
}
__device__ __forceinline__ double quad_sum(double v) {
  v += __shfl_xor_sync(kFull, v, 1);
  return v + __shfl_xor_sync(kFull, v, 2);
}
__device__ __forceinline__ unsigned quad_or(unsigned v) {
  v |= __shfl_xor_sync(kFull, v, 1);
  return v | __shfl_xor_sync(kFull, v, 2);
}

// Tolerances of the two arithmetic types, relative to the scale of the quantity they judge, with no absolute floor
// (a floor makes a state's result depend on the units of its inputs: forces of 1e-7 N against a 1 N floor of the
// feasibility test, or multipliers that scale with W against a floor that does not).
template <typename T> struct Tol;
template <> struct Tol<double> {
  __device__ static double feas() { return 1e-10; }   // a row counts as violated below -feas * max |y| of the state
  __device__ static double mult() { return 1e-13; }   // a multiplier counts as negative below -mult * max(|W y|, |A' t|)
  __device__ static float ipm(float tol) { return tol; }
  static constexpr bool refine = false;
  static constexpr bool rescue = false;
};
template <> struct Tol<float> {
  __device__ static float feas() { return 1e-5f; }
  __device__ static float mult() { return 3e-6f; }
  __device__ static float ipm(float tol) { return fmaxf(tol, 1e-4f); }  // FP32 residuals stall near 1e-5 * scale
  static constexpr bool refine = true;  // iterative refinement of the polish solves
  static constexpr bool rescue = true;  // states the FP32 core cannot verify go to a.list3 (FP64-core pass)
};

#define QLB_TRI(i, j) ((i) * ((i) + 1) / 2 + (j))

// In-thread Cholesky of a packed lower-triangular 6x6 SPD matrix; A <- L (strict lower part), rdg = 1/diag(L).
// All loops have constant trip counts and the triangle is cut with `if`: nvcc does not unroll loops whose
// bounds depend on an outer induction variable, and a rolled loop would put the matrix in local memory.
template <typename real>
__device__ __forceinline__ bool chol6_thread(real (&A)[21], real (&rdg)[6]) {
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; j++) {
    real d = A[QLB_TRI(j, j)];
#pragma unroll
    for (int k = 0; k < 6; k++)
      if (k < j) d = fma(-A[QLB_TRI(j, k)], A[QLB_TRI(j, k)], d);
    ok = ok && (d > real(0.0));
    const real r = fast_rsqrt(d);
    rdg[j] = r;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      if (i > j) {
        real s = A[QLB_TRI(i, j)];
#pragma unroll
        for (int k = 0; k < 6; k++)
          if (k < j) s = fma(-A[QLB_TRI(i, k)], A[QLB_TRI(j, k)], s);
        A[QLB_TRI(i, j)] = s * r;
      }
    }
  }
  return ok;
}
template <typename real>
__device__ __forceinline__ void solve6_thread(const real (&L)[21], const real (&rdg)[6], real (&x)[6]) {
#pragma unroll
  for (int i = 0; i < 6; i++) {
    real s = x[i];
#pragma unroll
    for (int k = 0; k < 6; k++)
      if (k < i) s = fma(-L[QLB_TRI(i, k)], x[k], s);
    x[i] = s * rdg[i];
  }
#pragma unroll
  for (int i = 5; i >= 0; i--) {
    real s = x[i];
#pragma unroll
    for (int k = 0; k < 6; k++)
      if (k > i) s = fma(-L[QLB_TRI(k, i)], x[k], s);
    x[i] = s * rdg[i];
  }
}

// In-thread LDL' of a packed lower-triangular 6x6 SPD matrix; A <- L (strict lower part, unit diagonal), rd = 1/D.
// The same pivots as chol6_thread (D_j is the square of its diagonal; a non-positive one is a failure), built row by
// row from the unscaled row s_jk = L_jk D_k.  What differs is the dependent chain between two pivots: one reciprocal
// (seed + two Newton steps, 4 dependent operations) and one FMA (D_j's last term s^2 / D_{j-1}) instead of a
// reciprocal square root (6), the column scaling and an FMA.
template <typename real>
__device__ __forceinline__ bool ldl6_thread(real (&A)[21], real (&rd)[6]) {
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; j++) {
    real s[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
      if (k < j) {
        real t = A[QLB_TRI(j, k)];
#pragma unroll
        for (int m = 0; m < 6; m++)
          if (m < k) t = fma(-s[m], A[QLB_TRI(k, m)], t);
        s[k] = t;
      }
    }
    real d = A[QLB_TRI(j, j)];
#pragma unroll
    for (int k = 0; k < 6; k++) {
      if (k < j) {
        A[QLB_TRI(j, k)] = s[k] * rd[k];
        d = (k + 1 < j) ? fma(-s[k], A[QLB_TRI(j, k)], d) : fma(-(s[k] * s[k]), rd[k], d);
      }
    }
    ok = ok && (d > real(0.0));
    rd[j] = fast_rcp(d);
  }
  return ok;
}
// L D L' x = b for the factors of ldl6_thread (x: b in, solution out).  Each substitution sums its terms with the one
// that was computed last at the end of the chain.
template <typename real>
__device__ __forceinline__ void ldl6_solve(const real (&L)[21], const real (&rd)[6], real (&x)[6]) {
#pragma unroll
  for (int i = 1; i < 6; i++) {
    real s = x[i];
#pragma unroll
    for (int k = 0; k < 6; k++)
      if (k < i) s = fma(-L[QLB_TRI(i, k)], x[k], s);
    x[i] = s;
  }
#pragma unroll
  for (int i = 0; i < 6; i++) x[i] *= rd[i];
#pragma unroll
  for (int i = 4; i >= 0; i--) {
    real s = x[i];
#pragma unroll
    for (int k = 5; k > 0; k--)
      if (k > i) s = fma(-L[QLB_TRI(k, i)], x[k], s);
    x[i] = s;
  }
}

// One step of iterative refinement for (S^-1 + sum_legs sum_c al_c v_c v_c') t = rhs with the residual
// evaluated through the factors v_c (not through the assembled matrix, whose large entries have already
// rounded the S^-1 part away).  Used by the FP32 core only: it brings the solve from cond * eps ~ 5e-3
// to the level of the input rounding.  Whole warp (quad shuffles).
template <typename real>
__device__ __forceinline__ void refine6(const real (&N)[21], const real (&rdg)[6], const real (&v)[3][6], const real (&al)[3],
                                        const real* sinv, const real (&rhs)[6], real (&t)[6]) {
  real d[3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    real acc = real(0.0);
#pragma unroll
    for (int r = 0; r < 6; r++) acc = fma(v[c][r], t[r], acc);
    d[c] = al[c] * acc;
  }
  real res[6];
#pragma unroll
  for (int r = 0; r < 6; r++) {
    const real kt = quad_sum(fma(d[0], v[0][r], fma(d[1], v[1][r], d[2] * v[2][r])));
    res[r] = (rhs[r] - sinv[r] * t[r]) - kt;
  }
  solve6_thread(N, rdg, res);
#pragma unroll
  for (int r = 0; r < 6; r++) t[r] += res[r];
}

// D~ y and D~' v for one leg (rows: y_n >= F_min, mu y_n +- y_1 >= 0, mu y_n +- y_2 >= 0); slots (n, 1, 2)
template <typename real>
__device__ __forceinline__ void leg_rows(real yn, real y1, real y2, real mu, real (&e)[5]) {
  const real m = mu * yn;
  e[0] = yn; e[1] = m + y1; e[2] = m - y1; e[3] = m + y2; e[4] = m - y2;
}
template <typename real>
__device__ __forceinline__ void leg_rows_t(const real (&v)[5], real mu, real (&o)[3]) {
  o[0] = fma(mu, (v[1] + v[2]) + (v[3] + v[4]), v[0]);
  o[1] = v[1] - v[2];
  o[2] = v[3] - v[4];
}

// Per-leg quantities that stay fixed while the QP is solved.
template <typename real>
struct LegSetup {
  real At[3][6];   // the leg's block of the wrench map in contact coordinates, At[c] = [e_c; r x e_c]
                     // (rows 0..2 are the friction frame n, t1, t2 itself; zero for a swing leg)
  real nrm[3];     // the leg's contact normal in base frame (also for swing legs)
  real foot[3];    // foot position in base frame
  real b[6];       // desired wrench
  real mu, c0;     // friction coefficient; normal force of the strictly feasible interior-point start
  float rm;          // 1 / number of constraint rows
  unsigned mask;
  int ns;
  bool alive, qbad, qinf;   // qinf: a stance leg has mu < 0 (no feasible force while F_min > 0)
};

#ifndef QLB_UNIT_VECTORS
#define QLB_UNIT_VECTORS 1   // enforce the unit-vector contract of the base quaternion and the surface normals in the kernel
#endif
#ifndef QLB_SMEM_MODEL
#define QLB_SMEM_MODEL 1     // the leg-model table is read from a per-CTA shared copy instead of global memory
#endif
#ifndef QLB_PIPELINE_LOADS
#define QLB_PIPELINE_LOADS 1
#endif
#ifndef QLB_PREFETCH_LEVEL
#define QLB_PREFETCH_LEVEL 2   // 0 off, 1 prefetch.global.L1, 2 prefetch.global.L2
#endif
__device__ __forceinline__ void prefetch_global(const void* p) {
#if QLB_PREFETCH_LEVEL == 1
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#elif QLB_PREFETCH_LEVEL == 2
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#endif
}

// Prefetch the input rows of the state this lane will load next (the rows of its own leg; the rows shared
// by the quad are spread over its four lanes).  The loads of the next work item then hit in cache
// instead of stalling twelve warps per SM on DRAM latency (top stall of the first pass in ncu).
template <typename real, int MODE>
__device__ __forceinline__ void quad_prefetch(const SolveArgsT<real>& a, const unsigned long long bx, const int leg) {
#if QLB_PREFETCH_LEVEL > 0
  const unsigned long long B = a.B;
#pragma unroll
  for (int j = 0; j < 3; j++) prefetch_global(a.q + (size_t)(3 * leg + j) * B + bx);
  if (MODE == 1) {
    prefetch_global(a.pose + (size_t)leg * B + bx);
    if (leg < 3) prefetch_global(a.pose + (size_t)(4 + leg) * B + bx);
    prefetch_global(a.tpose + (size_t)leg * B + bx);
    if (leg < 3) prefetch_global(a.tpose + (size_t)(4 + leg) * B + bx);
    prefetch_global(a.twist + (size_t)leg * B + bx);
    if (leg < 2) prefetch_global(a.twist + (size_t)(4 + leg) * B + bx);
    prefetch_global(a.ttwist + (size_t)leg * B + bx);
    if (leg < 2) prefetch_global(a.ttwist + (size_t)(4 + leg) * B + bx);
  } else {
    prefetch_global(a.quat + (size_t)leg * B + bx);
    prefetch_global(a.wrench + (size_t)leg * B + bx);
    if (leg < 2) prefetch_global(a.wrench + (size_t)(4 + leg) * B + bx);
  }
  if (a.mu != nullptr) prefetch_global(a.mu + (size_t)leg * B + bx);
  if (a.normals != nullptr) {
#pragma unroll
    for (int c = 0; c < 3; c++) prefetch_global(a.normals + (size_t)(3 * leg + c) * B + bx);
  }
#endif
}

// The raw inputs of one state as this lane needs them (its own leg's joint angles, friction coefficient and
// normal; the base state and the wrench, which the four lanes of a quad load redundantly).
template <typename real, int MODE>
struct RawIn {
  real qj[3];
  real quat[4];              // wrench mode
  real b[6];                 // wrench mode: the desired wrench
  real pose[MODE == 1 ? 7 : 1], tw[MODE == 1 ? 6 : 1], tp[MODE == 1 ? 7 : 1], tt[MODE == 1 ? 6 : 1];  // state mode
  real mu;
  real nw[3];
  unsigned mask;
};

// Issue the loads of state bx (each row of 8 consecutive states is one 64-byte segment).  Kept apart from
// quad_setup so that the first pass can have the next work item's loads in flight while it writes the current one.
template <typename real, int MODE>
__device__ __forceinline__ void quad_load(const SolveArgsT<real>& a, const real mu_default, const unsigned long long bx,
                                          const bool valid, const int leg, RawIn<real, MODE>& in) {
  const unsigned long long B = a.B;
  in.mask = valid ? (unsigned)a.mask[bx] & 0xFu : 0u;
#pragma unroll
  for (int j = 0; j < 3; j++) in.qj[j] = __ldg(a.q + (size_t)(3 * leg + j) * B + bx);
  if (MODE == 1) {
#pragma unroll
    for (int r = 0; r < 7; r++) { in.pose[r] = __ldg(a.pose + (size_t)r * B + bx); in.tp[r] = __ldg(a.tpose + (size_t)r * B + bx); }
#pragma unroll
    for (int r = 0; r < 6; r++) { in.tw[r] = __ldg(a.twist + (size_t)r * B + bx); in.tt[r] = __ldg(a.ttwist + (size_t)r * B + bx); }
  } else {
#pragma unroll
    for (int r = 0; r < 4; r++) in.quat[r] = __ldg(a.quat + (size_t)r * B + bx);
#pragma unroll
    for (int r = 0; r < 6; r++) in.b[r] = __ldg(a.wrench + (size_t)r * B + bx);
  }
  in.mu = (a.mu != nullptr) ? __ldg(a.mu + (size_t)leg * B + bx) : mu_default;
  in.nw[0] = real(0.0); in.nw[1] = real(0.0); in.nw[2] = real(1.0);
  if (a.normals != nullptr) {
#pragma unroll
    for (int c = 0; c < 3; c++) in.nw[c] = __ldg(a.normals + (size_t)(3 * leg + c) * B + bx);
  }
}

// Per-CTA shared copy of the leg-model table (2.2 KB in FP64), filled by load_model_to_smem at kernel start.
__device__ __forceinline__ double* smem_model_buffer() {
  __shared__ double buf[sizeof(DeviceModelT<double>) / sizeof(double)];
  return buf;
}
template <typename real>
__device__ __forceinline__ void load_model_to_smem(const DeviceModelT<real>* src) {
#if QLB_SMEM_MODEL
  const uint32_t* s32 = reinterpret_cast<const uint32_t*>(src);
  uint32_t* d32 = reinterpret_cast<uint32_t*>(smem_model_buffer());
  for (int i = threadIdx.x; i < (int)(sizeof(DeviceModelT<real>) / 4); i += blockDim.x) d32[i] = s32[i];
#endif
}

// Everything from the raw inputs of one state (lane = leg `leg`) up to the QP data.
// creal: the type of the QP data (friction frame, wrench map, desired wrench).  With FP32 inputs and the FP64 solver
// core the frame is built in FP64 from the FP32 quaternion and normal, so that it is orthonormal to FP64 rounding and
// the solver may use the identities that rest on Q Q' = I; the leg kinematics (the bulk of the work) stay in `real`.
template <typename real, int MODE, typename creal = real>
__device__ __forceinline__ void quad_setup(const SolveArgsT<real>& a, const DeviceParamsT<real>& prm, const RawIn<real, MODE>& in,
                                           const unsigned long long bq, const bool valid, const bool write_wout,
                                           const int leg, LegSetup<creal>& L, real* const jgp, const int jgs) {
  // jgp / jgs: where this lane parks its leg's Jacobian (9) and gravity torques (3): element k at jgp[k * jgs]
  const unsigned long long B = a.B;
#if QLB_SMEM_MODEL
  const DeviceModelT<real>& mdl = *reinterpret_cast<const DeviceModelT<real>*>(smem_model_buffer());
#define QLB_MDL(x) (x)
#else
  const DeviceModelT<real>& mdl = *a.model;
#define QLB_MDL(x) __ldg(&(x))
#endif
    const unsigned mask = in.mask;
    L.mask = mask;
    const bool alive = (mask >> leg) & 1u;
    const int ns = __popc(mask);
    L.alive = alive; L.ns = ns;
    real qj[3] = {in.qj[0], in.qj[1], in.qj[2]};
    // joint angles beyond 1e6 rad are outside the range of the argument reduction (and NaN / Inf fail the comparison)
    bool bad = !(fabs(qj[0]) <= real(1e6) && fabs(qj[1]) <= real(1e6) && fabs(qj[2]) <= real(1e6));
    real quat[4];
    real b[6];
    if (MODE == 1) {
      // virtual model controller prologue (VirtualModelController.cpp:104-268), redundantly on the quad
      const real (&pose)[MODE == 1 ? 7 : 1] = in.pose;
      const real (&tw)[MODE == 1 ? 6 : 1] = in.tw;
      const real (&tp)[MODE == 1 ? 7 : 1] = in.tp;
      const real (&tt)[MODE == 1 ? 6 : 1] = in.tt;
#pragma unroll
      for (int r = 0; r < 7; r++) bad |= !isfinite(pose[r]) || !isfinite(tp[r]);
#pragma unroll
      for (int r = 0; r < 6; r++) bad |= !isfinite(tw[r]) || !isfinite(tt[r]);
#pragma unroll
      for (int r = 0; r < 4; r++) quat[r] = pose[3 + r];
      const real w = quat[0], x = quat[1], y = quat[2], z = quat[3];
      real R[9];
      R[0] = w * w + x * x - y * y - z * z; R[1] = real(2.0) * (x * y - w * z); R[2] = real(2.0) * (x * z + w * y);
      R[3] = real(2.0) * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = real(2.0) * (y * z - w * x);
      R[6] = real(2.0) * (x * z - w * y); R[7] = real(2.0) * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
      real ep[3], ev[3], ew[3], eR[3];
#pragma unroll
      for (int c = 0; c < 3; c++) { ep[c] = tp[c] - pose[c]; ev[c] = tt[c] - tw[c]; ew[c] = tt[3 + c] - tw[3 + c]; }
      quat_rel_log(tp + 3, quat, eR);
      real gbv[3], Fg[3], Tg[3], ft[3];
#pragma unroll
      for (int c = 0; c < 3; c++) { gbv[c] = -prm.gravity * R[6 + c]; ft[c] = -prm.grav_pct * prm.torso_mass * gbv[c]; Fg[c] = ft[c]; }
      Tg[0] = prm.com[1] * ft[2] - prm.com[2] * ft[1];
      Tg[1] = prm.com[2] * ft[0] - prm.com[0] * ft[2];
      Tg[2] = prm.com[0] * ft[1] - prm.com[1] * ft[0];
#pragma unroll
      for (int l = 0; l < 4; l++) {
        real fl[3], rr[3];
#pragma unroll
        for (int c = 0; c < 3; c++) { fl[c] = -prm.grav_pct * prm.leg_mass[l] * gbv[c]; Fg[c] += fl[c]; rr[c] = prm.leg_pos[l][c] - prm.com[c]; }
        Tg[0] += rr[1] * fl[2] - rr[2] * fl[1];
        Tg[1] += rr[2] * fl[0] - rr[0] * fl[2];
        Tg[2] += rr[0] * fl[1] - rr[1] * fl[0];
      }
      const real gfz = prm.kp_t[2] * ep[2], gdz = prm.kd_t[2] * ev[2], fwz = prm.kff_r[2] * tt[5];
      const real dwv[3] = {prm.kd_r[0] * ew[0], prm.kd_r[1] * ew[1], prm.kd_r[2] * ew[2]};
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const real epb = R[c] * ep[0] + R[3 + c] * ep[1] + R[6 + c] * ep[2];
        const real evb = R[c] * ev[0] + R[3 + c] * ev[1] + R[6 + c] * ev[2];
        const real ffb = R[c] * tt[0] + R[3 + c] * tt[1];
        b[c] = prm.kp_t[c] * epb + prm.kd_t[c] * evb + prm.kff_t[c] * ffb + Fg[c] + R[6 + c] * gfz + R[6 + c] * gdz;
        const real dwb = R[c] * dwv[0] + R[3 + c] * dwv[1] + R[6 + c] * dwv[2];
        b[3 + c] = -prm.kp_r[c] * eR[c] + dwb + R[6 + c] * fwz + Tg[c];
      }
      if (a.wrench_out && valid && leg == 0 && write_wout) {
#pragma unroll
        for (int r = 0; r < 6; r++) a.wrench_out[(size_t)r * B + bq] = b[r];
      }
    } else {
#pragma unroll
      for (int r = 0; r < 4; r++) { quat[r] = in.quat[r]; bad |= !isfinite(quat[r]); }
#pragma unroll
      for (int r = 0; r < 6; r++) { b[r] = in.b[r]; bad |= !isfinite(b[r]); }
    }
#pragma unroll
    for (int r = 0; r < 6; r++) L.b[r] = (creal)b[r];
    const real mu = in.mu;
    L.mu = (creal)mu;

    // ---------------- base rotation, friction frame (CFD.cpp:223,237,286-309), gravity in base frame (:518-519)
    // The contact coordinates rest on an orthonormal frame: the quaternion and the normal must be unit vectors.
    // Rounding-level deviations (FP32 inputs, a sloppy normalisation) are removed here; anything beyond 1e-5 is
    // refused as bad input (the reference would silently scale the normal force bound and the friction coefficient).
    creal E[3][3];  // E[0] = n, E[1] = t1, E[2] = t2 in base frame
    real gb[3];
    {
      creal w = (creal)quat[0], x = (creal)quat[1], y = (creal)quat[2], z = (creal)quat[3];
      creal nv[3] = {(creal)in.nw[0], (creal)in.nw[1], (creal)in.nw[2]};
#if QLB_UNIT_VECTORS
      // 1 / sqrt(1 + e) = 1 - e/2 + 3 e^2/8 + O(e^3): exact to rounding for |e| <= 1e-5, no branch, no special function
      const creal eq = (w * w + x * x + y * y + z * z) - creal(1.0), en = (nv[0] * nv[0] + nv[1] * nv[1] + nv[2] * nv[2]) - creal(1.0);
      bad |= !(fabs(eq) <= creal(1e-5)) || (alive && !(fabs(en) <= creal(1e-5)));
      const creal sq = fma(eq, fma(eq, creal(0.375), creal(-0.5)), creal(1.0));
      const creal sn = fma(en, fma(en, creal(0.375), creal(-0.5)), creal(1.0));
      w *= sq; x *= sq; y *= sq; z *= sq;
      nv[0] *= sn; nv[1] *= sn; nv[2] *= sn;
#endif
      const creal (&nw)[3] = nv;
      creal R[9];
      R[0] = w * w + x * x - y * y - z * z; R[1] = creal(2.0) * (x * y - w * z); R[2] = creal(2.0) * (x * z + w * y);
      R[3] = creal(2.0) * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = creal(2.0) * (y * z - w * x);
      R[6] = creal(2.0) * (x * z - w * y); R[7] = creal(2.0) * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
#pragma unroll
      for (int c = 0; c < 3; c++) {
        E[0][c] = R[c] * nw[0] + R[3 + c] * nw[1] + R[6 + c] * nw[2];
        gb[c] = -prm.gravity * (real)R[6 + c];
      }
      // t1 = n x (R' e_y) = R' (n_w x e_y), and n_w x e_y = (-n_z, 0, n_x) is exact: rotated as one vector it keeps its
      // direction to rounding however close the normal comes to the base y axis (the cross product of the two rotated
      // vectors, each rounded on its own, loses the digits that cancel: 1e-10 of the frame at |n x e_y| = 1e-6)
#pragma unroll
      for (int c = 0; c < 3; c++) E[1][c] = R[6 + c] * nw[0] - R[c] * nw[2];
      creal rn = fast_rsqrt(E[1][0] * E[1][0] + E[1][1] * E[1][1] + E[1][2] * E[1][2]);
#pragma unroll
      for (int c = 0; c < 3; c++) E[1][c] *= rn;
      E[2][0] = E[0][1] * E[1][2] - E[0][2] * E[1][1];
      E[2][1] = E[0][2] * E[1][0] - E[0][0] * E[1][2];
      E[2][2] = E[0][0] * E[1][1] - E[0][1] * E[1][0];
      rn = fast_rsqrt(E[2][0] * E[2][0] + E[2][1] * E[2][1] + E[2][2] * E[2][2]);
#pragma unroll
      for (int c = 0; c < 3; c++) E[2][c] *= rn;
      if (alive) {
        bad |= !isfinite(mu);
#pragma unroll
        for (int c = 0; c < 3; c++) bad |= !isfinite(E[0][c]) || !isfinite(E[1][c]) || !isfinite(E[2][c]);
      }
    }
    L.qbad = quad_or(bad ? 1u : 0u) != 0u;
    L.qinf = quad_or((alive && mu < real(0.0)) ? 1u : 0u) != 0u;

    // ---------------- leg forward kinematics, Jacobian, gravity torques (QK.cpp:143-278,485-552)
    real foot[3], J[3][3], gtau[3];  // J[j] = column j
    {
      real R[9], p[3], zj[3][3], pj[3][3], com[4][3];
#pragma unroll
      for (int e = 0; e < 9; e++) R[e] = QLB_MDL(mdl.rot[leg][0][e]);
#pragma unroll
      for (int c = 0; c < 3; c++) p[c] = QLB_MDL(mdl.xyz[leg][0][c]);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        if (j > 0) {
          // (Skipping the transforms that are trivial on all four legs - the knee's rpy and the thigh's xyz are zero in
          // both shipped models - through uniform branches executes 45 instructions less per tile and runs 1 % slower;
          // rolling the chain into a three-trip loop with the per-joint results in a shared-memory scratch removes 170
          // instructions from the kernel and runs 2.5 % slower: the schedule loses the interleaving across joints.)
          const real x0 = QLB_MDL(mdl.xyz[leg][j][0]), x1 = QLB_MDL(mdl.xyz[leg][j][1]), x2 = QLB_MDL(mdl.xyz[leg][j][2]);
#pragma unroll
          for (int c = 0; c < 3; c++) p[c] += R[3 * c] * x0 + R[3 * c + 1] * x1 + R[3 * c + 2] * x2;
          if (j < 3) {
            real Rj[9], T[9];
#pragma unroll
            for (int e = 0; e < 9; e++) Rj[e] = QLB_MDL(mdl.rot[leg][j][e]);
#pragma unroll
            for (int r = 0; r < 3; r++)
#pragma unroll
              for (int s = 0; s < 3; s++) T[3 * r + s] = R[3 * r] * Rj[s] + R[3 * r + 1] * Rj[3 + s] + R[3 * r + 2] * Rj[6 + s];
#pragma unroll
            for (int e = 0; e < 9; e++) R[e] = T[e];
          }
        }
        if (j < 3) {
#pragma unroll
          for (int c = 0; c < 3; c++) { zj[j][c] = R[3 * c + 2]; pj[j][c] = p[c]; }
          real sj, cj;
          sincos_small(qj[j], &sj, &cj);
#pragma unroll
          for (int r = 0; r < 3; r++) {
            const real a0 = R[3 * r], a1 = R[3 * r + 1];
            R[3 * r] = cj * a0 + sj * a1;
            R[3 * r + 1] = cj * a1 - sj * a0;
          }
        }
        const real c0 = QLB_MDL(mdl.com[leg][j][0]), c1 = QLB_MDL(mdl.com[leg][j][1]), c2 = QLB_MDL(mdl.com[leg][j][2]);
        const real mj = QLB_MDL(mdl.mass[leg][j]);
#pragma unroll
        for (int c = 0; c < 3; c++) com[j][c] = mj * (p[c] + R[3 * c] * c0 + R[3 * c + 1] * c1 + R[3 * c + 2] * c2);
      }
#pragma unroll
      for (int c = 0; c < 3; c++) foot[c] = p[c];
      real mcs[3] = {real(0.0), real(0.0), real(0.0)};
#pragma unroll
      for (int j = 3; j >= 0; j--) {
#pragma unroll
        for (int c = 0; c < 3; c++) mcs[c] += com[j][c];
        if (j < 3) {
          const real dv[3] = {foot[0] - pj[j][0], foot[1] - pj[j][1], foot[2] - pj[j][2]};
          J[j][0] = zj[j][1] * dv[2] - zj[j][2] * dv[1];
          J[j][1] = zj[j][2] * dv[0] - zj[j][0] * dv[2];
          J[j][2] = zj[j][0] * dv[1] - zj[j][1] * dv[0];
          const real ms = QLB_MDL(mdl.msuf[leg][j]);
          const real arm[3] = {mcs[0] - ms * pj[j][0], mcs[1] - ms * pj[j][1], mcs[2] - ms * pj[j][2]};
          gtau[j] = -(zj[j][0] * (arm[1] * gb[2] - arm[2] * gb[1]) + zj[j][1] * (arm[2] * gb[0] - arm[0] * gb[2]) +
                      zj[j][2] * (arm[0] * gb[1] - arm[1] * gb[0]));
        }
      }
    }

    // ---------------- the leg's block of the wrench map in contact coordinates: A_k = [E'; (r x e_c)] (6 x 3)
    creal (&At)[3][6] = L.At;  // At[c] = column of slot c (0 = normal, 1, 2 = tangents)
    const creal footc[3] = {(creal)foot[0], (creal)foot[1], (creal)foot[2]};
    // (a swing leg: zero force rows; its torque rows r x 0 vanish without a second select unless the foot position is
    // not finite, which the joint-angle check above has already turned into status BAD_INPUT)
#pragma unroll
    for (int c = 0; c < 3; c++) {
      At[c][0] = alive ? E[c][0] : creal(0.0);
      At[c][1] = alive ? E[c][1] : creal(0.0);
      At[c][2] = alive ? E[c][2] : creal(0.0);
      At[c][3] = footc[1] * At[c][2] - footc[2] * At[c][1];
      At[c][4] = footc[2] * At[c][0] - footc[0] * At[c][2];
      At[c][5] = footc[0] * At[c][1] - footc[1] * At[c][0];
    }
    // Jacobian and gravity torques are only needed again for the outputs: park them in shared memory
#pragma unroll
    for (int j = 0; j < 3; j++) {
#pragma unroll
      for (int c = 0; c < 3; c++) jgp[(3 * j + c) * jgs] = J[j][c];
      jgp[(9 + j) * jgs] = gtau[j];
    }
#pragma unroll
    for (int c = 0; c < 3; c++) { L.nrm[c] = E[0][c]; L.foot[c] = footc[c]; }
    L.c0 = fmax(fmax(creal(2.0) * (creal)prm.fmin, (L.b[0] * E[0][0] + L.b[1] * E[0][1] + L.b[2] * E[0][2]) * (ns > 0 ? creal(1.0) / ns : creal(0.0))),
                           (creal)prm.fmin + creal(1.0));
    L.rm = ns > 0 ? 1.f / (5.f * ns) : 0.f;

}

// The solver core may run in a wider type than the inputs / kinematics (FP32 interface, FP64 core).
template <typename real, typename creal>
__device__ __forceinline__ void widen_setup(const LegSetup<real>& s, LegSetup<creal>& d) {
#pragma unroll
  for (int c = 0; c < 3; c++) {
#pragma unroll
    for (int r = 0; r < 6; r++) d.At[c][r] = (creal)s.At[c][r];
    d.nrm[c] = (creal)s.nrm[c];
    d.foot[c] = (creal)s.foot[c];
  }
#pragma unroll
  for (int r = 0; r < 6; r++) d.b[r] = (creal)s.b[r];
  d.mu = (creal)s.mu; d.c0 = (creal)s.c0;
  d.rm = s.rm; d.mask = s.mask; d.ns = s.ns; d.alive = s.alive; d.qbad = s.qbad; d.qinf = s.qinf;
}

// value number `leg` of four, as two levels of selects (no divergent branches)
template <typename T>
__device__ __forceinline__ T sel4(const int leg, const T v0, const T v1, const T v2, const T v3) {
  const T lo = (leg & 1) ? v1 : v0, hi = (leg & 1) ? v3 : v2;
  return (leg & 2) ? hi : lo;
}

// Forces in base frame, joint torques, net wrench, flags word of one finished state.
template <typename real, typename creal, typename jreal>
__device__ __forceinline__ void quad_output(const SolveArgsT<real>& a, const LegSetup<creal>& L, creal (&y)[3], const int a0, const int sg1,
                                            const int sg2, const int status, const int it, const unsigned long long bq,
                                            const bool valid, const int leg, const jreal* const jgp, const int jgs,
                                            const creal* net_pre = nullptr) {
  const unsigned long long B = a.B;
  const bool alive = L.alive;
  const unsigned mask = L.mask;
  const creal (&At)[3][6] = L.At;
    // ---------------- outputs: forces in base frame, torques, net wrench, flags
    const bool solved = (status == 0 || status == 2 || status == 3);
    const bool live = alive && solved;
    creal f[3];
#pragma unroll
    for (int c = 0; c < 3; c++) f[c] = live ? y[0] * At[0][c] + y[1] * At[1][c] + y[2] * At[2][c] : creal(0.0);
    if (valid) {
#pragma unroll
      for (int c = 0; c < 3; c++) a.grf[(size_t)(3 * leg + c) * B + bq] = (real)f[c];
      // (the Jacobian slot is read by every lane - it is a valid address whatever the state - and the select comes
      // last: no divergent branch around the loads)
#pragma unroll
      for (int j = 0; j < 3; j++) {
        const creal tq = (creal)jgp[(9 + j) * jgs] - ((creal)jgp[(3 * j) * jgs] * f[0] + (creal)jgp[(3 * j + 1) * jgs] * f[1] + (creal)jgp[(3 * j + 2) * jgs] * f[2]);
        a.tau[(size_t)(3 * leg + j) * B + bq] = (real)(live ? tq : creal(0.0));
      }
    }
    if (a.netwrench) {
      // A x = sum over legs of A_k y_k (CFD.cpp:614-625)
      // (or, when the caller has the solution t of the 6x6 system: A x = b - S^-1 t, no reduction needed)
      // leg k writes components k and k+4 (k < 2)
      creal nk, n4;
      if (net_pre != nullptr) {
        nk = solved ? sel4(leg, net_pre[0], net_pre[1], net_pre[2], net_pre[3]) : creal(0.0);
        n4 = solved ? ((leg & 1) ? net_pre[5] : net_pre[4]) : creal(0.0);
      } else {
        // a reduce-scatter is enough: the lanes of even legs sum components 0, 2, 4 (exchanged across xor 1), those
        // of odd legs 1, 3, 5, then a butterfly across xor 2 - (x0 + x1) + (x2 + x3), as quad_sum, with 6 values
        // crossing lanes instead of 12
        const bool odd = (leg & 1) != 0;
        creal h[3];
#pragma unroll
        for (int i = 0; i < 3; i++) {
          const creal ce = live ? At[0][2 * i] * y[0] + At[1][2 * i] * y[1] + At[2][2 * i] * y[2] : creal(0.0);
          const creal co = live ? At[0][2 * i + 1] * y[0] + At[1][2 * i + 1] * y[1] + At[2][2 * i + 1] * y[2] : creal(0.0);
          h[i] = (odd ? co : ce) + __shfl_xor_sync(kFull, odd ? ce : co, 1);
        }
#pragma unroll
        for (int i = 0; i < 3; i++) h[i] += __shfl_xor_sync(kFull, h[i], 2);
        nk = (leg & 2) ? h[1] : h[0];
        n4 = h[2];
      }
      if (valid) {
        a.netwrench[(size_t)leg * B + bq] = (real)nk;
        if (leg < 2) a.netwrench[(size_t)(4 + leg) * B + bq] = (real)n4;
      }
    }
    {
      unsigned bits = 0u;
      if (live) {
        bits = (a0 != 0 ? 1u : 0u) | (sg1 == -1 ? 2u : 0u) | (sg1 == 1 ? 4u : 0u) | (sg2 == -1 ? 8u : 0u) | (sg2 == 1 ? 16u : 0u);
        bits <<= (4 + 5 * leg);
      }
      bits = quad_or(bits);
      if (valid && leg == 0) {
        const unsigned itc = it > 31 ? 31u : (unsigned)it;
        a.flags[bq] = mask | bits | ((unsigned)status << 24) | (itc << 27);
      }
    }
}

// The unconstrained minimiser of one state (all rows free) and its first repair: which rows does it violate?
// Whole warp (quad shuffles).  Out: y (contact coordinates), t (solution of the 6x6 system; A x = b - S^-1 t),
// status (0 ok / 1 no stance / 4 bad), hard (some row is violated: the state needs active-set rounds),
// pat (first pattern: every violated row active, 5 bits per leg, OR-ed over the quad).
// (The friction frames are orthonormal to the rounding of creal - quad_setup builds them in creal - which the short
// form of the system below relies on.)
template <typename real, typename creal>
__device__ __forceinline__ void quad_first_solve(const LegSetup<creal>& L, const creal* sinv, const creal winv, const creal cfmin,
                                                 const int leg, creal (&y)[3], creal (&t)[6], int& status, bool& hard,
                                                 unsigned& pat_out) {
  const bool alive = L.alive;
  const creal (&At)[3][6] = L.At;
  status = L.qbad ? 4 : (L.ns == 0 ? 1 : (L.qinf ? 5 : 0));
  y[0] = y[1] = y[2] = creal(0.0);
  hard = false;
  // unconstrained minimiser through the 6x6 system: (S^-1 + A~ A~'/w) t = b,  y = A~' t / w
  const creal al = alive ? winv : creal(0.0);
  bool pd;
  if (Tol<creal>::refine) {
    // FP32 core: generic assembly + iterative refinement through the factors.
    creal N[21], rdg[6];
#pragma unroll
    for (int i = 0; i < 6; i++) {
      const creal w0 = al * At[0][i], w1 = al * At[1][i], w2 = al * At[2][i];
#pragma unroll
      for (int j = 0; j < 6; j++) {
        if (j <= i) {
          creal acc = (i == j && leg == 0) ? sinv[i] : creal(0.0);
          acc = fma(w0, At[0][j], acc);
          acc = fma(w1, At[1][j], acc);
          acc = fma(w2, At[2][j], acc);
          N[QLB_TRI(i, j)] = quad_sum(acc);
        }
      }
      t[i] = L.b[i];
    }
    pd = chol6_thread(N, rdg);
    solve6_thread(N, rdg, t);
    if (Tol<creal>::refine) {
      const creal al3[3] = {al, al, al};
      refine6(N, rdg, At, al3, sinv, L.b, t);
    }
  } else {
    // With every slot free the friction frames drop out (Q Q' = I):  A~ A~' = sum_k [I; X_k][I, X_k'],
    // X_k = [r_k]x, so the system is  [[D, B'], [B, C]]  with D = S_F^-1 + ns/w diagonal, B = [sum r]x / w and
    // C = S_T^-1 + sum(|r|^2 I - r r') / w: nine sums over the quad instead of twenty-one, and a 3x3 Schur
    // complement  (C - B D^-1 B') t_T = b_T - B D^-1 b_F  instead of a 6x6 factorisation.
    const creal rx = alive ? L.foot[0] : creal(0.0), ry = alive ? L.foot[1] : creal(0.0), rz = alive ? L.foot[2] : creal(0.0);
    const creal xs = winv * quad_sum(rx), ys = winv * quad_sum(ry), zs = winv * quad_sum(rz);
    const creal qxx = quad_sum(rx * rx), qyy = quad_sum(ry * ry), qzz = quad_sum(rz * rz);
    const creal qxy = quad_sum(rx * ry), qxz = quad_sum(rx * rz), qyz = quad_sum(ry * rz);
    const creal nsw = (creal)L.ns * winv;
    const creal d0 = full_rcp(sinv[0] + nsw), d1 = full_rcp(sinv[1] + nsw), d2 = full_rcp(sinv[2] + nsw);  // full precision: the Schur complement cancels
    // Schur complement, packed lower 3x3
    creal c00 = fma(winv, qyy + qzz, sinv[3]) - (zs * zs * d1 + ys * ys * d2);
    creal c11 = fma(winv, qxx + qzz, sinv[4]) - (zs * zs * d0 + xs * xs * d2);
    creal c22 = fma(winv, qxx + qyy, sinv[5]) - (ys * ys * d0 + xs * xs * d1);
    creal c10 = fma(-winv, qxy, xs * ys * d2);
    creal c20 = fma(-winv, qxz, xs * zs * d1);
    creal c21 = fma(-winv, qyz, ys * zs * d0);
    const creal u0 = d0 * L.b[0], u1 = d1 * L.b[1], u2 = d2 * L.b[2];
    creal g0 = L.b[3] - (ys * u2 - zs * u1);
    creal g1 = L.b[4] - (zs * u0 - xs * u2);
    creal g2 = L.b[5] - (xs * u1 - ys * u0);
    // 3x3 Cholesky and the two substitutions
    pd = c00 > creal(0.0);
    const creal r0 = fast_rsqrt(c00);
    c10 *= r0; c20 *= r0;
    c11 = fma(-c10, c10, c11);
    pd = pd && (c11 > creal(0.0));
    const creal r1 = fast_rsqrt(c11);
    c21 = fma(-c20, c10, c21) * r1;
    c22 = fma(-c21, c21, fma(-c20, c20, c22));
    pd = pd && (c22 > creal(0.0));
    const creal r2 = fast_rsqrt(c22);
    g0 *= r0;
    g1 = fma(-c10, g0, g1) * r1;
    g2 = fma(-c21, g1, fma(-c20, g0, g2)) * r2;
    g2 *= r2;
    g1 = fma(-c21, g2, g1) * r1;
    g0 = fma(-c20, g2, fma(-c10, g1, g0)) * r0;
    t[3] = g0; t[4] = g1; t[5] = g2;
    // t_F = D^-1 (b_F - B' t_T),  B' v = -(s x v) / w ... written out
    t[0] = d0 * (L.b[0] - (zs * g1 - ys * g2));
    t[1] = d1 * (L.b[1] - (xs * g2 - zs * g0));
    t[2] = d2 * (L.b[2] - (ys * g0 - xs * g1));
  }
  const bool pd_fail = !pd && status == 0;   // quad-uniform: every lane factors the same matrix
  if (pd_fail && !Tol<creal>::rescue) status = 4;
  creal e[5];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    creal d = creal(0.0);
#pragma unroll
    for (int r = 0; r < 6; r++) d = fma(At[c][r], t[r], d);
    y[c] = al * d;
  }
  leg_rows(y[0], y[1], y[2], L.mu, e);
  e[0] -= cfmin;
  const creal tol_s = Tol<creal>::feas() * quad_max_abs(y[0], y[1], y[2]);
  bool viol = false;
#pragma unroll
  for (int r = 0; r < 5; r++) viol = viol || (alive && e[r] < -tol_s);
  const bool quad_viol = quad_or(viol ? 1u : 0u) != 0u;  // not inside the && : every lane must reach the shuffle
  hard = (status == 0) && (quad_viol || pd_fail);
  // first repair of the empty pattern: every violated row becomes active (the more violated one of a +- pair)
  unsigned pat = 0u;
  if (alive && !pd_fail) {
    const bool v0 = e[0] < -tol_s, v1 = e[1] < -tol_s, v2 = e[2] < -tol_s, v3 = e[3] < -tol_s, v4 = e[4] < -tol_s;
    pat = v0 ? 1u : 0u;
    if (v1 || v2) pat |= ((v1 && (!v2 || e[1] <= e[2])) ? 1u : 2u) << 1;
    if (v3 || v4) pat |= ((v3 && (!v4 || e[3] <= e[4])) ? 1u : 2u) << 3;
  }
  pat_out = quad_or(pat << (5 * leg));
}

// First pass: kinematics + QP data + the unconstrained minimiser (polish round with the empty pattern).
// States whose unconstrained minimiser is feasible (most of them) are finished here; the others are
// appended to a.list for the second pass.  Fixed trip count: no divergence between the eight states of a warp.
template <typename real, typename creal, int MODE>
__global__ void __launch_bounds__(kQuadThreads, QLB_FIRST_MIN_CTAS) qlb_quad_first_kernel(const SolveArgsT<real> a) {
  __shared__ DeviceParamsT<real> prm;
  __shared__ creal sinv[6], cS[6];
  __shared__ creal winv, cW, cfmin;
  __shared__ real jg[12][kQuadThreads];  // per thread: Jacobian (9) and gravity torques (3) of its leg
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.params);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&prm);
    for (int i = threadIdx.x; i < (int)(sizeof(DeviceParamsT<real>) / 4); i += blockDim.x) dst[i] = src[i];
    // the solver core reads its weights from the FP64 parameter block, in its own type
    if (threadIdx.x < 6) { cS[threadIdx.x] = (creal)a.params64->S[threadIdx.x]; sinv[threadIdx.x] = (creal)(1.0 / a.params64->S[threadIdx.x]); }
    if (threadIdx.x == 6) { cW = (creal)a.params64->W; winv = (creal)(1.0 / a.params64->W); cfmin = (creal)a.params64->fmin; }
    load_model_to_smem(a.model);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int leg = lane & 3, quad = lane >> 2;
  const unsigned long long B = a.B;
  const unsigned long long nbatch = (B + 7) / 8;

  // Software pipeline over the work items of this warp: the next item is claimed and its loads are issued
  // before the outputs of the current one are written, so the input latency is hidden behind the stores
  // (the FP64 kernel runs only twelve warps per SM).  QLB_PIPELINE_LOADS=0: prefetch instructions only.
  unsigned long long bi = 0;
  if (lane == 0) bi = atomicAdd(a.counter, 1ull);
  bi = __shfl_sync(kFull, bi, 0);
  RawIn<real, MODE> in;
  if (bi < nbatch) {
    const unsigned long long s0 = bi * 8 + quad;
    quad_load<real, MODE>(a, prm.mu_default, s0 < B ? s0 : (B - 1), s0 < B, leg, in);
  }
  while (bi < nbatch) {
    unsigned long long bn = 0;
    if (lane == 0) bn = atomicAdd(a.counter, 1ull);
    bn = __shfl_sync(kFull, bn, 0);
    const unsigned long long sn = bn * 8 + quad;
    const unsigned long long bqn = sn < B ? sn : (B - 1);
    if (bn < nbatch) quad_prefetch<real, MODE>(a, bqn, leg);
    const unsigned long long slot = bi * 8 + quad;
    const bool valid = slot < B;
    const unsigned long long bq = valid ? slot : (B - 1);
    LegSetup<creal> L;
    quad_setup<real, MODE, creal>(a, prm, in, bq, valid, true, leg, L, &jg[0][threadIdx.x], kQuadThreads);
    int status;
    creal y[3], t[6];
    bool hard;
    unsigned pat;
    quad_first_solve<real, creal>(L, sinv, winv, cfmin, leg, y, t, status, hard, pat);
    // append the unfinished states to the list of the second pass (one atomic per warp).  The atomic is issued
    // here and its result consumed after the outputs are written, so its round trip to L2 is not waited for.
    const unsigned hm = __ballot_sync(kFull, hard && valid && leg == 0);
    unsigned base = 0;
    if (hm != 0u && lane == 0) base = atomicAdd(a.list_count, __popc(hm));
    // Every state is written, the listed ones provisionally (a later pass overwrites them): a row segment
    // with holes would be a partial-sector write, which costs a DRAM read to fill (ncu: +250 MB per 2^20 states).
#if QLB_PIPELINE_LOADS
    if (bn < nbatch) quad_load<real, MODE>(a, prm.mu_default, bqn, sn < B, leg, in);
#endif
    creal net[6];
#pragma unroll
    for (int r = 0; r < 6; r++) net[r] = fma(-sinv[r], t[r], L.b[r]);   // A x = b - S^-1 t
    quad_output<real, creal, real>(a, L, y, 0, 0, 0, status, 0, bq, valid, leg, &jg[0][threadIdx.x], kQuadThreads, net);  // whole warp: it contains quad shuffles
#if !QLB_PIPELINE_LOADS
    if (bn < nbatch) quad_load<real, MODE>(a, prm.mu_default, bqn, sn < B, leg, in);
#endif
    if (hm != 0u) {
      base = __shfl_sync(kFull, base, 0);
      if (hard && valid && leg == 0) {
        const unsigned at = base + __popc(hm & ((1u << lane) - 1u));
        a.list[at] = (unsigned)bq;
        a.list_pat[at] = pat;
      }
    }
    bi = bn;
  }
}

// Shared constants of the solver core, in the core's arithmetic type.
template <typename creal>
struct CoreConst {
  creal sinv[6], S[6];
  creal winv, W, fmin;
  float tol;
  int max_iter;
  // filled by the first threads of the CTA from the FP64 parameter block (followed by __syncthreads)
  __device__ void load(const DeviceParamsT<double>* p) {
    if (threadIdx.x < 6) { S[threadIdx.x] = (creal)p->S[threadIdx.x]; sinv[threadIdx.x] = (creal)(1.0 / p->S[threadIdx.x]); }
    if (threadIdx.x == 6) {
      W = (creal)p->W; winv = (creal)(1.0 / p->W); fmin = (creal)p->fmin;
      tol = (float)p->tol; max_iter = p->max_iter;
    }
  }
};

// The QP of one state, one leg per lane (whole warp: eight states side by side).
//   STAGE 0: the full algorithm - active-set rounds from the unconstrained minimiser, then the interior
//            point, each candidate pattern verified by an exact polish round;
//   STAGE 1: active-set rounds only, starting from the pattern pat0 of this leg; `defer` is set when they do not verify (and, with DEFER_FAIL, when a
//            factorisation fails): the state goes to the interior-point pass;
//   STAGE 2: interior point from the strictly feasible start, then polish rounds.
// enable = false: the quad idles (used when only some states of a warp are solved again).
// Out: y = forces in contact coordinates, pattern (a0, sg1, sg2), status, interior-point iterations.
template <typename creal, int STAGE, bool DEFER_FAIL>
__device__ __forceinline__ void quad_solve(const LegSetup<creal>& L, const CoreConst<creal>& cc, const int leg, const int quad,
                                           const bool enable, const unsigned pat0, creal (&y)[3], int& a0, int& sg1, int& sg2,
                                           int& status, int& it, bool& defer) {
  const bool alive = L.alive;
  const int ns = L.ns;
  const creal mu = L.mu, c0 = L.c0;
  const float rm = L.rm;
  const bool qbad = L.qbad;
  const creal (&At)[3][6] = L.At;
  const creal (&b)[6] = L.b;

  // ---------------- solver state of this leg
  y[0] = y[1] = y[2] = creal(0.0);   // (y_n, y_1, y_2)
  creal rdl[3] = {creal(0.0), creal(0.0), creal(0.0)}; // dual residual of the three slots
  creal s[5], lam[5], rp[5];
#pragma unroll
  for (int r = 0; r < 5; r++) { s[r] = creal(1.0); lam[r] = creal(0.0); rp[r] = creal(0.0); }
  a0 = 0; sg1 = 0; sg2 = 0;    // pattern: y_n pinned at F_min; y_1 = sg1 mu y_n; y_2 = sg2 mu y_n
  int mode = kModePolish, pass = 0;
  it = 0; status = 0;
  bool first = true, converged = false, want_polish = false;
  float gap_shrink = 1.f;  // a converged iterate whose pattern does not verify: iterate on to a smaller gap
  creal alpha_prev = creal(1.0);
  defer = false;  // STAGE 1: hand the state to the interior-point pass
  bool need_start = false;  // set when this quad begins its interior-point iteration
  if (!enable) { mode = kModeDone; }
  else if (qbad) { mode = kModeDone; status = 4; }
  else if (ns == 0) { mode = kModeDone; status = 1; }
  else if (L.qinf) { mode = kModeDone; status = 5; }
  else if (STAGE == 2) { mode = kModeIpm; first = false; need_start = true; }
  else if (STAGE == 1) {
    // the first pass already repaired the empty pattern once: start from its result (bit 0: y_n pinned;
    // bits 1-2 / 3-4: tangent tied to -mu y_n (1) or +mu y_n (2))
    a0 = (int)(pat0 & 1u);
    sg1 = ((pat0 >> 1) & 3u) == 1u ? -1 : (((pat0 >> 1) & 3u) == 2u ? 1 : 0);
    sg2 = ((pat0 >> 3) & 3u) == 1u ? -1 : (((pat0 >> 3) & 3u) == 2u ? 1 : 0);
    pass = 1;
  }

  int rounds = 0;
#pragma unroll 1
  for (;;) {
    if (__all_sync(kFull, mode == kModeDone)) break;
    if (++rounds > 200 && mode != kModeDone) { mode = kModeDone; status = 2; }
    // ---- a quad starts its interior-point iteration: strictly feasible start, centred multipliers
    if (STAGE != 1 && __any_sync(kFull, need_start)) {
      const creal y0 = alive ? c0 : creal(0.0);
      creal t0[6];
#pragma unroll
      for (int r = 0; r < 6; r++) t0[r] = cc.S[r] * (b[r] - quad_sum(At[0][r] * y0));  // S (b - A~ y0)
      creal g[3];
      float gm = 0.f;
#pragma unroll
      for (int c = 0; c < 3; c++) {
        creal d = (c == 0) ? cc.W * y0 : creal(0.0);
#pragma unroll
        for (int r = 0; r < 6; r++) d = fma(-At[c][r], t0[r], d);
        g[c] = d;
        gm = fmaxf(gm, fabsf((float)d));
      }
      const creal gmax = (creal)fmaxf(1.f, quad_max(gm));
      if (need_start) {
        need_start = false;
        creal e0[5], dt[3];
        leg_rows(c0, creal(0.0), creal(0.0), mu, e0);
        e0[0] -= cc.fmin;
#pragma unroll
        for (int r = 0; r < 5; r++) {
          const creal sr = fmax(e0[r], creal(1e-3) * c0);
          s[r] = alive ? sr : creal(1.0);
          lam[r] = alive ? gmax * fast_rcp(sr) : creal(0.0);
          rp[r] = alive ? sr - e0[r] : creal(0.0);
        }
        leg_rows_t(lam, mu, dt);
        y[0] = y0; y[1] = creal(0.0); y[2] = creal(0.0);
#pragma unroll
        for (int c = 0; c < 3; c++) rdl[c] = alive ? g[c] - dt[c] : creal(0.0);
      }
    }
    const bool pol_round = (mode == kModePolish), ipm_round = (STAGE != 1) && (mode == kModeIpm);  // STAGE 1 never iterates: keeps that code out of its kernel
    const bool any_ipm = __any_sync(kFull, ipm_round);
    const bool any_pol = __any_sync(kFull, pol_round);

    // ---- build: three vectors v_c and weights al_c with  A_k K_k^-1 A_k' = sum_c al_c v_c v_c'
    creal v[3][6], al[3] = {creal(0.0), creal(0.0), creal(0.0)}, r6[6];
    creal rs[5], th[5], e1 = creal(0.0), e2 = creal(0.0), rr[3] = {creal(0.0), creal(0.0), creal(0.0)};
#pragma unroll
    for (int r = 0; r < 5; r++) { rs[r] = creal(1.0); th[r] = creal(0.0); }
#pragma unroll
    for (int r = 0; r < 6; r++) { v[0][r] = creal(0.0); v[1][r] = creal(0.0); v[2][r] = creal(0.0); r6[r] = creal(0.0); }
    if (pol_round) {
      // reduced columns of the equality-constrained QP for the current pattern
      const creal q1 = sg1 * mu, q2 = sg2 * mu;
      const bool fn = alive && a0 == 0, f1 = alive && sg1 == 0, f2 = alive && sg2 == 0;
      const creal wn = cc.W * fma(mu * mu, (creal)(sg1 * sg1 + sg2 * sg2), creal(1.0));
      al[0] = fn ? fast_rcp(wn) : creal(0.0);
      al[1] = f1 ? cc.winv : creal(0.0);
      al[2] = f2 ? cc.winv : creal(0.0);
      const creal pin = (alive && a0 != 0) ? cc.fmin : creal(0.0);
#pragma unroll
      for (int r = 0; r < 6; r++) {
        const creal cn = fma(q2, At[2][r], fma(q1, At[1][r], At[0][r]));
        v[0][r] = fn ? cn : creal(0.0);
        v[1][r] = f1 ? At[1][r] : creal(0.0);
        v[2][r] = f2 ? At[2][r] : creal(0.0);
        r6[r] = ((leg == 0) ? b[r] : creal(0.0)) - pin * cn;
      }
    } else if (ipm_round) {
      // K = w I + D~' diag(lam/s) D~ is an arrow matrix; K^-1 = M' diag(al) M with M = [[1,0,0],[0,1,0],[-e1,-e2,1]]
      // (slots ordered 1, 2, n), so v = (a_1, a_2, a_n - e1 a_1 - e2 a_2), al = (1/d1, 1/d2, 1/sigma)
      creal vv[5];
#pragma unroll
      for (int r = 0; r < 5; r++) { rs[r] = fast_rcp(s[r]); th[r] = lam[r] * rs[r]; vv[r] = fma(-th[r], rp[r], lam[r]); }
      const creal T1 = th[1] + th[2], T2 = th[3] + th[4];
      const creal b1 = mu * (th[1] - th[2]), b2 = mu * (th[3] - th[4]);
      const creal d1 = cc.W + T1, d2 = cc.W + T2;
      al[1] = fast_rcp(d1); al[2] = fast_rcp(d2);
      e1 = b1 * al[1]; e2 = b2 * al[2];
      // Schur complement of the arrow matrix, sigma = w + th0 + mu^2 (T1 + T2) - b1 e1 - b2 e2, written without
      // the cancellation: mu^2 T - b^2 / d = mu^2 (T w + 4 th+ th-) / d  (all terms positive)
      const creal sc1 = fma(T1, cc.W, creal(4.0) * th[1] * th[2]) * al[1];
      const creal sc2 = fma(T2, cc.W, creal(4.0) * th[3] * th[4]) * al[2];
      al[0] = fast_rcp(cc.W + fma(mu * mu, sc1 + sc2, th[0]));
      creal dt[3];
      leg_rows_t(vv, mu, dt);
#pragma unroll
      for (int c = 0; c < 3; c++) rr[c] = alive ? -rdl[c] - dt[c] : creal(0.0);
      const creal m0 = rr[0] - e1 * rr[1] - e2 * rr[2];
#pragma unroll
      for (int r = 0; r < 6; r++) {
        v[1][r] = At[1][r];
        v[2][r] = At[2][r];
        v[0][r] = At[0][r] - e1 * At[1][r] - e2 * At[2][r];
        r6[r] = al[0] * m0 * v[0][r] + al[1] * rr[1] * v[1][r] + al[2] * rr[2] * v[2][r];
      }
    }

    // ---- this leg's contribution to the 6x6 system, summed over the quad
    creal N[21], rdg[6];
#pragma unroll
    for (int i = 0; i < 6; i++) {
      const creal w0 = al[0] * v[0][i], w1 = al[1] * v[1][i], w2 = al[2] * v[2][i];
#pragma unroll
      for (int j = 0; j < 6; j++) {
        if (j <= i) {
          creal acc = (i == j && leg == 0) ? cc.sinv[i] : creal(0.0);
          acc = fma(w0, v[0][j], acc);
          acc = fma(w1, v[1][j], acc);
          acc = fma(w2, v[2][j], acc);
          N[QLB_TRI(i, j)] = quad_sum(acc);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 6; r++) r6[r] = quad_sum(r6[r]);
    const bool pd = chol6_thread(N, rdg);
    if (Tol<creal>::refine && any_pol) {
      creal rhs6[6];
#pragma unroll
      for (int r = 0; r < 6; r++) rhs6[r] = r6[r];
      solve6_thread(N, rdg, r6);  // r6 <- t
      refine6(N, rdg, v, al, cc.sinv, rhs6, r6);
    } else {
      solve6_thread(N, rdg, r6);  // r6 <- t
    }
    if (!pd && mode != kModeDone) {
      mode = kModeDone; y[0] = y[1] = y[2] = creal(0.0);
      if (DEFER_FAIL && STAGE == 1) defer = true; else status = 4;
    }

    // ---- polish: recover y, gradient, multipliers, slacks; verify; repair the pattern
    if (any_pol) {
      creal zt[3], att[3];
#pragma unroll
      for (int c = 0; c < 3; c++) {
        creal d0 = creal(0.0), d1 = creal(0.0);
#pragma unroll
        for (int r = 0; r < 6; r++) { d0 = fma(v[c][r], r6[r], d0); d1 = fma(At[c][r], r6[r], d1); }
        zt[c] = al[c] * d0;
        att[c] = d1;
      }
      const creal yn = (a0 != 0) ? cc.fmin : zt[0];
      creal yp[3];
      yp[0] = alive ? yn : creal(0.0);
      yp[1] = alive ? ((sg1 != 0) ? sg1 * mu * yn : zt[1]) : creal(0.0);
      yp[2] = alive ? ((sg2 != 0) ? sg2 * mu * yn : zt[2]) : creal(0.0);
      // gradient G~ y + g~ = w y - A_k' t,  t = S (b - A~ y)
      const creal g0 = fma(cc.W, yp[0], -att[0]), g1 = fma(cc.W, yp[1], -att[1]), g2 = fma(cc.W, yp[2], -att[2]);
      creal e[5], u[5];
      leg_rows(yp[0], yp[1], yp[2], mu, e);
      e[0] -= cc.fmin;
      u[1] = (sg1 == -1) ? g1 : creal(0.0);
      u[2] = (sg1 == 1) ? -g1 : creal(0.0);
      u[3] = (sg2 == -1) ? g2 : creal(0.0);
      u[4] = (sg2 == 1) ? -g2 : creal(0.0);
      u[0] = (a0 != 0) ? g0 - mu * ((u[1] + u[2]) + (u[3] + u[4])) : creal(0.0);
      const bool act[5] = {a0 != 0, sg1 == -1, sg1 == 1, sg2 == -1, sg2 == 1};
      const creal tol_s = Tol<creal>::feas() * quad_max_abs(yp[0], yp[1], yp[2]);
      const creal tol_u = Tol<creal>::mult() * quad_max_abs(att[0], att[1], att[2], cc.W * lane_max_abs(yp[0], yp[1], yp[2]));
      // violations of this leg: negative multipliers (drop), else negative slacks (add; one per tangent pair)
      creal wd_v = -tol_u, wp_v = -tol_s;
      int wd_r = -1, wp_r = -1, nviol = 0;
      bool drop[5], add[5];
#pragma unroll
      for (int r = 0; r < 5; r++) {
        drop[r] = alive && pol_round && act[r] && u[r] < -tol_u;
        add[r] = alive && pol_round && !act[r] && e[r] < -tol_s;
        if (drop[r] && u[r] < wd_v) { wd_v = u[r]; wd_r = r; }
        if (add[r] && e[r] < wp_v) { wp_v = e[r]; wp_r = r; }
        nviol += (drop[r] || add[r]) ? 1 : 0;
      }
      const bool leg_viol = nviol > 0;
      const bool any_viol = quad_or(leg_viol ? 1u : 0u) != 0u;
      const float keyf = (wd_r >= 0) ? (float)(wd_v * creal(1e6)) : ((wp_r >= 0) ? (float)wp_v : 0.f);
      const float best = quad_min(keyf);
      const unsigned tie = (__ballot_sync(kFull, leg_viol && keyf == best) >> (4 * quad)) & 0xFu;
      if (pol_round && mode == kModePolish) {
        if (!any_viol) {
          y[0] = yp[0]; y[1] = yp[1]; y[2] = yp[2];
          mode = kModeDone;
          if (status == 2) status = 0;
        } else {
          pass++;
          const bool give_up = first ? (pass > QLB_PDAS_ROUNDS) : (pass >= kPolishPasses);
          if (!give_up) {
            if (pass <= 2) {
              // every violated row of every leg moves
              if (drop[0]) a0 = 0; else if (add[0]) a0 = 1;
              if (drop[1] || drop[2]) sg1 = 0; else if (add[1] || add[2]) sg1 = (add[1] && (!add[2] || e[1] <= e[2])) ? -1 : 1;
              if (drop[3] || drop[4]) sg2 = 0; else if (add[3] || add[4]) sg2 = (add[3] && (!add[4] || e[3] <= e[4])) ? -1 : 1;
            } else if (leg_viol && tie != 0u && (__ffs(tie) - 1) == leg) {
              // only the globally worst row moves (prevents cycling)
              if (wd_r >= 0) {
                if (wd_r == 0) a0 = 0; else if (wd_r <= 2) sg1 = 0; else sg2 = 0;
              } else {
                if (wp_r == 0) a0 = 1; else if (wp_r == 1) sg1 = -1; else if (wp_r == 2) sg1 = 1; else if (wp_r == 3) sg2 = -1; else sg2 = 1;
              }
            }
          } else if (first) {
            first = false;
            a0 = 0; sg1 = 0; sg2 = 0;
            if (STAGE == 1) { defer = true; mode = kModeDone; }  // the interior-point pass takes over
            else { mode = kModeIpm; need_start = true; }
          } else if (converged && status == 0 && !Tol<creal>::rescue && gap_shrink > 1e-5f) {
            // The rows with lambda > s were not the active set although the gap is at tolerance (a multiplier
            // below sqrt(gap)): two more decades of the interior point separate them.  Rare (1 in 10^5).
            gap_shrink *= 1e-2f;
            converged = false;
            mode = kModeIpm;
          } else if (converged || status == 2) {
            mode = kModeDone;
            if (status == 0) status = 3;
          } else {
            mode = kModeIpm;
          }
        }
      }
    }

    // ---- interior point: predictor direction, centring, corrector, step
    if (STAGE != 1 && any_ipm) {
      creal ds[5], dl[5], de[5], rc[5], x[3];
      float ratio = 0.f, pa = 0.f;
      {
        // x = K^-1 (r - A_k' t)
        creal g[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
          creal d = rr[c];
#pragma unroll
          for (int r = 0; r < 6; r++) d = fma(-At[c][r], r6[r], d);
          g[c] = d;
        }
        const creal hn = al[0] * (g[0] - e1 * g[1] - e2 * g[2]);
        x[0] = hn; x[1] = fma(-e1, hn, al[1] * g[1]); x[2] = fma(-e2, hn, al[2] * g[2]);
      }
      leg_rows(x[0], x[1], x[2], mu, de);
#pragma unroll
      for (int r = 0; r < 5; r++) {
        de[r] = (alive && ipm_round) ? de[r] : creal(0.0);
        ds[r] = de[r] - rp[r];
        dl[r] = (alive && ipm_round) ? -fma(lam[r], ds[r], s[r] * lam[r]) * rs[r] : creal(0.0);
        if (alive && ipm_round) ratio = fmaxf(ratio, fmaxf(-(float)ds[r] * (float)rs[r], -(float)dl[r] * rcp_approx((float)lam[r])));
        pa += (float)(s[r] * lam[r]);
      }
      ratio = quad_max(ratio);
      const float mu_c = quad_sum(ipm_round ? pa : 0.f) * rm;
      const creal ala = (ratio > 1.f) ? creal(1.0) / (creal)ratio : creal(1.0);
      float pb = 0.f;
#pragma unroll
      for (int r = 0; r < 5; r++) pb += (float)(fma(ala, ds[r], s[r]) * fma(ala, dl[r], lam[r]));
      const float mua = quad_sum(ipm_round ? pb : 0.f) * rm;
      const float q3 = (ipm_round && mu_c > 0.f) ? mua / mu_c : 0.f;
      float sigma = q3 * q3 * q3;
      if (alpha_prev < creal(0.1) && sigma < 0.5f) sigma = 0.5f;
      const creal sigmu = (creal)sigma * (creal)mu_c;
      creal vv[5], dt[3], r2[3];
#pragma unroll
      for (int r = 0; r < 5; r++) {
        rc[r] = (alive && ipm_round) ? fma(ds[r], dl[r], s[r] * lam[r]) - sigmu : creal(0.0);
        vv[r] = (rc[r] - lam[r] * rp[r]) * rs[r];
      }
      leg_rows_t(vv, mu, dt);
#pragma unroll
      for (int c = 0; c < 3; c++) r2[c] = (alive && ipm_round) ? -rdl[c] - dt[c] : creal(0.0);
      // corrector: same matrix, new right-hand side
      creal t2[6];
      {
        const creal m0 = r2[0] - e1 * r2[1] - e2 * r2[2];
#pragma unroll
        for (int r = 0; r < 6; r++)
          t2[r] = quad_sum(al[0] * m0 * v[0][r] + al[1] * r2[1] * v[1][r] + al[2] * r2[2] * v[2][r]);
      }
      solve6_thread(N, rdg, t2);
      {
        creal g[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
          creal d = r2[c];
#pragma unroll
          for (int r = 0; r < 6; r++) d = fma(-At[c][r], t2[r], d);
          g[c] = d;
        }
        const creal hn = al[0] * (g[0] - e1 * g[1] - e2 * g[2]);
        x[0] = hn; x[1] = fma(-e1, hn, al[1] * g[1]); x[2] = fma(-e2, hn, al[2] * g[2]);
      }
      leg_rows(x[0], x[1], x[2], mu, de);
      ratio = 0.f;
#pragma unroll
      for (int r = 0; r < 5; r++) {
        de[r] = (alive && ipm_round) ? de[r] : creal(0.0);
        ds[r] = de[r] - rp[r];
        dl[r] = (alive && ipm_round) ? -fma(lam[r], ds[r], rc[r]) * rs[r] : creal(0.0);
        if (alive && ipm_round) ratio = fmaxf(ratio, fmaxf(-(float)ds[r] * (float)rs[r], -(float)dl[r] * rcp_approx((float)lam[r])));
      }
      ratio = quad_max(ratio);
      creal alp = (ratio > 0.995f) ? creal(0.995) / (creal)ratio : creal(1.0);
#pragma unroll 1
      for (int tries = 0; tries < 20; tries++) {
        float ps = 0.f, pm = 3e38f;
#pragma unroll
        for (int r = 0; r < 5; r++) {
          const float pr = (float)(fma(alp, ds[r], s[r]) * fma(alp, dl[r], lam[r]));
          ps += pr;
          pm = fminf(pm, pr);
        }
        ps = quad_sum((alive && ipm_round) ? ps : 0.f) * rm;
        pm = quad_min((alive && ipm_round) ? pm : 3e38f);
        const bool ok = !ipm_round || (pm >= (float)kNeighbourhood * ps && pm > 0.f);
        if (__all_sync(kFull, ok)) break;
        if (!ok) alp *= creal(0.7);
      }
      // step; residuals without a mat-vec: rd += al (r2 - D~'(theta .* de + dl)), rp *= (1 - al)
      creal w5[5];
#pragma unroll
      for (int r = 0; r < 5; r++) w5[r] = fma(th[r], de[r], dl[r]);
      leg_rows_t(w5, mu, dt);
      float pn = 0.f, nrp = 0.f, nrd = 0.f, ymax = 0.f;
      if (ipm_round) {
#pragma unroll
        for (int r = 0; r < 5; r++) {
          s[r] = fma(alp, ds[r], s[r]);
          lam[r] = fma(alp, dl[r], lam[r]);
          rp[r] *= (creal(1.0) - alp);
          pn += (float)(s[r] * lam[r]);
          nrp = fmaxf(nrp, fabsf((float)rp[r]));
        }
#pragma unroll
        for (int c = 0; c < 3; c++) {
          rdl[c] = alive ? fma(alp, r2[c] - dt[c], rdl[c]) : creal(0.0);
          y[c] = fma(alp, x[c], y[c]);
          nrd = fmaxf(nrd, fabsf((float)rdl[c]));
          ymax = fmaxf(ymax, fabsf((float)y[c]));
        }
        alpha_prev = alp;
        it++;
      }
      const float mu_n = quad_sum((alive && ipm_round) ? pn : 0.f) * rm;
      nrd = quad_max(nrd);
      nrp = quad_max(nrp);
      const float scale = fmaxf(1.f, quad_max(ymax));
      if (ipm_round) {
        const float tolf = Tol<creal>::ipm(cc.tol) * scale;
        converged = (mu_n <= tolf * gap_shrink) && (nrp <= tolf) && (nrd <= 100.f * tolf);
        const bool out_of_iters = it >= cc.max_iter;
        want_polish = converged || out_of_iters || (it >= QLB_POLISH_MIN_IT && mu_n <= QLB_POLISH_MU * scale);
        if (out_of_iters && !converged) status = 2;
      }
    }

    if (mode == kModeIpm && want_polish) {
      want_polish = false;
      mode = kModePolish;
      pass = 0;
      a0 = 0; sg1 = 0; sg2 = 0;
      if (alive) {
        a0 = lam[0] > s[0];
        sg1 = (lam[1] > s[1]) ? -1 : ((lam[2] > s[2]) ? 1 : 0);
        sg2 = (lam[3] > s[3]) ? -1 : ((lam[4] > s[4]) ? 1 : 0);
      }
    }
  }

}

// One work item (eight consecutive entries of a list, or eight consecutive states for STAGE 0) of a later
// pass, whole warp.  STAGE 0: the full algorithm (stand-alone, no lists).  STAGE 1: states of a.list;
// active-set rounds from the pattern the first pass left in a.list_pat; what is still not verified after
// QLB_PDAS_ROUNDS repairs is appended to a.list2.  STAGE 2: states of a.list2; interior-point iteration
// from the strictly feasible start, polish rounds when the complementarity gap is small.  Compacted lists
// give the eight states of a warp similar numbers of rounds.
template <typename real, typename creal, int MODE, int STAGE>
__device__ __forceinline__ void quad_batch(const SolveArgsT<real>& a, const DeviceParamsT<real>& prm, const CoreConst<creal>& cc,
                                           const CoreConst<double>& cc64, real (*jg)[kQuadThreads], const unsigned long long bq,
                                           const unsigned pat_word, const bool valid, const int lane, const int leg, const int quad) {
  constexpr bool kRescue = Tol<creal>::rescue && (STAGE == 1 || STAGE == 2);
  LegSetup<creal> L;
  {
    RawIn<real, MODE> in;
    quad_load<real, MODE>(a, prm.mu_default, bq, valid, leg, in);
    quad_setup<real, MODE, creal>(a, prm, in, bq, valid, STAGE == 0, leg, L, &jg[0][threadIdx.x], kQuadThreads);
  }
  creal y[3];
  int a0, sg1, sg2, status, it;
  bool defer;
  const unsigned pat0 = (STAGE == 1 && valid) ? (pat_word >> (5 * leg)) & 31u : 0u;
  quad_solve<creal, STAGE, kRescue>(L, cc, leg, quad, true, pat0, y, a0, sg1, sg2, status, it, defer);
  if (kRescue && STAGE == 2) {
    // not verified by the FP32 core (iteration limit, pattern not confirmed, factorisation failed): the
    // same warp solves these states again with the FP64 core, from scratch.  Rare (a few per 10^5).
    const bool again = (status == 2 || status == 3 || (status == 4 && !L.qbad));
    if (__any_sync(kFull, again)) {
      LegSetup<double> Ld;
      widen_setup(L, Ld);
      double yd[3];
      int a0d, sg1d, sg2d, statusd, itd;
      bool deferd;
      quad_solve<double, 0, false>(Ld, cc64, leg, quad, again, 0u, yd, a0d, sg1d, sg2d, statusd, itd, deferd);
      if (again) {
        y[0] = (creal)yd[0]; y[1] = (creal)yd[1]; y[2] = (creal)yd[2];
        a0 = a0d; sg1 = sg1d; sg2 = sg2d; status = statusd; it = itd;
      }
    }
  }
  if (STAGE == 1) {
    const unsigned hm = __ballot_sync(kFull, defer && valid && leg == 0);
    if (hm != 0u) {
      unsigned base = 0;
      if (lane == 0) base = atomicAdd(a.list2_count, __popc(hm));
      base = __shfl_sync(kFull, base, 0);
      if (defer && valid && leg == 0) a.list2[base + __popc(hm & ((1u << lane) - 1u))] = (unsigned)bq;
    }
  }
  quad_output<real, creal, real>(a, L, y, a0, sg1, sg2, status, it, bq, valid && !defer, leg, &jg[0][threadIdx.x], kQuadThreads);
}

// A later pass (STAGE as in quad_batch).  Two experiments that did not pay at 2^20 states (each pass has a
// latency floor of one warp's serial work, ~100 us): splitting pass 2 into "one round" + "remaining rounds"
// for better packing (measured 1.04 ms against 0.95 ms), and the opposite, fusing passes 2 and 3.  Cutting the
// batch into sub-batches on several streams so that tails overlap bulk work did not pay either (0.97 - 1.3 ms),
// nor did sorting the list into "one violated row" / "several violated rows" classes (0.86 against 0.84 ms).
// A one-state-per-thread version of pass 2 (blocks in thread-local memory, one factorisation per state, no
// shuffles) executes 31 % fewer instructions but runs slower (0.43 against 0.37 ms): eight warps per SM, the
// kinematics of the four legs in sequence, and a warp waits for the slowest of 32 states instead of 8.
// Passes 2 and 3 stay separate launches: fused into one persistent
// kernel (warps taking interior-point items as soon as they are published) the code grows to 190 KB, past the
// instruction cache, and the pair runs 3x slower (measured: 2.9 ms against 0.96 ms per 2^20 states).
template <typename real, typename creal, int MODE, int STAGE>
__global__ void __launch_bounds__(kQuadThreads, STAGE == 1 ? QLB_QUAD_MIN_CTAS : QLB_IPM_MIN_CTAS) qlb_quad_kernel(const SolveArgsT<real> a) {
  __shared__ DeviceParamsT<real> prm;
  __shared__ CoreConst<creal> cc;
  __shared__ CoreConst<double> cc64;  // in-kernel rescue of the FP32 core
  __shared__ real jg[12][kQuadThreads];  // per thread: Jacobian (9) and gravity torques (3) of its leg
  // a list pass with an empty list (the usual case for the interior-point pass behind the fused kernel): nothing to set up
  if (STAGE != 0 && __ldcg(STAGE == 1 ? a.list_count : a.list2_count) == 0u) return;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.params);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&prm);
    for (int i = threadIdx.x; i < (int)(sizeof(DeviceParamsT<real>) / 4); i += blockDim.x) dst[i] = src[i];
    // the solver core reads its weights from the FP64 parameter block, in its own type
    cc.load(a.params64);
    load_model_to_smem(a.model);
    if (Tol<creal>::rescue && STAGE == 2) cc64.load(a.params64);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int leg = lane & 3, quad = lane >> 2;
  const unsigned long long total = (STAGE == 0) ? a.B : (unsigned long long)(*(STAGE == 1 ? a.list_count : a.list2_count));
  unsigned long long* const work = (STAGE == 0) ? a.counter : (STAGE == 1 ? a.counter2 : a.counter3);
  // The interior-point pass takes ONE state per warp (quad 0; the other quads idle).  With eight states per warp it
  // has returned, about once in 10^5 states of a sweep with F_min = 0, a state solved as if some of its legs were not
  // standing - depending on which states shared the warp, invisible to compute-sanitizer, gone with any
  // instrumentation (DESIGN.md 8).  One state per warp rules out every interaction between the quads of a warp;
  // the pass sees at most 1 % of the states of the three-pass pipeline and normally none behind the fused kernel.
  const unsigned long long nbatch = (STAGE == 2) ? total : (total + 7) / 8;
  const unsigned long long B = a.B;
  const unsigned* const in_list = (STAGE == 1) ? a.list : a.list2;
  // Software pipeline over the work items of this warp, two deep: the index (and pattern) of item i+2 is being
  // loaded, the input rows of item i+1 are being prefetched, while item i is solved - the gathers of a listed
  // state are scattered 32-byte sectors and would otherwise stall the warp at the start of every item.
  // (Static first items - warp w takes w and w + #warps - were measured and are slower: 0.84 against 0.79 ms.)
  auto claim = [&]() {
    unsigned long long b = 0;
    if (lane == 0) b = atomicAdd(work, 1ull);
    return __shfl_sync(kFull, b, 0);
  };
  auto fetch = [&](const unsigned long long b, unsigned long long& idx, unsigned& pat, bool& ok) {
    const unsigned long long slot = (STAGE == 2) ? b : b * 8 + quad;
    ok = (b < nbatch) && (slot < total) && (STAGE != 2 || quad == 0);
    idx = B - 1; pat = 0u;
    if (ok) {
      idx = (STAGE == 0) ? slot : (unsigned long long)__ldcg(in_list + slot);
      if (STAGE == 1) pat = __ldcg(a.list_pat + slot);
    }
  };
  unsigned long long b0 = claim(), b1 = claim();
  unsigned long long idx0, idx1;
  unsigned pat0w, pat1w;
  bool ok0, ok1;
  fetch(b0, idx0, pat0w, ok0);
  fetch(b1, idx1, pat1w, ok1);
  while (b0 < nbatch) {
    const unsigned long long b2 = claim();
    unsigned long long idx2;
    unsigned pat2w;
    bool ok2;
    fetch(b2, idx2, pat2w, ok2);
    if (b1 < nbatch) quad_prefetch<real, MODE>(a, idx1, leg);
    quad_batch<real, creal, MODE, STAGE>(a, prm, cc, cc64, jg, idx0, pat0w, ok0, lane, leg, quad);
    b0 = b1; idx0 = idx1; pat0w = pat1w; ok0 = ok1;
    b1 = b2; idx1 = idx2; pat1w = pat2w; ok1 = ok2;
  }
}

}  // namespace qlb
