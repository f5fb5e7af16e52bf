// qlb_aux.cuh - small companion kernels: stand-alone leg kinematics and batch statistics.
#pragma once

#include "qlb.h"
#include "qlb_device.cuh"

namespace qlb {

// One thread per (state, leg): foot position, translational Jacobian, gravity torques.
// Replaces QuadrupedKinematics::FowardKinematicsSolve / AnalysticJacobian /
// getGravityCompensationForLimb (quadruped_model/src/quadrupedkinematics.cpp:143-278,485-552).
// Consecutive threads handle consecutive states of the same leg, so all global accesses coalesce.
__global__ void __launch_bounds__(128) qlb_kinematics_kernel(unsigned long long B, const double* __restrict__ q,
                                                             const double* __restrict__ quat, double* __restrict__ foot,
                                                             double* __restrict__ jac, double* __restrict__ gtau,
                                                             const DeviceModel* __restrict__ mdl,
                                                             const DeviceParams* __restrict__ prm,
                                                             const double* __restrict__ pose = nullptr,
                                                             double* __restrict__ foot_world = nullptr) {
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 4ull * B) return;
  const int leg = (int)(t / B);
  const unsigned long long i = t - (unsigned long long)leg * B;
  double gb[3] = {0.0, 0.0, -prm->gravity};
  if (quat) {
    const double w = quat[i], x = quat[B + i], y = quat[2 * B + i], z = quat[3 * B + i];
    // third row of R_bw = R_wb * e_z
    gb[0] = -prm->gravity * 2.0 * (x * z - w * y);
    gb[1] = -prm->gravity * 2.0 * (y * z + w * x);
    gb[2] = -prm->gravity * (w * w - x * x - y * y + z * z);
  }
  double R[9], p[3], zax[3][3], pj[3][3], com[4][3];
#pragma unroll
  for (int e = 0; e < 9; e++) R[e] = mdl->rot[leg][0][e];
#pragma unroll
  for (int a = 0; a < 3; a++) p[a] = mdl->xyz[leg][0][a];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    if (j > 0) {
      const double* xj = mdl->xyz[leg][j];
#pragma unroll
      for (int a = 0; a < 3; a++) p[a] += R[3 * a] * xj[0] + R[3 * a + 1] * xj[1] + R[3 * a + 2] * xj[2];
      if (j < 3) {
        const double* Rj = mdl->rot[leg][j];
        double T[9];
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
      for (int a = 0; a < 3; a++) { zax[j][a] = R[3 * a + 2]; pj[j][a] = p[a]; }
      double sj, cj;
      sincos(q[(size_t)(3 * leg + j) * B + i], &sj, &cj);
#pragma unroll
      for (int r = 0; r < 3; r++) {
        const double a0 = R[3 * r], a1 = R[3 * r + 1];
        R[3 * r] = cj * a0 + sj * a1;
        R[3 * r + 1] = cj * a1 - sj * a0;
      }
    }
    const double* cm = mdl->com[leg][j];
#pragma unroll
    for (int a = 0; a < 3; a++) com[j][a] = p[a] + R[3 * a] * cm[0] + R[3 * a + 1] * cm[1] + R[3 * a + 2] * cm[2];
  }
  if (foot) {
#pragma unroll
    for (int a = 0; a < 3; a++) foot[(size_t)(3 * leg + a) * B + i] = p[a];
  }
  if (pose && foot_world) {
    // world <- base: position + R_bw * foot (StateBatchComputer.cpp:64-77, getPositionWorldToFootInWorldFrame)
    const double w = pose[3 * B + i], x = pose[4 * B + i], y = pose[5 * B + i], z = pose[6 * B + i];
    const double Rw[9] = {w * w + x * x - y * y - z * z, 2.0 * (x * y - w * z), 2.0 * (x * z + w * y),
                          2.0 * (x * y + w * z), w * w - x * x + y * y - z * z, 2.0 * (y * z - w * x),
                          2.0 * (x * z - w * y), 2.0 * (y * z + w * x), w * w - x * x - y * y + z * z};
#pragma unroll
    for (int a = 0; a < 3; a++)
      foot_world[(size_t)(3 * leg + a) * B + i] = pose[(size_t)a * B + i] + Rw[3 * a] * p[0] + Rw[3 * a + 1] * p[1] + Rw[3 * a + 2] * p[2];
  }
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const double dv[3] = {p[0] - pj[k][0], p[1] - pj[k][1], p[2] - pj[k][2]};
    const double col[3] = {zax[k][1] * dv[2] - zax[k][2] * dv[1], zax[k][2] * dv[0] - zax[k][0] * dv[2],
                           zax[k][0] * dv[1] - zax[k][1] * dv[0]};
    if (jac) {
#pragma unroll
      for (int a = 0; a < 3; a++) jac[(size_t)(9 * leg + 3 * a + k) * B + i] = col[a];
    }
    if (gtau) {
      double acc[3] = {0.0, 0.0, 0.0};
#pragma unroll
      for (int l = 0; l < 4; l++) {
        if (l < k) continue;
        const double m = mdl->mass[leg][l];
        const double arm[3] = {com[l][0] - pj[k][0], com[l][1] - pj[k][1], com[l][2] - pj[k][2]};
        acc[0] += m * (arm[1] * gb[2] - arm[2] * gb[1]);
        acc[1] += m * (arm[2] * gb[0] - arm[0] * gb[2]);
        acc[2] += m * (arm[0] * gb[1] - arm[1] * gb[0]);
      }
      gtau[(size_t)(3 * leg + k) * B + i] = -(zax[k][0] * acc[0] + zax[k][1] * acc[1] + zax[k][2] * acc[2]);
    }
  }
}

// RobotState records (array of structs, the fields RosBalanceController::baseCommandCallback reads from
// free_gait_msgs/RobotState, ros_balance_controller.cpp:761-811,860-...) -> the SoA arrays of the solver.
// Pure byte movement, HBM-bound: a CTA copies kPackTile records with 16-byte coalesced loads into shared
// memory (row stride padded by 8 bytes against bank conflicts), then every thread walks one record and the
// warp writes 256 contiguous bytes per component row.
constexpr int kPackTile = 128;
constexpr int kRecWords = (int)(sizeof(qlb_robot_state_record) / 8);   // 38 doubles
__global__ void __launch_bounds__(kPackTile) qlb_pack_kernel(unsigned long long B, const qlb_robot_state_record* __restrict__ rec,
                                                             double* __restrict__ q, double* __restrict__ pose,
                                                             double* __restrict__ twist, uint8_t* __restrict__ mask,
                                                             double* __restrict__ normals) {
  __shared__ double tile[kPackTile * (kRecWords + 1)];
  const unsigned long long base = (unsigned long long)blockIdx.x * kPackTile;
  const unsigned long long left = B - base;
  const int n = left < (unsigned long long)kPackTile ? (int)left : kPackTile;
  const double2* src = reinterpret_cast<const double2*>(rec + base);   // records are 304 B = 19 x 16 B
  const int nvec = n * (kRecWords / 2);
  for (int v = threadIdx.x; v < nvec; v += kPackTile) {
    const double2 d = __ldg(src + v);
    const int r = v / (kRecWords / 2), c = 2 * (v - r * (kRecWords / 2));
    tile[r * (kRecWords + 1) + c] = d.x;
    tile[r * (kRecWords + 1) + c + 1] = d.y;
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t >= n) return;
  const double* r = tile + t * (kRecWords + 1);
  const unsigned long long i = base + t;
  // record layout: position 0-2, orientation xyzw 3-6, linear velocity 7-9, angular velocity 10-12,
  // joint positions 13-24, surface normals 25-36, support flags in word 37
  if (pose) {
#pragma unroll
    for (int a = 0; a < 3; a++) pose[(size_t)a * B + i] = r[a];
    pose[(size_t)3 * B + i] = r[6];   // w first: kindr RotationQuaternion(w, x, y, z), ros_balance_controller.cpp:766-769
    pose[(size_t)4 * B + i] = r[3];
    pose[(size_t)5 * B + i] = r[4];
    pose[(size_t)6 * B + i] = r[5];
  }
  if (twist) {
#pragma unroll
    for (int a = 0; a < 6; a++) twist[(size_t)a * B + i] = r[7 + a];
  }
  if (q) {
#pragma unroll
    for (int a = 0; a < 12; a++) q[(size_t)a * B + i] = r[13 + a];
  }
  if (normals) {
#pragma unroll
    for (int a = 0; a < 12; a++) normals[(size_t)a * B + i] = r[25 + a];
  }
  if (mask) {
    const unsigned long long w = (unsigned long long)__double_as_longlong(r[37]);
    unsigned m = 0;
#pragma unroll
    for (int l = 0; l < 4; l++) m |= (((w >> (8 * l)) & 0xFFull) != 0ull ? 1u : 0u) << l;
    mask[i] = (uint8_t)m;
  }
}

// Batch statistics: counts per status, iteration sum/max, weighted wrench error sum/max, active-row histogram.
// HBM-bound byte movement (100 bytes per state: the flags word and the two wrench rows).  Every counter is an integer
// per thread; a warp folds each with one redux instruction, lane 0 adds the 28 integers to the block's shared-memory
// counters, the two floating-point statistics go through a shuffle butterfly; one global atomic per block and
// statistic.  (The first version did 31 shared-memory double atomics per THREAD: 173 us per 2^20 states, atomics-bound.)
__global__ void __launch_bounds__(256) qlb_stats_kernel(unsigned long long B, const uint32_t* __restrict__ flags,
                                                        const double* __restrict__ wrench,
                                                        const double* __restrict__ netwrench,
                                                        const DeviceParams* __restrict__ prm, double* __restrict__ out) {
  __shared__ unsigned long long shi[29];   // count, status[5], iterations, (unused), hist[20], infeasible
  __shared__ double sh_err;
  __shared__ unsigned long long sh_maxerr, sh_maxit;
  if (threadIdx.x < 29) shi[threadIdx.x] = 0ull;
  if (threadIdx.x == 32) { sh_err = 0.0; sh_maxerr = 0ull; sh_maxit = 0ull; }
  __syncthreads();
  unsigned cnt[7] = {0u, 0u, 0u, 0u, 0u, 0u, 0u};   // count, status 0..4, infeasible
  unsigned its = 0u, max_it = 0u;
  unsigned hist_local[20];
#pragma unroll
  for (int k = 0; k < 20; k++) hist_local[k] = 0u;
  double err_sum = 0.0, max_err = 0.0;
  const double S0 = prm->S[0], S1 = prm->S[1], S2 = prm->S[2], S3 = prm->S[3], S4 = prm->S[4], S5 = prm->S[5];
  const double Sw[6] = {S0, S1, S2, S3, S4, S5};
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < B;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const uint32_t f = flags[i];
    const unsigned st = (f >> QLB_FLAG_STATUS_SHIFT) & 7u;
    const unsigned it = f >> QLB_FLAG_ITER_SHIFT;
    cnt[0]++;
#pragma unroll
    for (int k = 0; k < 5; k++) cnt[1 + k] += (st == (unsigned)k) ? 1u : 0u;
    cnt[6] += (st == 5u) ? 1u : 0u;
    its += it;
    max_it = max(max_it, it);
    const unsigned act = (f & QLB_FLAG_ACTIVE_MASK) >> QLB_FLAG_ACTIVE_SHIFT;
#pragma unroll
    for (int k = 0; k < 20; k++) hist_local[k] += (act >> k) & 1u;
    if (wrench && netwrench && (st == 0 || st == 2 || st == 3)) {
      double e2 = 0.0;
#pragma unroll
      for (int r = 0; r < 6; r++) {
        const double d = netwrench[(size_t)r * B + i] - wrench[(size_t)r * B + i];
        e2 += Sw[r] * d * d;
      }
      const double e = sqrt(e2);
      err_sum += e;
      max_err = fmax(max_err, e);
    }
  }
  // warp level: integers through redux, the two doubles through a butterfly
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 7; k++) cnt[k] = __reduce_add_sync(full, cnt[k]);
  its = __reduce_add_sync(full, its);
  max_it = __reduce_max_sync(full, max_it);
#pragma unroll
  for (int k = 0; k < 20; k++) hist_local[k] = __reduce_add_sync(full, hist_local[k]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    err_sum += __shfl_xor_sync(full, err_sum, o);
    max_err = fmax(max_err, __shfl_xor_sync(full, max_err, o));
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 6; k++) atomicAdd(&shi[k], (unsigned long long)cnt[k]);
    atomicAdd(&shi[6], (unsigned long long)its);
#pragma unroll
    for (int k = 0; k < 20; k++) atomicAdd(&shi[8 + k], (unsigned long long)hist_local[k]);
    atomicAdd(&shi[28], (unsigned long long)cnt[6]);
    atomicAdd(&sh_err, err_sum);
    // max via atomicMax on the bit pattern (values are non-negative)
    atomicMax(&sh_maxerr, (unsigned long long)__double_as_longlong(max_err));
    atomicMax(&sh_maxit, (unsigned long long)max_it);
  }
  __syncthreads();
  // out[] in the order of qlb_stats: 0 count, 1..5 status, 6 iterations, 7 error sum, 8..27 histogram, 28 infeasible, 29 / 30 maxima
  const int t = threadIdx.x;
  if (t < 29 && t != 7) { if (shi[t] != 0ull) atomicAdd(&out[t], (double)shi[t]); }
  else if (t == 7) atomicAdd(&out[7], sh_err);
  else if (t == 29) atomicMax(reinterpret_cast<unsigned long long*>(&out[29]), sh_maxerr);
  else if (t == 30) atomicMax(reinterpret_cast<unsigned long long*>(&out[30]), (unsigned long long)__double_as_longlong((double)sh_maxit));
}

// Batched per-leg contact state machine: RosBalanceController::footContactsCallback
// (balance_controller/src/ros_controller/ros_balance_controller.cpp:1086-1140) and the support-leg decision that
// update() derives from the limb state (:242-366).  One thread per state, the four legs in sequence.
//   desired   bit k = the plan says leg k is a stance leg (limbs_desired_state == StanceNormal, else SwingNormal)
//   footstep  bit k = is_footstep_ (the leg takes part in contact supervision)
//   contact   bit k = measured foot contact (FootContacts.is_contact)
//   phase     [4][B] the phase of the leg's current stance or swing (st_phase / sw_phase, :979-1077)
//   limb_state[4][B] in: previous state, out: new state (qlb_limb_state values = StateSwitcher::States order)
//   stance    [B] out: bit k = leg k is a support leg for the force distribution
// (The reference advances its limb index only at the end of the loop body, so a `continue` makes the next foot
// overwrite the same limb; the per-limb rules below are the evident intent.)
// One robot i: phase has row pitch ld_phase, limb_state row pitch ld_limb (the controller tick keeps its limb states
// in arrays of its own batch size).  Returns the stance mask.  A float phase is widened before the comparisons, so the
// states are those of the double phase of the same value (against float literals, 0.1f > 0.1 would differ).
template <typename P>
__device__ __forceinline__ unsigned contact_fsm_robot(unsigned long long i, unsigned des, unsigned fs, unsigned con,
                                                      const P* __restrict__ phase, unsigned long long ld_phase,
                                                      uint8_t* __restrict__ limb_state, unsigned long long ld_limb) {
  unsigned mask = 0u;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const bool d = (des >> k) & 1u, f = (fs >> k) & 1u, c = (con >> k) & 1u;
    const double ph = (double)phase[(size_t)k * ld_phase + i];
    unsigned st = limb_state[(size_t)k * ld_limb + i];
    if (!d) {
      st = QLB_LIMB_SWING_NORMAL;
      if (f) {
        if (ph > 0.5) { if (c) st = QLB_LIMB_SWING_EARLY_TOUCHDOWN; }
        else if (ph > 0.2) { if (c) st = QLB_LIMB_SWING_BUMPED_INTO_OBSTACLE; }
      }
    } else {
      if (!f) {
        st = QLB_LIMB_STANCE_NORMAL;
      } else {
        if (c) st = QLB_LIMB_STANCE_NORMAL;
        else if (ph < 0.1) st = QLB_LIMB_SWING_LATELY_TOUCHDOWN;
        if (ph > 0.5 && !c) st = QLB_LIMB_STANCE_LOST_CONTACT;
      }
    }
    limb_state[(size_t)k * ld_limb + i] = (uint8_t)st;
    const bool support = st == QLB_LIMB_STANCE_NORMAL || st == QLB_LIMB_SWING_EARLY_TOUCHDOWN || st == QLB_LIMB_INIT;
    mask |= (support ? 1u : 0u) << k;
  }
  return mask;
}

__global__ void __launch_bounds__(256) qlb_contact_fsm_kernel(unsigned long long B, const uint8_t* __restrict__ desired,
                                                              const uint8_t* __restrict__ footstep, const uint8_t* __restrict__ contact,
                                                              const double* __restrict__ phase, uint8_t* __restrict__ limb_state,
                                                              uint8_t* __restrict__ stance) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const unsigned mask = contact_fsm_robot(i, desired[i], footstep ? footstep[i] : 0xFu, contact[i], phase, B, limb_state, B);
  if (stance) stance[i] = (uint8_t)mask;
}

// Friction margins of a solved batch: for every state the smallest slack of the friction-pyramid and minimal-force
// rows over its stance legs, relative to the normal force - how far the planned motion stays from slipping (0 = a
// friction row is active, negative = infeasible answer).  What a preview of a planned motion reads next to the
// forces (SURVEY 8f rank 2; the rows are those of ContactForceDistribution.cpp:210-336).  One thread per state.
__global__ void __launch_bounds__(256) qlb_friction_margin_kernel(unsigned long long B, const double* __restrict__ grf,
                                                                  const double* __restrict__ quat, const uint8_t* __restrict__ mask,
                                                                  const double* __restrict__ mu, const double* __restrict__ normals,
                                                                  const DeviceParams* __restrict__ prm, double* __restrict__ margin,
                                                                  double* __restrict__ min_normal) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const double w = quat[i], x = quat[B + i], y = quat[2 * B + i], z = quat[3 * B + i];
  const double R[9] = {w * w + x * x - y * y - z * z, 2.0 * (x * y - w * z), 2.0 * (x * z + w * y),
                       2.0 * (x * y + w * z), w * w - x * x + y * y - z * z, 2.0 * (y * z - w * x),
                       2.0 * (x * z - w * y), 2.0 * (y * z + w * x), w * w - x * x - y * y + z * z};
  const unsigned m = mask[i];
  double best = 1e300, bestn = 1e300;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    if (!((m >> k) & 1u)) continue;
    double nw[3] = {0.0, 0.0, 1.0};
    if (normals) { nw[0] = normals[(size_t)(3 * k) * B + i]; nw[1] = normals[(size_t)(3 * k + 1) * B + i]; nw[2] = normals[(size_t)(3 * k + 2) * B + i]; }
    double n[3], t1[3], t2[3];
#pragma unroll
    for (int c = 0; c < 3; c++) n[c] = R[c] * nw[0] + R[3 + c] * nw[1] + R[6 + c] * nw[2];   // R_wb n_world
    const double ey[3] = {R[3], R[4], R[5]};
    t1[0] = n[1] * ey[2] - n[2] * ey[1]; t1[1] = n[2] * ey[0] - n[0] * ey[2]; t1[2] = n[0] * ey[1] - n[1] * ey[0];
    double rn = rsqrt(t1[0] * t1[0] + t1[1] * t1[1] + t1[2] * t1[2]);
    t1[0] *= rn; t1[1] *= rn; t1[2] *= rn;
    t2[0] = n[1] * t1[2] - n[2] * t1[1]; t2[1] = n[2] * t1[0] - n[0] * t1[2]; t2[2] = n[0] * t1[1] - n[1] * t1[0];
    rn = rsqrt(t2[0] * t2[0] + t2[1] * t2[1] + t2[2] * t2[2]);
    t2[0] *= rn; t2[1] *= rn; t2[2] *= rn;
    const double f[3] = {grf[(size_t)(3 * k) * B + i], grf[(size_t)(3 * k + 1) * B + i], grf[(size_t)(3 * k + 2) * B + i]};
    const double fn = f[0] * n[0] + f[1] * n[1] + f[2] * n[2];
    const double f1 = f[0] * t1[0] + f[1] * t1[1] + f[2] * t1[2];
    const double f2 = f[0] * t2[0] + f[1] * t2[1] + f[2] * t2[2];
    const double muk = mu ? mu[(size_t)k * B + i] : prm->mu_default;
    const double slack = fmin(muk * fn - fabs(f1), muk * fn - fabs(f2));
    const double rel = slack / fmax(muk * fn, 1e-300);
    best = fmin(best, rel);
    bestn = fmin(bestn, fn - prm->fmin);
  }
  margin[i] = (m & 0xFu) ? best : 0.0;
  if (min_normal) min_normal[i] = (m & 0xFu) ? bestn : 0.0;
}

// FP64 FMA throughput probe: the roofline denominator for this path (SURVEY.md 8d asks for a measured
// figure; MEASURED_PEAKS.json only has HBM and bf16).  8 independent DFMA chains per thread.
__global__ void __launch_bounds__(256) qlb_fp64_peak_kernel(double* __restrict__ sink, int iters, double seed) {
  double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
  const double m = 1.0000001, c = 1e-9;
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 16; u++) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (r == 12345.678) sink[0] = r;  // never true; keeps the chains alive
}

}  // namespace qlb
