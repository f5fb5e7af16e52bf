// qlb_swing.cuh - swing-leg joint torques for a batch of states: limb inverse dynamics + Cartesian PD.
//
// Replaces MyRobotSolver::update (single_leg_test/lib/model_test_header.cpp:412-502), which the balance
// controller calls for every leg that is not in stance (ros_balance_controller.cpp:472-603):
//     tau = InverseDynamics(limb model, q, qd, 0.5 qdd)                       (:460)
//         + J^T (kp .* (p* - p) + kd .* (v* - v)),   v = J qd                 (:481-498)
// One thread per (state, leg); consecutive threads take consecutive states of one leg, so every access to the
// SoA arrays coalesces.  The recursive Newton-Euler algorithm is written in the base frame as plain sums
// (three bodies): angular velocity / acceleration and the acceleration of every joint origin outward, then
// tau_j = z_j . sum_{i>=j} [ N_i + (c_i - p_j) x F_i ].  Gravity enters as the base acceleration -g.
#pragma once

#include "qlb.h"
#include "qlb_device.cuh"

namespace qlb {

template <typename T>
struct DeviceLimbDynamicsT {
  T rot[4][3][9];      // [leg][joint] rotation of <origin rpy>, row-major
  T xyz[4][3][3];      // [leg][joint] <origin xyz>
  T mass[4][3];
  T com[4][3][3];      // link frame
  T inertia[4][3][6];  // Ixx Ixy Ixz Iyy Iyz Izz about the centre of mass, link axes
};
using DeviceLimbDynamics = DeviceLimbDynamicsT<double>;

// T = double, or float for the FP32 controller tick (the acceleration is then differenced in FP32 from the newest
// float sample and the FP64 ring slot rounded to float).
template <typename T>
struct SwingArgsT {
  unsigned long long B;
  const T* q;
  const T* qd;
  const T* qdd;            // null when the acceleration comes from the velocity queue
  const double* qd_front;  // oldest entry of the caller's joint-velocity queue (qd is its newest entry), or null
  unsigned long long ld_front;  // row pitch of qd_front (B, or the batch size of the controller that owns the queue)
  T inv_window;            // 1 / (10 * period): the reference's Time_derta (model_test_header.cpp:421,428)
  const T* ptarget;        // may be null
  const T* vtarget;        // may be null
  T* tau;
  T gravity[3];
  T acc_scale;
  T kp[3], kd[3];
  const DeviceLimbDynamicsT<T>* dyn;
  const DeviceModelT<T>* model;  // foot frame of the kinematic model (the Jacobian the controller uses)
};
using SwingArgs = SwingArgsT<double>;

// sin and cos of a joint angle.  FP32 goes through sincospif, whose range reduction is exact: sincosf would carry a
// Payne-Hanek slow path for huge arguments (local memory and FP64 arithmetic).  The product q / pi rounds once, an
// angle error of the order of rounding q itself to float.
__device__ __forceinline__ void joint_sincos(const double x, double* s, double* c) { sincos(x, s, c); }
__device__ __forceinline__ void joint_sincos(const float x, float* s, float* c) { sincospif(x * 0.318309886183790672f, s, c); }

template <typename T>
__device__ __forceinline__ void cross3(const T (&a)[3], const T (&b)[3], T (&o)[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}

// The three joint torques of leg `leg` of state i (used by qlb_swing_kernel and the controller tick's epilogue).
template <typename T>
__device__ __forceinline__ void swing_leg_torque(const SwingArgsT<T>& a, const int leg, const unsigned long long i, T (&tau)[3]) {
  const unsigned long long B = a.B;
  const DeviceLimbDynamicsT<T>& dyn = *a.dyn;
  T qv[3], qdv[3], qddv[3];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    qv[j] = a.q[(size_t)(3 * leg + j) * B + i];
    qdv[j] = a.qd[(size_t)(3 * leg + j) * B + i];
    // acceleration: given, or estimated as the reference does from the two ends of its velocity queue,
    // (qd_back - qd_front) / (10 * period)  (model_test_header.cpp:421-429; the windowed average it also computes is never used)
    const T acc = a.qd_front ? (qdv[j] - (T)a.qd_front[(size_t)(3 * leg + j) * a.ld_front + i]) * a.inv_window : a.qdd[(size_t)(3 * leg + j) * B + i];
    qddv[j] = a.acc_scale * acc;
  }
  // ---- outward pass in the base frame
  T R[9], p[3] = {T(0), T(0), T(0)};
  T w[3] = {T(0), T(0), T(0)}, al[3] = {T(0), T(0), T(0)};
  T acc[3] = {-a.gravity[0], -a.gravity[1], -a.gravity[2]};   // acceleration of the current joint origin
  T zj[3][3], pj[3][3], F[3][3], N[3][3], cw[3][3];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    // joint origin: p_j = p_{j-1} + R_{j-1} xyz_j; its acceleration from the parent link's motion
    T d[3];
    if (j == 0) {
#pragma unroll
      for (int c = 0; c < 3; c++) d[c] = dyn.xyz[leg][0][c];
#pragma unroll
      for (int e = 0; e < 9; e++) R[e] = dyn.rot[leg][0][e];
    } else {
      const T x0 = dyn.xyz[leg][j][0], x1 = dyn.xyz[leg][j][1], x2 = dyn.xyz[leg][j][2];
#pragma unroll
      for (int c = 0; c < 3; c++) d[c] = R[3 * c] * x0 + R[3 * c + 1] * x1 + R[3 * c + 2] * x2;
      T Tm[9];
      const T* Rj = dyn.rot[leg][j];
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int s = 0; s < 3; s++) Tm[3 * r + s] = R[3 * r] * Rj[s] + R[3 * r + 1] * Rj[3 + s] + R[3 * r + 2] * Rj[6 + s];
#pragma unroll
      for (int e = 0; e < 9; e++) R[e] = Tm[e];
    }
    {
      T wd[3], t1[3], t2[3];
      cross3(al, d, t1);
      cross3(w, d, wd);
      cross3(w, wd, t2);
#pragma unroll
      for (int c = 0; c < 3; c++) { acc[c] += t1[c] + t2[c]; p[c] += d[c]; }
    }
#pragma unroll
    for (int c = 0; c < 3; c++) { zj[j][c] = R[3 * c + 2]; pj[j][c] = p[c]; }
    // joint rotation, then the link's angular velocity and acceleration
    T sj, cj;
    joint_sincos(qv[j], &sj, &cj);
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const T a0 = R[3 * r], a1 = R[3 * r + 1];
      R[3 * r] = cj * a0 + sj * a1;
      R[3 * r + 1] = cj * a1 - sj * a0;
    }
    {
      T zq[3] = {zj[j][0] * qdv[j], zj[j][1] * qdv[j], zj[j][2] * qdv[j]}, wz[3];
      cross3(w, zq, wz);
#pragma unroll
      for (int c = 0; c < 3; c++) { al[c] += zj[j][c] * qddv[j] + wz[c]; w[c] += zq[c]; }
    }
    // the body: centre of mass, its acceleration, force and moment about the centre of mass
    T rc[3];
    {
      const T c0 = dyn.com[leg][j][0], c1 = dyn.com[leg][j][1], c2 = dyn.com[leg][j][2];
#pragma unroll
      for (int c = 0; c < 3; c++) rc[c] = R[3 * c] * c0 + R[3 * c + 1] * c1 + R[3 * c + 2] * c2;
    }
    T t1[3], wr[3], t2[3];
    cross3(al, rc, t1);
    cross3(w, rc, wr);
    cross3(w, wr, t2);
    const T m = dyn.mass[leg][j];
#pragma unroll
    for (int c = 0; c < 3; c++) { F[j][c] = m * (acc[c] + t1[c] + t2[c]); cw[j][c] = p[c] + rc[c]; }
    // I_base = R I R^T applied to a vector: R (I (R^T v))
    const T* I6 = dyn.inertia[leg][j];
    auto apply_inertia = [&](const T (&v)[3], T (&o)[3]) {
      T l[3], u[3];
#pragma unroll
      for (int c = 0; c < 3; c++) l[c] = R[c] * v[0] + R[3 + c] * v[1] + R[6 + c] * v[2];
      u[0] = I6[0] * l[0] + I6[1] * l[1] + I6[2] * l[2];
      u[1] = I6[1] * l[0] + I6[3] * l[1] + I6[4] * l[2];
      u[2] = I6[2] * l[0] + I6[4] * l[1] + I6[5] * l[2];
#pragma unroll
      for (int c = 0; c < 3; c++) o[c] = R[3 * c] * u[0] + R[3 * c + 1] * u[1] + R[3 * c + 2] * u[2];
    };
    T Ia[3], Iw[3], wIw[3];
    apply_inertia(al, Ia);
    apply_inertia(w, Iw);
    cross3(w, Iw, wIw);
#pragma unroll
    for (int c = 0; c < 3; c++) N[j][c] = Ia[c] + wIw[c];
  }
  // ---- inward pass: tau_j = z_j . sum_{i >= j} [N_i + (c_i - p_j) x F_i]
#pragma unroll
  for (int j = 0; j < 3; j++) {
    T s[3] = {T(0), T(0), T(0)};
#pragma unroll
    for (int k = 0; k < 3; k++) {
      if (k >= j) {
        const T arm[3] = {cw[k][0] - pj[j][0], cw[k][1] - pj[j][1], cw[k][2] - pj[j][2]};
        T mf[3];
        cross3(arm, F[k], mf);
#pragma unroll
        for (int c = 0; c < 3; c++) s[c] += N[k][c] + mf[c];
      }
    }
    tau[j] = zj[j][0] * s[0] + zj[j][1] * s[1] + zj[j][2] * s[2];
  }
  // ---- Cartesian PD on the foot, with the kinematic model's foot frame and Jacobian (the controller takes them
  //      from QuadrupedState, i.e. the full URDF: model_test_header.cpp:418,481-498)
  if (a.ptarget != nullptr || a.vtarget != nullptr) {
    const DeviceModelT<T>& mdl = *a.model;
    T Rk[9], pk[3], zk[3][3], pjk[3][3];
#pragma unroll
    for (int e = 0; e < 9; e++) Rk[e] = mdl.rot[leg][0][e];
#pragma unroll
    for (int c = 0; c < 3; c++) pk[c] = mdl.xyz[leg][0][c];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      if (j > 0) {
        const T x0 = mdl.xyz[leg][j][0], x1 = mdl.xyz[leg][j][1], x2 = mdl.xyz[leg][j][2];
#pragma unroll
        for (int c = 0; c < 3; c++) pk[c] += Rk[3 * c] * x0 + Rk[3 * c + 1] * x1 + Rk[3 * c + 2] * x2;
        if (j < 3) {
          T Tm[9];
          const T* Rj = mdl.rot[leg][j];
#pragma unroll
          for (int r = 0; r < 3; r++)
#pragma unroll
            for (int s = 0; s < 3; s++) Tm[3 * r + s] = Rk[3 * r] * Rj[s] + Rk[3 * r + 1] * Rj[3 + s] + Rk[3 * r + 2] * Rj[6 + s];
#pragma unroll
          for (int e = 0; e < 9; e++) Rk[e] = Tm[e];
        }
      }
      if (j < 3) {
#pragma unroll
        for (int c = 0; c < 3; c++) { zk[j][c] = Rk[3 * c + 2]; pjk[j][c] = pk[c]; }
        T sj, cj;
        joint_sincos(qv[j], &sj, &cj);
#pragma unroll
        for (int r = 0; r < 3; r++) {
          const T a0 = Rk[3 * r], a1 = Rk[3 * r + 1];
          Rk[3 * r] = cj * a0 + sj * a1;
          Rk[3 * r + 1] = cj * a1 - sj * a0;
        }
      }
    }
    T J[3][3], v[3] = {T(0), T(0), T(0)};
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const T dv[3] = {pk[0] - pjk[j][0], pk[1] - pjk[j][1], pk[2] - pjk[j][2]};
      cross3(zk[j], dv, J[j]);
#pragma unroll
      for (int c = 0; c < 3; c++) v[c] += J[j][c] * qdv[j];
    }
    T f[3];
#pragma unroll
    for (int c = 0; c < 3; c++) {
      const T ep = a.ptarget ? a.ptarget[(size_t)(3 * leg + c) * B + i] - pk[c] : T(0);
      const T ev = a.vtarget ? a.vtarget[(size_t)(3 * leg + c) * B + i] - v[c] : T(0);
      f[c] = a.kp[c] * ep + a.kd[c] * ev;
    }
#pragma unroll
    for (int j = 0; j < 3; j++) tau[j] += J[j][0] * f[0] + J[j][1] * f[1] + J[j][2] * f[2];
  }
}

__global__ void __launch_bounds__(128) qlb_swing_kernel(const SwingArgs a) {
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long B = a.B;
  if (t >= 4ull * B) return;
  const int leg = (int)(t / B);
  const unsigned long long i = t - (unsigned long long)leg * B;
  double tau[3];
  swing_leg_torque(a, leg, i, tau);
#pragma unroll
  for (int j = 0; j < 3; j++) a.tau[(size_t)(3 * leg + j) * B + i] = tau[j];
}

}  // namespace qlb
