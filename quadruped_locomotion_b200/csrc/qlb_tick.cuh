// qlb_tick.cuh - the two kernels around the state-mode solve in one controller tick (qlb_controller_update):
// RosBalanceController::update (ros_balance_controller.cpp:198-716) for B robots.
//
//   prologue (one thread per robot): contact state machine -> limb states + stance mask; the joint-velocity sample
//       goes into the robot's ring of the last kTickRing samples
//   solve    (qlb_solve_state, unchanged): forces and stance-leg torques for that stance mask
//   epilogue (one thread per (robot, leg), consecutive threads = consecutive robots of one leg): stance rows of the
//       persistent efforts from the solve (kept when the solve failed, RBC.cpp:418,455-458), swing rows from the
//       swing-leg dynamics with the acceleration differenced over the ring, then the clamped command (RBC.cpp:450-454)
//
// Arrays of the caller have row pitch n (the robots of this call); arrays the controller owns have row pitch ld (its
// batch size) and are passed already offset to the first robot of the call.
//
// T is the type of the caller's arrays: double (qlb_controller_update) or float (qlb_controller_update_f32).  The state
// the controller owns is double either way: a float qd sample goes into the ring exactly, the solve's float torques
// and the float swing-leg torques are widened into the efforts, and the command is the clamp of the efforts in double,
// rounded to T.  So the two entry points act on one controller and may be mixed from tick to tick.
#pragma once

#include "qlb.h"
#include "qlb_aux.cuh"
#include "qlb_swing.cuh"

namespace qlb {

constexpr int kTickRing = 11;   // joint-velocity samples per robot: the newest and the one 10 periods older

template <typename T>
struct TickArgsT {
  unsigned long long n;    // robots in this call = row pitch of the caller's arrays
  unsigned long long ld;   // row pitch of the controller's arrays
  int head;                // ring slot of this tick's sample; the oldest sample is in slot (head + 1) % kTickRing
  // prologue
  const uint8_t* desired;
  const uint8_t* footstep;   // may be null: every leg supervised
  const uint8_t* contact;
  const T* phase;            // [4][n]
  const T* qd;               // [12][n]
  uint8_t* limb;             // [4][ld]
  uint8_t* refill;           // [ld]: 1 = fill every ring slot with the next sample
  double* ring;              // [kTickRing][12][ld]
  uint8_t* stance;           // [n] out of the prologue, in of the solve and the epilogue
  // epilogue
  const uint32_t* flags;     // [n] of the solve
  const T* tau;              // [12][n] of the solve
  double* efforts;           // [12][ld]
  T* command;                // [12][n]
  double limit;
  SwingArgsT<T> swing;       // B = n, q, qd, qd_front = oldest ring slot with ld_front = ld, targets, gains
};

template <typename T>
__global__ void __launch_bounds__(256) qlb_tick_prologue_kernel(const TickArgsT<T> a) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long n = a.n, ld = a.ld;
  if (i >= n) return;
  const unsigned mask = contact_fsm_robot(i, a.desired[i], a.footstep ? a.footstep[i] : 0xFu, a.contact[i], a.phase, n, a.limb, ld);
  a.stance[i] = (uint8_t)mask;
  const bool refill = a.refill[i] != 0;
  const int s0 = refill ? 0 : a.head, s1 = refill ? kTickRing : a.head + 1;   // every slot, or this tick's
#pragma unroll 1
  for (int s = s0; s < s1; s++) {
    double* slot = a.ring + (size_t)s * 12 * ld + i;
#pragma unroll
    for (int c = 0; c < 12; c++) slot[(size_t)c * ld] = (double)a.qd[(size_t)c * n + i];
  }
  if (refill) a.refill[i] = 0;
}

template <typename T>
__global__ void __launch_bounds__(128) qlb_tick_epilogue_kernel(const TickArgsT<T> a) {
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long n = a.n, ld = a.ld;
  if (t >= 4ull * n) return;
  const int leg = (int)(t / n);
  const unsigned long long i = t - (unsigned long long)leg * n;
  double e[3];
#pragma unroll
  for (int j = 0; j < 3; j++) e[j] = a.efforts[(size_t)(3 * leg + j) * ld + i];
  if ((a.stance[i] >> leg) & 1u) {
    const unsigned status = (a.flags[i] & QLB_FLAG_STATUS_MASK) >> QLB_FLAG_STATUS_SHIFT;
    if (status == QLB_STATE_OK || status == QLB_STATE_NO_STANCE) {
#pragma unroll
      for (int j = 0; j < 3; j++) e[j] = (double)a.tau[(size_t)(3 * leg + j) * n + i];
    }
  } else {
    T tq[3];
    swing_leg_torque(a.swing, leg, i, tq);
    if (isfinite(tq[0]) && isfinite(tq[1]) && isfinite(tq[2])) {
#pragma unroll
      for (int j = 0; j < 3; j++) e[j] = (double)tq[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 3; j++) {
    a.efforts[(size_t)(3 * leg + j) * ld + i] = e[j];
    a.command[(size_t)(3 * leg + j) * n + i] = (T)fmin(fmax(e[j], -a.limit), a.limit);
  }
}

// qlb_controller_reset: robots with mask[i] != 0 (every robot when mask is null) start again as after create.
__global__ void __launch_bounds__(256) qlb_tick_reset_kernel(unsigned long long B, const uint8_t* __restrict__ mask,
                                                             uint8_t* __restrict__ limb, double* __restrict__ efforts,
                                                             uint8_t* __restrict__ refill) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B || (mask && !mask[i])) return;
#pragma unroll
  for (int k = 0; k < 4; k++) limb[(size_t)k * B + i] = QLB_LIMB_INIT;
#pragma unroll
  for (int c = 0; c < 12; c++) efforts[(size_t)c * B + i] = 0.0;
  refill[i] = 1;
}

}  // namespace qlb
