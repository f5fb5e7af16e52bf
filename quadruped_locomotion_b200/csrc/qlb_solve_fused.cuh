// qlb_solve_fused.cuh - building blocks of the fused solve kernel (qlb_solve_single.cuh): staging of the raw input rows
// in shared memory (TMA tensor boxes or cp.async), mbarrier / TMA primitives, and one round of the dual block
// active-set method on the 6x6 dual system.
//
// The rounds are a DUAL BLOCK ACTIVE-SET method (the Goldfarb-Idnani idea with block additions; the dual of
// the QP is a bound-constrained QP in the multipliers and this is the primal active-set method on it):
//   state  (y, u, F): primal iterate, multipliers u >= 0 of the rows in the working set F
//   round  (y+, u+) = solution of the equality-constrained QP for F (the 6x6 Woodbury system);
//          ratio test: the largest step t in [0, 1] towards (y+, u+) that keeps every multiplier >= 0;
//          t < 1: move by t, drop the blocking rows from F;
//          t = 1: move; every violated row joins F (multiplier 0); no violated row -> optimal.
// Each non-zero step increases the dual objective, so no working set repeats: finite, no cycling, and in
// the common cases it takes the same steps as the "repair every violated row" heuristic of round 1 (which
// needed an interior-point pass as a safety net for 1 % of the states).  Measured on 60 000 C3 / C5 states
// (tools/proto/rounds_proto.py): 1.69 / 1.45 rounds per hard state, at most 14, no failure, active set equal to
// the reference solver's on every state.  States that exhaust the round limit (none seen) go to a.list2 for
// the interior-point kernel of qlb_solve_quad.cuh.
//
// Reference path: ContactForceDistribution.cpp:99-136,138-336,385-578,614-625;
// quadrupedkinematics.cpp:143-278,485-552; VirtualModelController.cpp:89-268 (as in qlb_solve_quad.cuh).
#pragma once

#include <cuda.h>

#include "qlb_solve_quad.cuh"

namespace qlb {

#ifndef QLB_SUPER
#define QLB_SUPER 2      // tiles (of eight states) per staged box: TMA boxes are 8 QLB_SUPER states wide
#endif
#ifndef QLB_DBAS_MAX_ROUNDS
#define QLB_DBAS_MAX_ROUNDS 40
#endif

// ---------------------------------------------------------------------------------------------------------
// Staging of the raw input rows: one segment per input array, each a dense [rows][8 states] box.
template <typename real, int MODE, int SUPER>
struct Staging {
  static constexpr int kCols = 8 * SUPER;                                       // states per box
  static constexpr int kRow = kCols * (int)sizeof(real);                        // bytes of one row of a box
  __host__ __device__ static constexpr int align(int x) { return (x + 127) & ~127; }   // TMA destinations: 128-byte aligned
  // wrench mode: q, quat, wrench, mu, normals;  state mode: q, pose, twist, tpose, ttwist, mu, normals.  (Arrays the
  // caller does not pass - mu, normals - are skipped: no transfer, the space stays unused.)
  static constexpr int kNumSeg = (MODE == 1) ? 7 : 5;
  __host__ __device__ static constexpr int rows(int s) {
    return (MODE == 1) ? (s == 0 ? 12 : s == 1 ? 7 : s == 2 ? 6 : s == 3 ? 7 : s == 4 ? 6 : s == 5 ? 4 : 12)
                       : (s == 0 ? 12 : s == 1 ? 4 : s == 2 ? 6 : s == 3 ? 4 : 12);
  }
  // (closed form, no recursion: a recursive constexpr function called with a run-time-looking argument is compiled
  // as a real recursive device function - found in the SASS as CALL/RET, 29 % of all executed instructions)
  static constexpr int kO1 = align(rows(0) * kRow), kO2 = kO1 + align(rows(1) * kRow), kO3 = kO2 + align(rows(2) * kRow),
                       kO4 = kO3 + align(rows(3) * kRow), kO5 = kO4 + align(rows(4) * kRow),
                       kO6 = kO5 + align((MODE == 1 ? rows(5) : 0) * kRow), kO7 = kO6 + align((MODE == 1 ? rows(6) : 0) * kRow);
  __host__ __device__ static constexpr int offset(int s) {
    return s == 0 ? 0 : s == 1 ? kO1 : s == 2 ? kO2 : s == 3 ? kO3 : s == 4 ? kO4 : s == 5 ? kO5 : s == 6 ? kO6 : kO7;
  }
  static constexpr int kMaskOff = (MODE == 1) ? kO7 : kO5;     // the stance masks of the box: one byte per state
  static constexpr int kBytes = kMaskOff + 128;
  static constexpr int kSegMu = (MODE == 1) ? 5 : 3;
  static constexpr int kSegNrm = kSegMu + 1;
  // the global array behind segment s (nullptr: not passed)
  template <typename Args>
  __host__ __device__ static const real* source(const Args& a, const int s) {
    if (MODE == 1) return s == 0 ? a.q : s == 1 ? a.pose : s == 2 ? a.twist : s == 3 ? a.tpose : s == 4 ? a.ttwist : s == 5 ? a.mu : a.normals;
    return s == 0 ? a.q : s == 1 ? a.quat : s == 2 ? a.wrench : s == 3 ? a.mu : a.normals;
  }
};

// Tensor maps of the input arrays of one call (built on the host, qlb_api.cu), in Staging segment order.
struct alignas(64) FusedMaps {
  CUtensorMap seg[7];
  CUtensorMap mask;    // rank 1, uint8, boxes of 8 SUPER states
};

// ---------------------------------------------------------------------------------------------------------
// mbarrier / TMA / cp.async primitives (shared::cta addresses as 32-bit)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0u;
}
// Whole warp.  The exit is decided by a vote, so the warp leaves the loop converged (a per-lane exit, or a trap
// inside the loop, makes the compiler treat everything after it as possibly divergent: every later shuffle then
// gets an out-of-line slow path and the kernel doubles in size).  Bounded: a transfer that never completes (a bad
// tensor map) lets the kernel finish with wrong data instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  for (unsigned spins = 0; spins < (1u << 24); spins++) {
    const bool ok = mbar_try_wait(bar, parity);
    if (__all_sync(kFull, ok)) break;
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const CUtensorMap* map, int c0, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.1d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2}], [%3];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(bar) : "memory");
}
// four bytes, of which only `valid` (0..4) are read from global memory; the rest is zero-filled
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void* src, int valid) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(valid) : "memory");
}
__device__ __forceinline__ void cp_async_elem(uint32_t dst, const double* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_elem(uint32_t dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// the j-th (0-based) set bit of m, or -1
__device__ __forceinline__ int nth_set_bit(unsigned m, const int j) {
#pragma unroll
  for (int i = 0; i < 7; i++)
    if (i < j) m &= m - 1u;
  return m ? (__ffs(m) - 1) : -1;
}

// Issue the loads of box `box` (8 SUPER consecutive states) into this warp's staging buffer.
// TMA: lane 0 arms the mbarrier with the byte count and issues one tensor box per input array (out-of-range
// columns of the last box are zero-filled by the unit).  Otherwise (batch size or pointers not 16-byte
// aligned): every lane copies its share with 8-/4-byte cp.async, column index clamped to B - 1.
template <typename real, int MODE, int SUPER, bool TMA>
__device__ __forceinline__ void stage_issue(const SolveArgsT<real>& a, const FusedMaps& maps, const unsigned long long box,
                                            unsigned char* stage, const uint32_t bar, const int lane) {
  using SG = Staging<real, MODE, SUPER>;
  const real* src[SG::kNumSeg];
#pragma unroll
  for (int s = 0; s < SG::kNumSeg; s++) src[s] = SG::source(a, s);
  if (TMA) {
    if (lane == 0) {
      uint32_t bytes = 0;
#pragma unroll
      for (int s = 0; s < SG::kNumSeg; s++)
        if (src[s] != nullptr) bytes += SG::rows(s) * SG::kRow;
      bytes += SG::kCols;   // the stance masks
      mbar_expect_tx(bar, bytes);
      const uint32_t dst = smem_u32(stage);
#pragma unroll
      for (int s = 0; s < SG::kNumSeg; s++)
        if (src[s] != nullptr) tma_load_2d(dst + SG::offset(s), &maps.seg[s], (int)(box * (unsigned long long)SG::kCols), 0, bar);
      tma_load_1d(dst + SG::kMaskOff, &maps.mask, (int)(box * (unsigned long long)SG::kCols), bar);
    }
  } else {
    const unsigned long long B = a.B;
    constexpr int kRowsPerPass = 32 / SG::kCols;
    const int col = lane % SG::kCols;
    unsigned long long bx = box * (unsigned long long)SG::kCols + col;
    if (bx >= B) bx = B - 1;
#pragma unroll
    for (int s = 0; s < SG::kNumSeg; s++) {
      if (src[s] == nullptr) continue;
      const uint32_t dst = smem_u32(stage) + SG::offset(s);
#pragma unroll
      for (int r0 = 0; r0 < SG::rows(s); r0 += kRowsPerPass) {
        const int r = r0 + lane / SG::kCols;
        if (r < SG::rows(s)) cp_async_elem(dst + (r * SG::kCols + col) * (int)sizeof(real), src[s] + (size_t)r * B + bx);
      }
    }
    // stance masks: four bytes per lane when the array is word-aligned (bytes past the end of the batch are not read),
    // else byte by byte (synchronous; only for callers with an odd mask pointer)
    const unsigned long long m0 = box * (unsigned long long)SG::kCols;
    if ((reinterpret_cast<uintptr_t>(a.mask) & 3u) == 0) {
      if (lane < SG::kCols / 4) {
        const unsigned long long first = m0 + 4ull * lane;
        const int valid = first >= B ? 0 : (B - first < 4 ? (int)(B - first) : 4);
        cp_async_4(smem_u32(stage) + SG::kMaskOff + 4 * lane, a.mask + (valid ? first : 0), valid);
      }
    } else if (lane < SG::kCols) {
      stage[SG::kMaskOff + lane] = (m0 + lane < B) ? a.mask[m0 + lane] : (unsigned char)0;
    }
    cp_async_commit();
  }
}

// The raw inputs of this lane's state (column `col` of the staged box) in the layout RawIn of qlb_solve_quad.cuh.
template <typename real, int MODE, int SUPER>
__device__ __forceinline__ void stage_read(const SolveArgsT<real>& a, const unsigned char* stage, const real mu_default,
                                           const int leg, const int col, const unsigned long long bq, RawIn<real, MODE>& in) {
  using SG = Staging<real, MODE, SUPER>;
  auto at = [&](const int seg, const int row) { return reinterpret_cast<const real*>(stage + SG::offset(seg))[row * SG::kCols + col]; };
#pragma unroll
  for (int j = 0; j < 3; j++) in.qj[j] = at(0, 3 * leg + j);
  if (MODE == 1) {
#pragma unroll
    for (int r = 0; r < 7; r++) { in.pose[r] = at(1, r); in.tp[r] = at(3, r); }
#pragma unroll
    for (int r = 0; r < 6; r++) { in.tw[r] = at(2, r); in.tt[r] = at(4, r); }
  } else {
#pragma unroll
    for (int r = 0; r < 4; r++) in.quat[r] = at(1, r);
#pragma unroll
    for (int r = 0; r < 6; r++) in.b[r] = at(2, r);
  }
  in.mask = (unsigned)stage[SG::kMaskOff + col] & 0xFu;
  in.mu = (a.mu != nullptr) ? at(SG::kSegMu, leg) : mu_default;
  in.nw[0] = real(0.0); in.nw[1] = real(0.0); in.nw[2] = real(1.0);
  if (a.normals != nullptr) {
#pragma unroll
    for (int c = 0; c < 3; c++) in.nw[c] = at(SG::kSegNrm, 3 * leg + c);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Registers of one lane while its quad runs rounds on a hard state.
template <typename creal>
struct RoundState {
  creal At[3][6];   // the leg's block of the wrench map in contact coordinates (zero for a swing leg)
  creal mu;
  creal y[3];       // primal iterate (y_n, y_1, y_2)
  creal u[3];       // multipliers of the rows held by the slots n, 1, 2 (0 where the slot is free)
  int a0, sg1, sg2; // working set: y_n pinned at F_min; y_1 = sg1 mu y_n; y_2 = sg2 mu y_n
  unsigned mask;
  bool alive;
  int rounds;
  unsigned idx;
};

// One round of the dual block active-set method for the states held by the eight quads (whole warp).
// b: the quad's desired wrench in shared memory (element r at b[r * bstride]).
// done: the iterate is optimal (KKT verified).  fail: factorisation failed or the round limit is reached.
template <typename creal>
__device__ __forceinline__ void dbas_round(RoundState<creal>& q, const creal* b, const int bstride, const CoreConst<creal>& cc,
                                           const int leg, const bool active, bool& done, bool& fail) {
  const bool alive = q.alive && active;
  const creal mu = q.mu;
  const creal (&At)[3][6] = q.At;
  const int a0 = q.a0, sg1 = q.sg1, sg2 = q.sg2;
  // ---- reduced columns of the equality-constrained QP for the working set
  // (a slot that is not free gets the weight al = 0: its column needs no masking - it enters the system and the
  // recovery of y+ only through al - and the columns of a swing leg are zero anyway)
  creal v[3][6], al[3], r6[6];
  {
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
      v[0][r] = cn;
      v[1][r] = At[1][r];
      v[2][r] = At[2][r];
      r6[r] = fma(-pin, cn, (leg == 0 && active) ? b[r * bstride] : creal(0.0));
    }
  }
  // ---- the 6x6 system, summed over the quad
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
  bool pd;
  if (Tol<creal>::refine) {
    pd = chol6_thread(N, rdg);
    creal rhs6[6];
#pragma unroll
    for (int r = 0; r < 6; r++) rhs6[r] = r6[r];
    solve6_thread(N, rdg, r6);
    refine6(N, rdg, v, al, cc.sinv, rhs6, r6);
  } else {
    pd = ldl6_thread(N, rdg);
    ldl6_solve(N, rdg, r6);   // r6 <- t = S (b - A y+)
  }
  // ---- y+ and the multipliers u+ of the working set
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
  // gradient w y - A_k' t; stationarity g = D~' u gives the multipliers of the active rows
  const creal g0 = fma(cc.W, yp[0], -att[0]), g1 = fma(cc.W, yp[1], -att[1]), g2 = fma(cc.W, yp[2], -att[2]);
  creal up[3];
  up[1] = (alive && sg1 != 0) ? -sg1 * g1 : creal(0.0);
  up[2] = (alive && sg2 != 0) ? -sg2 * g2 : creal(0.0);
  up[0] = (alive && a0 != 0) ? g0 - mu * (up[1] + up[2]) : creal(0.0);
  // ---- ratio test: the step towards (y+, u+) that keeps every multiplier non-negative
  // (the scale of the gradient w y - A_k' t: the multipliers scale with W wherever the W term decides the internal forces)
  const creal tol_u = Tol<creal>::mult() * quad_max_abs(att[0], att[1], att[2], cc.W * lane_max_abs(yp[0], yp[1], yp[2]));
  const bool act[3] = {alive && a0 != 0, alive && sg1 != 0, alive && sg2 != 0};
  creal tr[3], tl = creal(2.0);
#pragma unroll
  for (int s = 0; s < 3; s++) {
    tr[s] = creal(2.0);
    if (act[s] && up[s] < -tol_u) tr[s] = (q.u[s] > creal(0.0)) ? q.u[s] * fast_rcp(q.u[s] - up[s]) : creal(0.0);
    tl = fmin(tl, tr[s]);
  }
  creal tq = tl;
  tq = fmin(tq, __shfl_xor_sync(kFull, tq, 1));
  tq = fmin(tq, __shfl_xor_sync(kFull, tq, 2));
  const bool blocked = tq < creal(1.5);   // some multiplier turns negative on the way (tr <= 1 by construction)
  const creal step = blocked ? fmin(tq, creal(1.0)) : creal(1.0);
  // ---- move
  creal yn3[3], un3[3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    yn3[c] = blocked ? fma(step, yp[c] - q.y[c], q.y[c]) : yp[c];
    un3[c] = blocked ? fmax(fma(step, up[c] - q.u[c], q.u[c]), creal(0.0)) : fmax(up[c], creal(0.0));
  }
  int na0 = a0, nsg1 = sg1, nsg2 = sg2;
  if (blocked) {
    // drop the blocking rows (all rows that share the smallest ratio: the fresh rows with a negative multiplier at t = 0)
    if (act[0] && tr[0] <= tq) { na0 = 0; un3[0] = creal(0.0); }
    if (act[1] && tr[1] <= tq) { nsg1 = 0; un3[1] = creal(0.0); }
    if (act[2] && tr[2] <= tq) { nsg2 = 0; un3[2] = creal(0.0); }
  }
  // ---- at the minimiser of the face: which rows does it violate?
  creal e[5];
  leg_rows(yn3[0], yn3[1], yn3[2], mu, e);
  e[0] -= cc.fmin;
  const creal tol_s = Tol<creal>::feas() * quad_max_abs(yn3[0], yn3[1], yn3[2]);
  bool viol = false;
  if (!blocked && alive) {
    if (na0 == 0 && e[0] < -tol_s) { na0 = 1; viol = true; }
    if (nsg1 == 0) {
      const bool v1 = e[1] < -tol_s, v2 = e[2] < -tol_s;
      if (v1 || v2) { nsg1 = (v1 && (!v2 || e[1] <= e[2])) ? -1 : 1; viol = true; }
    }
    if (nsg2 == 0) {
      const bool v3 = e[3] < -tol_s, v4 = e[4] < -tol_s;
      if (v3 || v4) { nsg2 = (v3 && (!v4 || e[3] <= e[4])) ? -1 : 1; viol = true; }
    }
  }
  const bool quad_viol = quad_or(viol ? 1u : 0u) != 0u;
  done = false; fail = false;
  if (active) {
    q.rounds++;
    if (!pd) {
      fail = true;
    } else {
      q.y[0] = yn3[0]; q.y[1] = yn3[1]; q.y[2] = yn3[2];
      q.u[0] = un3[0]; q.u[1] = un3[1]; q.u[2] = un3[2];
      if (!blocked && !quad_viol) {
        done = true;            // the working set (q.a0, q.sg1, q.sg2) is the active set
      } else {
        q.a0 = na0; q.sg1 = nsg1; q.sg2 = nsg2;
        if (q.rounds >= QLB_DBAS_MAX_ROUNDS) fail = true;
      }
    }
  }
}

}  // namespace qlb
