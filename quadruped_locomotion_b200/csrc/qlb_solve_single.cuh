// qlb_solve_single.cuh - the fused solve kernel: tile phase and round phase in ONE persistent kernel, every warp
// autonomous, the states that need active-set rounds parked in a per-warp shared-memory stash (nothing goes back to
// HBM between the two phases; the outputs of those states are overwritten while their lines are still in L2).
//
//   tile phase   eight consecutive states per step (one leg per lane, as in qlb_solve_quad.cuh).  The raw SoA input
//                rows of 8 QLB_SUPER states are staged in shared memory by the TMA unit (one cp.async.bulk.tensor box
//                per input array, completion on a per-warp mbarrier) while the previous box is computed.
//                Kinematics, friction frames, wrench map, the unconstrained minimiser.  States whose minimiser is
//                feasible (72 % of config C3) are finished.  The record of a "hard" state - normal and first tangent
//                of the friction frame, foot position, Jacobian, gravity torques, the minimiser - goes into one of the
//                warp's CAP stash slots (the Jacobian of every state of the tile is written straight into the slot its
//                quad would keep, which is why a tile needs eight free slots).
//   round phase  entered when fewer than eight slots are free: each quad takes a pending state and runs rounds of
//                the dual block active-set method (qlb_solve_fused.cuh); a quad that finishes writes its outputs and
//                takes the next pending slot, so the eight quads stay busy whatever the number of rounds their states
//                need (measured: 93 % of the quad-rounds executed are useful); when fewer than min(CAP - 7,
//                QLB_ROUND_LOW) states are left the unfinished ones are written back (iterate, multipliers, working
//                set) and the warp fetches tiles again.
// Launch: one CTA of twelve warps per SM, 168 registers, 222 KB of shared memory (staging buffer, stash and loop-control
// words per warp; parameters, solver constants, leg model and one mbarrier per warp per CTA).
#pragma once

#include "qlb_solve_fused.cuh"

namespace qlb {

// Launch shape: ONE CTA of twelve warps per SM (168 registers, three warps per scheduler).  Measured on 2^20 C3 states:
//   2 CTAs x 4 warps (194 registers)  0.576 ms      3 CTAs x 4 warps  0.550 ms      1 CTA x 12 warps  0.490 ms
//   2 CTAs x 5 warps                  0.640 ms (schedulers loaded 3-3-2-2, spills)
// (while the kernel still spilled at 168 registers, two CTAs of four warps were the fastest: 0.613 against 0.667 ms)
#ifndef QLB_FUSED_MIN_CTAS
#define QLB_FUSED_MIN_CTAS 1
#endif
#ifndef QLB_FUSED_MIN_CTAS_F32
#define QLB_FUSED_MIN_CTAS_F32 1
#endif
#ifndef QLB_FUSED_THREADS
#define QLB_FUSED_THREADS 384
#endif
#ifndef QLB_DYNAMIC_PART
#define QLB_DYNAMIC_PART 4       // one box in this many is claimed dynamically (the rest is dealt out statically)
#endif
#ifndef QLB_STASH_CAP
#define QLB_STASH_CAP 22         // stash slots per warp (as many as the shared-memory budget allows, at most this)
#endif
#ifndef QLB_ROUND_LOW
#define QLB_ROUND_LOW 8          // the round phase runs until fewer than this many states are pending: all eight quads
#endif                           // stay busy
constexpr int kFusedThreads = QLB_FUSED_THREADS;
constexpr int kFusedWarps = kFusedThreads / 32;
template <typename real> constexpr int fused_min_ctas() { return sizeof(real) == 4 ? QLB_FUSED_MIN_CTAS_F32 : QLB_FUSED_MIN_CTAS; }
// shared memory per CTA: fused_min_ctas CTAs per SM (228 KB, 1 KB reserved per CTA)
template <typename real> constexpr int fused_smem_budget() { return (228 / fused_min_ctas<real>() - 1) * 1024; }

// ---------------------------------------------------------------------------------------------------------
// The stash of one warp: CAP entries.  Per-lane planes (element k of the entry in slot s, leg l at
// plane[k * 4 CAP + 4 s + l]) and a per-entry header.
// The entry is kept small - the number of slots decides how full the quads of a round phase run (measured on 2^20 C3
// states, two CTAs of four warps: 12 slots 0.629 ms, 16 slots 0.573 ms, 22 slots 0.576 ms).  Per leg: normal and first
// tangent of the friction frame (6; the second tangent is rebuilt from them when the entry is loaded), foot (3), mu,
// y (3), u (3).  (Going further - the tangents rebuilt from the normal and the base frame's y axis, the multipliers as
// FP32: 16 slots instead of 14 - measured no gain for FP64 arrays and 4 % loss for FP32 arrays, which have room anyway.)
constexpr int kStashLane = 16;
constexpr int kSlFoot = 6, kSlMu = 9, kSlY = 10, kSlU = 13;
template <typename real, typename creal, int CAP>
struct StashLayout {
  static constexpr int kQ = 4 * CAP;
  static constexpr int kLaneBytes = kStashLane * kQ * (int)sizeof(creal);
  static constexpr int kJBytes = 12 * kQ * (int)sizeof(real);
  static constexpr int kBBytes = 6 * CAP * (int)sizeof(creal);
  static constexpr int kHBytes = 4 * CAP * 4;
  static constexpr int kBytes = ((kLaneBytes + kJBytes + kBBytes + kHBytes) + 15) & ~15;
};

template <typename real, typename creal, int MODE, int SUPER>
struct FusedLayout {
  // fixed part: parameter block, solver constants, one mbarrier per warp (the leg-model table is a static array)
  static constexpr int kCtlWords = 8;   // per warp: loop-control words that are read once per box (kept out of the registers)
  static constexpr int kBarBytes = (kFusedWarps * 8 + 63) & ~63;   // one mbarrier per warp
  static constexpr int kFixed = ((((int)sizeof(DeviceParamsT<real>) + 15) & ~15) + (((int)sizeof(CoreConst<creal>) + 15) & ~15) + kBarBytes +
                                 kFusedWarps * kCtlWords * 4 + 127) & ~127;
  static constexpr int kStatic = (int)sizeof(DeviceModelT<double>) + 128;
  static constexpr int kStage = Staging<real, MODE, SUPER>::kBytes;
  static constexpr int stash_bytes(int c) {
    return ((kStashLane * 4 * c * (int)sizeof(creal) + 12 * 4 * c * (int)sizeof(real) + 6 * c * (int)sizeof(creal) + 16 * c) + 15) & ~15;
  }
  static constexpr int warp_bytes(int c) { return (kStage + stash_bytes(c) + 127) & ~127; }
  static constexpr int cap_for(int c) { return (kStatic + kFixed + kFusedWarps * warp_bytes(c) <= fused_smem_budget<real>() || c <= 8) ? c : cap_for(c - 1); }
  static constexpr int kCap = cap_for(QLB_STASH_CAP);
  static_assert(kCap >= 10, "stash too small");
  static_assert(stash_bytes(kCap) == StashLayout<real, creal, kCap>::kBytes, "layout mismatch");
  static constexpr int kWarpBytes = warp_bytes(kCap);
  static constexpr int kTotal = kFixed + kFusedWarps * kWarpBytes;   // dynamic shared memory of the kernel
  static_assert(kStatic + kTotal <= fused_smem_budget<real>(), "shared memory budget");
};

template <typename real, typename creal, int CAP>
struct WarpStash {
  creal* sl;      // [kStashLane][4 CAP]
  real* sj;       // [12][4 CAP]   Jacobian (9) and gravity torques (3); also the scratch of the tile phase
  creal* sb;      // [6][CAP]      desired wrench
  uint32_t* sh;   // [4][CAP]      state index; mask | pattern << 4 | rounds << 24; two spare words
  __device__ WarpStash(unsigned char* base) {
    using SL = StashLayout<real, creal, CAP>;
    sl = reinterpret_cast<creal*>(base);
    sj = reinterpret_cast<real*>(base + SL::kLaneBytes);
    sb = reinterpret_cast<creal*>(base + SL::kLaneBytes + SL::kJBytes);
    sh = reinterpret_cast<uint32_t*>(base + SL::kLaneBytes + SL::kJBytes + SL::kBBytes);
  }
};


template <typename real, typename creal, int CAP>
__device__ __forceinline__ void stash_load(const WarpStash<real, creal, CAP>& ws, const int slot, const int leg, RoundState<creal>& q) {
  constexpr int Q = 4 * CAP;
  const int e = 4 * slot + leg;
  const uint32_t w1 = ws.sh[CAP + slot];
  q.idx = ws.sh[slot];
  q.mask = w1 & 0xFu;
  q.alive = (w1 >> leg) & 1u;
  q.rounds = (int)(w1 >> 24);
  const unsigned pat = (w1 >> (4 + 5 * leg)) & 31u;
  q.a0 = (int)(pat & 1u);
  q.sg1 = ((pat >> 1) & 3u) == 1u ? -1 : (((pat >> 1) & 3u) == 2u ? 1 : 0);
  q.sg2 = ((pat >> 3) & 3u) == 1u ? -1 : (((pat >> 3) & 3u) == 2u ? 1 : 0);
  creal foot[3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    q.At[0][c] = ws.sl[c * Q + e];
    q.At[1][c] = ws.sl[(3 + c) * Q + e];
    foot[c] = ws.sl[(kSlFoot + c) * Q + e];
  }
  {
    // second tangent t2 = n x t1, normalised - the operations of quad_setup (CFD.cpp:306-309); a swing leg's rows are zero
    creal t2[3];
    t2[0] = q.At[0][1] * q.At[1][2] - q.At[0][2] * q.At[1][1];
    t2[1] = q.At[0][2] * q.At[1][0] - q.At[0][0] * q.At[1][2];
    t2[2] = q.At[0][0] * q.At[1][1] - q.At[0][1] * q.At[1][0];
    const creal rn = q.alive ? fast_rsqrt(t2[0] * t2[0] + t2[1] * t2[1] + t2[2] * t2[2]) : creal(0.0);
#pragma unroll
    for (int c = 0; c < 3; c++) q.At[2][c] = t2[c] * rn;
  }
  q.mu = ws.sl[kSlMu * Q + e];
#pragma unroll
  for (int c = 0; c < 3; c++) { q.y[c] = ws.sl[(kSlY + c) * Q + e]; q.u[c] = ws.sl[(kSlU + c) * Q + e]; }
  // torque rows of the wrench map: r x e_c (zero for a swing leg: its force rows are stored as zero)
#pragma unroll
  for (int c = 0; c < 3; c++) {
    q.At[c][3] = foot[1] * q.At[c][2] - foot[2] * q.At[c][1];
    q.At[c][4] = foot[2] * q.At[c][0] - foot[0] * q.At[c][2];
    q.At[c][5] = foot[0] * q.At[c][1] - foot[1] * q.At[c][0];
  }
}

__device__ __forceinline__ unsigned pattern_bits(const int a0, const int sg1, const int sg2) {
  return (a0 != 0 ? 1u : 0u) | (sg1 == -1 ? 2u : (sg1 == 1 ? 4u : 0u)) | (sg2 == -1 ? 8u : (sg2 == 1 ? 16u : 0u));
}

// Write the iterate of an unfinished state back to its slot (the fixed part of the entry is still there).
template <typename real, typename creal, int CAP>
__device__ __forceinline__ void stash_save(const WarpStash<real, creal, CAP>& ws, const int slot, const int leg, const RoundState<creal>& q,
                                           const bool doit) {
  constexpr int Q = 4 * CAP;
  const unsigned pat = quad_or(pattern_bits(q.a0, q.sg1, q.sg2) << (5 * leg));   // whole warp
  if (doit) {
    const int e = 4 * slot + leg;
#pragma unroll
    for (int c = 0; c < 3; c++) { ws.sl[(kSlY + c) * Q + e] = q.y[c]; ws.sl[(kSlU + c) * Q + e] = q.u[c]; }
    if (leg == 0) ws.sh[CAP + slot] = q.mask | (pat << 4) | ((unsigned)q.rounds << 24);
  }
}

// The round phase of one warp (see the header).  occ: bit s = slot s holds a pending state.
template <typename real, typename creal, int CAP>
__device__ __forceinline__ void round_phase(const SolveArgsT<real>& a, const CoreConst<creal>& cc, const WarpStash<real, creal, CAP>& ws,
                                            unsigned& occ, const bool final, const int run_min, const int lane, const int leg,
                                            const int quad) {
  constexpr int Q = 4 * CAP;
  unsigned unassigned = occ;
  RoundState<creal> q;
#pragma unroll
  for (int c = 0; c < 3; c++) {
#pragma unroll
    for (int r = 0; r < 6; r++) q.At[c][r] = creal(0.0);
    q.y[c] = creal(0.0); q.u[c] = creal(0.0);
  }
  q.mu = creal(0.0); q.a0 = 0; q.sg1 = 0; q.sg2 = 0; q.mask = 0u; q.alive = false; q.rounds = 0; q.idx = 0u;
  int slot = nth_set_bit(unassigned, quad);
  bool active = slot >= 0;
  {
    const int ntake = min(8, __popc(unassigned));
#pragma unroll 1
    for (int i = 0; i < ntake; i++) unassigned &= unassigned - 1u;   // the eight lowest pending slots are taken
  }
  bool fresh = active;   // this lane's quad has been handed a slot whose entry is not in registers yet
#pragma unroll 1
  for (;;) {
    if (fresh) stash_load(ws, slot, leg, q);   // (one copy of the load code: 56 instructions less, 1.8 % faster)
    fresh = false;
    bool done, fail;
    const int bslot = active ? slot : 0;
    dbas_round<creal>(q, ws.sb + bslot, CAP, cc, leg, active, done, fail);
    const bool leave = active && (done || fail);
    // ---- finished states: forces, torques, net wrench, flags (whole warp: quad shuffles inside)
    if (__any_sync(kFull, leave)) {
      LegSetup<creal> L;
#pragma unroll
      for (int c = 0; c < 3; c++) {
#pragma unroll
        for (int r = 0; r < 6; r++) L.At[c][r] = q.At[c][r];
      }
      L.alive = q.alive; L.mask = q.mask;
      const int oslot = active ? slot : 0;
      quad_output<real, creal, real>(a, L, q.y, q.a0, q.sg1, q.sg2, 0, q.rounds, (unsigned long long)q.idx, active && done, leg,
                               ws.sj + 4 * oslot + leg, Q);
      // not verified within the round limit (or a factorisation failed): the interior-point kernel takes the state
      const unsigned fm = __ballot_sync(kFull, active && fail && leg == 0);
      if (fm != 0u) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(a.list2_count, __popc(fm));
        base = __shfl_sync(kFull, base, 0);
        if (active && fail && leg == 0) a.list2[base + __popc(fm & ((1u << lane) - 1u))] = q.idx;
      }
      // release the slots, hand the next pending states to the quads that became free
      const unsigned freed = __reduce_or_sync(kFull, leave ? (1u << slot) : 0u);
      occ &= ~freed;
      const unsigned wm = __ballot_sync(kFull, leave && leg == 0);
      const int rank = __popc(wm & ((1u << (lane & ~3)) - 1u));
      __syncwarp();
      if (leave) {
        slot = nth_set_bit(unassigned, rank);
        active = slot >= 0;
        fresh = active;
      }
      {
        const int ntake = min(__popc(wm), __popc(unassigned));
#pragma unroll 1
        for (int i = 0; i < ntake; i++) unassigned &= unassigned - 1u;
      }
    }
    const int nact = __popc(__ballot_sync(kFull, active && leg == 0));
    if (nact == 0) break;
    if (!final && nact + __popc(unassigned) < run_min) {
      // too few states left to keep the warp busy: park the unfinished ones and fetch more tiles
      // (a quad that has just been handed a slot has not loaded it: that entry is still as it was parked)
      stash_save(ws, active ? slot : 0, leg, q, active && !fresh);
      break;
    }
  }
  __syncwarp();
}

// ---------------------------------------------------------------------------------------------------------
template <typename real, typename creal, int MODE, int SUPER, bool TMA>
__global__ void __launch_bounds__(kFusedThreads, fused_min_ctas<real>())
qlb_single_kernel(const SolveArgsT<real> a, const __grid_constant__ FusedMaps maps) {
  using FL = FusedLayout<real, creal, MODE, SUPER>;
  constexpr int CAP = FL::kCap;
  constexpr int Q = 4 * CAP;
  constexpr int kRunMin = CAP - 7;            // a tile needs eight free slots: the round phase starts at CAP - 7 pending ...
  constexpr int kRunLow = QLB_ROUND_LOW < kRunMin ? QLB_ROUND_LOW : kRunMin;   // ... and runs until fewer than this are left
  constexpr int kCols = 8 * SUPER;
  extern __shared__ __align__(128) unsigned char smem[];
  DeviceParamsT<real>& prm = *reinterpret_cast<DeviceParamsT<real>*>(smem);
  CoreConst<creal>& cc = *reinterpret_cast<CoreConst<creal>*>(smem + ((sizeof(DeviceParamsT<real>) + 15) & ~15));
  static_assert(((sizeof(DeviceParamsT<real>) + 15) & ~15) + sizeof(CoreConst<creal>) + FL::kBarBytes + kFusedWarps * FL::kCtlWords * 4 <= FL::kFixed, "fixed part");
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + FL::kFixed - FL::kBarBytes);
  volatile unsigned* ctl = reinterpret_cast<volatile unsigned*>(smem + FL::kFixed - FL::kBarBytes - kFusedWarps * FL::kCtlWords * 4) +
                           (threadIdx.x >> 5) * FL::kCtlWords;   // [0] share [1] dyn_base [2] taken [3] nbox [4] B
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int leg = lane & 3, quad = lane >> 2;
  unsigned char* wbase = smem + FL::kFixed + warp * FL::kWarpBytes;
  unsigned char* stage = wbase;
  const WarpStash<real, creal, CAP> ws(wbase + FL::kStage);
  const uint32_t bar = smem_u32(&bars[warp]);
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a.params);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&prm);
    for (int i = threadIdx.x; i < (int)(sizeof(DeviceParamsT<real>) / 4); i += blockDim.x) dst[i] = src[i];
    cc.load(a.params64);
    load_model_to_smem(a.model);
    if (TMA && lane == 0) {
      mbar_init(bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
  }
  __syncthreads();
  // Box and state numbers are 32-bit (B < 2^32), and what the loop needs only once per box - its share of the boxes,
  // how many it has taken, the totals - lives in shared-memory control words, not in loop-carried registers: the FP32
  // twin runs with 168 registers and spilled exactly these to local memory (long-scoreboard stalls behind a small L1).
  const unsigned nbox = (unsigned)((a.B + kCols - 1) / kCols);
  unsigned occ = 0u;           // pending slots of the stash (warp-uniform)

  // Work distribution: the first three quarters of the boxes are dealt out to the warps of the grid round robin
  // (box b to warp b mod #warps: no atomics, no latency, and neighbouring boxes - whose states are correlated in a
  // sweep of perturbations around nominal states - go to different warps); the last quarter is claimed dynamically,
  // one atomic per box, issued a whole box ahead - its result stays in lane 0 and is broadcast only when the box number is needed - so warps that
  // drew cheap states take more of it.  (The stance masks travel with the staged box: a loop-carried register loaded
  // from global memory gets spilled right behind its load, which exposes the full latency.)
  const unsigned nwarps = gridDim.x * kFusedWarps;
  const unsigned gwarp = blockIdx.x * kFusedWarps + warp;
  const unsigned share = (nbox - nbox / QLB_DYNAMIC_PART) / nwarps;     // static boxes per warp
  const unsigned dyn_base = share * nwarps;              // first dynamically claimed box
  // [2]: boxes started, [5]: tile of the current box, [6]: phase bit of the staging barrier
  if (lane == 0) { ctl[0] = share; ctl[1] = dyn_base; ctl[2] = 0u; ctl[3] = nbox; ctl[4] = (unsigned)a.B; ctl[5] = 0u; ctl[6] = 0u; }
  __syncwarp();
  auto claim_raw = [&](const bool doit) -> unsigned {   // 32 bits: the value is carried through the whole tile body
    unsigned b = 0;
    if (lane == 0 && doit) b = atomicAdd(reinterpret_cast<unsigned*>(a.counter), 1u);
    return b;
  };
  unsigned pending_claim = claim_raw(share <= 1);
  unsigned cur;
  {
    // (box numbers go through a broadcast from lane 0 even when every lane computes the same value: the compiler
    // then knows they are warp-uniform; a box number derived from threadIdx would make it treat the whole tile body
    // as divergent code and give every shuffle an out-of-line slow path)
    cur = __shfl_sync(kFull, share > 0 ? gwarp : dyn_base + pending_claim, 0);
    if (share == 0) pending_claim = claim_raw(true);
  }
  if (cur < nbox) stage_issue<real, MODE, SUPER, TMA>(a, maps, cur, stage, bar, lane);
  if (lane == 0) ctl[5] = (cur < nbox) ? 0x200u : 0u;
  __syncwarp();
  unsigned nxt = 0;
#pragma unroll 1
  for (;;) {
    // (control words go through a broadcast: the compiler must see warp-uniform values in everything that steers the loop)
    // ONE control word steers the step (one shared-memory read and one broadcast in front of the tile, not three):
    // bits 0-7 tile of the current box, bit 8 phase of the staging barrier, bit 9 "there is a current box"
    const unsigned cw = __shfl_sync(kFull, ctl[5], 0);
    const bool have = (cw & 0x200u) != 0u;
    if (have) {
      const int sub = (int)(cw & 0xffu);
      const unsigned cw_wait = (sub == 0 && TMA) ? (cw ^ 0x100u) : cw;   // the wait below consumes one barrier phase
      if (sub + 1 < SUPER && lane == 0) ctl[5] = cw_wait + 1u;           // (the last tile of a box writes the word below)
      if (sub == 0) {
        if (TMA) mbar_wait(bar, (cw >> 8) & 1u);
        else { cp_async_wait_all(); __syncwarp(); }
      }
      const int col = sub * 8 + quad;
      const unsigned s0 = cur * kCols + col, Bu = ctl[4];
      const bool valid = s0 < Bu;
      const unsigned bq = valid ? s0 : (Bu - 1u);
      RawIn<real, MODE> in;
      stage_read<real, MODE, SUPER>(a, stage, prm.mu_default, leg, col, bq, in);
      if (!valid) in.mask = 0u;
      if (sub == SUPER - 1) {
        __syncwarp();     // every lane has read the last tile of the box: the next box may land in the buffer
        const unsigned taken = __shfl_sync(kFull, ctl[2], 0) + 1u, shr = __shfl_sync(kFull, ctl[0], 0);
        if (lane == 0) ctl[2] = taken;
        nxt = __shfl_sync(kFull, taken < shr ? blockIdx.x * kFusedWarps + warp + taken * (gridDim.x * kFusedWarps) : ctl[1] + pending_claim, 0);
        // the claim for the box after `nxt`: needed once the static share is used up
        pending_claim = claim_raw(taken + 1 >= shr);
        const bool more = nxt < __shfl_sync(kFull, ctl[3], 0);
        if (lane == 0) ctl[5] = (cw_wait & 0x100u) | (more ? 0x200u : 0u);
        if (more) stage_issue<real, MODE, SUPER, TMA>(a, maps, nxt, stage, bar, lane);
      }
      // ---- kinematics and QP data; the Jacobian goes straight into the slot this quad would keep
      const int slot = nth_set_bit(~occ & ((1u << CAP) - 1u), quad);
      LegSetup<creal> L;
      quad_setup<real, MODE, creal>(a, prm, in, bq, valid, true, leg, L, ws.sj + 4 * slot + leg, Q);
      int status;
      creal y[3], t[6];
      bool hard;
      unsigned pat;
      quad_first_solve<real, creal>(L, cc.sinv, cc.winv, cc.fmin, leg, y, t, status, hard, pat);
      hard = hard && valid;
      creal net[6];
#pragma unroll
      for (int r = 0; r < 6; r++) net[r] = fma(-cc.sinv[r], t[r], L.b[r]);   // A x = b - S^-1 t
      // every state is written, the hard ones provisionally (full sectors; the round phase overwrites them while the
      // lines are still in L2)
      quad_output<real, creal, real>(a, L, y, 0, 0, 0, status, 0, bq, valid, leg, ws.sj + 4 * slot + leg, Q, net);
      // ---- park the hard states
      if (hard) {
        const int e = 4 * slot + leg;
#pragma unroll
        for (int c = 0; c < 3; c++) {
#pragma unroll
          for (int k = 0; k < 2; k++) ws.sl[(3 * k + c) * Q + e] = L.At[k][c];
          ws.sl[(kSlFoot + c) * Q + e] = L.foot[c];
          ws.sl[(kSlY + c) * Q + e] = y[c];
          ws.sl[(kSlU + c) * Q + e] = creal(0.0);
        }
        ws.sl[kSlMu * Q + e] = L.mu;
        // lane `leg` stores components leg and leg + 4 (no dynamic register indexing)
        ws.sb[leg * CAP + slot] = sel4(leg, L.b[0], L.b[1], L.b[2], L.b[3]);
        if (leg < 2) ws.sb[(4 + leg) * CAP + slot] = (leg & 1) ? L.b[5] : L.b[4];
        if (leg == 0) {
          ws.sh[slot] = (unsigned)bq;
          ws.sh[CAP + slot] = L.mask | (pat << 4);
        }
      }
      occ |= __reduce_or_sync(kFull, hard ? (1u << slot) : 0u);
      __syncwarp();
      if (sub + 1 == SUPER) cur = nxt;
    }
    // one call site (the code of the round phase exists once): after a tile when the stash is full enough, and
    // once more when the boxes are exhausted, until the stash is empty
    const int pending = __popc(occ);
    if (have ? (pending >= kRunMin) : (pending > 0)) round_phase<real, creal, CAP>(a, cc, ws, occ, !have, kRunLow, lane, leg, quad);
    if (!have) break;
  }
}

}  // namespace qlb
