// qlb_api.cu - the C ABI declared in include/qlb.h: context management and kernel launches.
// No CPU fallback lives here: every compute entry point launches sm_100a kernels or returns an error.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>

#include "qlb.h"
#include "qlb_aux.cuh"
#include "qlb_gen.cuh"
#include "qlb_qp_dense.cuh"
#include "qlb_records.cuh"
#include "qlb_solve.cuh"
#include "qlb_solve_quad.cuh"
#include "qlb_solve_fused.cuh"
#include "qlb_solve_single.cuh"
#include "qlb_swing.cuh"
#include "qlb_tick.cuh"

using namespace qlb;

#ifndef QLB_PIPE
#define QLB_PIPE 3
#endif
constexpr int kPipe = QLB_PIPE;   // host entry points: chunks in flight (H2D / kernel / D2H overlap)

// Device memory of a context that only grows (reserve)
struct DeviceBuffer {
  unsigned char* p = nullptr;
  size_t bytes = 0;
};

// CTAs per SM of the solve kernels of one (interface, core) type pair, [MODE]: the three-pass kernels, and the fused
// kernel without / with TMA staging (FP64 core only)
struct SolveOccupancy {
  int first[2] = {0, 0};
  int quad[2] = {0, 0};
  int single[2][2] = {};
};

struct qlb_context {
  int device = 0;
  int sm_count = 0;
  SolveOccupancy occ[3];   // [occ_index<T, C>]: double/double, float/double, float/float
  qlb_params params;
  qlb_leg_model legs[QLB_NUM_LEGS];
  DeviceModel* d_model = nullptr;
  DeviceParams* d_params = nullptr;
  DeviceLimbDynamics* d_limb = nullptr;        // qlb_set_limb_dynamics
  DeviceLimbDynamicsT<float>* d_limb_f = nullptr;   // its FP32 copy (swing legs of qlb_controller_update_f32)
  bool have_limb = false;
  DeviceModelT<float>* d_model_f = nullptr;    // FP32 copies for the _f32 entry points
  DeviceParamsT<float>* d_params_f = nullptr;
  int pipeline = QLB_PIPELINE_FUSED;   // qlb_set_pipeline
  std::recursive_mutex mu;                  // calls on one context from several host threads are serialised (QLB_GUARD)
  int fused_bps_cap = 0;                    // experiments (env QLB_FUSED_BPS): fewer CTAs of the fused kernel per SM
  bool f32_pure = false;  // qlb_set_f32_core: FP32 solver core with in-kernel FP64 rescue, or FP64 core for every state
  unsigned long long* d_counter = nullptr;
  DeviceBuffer lists;         // second-pass index lists: 8 launch slots x 3 lists of list_cap entries
  size_t list_cap = 0;
  uint64_t solve_calls = 0;   // picks the launch slot (counters + list): concurrent launches never share one
  cudaEvent_t slot_done[8] = {};  // recorded after the last pass of the call that used the slot; the next user waits on it
  int last_slot = 0;
  double* d_stats = nullptr;
  cudaStream_t stream = nullptr;  // used by the *_host entry points
  cudaStream_t pipe[kPipe] = {};  // chunk pipeline of the *_host entry points
  // staging of the host entry points and qlb_solve_records
  DeviceBuffer soa;    // SoA rows of kPipe slots of `cap` states (soa_slot)
  size_t cap = 0;
  cudaEvent_t soa_free = nullptr;   // recorded after the last asynchronous use of `soa` (qlb_solve_records)
  DeviceBuffer rec;    // records of qlb_solve_records_host: kPipe x cap x (216 + 248) bytes
  DeviceBuffer prev;   // qlb_preview_plan_host
  DeviceBuffer qp;     // qlb_qp_dense_host
  uint64_t launches = 0;
  char last_error[256] = {0};
};

namespace {

constexpr int kHostInRows = 12 + 7 + 6 + 7 + 6 + 4 + 12;  // state mode is the larger one (54)
constexpr int kHostOutRows = 12 + 12 + 6 + 6;
#ifndef QLB_CHUNK_LOG2
#define QLB_CHUNK_LOG2 17
#endif
constexpr size_t kChunk = size_t(1) << QLB_CHUNK_LOG2;  // states per pipeline chunk

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

int cuda_fail(qlb_context* ctx, cudaError_t e, const char* what) {
  if (ctx) std::snprintf(ctx->last_error, sizeof ctx->last_error, "%s: %s", what, cudaGetErrorString(e));
  return QLB_ERR_CUDA;
}
// Every entry point that touches the state of a context (launch slots, staging buffers, parameter blocks) holds the
// context's lock while it enqueues its work: one context may be shared by several host threads.  Device work stays
// asynchronous (the lock covers the enqueue, not the execution); the *_host entry points hold it until they return.
#define QLB_GUARD(ctx) \
  std::unique_lock<std::recursive_mutex> qlb_guard_; \
  if ((ctx) != nullptr) qlb_guard_ = std::unique_lock<std::recursive_mutex>((ctx)->mu)

#define QLB_CUDA(ctx, call)                                   \
  do {                                                        \
    cudaError_t e__ = (call);                                 \
    if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); \
  } while (0)

#define QLB_TRY(call)                        \
  do {                                       \
    const int rc__ = (call);                 \
    if (rc__ != QLB_OK) return rc__;         \
  } while (0)

// The one rule of every staging buffer: the device is synchronised before the old buffer is freed (work on any stream
// may still use it); when the allocation fails the buffer is left empty.
int reserve(qlb_context* ctx, DeviceBuffer& b, size_t bytes) {
  if (bytes <= b.bytes) return QLB_OK;
  QLB_CUDA(ctx, cudaDeviceSynchronize());
  cudaFree(b.p);
  b.p = nullptr;
  b.bytes = 0;
  if (cudaMalloc(&b.p, bytes) != cudaSuccess) { cudaGetLastError(); return QLB_ERR_ALLOC; }
  b.bytes = bytes;
  return QLB_OK;
}

size_t pow2_at_least(size_t n, size_t lo) {
  while (lo < n) lo *= 2;
  return lo;
}

// One thread per item: ceil(items / threads) blocks of `threads`.
template <typename... P, typename... A>
int launch_items(qlb_context* ctx, unsigned long long items, unsigned threads, cudaStream_t st, void (*kernel)(P...), A... args) {
  const unsigned long long blocks = (items + threads - 1) / threads;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  kernel<<<(unsigned)blocks, threads, 0, st>>>(args...);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

// URDF <origin rpy> -> rotation matrix, through the quaternion like urdfdom + KDL do.
void rpy_to_rot(const double rpy[3], double R[9]) {
  const double hr = 0.5 * rpy[0], hp = 0.5 * rpy[1], hy = 0.5 * rpy[2];
  double x = std::sin(hr) * std::cos(hp) * std::cos(hy) - std::cos(hr) * std::sin(hp) * std::sin(hy);
  double y = std::cos(hr) * std::sin(hp) * std::cos(hy) + std::sin(hr) * std::cos(hp) * std::sin(hy);
  double z = std::cos(hr) * std::cos(hp) * std::sin(hy) - std::sin(hr) * std::sin(hp) * std::cos(hy);
  double w = std::cos(hr) * std::cos(hp) * std::cos(hy) + std::sin(hr) * std::sin(hp) * std::sin(hy);
  const double n = std::sqrt(x * x + y * y + z * z + w * w);
  x /= n; y /= n; z /= n; w /= n;
  R[0] = w * w + x * x - y * y - z * z; R[1] = 2.0 * (x * y - w * z); R[2] = 2.0 * (x * z + w * y);
  R[3] = 2.0 * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = 2.0 * (y * z - w * x);
  R[6] = 2.0 * (x * z - w * y); R[7] = 2.0 * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
}

void build_device_model(const qlb_leg_model legs[QLB_NUM_LEGS], DeviceModel* m) {
  std::memset(m, 0, sizeof *m);
  for (int l = 0; l < 4; l++) {
    for (int j = 0; j < 4; j++) {
      rpy_to_rot(legs[l].joint_rpy[j], m->rot[l][j]);
      for (int a = 0; a < 3; a++) m->xyz[l][j][a] = legs[l].joint_xyz[j][a];
      m->mass[l][j] = legs[l].link_mass[j];
      for (int a = 0; a < 3; a++) m->com[l][j][a] = legs[l].link_com[j][a];
    }
    // the foot frame is never rotated in the kernel: fold its fixed rotation into the foot link's COM
    const double* R3 = m->rot[l][3];
    const double* c3 = legs[l].link_com[3];
    for (int a = 0; a < 3; a++) m->com[l][3][a] = R3[3 * a] * c3[0] + R3[3 * a + 1] * c3[1] + R3[3 * a + 2] * c3[2];
    double acc = 0.0;
    for (int j = 3; j >= 0; j--) { acc += legs[l].link_mass[j]; m->msuf[l][j] = acc; }
  }
}

void build_device_params(const qlb_params* p, DeviceParams* d) {
  std::memset(d, 0, sizeof *d);
  for (int i = 0; i < 6; i++) d->S[i] = p->wrench_weights[i];
  d->W = p->ground_force_weight;
  d->fmin = p->min_normal_force > 0.0 ? p->min_normal_force : 0.0;   // with mu > 0 the friction rows imply n.f >= 0
  d->mu_default = p->friction_default;
  d->gravity = p->gravity;
  d->tol = p->ipm_tolerance;
  d->max_iter = p->ipm_max_iterations;
  for (int i = 0; i < 3; i++) {
    d->kp_t[i] = p->kp_translation[i]; d->kd_t[i] = p->kd_translation[i]; d->kff_t[i] = p->kff_translation[i];
    d->kp_r[i] = p->kp_rotation[i]; d->kd_r[i] = p->kd_rotation[i]; d->kff_r[i] = p->kff_rotation[i];
    d->com[i] = p->com_in_base[i];
  }
  d->torso_mass = p->torso_mass;
  for (int l = 0; l < 4; l++) {
    d->leg_mass[l] = p->leg_mass[l];
    for (int a = 0; a < 3; a++) d->leg_pos[l][a] = p->leg_base_position[l][a];
  }
  d->grav_pct = p->gravity_compensation_percentage;
}

// FP32 copies: same fields, rounded once on the host
void narrow_model(const DeviceModel& m, DeviceModelT<float>* f) {
  const double* src = reinterpret_cast<const double*>(&m);
  float* dst = reinterpret_cast<float*>(f);
  for (size_t i = 0; i < sizeof(DeviceModel) / sizeof(double); i++) dst[i] = (float)src[i];
}
void narrow_params(const DeviceParams& d, DeviceParamsT<float>* f) {
  std::memset(f, 0, sizeof *f);
  for (int i = 0; i < 6; i++) f->S[i] = (float)d.S[i];
  f->W = (float)d.W; f->fmin = (float)d.fmin; f->mu_default = (float)d.mu_default; f->gravity = (float)d.gravity;
  f->tol = (float)d.tol; f->max_iter = d.max_iter;
  for (int i = 0; i < 3; i++) {
    f->kp_t[i] = (float)d.kp_t[i]; f->kd_t[i] = (float)d.kd_t[i]; f->kff_t[i] = (float)d.kff_t[i];
    f->kp_r[i] = (float)d.kp_r[i]; f->kd_r[i] = (float)d.kd_r[i]; f->kff_r[i] = (float)d.kff_r[i];
    f->com[i] = (float)d.com[i];
  }
  f->torso_mass = (float)d.torso_mass;
  for (int l = 0; l < 4; l++) {
    f->leg_mass[l] = (float)d.leg_mass[l];
    for (int a = 0; a < 3; a++) f->leg_pos[l][a] = (float)d.leg_pos[l][a];
  }
  f->grav_pct = (float)d.grav_pct;
}

// The FP32-core kernels seed reciprocals and reciprocal square roots from FP32 (qlb_device.cuh; the FP64 kernels use
// the FP64 seed instructions and have no such limit): weights, their inverses and the pivots built from them must stay
// inside the FP32 normal range for that core, so the weights are bounded here for every core alike.
bool params_ok(const qlb_params* p) {
  const double lo = 1e-12, hi = 1e12;
  if (!(p->ground_force_weight >= lo && p->ground_force_weight <= hi) || !(p->ipm_tolerance > 0.0) || p->ipm_max_iterations < 1)
    return false;
  for (int i = 0; i < 6; i++)
    if (!(p->wrench_weights[i] >= lo && p->wrench_weights[i] <= hi)) return false;  // the 6x6 dual system needs S^-1
  if (!(p->friction_default >= 0.0) || !std::isfinite(p->friction_default)) return false;
  if (!(std::fabs(p->min_normal_force) <= 1e9)) return false;
  return std::isfinite(p->gravity);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Launch slot of one solve call: work counters of the three passes, lengths and storage of the two
// compacted index lists.  Concurrent launches (the host pipeline's streams) never share a slot.
template <typename T>
int prepare_slot(qlb_context* ctx, SolveArgsT<T>& a, cudaStream_t st) {
  if (a.B > 0xFFFFFFF0ull) return QLB_ERR_BATCH_TOO_LARGE;
  // the lowest slot whose previous call has finished (so that a serial caller keeps using one set of buffers); if all
  // eight are busy, round robin: the call is ordered behind the previous user of its slot
  int slot = -1;
  for (int i = 0; i < 8 && slot < 0; i++)
    if (cudaEventQuery(ctx->slot_done[i]) == cudaSuccess) slot = i;
  cudaGetLastError();
  if (slot < 0) slot = (int)(ctx->solve_calls % 8);
  ctx->solve_calls++;
  ctx->last_slot = slot;
  QLB_CUDA(ctx, cudaStreamWaitEvent(st, ctx->slot_done[slot], 0));
  a.counter = ctx->d_counter + 8 * slot;
  a.counter2 = a.counter + 1;
  a.counter3 = a.counter + 2;
  a.list_count = reinterpret_cast<unsigned*>(a.counter + 3);
  a.list2_count = reinterpret_cast<unsigned*>(a.counter + 4);
  QLB_CUDA(ctx, cudaMemsetAsync(a.counter, 0, 8 * sizeof(unsigned long long), st));
  if (ctx->list_cap < a.B) {  // grow the index lists of all slots at once (rare; synchronises)
    const size_t cap = pow2_at_least(a.B, 1024);
    ctx->list_cap = 0;
    QLB_TRY(reserve(ctx, ctx->lists, 8 * 3 * cap * sizeof(unsigned)));
    ctx->list_cap = cap;
  }
  unsigned* list = reinterpret_cast<unsigned*>(ctx->lists.p) + (size_t)slot * 3 * ctx->list_cap;
  a.list = list;
  a.list2 = list + ctx->list_cap;
  a.list_pat = list + 2 * ctx->list_cap;
  return QLB_OK;
}

template <typename T, typename C>
constexpr int occ_index() { return sizeof(T) == 8 ? 0 : sizeof(C) == 8 ? 1 : 2; }

// The three passes of the leg-per-lane kernels.  pass 1: everything up to the unconstrained minimiser;
// pass 2: active-set rounds on what is left; pass 3: interior point on what is still left.  The later
// grids are sized for the worst case and read the list lengths on the device (no host synchronisation
// between the passes).
template <typename T, typename C, int MODE>
int launch_quad(qlb_context* ctx, SolveArgsT<T>& a, cudaStream_t st) {
  const SolveOccupancy& occ = ctx->occ[occ_index<T, C>()];
  const unsigned long long nb8 = (a.B + 7) / 8;
  const unsigned long long wantq = (nb8 + (kQuadThreads / 32) - 1) / (kQuadThreads / 32);
  const unsigned long long capq = (unsigned long long)ctx->sm_count * occ.quad[MODE];
  const unsigned long long capf = (unsigned long long)ctx->sm_count * occ.first[MODE];
  const unsigned gq = (unsigned)(wantq < capq ? wantq : capq);
  qlb_quad_first_kernel<T, C, MODE><<<(unsigned)(wantq < capf ? wantq : capf), kQuadThreads, 0, st>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  qlb_quad_kernel<T, C, MODE, 1><<<gq, kQuadThreads, 0, st>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  qlb_quad_kernel<T, C, MODE, 2><<<gq, kQuadThreads, 0, st>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  QLB_CUDA(ctx, cudaEventRecord(ctx->slot_done[ctx->last_slot], st));
  return QLB_OK;
}

// ---- the fused pipeline (qlb_solve_fused.cuh): one persistent kernel + the interior-point kernel for the
// states the rounds could not verify (normally none: it finds an empty list and returns)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// Tensor map of one SoA input array [rows][B]: boxes of {8 QLB_SUPER states, rows}, out-of-range columns read as zero.
template <typename T>
bool make_map(CUtensorMap* m, const T* ptr, unsigned long long B, int rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  const cuuint64_t gdim[2] = {(cuuint64_t)B, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)B * sizeof(T)};
  const cuuint32_t box[2] = {8u * QLB_SUPER, (cuuint32_t)rows};
  const cuuint32_t estr[2] = {1u, 1u};
  return fn(m, sizeof(T) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<T*>(ptr), gdim,
            gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// rank-1 tensor map of the stance masks (one byte per state), boxes of `cols` states
bool make_mask_map(CUtensorMap* m, const uint8_t* ptr, unsigned long long B, int cols) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  const cuuint64_t gdim[1] = {(cuuint64_t)B};
  const cuuint64_t gstride[1] = {0};
  const cuuint32_t box[1] = {(cuuint32_t)cols};
  const cuuint32_t estr[1] = {1u};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, const_cast<uint8_t*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// the fused kernel (qlb_solve_single.cuh) + the interior-point kernel for the states its rounds could not verify
// (normally none: it finds an empty list and returns)
template <typename T, typename C, int MODE>
int launch_single(qlb_context* ctx, SolveArgsT<T>& a, cudaStream_t st) {
  const SolveOccupancy& occ = ctx->occ[occ_index<T, C>()];
  using SG = Staging<T, MODE, QLB_SUPER>;
  using FL = FusedLayout<T, C, MODE, QLB_SUPER>;
  const T* src[SG::kNumSeg];
  for (int s = 0; s < SG::kNumSeg; s++) src[s] = SG::source(a, s);
  bool tma = a.B >= 64 && a.B < 0x7fffff00ull && ((a.B * sizeof(T)) % 16 == 0);
  for (int s = 0; s < SG::kNumSeg && tma; s++)
    if (src[s] && !aligned16(src[s])) tma = false;
  FusedMaps maps;
  std::memset(&maps, 0, sizeof maps);
  for (int s = 0; s < SG::kNumSeg && tma; s++)
    if (src[s] && !make_map<T>(&maps.seg[s], src[s], a.B, SG::rows(s))) tma = false;
  if (tma && (SG::kCols < 16 || !aligned16(a.mask) || !make_mask_map(&maps.mask, a.mask, a.B, SG::kCols))) tma = false;
  const unsigned long long ntiles = (a.B + 7) / 8;
  const unsigned long long want = (ntiles + kFusedWarps - 1) / kFusedWarps;
  int bps = occ.single[MODE][tma ? 1 : 0];
  if (ctx->fused_bps_cap > 0 && bps > ctx->fused_bps_cap) bps = ctx->fused_bps_cap;
  const unsigned long long cap = (unsigned long long)ctx->sm_count * bps;
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  if (tma) qlb_single_kernel<T, C, MODE, QLB_SUPER, true><<<grid, kFusedThreads, FL::kTotal, st>>>(a, maps);
  else qlb_single_kernel<T, C, MODE, QLB_SUPER, false><<<grid, kFusedThreads, FL::kTotal, st>>>(a, maps);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  const unsigned long long capq = (unsigned long long)ctx->sm_count * occ.quad[MODE];
  const unsigned long long wantq = (ntiles + 3) / 4;
  qlb_quad_kernel<T, C, MODE, 2><<<(unsigned)(wantq < capq ? wantq : capq), kQuadThreads, 0, st>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  QLB_CUDA(ctx, cudaEventRecord(ctx->slot_done[ctx->last_slot], st));
  return QLB_OK;
}

// ctx->occ of one type pair: the three-pass kernels of both modes
template <typename T, typename C>
bool query_occupancy(qlb_context* ctx) {
  SolveOccupancy& o = ctx->occ[occ_index<T, C>()];
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.quad[0], qlb_quad_kernel<T, C, 0, 2>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.quad[1], qlb_quad_kernel<T, C, 1, 2>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.first[0], qlb_quad_first_kernel<T, C, 0>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o.first[1], qlb_quad_first_kernel<T, C, 1>, kQuadThreads, 0) != cudaSuccess)
    return false;
  return o.quad[0] >= 1 && o.quad[1] >= 1 && o.first[0] >= 1 && o.first[1] >= 1;
}

// ctx->occ.single of the fused kernel (FP64 core) for one interface type and mode
template <typename T, int MODE>
bool prepare_single_kernels(qlb_context* ctx) {
  using C = double;
  using FL = FusedLayout<T, C, MODE, QLB_SUPER>;
  int* out = ctx->occ[occ_index<T, C>()].single[MODE];
  if (cudaFuncSetAttribute(qlb_single_kernel<T, C, MODE, QLB_SUPER, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FL::kTotal) != cudaSuccess ||
      cudaFuncSetAttribute(qlb_single_kernel<T, C, MODE, QLB_SUPER, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FL::kTotal) != cudaSuccess ||
      cudaFuncSetAttribute(qlb_single_kernel<T, C, MODE, QLB_SUPER, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess ||
      cudaFuncSetAttribute(qlb_single_kernel<T, C, MODE, QLB_SUPER, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess)
    return false;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&out[0], qlb_single_kernel<T, C, MODE, QLB_SUPER, false>, kFusedThreads, FL::kTotal) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&out[1], qlb_single_kernel<T, C, MODE, QLB_SUPER, true>, kFusedThreads, FL::kTotal) != cudaSuccess)
    return false;
  return out[0] >= 1 && out[1] >= 1;
}

// The FP64 interface runs the FP64 core; the FP32 interface the FP64 core or, with qlb_set_f32_core, the FP32 core
// (three-pass pipeline only).
template <typename T, int MODE>
int launch_solve(qlb_context* ctx, SolveArgsT<T>& a, cudaStream_t st) {
  QLB_TRY(prepare_slot(ctx, a, st));
  if constexpr (sizeof(T) == 4) {
    if (ctx->f32_pure) return launch_quad<float, float, MODE>(ctx, a, st);
  }
  if (ctx->pipeline == QLB_PIPELINE_FUSED) return launch_single<T, double, MODE>(ctx, a, st);
  return launch_quad<T, double, MODE>(ctx, a, st);
}

// SoA staging of the host entry points and qlb_solve_records: kPipe slots of `cap` states, laid out as
// [kPipe][kHostInRows][cap] and [kPipe][kHostOutRows][cap] doubles, [kPipe][cap] flags and [kPipe][cap] mask bytes.
// cap is a power of two >= 1024: cap % 16 == 0 keeps every row block 16-byte aligned, so that launch_single's choice of
// TMA does not depend on the chunk.
constexpr size_t kSoaBytesPerState = (kHostInRows + kHostOutRows) * sizeof(double) + sizeof(uint32_t) + 1;
struct SoaSlot {
  double* in;
  double* out;
  uint32_t* flags;
  uint8_t* mask;
};
SoaSlot soa_slot(const qlb_context* ctx, int slot) {
  const size_t cap = ctx->cap;
  double* in = reinterpret_cast<double*>(ctx->soa.p);
  double* out = in + kPipe * cap * kHostInRows;
  uint32_t* flags = reinterpret_cast<uint32_t*>(out + kPipe * cap * kHostOutRows);
  uint8_t* mask = reinterpret_cast<uint8_t*>(flags + kPipe * cap);
  return {in + slot * cap * kHostInRows, out + slot * cap * kHostOutRows, flags + slot * cap, mask + slot * cap};
}

int reserve_soa(qlb_context* ctx, size_t B) {
  if (B > kChunk) B = kChunk;
  if (B <= ctx->cap) return QLB_OK;
  const size_t cap = pow2_at_least(B, ctx->cap ? ctx->cap : 1024);
  ctx->cap = 0;
  QLB_TRY(reserve(ctx, ctx->soa, kPipe * cap * kSoaBytesPerState));
  ctx->cap = cap;
  return QLB_OK;
}

// Runs body(b0, n, slot, stream) over [0, B) in chunks of `chunk` states: chunk i on pipeline stream i % kPipe with
// staging slot i % kPipe, or all of them on the context stream with slot 0.  Each stream waits for the last
// asynchronous user of the SoA staging before its first chunk.  Every stream it enqueued on is synchronised before it
// returns, on failure too: no copy may still be reading or writing the caller's buffers.
template <typename F>
int for_chunks(qlb_context* ctx, size_t B, size_t chunk, bool pipelined, F&& body) {
  cudaStream_t* streams = pipelined ? ctx->pipe : &ctx->stream;
  const int nstreams = pipelined ? kPipe : 1;
  int used = 0, rc = QLB_OK;
  for (size_t b0 = 0, i = 0; b0 < B && rc == QLB_OK; b0 += chunk, i++) {
    const int slot = (int)(i % nstreams);
    if (used <= slot) {
      used = slot + 1;
      const cudaError_t e = cudaStreamWaitEvent(streams[slot], ctx->soa_free, 0);
      if (e != cudaSuccess) { rc = cuda_fail(ctx, e, "cudaStreamWaitEvent"); break; }
    }
    rc = body(b0, B - b0 < chunk ? B - b0 : chunk, slot, streams[slot]);
  }
  for (int i = 0; i < used; i++) {
    const cudaError_t e = cudaStreamSynchronize(streams[i]);
    if (e != cudaSuccess && rc == QLB_OK) rc = cuda_fail(ctx, e, "cudaStreamSynchronize");
  }
  return rc;
}

// Rows [0, rows) of columns [b0, b0 + n) of a host array with row pitch B, to or from a device block with row pitch n.
// A null host array is skipped.
template <typename T>
int rows_to_device(qlb_context* ctx, T* d, const T* h, size_t rows, size_t b0, size_t n, size_t B, cudaStream_t st) {
  if (h) QLB_CUDA(ctx, cudaMemcpy2DAsync(d, n * sizeof(T), h + b0, B * sizeof(T), n * sizeof(T), rows, cudaMemcpyHostToDevice, st));
  return QLB_OK;
}
template <typename T>
int rows_to_host(qlb_context* ctx, T* h, const T* d, size_t rows, size_t b0, size_t n, size_t B, cudaStream_t st) {
  if (h) QLB_CUDA(ctx, cudaMemcpy2DAsync(h + b0, B * sizeof(T), d, n * sizeof(T), n * sizeof(T), rows, cudaMemcpyDeviceToHost, st));
  return QLB_OK;
}

}  // namespace

extern "C" {

int qlb_abi_version(void) { return QLB_ABI_VERSION; }

const char* qlb_strerror(int status) {
  switch (status) {
    case QLB_OK: return "ok";
    case QLB_ERR_INVALID_ARGUMENT: return "invalid argument";
    case QLB_ERR_CUDA: return "CUDA error (see qlb_last_cuda_error)";
    case QLB_ERR_BATCH_TOO_LARGE: return "batch too large";
    case QLB_ERR_NOT_INITIALISED: return "context not initialised";
    case QLB_ERR_ALLOC: return "device allocation failed";
    default: return "unknown status";
  }
}

const char* qlb_last_cuda_error(const qlb_context* ctx) { return ctx ? ctx->last_error : ""; }

int qlb_default_params(qlb_params* p) {
  if (!p) return QLB_ERR_INVALID_ARGUMENT;
  std::memset(p, 0, sizeof *p);
  // balance_controller/config/controller_gains.yaml:27-41
  const double S[6] = {1.0, 5.0, 1.0, 10.0, 10.0, 5.0};
  for (int i = 0; i < 6; i++) p->wrench_weights[i] = S[i];
  p->ground_force_weight = 0.0001;
  p->min_normal_force = 10.0;
  p->friction_default = 0.6;
  p->gravity = 9.8;  // ContactForceDistribution.cpp:518, VirtualModelController.cpp:165
  // controller_gains.yaml:3-26 (heading, lateral, vertical / roll, pitch, yaw)
  const double kp_t[3] = {5000, 5000, 10000}, kd_t[3] = {5000, 4000, 5000}, kff_t[3] = {10, 10, 100};
  const double kp_r[3] = {10000, 10000, 4000}, kd_r[3] = {1000, 1000, 1000}, kff_r[3] = {0.2, 0.2, 1000};
  for (int i = 0; i < 3; i++) {
    p->kp_translation[i] = kp_t[i]; p->kd_translation[i] = kd_t[i]; p->kff_translation[i] = kff_t[i];
    p->kp_rotation[i] = kp_r[i]; p->kd_rotation[i] = kd_r[i]; p->kff_rotation[i] = kff_r[i];
    p->com_in_base[i] = 0.0;
  }
  p->torso_mass = 27.0;  // quadruped_state.cpp:28
  // quadruped_state.cpp:83-97, LF RF RH LH
  const double pos[4][3] = {{0.42, 0.075, 0.0}, {0.42, -0.075, 0.0}, {-0.42, -0.075, 0.0}, {-0.42, 0.075, 0.0}};
  for (int l = 0; l < 4; l++) {
    p->leg_mass[l] = 6.0;  // quadruped_state.cpp:36-41
    for (int a = 0; a < 3; a++) p->leg_base_position[l][a] = pos[l][a];
  }
  p->gravity_compensation_percentage = 1.0;  // VirtualModelController.cpp:57
  p->ipm_tolerance = 1e-9;
  p->ipm_max_iterations = 40;
  return QLB_OK;
}

// ---- parameters from the reference's own keys (ROS parameter paths / controller_gains.yaml)
namespace {
struct ParamKey { const char* path; int group; int index; };
// group 0: wrench_weights[i]; 1: ground_force_weight; 2: friction_default; 3: min_normal_force;
// 4/5/6: kp/kd/kff translation[i]; 7/8/9: kp/kd/kff rotation[i]
const ParamKey kParamKeys[] = {
    {"/balance_controller/contact_force_distribution/weights/force/heading", 0, 0},
    {"/balance_controller/contact_force_distribution/weights/force/lateral", 0, 1},
    {"/balance_controller/contact_force_distribution/weights/force/vertical", 0, 2},
    {"/balance_controller/contact_force_distribution/weights/torque/roll", 0, 3},
    {"/balance_controller/contact_force_distribution/weights/torque/pitch", 0, 4},
    {"/balance_controller/contact_force_distribution/weights/torque/yaw", 0, 5},
    {"/balance_controller/contact_force_distribution/weights/regularizer/value", 1, 0},
    {"/balance_controller/contact_force_distribution/constraints/friction_coefficient", 2, 0},
    {"/balance_controller/contact_force_distribution/constraints/minimal_normal_force", 3, 0},
    {"/balance_controller/virtual_model_controller/heading/kp", 4, 0}, {"/balance_controller/virtual_model_controller/heading/kd", 5, 0},
    {"/balance_controller/virtual_model_controller/heading/kff", 6, 0}, {"/balance_controller/virtual_model_controller/lateral/kp", 4, 1},
    {"/balance_controller/virtual_model_controller/lateral/kd", 5, 1}, {"/balance_controller/virtual_model_controller/lateral/kff", 6, 1},
    {"/balance_controller/virtual_model_controller/vertical/kp", 4, 2}, {"/balance_controller/virtual_model_controller/vertical/kd", 5, 2},
    {"/balance_controller/virtual_model_controller/vertical/kff", 6, 2}, {"/balance_controller/virtual_model_controller/roll/kp", 7, 0},
    {"/balance_controller/virtual_model_controller/roll/kd", 8, 0}, {"/balance_controller/virtual_model_controller/roll/kff", 9, 0},
    {"/balance_controller/virtual_model_controller/pitch/kp", 7, 1}, {"/balance_controller/virtual_model_controller/pitch/kd", 8, 1},
    {"/balance_controller/virtual_model_controller/pitch/kff", 9, 1}, {"/balance_controller/virtual_model_controller/yaw/kp", 7, 2},
    {"/balance_controller/virtual_model_controller/yaw/kd", 8, 2}, {"/balance_controller/virtual_model_controller/yaw/kff", 9, 2},
};
constexpr int kNumParamKeys = (int)(sizeof(kParamKeys) / sizeof(kParamKeys[0]));

// index of a key in kParamKeys, or -1
int find_param_key(const char* key) {
  for (int k = 0; k < kNumParamKeys; k++)
    if (std::strcmp(key, kParamKeys[k].path) == 0) return k;
  return -1;
}

double* param_field(qlb_params* p, int k) {
  const int i = kParamKeys[k].index;
  switch (kParamKeys[k].group) {
    case 0: return &p->wrench_weights[i];
    case 1: return &p->ground_force_weight;
    case 2: return &p->friction_default;
    case 3: return &p->min_normal_force;
    case 4: return &p->kp_translation[i];
    case 5: return &p->kd_translation[i];
    case 6: return &p->kff_translation[i];
    case 7: return &p->kp_rotation[i];
    case 8: return &p->kd_rotation[i];
    default: return &p->kff_rotation[i];
  }
}
}  // namespace

int qlb_params_set_key(qlb_params* p, const char* key, double value) {
  if (!p || !key) return QLB_ERR_INVALID_ARGUMENT;
  const int k = find_param_key(key);
  if (k < 0) return QLB_ERR_INVALID_ARGUMENT;
  *param_field(p, k) = value;
  return k;   // index of the key (>= 0)
}

int qlb_params_get_key(const qlb_params* p, const char* key, double* value) {
  if (!p || !key || !value) return QLB_ERR_INVALID_ARGUMENT;
  const int k = find_param_key(key);
  if (k < 0) return QLB_ERR_INVALID_ARGUMENT;
  *value = *param_field(const_cast<qlb_params*>(p), k);
  return k;
}

int qlb_params_num_keys(void) { return kNumParamKeys; }
const char* qlb_params_key(int index) { return (index >= 0 && index < kNumParamKeys) ? kParamKeys[index].path : nullptr; }

// A YAML subset is enough for the reference's parameter files: nested mappings by indentation, `key: scalar` leaves,
// comments and blank lines.  Every leaf becomes a parameter path "/a/b/c" and goes through qlb_params_set_key;
// unknown paths are ignored (the files also configure other controllers).
int qlb_params_from_yaml(qlb_params* p, const char* text, const char** first_missing) {
  if (!p || !text) return QLB_ERR_INVALID_ARGUMENT;
  bool seen[kNumParamKeys] = {};
  struct Level { int indent; size_t len; };
  Level stack[32];
  int depth = 0;
  char path[512];
  size_t plen = 0;
  const char* c = text;
  while (*c) {
    const char* eol = c;
    while (*eol && *eol != '\n') eol++;
    int indent = 0;
    const char* t = c;
    while (t < eol && *t == ' ') { indent++; t++; }
    const char* hash = t;
    while (hash < eol && *hash != '#') hash++;
    const char* end = hash;
    while (end > t && (end[-1] == ' ' || end[-1] == '\t' || end[-1] == '\r')) end--;
    if (end > t && *t != '-') {
      const char* colon = t;
      while (colon < end && *colon != ':') colon++;
      if (colon < end) {
        while (depth > 0 && stack[depth - 1].indent >= indent) depth--;
        plen = depth > 0 ? stack[depth - 1].len : 0;
        const size_t klen = (size_t)(colon - t);
        if (plen + 1 + klen + 1 < sizeof path && depth < 32) {
          path[plen] = '/';
          std::memcpy(path + plen + 1, t, klen);
          const size_t nlen = plen + 1 + klen;
          path[nlen] = 0;
          const char* v = colon + 1;
          while (v < end && *v == ' ') v++;
          if (v < end) {
            char buf[64];
            const size_t vl = (size_t)(end - v) < sizeof buf - 1 ? (size_t)(end - v) : sizeof buf - 1;
            std::memcpy(buf, v, vl);
            buf[vl] = 0;
            char* stop = nullptr;
            const double val = std::strtod(buf, &stop);
            if (stop != buf) {
              const int k = qlb_params_set_key(p, path, val);
              if (k >= 0) seen[k] = true;
            }
          } else {
            stack[depth].indent = indent; stack[depth].len = nlen; depth++;
          }
        }
      }
    }
    c = *eol ? eol + 1 : eol;
  }
  int found = 0;
  const char* miss = nullptr;
  for (int k = 0; k < kNumParamKeys; k++) {
    if (seen[k]) found++;
    else if (!miss) miss = kParamKeys[k].path;
  }
  if (first_missing) *first_missing = miss;
  return found;
}

int qlb_create(qlb_context** out, const qlb_leg_model legs[QLB_NUM_LEGS], const qlb_params* params, int device,
               size_t max_batch) {
  if (!out || !legs) return QLB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  qlb_params defaults;
  qlb_default_params(&defaults);
  const qlb_params* p = params ? params : &defaults;
  if (!params_ok(p)) return QLB_ERR_INVALID_ARGUMENT;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    cudaGetLastError();
    return QLB_ERR_CUDA;
  }
  qlb_context* ctx = new (std::nothrow) qlb_context();
  if (!ctx) return QLB_ERR_ALLOC;
  ctx->device = device;
  ctx->params = *p;
  std::memcpy(ctx->legs, legs, sizeof ctx->legs);
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { delete ctx; return QLB_ERR_CUDA; }
  ctx->sm_count = prop.multiProcessorCount;
  auto fail = [&](int code) { qlb_destroy(ctx); return code; };
  if (cudaMalloc(&ctx->d_model, sizeof(DeviceModel)) != cudaSuccess || cudaMalloc(&ctx->d_params, sizeof(DeviceParams)) != cudaSuccess ||
      cudaMalloc(&ctx->d_model_f, sizeof(DeviceModelT<float>)) != cudaSuccess ||
      cudaMalloc(&ctx->d_params_f, sizeof(DeviceParamsT<float>)) != cudaSuccess ||
      cudaMalloc(&ctx->d_counter, 64 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMalloc(&ctx->d_stats, QLB_STATS_NUM * sizeof(double)) != cudaSuccess)
    return fail(QLB_ERR_ALLOC);
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(QLB_ERR_CUDA);
  for (int i = 0; i < kPipe; i++)
    if (cudaStreamCreateWithFlags(&ctx->pipe[i], cudaStreamNonBlocking) != cudaSuccess) return fail(QLB_ERR_CUDA);
  for (int i = 0; i < 8; i++)
    if (cudaEventCreateWithFlags(&ctx->slot_done[i], cudaEventDisableTiming) != cudaSuccess) return fail(QLB_ERR_CUDA);
  if (cudaEventCreateWithFlags(&ctx->soa_free, cudaEventDisableTiming) != cudaSuccess) return fail(QLB_ERR_CUDA);
  DeviceModel hm;
  build_device_model(legs, &hm);
  if (cudaMemcpy(ctx->d_model, &hm, sizeof hm, cudaMemcpyHostToDevice) != cudaSuccess) return fail(QLB_ERR_CUDA);
  DeviceModelT<float> hmf;
  narrow_model(hm, &hmf);
  if (cudaMemcpy(ctx->d_model_f, &hmf, sizeof hmf, cudaMemcpyHostToDevice) != cudaSuccess) return fail(QLB_ERR_CUDA);
  if (qlb_set_params(ctx, p) != QLB_OK) return fail(QLB_ERR_CUDA);
  if (!query_occupancy<double, double>(ctx) || !query_occupancy<float, float>(ctx) || !query_occupancy<float, double>(ctx) ||
      !prepare_single_kernels<double, 0>(ctx) || !prepare_single_kernels<double, 1>(ctx) ||
      !prepare_single_kernels<float, 0>(ctx) || !prepare_single_kernels<float, 1>(ctx)) {
    cudaGetLastError();
    return fail(QLB_ERR_CUDA);
  }
  if (const char* e = std::getenv("QLB_FUSED_BPS")) ctx->fused_bps_cap = std::atoi(e);
  if (max_batch > 0 && reserve_soa(ctx, max_batch) != QLB_OK) return fail(QLB_ERR_ALLOC);
  *out = ctx;
  return QLB_OK;
}

int qlb_destroy(qlb_context* ctx) {
  if (!ctx) return QLB_OK;
  DeviceGuard guard(ctx->device);
  if (ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
  for (int i = 0; i < kPipe; i++)
    if (ctx->pipe[i]) { cudaStreamSynchronize(ctx->pipe[i]); cudaStreamDestroy(ctx->pipe[i]); }
  cudaFree(ctx->d_model); cudaFree(ctx->d_params); cudaFree(ctx->d_counter); cudaFree(ctx->d_stats);
  cudaFree(ctx->d_model_f); cudaFree(ctx->d_params_f); cudaFree(ctx->d_limb); cudaFree(ctx->d_limb_f);
  for (DeviceBuffer* b : {&ctx->lists, &ctx->soa, &ctx->rec, &ctx->prev, &ctx->qp}) cudaFree(b->p);
  for (int i = 0; i < 8; i++)
    if (ctx->slot_done[i]) cudaEventDestroy(ctx->slot_done[i]);
  if (ctx->soa_free) cudaEventDestroy(ctx->soa_free);
  cudaGetLastError();
  delete ctx;
  return QLB_OK;
}

int qlb_set_params(qlb_context* ctx, const qlb_params* params) {
  QLB_GUARD(ctx);
  if (!ctx || !params) return QLB_ERR_INVALID_ARGUMENT;
  if (!params_ok(params)) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  DeviceParams hp;
  build_device_params(params, &hp);
  // ordered after any solve already queued on the context stream
  QLB_CUDA(ctx, cudaDeviceSynchronize());
  QLB_CUDA(ctx, cudaMemcpy(ctx->d_params, &hp, sizeof hp, cudaMemcpyHostToDevice));
  DeviceParamsT<float> hpf;
  narrow_params(hp, &hpf);
  QLB_CUDA(ctx, cudaMemcpy(ctx->d_params_f, &hpf, sizeof hpf, cudaMemcpyHostToDevice));
  ctx->params = *params;
  return QLB_OK;
}

int qlb_get_params(const qlb_context* ctx, qlb_params* params) {
  if (!ctx || !params) return QLB_ERR_INVALID_ARGUMENT;
  *params = ctx->params;
  return QLB_OK;
}

int qlb_set_f32_core(qlb_context* ctx, int core) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (core != QLB_F32_CORE_FP32 && core != QLB_F32_CORE_FP64) return QLB_ERR_INVALID_ARGUMENT;
  ctx->f32_pure = (core == QLB_F32_CORE_FP32);
  return QLB_OK;
}

int qlb_set_pipeline(qlb_context* ctx, int pipeline) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (pipeline != QLB_PIPELINE_FUSED && pipeline != QLB_PIPELINE_THREE_PASS) return QLB_ERR_INVALID_ARGUMENT;
  ctx->pipeline = pipeline;
  return QLB_OK;
}

uint64_t qlb_launch_count(const qlb_context* ctx) { return ctx ? ctx->launches : 0; }

// ---- solve entry points (T = double, and float for the _f32 twins).  Each device-pointer / host-pointer twin pair goes
// through one function that checks the arguments and then launches on `stream` or runs the host pipeline.
extern "C++" {
namespace {

template <typename T> struct Typed;
template <> struct Typed<double> {
  static const DeviceModel* model(const qlb_context* c) { return c->d_model; }
  static const DeviceLimbDynamics* limb(const qlb_context* c) { return c->d_limb; }
  static const DeviceParams* params(const qlb_context* c) { return c->d_params; }
};
template <> struct Typed<float> {
  static const DeviceModelT<float>* model(const qlb_context* c) { return c->d_model_f; }
  static const DeviceLimbDynamicsT<float>* limb(const qlb_context* c) { return c->d_limb_f; }
  static const DeviceParamsT<float>* params(const qlb_context* c) { return c->d_params_f; }
};

// Host pipeline of the solve: copy in, solve, copy out, synchronise.
// Large batches are cut into chunks of kChunk states that flow through kPipe streams, so that the H2D
// copy of chunk i+1, the kernel of chunk i and the D2H copy of chunk i-1 overlap (PCIe is full duplex).
// The arrays are SoA with row pitch B, so a chunk is a column range: one 2-D copy per array.
// solve(n, in, mask, out, flags, stream) runs the device-pointer solve on the staged arrays of one chunk.
template <typename P> struct HostRows { P h; int rows; };   // array (may be null) and its component count

template <typename T, typename F>
int run_host_pipeline(qlb_context* ctx, size_t B, const HostRows<const T*>* in, int nin, const uint8_t* mask,
                      const HostRows<T*>* out, int nout, uint32_t* flags, F&& solve) {
  QLB_TRY(reserve_soa(ctx, B));
  const size_t cap = ctx->cap;
  return for_chunks(ctx, B, cap, true, [&](size_t b0, size_t n, int slot, cudaStream_t st) -> int {
    // the staging is sized for FP64; the FP32 twins use the first half of each slot
    const SoaSlot s = soa_slot(ctx, slot);
    T* din = reinterpret_cast<T*>(s.in);
    T* dout = reinterpret_cast<T*>(s.out);
    const T* dptr_in[8];
    T* dptr_out[4];
    for (int k = 0; k < nin; k++) {
      dptr_in[k] = in[k].h ? din : nullptr;
      QLB_TRY(rows_to_device(ctx, din, in[k].h, in[k].rows, b0, n, B, st));
      din += (size_t)in[k].rows * cap;   // fixed block sizes keep every block 16-byte aligned (cap % 16 == 0)
    }
    QLB_CUDA(ctx, cudaMemcpyAsync(s.mask, mask + b0, n, cudaMemcpyHostToDevice, st));
    for (int k = 0; k < nout; k++) {
      dptr_out[k] = out[k].h ? dout : nullptr;
      dout += (size_t)out[k].rows * cap;
    }
    QLB_TRY(solve(n, dptr_in, s.mask, dptr_out, s.flags, st));
    for (int k = 0; k < nout; k++) QLB_TRY(rows_to_host(ctx, out[k].h, dptr_out[k], out[k].rows, b0, n, B, st));
    QLB_CUDA(ctx, cudaMemcpyAsync(flags + b0, s.flags, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    return QLB_OK;
  });
}

template <typename T>
int solve_wrench_t(qlb_context* ctx, size_t B, const T* q, const T* quat_wxyz, const T* wrench, const uint8_t* stance_mask,
                   const T* mu, const T* normals_world, T* grf, T* tau, uint32_t* flags, T* netwrench, void* stream, bool host) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !quat_wxyz || !wrench || !stance_mask || !grf || !tau || !flags) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  if (host) {
    const HostRows<const T*> in[5] = {{q, 12}, {quat_wxyz, 4}, {wrench, 6}, {mu, 4}, {normals_world, 12}};
    const HostRows<T*> out[3] = {{grf, 12}, {tau, 12}, {netwrench, 6}};
    return run_host_pipeline<T>(ctx, B, in, 5, stance_mask, out, 3, flags,
                                [&](size_t n, const T* const* i, const uint8_t* m, T* const* o, uint32_t* f, cudaStream_t st) {
                                  return solve_wrench_t<T>(ctx, n, i[0], i[1], i[2], m, i[3], i[4], o[0], o[1], f, o[2], st, false);
                                });
  }
  SolveArgsT<T> a;
  std::memset(&a, 0, sizeof a);
  a.B = B; a.q = q; a.quat = quat_wxyz; a.wrench = wrench; a.mask = stance_mask; a.mu = mu; a.normals = normals_world;
  a.grf = grf; a.tau = tau; a.flags = flags; a.netwrench = netwrench;
  a.model = Typed<T>::model(ctx); a.params = Typed<T>::params(ctx); a.params64 = ctx->d_params;
  return launch_solve<T, 0>(ctx, a, static_cast<cudaStream_t>(stream));
}

template <typename T>
int solve_state_t(qlb_context* ctx, size_t B, const T* q, const T* base_pose, const T* base_twist, const T* target_pose,
                  const T* target_twist, const uint8_t* stance_mask, const T* mu, const T* normals_world, T* grf, T* tau,
                  uint32_t* flags, T* netwrench, T* wrench_out, void* stream, bool host) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !base_pose || !base_twist || !target_pose || !target_twist || !stance_mask || !grf || !tau || !flags)
    return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  if (host) {
    const HostRows<const T*> in[7] = {{q, 12}, {base_pose, 7}, {base_twist, 6}, {target_pose, 7}, {target_twist, 6}, {mu, 4}, {normals_world, 12}};
    const HostRows<T*> out[4] = {{grf, 12}, {tau, 12}, {netwrench, 6}, {wrench_out, 6}};
    return run_host_pipeline<T>(ctx, B, in, 7, stance_mask, out, 4, flags,
                                [&](size_t n, const T* const* i, const uint8_t* m, T* const* o, uint32_t* f, cudaStream_t st) {
                                  return solve_state_t<T>(ctx, n, i[0], i[1], i[2], i[3], i[4], m, i[5], i[6], o[0], o[1], f, o[2],
                                                          o[3], st, false);
                                });
  }
  SolveArgsT<T> a;
  std::memset(&a, 0, sizeof a);
  a.B = B; a.q = q; a.pose = base_pose; a.twist = base_twist; a.tpose = target_pose; a.ttwist = target_twist;
  a.mask = stance_mask; a.mu = mu; a.normals = normals_world;
  a.grf = grf; a.tau = tau; a.flags = flags; a.netwrench = netwrench; a.wrench_out = wrench_out;
  a.model = Typed<T>::model(ctx); a.params = Typed<T>::params(ctx); a.params64 = ctx->d_params;
  return launch_solve<T, 1>(ctx, a, static_cast<cudaStream_t>(stream));
}

}  // namespace
}  // extern "C++"

int qlb_solve_wrench(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz, const double* wrench,
                     const uint8_t* stance_mask, const double* mu, const double* normals_world, double* grf,
                     double* tau, uint32_t* flags, double* netwrench, void* stream) {
  QLB_GUARD(ctx);
  return solve_wrench_t<double>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench, stream, false);
}
int qlb_solve_wrench_f32(qlb_context* ctx, size_t B, const float* q, const float* quat_wxyz, const float* wrench,
                         const uint8_t* stance_mask, const float* mu, const float* normals_world, float* grf, float* tau,
                         uint32_t* flags, float* netwrench, void* stream) {
  QLB_GUARD(ctx);
  return solve_wrench_t<float>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench, stream, false);
}
int qlb_solve_state(qlb_context* ctx, size_t B, const double* q, const double* base_pose, const double* base_twist,
                    const double* target_pose, const double* target_twist, const uint8_t* stance_mask,
                    const double* mu, const double* normals_world, double* grf, double* tau, uint32_t* flags,
                    double* netwrench, double* wrench_out, void* stream) {
  QLB_GUARD(ctx);
  return solve_state_t<double>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world, grf,
                               tau, flags, netwrench, wrench_out, stream, false);
}
int qlb_solve_state_f32(qlb_context* ctx, size_t B, const float* q, const float* base_pose, const float* base_twist,
                        const float* target_pose, const float* target_twist, const uint8_t* stance_mask, const float* mu,
                        const float* normals_world, float* grf, float* tau, uint32_t* flags, float* netwrench,
                        float* wrench_out, void* stream) {
  QLB_GUARD(ctx);
  return solve_state_t<float>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world, grf,
                              tau, flags, netwrench, wrench_out, stream, false);
}
int qlb_solve_wrench_host(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz, const double* wrench,
                          const uint8_t* stance_mask, const double* mu, const double* normals_world, double* grf,
                          double* tau, uint32_t* flags, double* netwrench) {
  QLB_GUARD(ctx);
  return solve_wrench_t<double>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench, nullptr, true);
}
int qlb_solve_wrench_f32_host(qlb_context* ctx, size_t B, const float* q, const float* quat_wxyz, const float* wrench,
                              const uint8_t* stance_mask, const float* mu, const float* normals_world, float* grf, float* tau,
                              uint32_t* flags, float* netwrench) {
  QLB_GUARD(ctx);
  return solve_wrench_t<float>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench, nullptr, true);
}
int qlb_solve_state_host(qlb_context* ctx, size_t B, const double* q, const double* base_pose, const double* base_twist,
                         const double* target_pose, const double* target_twist, const uint8_t* stance_mask,
                         const double* mu, const double* normals_world, double* grf, double* tau, uint32_t* flags,
                         double* netwrench, double* wrench_out) {
  QLB_GUARD(ctx);
  return solve_state_t<double>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world,
                               grf, tau, flags, netwrench, wrench_out, nullptr, true);
}
int qlb_solve_state_f32_host(qlb_context* ctx, size_t B, const float* q, const float* base_pose, const float* base_twist,
                             const float* target_pose, const float* target_twist, const uint8_t* stance_mask, const float* mu,
                             const float* normals_world, float* grf, float* tau, uint32_t* flags, float* netwrench,
                             float* wrench_out) {
  QLB_GUARD(ctx);
  return solve_state_t<float>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world,
                              grf, tau, flags, netwrench, wrench_out, nullptr, true);
}

int qlb_leg_kinematics(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz, double* foot, double* jac,
                       double* gravity_tau, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  return launch_items(ctx, B * 4ull, 128, static_cast<cudaStream_t>(stream), qlb_kinematics_kernel, (unsigned long long)B, q,
                      quat_wxyz, foot, jac, gravity_tau, ctx->d_model, ctx->d_params, nullptr, nullptr);
}

int qlb_pack_robot_states(qlb_context* ctx, size_t B, const qlb_robot_state_record* records, double* q, double* base_pose,
                          double* base_twist, uint8_t* stance_mask, double* normals_world, void* stream) {
  QLB_GUARD(ctx);
  static_assert(sizeof(qlb_robot_state_record) == 304, "record layout is part of the ABI");
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!records || !aligned16(records)) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  return launch_items(ctx, B, kPackTile, static_cast<cudaStream_t>(stream), qlb_pack_kernel, (unsigned long long)B, records, q,
                      base_pose, base_twist, stance_mask, normals_world);
}

int qlb_feet_in_world(qlb_context* ctx, size_t B, const double* q, const double* base_pose, double* feet_world, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !base_pose || !feet_world) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  return launch_items(ctx, B * 4ull, 128, static_cast<cudaStream_t>(stream), qlb_kinematics_kernel, (unsigned long long)B, q,
                      nullptr, nullptr, nullptr, nullptr, ctx->d_model, ctx->d_params, base_pose, feet_world);
}

int qlb_default_swing_params(qlb_swing_params* p) {
  if (!p) return QLB_ERR_INVALID_ARGUMENT;
  std::memset(p, 0, sizeof *p);
  p->gravity[1] = -9.81;            // the dynamics library's default, never overridden for the limb models
  p->acceleration_scale = 0.5;      // model_test_header.cpp:460
  return QLB_OK;
}

int qlb_set_limb_dynamics(qlb_context* ctx, const qlb_limb_dynamics legs[QLB_NUM_LEGS]) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (!legs) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  DeviceLimbDynamics h;
  std::memset(&h, 0, sizeof h);
  for (int l = 0; l < 4; l++)
    for (int j = 0; j < 3; j++) {
      rpy_to_rot(legs[l].joint_rpy[j], h.rot[l][j]);
      for (int a = 0; a < 3; a++) { h.xyz[l][j][a] = legs[l].joint_xyz[j][a]; h.com[l][j][a] = legs[l].body_com[j][a]; }
      h.mass[l][j] = legs[l].body_mass[j];
      for (int a = 0; a < 6; a++) h.inertia[l][j][a] = legs[l].body_inertia[j][a];
    }
  // FP32 copy: same fields, rounded once on the host (as narrow_model)
  DeviceLimbDynamicsT<float> hf;
  static_assert(sizeof hf * 2 == sizeof h, "the FP32 copy narrows every field");
  const double* src = reinterpret_cast<const double*>(&h);
  float* dst = reinterpret_cast<float*>(&hf);
  for (size_t i = 0; i < sizeof h / sizeof(double); i++) dst[i] = (float)src[i];
  if (!ctx->d_limb && cudaMalloc(&ctx->d_limb, sizeof h) != cudaSuccess) { cudaGetLastError(); return QLB_ERR_ALLOC; }
  if (!ctx->d_limb_f && cudaMalloc(&ctx->d_limb_f, sizeof hf) != cudaSuccess) { cudaGetLastError(); return QLB_ERR_ALLOC; }
  QLB_CUDA(ctx, cudaDeviceSynchronize());
  QLB_CUDA(ctx, cudaMemcpy(ctx->d_limb, &h, sizeof h, cudaMemcpyHostToDevice));
  QLB_CUDA(ctx, cudaMemcpy(ctx->d_limb_f, &hf, sizeof hf, cudaMemcpyHostToDevice));
  ctx->have_limb = true;
  return QLB_OK;
}

extern "C++" {
namespace {
// The swing-leg arguments every caller fills alike; the caller sets qdd, or qd_front / ld_front / inv_window.
template <typename T>
void fill_swing(SwingArgsT<T>& s, const qlb_context* ctx, const qlb_swing_params& p, size_t B, const T* q, const T* qd,
                const T* ptarget, const T* vtarget, T* tau) {
  std::memset(&s, 0, sizeof s);
  s.B = B; s.q = q; s.qd = qd; s.ptarget = ptarget; s.vtarget = vtarget; s.tau = tau;
  for (int k = 0; k < 3; k++) { s.gravity[k] = (T)p.gravity[k]; s.kp[k] = (T)p.kp[k]; s.kd[k] = (T)p.kd[k]; }
  s.acc_scale = (T)p.acceleration_scale;
  s.dyn = Typed<T>::limb(ctx); s.model = Typed<T>::model(ctx);
}

// qlb_swing_leg_torques and its host twin: checks, then one launch on `stream`, or chunks of the staging capacity on
// the context stream
int swing_leg_torques(qlb_context* ctx, size_t B, const double* q, const double* qd, const double* qdd,
                      const double* foot_target_position, const double* foot_target_velocity, const qlb_swing_params* params,
                      double* tau, void* stream, bool host) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (!ctx->have_limb) return QLB_ERR_NOT_INITIALISED;   // qlb_set_limb_dynamics first
  if (B == 0) return QLB_OK;
  if (!q || !qd || !qdd || !params || !tau) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  if (host) {
    QLB_TRY(reserve_soa(ctx, B));
    const size_t cap = ctx->cap;   // the input staging area holds kPipe * cap * 54 doubles >= 5 * 12 * cap
    static_assert(kPipe * kHostInRows >= 60 && kPipe * kHostOutRows >= 12, "staging too small for the swing-leg arrays");
    const SoaSlot s = soa_slot(ctx, 0);
    const double* src[5] = {q, qd, qdd, foot_target_position, foot_target_velocity};
    return for_chunks(ctx, B, cap, false, [&](size_t b0, size_t n, int, cudaStream_t st) -> int {
      const double* dptr[5];
      for (int k = 0; k < 5; k++) {
        double* d = s.in + (size_t)k * 12 * cap;
        dptr[k] = src[k] ? d : nullptr;
        QLB_TRY(rows_to_device(ctx, d, src[k], 12, b0, n, B, st));
      }
      QLB_TRY(swing_leg_torques(ctx, n, dptr[0], dptr[1], dptr[2], dptr[3], dptr[4], params, s.out, st, false));
      return rows_to_host(ctx, tau, s.out, 12, b0, n, B, st);
    });
  }
  SwingArgs a;
  fill_swing(a, ctx, *params, B, q, qd, foot_target_position, foot_target_velocity, tau);
  a.qdd = qdd;
  return launch_items(ctx, B * 4ull, 128, static_cast<cudaStream_t>(stream), qlb_swing_kernel, a);
}
}  // namespace
}  // extern "C++"

int qlb_swing_leg_torques(qlb_context* ctx, size_t B, const double* q, const double* qd, const double* qdd,
                          const double* foot_target_position, const double* foot_target_velocity,
                          const qlb_swing_params* params, double* tau, void* stream) {
  QLB_GUARD(ctx);
  return swing_leg_torques(ctx, B, q, qd, qdd, foot_target_position, foot_target_velocity, params, tau, stream, false);
}

// HOST pointers: staged through the context's SoA staging in chunks, on the context stream; synchronises.
int qlb_swing_leg_torques_host(qlb_context* ctx, size_t B, const double* q, const double* qd, const double* qdd,
                               const double* foot_target_position, const double* foot_target_velocity,
                               const qlb_swing_params* params, double* tau) {
  QLB_GUARD(ctx);
  return swing_leg_torques(ctx, B, q, qd, qdd, foot_target_position, foot_target_velocity, params, tau, nullptr, true);
}

int qlb_swing_leg_torques_from_queue(qlb_context* ctx, size_t B, const double* q, const double* qd_back, const double* qd_front,
                                     double period, const double* foot_target_position, const double* foot_target_velocity,
                                     const qlb_swing_params* params, double* tau, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (!ctx->have_limb) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !qd_back || !qd_front || !params || !tau || !(period > 0.0)) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  SwingArgs a;
  fill_swing(a, ctx, *params, B, q, qd_back, foot_target_position, foot_target_velocity, tau);
  a.qd_front = qd_front; a.ld_front = B; a.inv_window = 1.0 / (10.0 * period);
  return launch_items(ctx, B * 4ull, 128, static_cast<cudaStream_t>(stream), qlb_swing_kernel, a);
}

int qlb_contact_fsm(qlb_context* ctx, size_t B, const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                    const uint8_t* contact_mask, const double* phase, uint8_t* limb_state, uint8_t* stance_mask, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!desired_stance_mask || !contact_mask || !phase || !limb_state) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  return launch_items(ctx, B, 256, static_cast<cudaStream_t>(stream), qlb_contact_fsm_kernel, (unsigned long long)B,
                      desired_stance_mask, footstep_mask, contact_mask, phase, limb_state, stance_mask);
}

int qlb_friction_margins(qlb_context* ctx, size_t B, const double* grf, const double* quat_wxyz, const uint8_t* stance_mask,
                         const double* mu, const double* normals_world, double* margin, double* min_normal, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!grf || !quat_wxyz || !stance_mask || !margin) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  return launch_items(ctx, B, 256, static_cast<cudaStream_t>(stream), qlb_friction_margin_kernel, (unsigned long long)B, grf,
                      quat_wxyz, stance_mask, mu, normals_world, ctx->d_params, margin, min_normal);
}

namespace {
// one chunk of records on one stream: unpack, solve, pack (device pointers; `slot` selects the SoA staging area)
int records_chunk(qlb_context* ctx, size_t n, const qlb_wrench_record* d_in, qlb_result_record* d_out, int slot, cudaStream_t st) {
  const size_t cap = ctx->cap;
  const SoaSlot s = soa_slot(ctx, slot);
  double* q = s.in; double* quat = s.in + 12 * cap; double* wrench = s.in + 16 * cap; double* mu = s.in + 22 * cap;
  double* grf = s.out; double* tau = s.out + 12 * cap; double* net = s.out + 24 * cap;
  // the SoA staging rows have pitch n inside this chunk
  QLB_TRY(launch_items(ctx, n, kRecTile, st, qlb_unpack_records_kernel, (unsigned long long)n, d_in, q, quat, wrench, mu, s.mask));
  QLB_TRY(solve_wrench_t<double>(ctx, n, q, quat, wrench, s.mask, mu, nullptr, grf, tau, s.flags, net, st, false));
  return launch_items(ctx, n, kRecTile, st, qlb_pack_results_kernel, (unsigned long long)n, grf, tau, net, s.flags, d_out);
}

// qlb_solve_records and its host twin: checks, then the chunks on `stream` (one staging area: the caller's arrays are
// already on the device, nothing to overlap), or on the pipeline with one 1-D copy per chunk and direction
int solve_records(qlb_context* ctx, size_t B, const qlb_wrench_record* records, qlb_result_record* results, void* stream,
                  bool host) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!records || !results) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  QLB_TRY(reserve_soa(ctx, B));
  const size_t cap = ctx->cap;
  if (host) {
    constexpr size_t per_state = sizeof(qlb_wrench_record) + sizeof(qlb_result_record);
    QLB_TRY(reserve(ctx, ctx->rec, kPipe * cap * per_state));
    return for_chunks(ctx, B, cap, true, [&](size_t b0, size_t n, int slot, cudaStream_t st) -> int {
      unsigned char* base = ctx->rec.p + (size_t)slot * cap * per_state;
      qlb_wrench_record* d_in = reinterpret_cast<qlb_wrench_record*>(base);
      qlb_result_record* d_out = reinterpret_cast<qlb_result_record*>(base + cap * sizeof(qlb_wrench_record));
      QLB_CUDA(ctx, cudaMemcpyAsync(d_in, records + b0, n * sizeof(qlb_wrench_record), cudaMemcpyHostToDevice, st));
      QLB_TRY(records_chunk(ctx, n, d_in, d_out, slot, st));
      QLB_CUDA(ctx, cudaMemcpyAsync(results + b0, d_out, n * sizeof(qlb_result_record), cudaMemcpyDeviceToHost, st));
      return QLB_OK;
    });
  }
  // the only asynchronous user of the SoA staging: ordered after the previous one, and recorded (on failure too) for
  // the next user to wait on
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  QLB_CUDA(ctx, cudaStreamWaitEvent(st, ctx->soa_free, 0));
  int rc = QLB_OK;
  for (size_t b0 = 0; b0 < B && rc == QLB_OK; b0 += cap)
    rc = records_chunk(ctx, B - b0 < cap ? B - b0 : cap, records + b0, results + b0, 0, st);
  const cudaError_t e = cudaEventRecord(ctx->soa_free, st);
  if (e != cudaSuccess && rc == QLB_OK) rc = cuda_fail(ctx, e, "cudaEventRecord");
  return rc;
}
}  // namespace

int qlb_solve_records(qlb_context* ctx, size_t B, const qlb_wrench_record* records, qlb_result_record* results, void* stream) {
  QLB_GUARD(ctx);
  return solve_records(ctx, B, records, results, stream, false);
}

int qlb_solve_records_host(qlb_context* ctx, size_t B, const qlb_wrench_record* records, qlb_result_record* results) {
  QLB_GUARD(ctx);
  return solve_records(ctx, B, records, results, nullptr, true);
}

int qlb_preview_plan_host(qlb_context* ctx, size_t B, const qlb_robot_state_record* records, const double mu[4],
                          qlb_preview_record* preview) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!records || !preview) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  QLB_TRY(reserve_soa(ctx, B));
  const size_t cap = ctx->cap;
  // per state: the input record, the result record, and SoA rows for feet (12), friction coefficients (4), margins (2)
  constexpr size_t per_state = sizeof(qlb_robot_state_record) + sizeof(qlb_preview_record) + 18 * sizeof(double);
  QLB_TRY(reserve(ctx, ctx->prev, cap * per_state));
  qlb_robot_state_record* d_rec = reinterpret_cast<qlb_robot_state_record*>(ctx->prev.p);
  qlb_preview_record* d_res = reinterpret_cast<qlb_preview_record*>(ctx->prev.p + cap * sizeof(qlb_robot_state_record));
  double* extra = reinterpret_cast<double*>(ctx->prev.p + cap * (sizeof(qlb_robot_state_record) + sizeof(qlb_preview_record)));
  double* feet = extra; double* dmu = mu ? extra + 12 * cap : nullptr; double* margin = extra + 16 * cap; double* minn = extra + 17 * cap;
  const SoaSlot s = soa_slot(ctx, 0);
  double* q = s.in; double* pose = s.in + 12 * cap; double* twist = s.in + 19 * cap; double* nrm = s.in + 25 * cap;
  double* grf = s.out; double* tau = s.out + 12 * cap; double* net = s.out + 24 * cap; double* wout = s.out + 30 * cap;
  return for_chunks(ctx, B, cap, false, [&](size_t b0, size_t n, int, cudaStream_t st) -> int {
    QLB_CUDA(ctx, cudaMemcpyAsync(d_rec, records + b0, n * sizeof(qlb_robot_state_record), cudaMemcpyHostToDevice, st));
    QLB_TRY(qlb_pack_robot_states(ctx, n, d_rec, q, pose, twist, s.mask, nrm, st));
    QLB_TRY(qlb_feet_in_world(ctx, n, q, pose, feet, st));
    if (mu) QLB_TRY(launch_items(ctx, n, 256, st, qlb_fill_rows_kernel, (unsigned long long)n, 4, dmu, mu[0], mu[1], mu[2], mu[3]));
    // the planned state is feedback AND target: zero tracking error
    QLB_TRY(solve_state_t<double>(ctx, n, q, pose, twist, pose, twist, s.mask, dmu, nrm, grf, tau, s.flags, net, wout, st, false));
    QLB_TRY(qlb_friction_margins(ctx, n, grf, pose + 3 * n, s.mask, dmu, nrm, margin, minn, st));
    QLB_TRY(launch_items(ctx, n, kPrevTile, st, qlb_pack_preview_kernel, (unsigned long long)n, feet, grf, tau, net, wout, margin,
                         minn, s.flags, d_res));
    QLB_CUDA(ctx, cudaMemcpyAsync(preview + b0, d_res, n * sizeof(qlb_preview_record), cudaMemcpyDeviceToHost, st));
    return QLB_OK;
  });
}

namespace {
int generate_common(qlb_context* ctx, int config, size_t B, uint64_t start, uint64_t seed, GenArgs& g, void* stream) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (config == 4) config = 3;   // C4 = the C3 states through the FP32 interface
  if (config != 1 && config != 2 && config != 3 && config != 5) return QLB_ERR_INVALID_ARGUMENT;
  if (B == 0) return QLB_OK;
  DeviceGuard guard(ctx->device);
  g.B = B; g.start = start; g.config = config;
  g.seed = seed ? seed : (0x5EED0000ull + (unsigned long long)config);
  return launch_items(ctx, B, 256, static_cast<cudaStream_t>(stream), qlb_generate_kernel, g);
}
}  // namespace

int qlb_generate_states(qlb_context* ctx, int config, size_t B, uint64_t start, uint64_t seed, double* q, double* quat_wxyz,
                        double* wrench, uint8_t* stance_mask, double* mu, double* normals_world, void* stream) {
  QLB_GUARD(ctx);
  GenArgs g;
  std::memset(&g, 0, sizeof g);
  g.q = q; g.quat = quat_wxyz; g.wrench = wrench; g.mask = stance_mask; g.mu = mu; g.normals = normals_world;
  return generate_common(ctx, config, B, start, seed, g, stream);
}

int qlb_generate_states_f32(qlb_context* ctx, int config, size_t B, uint64_t start, uint64_t seed, float* q, float* quat_wxyz,
                            float* wrench, uint8_t* stance_mask, float* mu, float* normals_world, void* stream) {
  QLB_GUARD(ctx);
  GenArgs g;
  std::memset(&g, 0, sizeof g);
  g.q32 = q; g.quat32 = quat_wxyz; g.wrench32 = wrench; g.mask = stance_mask; g.mu32 = mu; g.normals32 = normals_world;
  return generate_common(ctx, config, B, start, seed, g, stream);
}

int qlb_batch_stats(qlb_context* ctx, size_t B, const uint32_t* flags, const double* wrench, const double* netwrench,
                    qlb_stats* stats_out, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (!flags || !stats_out) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  QLB_CUDA(ctx, cudaMemsetAsync(ctx->d_stats, 0, QLB_STATS_NUM * sizeof(double), st));
  if (B > 0) {
    const unsigned threads = 256;
    unsigned long long blocks = (B + threads - 1) / threads;
    const unsigned long long cap = (unsigned long long)ctx->sm_count * 8ull;   // resident in one wave: a grid-stride loop per thread
    if (blocks > cap) blocks = cap;
    qlb_stats_kernel<<<(unsigned)blocks, threads, 0, st>>>(B, flags, wrench, netwrench, ctx->d_params, ctx->d_stats);
    QLB_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
  }
  double h[QLB_STATS_NUM];
  QLB_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_stats, sizeof h, cudaMemcpyDeviceToHost, st));
  QLB_CUDA(ctx, cudaStreamSynchronize(st));
  std::memcpy(stats_out, h, sizeof h);
  return QLB_OK;
}

// The one collective of the design (SURVEY 8e): all-reduce of the statistics vector over the ranks of an NCCL
// communicator.  NCCL is resolved at run time (dlopen of libnccl.so.2: the copy already loaded by the process - the
// caller created `comm` with it - or the system library), so libqlb.so itself has no link-time dependency on it.
namespace {
struct NcclApi {
  ncclResult_t (*all_reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*group_start)() = nullptr;
  ncclResult_t (*group_end)() = nullptr;
  bool ok = false;
};
const NcclApi& nccl_api() {
  static NcclApi api = []() {
    NcclApi a;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return a;
    a.all_reduce = reinterpret_cast<decltype(a.all_reduce)>(dlsym(h, "ncclAllReduce"));
    a.group_start = reinterpret_cast<decltype(a.group_start)>(dlsym(h, "ncclGroupStart"));
    a.group_end = reinterpret_cast<decltype(a.group_end)>(dlsym(h, "ncclGroupEnd"));
    a.ok = a.all_reduce && a.group_start && a.group_end;
    return a;
  }();
  return api;
}
}  // namespace

int qlb_stats_allreduce(qlb_context* ctx, void* nccl_comm, qlb_stats* stats, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (!nccl_comm || !stats) return QLB_ERR_INVALID_ARGUMENT;
  const NcclApi& nccl = nccl_api();
  if (!nccl.ok) {
    std::snprintf(ctx->last_error, sizeof ctx->last_error, "libnccl.so.2 not found");
    return QLB_ERR_CUDA;
  }
  DeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ncclComm_t comm = static_cast<ncclComm_t>(nccl_comm);
  static_assert(sizeof(qlb_stats) == QLB_STATS_NUM * sizeof(double), "qlb_stats is a vector of doubles");
  QLB_CUDA(ctx, cudaMemcpyAsync(ctx->d_stats, stats, sizeof(qlb_stats), cudaMemcpyHostToDevice, st));
  bool ok = nccl.group_start() == ncclSuccess;
  ok = ok && nccl.all_reduce(ctx->d_stats, ctx->d_stats, QLB_STATS_NUM_SUM, ncclDouble, ncclSum, comm, st) == ncclSuccess;
  ok = ok && nccl.all_reduce(ctx->d_stats + QLB_STATS_NUM_SUM, ctx->d_stats + QLB_STATS_NUM_SUM, QLB_STATS_NUM - QLB_STATS_NUM_SUM,
                             ncclDouble, ncclMax, comm, st) == ncclSuccess;
  ok = (nccl.group_end() == ncclSuccess) && ok;
  if (!ok) {
    std::snprintf(ctx->last_error, sizeof ctx->last_error, "ncclAllReduce failed");
    return QLB_ERR_CUDA;
  }
  QLB_CUDA(ctx, cudaMemcpyAsync(stats, ctx->d_stats, sizeof(qlb_stats), cudaMemcpyDeviceToHost, st));
  QLB_CUDA(ctx, cudaStreamSynchronize(st));
  return QLB_OK;
}

extern "C++" {
namespace {
// qlb_qp_dense and its host twin: checks, then one launch on `stream`, or one call on the context stream through the
// context's staging
int qp_dense(qlb_context* ctx, size_t B, int n, int m, int p, const double* G, const double* g0, const double* CE,
             const double* ce0, const double* CI, const double* ci0, double* x, double* cost, uint32_t* status,
             uint32_t* active, void* stream, bool host) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (n < 1 || n > kQpMaxN || m < 0 || m > kQpMaxM || p < 0 || p > kQpMaxP) return QLB_ERR_INVALID_ARGUMENT;
  if (B == 0) return QLB_OK;
  if (!G || !g0 || !x || !status || (p > 0 && (!CE || !ce0)) || (m > 0 && (!CI || !ci0))) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  if (host) {
    const size_t nin = (size_t)(n * n + n + n * p + p + n * m + m) * B, nout = (size_t)(n + 1) * B;
    // grown on demand (a controller calls this every tick with the same shape)
    QLB_TRY(reserve(ctx, ctx->qp, pow2_at_least((nin + nout) * sizeof(double) + 2 * B * sizeof(uint32_t), 4096)));
    double* dG = reinterpret_cast<double*>(ctx->qp.p); double* dg = dG + (size_t)n * n * B; double* dCE = dg + (size_t)n * B;
    double* dce = dCE + (size_t)n * p * B; double* dCI = dce + (size_t)p * B; double* dci = dCI + (size_t)n * m * B;
    double* d_out = dG + nin;
    uint32_t* d_u = reinterpret_cast<uint32_t*>(d_out + nout);
    if (p == 0) CE = ce0 = nullptr;   // may be set; nothing to copy
    if (m == 0) CI = ci0 = nullptr;
    return for_chunks(ctx, B, B, false, [&](size_t, size_t, int, cudaStream_t st) -> int {
      QLB_TRY(rows_to_device(ctx, dG, G, (size_t)n * n, 0, B, B, st));
      QLB_TRY(rows_to_device(ctx, dg, g0, n, 0, B, B, st));
      QLB_TRY(rows_to_device(ctx, dCE, CE, (size_t)n * p, 0, B, B, st));
      QLB_TRY(rows_to_device(ctx, dce, ce0, p, 0, B, B, st));
      QLB_TRY(rows_to_device(ctx, dCI, CI, (size_t)n * m, 0, B, B, st));
      QLB_TRY(rows_to_device(ctx, dci, ci0, m, 0, B, B, st));
      QLB_TRY(qp_dense(ctx, B, n, m, p, dG, dg, p ? dCE : nullptr, p ? dce : nullptr, m ? dCI : nullptr, m ? dci : nullptr,
                       d_out, d_out + (size_t)n * B, d_u, d_u + B, st, false));
      QLB_TRY(rows_to_host(ctx, x, d_out, n, 0, B, B, st));
      QLB_TRY(rows_to_host(ctx, cost, d_out + (size_t)n * B, 1, 0, B, B, st));
      QLB_TRY(rows_to_host(ctx, status, d_u, 1, 0, B, B, st));
      return rows_to_host(ctx, active, d_u + B, 1, 0, B, B, st);
    });
  }
  QpDenseArgs a;
  a.B = B; a.n = n; a.m = m; a.p = p; a.G = G; a.g0 = g0; a.CE = CE; a.ce0 = ce0; a.CI = CI; a.ci0 = ci0;
  a.x = x; a.cost = cost; a.status = status; a.active = active;
  // one warp per problem, four problems per CTA, grid-stride over the batch
  unsigned long long blocks = (B + kQpWarpsPerCta - 1) / kQpWarpsPerCta;
  const unsigned long long cap = (unsigned long long)ctx->sm_count * 8ull;
  if (blocks > cap) blocks = cap;
  qlb_qp_dense_kernel<<<(unsigned)blocks, 32 * kQpWarpsPerCta, 0, static_cast<cudaStream_t>(stream)>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}
}  // namespace
}  // extern "C++"

int qlb_qp_dense(qlb_context* ctx, size_t B, int n, int m, int p, const double* G, const double* g0, const double* CE,
                 const double* ce0, const double* CI, const double* ci0, double* x, double* cost, uint32_t* status,
                 uint32_t* active, void* stream) {
  QLB_GUARD(ctx);
  return qp_dense(ctx, B, n, m, p, G, g0, CE, ce0, CI, ci0, x, cost, status, active, stream, false);
}

int qlb_qp_dense_host(qlb_context* ctx, size_t B, int n, int m, int p, const double* G, const double* g0,
                      const double* CE, const double* ce0, const double* CI, const double* ci0, double* x, double* cost,
                      uint32_t* status, uint32_t* active) {
  QLB_GUARD(ctx);
  return qp_dense(ctx, B, n, m, p, G, g0, CE, ce0, CI, ci0, x, cost, status, active, nullptr, true);
}

int qlb_measure_fp64_peak(qlb_context* ctx, double* tflops_out) {
  QLB_GUARD(ctx);
  if (!ctx || !tflops_out) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  cudaStream_t st = ctx->stream;
  cudaEvent_t e0, e1;
  QLB_CUDA(ctx, cudaEventCreate(&e0));
  QLB_CUDA(ctx, cudaEventCreate(&e1));
  const int iters = 4096, threads = 256;
  const int blocks = ctx->sm_count * 8;
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    QLB_CUDA(ctx, cudaEventRecord(e0, st));
    qlb_fp64_peak_kernel<<<blocks, threads, 0, st>>>(ctx->d_stats, iters, 1.0 + rep);
    QLB_CUDA(ctx, cudaGetLastError());
    QLB_CUDA(ctx, cudaEventRecord(e1, st));
    QLB_CUDA(ctx, cudaEventSynchronize(e1));
    float ms = 0.f;
    QLB_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * 16.0 * (double)iters * (double)threads * (double)blocks;
    const double tf = flops / (ms * 1e-3) * 1e-12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tflops_out = best;
  return QLB_OK;
}

}  // extern "C"

// ---- the controller tick (qlb_controller_*)
struct qlb_controller {
  qlb_context* ctx = nullptr;
  size_t B = 0;
  qlb_tick_params p;
  int head = 0;                 // ring slot of the next tick's sample
  cudaEvent_t reset_done = nullptr;   // recorded by qlb_controller_reset: every update waits for it, whatever its stream
  uint8_t* limb = nullptr;      // [4][B]
  uint8_t* refill = nullptr;    // [B]
  double* efforts = nullptr;    // [12][B]
  double* ring = nullptr;       // [kTickRing][12][B]
  uint8_t* stance = nullptr;    // scratch [B]: stance mask of the current tick
  double* tau = nullptr;        // scratch [12][B]: torques of the solve
  double* grf = nullptr;        // scratch [12][B]: forces of the solve when the caller passes none
};

namespace {

// One tick for robots b0 .. b0 + n - 1 of the controller; the caller's arrays have row pitch n.  T = float: the
// swing legs in FP32 on the FP32 tables, the stance legs by solve_state_t<float> on the scratch reinterpreted as float
// (12 n doubles hold 12 n floats); the solver core follows the context's qlb_set_f32_core.
template <typename T>
int controller_tick(qlb_controller* c, size_t n, size_t b0, const T* q, const T* qd, const T* pose, const T* twist,
                    const T* tpose, const T* ttwist, const uint8_t* desired, const uint8_t* footstep, const uint8_t* contact,
                    const T* phase, const T* mu, const T* normals, const T* ptarget, const T* vtarget, T* command,
                    uint32_t* flags, T* grf, cudaStream_t st) {
  qlb_context* ctx = c->ctx;
  const size_t ld = c->B;
  T* tau = reinterpret_cast<T*>(c->tau);
  TickArgsT<T> a;
  std::memset(&a, 0, sizeof a);
  a.n = n; a.ld = ld; a.head = c->head;
  a.desired = desired; a.footstep = footstep; a.contact = contact; a.phase = phase; a.qd = qd;
  a.limb = c->limb + b0; a.refill = c->refill + b0; a.ring = c->ring + b0; a.stance = c->stance;
  a.flags = flags; a.tau = tau; a.efforts = c->efforts + b0; a.command = command; a.limit = c->p.effort_limit;
  fill_swing<T>(a.swing, ctx, c->p.swing, n, q, qd, ptarget, vtarget, nullptr);
  a.swing.qd_front = c->ring + (size_t)((c->head + 1) % kTickRing) * 12 * ld + b0; a.swing.ld_front = ld;
  a.swing.inv_window = (T)(1.0 / (10.0 * c->p.period));
  QLB_CUDA(ctx, cudaStreamWaitEvent(st, c->reset_done, 0));
  QLB_TRY(launch_items(ctx, n, 256, st, qlb_tick_prologue_kernel<T>, a));
  QLB_TRY(solve_state_t<T>(ctx, n, q, pose, twist, tpose, ttwist, c->stance, mu, normals, grf ? grf : reinterpret_cast<T*>(c->grf),
                           tau, flags, nullptr, nullptr, st, false));
  return launch_items(ctx, 4ull * n, 128, st, qlb_tick_epilogue_kernel<T>, a);
}

// qlb_controller_update[_f32] and the host twins: checks, then one tick of the whole batch on `stream`, or chunks of the
// context's staging capacity one after the other on the context stream (they share the controller's stance and tau
// scratch, which is not offset by b0).  The staging is sized for FP64; the FP32 twin uses the same row offsets in
// float, i.e. the first half.
template <typename T>
int controller_update_t(qlb_controller* c, const T* q, const T* qd, const T* base_pose, const T* base_twist,
                        const T* target_pose, const T* target_twist, const uint8_t* desired_stance_mask,
                        const uint8_t* footstep_mask, const uint8_t* contact_mask, const T* phase, const T* mu,
                        const T* normals_world, const T* foot_target_position, const T* foot_target_velocity, T* command,
                        uint32_t* flags, T* grf, void* stream, bool host) {
  if (!c) return QLB_ERR_NOT_INITIALISED;
  QLB_GUARD(c->ctx);
  if (!c->ctx || !c->ctx->have_limb) return QLB_ERR_NOT_INITIALISED;   // qlb_set_limb_dynamics first
  if (!q || !qd || !base_pose || !base_twist || !target_pose || !target_twist || !desired_stance_mask || !contact_mask ||
      !phase || !command || !flags)
    return QLB_ERR_INVALID_ARGUMENT;
  qlb_context* ctx = c->ctx;
  DeviceGuard guard(ctx->device);
  const size_t B = c->B;
  int rc;
  if (!host) {
    rc = controller_tick<T>(c, B, 0, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask, footstep_mask,
                            contact_mask, phase, mu, normals_world, foot_target_position, foot_target_velocity, command, flags,
                            grf, static_cast<cudaStream_t>(stream));
  } else {
    QLB_TRY(reserve_soa(ctx, B));
    const size_t cap = ctx->cap;
    const SoaSlot s = soa_slot(ctx, 0);
    // inputs: 94 rows in the input staging (kPipe * 54 rows of cap), outputs 24 rows, the three masks one row each
    constexpr int kIn = 11, kOut = 2;
    const T* src[kIn] = {q, qd, base_pose, base_twist, target_pose, target_twist, phase, mu, normals_world,
                         foot_target_position, foot_target_velocity};
    const int rows[kIn] = {12, 12, 7, 6, 7, 6, 4, 4, 12, 12, 12};
    static_assert(kPipe * kHostInRows >= 94 && kPipe * kHostOutRows >= 24 && kPipe >= 3, "staging too small for a tick");
    const uint8_t* msrc[3] = {desired_stance_mask, footstep_mask, contact_mask};
    T* const dst_out[kOut] = {command, grf};
    T* const dout[kOut] = {reinterpret_cast<T*>(s.out), reinterpret_cast<T*>(s.out) + 12 * cap};
    rc = for_chunks(ctx, B, cap, false, [&](size_t b0, size_t n, int, cudaStream_t st) -> int {
      const T* din[kIn];
      T* d = reinterpret_cast<T*>(s.in);
      for (int k = 0; k < kIn; d += (size_t)rows[k] * cap, k++) {
        din[k] = src[k] ? d : nullptr;
        QLB_TRY(rows_to_device(ctx, d, src[k], rows[k], b0, n, B, st));
      }
      const uint8_t* dmask[3];
      for (int k = 0; k < 3; k++) {
        dmask[k] = msrc[k] ? s.mask + (size_t)k * cap : nullptr;
        if (msrc[k]) QLB_CUDA(ctx, cudaMemcpyAsync(s.mask + (size_t)k * cap, msrc[k] + b0, n, cudaMemcpyHostToDevice, st));
      }
      QLB_TRY(controller_tick<T>(c, n, b0, din[0], din[1], din[2], din[3], din[4], din[5], dmask[0], dmask[1], dmask[2], din[6],
                                 din[7], din[8], din[9], din[10], dout[0], s.flags, dout[1], st));
      for (int k = 0; k < kOut; k++) QLB_TRY(rows_to_host(ctx, dst_out[k], dout[k], 12, b0, n, B, st));
      QLB_CUDA(ctx, cudaMemcpyAsync(flags + b0, s.flags, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      return QLB_OK;
    });
  }
  if (rc == QLB_OK) c->head = (c->head + 1) % kTickRing;
  return rc;
}

}  // namespace

extern "C" {

int qlb_default_tick_params(qlb_tick_params* p) {
  if (!p) return QLB_ERR_INVALID_ARGUMENT;
  std::memset(p, 0, sizeof *p);
  p->period = 0.0025;        // 400 Hz (balance_controller_manager.cpp:48,70)
  p->effort_limit = 300.0;   // RBC.cpp:450-454
  return qlb_default_swing_params(&p->swing);
}

int qlb_controller_create(qlb_context* ctx, size_t B, const qlb_tick_params* params, qlb_controller** out) {
  static_assert(sizeof(qlb_tick_params) == 96, "qlb_tick_params layout is part of the ABI");
  if (!out) return QLB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    cudaGetLastError();
    return QLB_ERR_CUDA;
  }
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  qlb_tick_params defaults;
  qlb_default_tick_params(&defaults);
  const qlb_tick_params* p = params ? params : &defaults;
  if (B == 0 || !(p->period > 0.0) || !std::isfinite(p->period) || !(p->effort_limit >= 0.0) || !std::isfinite(p->effort_limit))
    return QLB_ERR_INVALID_ARGUMENT;
  if (B > 0xFFFFFFF0ull) return QLB_ERR_BATCH_TOO_LARGE;
  QLB_GUARD(ctx);
  DeviceGuard guard(ctx->device);
  qlb_controller* c = new (std::nothrow) qlb_controller();
  if (!c) return QLB_ERR_ALLOC;
  c->ctx = ctx; c->B = B; c->p = *p;
  if (cudaMalloc(&c->limb, 4 * B) != cudaSuccess || cudaMalloc(&c->refill, B) != cudaSuccess ||
      cudaMalloc(&c->stance, B) != cudaSuccess || cudaMalloc(&c->efforts, 12 * B * sizeof(double)) != cudaSuccess ||
      cudaMalloc(&c->ring, (size_t)kTickRing * 12 * B * sizeof(double)) != cudaSuccess ||
      cudaMalloc(&c->tau, 12 * B * sizeof(double)) != cudaSuccess || cudaMalloc(&c->grf, 12 * B * sizeof(double)) != cudaSuccess) {
    cudaGetLastError();
    qlb_controller_destroy(c);
    return QLB_ERR_ALLOC;
  }
  if (cudaEventCreateWithFlags(&c->reset_done, cudaEventDisableTiming) != cudaSuccess) {
    const int rc = cuda_fail(ctx, cudaGetLastError(), "qlb_controller_create");
    qlb_controller_destroy(c);
    return rc;
  }
  static_assert(QLB_LIMB_INIT == 0, "limb states start as zero bytes");
  if (cudaMemsetAsync(c->limb, 0, 4 * B, ctx->stream) != cudaSuccess || cudaMemsetAsync(c->refill, 1, B, ctx->stream) != cudaSuccess ||
      cudaMemsetAsync(c->efforts, 0, 12 * B * sizeof(double), ctx->stream) != cudaSuccess ||
      cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
    const int rc = cuda_fail(ctx, cudaGetLastError(), "qlb_controller_create");
    qlb_controller_destroy(c);
    return rc;
  }
  *out = c;
  return QLB_OK;
}

int qlb_controller_destroy(qlb_controller* c) {
  if (!c) return QLB_OK;
  QLB_GUARD(c->ctx);
  DeviceGuard guard(c->ctx->device);
  cudaFree(c->limb); cudaFree(c->refill); cudaFree(c->stance); cudaFree(c->efforts); cudaFree(c->ring);
  cudaFree(c->tau); cudaFree(c->grf);
  if (c->reset_done) cudaEventDestroy(c->reset_done);
  cudaGetLastError();
  delete c;
  return QLB_OK;
}

int qlb_controller_reset(qlb_controller* c, const uint8_t* reset_mask, void* stream) {
  if (!c) return QLB_ERR_NOT_INITIALISED;
  QLB_GUARD(c->ctx);
  DeviceGuard guard(c->ctx->device);
  QLB_TRY(launch_items(c->ctx, c->B, 256, static_cast<cudaStream_t>(stream), qlb_tick_reset_kernel, (unsigned long long)c->B,
                       reset_mask, c->limb, c->efforts, c->refill));
  QLB_CUDA(c->ctx, cudaEventRecord(c->reset_done, static_cast<cudaStream_t>(stream)));
  return QLB_OK;
}

int qlb_controller_update(qlb_controller* c, const double* q, const double* qd, const double* base_pose,
                          const double* base_twist, const double* target_pose, const double* target_twist,
                          const uint8_t* desired_stance_mask, const uint8_t* footstep_mask, const uint8_t* contact_mask,
                          const double* phase, const double* mu, const double* normals_world,
                          const double* foot_target_position, const double* foot_target_velocity, double* command,
                          uint32_t* flags, double* grf, void* stream) {
  return controller_update_t<double>(c, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                     footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                     foot_target_velocity, command, flags, grf, stream, false);
}
int qlb_controller_update_f32(qlb_controller* c, const float* q, const float* qd, const float* base_pose,
                              const float* base_twist, const float* target_pose, const float* target_twist,
                              const uint8_t* desired_stance_mask, const uint8_t* footstep_mask, const uint8_t* contact_mask,
                              const float* phase, const float* mu, const float* normals_world,
                              const float* foot_target_position, const float* foot_target_velocity, float* command,
                              uint32_t* flags, float* grf, void* stream) {
  return controller_update_t<float>(c, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                    footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                    foot_target_velocity, command, flags, grf, stream, false);
}
int qlb_controller_update_host(qlb_controller* c, const double* q, const double* qd, const double* base_pose,
                               const double* base_twist, const double* target_pose, const double* target_twist,
                               const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                               const uint8_t* contact_mask, const double* phase, const double* mu,
                               const double* normals_world, const double* foot_target_position,
                               const double* foot_target_velocity, double* command, uint32_t* flags, double* grf) {
  return controller_update_t<double>(c, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                     footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                     foot_target_velocity, command, flags, grf, nullptr, true);
}
int qlb_controller_update_f32_host(qlb_controller* c, const float* q, const float* qd, const float* base_pose,
                                   const float* base_twist, const float* target_pose, const float* target_twist,
                                   const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                                   const uint8_t* contact_mask, const float* phase, const float* mu,
                                   const float* normals_world, const float* foot_target_position,
                                   const float* foot_target_velocity, float* command, uint32_t* flags, float* grf) {
  return controller_update_t<float>(c, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                    footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                    foot_target_velocity, command, flags, grf, nullptr, true);
}

int qlb_controller_get_state(const qlb_controller* c, uint8_t* limb_state, double* efforts, void* stream) {
  if (!c) return QLB_ERR_NOT_INITIALISED;
  QLB_GUARD(c->ctx);
  DeviceGuard guard(c->ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (limb_state) QLB_CUDA(c->ctx, cudaMemcpyAsync(limb_state, c->limb, 4 * c->B, cudaMemcpyDeviceToDevice, st));
  if (efforts) QLB_CUDA(c->ctx, cudaMemcpyAsync(efforts, c->efforts, 12 * c->B * sizeof(double), cudaMemcpyDeviceToDevice, st));
  return QLB_OK;
}

}  // extern "C"
