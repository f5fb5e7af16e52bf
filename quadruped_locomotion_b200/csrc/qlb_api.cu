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

struct qlb_context {
  int device = 0;
  int sm_count = 0;
  int blocks_per_sm_quad[2] = {0, 0};
  int blocks_per_sm_first[2] = {0, 0};
  qlb_params params;
  qlb_leg_model legs[QLB_NUM_LEGS];
  DeviceModel* d_model = nullptr;
  DeviceParams* d_params = nullptr;
  DeviceLimbDynamics* d_limb = nullptr;        // qlb_set_limb_dynamics
  DeviceLimbDynamicsT<float>* d_limb_f = nullptr;   // its FP32 copy (swing legs of qlb_controller_update_f32)
  bool have_limb = false;
  DeviceModelT<float>* d_model_f = nullptr;    // FP32 copies for the _f32 entry points
  DeviceParamsT<float>* d_params_f = nullptr;
  int blocks_per_sm_quad_f[2] = {0, 0};
  int blocks_per_sm_first_f[2] = {0, 0};
  int blocks_per_sm_quad_m[2] = {0, 0};   // FP32 interface + FP64 solver core
  int blocks_per_sm_first_m[2] = {0, 0};
  int pipeline = QLB_PIPELINE_FUSED;   // qlb_set_pipeline
  int blocks_per_sm_single[2][2][2] = {};   // [interface type: 0 double, 1 float][MODE][TMA]
  std::recursive_mutex mu;                  // calls on one context from several host threads are serialised (QLB_GUARD)
  int fused_bps_cap = 0;                    // experiments (env QLB_FUSED_BPS): fewer CTAs of the fused kernel per SM
  bool use_tma = true;    // fused pipeline: stage the inputs with the TMA unit when the arrays allow it
  bool f32_pure = false;  // qlb_set_f32_core: FP32 solver core with in-kernel FP64 rescue, or FP64 core for every state
  unsigned long long* d_counter = nullptr;
  unsigned* d_list[8] = {};   // second-pass index lists, one per launch slot
  size_t list_cap[8] = {};
  uint64_t solve_calls = 0;   // picks the launch slot (counters + list): concurrent launches never share one
  cudaEvent_t slot_done[8] = {};  // recorded after the last pass of the call that used the slot; the next user waits on it
  int last_slot = 0;
  double* d_stats = nullptr;
  cudaStream_t stream = nullptr;  // used by the *_host entry points
  cudaStream_t pipe[kPipe] = {};  // chunk pipeline of the *_host entry points
  // device staging for the *_host entry points
  double* d_in = nullptr;
  double* d_out = nullptr;
  uint8_t* d_mask = nullptr;
  uint32_t* d_flags = nullptr;
  unsigned char* d_prev = nullptr;  // staging of qlb_preview_plan_host
  size_t prev_cap = 0;
  unsigned char* d_qp = nullptr;    // staging of qlb_qp_dense_host
  size_t qp_bytes = 0;
  unsigned char* d_rec = nullptr;   // record staging of qlb_solve_records_host: kPipe x cap x (216 + 248) bytes
  size_t rec_cap = 0;
  size_t cap = 0;
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
  if (ctx->list_cap[slot] < a.B) {  // grow the index lists of all slots at once (rare; synchronises)
    QLB_CUDA(ctx, cudaDeviceSynchronize());
    size_t cap = 1024;
    while (cap < a.B) cap *= 2;
    for (int i = 0; i < 8; i++) {
      if (ctx->list_cap[i] >= cap) continue;
      cudaFree(ctx->d_list[i]);
      ctx->d_list[i] = nullptr;
      ctx->list_cap[i] = 0;
      if (cudaMalloc(&ctx->d_list[i], 3 * cap * sizeof(unsigned)) != cudaSuccess) { cudaGetLastError(); return QLB_ERR_ALLOC; }
      ctx->list_cap[i] = cap;
    }
  }
  a.list = ctx->d_list[slot];
  a.list2 = ctx->d_list[slot] + ctx->list_cap[slot];
  a.list_pat = ctx->d_list[slot] + 2 * ctx->list_cap[slot];
  return QLB_OK;
}

// The three passes of the leg-per-lane kernels.  pass 1: everything up to the unconstrained minimiser;
// pass 2: active-set rounds on what is left; pass 3: interior point on what is still left.  The later
// grids are sized for the worst case and read the list lengths on the device (no host synchronisation
// between the passes).
template <typename T, typename C, int MODE>
int launch_quad(qlb_context* ctx, SolveArgsT<T>& a, cudaStream_t st, const int bps_first, const int bps_quad) {
  const unsigned long long nb8 = (a.B + 7) / 8;
  const unsigned long long wantq = (nb8 + (kQuadThreads / 32) - 1) / (kQuadThreads / 32);
  const unsigned long long capq = (unsigned long long)ctx->sm_count * bps_quad;
  const unsigned long long capf = (unsigned long long)ctx->sm_count * bps_first;
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
int launch_single(qlb_context* ctx, SolveArgsT<T>& a, cudaStream_t st, const int bps_ipm) {
  using SG = Staging<T, MODE, QLB_SUPER>;
  using FL = FusedLayout<T, C, MODE, QLB_SUPER>;
  const T* src[SG::kNumSeg];
  for (int s = 0; s < SG::kNumSeg; s++) src[s] = SG::source(a, s);
  bool tma = ctx->use_tma && a.B >= 64 && a.B < 0x7fffff00ull && ((a.B * sizeof(T)) % 16 == 0);
  for (int s = 0; s < SG::kNumSeg && tma; s++)
    if (src[s] && !aligned16(src[s])) tma = false;
  FusedMaps maps;
  std::memset(&maps, 0, sizeof maps);
  for (int s = 0; s < SG::kNumSeg && tma; s++)
    if (src[s] && !make_map<T>(&maps.seg[s], src[s], a.B, SG::rows(s))) tma = false;
  if (tma && (SG::kCols < 16 || !aligned16(a.mask) || !make_mask_map(&maps.mask, a.mask, a.B, SG::kCols))) tma = false;
  const unsigned long long ntiles = (a.B + 7) / 8;
  const unsigned long long want = (ntiles + kFusedWarps - 1) / kFusedWarps;
  int bps = ctx->blocks_per_sm_single[sizeof(T) == 4 ? 1 : 0][MODE][tma ? 1 : 0];
  if (ctx->fused_bps_cap > 0 && bps > ctx->fused_bps_cap) bps = ctx->fused_bps_cap;
  const unsigned long long cap = (unsigned long long)ctx->sm_count * bps;
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  if (tma) qlb_single_kernel<T, C, MODE, QLB_SUPER, true><<<grid, kFusedThreads, FL::kTotal, st>>>(a, maps);
  else qlb_single_kernel<T, C, MODE, QLB_SUPER, false><<<grid, kFusedThreads, FL::kTotal, st>>>(a, maps);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  const unsigned long long capq = (unsigned long long)ctx->sm_count * bps_ipm;
  const unsigned long long wantq = (ntiles + 3) / 4;
  qlb_quad_kernel<T, C, MODE, 2><<<(unsigned)(wantq < capq ? wantq : capq), kQuadThreads, 0, st>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  QLB_CUDA(ctx, cudaEventRecord(ctx->slot_done[ctx->last_slot], st));
  return QLB_OK;
}

template <typename T, typename C, int MODE>
bool prepare_single_kernels(qlb_context* ctx) {
  using FL = FusedLayout<T, C, MODE, QLB_SUPER>;
  int* out = ctx->blocks_per_sm_single[sizeof(T) == 4 ? 1 : 0][MODE];
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

template <int MODE>
int launch_solve(qlb_context* ctx, SolveArgs& a, cudaStream_t st) {
  const int rc = prepare_slot(ctx, a, st);
  if (rc != QLB_OK) return rc;
  if (ctx->pipeline == QLB_PIPELINE_FUSED) return launch_single<double, double, MODE>(ctx, a, st, ctx->blocks_per_sm_quad[MODE]);
  return launch_quad<double, double, MODE>(ctx, a, st, ctx->blocks_per_sm_first[MODE], ctx->blocks_per_sm_quad[MODE]);
}

// FP32 twins: FP32 interface with the FP64 or the FP32 solver core (qlb_set_f32_core)
template <int MODE>
int launch_solve_f32(qlb_context* ctx, SolveArgsT<float>& a, cudaStream_t st) {
  const int rc = prepare_slot(ctx, a, st);
  if (rc != QLB_OK) return rc;
  if (ctx->f32_pure) return launch_quad<float, float, MODE>(ctx, a, st, ctx->blocks_per_sm_first_f[MODE], ctx->blocks_per_sm_quad_f[MODE]);
  if (ctx->pipeline == QLB_PIPELINE_FUSED) return launch_single<float, double, MODE>(ctx, a, st, ctx->blocks_per_sm_quad_m[MODE]);
  return launch_quad<float, double, MODE>(ctx, a, st, ctx->blocks_per_sm_first_m[MODE], ctx->blocks_per_sm_quad_m[MODE]);
}

// staging of the host entry points: kPipe slots of `cap` states each (cap <= kChunk)
int ensure_capacity(qlb_context* ctx, size_t B) {
  if (B > kChunk) B = kChunk;
  if (B <= ctx->cap) return QLB_OK;
  size_t cap = ctx->cap ? ctx->cap : 1024;
  while (cap < B) cap *= 2;
  cap = (cap + 15) & ~size_t(15);
  cudaFree(ctx->d_in); cudaFree(ctx->d_out); cudaFree(ctx->d_mask); cudaFree(ctx->d_flags);
  ctx->d_in = ctx->d_out = nullptr; ctx->d_mask = nullptr; ctx->d_flags = nullptr; ctx->cap = 0;
  if (cudaMalloc(&ctx->d_in, kPipe * cap * kHostInRows * sizeof(double)) != cudaSuccess ||
      cudaMalloc(&ctx->d_out, kPipe * cap * kHostOutRows * sizeof(double)) != cudaSuccess ||
      cudaMalloc(&ctx->d_mask, kPipe * cap) != cudaSuccess || cudaMalloc(&ctx->d_flags, kPipe * cap * sizeof(uint32_t)) != cudaSuccess) {
    cudaGetLastError();
    return QLB_ERR_ALLOC;
  }
  ctx->cap = cap;
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
}  // namespace

int qlb_params_set_key(qlb_params* p, const char* key, double value) {
  if (!p || !key) return QLB_ERR_INVALID_ARGUMENT;
  for (int k = 0; k < kNumParamKeys; k++) {
    if (std::strcmp(key, kParamKeys[k].path) != 0) continue;
    const int i = kParamKeys[k].index;
    switch (kParamKeys[k].group) {
      case 0: p->wrench_weights[i] = value; break;
      case 1: p->ground_force_weight = value; break;
      case 2: p->friction_default = value; break;
      case 3: p->min_normal_force = value; break;
      case 4: p->kp_translation[i] = value; break;
      case 5: p->kd_translation[i] = value; break;
      case 6: p->kff_translation[i] = value; break;
      case 7: p->kp_rotation[i] = value; break;
      case 8: p->kd_rotation[i] = value; break;
      default: p->kff_rotation[i] = value; break;
    }
    return k;   // index of the key (>= 0)
  }
  return QLB_ERR_INVALID_ARGUMENT;
}

int qlb_params_get_key(const qlb_params* p, const char* key, double* value) {
  if (!p || !key || !value) return QLB_ERR_INVALID_ARGUMENT;
  for (int k = 0; k < kNumParamKeys; k++) {
    if (std::strcmp(key, kParamKeys[k].path) != 0) continue;
    const int i = kParamKeys[k].index;
    switch (kParamKeys[k].group) {
      case 0: *value = p->wrench_weights[i]; break;
      case 1: *value = p->ground_force_weight; break;
      case 2: *value = p->friction_default; break;
      case 3: *value = p->min_normal_force; break;
      case 4: *value = p->kp_translation[i]; break;
      case 5: *value = p->kd_translation[i]; break;
      case 6: *value = p->kff_translation[i]; break;
      case 7: *value = p->kp_rotation[i]; break;
      case 8: *value = p->kd_rotation[i]; break;
      default: *value = p->kff_rotation[i]; break;
    }
    return k;
  }
  return QLB_ERR_INVALID_ARGUMENT;
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
  DeviceModel hm;
  build_device_model(legs, &hm);
  if (cudaMemcpy(ctx->d_model, &hm, sizeof hm, cudaMemcpyHostToDevice) != cudaSuccess) return fail(QLB_ERR_CUDA);
  DeviceModelT<float> hmf;
  narrow_model(hm, &hmf);
  if (cudaMemcpy(ctx->d_model_f, &hmf, sizeof hmf, cudaMemcpyHostToDevice) != cudaSuccess) return fail(QLB_ERR_CUDA);
  if (qlb_set_params(ctx, p) != QLB_OK) return fail(QLB_ERR_CUDA);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_quad[0], qlb_quad_kernel<double, double, 0, 2>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_quad[1], qlb_quad_kernel<double, double, 1, 2>, kQuadThreads, 0) != cudaSuccess)
    return fail(QLB_ERR_CUDA);
  if (ctx->blocks_per_sm_quad[0] < 1 || ctx->blocks_per_sm_quad[1] < 1) return fail(QLB_ERR_CUDA);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_first[0], qlb_quad_first_kernel<double, double, 0>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_first[1], qlb_quad_first_kernel<double, double, 1>, kQuadThreads, 0) != cudaSuccess)
    return fail(QLB_ERR_CUDA);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_quad_f[0], qlb_quad_kernel<float, float, 0, 2>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_quad_f[1], qlb_quad_kernel<float, float, 1, 2>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_first_f[0], qlb_quad_first_kernel<float, float, 0>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_first_f[1], qlb_quad_first_kernel<float, float, 1>, kQuadThreads, 0) != cudaSuccess)
    return fail(QLB_ERR_CUDA);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_quad_m[0], qlb_quad_kernel<float, double, 0, 2>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_quad_m[1], qlb_quad_kernel<float, double, 1, 2>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_first_m[0], qlb_quad_first_kernel<float, double, 0>, kQuadThreads, 0) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->blocks_per_sm_first_m[1], qlb_quad_first_kernel<float, double, 1>, kQuadThreads, 0) != cudaSuccess)
    return fail(QLB_ERR_CUDA);
  if (!prepare_single_kernels<double, double, 0>(ctx) || !prepare_single_kernels<double, double, 1>(ctx) ||
      !prepare_single_kernels<float, double, 0>(ctx) || !prepare_single_kernels<float, double, 1>(ctx)) {
    cudaGetLastError();
    return fail(QLB_ERR_CUDA);
  }
  if (const char* e = std::getenv("QLB_FUSED_BPS")) ctx->fused_bps_cap = std::atoi(e);
  if (const char* e = std::getenv("QLB_PIPELINE")) {   // experiments: three_pass | fused | fused_notma
    if (!std::strcmp(e, "three_pass")) ctx->pipeline = QLB_PIPELINE_THREE_PASS;

    if (!std::strcmp(e, "fused_notma")) ctx->use_tma = false;
  }
  if (max_batch > 0 && ensure_capacity(ctx, max_batch) != QLB_OK) return fail(QLB_ERR_ALLOC);
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
  cudaFree(ctx->d_in); cudaFree(ctx->d_out); cudaFree(ctx->d_mask); cudaFree(ctx->d_flags); cudaFree(ctx->d_rec); cudaFree(ctx->d_qp); cudaFree(ctx->d_prev);
  for (int i = 0; i < 8; i++) cudaFree(ctx->d_list[i]);
  for (int i = 0; i < 8; i++)
    if (ctx->slot_done[i]) cudaEventDestroy(ctx->slot_done[i]);
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

// ---- device-pointer entry points (T = double, and float for the _f32 twins)
extern "C++" {
namespace {

template <typename T> struct Typed;
template <> struct Typed<double> {
  static const DeviceModel* model(const qlb_context* c) { return c->d_model; }
  static const DeviceLimbDynamics* limb(const qlb_context* c) { return c->d_limb; }
  static const DeviceParams* params(const qlb_context* c) { return c->d_params; }
  template <int MODE> static int launch(qlb_context* c, SolveArgs& a, cudaStream_t st) { return launch_solve<MODE>(c, a, st); }
};
template <> struct Typed<float> {
  static const DeviceModelT<float>* model(const qlb_context* c) { return c->d_model_f; }
  static const DeviceLimbDynamicsT<float>* limb(const qlb_context* c) { return c->d_limb_f; }
  static const DeviceParamsT<float>* params(const qlb_context* c) { return c->d_params_f; }
  template <int MODE> static int launch(qlb_context* c, SolveArgsT<float>& a, cudaStream_t st) { return launch_solve_f32<MODE>(c, a, st); }
};

template <typename T>
int solve_wrench_t(qlb_context* ctx, size_t B, const T* q, const T* quat_wxyz, const T* wrench, const uint8_t* stance_mask,
                   const T* mu, const T* normals_world, T* grf, T* tau, uint32_t* flags, T* netwrench, void* stream) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !quat_wxyz || !wrench || !stance_mask || !grf || !tau || !flags) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  SolveArgsT<T> a;
  std::memset(&a, 0, sizeof a);
  a.B = B; a.q = q; a.quat = quat_wxyz; a.wrench = wrench; a.mask = stance_mask; a.mu = mu; a.normals = normals_world;
  a.grf = grf; a.tau = tau; a.flags = flags; a.netwrench = netwrench;
  a.counter = ctx->d_counter; a.model = Typed<T>::model(ctx); a.params = Typed<T>::params(ctx); a.params64 = ctx->d_params;
  return Typed<T>::template launch<0>(ctx, a, static_cast<cudaStream_t>(stream));
}

template <typename T>
int solve_state_t(qlb_context* ctx, size_t B, const T* q, const T* base_pose, const T* base_twist, const T* target_pose,
                  const T* target_twist, const uint8_t* stance_mask, const T* mu, const T* normals_world, T* grf, T* tau,
                  uint32_t* flags, T* netwrench, T* wrench_out, void* stream) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !base_pose || !base_twist || !target_pose || !target_twist || !stance_mask || !grf || !tau || !flags)
    return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  SolveArgsT<T> a;
  std::memset(&a, 0, sizeof a);
  a.B = B; a.q = q; a.pose = base_pose; a.twist = base_twist; a.tpose = target_pose; a.ttwist = target_twist;
  a.mask = stance_mask; a.mu = mu; a.normals = normals_world;
  a.grf = grf; a.tau = tau; a.flags = flags; a.netwrench = netwrench; a.wrench_out = wrench_out;
  a.counter = ctx->d_counter; a.model = Typed<T>::model(ctx); a.params = Typed<T>::params(ctx); a.params64 = ctx->d_params;
  return Typed<T>::template launch<1>(ctx, a, static_cast<cudaStream_t>(stream));
}

// ---- host-pointer entry points: copy in, solve, copy out, synchronise.
// Large batches are cut into chunks of kChunk states that flow through kPipe streams, so that the H2D
// copy of chunk i+1, the kernel of chunk i and the D2H copy of chunk i-1 overlap (PCIe is full duplex).
// The arrays are SoA with row pitch B, so a chunk is a column range: one 2-D copy per array.
template <typename T> struct HostRow { const T* h; int rows; };   // input array (may be null) and its component count
template <typename T> struct HostOut { T* h; int rows; };

template <typename T>
int host_pipeline_chunks(qlb_context* ctx, size_t B, bool state_mode, const HostRow<T>* in, int nin, const uint8_t* mask,
                      const HostOut<T>* out, int nout, uint32_t* flags) {
  int rc = QLB_OK;
  const size_t cap = ctx->cap;
  const size_t nchunks = (B + cap - 1) / cap;
  for (size_t ci = 0; ci < nchunks; ci++) {
    const int slot = (int)(ci % kPipe);
    cudaStream_t st = ctx->pipe[slot];
    const size_t b0 = ci * cap, n = (B - b0 < cap) ? (B - b0) : cap;
    // the staging buffers are sized for FP64; the FP32 twins use the first half of each slot
    T* din = reinterpret_cast<T*>(ctx->d_in + (size_t)slot * cap * kHostInRows);
    T* dout = reinterpret_cast<T*>(ctx->d_out + (size_t)slot * cap * kHostOutRows);
    uint8_t* dmask = ctx->d_mask + (size_t)slot * cap;
    uint32_t* dflags = ctx->d_flags + (size_t)slot * cap;
    const T* dptr_in[8];
    size_t off = 0;
    for (int k = 0; k < nin; k++) {
      dptr_in[k] = nullptr;
      if (in[k].h) {
        dptr_in[k] = din + off;
        QLB_CUDA(ctx, cudaMemcpy2DAsync(din + off, n * sizeof(T), in[k].h + b0, B * sizeof(T), n * sizeof(T), in[k].rows,
                                        cudaMemcpyHostToDevice, st));
      }
      off += (size_t)in[k].rows * cap;   // fixed block sizes keep every block 16-byte aligned (cap % 16 == 0)
    }
    QLB_CUDA(ctx, cudaMemcpyAsync(dmask, mask + b0, n, cudaMemcpyHostToDevice, st));
    T* dptr_out[4];
    off = 0;
    for (int k = 0; k < nout; k++) {
      dptr_out[k] = out[k].h ? dout + off : nullptr;
      off += (size_t)out[k].rows * cap;
    }
    if (!state_mode)
      rc = solve_wrench_t<T>(ctx, n, dptr_in[0], dptr_in[1], dptr_in[2], dmask, dptr_in[3], dptr_in[4], dptr_out[0], dptr_out[1],
                             dflags, dptr_out[2], st);
    else
      rc = solve_state_t<T>(ctx, n, dptr_in[0], dptr_in[1], dptr_in[2], dptr_in[3], dptr_in[4], dmask, dptr_in[5], dptr_in[6],
                            dptr_out[0], dptr_out[1], dflags, dptr_out[2], dptr_out[3], st);
    if (rc != QLB_OK) return rc;
    for (int k = 0; k < nout; k++)
      if (out[k].h)
        QLB_CUDA(ctx, cudaMemcpy2DAsync(out[k].h + b0, B * sizeof(T), dptr_out[k], n * sizeof(T), n * sizeof(T), out[k].rows,
                                        cudaMemcpyDeviceToHost, st));
    QLB_CUDA(ctx, cudaMemcpyAsync(flags + b0, dflags, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  }
  return QLB_OK;
}


template <typename T>
int run_host_pipeline(qlb_context* ctx, size_t B, bool state_mode, const HostRow<T>* in, int nin, const uint8_t* mask,
                      const HostOut<T>* out, int nout, uint32_t* flags) {
  int rc = ensure_capacity(ctx, B);
  if (rc != QLB_OK) return rc;
  rc = host_pipeline_chunks<T>(ctx, B, state_mode, in, nin, mask, out, nout, flags);
  // also on failure: no copy may still be reading or writing the caller's buffers when the call returns
  for (int i = 0; i < kPipe; i++)
    if (cudaStreamSynchronize(ctx->pipe[i]) != cudaSuccess && rc == QLB_OK) rc = cuda_fail(ctx, cudaGetLastError(), "cudaStreamSynchronize");
  return rc;
}

template <typename T>
int solve_wrench_host_t(qlb_context* ctx, size_t B, const T* q, const T* quat_wxyz, const T* wrench, const uint8_t* stance_mask,
                        const T* mu, const T* normals_world, T* grf, T* tau, uint32_t* flags, T* netwrench) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !quat_wxyz || !wrench || !stance_mask || !grf || !tau || !flags) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  const HostRow<T> in[5] = {{q, 12}, {quat_wxyz, 4}, {wrench, 6}, {mu, 4}, {normals_world, 12}};
  const HostOut<T> out[3] = {{grf, 12}, {tau, 12}, {netwrench, 6}};
  return run_host_pipeline<T>(ctx, B, false, in, 5, stance_mask, out, 3, flags);
}

template <typename T>
int solve_state_host_t(qlb_context* ctx, size_t B, const T* q, const T* base_pose, const T* base_twist, const T* target_pose,
                       const T* target_twist, const uint8_t* stance_mask, const T* mu, const T* normals_world, T* grf, T* tau,
                       uint32_t* flags, T* netwrench, T* wrench_out) {
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !base_pose || !base_twist || !target_pose || !target_twist || !stance_mask || !grf || !tau || !flags)
    return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  const HostRow<T> in[7] = {{q, 12}, {base_pose, 7}, {base_twist, 6}, {target_pose, 7}, {target_twist, 6}, {mu, 4}, {normals_world, 12}};
  const HostOut<T> out[4] = {{grf, 12}, {tau, 12}, {netwrench, 6}, {wrench_out, 6}};
  return run_host_pipeline<T>(ctx, B, true, in, 7, stance_mask, out, 4, flags);
}

}  // namespace
}  // extern "C++"

int qlb_solve_wrench(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz, const double* wrench,
                     const uint8_t* stance_mask, const double* mu, const double* normals_world, double* grf,
                     double* tau, uint32_t* flags, double* netwrench, void* stream) {
  QLB_GUARD(ctx);
  return solve_wrench_t<double>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench, stream);
}
int qlb_solve_wrench_f32(qlb_context* ctx, size_t B, const float* q, const float* quat_wxyz, const float* wrench,
                         const uint8_t* stance_mask, const float* mu, const float* normals_world, float* grf, float* tau,
                         uint32_t* flags, float* netwrench, void* stream) {
  QLB_GUARD(ctx);
  return solve_wrench_t<float>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench, stream);
}
int qlb_solve_state(qlb_context* ctx, size_t B, const double* q, const double* base_pose, const double* base_twist,
                    const double* target_pose, const double* target_twist, const uint8_t* stance_mask,
                    const double* mu, const double* normals_world, double* grf, double* tau, uint32_t* flags,
                    double* netwrench, double* wrench_out, void* stream) {
  QLB_GUARD(ctx);
  return solve_state_t<double>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world, grf,
                               tau, flags, netwrench, wrench_out, stream);
}
int qlb_solve_state_f32(qlb_context* ctx, size_t B, const float* q, const float* base_pose, const float* base_twist,
                        const float* target_pose, const float* target_twist, const uint8_t* stance_mask, const float* mu,
                        const float* normals_world, float* grf, float* tau, uint32_t* flags, float* netwrench,
                        float* wrench_out, void* stream) {
  QLB_GUARD(ctx);
  return solve_state_t<float>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world, grf,
                              tau, flags, netwrench, wrench_out, stream);
}
int qlb_solve_wrench_host(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz, const double* wrench,
                          const uint8_t* stance_mask, const double* mu, const double* normals_world, double* grf,
                          double* tau, uint32_t* flags, double* netwrench) {
  QLB_GUARD(ctx);
  return solve_wrench_host_t<double>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench);
}
int qlb_solve_wrench_f32_host(qlb_context* ctx, size_t B, const float* q, const float* quat_wxyz, const float* wrench,
                              const uint8_t* stance_mask, const float* mu, const float* normals_world, float* grf, float* tau,
                              uint32_t* flags, float* netwrench) {
  QLB_GUARD(ctx);
  return solve_wrench_host_t<float>(ctx, B, q, quat_wxyz, wrench, stance_mask, mu, normals_world, grf, tau, flags, netwrench);
}
int qlb_solve_state_host(qlb_context* ctx, size_t B, const double* q, const double* base_pose, const double* base_twist,
                         const double* target_pose, const double* target_twist, const uint8_t* stance_mask,
                         const double* mu, const double* normals_world, double* grf, double* tau, uint32_t* flags,
                         double* netwrench, double* wrench_out) {
  QLB_GUARD(ctx);
  return solve_state_host_t<double>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world,
                                    grf, tau, flags, netwrench, wrench_out);
}
int qlb_solve_state_f32_host(qlb_context* ctx, size_t B, const float* q, const float* base_pose, const float* base_twist,
                             const float* target_pose, const float* target_twist, const uint8_t* stance_mask, const float* mu,
                             const float* normals_world, float* grf, float* tau, uint32_t* flags, float* netwrench,
                             float* wrench_out) {
  QLB_GUARD(ctx);
  return solve_state_host_t<float>(ctx, B, q, base_pose, base_twist, target_pose, target_twist, stance_mask, mu, normals_world,
                                   grf, tau, flags, netwrench, wrench_out);
}

int qlb_leg_kinematics(qlb_context* ctx, size_t B, const double* q, const double* quat_wxyz, double* foot, double* jac,
                       double* gravity_tau, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  const unsigned long long total = (unsigned long long)B * 4ull;
  const unsigned threads = 128;
  const unsigned long long blocks = (total + threads - 1) / threads;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_kinematics_kernel<<<(unsigned)blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(
      B, q, quat_wxyz, foot, jac, gravity_tau, ctx->d_model, ctx->d_params);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

int qlb_pack_robot_states(qlb_context* ctx, size_t B, const qlb_robot_state_record* records, double* q, double* base_pose,
                          double* base_twist, uint8_t* stance_mask, double* normals_world, void* stream) {
  QLB_GUARD(ctx);
  static_assert(sizeof(qlb_robot_state_record) == 304, "record layout is part of the ABI");
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!records || !aligned16(records)) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  const unsigned long long blocks = ((unsigned long long)B + kPackTile - 1) / kPackTile;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_pack_kernel<<<(unsigned)blocks, kPackTile, 0, static_cast<cudaStream_t>(stream)>>>(B, records, q, base_pose, base_twist,
                                                                                       stance_mask, normals_world);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

int qlb_feet_in_world(qlb_context* ctx, size_t B, const double* q, const double* base_pose, double* feet_world, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !base_pose || !feet_world) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  const unsigned long long total = (unsigned long long)B * 4ull;
  const unsigned threads = 128;
  const unsigned long long blocks = (total + threads - 1) / threads;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_kinematics_kernel<<<(unsigned)blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(
      B, q, nullptr, nullptr, nullptr, nullptr, ctx->d_model, ctx->d_params, base_pose, feet_world);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
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

int qlb_swing_leg_torques(qlb_context* ctx, size_t B, const double* q, const double* qd, const double* qdd,
                          const double* foot_target_position, const double* foot_target_velocity,
                          const qlb_swing_params* params, double* tau, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (!ctx->have_limb) return QLB_ERR_NOT_INITIALISED;   // qlb_set_limb_dynamics first
  if (B == 0) return QLB_OK;
  if (!q || !qd || !qdd || !params || !tau) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  SwingArgs a;
  std::memset(&a, 0, sizeof a);
  a.B = B; a.q = q; a.qd = qd; a.qdd = qdd; a.ptarget = foot_target_position; a.vtarget = foot_target_velocity; a.tau = tau;
  for (int c = 0; c < 3; c++) { a.gravity[c] = params->gravity[c]; a.kp[c] = params->kp[c]; a.kd[c] = params->kd[c]; }
  a.acc_scale = params->acceleration_scale;
  a.dyn = ctx->d_limb; a.model = ctx->d_model;
  const unsigned long long total = (unsigned long long)B * 4ull;
  const unsigned long long blocks = (total + 127) / 128;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_swing_kernel<<<(unsigned)blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
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
  std::memset(&a, 0, sizeof a);
  a.B = B; a.q = q; a.qd = qd_back; a.qdd = nullptr; a.qd_front = qd_front; a.ld_front = B; a.inv_window = 1.0 / (10.0 * period);
  a.ptarget = foot_target_position; a.vtarget = foot_target_velocity; a.tau = tau;
  for (int c = 0; c < 3; c++) { a.gravity[c] = params->gravity[c]; a.kp[c] = params->kp[c]; a.kd[c] = params->kd[c]; }
  a.acc_scale = params->acceleration_scale;
  a.dyn = ctx->d_limb; a.model = ctx->d_model;
  const unsigned long long total = (unsigned long long)B * 4ull;
  const unsigned long long blocks = (total + 127) / 128;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_swing_kernel<<<(unsigned)blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

int qlb_contact_fsm(qlb_context* ctx, size_t B, const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                    const uint8_t* contact_mask, const double* phase, uint8_t* limb_state, uint8_t* stance_mask, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!desired_stance_mask || !contact_mask || !phase || !limb_state) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  const unsigned long long blocks = ((unsigned long long)B + 255) / 256;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_contact_fsm_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(B, desired_stance_mask, footstep_mask,
                                                                                         contact_mask, phase, limb_state, stance_mask);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

int qlb_friction_margins(qlb_context* ctx, size_t B, const double* grf, const double* quat_wxyz, const uint8_t* stance_mask,
                         const double* mu, const double* normals_world, double* margin, double* min_normal, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!grf || !quat_wxyz || !stance_mask || !margin) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  const unsigned long long blocks = ((unsigned long long)B + 255) / 256;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_friction_margin_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(B, grf, quat_wxyz, stance_mask, mu,
                                                                                             normals_world, ctx->d_params, margin, min_normal);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

// HOST pointers: staged through the context's pipeline buffers in chunks, on the context stream; synchronises.
int qlb_swing_leg_torques_host(qlb_context* ctx, size_t B, const double* q, const double* qd, const double* qdd,
                               const double* foot_target_position, const double* foot_target_velocity,
                               const qlb_swing_params* params, double* tau) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (!ctx->have_limb) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!q || !qd || !qdd || !params || !tau) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  int rc = ensure_capacity(ctx, B);
  if (rc != QLB_OK) return rc;
  const size_t cap = ctx->cap;   // the input staging area holds kPipe * cap * 54 doubles >= 5 * 12 * cap
  static_assert(kPipe * kHostInRows >= 60 && kPipe * kHostOutRows >= 12, "staging too small for the swing-leg arrays");
  const double* src[5] = {q, qd, qdd, foot_target_position, foot_target_velocity};
  for (size_t b0 = 0; b0 < B; b0 += cap) {
    const size_t n = (B - b0 < cap) ? (B - b0) : cap;
    const double* dptr[5];
    for (int k = 0; k < 5; k++) {
      dptr[k] = nullptr;
      if (!src[k]) continue;
      double* d = ctx->d_in + (size_t)k * 12 * cap;
      dptr[k] = d;
      QLB_CUDA(ctx, cudaMemcpy2DAsync(d, n * sizeof(double), src[k] + b0, B * sizeof(double), n * sizeof(double), 12,
                                      cudaMemcpyHostToDevice, ctx->stream));
    }
    rc = qlb_swing_leg_torques(ctx, n, dptr[0], dptr[1], dptr[2], dptr[3], dptr[4], params, ctx->d_out, ctx->stream);
    if (rc != QLB_OK) { cudaStreamSynchronize(ctx->stream); return rc; }
    QLB_CUDA(ctx, cudaMemcpy2DAsync(tau + b0, B * sizeof(double), ctx->d_out, n * sizeof(double), n * sizeof(double), 12,
                                    cudaMemcpyDeviceToHost, ctx->stream));
    QLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return QLB_OK;
}

namespace {
// one chunk of records on one stream: unpack, solve, pack (device pointers; `slot` selects the SoA staging area)
int records_chunk(qlb_context* ctx, size_t n, const qlb_wrench_record* d_in, qlb_result_record* d_out, int slot, cudaStream_t st) {
  const size_t cap = ctx->cap;
  double* din = ctx->d_in + (size_t)slot * cap * kHostInRows;
  double* dout = ctx->d_out + (size_t)slot * cap * kHostOutRows;
  uint8_t* dmask = ctx->d_mask + (size_t)slot * cap;
  uint32_t* dflags = ctx->d_flags + (size_t)slot * cap;
  double* q = din; double* quat = din + 12 * cap; double* wrench = din + 16 * cap; double* mu = din + 22 * cap;
  double* grf = dout; double* tau = dout + 12 * cap; double* net = dout + 24 * cap;
  const unsigned blocks = (unsigned)((n + kRecTile - 1) / kRecTile);
  // the SoA staging rows have pitch n inside this chunk
  qlb_unpack_records_kernel<<<blocks, kRecTile, 0, st>>>(n, d_in, q, quat, wrench, mu, dmask);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  const int rc = solve_wrench_t<double>(ctx, n, q, quat, wrench, dmask, mu, nullptr, grf, tau, dflags, net, st);
  if (rc != QLB_OK) return rc;
  qlb_pack_results_kernel<<<blocks, kRecTile, 0, st>>>(n, grf, tau, net, dflags, d_out);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

int records_host_chunks(qlb_context* ctx, size_t B, const qlb_wrench_record* in, qlb_result_record* out) {
  const size_t cap = ctx->cap;
  const size_t nchunks = (B + cap - 1) / cap;
  for (size_t ci = 0; ci < nchunks; ci++) {
    const int slot = (int)(ci % kPipe);
    cudaStream_t st = ctx->pipe[slot];
    const size_t b0 = ci * cap, n = (B - b0 < cap) ? (B - b0) : cap;
    unsigned char* base = ctx->d_rec + (size_t)slot * cap * (sizeof(qlb_wrench_record) + sizeof(qlb_result_record));
    qlb_wrench_record* d_in = reinterpret_cast<qlb_wrench_record*>(base);
    qlb_result_record* d_out = reinterpret_cast<qlb_result_record*>(base + cap * sizeof(qlb_wrench_record));
    QLB_CUDA(ctx, cudaMemcpyAsync(d_in, in + b0, n * sizeof(qlb_wrench_record), cudaMemcpyHostToDevice, st));
    const int rc = records_chunk(ctx, n, d_in, d_out, slot, st);
    if (rc != QLB_OK) return rc;
    QLB_CUDA(ctx, cudaMemcpyAsync(out + b0, d_out, n * sizeof(qlb_result_record), cudaMemcpyDeviceToHost, st));
  }
  return QLB_OK;
}
}  // namespace

int qlb_solve_records(qlb_context* ctx, size_t B, const qlb_wrench_record* records, qlb_result_record* results, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!records || !results) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  int rc = ensure_capacity(ctx, B);
  if (rc != QLB_OK) return rc;
  const size_t cap = ctx->cap;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // one staging area, chunks in stream order (the caller's arrays are already on the device: nothing to overlap)
  for (size_t b0 = 0; b0 < B; b0 += cap) {
    const size_t n = (B - b0 < cap) ? (B - b0) : cap;
    rc = records_chunk(ctx, n, records + b0, results + b0, 0, st);
    if (rc != QLB_OK) return rc;
  }
  return QLB_OK;
}

int qlb_solve_records_host(qlb_context* ctx, size_t B, const qlb_wrench_record* records, qlb_result_record* results) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!records || !results) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  int rc = ensure_capacity(ctx, B);
  if (rc != QLB_OK) return rc;
  if (ctx->rec_cap < ctx->cap) {
    QLB_CUDA(ctx, cudaDeviceSynchronize());
    cudaFree(ctx->d_rec);
    ctx->d_rec = nullptr; ctx->rec_cap = 0;
    if (cudaMalloc(&ctx->d_rec, (size_t)kPipe * ctx->cap * (sizeof(qlb_wrench_record) + sizeof(qlb_result_record))) != cudaSuccess) {
      cudaGetLastError();
      return QLB_ERR_ALLOC;
    }
    ctx->rec_cap = ctx->cap;
  }
  rc = records_host_chunks(ctx, B, records, results);
  for (int i = 0; i < kPipe; i++)
    if (cudaStreamSynchronize(ctx->pipe[i]) != cudaSuccess && rc == QLB_OK) rc = cuda_fail(ctx, cudaGetLastError(), "cudaStreamSynchronize");
  return rc;
}

int qlb_preview_plan_host(qlb_context* ctx, size_t B, const qlb_robot_state_record* records, const double mu[4],
                          qlb_preview_record* preview) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (B == 0) return QLB_OK;
  if (!records || !preview) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  int rc = ensure_capacity(ctx, B);
  if (rc != QLB_OK) return rc;
  const size_t cap = ctx->cap;
  // per state: the input record, the result record, and SoA rows for feet (12), friction coefficients (4), margins (2)
  const size_t per_state = sizeof(qlb_robot_state_record) + sizeof(qlb_preview_record) + 18 * sizeof(double);
  if (ctx->prev_cap < cap) {
    QLB_CUDA(ctx, cudaDeviceSynchronize());
    cudaFree(ctx->d_prev);
    ctx->d_prev = nullptr; ctx->prev_cap = 0;
    if (cudaMalloc(&ctx->d_prev, cap * per_state) != cudaSuccess) { cudaGetLastError(); return QLB_ERR_ALLOC; }
    ctx->prev_cap = cap;
  }
  cudaStream_t st = ctx->stream;
  qlb_robot_state_record* d_rec = reinterpret_cast<qlb_robot_state_record*>(ctx->d_prev);
  qlb_preview_record* d_res = reinterpret_cast<qlb_preview_record*>(ctx->d_prev + cap * sizeof(qlb_robot_state_record));
  double* extra = reinterpret_cast<double*>(ctx->d_prev + cap * (sizeof(qlb_robot_state_record) + sizeof(qlb_preview_record)));
  double* feet = extra; double* dmu = extra + 12 * cap; double* margin = extra + 16 * cap; double* minn = extra + 17 * cap;
  double* din = ctx->d_in; double* dout = ctx->d_out;
  double* q = din; double* pose = din + 12 * cap; double* twist = din + 19 * cap; double* nrm = din + 25 * cap;
  double* grf = dout; double* tau = dout + 12 * cap; double* net = dout + 24 * cap; double* wout = dout + 30 * cap;
  for (size_t b0 = 0; b0 < B && rc == QLB_OK; b0 += cap) {
    const size_t n = (B - b0 < cap) ? (B - b0) : cap;
    if (cudaMemcpyAsync(d_rec, records + b0, n * sizeof(qlb_robot_state_record), cudaMemcpyHostToDevice, st) != cudaSuccess) { rc = QLB_ERR_CUDA; break; }
    rc = qlb_pack_robot_states(ctx, n, d_rec, q, pose, twist, ctx->d_mask, nrm, st);
    if (rc == QLB_OK) rc = qlb_feet_in_world(ctx, n, q, pose, feet, st);
    if (rc == QLB_OK && mu) {
      qlb_fill_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, 4, dmu, mu[0], mu[1], mu[2], mu[3]);
      ctx->launches++;
    }
    // the planned state is feedback AND target: zero tracking error
    if (rc == QLB_OK) rc = solve_state_t<double>(ctx, n, q, pose, twist, pose, twist, ctx->d_mask, mu ? dmu : nullptr, nrm, grf, tau,
                                                  ctx->d_flags, net, wout, st);
    if (rc == QLB_OK) rc = qlb_friction_margins(ctx, n, grf, pose + 3 * n, ctx->d_mask, mu ? dmu : nullptr, nrm, margin, minn, st);
    if (rc == QLB_OK) {
      qlb_pack_preview_kernel<<<(unsigned)((n + kPrevTile - 1) / kPrevTile), kPrevTile, 0, st>>>(n, feet, grf, tau, net, wout, margin, minn,
                                                                                             ctx->d_flags, d_res);
      ctx->launches++;
      if (cudaGetLastError() != cudaSuccess) rc = QLB_ERR_CUDA;
    }
    if (rc == QLB_OK && cudaMemcpyAsync(preview + b0, d_res, n * sizeof(qlb_preview_record), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QLB_ERR_CUDA;
    // the staging is reused by the next chunk
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == QLB_OK) rc = QLB_ERR_CUDA;
  }
  if (rc == QLB_ERR_CUDA) cuda_fail(ctx, cudaGetLastError(), "qlb_preview_plan_host");
  return rc;
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
  const unsigned long long blocks = ((unsigned long long)B + 255) / 256;
  if (blocks > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  qlb_generate_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(g);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
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

int qlb_qp_dense(qlb_context* ctx, size_t B, int n, int m, int p, const double* G, const double* g0, const double* CE,
                 const double* ce0, const double* CI, const double* ci0, double* x, double* cost, uint32_t* status,
                 uint32_t* active, void* stream) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (n < 1 || n > kQpMaxN || m < 0 || m > kQpMaxM || p < 0 || p > kQpMaxP) return QLB_ERR_INVALID_ARGUMENT;
  if (B == 0) return QLB_OK;
  if (!G || !g0 || !x || !status || (p > 0 && (!CE || !ce0)) || (m > 0 && (!CI || !ci0))) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
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

int qlb_qp_dense_host(qlb_context* ctx, size_t B, int n, int m, int p, const double* G, const double* g0,
                      const double* CE, const double* ce0, const double* CI, const double* ci0, double* x, double* cost,
                      uint32_t* status, uint32_t* active) {
  QLB_GUARD(ctx);
  if (!ctx) return QLB_ERR_NOT_INITIALISED;
  if (n < 1 || n > kQpMaxN || m < 0 || m > kQpMaxM || p < 0 || p > kQpMaxP) return QLB_ERR_INVALID_ARGUMENT;
  if (B == 0) return QLB_OK;
  if (!G || !g0 || !x || !status || (p > 0 && (!CE || !ce0)) || (m > 0 && (!CI || !ci0))) return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(ctx->device);
  cudaStream_t st = ctx->stream;
  const size_t nin = (size_t)(n * n + n + n * p + p + n * m + m) * B, nout = (size_t)(n + 1) * B;
  // staging owned by the context, grown on demand (a controller calls this every tick with the same shape)
  const size_t need = (nin + nout) * sizeof(double) + 2 * B * sizeof(uint32_t);
  if (ctx->qp_bytes < need) {
    QLB_CUDA(ctx, cudaStreamSynchronize(st));
    cudaFree(ctx->d_qp);
    ctx->d_qp = nullptr; ctx->qp_bytes = 0;
    size_t cap = 4096;
    while (cap < need) cap *= 2;
    if (cudaMalloc(&ctx->d_qp, cap) != cudaSuccess) { cudaGetLastError(); return QLB_ERR_ALLOC; }
    ctx->qp_bytes = cap;
  }
  double* d_in = reinterpret_cast<double*>(ctx->d_qp);
  double* d_out = d_in + nin;
  uint32_t* d_u = reinterpret_cast<uint32_t*>(d_out + nout);
  double* dG = d_in; double* dg = dG + (size_t)n * n * B; double* dCE = dg + (size_t)n * B; double* dce = dCE + (size_t)n * p * B;
  double* dCI = dce + (size_t)p * B; double* dci = dCI + (size_t)n * m * B;
  int rc = QLB_OK;
  auto H2D = [&](double* d, const double* h, size_t cnt) {
    if (cnt && rc == QLB_OK && cudaMemcpyAsync(d, h, cnt * sizeof(double), cudaMemcpyHostToDevice, st) != cudaSuccess) rc = QLB_ERR_CUDA;
  };
  H2D(dG, G, (size_t)n * n * B); H2D(dg, g0, (size_t)n * B); H2D(dCE, CE, (size_t)n * p * B); H2D(dce, ce0, (size_t)p * B);
  H2D(dCI, CI, (size_t)n * m * B); H2D(dci, ci0, (size_t)m * B);
  if (rc == QLB_OK) rc = qlb_qp_dense(ctx, B, n, m, p, dG, dg, p ? dCE : nullptr, p ? dce : nullptr, m ? dCI : nullptr,
                                       m ? dci : nullptr, d_out, d_out + (size_t)n * B, d_u, d_u + B, st);
  if (rc == QLB_OK) {
    if (cudaMemcpyAsync(x, d_out, (size_t)n * B * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QLB_ERR_CUDA;
    if (cost && cudaMemcpyAsync(cost, d_out + (size_t)n * B, B * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QLB_ERR_CUDA;
    if (cudaMemcpyAsync(status, d_u, B * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QLB_ERR_CUDA;
    if (active && cudaMemcpyAsync(active, d_u + B, B * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = QLB_ERR_CUDA;
  }
  if (cudaStreamSynchronize(st) != cudaSuccess && rc == QLB_OK) rc = QLB_ERR_CUDA;
  if (rc == QLB_ERR_CUDA) cuda_fail(ctx, cudaGetLastError(), "qlb_qp_dense_host");
  return rc;
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
  const unsigned long long blocks_pro = ((unsigned long long)n + 255) / 256;
  const unsigned long long blocks_epi = (4ull * n + 127) / 128;
  if (blocks_epi > 0x7fffffffull) return QLB_ERR_BATCH_TOO_LARGE;
  const size_t ld = c->B;
  T* tau = reinterpret_cast<T*>(c->tau);
  TickArgsT<T> a;
  std::memset(&a, 0, sizeof a);
  a.n = n; a.ld = ld; a.head = c->head;
  a.desired = desired; a.footstep = footstep; a.contact = contact; a.phase = phase; a.qd = qd;
  a.limb = c->limb + b0; a.refill = c->refill + b0; a.ring = c->ring + b0; a.stance = c->stance;
  a.flags = flags; a.tau = tau; a.efforts = c->efforts + b0; a.command = command; a.limit = c->p.effort_limit;
  SwingArgsT<T>& s = a.swing;
  s.B = n; s.q = q; s.qd = qd;
  s.qd_front = c->ring + (size_t)((c->head + 1) % kTickRing) * 12 * ld + b0; s.ld_front = ld;
  s.inv_window = (T)(1.0 / (10.0 * c->p.period));
  s.ptarget = ptarget; s.vtarget = vtarget;
  for (int k = 0; k < 3; k++) { s.gravity[k] = (T)c->p.swing.gravity[k]; s.kp[k] = (T)c->p.swing.kp[k]; s.kd[k] = (T)c->p.swing.kd[k]; }
  s.acc_scale = (T)c->p.swing.acceleration_scale;
  s.dyn = Typed<T>::limb(ctx); s.model = Typed<T>::model(ctx);
  QLB_CUDA(ctx, cudaStreamWaitEvent(st, c->reset_done, 0));
  qlb_tick_prologue_kernel<T><<<(unsigned)blocks_pro, 256, 0, st>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  const int rc = solve_state_t<T>(ctx, n, q, pose, twist, tpose, ttwist, c->stance, mu, normals,
                                  grf ? grf : reinterpret_cast<T*>(c->grf), tau, flags, nullptr, nullptr, st);
  if (rc != QLB_OK) return rc;
  qlb_tick_epilogue_kernel<T><<<(unsigned)blocks_epi, 128, 0, st>>>(a);
  QLB_CUDA(ctx, cudaGetLastError());
  ctx->launches++;
  return QLB_OK;
}

bool controller_ready(const qlb_controller* c) { return c && c->ctx && c->ctx->have_limb; }

template <typename T>
int controller_update_t(qlb_controller* c, const T* q, const T* qd, const T* base_pose, const T* base_twist,
                        const T* target_pose, const T* target_twist, const uint8_t* desired_stance_mask,
                        const uint8_t* footstep_mask, const uint8_t* contact_mask, const T* phase, const T* mu,
                        const T* normals_world, const T* foot_target_position, const T* foot_target_velocity, T* command,
                        uint32_t* flags, T* grf, void* stream) {
  if (!c) return QLB_ERR_NOT_INITIALISED;
  QLB_GUARD(c->ctx);
  if (!controller_ready(c)) return QLB_ERR_NOT_INITIALISED;   // qlb_set_limb_dynamics first
  if (!q || !qd || !base_pose || !base_twist || !target_pose || !target_twist || !desired_stance_mask || !contact_mask ||
      !phase || !command || !flags)
    return QLB_ERR_INVALID_ARGUMENT;
  DeviceGuard guard(c->ctx->device);
  const int rc = controller_tick<T>(c, c->B, 0, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                    footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                    foot_target_velocity, command, flags, grf, static_cast<cudaStream_t>(stream));
  if (rc == QLB_OK) c->head = (c->head + 1) % kTickRing;
  return rc;
}

// HOST pointers: chunks of the context's staging capacity, one after the other on the context stream; synchronises.
// The staging buffers are sized for FP64; the FP32 twin uses the same row offsets in float, i.e. the first half.
template <typename T>
int controller_update_host_t(qlb_controller* c, const T* q, const T* qd, const T* base_pose, const T* base_twist,
                             const T* target_pose, const T* target_twist, const uint8_t* desired_stance_mask,
                             const uint8_t* footstep_mask, const uint8_t* contact_mask, const T* phase, const T* mu,
                             const T* normals_world, const T* foot_target_position, const T* foot_target_velocity,
                             T* command, uint32_t* flags, T* grf) {
  if (!c) return QLB_ERR_NOT_INITIALISED;
  QLB_GUARD(c->ctx);
  if (!controller_ready(c)) return QLB_ERR_NOT_INITIALISED;
  if (!q || !qd || !base_pose || !base_twist || !target_pose || !target_twist || !desired_stance_mask || !contact_mask ||
      !phase || !command || !flags)
    return QLB_ERR_INVALID_ARGUMENT;
  qlb_context* ctx = c->ctx;
  DeviceGuard guard(ctx->device);
  int rc = ensure_capacity(ctx, c->B);
  if (rc != QLB_OK) return rc;
  const size_t B = c->B, cap = ctx->cap;
  cudaStream_t st = ctx->stream;
  T* const d_in = reinterpret_cast<T*>(ctx->d_in);
  T* const d_out = reinterpret_cast<T*>(ctx->d_out);
  // inputs: 94 rows in the input staging (kPipe * 54 rows of cap), outputs 24 rows, the three masks one row each
  constexpr int kIn = 11, kOut = 2;
  const T* src[kIn] = {q, qd, base_pose, base_twist, target_pose, target_twist, phase, mu, normals_world,
                       foot_target_position, foot_target_velocity};
  const int rows[kIn] = {12, 12, 7, 6, 7, 6, 4, 4, 12, 12, 12};
  static_assert(kPipe * kHostInRows >= 94 && kPipe * kHostOutRows >= 24 && kPipe >= 3, "staging too small for a tick");
  const uint8_t* msrc[3] = {desired_stance_mask, footstep_mask, contact_mask};
  T* dst_out[kOut] = {command, grf};
  for (size_t b0 = 0; b0 < B && rc == QLB_OK; b0 += cap) {
    const size_t n = (B - b0 < cap) ? (B - b0) : cap;
    const T* din[kIn];
    size_t off = 0;
    for (int k = 0; k < kIn && rc == QLB_OK; k++) {
      din[k] = src[k] ? d_in + off : nullptr;
      if (src[k] && cudaMemcpy2DAsync(d_in + off, n * sizeof(T), src[k] + b0, B * sizeof(T), n * sizeof(T), rows[k],
                                      cudaMemcpyHostToDevice, st) != cudaSuccess)
        rc = QLB_ERR_CUDA;
      off += (size_t)rows[k] * cap;
    }
    const uint8_t* dmask[3];
    for (int k = 0; k < 3 && rc == QLB_OK; k++) {
      dmask[k] = msrc[k] ? ctx->d_mask + (size_t)k * cap : nullptr;
      if (msrc[k] && cudaMemcpyAsync(ctx->d_mask + (size_t)k * cap, msrc[k] + b0, n, cudaMemcpyHostToDevice, st) != cudaSuccess)
        rc = QLB_ERR_CUDA;
    }
    if (rc != QLB_OK) break;
    T* dout[kOut] = {d_out, d_out + 12 * cap};
    rc = controller_tick<T>(c, n, b0, din[0], din[1], din[2], din[3], din[4], din[5], dmask[0], dmask[1], dmask[2], din[6],
                            din[7], din[8], din[9], din[10], dout[0], ctx->d_flags, dout[1], st);
    for (int k = 0; k < kOut && rc == QLB_OK; k++)
      if (dst_out[k] && cudaMemcpy2DAsync(dst_out[k] + b0, B * sizeof(T), dout[k], n * sizeof(T), n * sizeof(T), 12,
                                          cudaMemcpyDeviceToHost, st) != cudaSuccess)
        rc = QLB_ERR_CUDA;
    if (rc == QLB_OK && cudaMemcpyAsync(flags + b0, ctx->d_flags, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess)
      rc = QLB_ERR_CUDA;
  }
  // also on failure: no copy may still be reading or writing the caller's buffers when the call returns
  if (cudaStreamSynchronize(st) != cudaSuccess && rc == QLB_OK) rc = QLB_ERR_CUDA;
  if (rc == QLB_ERR_CUDA) return cuda_fail(ctx, cudaGetLastError(), "qlb_controller_update_host");
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
  const unsigned long long blocks = ((unsigned long long)c->B + 255) / 256;
  qlb_tick_reset_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(c->B, reset_mask, c->limb, c->efforts,
                                                                                         c->refill);
  QLB_CUDA(c->ctx, cudaGetLastError());
  c->ctx->launches++;
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
                                     foot_target_velocity, command, flags, grf, stream);
}
int qlb_controller_update_f32(qlb_controller* c, const float* q, const float* qd, const float* base_pose,
                              const float* base_twist, const float* target_pose, const float* target_twist,
                              const uint8_t* desired_stance_mask, const uint8_t* footstep_mask, const uint8_t* contact_mask,
                              const float* phase, const float* mu, const float* normals_world,
                              const float* foot_target_position, const float* foot_target_velocity, float* command,
                              uint32_t* flags, float* grf, void* stream) {
  return controller_update_t<float>(c, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                    footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                    foot_target_velocity, command, flags, grf, stream);
}
int qlb_controller_update_host(qlb_controller* c, const double* q, const double* qd, const double* base_pose,
                               const double* base_twist, const double* target_pose, const double* target_twist,
                               const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                               const uint8_t* contact_mask, const double* phase, const double* mu,
                               const double* normals_world, const double* foot_target_position,
                               const double* foot_target_velocity, double* command, uint32_t* flags, double* grf) {
  return controller_update_host_t<double>(c, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                          footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                          foot_target_velocity, command, flags, grf);
}
int qlb_controller_update_f32_host(qlb_controller* c, const float* q, const float* qd, const float* base_pose,
                                   const float* base_twist, const float* target_pose, const float* target_twist,
                                   const uint8_t* desired_stance_mask, const uint8_t* footstep_mask,
                                   const uint8_t* contact_mask, const float* phase, const float* mu,
                                   const float* normals_world, const float* foot_target_position,
                                   const float* foot_target_velocity, float* command, uint32_t* flags, float* grf) {
  return controller_update_host_t<float>(c, q, qd, base_pose, base_twist, target_pose, target_twist, desired_stance_mask,
                                         footstep_mask, contact_mask, phase, mu, normals_world, foot_target_position,
                                         foot_target_velocity, command, flags, grf);
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
