// Shared declarations of libdrs: error handling, the handle, device arena, tensor-map encoding.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/drs.h"

#define DRS_VERSION 100

// ------------------------------------------------------------------ errors
extern thread_local char g_drs_err[1024];
struct DrsError {
  int code;
};
#define DRS_FAIL(...)                                   \
  do {                                                  \
    snprintf(g_drs_err, sizeof(g_drs_err), __VA_ARGS__); \
    throw DrsError{1};                                  \
  } while (0)
#define CUDA_CHECK(expr)                                                                               \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess) DRS_FAIL("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
  } while (0)
#define DRS_CHECK(cond, ...)          \
  do {                                \
    if (!(cond)) DRS_FAIL(__VA_ARGS__); \
  } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

// ------------------------------------------------------------------ network description
enum { ACT_NONE = 0, ACT_RELU = 1, ACT_LRELU = 2 };

struct ConvLayer {
  std::string scope;
  int k, rate, ci, co;
  int pad_b, pad_a;       // SAME padding before/after (Appendix A)
  int in_coff;            // channel offset of the input inside its buffer (dense nets read [0,ci))
  int out_coff;           // channel offset of the output inside its buffer (dense nets write a slice)
  // offsets (in floats) into the flat trainable buffer
  int64_t w_off, b_off;
  // offsets into the flat BN-statistics buffer
  int64_t mm_off, mv_off;
  // packed low-precision operand matrices
  void* w_fprop = nullptr;   // [co][k*k*ci]  (K index = tap*ci + c)
  void* w_dgrad = nullptr;   // [ci][k*k*co]  (flipped taps)
  float* fold_scale = nullptr;  // [co] eval-mode BN folded: y = act(conv*scale + shift)
  float* fold_shift = nullptr;
  float* raw_scale = nullptr;   // [co] ones
  // structural variants (variants.cuh): a post-op behind the activation, and explicit buffer routing for the squeeze modules
  int post = 0;           // 0 none, 1 SAME average pooling post_k x post_k (isprs:753-758), 2 squeeze-and-excitation gate
  int post_k = 0;
  int se = -1;            // index into NetDesc::se
  int in_group = -1;      // layer that leads the buffer this layer reads (-1: the previous layer / the network input)
  int in_cs = 0;          // channel stride of that buffer
  int out_group = -1;     // layer that leads the buffer this layer writes a channel slice of (-1: its own buffer)
  int out_cs = 0;         // channel stride of the output buffer (0: co)
};

// _squeeze_excitation_layer (isprs:682-697): two fully connected layers on the per-image channel means
struct SeBlock {
  std::string name;       // "se1": variables se1_fc1/{weights,biases}, se1_fc2/{weights,biases}
  int c, r;               // channels, channels / ratio
  int64_t w1_off, b1_off, w2_off, b2_off;   // offsets into the flat trainable buffer, in this order, right behind the layer
};

struct NetDesc {
  int net_type;
  int channels, classes;
  int act;            // ACT_RELU / ACT_LRELU
  bool pool, dense;
  bool squeeze = false;   // dilated_icpr_rate6_squeeze: conv2..6 are squeeze modules (three convs, two share an output buffer)
  std::vector<SeBlock> se;
  std::vector<ConvLayer> convs;
  int cls_in;         // classifier input width
  int64_t cls_w_off, cls_b_off;
  int feat_stride;    // channel stride of the feature buffers (dense: 448; else max co)
  int64_t n_trainable; // floats in the flat trainable buffer
  int64_t n_bnstat;
};

struct Scene {
  void* data = nullptr;   // [H,W,C] f64 or f32
  uint8_t* labels = nullptr;
  int H = 0, W = 0, C = 0, dtype = 0;
  size_t data_cap = 0, labels_cap = 0;   // allocation sizes (re-uploads of the same shape reuse the buffers)
  int row0 = 0, rows = 0;   // resident rows [row0, row0+rows) of the H-row scene (a rank keeps only its stripe + halo)
};

constexpr int MAX_SCENES = 64;
struct SceneDesc {
  const void* data;       // rows [row0, row0 + rows) of the scene
  const uint8_t* labels;
  int H, W, C, dtype;
  int row0, rows;
};
struct SceneTable {
  SceneDesc s[MAX_SCENES];
};

constexpr int MAX_CLASSES = 8;

struct Arena {
  char* base = nullptr;
  size_t cap = 0, used = 0;
  void reset() { used = 0; }
  void* take(size_t bytes) {
    size_t off = (used + 1023) & ~size_t(1023);
    if (off + bytes > cap) return nullptr;
    used = off + bytes;
    return base + off;
  }
};

struct InferLane {
  cudaStream_t stream = nullptr;
  Arena arena;
  float* x = nullptr;
  float* lg = nullptr;
  size_t x_cap = 0, lg_cap = 0;
  cudaEvent_t fwd_done = nullptr, acc_done = nullptr;
};

// One captured training step (CUDA graph) per (batch, patch size, buffers, learning rate): the step is ~65 small
// dependent launches, so replaying it as a graph removes the launch gaps between them.
struct TrainGraphKey {
  int B, crop, ignore_label, profiling;
  const void *x, *y, *mask, *acc_mask, *pred, *cm;
  uint64_t lr_bits;
  uint64_t arena_epoch;
  bool operator<(const TrainGraphKey& o) const { return memcmp(this, &o, sizeof(*this)) < 0; }
};
struct TrainGraph {
  cudaGraphExec_t exec = nullptr;
  int64_t launches = 0, conv_launches = 0;
  double conv_flops = 0;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> events;   // external event-record nodes around the tensor-core launches
};

// cell tables of an ordered position list (host)
struct CellTables {
  int nh, nw, stride;
  std::vector<int32_t> off, seq;
};
// a scene pass's visiting order and cell tables, memoised per geometry (drs_scene_api.cuh: pass_geometry)
struct PassGeometry {
  int key[8];
  std::vector<int32_t> pos, inst;
  CellTables ct;
};

constexpr int RESULT_STRIDE = 64 + MAX_CLASSES * MAX_CLASSES;   // floats per pinned result slot: loss, then K*K+1 counts

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                     const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Tensor maps are pure functions of (base pointer, geometry); encoding one costs a few microseconds on the host and every
// convolution launch needs three, so they are memoised per handle (workspace addresses repeat from step to step).
struct TmKey {
  uint64_t v[8];
  bool operator<(const TmKey& o) const { return memcmp(v, o.v, sizeof(v)) < 0; }
};

struct drs_handle_s {
  drs_config cfg;
  NetDesc net;
  int sm_count = 148;
  int driver_version = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  int64_t launches = 0;
  // Programmatic dependent launch (training step, main stream): pdl_on = the step allows it, pdl_prev = the last operation
  // enqueued on `stream` was one of our kernels (anything else -- memset, copy, collective, stream switch -- clears it)
  bool pdl_on = false, pdl_prev = false;

  // variables
  float* params = nullptr;   // flat trainables: all weights & biases
  float* grads = nullptr;
  float* moms = nullptr;
  float* bnstat = nullptr;   // moving_mean / moving_variance
  int64_t global_step = 0;
  int ignore_label = -1;     // contest: label excluded from loss / confusion when no mask is passed
  bool packed_dirty = true;  // packed operand matrices need refresh
  bool eval_dirty = true;    // folded eval-mode BN / conv1 tensor-core operand need refresh

  // workspace
  Arena arena;
  uint64_t arena_epoch = 0;
  // pinned staging for *_host entry points
  void* pinned = nullptr;
  size_t pinned_cap = 0;
  void* dstage = nullptr;    // device staging for host entry points
  size_t dstage_cap = 0;

  // host-mapped diagnostics written by bounded waits
  uint32_t* diag_host = nullptr;
  uint32_t* diag_dev = nullptr;

  // scenes
  std::map<int, Scene> scenes;
  double norm_mean[3] = {0, 0, 0}, norm_std[3] = {1, 1, 1};
  int gather_fp16 = 0;       // coffee training patches are float16 before normalisation (coffee:293)

  // data parallel
  drs_allreduce_fn allreduce = nullptr;
  void* allreduce_user = nullptr;
  int world = 1;
  int sync_bn = 0;

  // timing of conv kernels
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> conv_events;
  size_t conv_events_used = 0;
  bool time_convs = false;

  // debug taps: scope -> (device ptr, elem type (0 f32, 1 f16, 2 bf16), cstride, coff, co, pixels)
  struct Tap { const void* ptr; int type; int cstride, coff, co; int64_t pixels; };
  std::map<std::string, Tap> taps;

  PFN_encodeTiled encodeTiled = nullptr;
  PFN_encodeIm2col encodeIm2col = nullptr;
  std::map<TmKey, CUtensorMap> tm_cache;

  // persistent scene-pass buffers (score map, occurrence counts, cell tables, label map ...): cudaMalloc / cudaFree of
  // gigabyte-sized buffers per call costs hundreds of milliseconds, so each named slot only ever grows
  // the label map of the last scene pass stays in slot 4 for drs_scene_confusion
  int last_scene = -1, last_row_begin = 0, last_rows = 0, last_W = 0;
  void* slot_ptr[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  size_t slot_cap[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::vector<PassGeometry> pass_geometry;   // the last few scene-pass geometries, oldest first
  std::map<TrainGraphKey, TrainGraph> graphs;
  TrainGraph* capturing = nullptr;   // non-null while a training step is being captured
  cudaStream_t side_stream = nullptr;     // filter gradients run here, overlapped with the backward's HBM-bound kernels
  cudaEvent_t ev_dz[2] = {nullptr, nullptr}, ev_wgrad[2] = {nullptr, nullptr};
  // data-parallel exchange of the late layers' gradients, overlapped with the rest of the backward
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t ev_bucket_ready = nullptr, ev_bucket_done = nullptr;
  cudaEvent_t ev_x8 = nullptr;          // conv1's padded input is ready: the side stream builds the im2col matrix under the forward
  bool use_graphs = true;           // DRS_GRAPHS=0 turns the whole-step CUDA graphs off (drs_create)
  double conv_ms_acc = 0;            // device time of profiled launches already read back
  InferLane lane;                 // scene-inference lane (drs_scene_api.cuh)
  cudaEvent_t lane_ready = nullptr;
  // streamed scene upload (drs_scene_infer_host): copy stream + "rows uploaded" event
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t up_ev[1] = {nullptr};
  uint8_t* is_weight = nullptr;   // [n_trainable] 1 for `weights` variables
  SceneTable table;               // host copy of the device scene table
  // training scratch kept between calls
  float* mean = nullptr;          // [sum co] batch mean of the last train step (per layer, same offsets as mm_off/2)
  float* inv_std = nullptr;
  float* sums = nullptr;          // [2*256]
  float* loss_dev = nullptr;      // [4]: ce, l2, count, spare
  unsigned int* cm_dev = nullptr; // [K*K+1]
  unsigned int* count_dev = nullptr;
  unsigned int* bn_counter = nullptr;   // last-block-done counter of bn_partial_kernel (self-resetting)
  long long* bn_acc = nullptr;          // [BN_ACC_REPLICAS][2*512] fixed-point accumulators of bn_partial_kernel (self-clearing)
  float* ones = nullptr;          // [512]
  float* zeros = nullptr;         // [512]
  // profiling
  double conv_flops = 0;
  int64_t conv_launches = 0;
  // pipelined training loop (drs_gather_plan_dev / drs_train_step_async / drs_train_result): the plan of step i+1 is
  // uploaded on plan_stream into a two-slot device staging ring while step i runs; loss + confusion counts of each step
  // land in a ring of pinned result slots behind an event, so the host never blocks on the step it has just enqueued
  void* nccl = nullptr;             // ncclComm_t of drs_comm_init (drs_comm.cuh); null: single process or callback exchange
  int rank = 0;
  cudaStream_t plan_stream = nullptr;
  void* plan_stage[2] = {nullptr, nullptr};
  size_t plan_stage_cap[2] = {0, 0};
  cudaEvent_t plan_uploaded[2] = {nullptr, nullptr}, plan_consumed[2] = {nullptr, nullptr};
  bool plan_consumed_valid[2] = {false, false};
  int64_t plan_calls = 0;
  static constexpr int RESULT_RING = 8;
  float* result_host = nullptr;     // pinned [RESULT_RING][RESULT_STRIDE]
  cudaEvent_t result_ev[RESULT_RING] = {};
  int64_t next_ticket = 0;
  // DRS_DEBUG_KEEP=1: fp32 copies of backward intermediates ("dz:<scope>", "da:<scope>")
  std::vector<float*> keep;
  bool debug_keep = false;
};
typedef drs_handle_s Handle;

static inline void ensure_arena(Handle* h, size_t bytes) {
  if (h->arena.cap >= bytes) return;
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (h->arena.base) CUDA_CHECK(cudaFree(h->arena.base));
  h->arena.base = nullptr;
  h->arena.cap = 0;
  h->arena_epoch++;          // cached CUDA graphs hold pointers into the old arena
  size_t want = bytes + (bytes >> 3) + (size_t(1) << 20);
  CUDA_CHECK(cudaMalloc(&h->arena.base, want));
  h->arena.cap = want;
}
static inline void* arena_take(Handle* h, size_t bytes) {
  void* p = h->arena.take(bytes);
  DRS_CHECK(p != nullptr, "workspace arena exhausted (need %zu more bytes, cap %zu)", bytes, h->arena.cap);
  return p;
}
// What a workspace layout (TrainWs, EvalWs) runs against: with an arena it carves the buffers from it; without one it only
// adds up what the same requests take, and that sum is what the arena is sized by.
struct WsAlloc {
  Arena* arena = nullptr;
  size_t used = 0;
  template <typename T> T* take(size_t bytes) {
    used = round_up(used, 1024) + bytes;
    if (!arena) return nullptr;
    void* p = arena->take(bytes);
    DRS_CHECK(p != nullptr, "workspace arena exhausted (need %zu more bytes, cap %zu)", bytes, arena->cap);
    return (T*)p;
  }
};

// Launches inside the scope go to stream `s` (and carve from `arena`, when given) if `on`; the handle's stream, arena and
// PDL state are restored when the scope ends, also when a launch throws.  The first launch on `s` gets no programmatic
// dependency: its predecessor on that stream is not known.
struct StreamScope {
  drs_handle_s* h;
  bool on, swap_arena, pdl_prev;
  cudaStream_t stream;
  Arena arena;
  StreamScope(drs_handle_s* h_, bool on_, cudaStream_t s, const Arena* a = nullptr)
      : h(h_), on(on_), swap_arena(on_ && a), pdl_prev(h_->pdl_prev), stream(h_->stream), arena(h_->arena) {
    if (on) { h->stream = s; h->pdl_prev = false; }
    if (swap_arena) h->arena = *a;
  }
  ~StreamScope() {
    if (on) { h->stream = stream; h->pdl_prev = pdl_prev; }
    if (swap_arena) h->arena = arena;
  }
};
static inline void ensure_pinned(Handle* h, size_t bytes) {
  if (h->pinned_cap >= bytes) return;
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (h->pinned) CUDA_CHECK(cudaFreeHost(h->pinned));
  h->pinned = nullptr;
  size_t want = bytes + (bytes >> 2) + 4096;
  CUDA_CHECK(cudaHostAlloc(&h->pinned, want, cudaHostAllocDefault));
  h->pinned_cap = want;
}
static inline void ensure_dstage(Handle* h, size_t bytes) {
  if (h->dstage_cap >= bytes) return;
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  if (h->dstage) CUDA_CHECK(cudaFree(h->dstage));
  h->dstage = nullptr;
  size_t want = bytes + (bytes >> 2) + 4096;
  CUDA_CHECK(cudaMalloc(&h->dstage, want));
  h->dstage_cap = want;
}

// Train-mode BN statistics: what the last block of a statistics-producing kernel (bn_partial_kernel, or the conv epilogue)
// does with the grid-wide sums.
struct BnFinish {
  long long* acc;          // [2][C] fixed-point accumulators, zero before the launch; cleared by the kernel
  double fx_scale;         // fixed-point scale (2^20 forward statistics, 2^40 backward sums)
  unsigned int* counter;   // zero before the launch; reset by the kernel
  float* sums;             // [2][C] out
  float* mean;             // non-null: also finalize (batch mean / inv_std, moving-average update)
  float* inv_std;
  float* mov_mean;
  float* mov_var;
  double count;
  float eps, decay;
  int unbiased_ema;
};

// The fixed-point accumulators are replicated: a block adds into replica (blockIdx.x mod BN_ACC_REPLICAS) and the finishing
// block sums the replicas (integers: still order-independent).  With one copy, a 1184-block launch put 600 k 64-bit atomics on
// 4 KB of addresses -- a handful of L2 slices -- and the statistics tail cost more than the pass it was fused into.
constexpr int BN_ACC_REPLICAS = 16;
constexpr int BN_ACC_STRIDE = 1024;      // entries per replica: [2][512 channels]
__device__ __forceinline__ unsigned long long* bn_acc_mine(const BnFinish& f) {
  return reinterpret_cast<unsigned long long*>(f.acc) + (size_t)(blockIdx.x & (BN_ACC_REPLICAS - 1)) * BN_ACC_STRIDE;
}
// finishing block only: total of entry i over the replicas; clears them for the next launch
__device__ __forceinline__ long long bn_acc_take(const BnFinish& f, int i) {
  long long t = 0;
#pragma unroll
  for (int r = 0; r < BN_ACC_REPLICAS; ++r) {
    long long* q = f.acc + (size_t)r * BN_ACC_STRIDE + i;
    t += __ldcg(q);
    *q = 0;
  }
  return t;
}

// ---- programmatic dependent launch ------------------------------------------------------------------------------------
// A kernel launched through launch_pdl may be made resident while the previous kernel of the stream is still draining: its
// blocks run up to pdl_wait() and stop there until that kernel has completed and its writes are visible.  Every kernel
// launched this way executes pdl_wait() before its first global access (without a programmatic dependency the instruction
// returns at once), so completion stays transitive along the stream; pdl_trigger() right behind it allows the launch of the
// next kernel as soon as every block of this one has started.  Measured on the training step: the 1.2-3 us between two
// consecutive kernels of the graph shrink to ~0.5 us.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_sync() { pdl_wait(); pdl_trigger(); }

static bool pdl_env() {
  static const bool on = !getenv("DRS_NO_PDL");
  return on;
}
template <typename... P, typename... A>
static void launch_pdl(drs_handle_s* h, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = h->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = (h->pdl_on && h->pdl_prev && pdl_env()) ? 1 : 0;
  CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, static_cast<P>(args)...));
}

#define LAUNCH_CHECK(h)                 \
  do {                                  \
    (h)->launches++;                    \
    (h)->pdl_prev = true;               \
    CUDA_CHECK(cudaGetLastError());     \
  } while (0)

// element type tags shared by templated kernels
enum { ET_F32 = 0, ET_F16 = 1, ET_BF16 = 2 };
template <typename T> struct ElemTag;
template <> struct ElemTag<float> { static constexpr int v = ET_F32; };
template <> struct ElemTag<__half> { static constexpr int v = ET_F16; };
template <> struct ElemTag<__nv_bfloat16> { static constexpr int v = ET_BF16; };

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == ACT_RELU) return fmaxf(v, 0.0f);
  if (act == ACT_LRELU) return fmaxf(0.1f * v, v);   // isprs:620-621 tf.maximum(alpha*x, x)
  return v;
}
