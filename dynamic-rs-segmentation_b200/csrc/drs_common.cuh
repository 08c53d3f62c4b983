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

#include <initializer_list>
#include <map>
#include <memory>
#include <string>
#include <utility>
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

// ------------------------------------------------------------------ owned CUDA resources
// A stream, event, graph exec or allocation that releases itself: whatever holds one (the handle, a scene, a debug entry
// point) frees it by going away, so no list of frees has to mirror the allocations.  The destructor ignores the error of the
// release (nothing could be done about it there); reset() returns it.
template <typename T, auto Destroy>
class Owner {
 public:
  Owner() = default;
  explicit Owner(T p) : p_(p) {}
  Owner(Owner&& o) noexcept : p_(o.p_) { o.p_ = nullptr; }
  Owner& operator=(Owner&& o) noexcept {
    if (this != &o) { reset(); p_ = o.p_; o.p_ = nullptr; }
    return *this;
  }
  ~Owner() { reset(); }
  cudaError_t reset() {
    const cudaError_t e = p_ ? Destroy(p_) : cudaSuccess;
    p_ = nullptr;
    return e;
  }
  T get() const { return p_; }
  operator T() const { return p_; }

 private:
  T p_ = nullptr;
};
using Stream = Owner<cudaStream_t, cudaStreamDestroy>;
using Event = Owner<cudaEvent_t, cudaEventDestroy>;
using GraphExec = Owner<cudaGraphExec_t, cudaGraphExecDestroy>;
template <typename T> using PinnedMem = Owner<T*, cudaFreeHost>;

static inline Stream new_stream() {
  cudaStream_t s = nullptr;
  CUDA_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  return Stream(s);
}
static inline Event new_event(unsigned flags = cudaEventDisableTiming) {
  cudaEvent_t e = nullptr;
  CUDA_CHECK(cudaEventCreateWithFlags(&e, flags));
  return Event(e);
}
template <typename T>
static PinnedMem<T> new_pinned(size_t bytes, unsigned flags) {
  void* p = nullptr;
  CUDA_CHECK(cudaHostAlloc(&p, bytes, flags));
  return PinnedMem<T>((T*)p);
}

// Device memory and its size in bytes.
template <typename T>
struct DevMem {
  Owner<T*, cudaFree> p;
  size_t cap = 0;

  DevMem() = default;
  explicit DevMem(size_t bytes) { grow(bytes, bytes); }
  DevMem(DevMem&& o) noexcept : p(std::move(o.p)), cap(std::exchange(o.cap, 0)) {}
  DevMem& operator=(DevMem&& o) noexcept {
    p = std::move(o.p);
    cap = std::exchange(o.cap, 0);
    return *this;
  }
  T* get() const { return p; }
  operator T*() const { return p; }
  // Makes room for `need` bytes.  A smaller buffer is freed, once the streams in `sync` (whose queued work may still use it)
  // have drained, and replaced by `want` >= need bytes.  Returns whether it was.
  bool grow(size_t need, size_t want, std::initializer_list<cudaStream_t> sync = {}) {
    if (cap >= need) return false;
    for (cudaStream_t s : sync) CUDA_CHECK(cudaStreamSynchronize(s));
    reset();
    void* q = nullptr;
    CUDA_CHECK(cudaMalloc(&q, want));
    p = Owner<T*, cudaFree>((T*)q);
    cap = want;
    return true;
  }
  void reset() {
    cap = 0;
    CUDA_CHECK(p.reset());
  }
};

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
  DevMem<void> w_fprop;      // [co][k*k*ci]  (K index = tap*ci + c)
  DevMem<void> w_dgrad;      // [ci][k*k*co]  (flipped taps)
  DevMem<float> fold_scale;  // [co] eval-mode BN folded: y = act(conv*scale + shift)
  DevMem<float> fold_shift;
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
  DevMem<void> data;       // [H,W,C] f64 or f32 (re-uploads of the same shape reuse the buffers)
  DevMem<uint8_t> labels;
  int H = 0, W = 0, C = 0, dtype = 0;
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
  DevMem<char> mem;
  size_t used = 0;
  void reset() { used = 0; }
  void* take(size_t bytes) {
    size_t off = (used + 1023) & ~size_t(1023);
    if (off + bytes > mem.cap) return nullptr;
    used = off + bytes;
    return mem.get() + off;
  }
};

struct InferLane {
  Stream stream;
  Arena arena;
  DevMem<float> x, lg;
  Event fwd_done, acc_done;
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
  std::vector<std::pair<Event, Event>> events;   // external event-record nodes around the tensor-core launches
  GraphExec exec;                                // (declared after the events: destroyed before them)
  int64_t launches = 0, conv_launches = 0;
  double conv_flops = 0;
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
  int chunk = 0;                   // chunk size the accumulation ranges were split for
  std::vector<int32_t> cuts;       // accumulation ranges [cuts[r], cuts[r+1]) (drs_scene_api.cuh: accum_ranges)
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
  Stream own_stream;
  cudaStream_t stream = nullptr;
  int64_t launches = 0;
  // Programmatic dependent launch (training step, main stream): pdl_on = the step allows it, pdl_prev = the last operation
  // enqueued on `stream` was one of our kernels (anything else -- memset, copy, collective, stream switch -- clears it)
  bool pdl_on = false, pdl_prev = false;

  // variables
  DevMem<float> params;      // flat trainables: all weights & biases
  DevMem<float> grads;
  DevMem<float> moms;
  DevMem<float> bnstat;      // moving_mean / moving_variance
  int64_t global_step = 0;
  int ignore_label = -1;     // contest: label excluded from loss / confusion when no mask is passed
  bool packed_dirty = true;  // packed operand matrices need refresh
  bool eval_dirty = true;    // folded eval-mode BN / conv1 tensor-core operand need refresh

  // workspace: launches carve from *arena, the handle's own arena or, inside its StreamScope, the scene lane's
  Arena own_arena;
  Arena* arena = &own_arena;
  uint64_t arena_epoch = 0;
  DevMem<char> dstage;       // device staging for host entry points

  // host-mapped diagnostics written by bounded waits
  PinnedMem<uint32_t> diag_host;
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
  std::vector<std::pair<Event, Event>> conv_events;
  size_t conv_events_used = 0;
  bool time_convs = false;

  // debug taps: scope -> (device ptr, elem type (0 f32, 1 f16, 2 bf16), cstride, coff, co, pixels)
  struct Tap { const void* ptr; int type; int cstride, coff, co; int64_t pixels; };
  std::map<std::string, Tap> taps;

  PFN_encodeTiled encodeTiled = nullptr;
  PFN_encodeIm2col encodeIm2col = nullptr;
  std::map<TmKey, CUtensorMap> tm_cache;

  // persistent scene-pass buffers: cudaMalloc / cudaFree of gigabyte-sized buffers per call costs hundreds of milliseconds,
  // so each only ever grows.  The label map of the last pass stays for drs_scene_confusion and drs_scene_gather_labels.
  int last_scene = -1, last_row_begin = 0, last_rows = 0, last_W = 0;
  struct {
    DevMem<float> prob;                   // score map [rows][W][K]
    DevMem<uint32_t> occur;               // occurrence counts [rows][W]
    DevMem<int32_t> cell_off, cell_seq;   // cell tables of the visiting order
    DevMem<uint8_t> labels;               // label map [rows][W]
    DevMem<double> mean;                  // mean score map [rows][W][K]
    DevMem<float> prob_sum;               // multi-scale: sum over the scales of softmax(mean) [rows][W][K]
    DevMem<int32_t> inst;                 // (scene, row, col) of every patch of the pass
    DevMem<uint8_t> assembled;            // [H][W] label map assembled from every rank's stripe
  } pass;
  std::vector<PassGeometry> pass_geometry;   // the last few scene-pass geometries, oldest first
  std::map<TrainGraphKey, TrainGraph> graphs;
  TrainGraph* capturing = nullptr;   // non-null while a training step is being captured
  Stream side_stream;                // filter gradients run here, overlapped with the backward's HBM-bound kernels
  Event ev_dz[2], ev_wgrad[2];
  // data-parallel exchange of the late layers' gradients, overlapped with the rest of the backward
  Stream comm_stream;
  Event ev_bucket_ready, ev_bucket_done;
  Event ev_x8;                       // conv1's padded input is ready: the side stream builds the im2col matrix under the forward
  bool use_graphs = true;           // DRS_GRAPHS=0 turns the whole-step CUDA graphs off (drs_create)
  double conv_ms_acc = 0;            // device time of profiled launches already read back
  InferLane lane;                 // scene-inference lane (drs_scene_api.cuh)
  Event lane_ready;
  // streamed scene upload (drs_scene_infer_host): copy stream + "rows uploaded" event
  Stream copy_stream;
  Event up_ev;
  DevMem<uint8_t> is_weight;      // [n_trainable] 1 for `weights` variables
  SceneTable table;               // host copy of the device scene table
  // training scratch kept between calls
  DevMem<float> mean;             // [sum co] batch mean of the last train step (per layer, same offsets as mm_off/2)
  DevMem<float> inv_std;
  DevMem<float> sums;             // [2*256]
  DevMem<float> loss_dev;         // [4]: ce, l2, count, spare
  DevMem<unsigned int> cm_dev;    // [K*K+1]
  DevMem<unsigned int> count_dev;
  unsigned int* bn_counter = nullptr;   // last-block-done counter of bn_partial_kernel (self-resetting)
  DevMem<long long> bn_acc;             // [BN_ACC_REPLICAS][2*512] fixed-point accumulators of bn_partial_kernel (self-clearing)
  DevMem<float> ones;             // [512]
  DevMem<float> zeros;            // [512]
  // profiling
  double conv_flops = 0;
  int64_t conv_launches = 0;
  // pipelined training loop (drs_gather_plan_dev / drs_train_step_async / drs_train_result): the plan of step i+1 is
  // uploaded on plan_stream into a two-slot device staging ring while step i runs; loss + confusion counts of each step
  // land in a ring of pinned result slots behind an event, so the host never blocks on the step it has just enqueued
  void* nccl = nullptr;             // ncclComm_t of drs_comm_init (drs_comm.cuh); null: single process or callback exchange
  int rank = 0;
  Stream plan_stream;
  DevMem<char> plan_stage[2];
  Event plan_uploaded[2], plan_consumed[2];
  bool plan_consumed_valid[2] = {false, false};
  int64_t plan_calls = 0;
  static constexpr int RESULT_RING = 8;
  PinnedMem<float> result_host;     // [RESULT_RING][RESULT_STRIDE]
  Event result_ev[RESULT_RING];
  int64_t next_ticket = 0;
  // DRS_DEBUG_KEEP=1: fp32 copies of training-step tensors whose buffers are reused ("z:", "dout:", "da:", "dz:<scope>")
  std::vector<DevMem<float>> keep;
  bool debug_keep = false;
};
typedef drs_handle_s Handle;

static inline void ensure_arena(Handle* h, size_t bytes) {
  if (h->arena->mem.grow(bytes, bytes + (bytes >> 3) + (size_t(1) << 20), {h->stream}))
    h->arena_epoch++;          // cached CUDA graphs hold pointers into the old arena
}
static inline void* arena_take(Handle* h, size_t bytes) {
  void* p = h->arena->take(bytes);
  DRS_CHECK(p != nullptr, "workspace arena exhausted (need %zu more bytes, cap %zu)", bytes, h->arena->mem.cap);
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
    DRS_CHECK(p != nullptr, "workspace arena exhausted (need %zu more bytes, cap %zu)", bytes, arena->mem.cap);
    return (T*)p;
  }
};

// Launches inside the scope go to stream `s` (and carve from `arena`, when given) if `on`; the handle's stream, arena and
// PDL state are restored when the scope ends, also when a launch throws.  The first launch on `s` gets no programmatic
// dependency: its predecessor on that stream is not known.
struct StreamScope {
  drs_handle_s* h;
  bool on, pdl_prev;
  cudaStream_t stream;
  Arena* arena;
  StreamScope(drs_handle_s* h_, bool on_, cudaStream_t s, Arena* a = nullptr)
      : h(h_), on(on_), pdl_prev(h_->pdl_prev), stream(h_->stream), arena(h_->arena) {
    if (on) { h->stream = s; h->pdl_prev = false; }
    if (on && a) h->arena = a;
  }
  ~StreamScope() {
    if (on) { h->stream = stream; h->pdl_prev = pdl_prev; }
    h->arena = arena;
  }
};
static inline void ensure_dstage(Handle* h, size_t bytes) { h->dstage.grow(bytes, bytes + (bytes >> 2) + 4096, {h->stream}); }
// a scene-pass buffer of the handle, grown to exactly `bytes` (an empty table still gets an address)
template <typename T>
static T* pass_buf(Handle* h, DevMem<T>& b, size_t bytes) {
  if (bytes == 0) bytes = 16;
  b.grow(bytes, bytes, {h->stream});
  return b;
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
