// In-library collectives: NCCL over NVLink / NVSwitch, resolved at run time.  Included by drs_api.cu.
//
// The reference is single-process (SURVEY.md section 2.1); the sharded path has exactly three exchanges (section 8e):
//   training    one sum-allreduce of [gradients ++ loss ++ confusion counts] per step (two buckets, the large one overlapped
//               with the backward), plus the per-layer BN sums when sync_bn (12-16 reductions of <= 2 KB per step);
//   inference   the uint8 label stripes of a scene pass are sent to rank 0 (no data-path collective otherwise).
// Calling ncclAllReduce directly from the step -- instead of a C -> Python -> torch.distributed callback per exchange --
// removes ~20 us of host work per reduction and makes the data-parallel step capturable as a CUDA graph.
//
// libnccl.so.2 is dlopen'ed: no link-time dependency, and a process that already holds a copy (torch's bundled one) gets
// that same instance.  Only the handful of entry points below is used; the prototypes follow nccl.h (2.27 / 2.28).
#pragma once
#include <dlfcn.h>

typedef struct drs_nccl_comm* drs_ncclComm_t;
struct drs_ncclUniqueId { char internal[128]; };
enum { DRS_NCCL_SUM = 0, DRS_NCCL_UINT8 = 1, DRS_NCCL_FLOAT32 = 7 };

struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(drs_ncclUniqueId*) = nullptr;
  int (*CommInitRank)(drs_ncclComm_t*, int, drs_ncclUniqueId, int) = nullptr;
  int (*CommDestroy)(drs_ncclComm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, drs_ncclComm_t, cudaStream_t) = nullptr;
  int (*Send)(const void*, size_t, int, int, drs_ncclComm_t, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, drs_ncclComm_t, cudaStream_t) = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, drs_ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};

static NcclApi* nccl_api() {
  static NcclApi api;
  if (api.lib) return &api;
  const char* names[] = {getenv("DRS_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    if (!n || !*n) continue;
    api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) break;
  }
  DRS_CHECK(api.lib, "NCCL not found (dlopen libnccl.so.2 failed: %s); set DRS_NCCL_LIB", dlerror());
  auto sym = [&](const char* s) {
    void* p = dlsym(api.lib, s);
    if (!p) { api.lib = nullptr; DRS_FAIL("NCCL symbol %s missing", s); }
    return p;
  };
  api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
  api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
  api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
  api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
  api.Send = (decltype(api.Send))sym("ncclSend");
  api.Recv = (decltype(api.Recv))sym("ncclRecv");
  api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
  api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
  api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
  api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
  return &api;
}

#define NCCL_CHECK(expr)                                                                             \
  do {                                                                                               \
    int _r = (expr);                                                                                 \
    if (_r != 0) DRS_FAIL("NCCL error %d (%s) at %s", _r, nccl_api()->GetErrorString(_r), #expr);    \
  } while (0)

extern "C" int drs_comm_unique_id(uint8_t* id_out) {
  API_BEGIN
  DRS_CHECK(id_out, "null argument");
  drs_ncclUniqueId id;
  NCCL_CHECK(nccl_api()->GetUniqueId(&id));
  memcpy(id_out, id.internal, 128);
  API_END
}

extern "C" int drs_comm_init(drs_handle_t h, const uint8_t* id128, int32_t rank, int32_t world, int32_t sync_bn) {
  API_BEGIN
  DRS_CHECK(h && id128, "null argument");
  DRS_CHECK(world >= 1 && rank >= 0 && rank < world, "comm_init: bad rank %d of %d", rank, world);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  if (h->nccl) { NCCL_CHECK(nccl_api()->CommDestroy((drs_ncclComm_t)h->nccl)); h->nccl = nullptr; }
  drs_ncclUniqueId id;
  memcpy(id.internal, id128, 128);
  drs_ncclComm_t comm = nullptr;
  NCCL_CHECK(nccl_api()->CommInitRank(&comm, world, id, rank));
  h->nccl = comm;
  h->rank = rank;
  h->world = world;
  h->sync_bn = sync_bn ? 1 : 0;
  h->allreduce = nullptr;
  h->allreduce_user = nullptr;
  API_END
}

extern "C" int drs_comm_destroy(drs_handle_t h) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  if (h->nccl) {
    CUDA_CHECK(cudaSetDevice(h->cfg.device));
    cudaStreamSynchronize(h->stream);
    if (h->comm_stream) cudaStreamSynchronize(h->comm_stream);
    NCCL_CHECK(nccl_api()->CommDestroy((drs_ncclComm_t)h->nccl));
    h->nccl = nullptr;
    h->world = 1;
  }
  API_END
}

// sum `count` floats over ranks in place, in the order of `on_stream` (default: the handle's stream)
static void do_allreduce(Handle* h, float* buf, int64_t count, cudaStream_t on_stream = (cudaStream_t)(uintptr_t)1) {
  if (h->world <= 1) return;
  h->pdl_prev = false;
  const cudaStream_t st = on_stream == (cudaStream_t)(uintptr_t)1 ? h->stream : on_stream;
  if (h->nccl) {
    NCCL_CHECK(nccl_api()->AllReduce(buf, buf, (size_t)count, DRS_NCCL_FLOAT32, DRS_NCCL_SUM, (drs_ncclComm_t)h->nccl, st));
    return;
  }
  if (!h->allreduce) return;
  int rc = h->allreduce(h->allreduce_user, buf, count, (void*)st);
  DRS_CHECK(rc == 0, "allreduce callback failed with %d", rc);
}

// Stripe-sharded scene pass: every rank's uint8 label stripe (the label map of the last drs_scene_infer) goes to rank 0 over
// NVLink, straight from device memory; rank 0 assembles [H, W] on the device and copies it to the host once.
//   row_cuts [world+1]: stripe r holds rows [row_cuts[r], row_cuts[r+1]) (dist.stripe_bounds)
extern "C" int drs_scene_gather_labels(drs_handle_t h, int32_t H, int32_t W, const int32_t* row_cuts, int32_t all_ranks,
                                       uint8_t* labels_out_host) {
  API_BEGIN
  DRS_CHECK(h && row_cuts, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  DRS_CHECK(h->nccl, "scene_gather_labels: drs_comm_init has not been called");
  const int world = h->world, rank = h->rank;
  DRS_CHECK(h->last_scene >= 0 && h->last_W == W && h->last_row_begin == row_cuts[rank] &&
                h->last_rows == row_cuts[rank + 1] - row_cuts[rank],
            "scene_gather_labels: the last scene pass covered rows [%d,%d), not this rank's stripe [%d,%d)", h->last_row_begin,
            h->last_row_begin + h->last_rows, row_cuts[rank], row_cuts[rank + 1]);
  DRS_CHECK(labels_out_host || (rank != 0 && !all_ranks), "scene_gather_labels: this rank needs the output buffer");
  const uint8_t* mine = h->pass.labels;
  NcclApi* n = nccl_api();
  drs_ncclComm_t comm = (drs_ncclComm_t)h->nccl;
  uint8_t* full = (rank == 0 || all_ranks) ? pass_buf(h, h->pass.assembled, (size_t)H * W) : nullptr;
  if (rank != 0) {
    if (h->last_rows > 0) NCCL_CHECK(n->Send(mine, (size_t)h->last_rows * W, DRS_NCCL_UINT8, 0, comm, h->stream));
  } else {
    NCCL_CHECK(n->GroupStart());
    for (int r = 1; r < world; ++r) {
      const int rows = row_cuts[r + 1] - row_cuts[r];
      if (rows > 0) NCCL_CHECK(n->Recv(full + (size_t)row_cuts[r] * W, (size_t)rows * W, DRS_NCCL_UINT8, r, comm, h->stream));
    }
    NCCL_CHECK(n->GroupEnd());
    CUDA_CHECK(cudaMemcpyAsync(full + (size_t)row_cuts[0] * W, mine, (size_t)h->last_rows * W, cudaMemcpyDeviceToDevice, h->stream));
  }
  if (all_ranks) NCCL_CHECK(n->Broadcast(full, full, (size_t)H * W, DRS_NCCL_UINT8, 0, comm, h->stream));
  if (labels_out_host && full) CUDA_CHECK(cudaMemcpyAsync(labels_out_host, full, (size_t)H * W, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  API_END
}
