// libdrs.so -- C-ABI entry points (include/drs.h) and the orchestration of the four dilated nets.
// Reference graph: dilated_icpr_original / dilated_grsl / dilated_icpr_rate6_densely / dilated_grsl_rate8
// (/root/reference/isprs_dilated_random.py:761-788, 962-993, 914-959, 996-1033), loss_def (1089-1099),
// MomentumOptimizer (1685-1687).  No CPU fallback: every compute entry point needs an sm_100 device.
#include "conv_simt.cuh"
#include "conv_tc.cuh"
#include "drs_common.cuh"
#include "ops.cuh"
#include "scene.cuh"
#include "wgrad_tc.cuh"
#include "conv1_tc.cuh"
#include "npz_io.h"

#include <functional>

thread_local char g_drs_err[1024] = {0};

#define API_BEGIN try {
#define API_END                                                        \
  }                                                                    \
  catch (const DrsError& e) { return e.code; }                         \
  catch (const std::exception& e) {                                    \
    snprintf(g_drs_err, sizeof(g_drs_err), "exception: %s", e.what()); \
    return 2;                                                          \
  }                                                                    \
  return 0;

static inline unsigned nblk(int64_t n, int t) { return (unsigned)ceil_div(n, t); }
#include "variants.cuh"
static inline int act_type(const Handle* h) { return h->cfg.precision == DRS_PREC_FP32 ? ET_F32 : (h->cfg.precision == DRS_PREC_F16 ? ET_F16 : ET_BF16); }

// ------------------------------------------------------------------------------------------------
// network description (SURVEY.md Appendix A)
// ------------------------------------------------------------------------------------------------
struct ConvSpec { int k, rate, co; };
static void build_net(NetDesc& n, const drs_config& cfg) {
  static const ConvSpec d6[] = {{5, 1, 64}, {5, 1, 64}, {4, 2, 128}, {4, 2, 128}, {3, 4, 256}, {3, 4, 256}};
  static const ConvSpec d6p[] = {{5, 1, 64}, {5, 2, 64}, {4, 3, 128}, {4, 4, 128}, {3, 5, 256}, {3, 6, 256}};
  static const ConvSpec dd6[] = {{5, 1, 32}, {5, 2, 32}, {4, 3, 64}, {4, 4, 64}, {3, 5, 128}, {3, 6, 128}};
  static const ConvSpec d8p[] = {{5, 1, 64}, {5, 2, 64}, {4, 3, 128}, {4, 4, 128}, {3, 5, 192}, {3, 6, 192}, {3, 7, 256}, {3, 8, 256}};
  static const ConvSpec r6[] = {{5, 1, 64}, {5, 2, 64}, {4, 3, 128}, {4, 4, 128}, {3, 5, 256}, {3, 6, 256}};
  static const ConvSpec r6s[] = {{5, 1, 64}, {5, 2, 64}, {4, 3, 64}, {4, 4, 128}, {3, 5, 128}, {3, 6, 128}};
  static const ConvSpec r6n[] = {{5, 1, 64}, {5, 1, 64}, {4, 1, 128}, {4, 1, 128}, {3, 1, 256}, {3, 1, 256}};
  static const ConvSpec r1[] = {{5, 1, 64}, {5, 1, 64}, {4, 1, 128}, {4, 1, 128}, {3, 1, 256}, {3, 1, 256}};    // coffee:788-813
  static const ConvSpec vr[] = {{5, 1, 64}, {5, 2, 64}, {4, 4, 128}, {4, 1, 128}, {3, 2, 256}, {3, 4, 256}};    // coffee:816-841
  static const ConvSpec old3[] = {{5, 1, 64}, {4, 2, 128}, {3, 4, 256}};                                         // contest:574-603
  static const int old3_scope[] = {1, 3, 5};        // the reference kept the scope numbers of the layers it commented out
  const int* scope_no = nullptr;
  const ConvSpec* sp = nullptr;
  int L = 0;
  n.net_type = cfg.net_type;
  n.channels = cfg.channels;
  n.classes = cfg.num_classes;
  n.pool = n.dense = false;
  n.squeeze = false;
  n.se.clear();
  const char* prefix = "conv";
  switch (cfg.net_type) {
    case DRS_NET_DILATED6: sp = d6; L = 6; n.act = ACT_RELU; if (cfg.isprs_scopes) prefix = "main_conv"; break;
    case DRS_NET_DILATED6_POOLING: sp = d6p; L = 6; n.act = ACT_LRELU; n.pool = true; break;
    case DRS_NET_DENSE_DILATED6: sp = dd6; L = 6; n.act = ACT_RELU; n.dense = true; break;
    case DRS_NET_DILATED8_POOLING: sp = d8p; L = 8; n.act = ACT_LRELU; n.pool = true; break;
    case DRS_NET_RATE6: sp = r6; L = 6; n.act = ACT_RELU; break;
    case DRS_NET_RATE6_SMALL: sp = r6s; L = 6; n.act = ACT_RELU; break;
    case DRS_NET_RATE6_NODILATION: sp = r6n; L = 6; n.act = ACT_RELU; break;
    case DRS_NET_RATE1: sp = r1; L = 6; n.act = ACT_RELU; break;
    case DRS_NET_VARY_RATE: sp = vr; L = 6; n.act = ACT_RELU; break;
    case DRS_NET_ICPR_OLD: sp = old3; L = 3; n.act = ACT_RELU; scope_no = old3_scope; break;
    case DRS_NET_RATE6_AVGPOOL: sp = r6; L = 6; n.act = ACT_RELU; break;
    case DRS_NET_RATE6_SE: sp = r6; L = 6; n.act = ACT_RELU; break;
    case DRS_NET_RATE6_SQUEEZE: sp = r6; L = 1; n.act = ACT_RELU; n.squeeze = true; break;
    default: DRS_FAIL("Error! Net type not identified: %d", cfg.net_type);
  }
  DRS_CHECK(cfg.channels >= 1 && cfg.channels <= 16, "channels=%d out of range", cfg.channels);
  DRS_CHECK(cfg.num_classes >= 2 && cfg.num_classes <= MAX_CLASSES, "num_classes=%d out of range [2,%d]", cfg.num_classes, MAX_CLASSES);
  int cin = cfg.channels;
  int64_t off = 0, boff = 0;
  int feat = 0;   // dense: running width of the concat buffer
  n.convs.clear();
  for (int i = 0; i < L; ++i) {
    ConvLayer c;
    c.scope = std::string(prefix) + std::to_string(scope_no ? scope_no[i] : i + 1);
    c.k = sp[i].k; c.rate = sp[i].rate; c.ci = cin; c.co = sp[i].co;
    const int total = (c.k - 1) * c.rate;
    c.pad_b = total / 2; c.pad_a = total - c.pad_b;
    c.in_coff = 0;
    c.out_coff = n.dense ? feat : 0;
    c.w_off = off; off += (int64_t)c.k * c.k * c.ci * c.co;
    c.b_off = off; off += c.co;
    c.mm_off = boff; boff += c.co;
    c.mv_off = boff; boff += c.co;
    if (cfg.net_type == DRS_NET_RATE6_AVGPOOL && i < 5) { c.post = 1; c.post_k = i < 3 ? 5 : 7; }     // isprs:824-837
    if (cfg.net_type == DRS_NET_RATE6_SE && (i & 1)) {                                               // isprs:1042-1051
      SeBlock sb;
      sb.name = "se" + std::to_string(i / 2 + 1);
      sb.c = c.co; sb.r = c.co / 4;
      sb.w1_off = off; off += (int64_t)sb.c * sb.r;
      sb.b1_off = off; off += sb.r;
      sb.w2_off = off; off += (int64_t)sb.r * sb.c;
      sb.b2_off = off; off += sb.c;
      c.post = 2; c.se = (int)n.se.size();
      n.se.push_back(sb);
    }
    n.convs.push_back(std::move(c));
    if (n.dense) { feat += c.co; cin = feat; } else cin = c.co;
  }
  if (n.squeeze) {
    // _squeeze_conv_layer (isprs:726-742, 1068-1075): name, in, out, k_dim, kernel, rate
    struct Sq { const char* name; int in, out, kd, ks, rate; };
    static const Sq sq[] = {{"conv2", 64, 64, 32, 5, 2}, {"conv3", 64, 128, 64, 4, 3}, {"conv4", 128, 128, 64, 4, 4},
                            {"conv5", 128, 256, 64, 3, 5}, {"conv6", 256, 256, 128, 3, 6}};
    int prev_group = 0, prev_cs = n.convs[0].co;
    for (const Sq& q : sq) {
      const int s1 = (int)n.convs.size();
      for (int part = 0; part < 3; ++part) {
        ConvLayer c;
        c.scope = std::string(q.name) + (part == 0 ? "_s1" : part == 1 ? "_s2_1" : "_s2_2");
        c.k = part == 2 ? q.ks : 1;
        c.rate = q.rate;
        c.ci = part == 0 ? q.in : q.kd;
        c.co = part == 0 ? q.kd : q.out / 2;
        const int total = (c.k - 1) * c.rate;
        c.pad_b = total / 2; c.pad_a = total - c.pad_b;
        c.in_coff = 0;
        c.in_group = part == 0 ? prev_group : s1;
        c.in_cs = part == 0 ? prev_cs : q.kd;
        c.out_group = part == 0 ? s1 : s1 + 1;
        c.out_cs = part == 0 ? q.kd : q.out;
        c.out_coff = part == 2 ? q.out / 2 : 0;
        c.w_off = off; off += (int64_t)c.k * c.k * c.ci * c.co;
        c.b_off = off; off += c.co;
        c.mm_off = boff; boff += c.co;
        c.mv_off = boff; boff += c.co;
        n.convs.push_back(std::move(c));
      }
      prev_group = s1 + 1;
      prev_cs = q.out;
      cin = q.out;
    }
  }
  n.cls_in = cin;
  n.cls_w_off = off; off += (int64_t)cin * cfg.num_classes;
  n.cls_b_off = off; off += cfg.num_classes;
  n.n_trainable = off;
  n.n_bnstat = boff;
  n.feat_stride = 0;
  for (auto& c : n.convs) n.feat_stride = std::max(n.feat_stride, std::max(c.co, c.out_cs));
  if (n.dense) n.feat_stride = feat;
}

// ------------------------------------------------------------------------------------------------
// life cycle
// ------------------------------------------------------------------------------------------------
extern "C" const char* drs_last_error(void) { return g_drs_err; }
extern "C" int drs_version(void) { return DRS_VERSION; }

extern "C" int drs_create(drs_handle_t* out, const drs_config* cfg) {
  API_BEGIN
  DRS_CHECK(out && cfg, "drs_create: null argument");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  DRS_CHECK(e == cudaSuccess && ndev > 0, "drs_create: no CUDA device (%s); libdrs has no CPU fallback", cudaGetErrorString(e));
  DRS_CHECK(cfg->device >= 0 && cfg->device < ndev, "drs_create: device %d out of range (%d devices)", cfg->device, ndev);
  CUDA_CHECK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CUDA_CHECK(cudaGetDeviceProperties(&prop, cfg->device));
  DRS_CHECK(prop.major == 10, "drs_create: device %s is sm_%d%d; libdrs is built for sm_100a only", prop.name, prop.major, prop.minor);
  std::unique_ptr<Handle> h(new Handle());   // everything created below is released with it if a later step throws
  h->cfg = *cfg;
  h->sm_count = prop.multiProcessorCount;
  CUDA_CHECK(cudaDriverGetVersion(&h->driver_version));
  build_net(h->net, *cfg);
  h->own_stream = new_stream();
  h->stream = h->own_stream;
  const int64_t nt = h->net.n_trainable;
  h->params = DevMem<float>(nt * 4);
  h->grads = DevMem<float>((nt + 1024) * 4);
  h->moms = DevMem<float>(nt * 4);
  h->bnstat = DevMem<float>(h->net.n_bnstat * 4);
  CUDA_CHECK(cudaMemset(h->params, 0, nt * 4));
  CUDA_CHECK(cudaMemset(h->grads, 0, (nt + 1024) * 4));
  CUDA_CHECK(cudaMemset(h->moms, 0, nt * 4));
  h->is_weight = DevMem<uint8_t>(nt);
  {
    std::vector<uint8_t> isw(nt, 0);
    for (auto& c : h->net.convs)
      for (int64_t i = c.w_off; i < c.b_off; ++i) isw[i] = 1;
    for (int64_t i = h->net.cls_w_off; i < h->net.cls_b_off; ++i) isw[i] = 1;
    for (auto& sb : h->net.se) {                         // _fc_layer weights carry weight decay too (isprs:668-670)
      for (int64_t i = sb.w1_off; i < sb.b1_off; ++i) isw[i] = 1;
      for (int64_t i = sb.w2_off; i < sb.b2_off; ++i) isw[i] = 1;
    }
    CUDA_CHECK(cudaMemcpy(h->is_weight, isw.data(), nt, cudaMemcpyHostToDevice));
    // moving_mean = 0, moving_variance = 1 (Appendix B.3)
    std::vector<float> bn(h->net.n_bnstat, 0.0f);
    for (auto& c : h->net.convs)
      for (int i = 0; i < c.co; ++i) bn[c.mv_off + i] = 1.0f;
    CUDA_CHECK(cudaMemcpy(h->bnstat, bn.data(), bn.size() * 4, cudaMemcpyHostToDevice));
  }
  h->mean = DevMem<float>(h->net.n_bnstat * 4);
  h->inv_std = DevMem<float>(h->net.n_bnstat * 4);
  h->sums = DevMem<float>(2 * 512 * 4);
  h->loss_dev = DevMem<float>(16 * 4);
  h->cm_dev = DevMem<unsigned int>((MAX_CLASSES * MAX_CLASSES + 1) * 4);
  h->count_dev = DevMem<unsigned int>(16);
  CUDA_CHECK(cudaMemset(h->count_dev, 0, 16));
  h->bn_counter = h->count_dev + 2;
  h->bn_acc = DevMem<long long>((size_t)BN_ACC_REPLICAS * BN_ACC_STRIDE * 8);
  CUDA_CHECK(cudaMemset(h->bn_acc, 0, (size_t)BN_ACC_REPLICAS * BN_ACC_STRIDE * 8));
  h->ones = DevMem<float>(512 * 4);
  h->zeros = DevMem<float>(512 * 4);
  CUDA_CHECK(cudaMemset(h->zeros, 0, 512 * 4));
  {
    std::vector<float> o(512, 1.0f);
    CUDA_CHECK(cudaMemcpy(h->ones, o.data(), 512 * 4, cudaMemcpyHostToDevice));
  }
  memset(&h->table, 0, sizeof(h->table));
  h->diag_host = new_pinned<uint32_t>(64, cudaHostAllocMapped);
  memset(h->diag_host, 0, 64);
  CUDA_CHECK(cudaHostGetDevicePointer((void**)&h->diag_dev, h->diag_host, 0));
  // driver entry points for tensor-map encoding (no link-time dependency on libcuda)
  {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    DRS_CHECK(fn && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    h->encodeTiled = (PFN_encodeTiled)fn;
    fn = nullptr;
    CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &qres));
    DRS_CHECK(fn && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeIm2col not available");
    h->encodeIm2col = (PFN_encodeIm2col)fn;
  }
  h->packed_dirty = true;
  h->eval_dirty = true;
  // whole-step CUDA graphs per (batch, patch size, buffers, lr): on by default (DRS_GRAPHS=0 turns them off); the drop-in
  // loops pre-capture the patch-size interval at start-up (drs_train_prepare), like TF building its graph before the loop
  h->use_graphs = getenv("DRS_GRAPHS") == nullptr || atoi(getenv("DRS_GRAPHS")) != 0;
  h->plan_stream = new_stream();
  for (int i = 0; i < 2; ++i) {
    h->plan_uploaded[i] = new_event();
    h->plan_consumed[i] = new_event();
  }
  h->result_host = new_pinned<float>((size_t)Handle::RESULT_RING * RESULT_STRIDE * 4, cudaHostAllocDefault);
  for (int i = 0; i < Handle::RESULT_RING; ++i) h->result_ev[i] = new_event();
  h->side_stream = new_stream();
  h->comm_stream = new_stream();
  h->ev_bucket_ready = new_event();
  h->ev_x8 = new_event();
  h->ev_bucket_done = new_event();
  for (int i = 0; i < 2; ++i) {
    h->ev_dz[i] = new_event();
    h->ev_wgrad[i] = new_event();
  }
  *out = h.release();
  API_END
}

// Everything the handle holds is released by its members' destructors, once no stream has work left that uses it.
extern "C" int drs_destroy(drs_handle_t h) {
  API_BEGIN
  if (!h) return 0;
  cudaSetDevice(h->cfg.device);
  cudaStreamSynchronize(h->stream);
  for (cudaStream_t s : {h->own_stream.get(), h->side_stream.get(), h->comm_stream.get(), h->copy_stream.get(),
                         h->plan_stream.get(), h->lane.stream.get()})
    if (s) cudaStreamSynchronize(s);
  if (h->nccl) drs_comm_destroy(h);
  delete h;
  API_END
}

extern "C" int drs_set_stream(drs_handle_t h, void* s) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  // (void*)-1 selects the handle's own non-blocking stream; any other value is a cudaStream_t, 0 = the legacy default stream
  h->stream = (s == (void*)(intptr_t)-1) ? h->own_stream : (cudaStream_t)s;
  API_END
}
extern "C" int drs_synchronize(drs_handle_t h) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  cudaError_t e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) {
    DRS_FAIL("stream failed: %s (diag %08x blk %u thr %u par %u)", cudaGetErrorString(e), h->diag_host[0], h->diag_host[1],
             h->diag_host[2], h->diag_host[3]);
  }
  API_END
}
extern "C" int64_t drs_launch_count(drs_handle_t h) { return h ? h->launches : -1; }

// ------------------------------------------------------------------------------------------------
// variables
// ------------------------------------------------------------------------------------------------
struct VarRef { float* ptr; int64_t count; int kind; };  // kind 0 device float, 1 global_step
static bool find_var(Handle* h, const std::string& name, VarRef& r, bool grad = false) {
  float* base = grad ? h->grads : h->params;
  auto slot = [&](const std::string& nm, float* p, float* m, int64_t cnt) -> bool {
    if (name == nm) { r = {p, cnt, 0}; return true; }
    if (!grad && m && name == nm + "/Momentum") { r = {m, cnt, 0}; return true; }
    return false;
  };
  for (auto& c : h->net.convs) {
    const int64_t wc = (int64_t)c.k * c.k * c.ci * c.co;
    if (slot(c.scope + "/weights", base + c.w_off, h->moms + c.w_off, wc)) return true;
    if (slot(c.scope + "/biases", base + c.b_off, h->moms + c.b_off, c.co)) return true;
    if (!grad) {
      if (slot(c.scope + "/moving_mean", h->bnstat + c.mm_off, nullptr, c.co)) return true;
      if (slot(c.scope + "/moving_variance", h->bnstat + c.mv_off, nullptr, c.co)) return true;
    }
  }
  for (auto& sb : h->net.se) {
    if (slot(sb.name + "_fc1/weights", base + sb.w1_off, h->moms + sb.w1_off, (int64_t)sb.c * sb.r)) return true;
    if (slot(sb.name + "_fc1/biases", base + sb.b1_off, h->moms + sb.b1_off, sb.r)) return true;
    if (slot(sb.name + "_fc2/weights", base + sb.w2_off, h->moms + sb.w2_off, (int64_t)sb.r * sb.c)) return true;
    if (slot(sb.name + "_fc2/biases", base + sb.b2_off, h->moms + sb.b2_off, sb.c)) return true;
  }
  if (slot("conv_classifier/weights", base + h->net.cls_w_off, h->moms + h->net.cls_w_off, (int64_t)h->net.cls_in * h->net.classes)) return true;
  if (slot("conv_classifier/biases", base + h->net.cls_b_off, h->moms + h->net.cls_b_off, h->net.classes)) return true;
  if (!grad && (name == "global_step" || name == "main_global_step")) { r = {nullptr, 1, 1}; return true; }
  return false;
}
static void list_vars(Handle* h, std::vector<std::pair<std::string, int64_t>>& v) {
  for (auto& c : h->net.convs) {
    const int64_t wc = (int64_t)c.k * c.k * c.ci * c.co;
    v.push_back({c.scope + "/weights", wc});
    v.push_back({c.scope + "/biases", c.co});
    v.push_back({c.scope + "/moving_mean", c.co});
    v.push_back({c.scope + "/moving_variance", c.co});
    v.push_back({c.scope + "/weights/Momentum", wc});
    v.push_back({c.scope + "/biases/Momentum", c.co});
  }
  for (auto& sb : h->net.se) {
    const std::pair<std::string, int64_t> vs[4] = {{sb.name + "_fc1/weights", (int64_t)sb.c * sb.r}, {sb.name + "_fc1/biases", sb.r},
                                                    {sb.name + "_fc2/weights", (int64_t)sb.r * sb.c}, {sb.name + "_fc2/biases", sb.c}};
    for (auto& pr : vs) v.push_back(pr);
    for (auto& pr : vs) v.push_back({pr.first + "/Momentum", pr.second});
  }
  v.push_back({"conv_classifier/weights", (int64_t)h->net.cls_in * h->net.classes});
  v.push_back({"conv_classifier/biases", h->net.classes});
  v.push_back({"conv_classifier/weights/Momentum", (int64_t)h->net.cls_in * h->net.classes});
  v.push_back({"conv_classifier/biases/Momentum", h->net.classes});
  v.push_back({"global_step", 1});
}
extern "C" int drs_num_variables(drs_handle_t h) {
  if (!h) return -1;
  std::vector<std::pair<std::string, int64_t>> v;
  list_vars(h, v);
  return (int)v.size();
}
extern "C" int drs_variable_name(drs_handle_t h, int index, char* name_out, int cap, int64_t* count_out) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  std::vector<std::pair<std::string, int64_t>> v;
  list_vars(h, v);
  DRS_CHECK(index >= 0 && index < (int)v.size(), "variable index %d out of range", index);
  if (name_out && cap > 0) snprintf(name_out, cap, "%s", v[index].first.c_str());
  if (count_out) *count_out = v[index].second;
  API_END
}
extern "C" int drs_set_variable(drs_handle_t h, const char* name, const float* data, int64_t count) {
  API_BEGIN
  DRS_CHECK(h && name && data, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  VarRef r;
  DRS_CHECK(find_var(h, name, r), "unknown variable '%s'", name);
  DRS_CHECK(r.count == count, "variable '%s' has %lld elements, got %lld", name, (long long)r.count, (long long)count);
  if (r.kind == 1) { h->global_step = (int64_t)data[0]; return 0; }
  CUDA_CHECK(cudaMemcpyAsync(r.ptr, data, count * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  h->packed_dirty = true;
  h->eval_dirty = true;
  API_END
}
extern "C" int drs_get_variable(drs_handle_t h, const char* name, float* data, int64_t count) {
  API_BEGIN
  DRS_CHECK(h && name && data, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  VarRef r;
  DRS_CHECK(find_var(h, name, r), "unknown variable '%s'", name);
  DRS_CHECK(r.count == count, "variable '%s' has %lld elements, got %lld", name, (long long)r.count, (long long)count);
  if (r.kind == 1) { data[0] = (float)h->global_step; return 0; }
  CUDA_CHECK(cudaMemcpyAsync(data, r.ptr, count * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  API_END
}
extern "C" int drs_get_gradient(drs_handle_t h, const char* name, float* data, int64_t count) {
  API_BEGIN
  DRS_CHECK(h && name && data, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  VarRef r;
  DRS_CHECK(find_var(h, name, r, true), "unknown trainable variable '%s'", name);
  DRS_CHECK(r.count == count, "variable '%s' has %lld elements, got %lld", name, (long long)r.count, (long long)count);
  CUDA_CHECK(cudaMemcpyAsync(data, r.ptr, count * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  API_END
}

// ------------------------------------------------------------------------------------------------
// checkpoints: tf.train.Saver.save / restore (isprs:1693-1717, 1797-1802) as an uncompressed .npz keyed by the TF variable
// names ('/' written as '__', which is what numpy.savez keyword arguments allow), shapes as TF holds them (HWIO filters)
// ------------------------------------------------------------------------------------------------
static std::vector<int64_t> var_shape(Handle* h, const std::string& full, int64_t count) {
  std::string name = full;
  const std::string mom = "/Momentum";
  if (name.size() > mom.size() && name.compare(name.size() - mom.size(), mom.size(), mom) == 0) name.resize(name.size() - mom.size());
  for (auto& c : h->net.convs)
    if (name == c.scope + "/weights") return {c.k, c.k, c.ci, c.co};
  for (auto& sb : h->net.se) {
    if (name == sb.name + "_fc1/weights") return {sb.c, sb.r};
    if (name == sb.name + "_fc2/weights") return {sb.r, sb.c};
  }
  if (name == "conv_classifier/weights") return {1, 1, h->net.cls_in, h->net.classes};
  return {count};
}
static std::string npz_key(std::string name) {
  for (size_t i = 0; (i = name.find('/', i)) != std::string::npos;) name.replace(i, 1, "__");
  return name;
}
static std::string npz_unkey(std::string key) {
  for (size_t i = 0; (i = key.find("__", i)) != std::string::npos; ++i) key.replace(i, 2, "/");
  return key;
}

extern "C" int drs_save(drs_handle_t h, const char* path) {
  API_BEGIN
  DRS_CHECK(h && path, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  std::vector<std::pair<std::string, int64_t>> v;
  list_vars(h, v);
  std::vector<drs_npz::Array> arrays(v.size());
  for (size_t i = 0; i < v.size(); ++i) {
    VarRef r;
    DRS_CHECK(find_var(h, v[i].first, r), "unknown variable '%s'", v[i].first.c_str());
    arrays[i].name = npz_key(v[i].first);
    arrays[i].shape = var_shape(h, v[i].first, r.count);
    arrays[i].data.resize((size_t)r.count);
    if (r.kind == 1) arrays[i].data[0] = (float)h->global_step;
    else CUDA_CHECK(cudaMemcpyAsync(arrays[i].data.data(), r.ptr, r.count * 4, cudaMemcpyDeviceToHost, h->stream));
  }
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  const std::string e = drs_npz::write(path, arrays);
  DRS_CHECK(e.empty(), "%s", e.c_str());
  API_END
}

extern "C" int drs_load(drs_handle_t h, const char* path) {
  API_BEGIN
  DRS_CHECK(h && path, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  std::vector<drs_npz::Array> arrays;
  const std::string e = drs_npz::read(path, arrays);
  DRS_CHECK(e.empty(), "%s", e.c_str());
  // validate everything before touching the model: a checkpoint of another net must not be applied half-way
  for (auto& a : arrays) {
    VarRef r;
    const std::string name = npz_unkey(a.name);
    DRS_CHECK(find_var(h, name, r), "checkpoint '%s': unknown variable '%s'", path, name.c_str());
    DRS_CHECK(r.count == a.count(), "checkpoint '%s': variable '%s' has %lld elements, the model expects %lld", path, name.c_str(),
              (long long)a.count(), (long long)r.count);
  }
  for (auto& a : arrays) {
    VarRef r;
    find_var(h, npz_unkey(a.name), r);
    if (r.kind == 1) { h->global_step = (int64_t)a.data[0]; continue; }
    CUDA_CHECK(cudaMemcpyAsync(r.ptr, a.data.data(), r.count * 4, cudaMemcpyHostToDevice, h->stream));
  }
  CUDA_CHECK(cudaStreamSynchronize(h->stream));      // the host arrays die with this scope
  h->packed_dirty = true;
  h->eval_dirty = true;
  API_END
}

// the container alone, no handle and no device: inspection / conversion tools and the CPU tests
extern "C" int drs_npz_write(const char* path, int32_t n, const char* const* names, const float* const* data, const int32_t* ndim,
                             const int64_t* dims) {
  API_BEGIN
  DRS_CHECK(path && n >= 0 && (n == 0 || (names && data && ndim && dims)), "bad argument");
  std::vector<drs_npz::Array> arrays((size_t)n);
  for (int i = 0; i < n; ++i) {
    DRS_CHECK(names[i] && data[i] && ndim[i] >= 0 && ndim[i] <= 4, "array %d: bad argument", i);
    arrays[i].name = names[i];
    arrays[i].shape.assign(dims + 4 * i, dims + 4 * i + ndim[i]);
    for (int64_t d : arrays[i].shape) DRS_CHECK(d >= 0, "array %d: negative dimension", i);
    arrays[i].data.assign(data[i], data[i] + arrays[i].count());
  }
  const std::string e = drs_npz::write(path, arrays);
  DRS_CHECK(e.empty(), "%s", e.c_str());
  API_END
}
extern "C" int drs_npz_entry(const char* path, int32_t index, char* name_out, int32_t name_cap, int32_t* ndim_out, int64_t* dims_out,
                             int64_t* count_out, int32_t* total_out) {
  API_BEGIN
  DRS_CHECK(path, "null argument");
  std::vector<drs_npz::Array> arrays;
  const std::string e = drs_npz::read(path, arrays);
  DRS_CHECK(e.empty(), "%s", e.c_str());
  if (total_out) *total_out = (int32_t)arrays.size();
  if (index < 0) return 0;                                  // count only
  DRS_CHECK(index < (int)arrays.size(), "entry %d out of range (%d arrays)", index, (int)arrays.size());
  const drs_npz::Array& a = arrays[index];
  DRS_CHECK(a.shape.size() <= 4, "array '%s' has %d dimensions", a.name.c_str(), (int)a.shape.size());
  if (name_out && name_cap > 0) snprintf(name_out, name_cap, "%s", a.name.c_str());
  if (ndim_out) *ndim_out = (int32_t)a.shape.size();
  if (dims_out) for (size_t i = 0; i < a.shape.size(); ++i) dims_out[i] = a.shape[i];
  if (count_out) *count_out = a.count();
  API_END
}
extern "C" int drs_npz_read(const char* path, const char* name, float* out, int64_t count) {
  API_BEGIN
  DRS_CHECK(path && name && out, "null argument");
  std::vector<drs_npz::Array> arrays;
  const std::string e = drs_npz::read(path, arrays);
  DRS_CHECK(e.empty(), "%s", e.c_str());
  for (auto& a : arrays)
    if (a.name == name) {
      DRS_CHECK(a.count() == count, "array '%s' has %lld elements, got room for %lld", name, (long long)a.count(), (long long)count);
      memcpy(out, a.data.data(), (size_t)count * 4);
      return 0;
    }
  DRS_FAIL("checkpoint '%s' has no array '%s'", path, name);
  API_END
}

// host-only: the units CTA `block` of a `grid`-CTA conv_tc launch works on, in order (ConvSched is the kernel's own code)
extern "C" int drs_debug_conv_schedule(int32_t num_units, int32_t mt, int32_t grid, int32_t block, int32_t* units_out,
                                       uint8_t* pair_out, int32_t cap, int32_t* n_out) {
  API_BEGIN
  DRS_CHECK(num_units >= 0 && (mt == 1 || mt == 2) && grid >= 1 && block >= 0 && block < grid && n_out, "bad argument");
  const ConvSched sc(num_units, mt, grid, block);
  *n_out = sc.iters;
  for (int i = 0; i < sc.iters && i < cap; ++i) {
    bool two;
    const int u = sc.unit(i, two);
    if (units_out) units_out[i] = u;
    if (pair_out) pair_out[i] = two ? 1 : 0;
  }
  API_END
}

extern "C" int drs_set_ignore_label(drs_handle_t h, int32_t label) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  h->ignore_label = label;
  API_END
}

extern "C" int drs_set_allreduce(drs_handle_t h, drs_allreduce_fn fn, void* user, int32_t world, int32_t sync_bn) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  h->allreduce = fn;
  h->allreduce_user = user;
  h->world = fn ? (world > 0 ? world : 1) : 1;
  h->sync_bn = fn ? sync_bn : 0;
  API_END
}
#include "drs_comm.cuh"

// ------------------------------------------------------------------------------------------------
// packed operands / folded BN refresh (after set_variable or an optimizer step)
// ------------------------------------------------------------------------------------------------
// One launch repacks the operand matrices of every tensor-core layer after set_variable / an optimizer step:
//   kind 0  fprop operand  Wf[co][tap*ci + c]            = W[tap][c][co]
//   kind 1  dgrad operand  Wd[c][tap'*co + o]            = W[taps-1-tap'][c][o]
//   kind 2  dgrad operand of the fp32 CUDA-core path  [tap'*co + o][c]
struct RepackSeg {
  const float* w;
  void* out;
  int taps, ci, co, kind;
  long long start;
};
struct RepackTable {
  RepackSeg seg[40];       // up to 20 tensor-core layers (the squeeze net has 15), fprop + dgrad operand each
  int n, etype;
  long long total;
};
__global__ void repack_kernel(const __grid_constant__ RepackTable t) {
  pdl_sync();
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= t.total) return;
  int si = 0;
  while (si + 1 < t.n && gid >= t.seg[si + 1].start) ++si;
  const RepackSeg& s = t.seg[si];
  const long long i = gid - s.start;
  float v;
  if (s.kind == 0) {
    const int o = (int)(i / ((long long)s.taps * s.ci));
    const int kk = (int)(i - (long long)o * s.taps * s.ci);
    v = s.w[(long long)kk * s.co + o];
  } else if (s.kind == 1) {
    const int c = (int)(i / ((long long)s.taps * s.co));
    const int r = (int)(i - (long long)c * s.taps * s.co);
    const int tp = r / s.co, o = r - tp * s.co;
    v = s.w[((long long)(s.taps - 1 - tp) * s.ci + c) * s.co + o];
  } else {
    const int c = (int)(i % s.ci);
    const int r = (int)(i / s.ci);
    const int tp = r / s.co, o = r - tp * s.co;
    v = s.w[((long long)(s.taps - 1 - tp) * s.ci + c) * s.co + o];
  }
  if (s.kind == 2 || t.etype == ET_F32) reinterpret_cast<float*>(s.out)[i] = v;
  else if (t.etype == ET_F16) reinterpret_cast<__half*>(s.out)[i] = __float2half_rn(v);
  else reinterpret_cast<__nv_bfloat16*>(s.out)[i] = __float2bfloat16_rn(v);
}

// one filter's operand matrix of the given kind, exactly as refresh_packed builds a layer's
static void repack_filter(Handle* h, const float* w, void* out, int taps, int ci, int co, int kind, int etype) {
  RepackTable t;
  memset(&t, 0, sizeof(t));
  t.etype = etype;
  t.seg[t.n++] = RepackSeg{w, out, taps, ci, co, kind, 0};
  t.total = (long long)taps * ci * co;
  repack_kernel<<<nblk(t.total, 256), 256, 0, h->stream>>>(t);
  LAUNCH_CHECK(h);
}

// conv1's tensor-core operand (conv1_tc.cuh): the HWIO filter in core-matrix order, C1_SLOTS * co * 8 16-bit elements
template <typename TA>
static void pack_conv1(Handle* h, const float* w, void* out, int ci, int co) {
  launch_pdl(h, pack_conv1_kernel<TA>, dim3(nblk(C1_SLOTS * co * 8, 256)), dim3(256), 0, w, (TA*)out, ci, co);
  LAUNCH_CHECK(h);
}

// training needs only the layer operands; inference additionally the folded eval-mode BN and conv1's tensor-core operand
static void refresh_packed(Handle* h, bool training) {
  const int et = act_type(h);
  if (h->packed_dirty) {
    RepackTable t;
    memset(&t, 0, sizeof(t));
    t.etype = et;
    long long off = 0;
    for (size_t l = 1; l < h->net.convs.size(); ++l) {
      ConvLayer& c = h->net.convs[l];
      const int taps = c.k * c.k;
      const long long n = (long long)taps * c.ci * c.co;
      const size_t es = et == ET_F32 ? 4 : 2;
      if (et != ET_F32) {
        c.w_fprop.grow(n * es, n * es);
        t.seg[t.n++] = RepackSeg{h->params + c.w_off, c.w_fprop, taps, c.ci, c.co, 0, off};
        off += n;
      }
      c.w_dgrad.grow(n * es, n * es);
      t.seg[t.n++] = RepackSeg{h->params + c.w_off, c.w_dgrad, taps, c.ci, c.co, et == ET_F32 ? 2 : 1, off};
      off += n;
    }
    t.total = off;
    if (off > 0) {
      repack_kernel<<<nblk(off, 256), 256, 0, h->stream>>>(t);
      LAUNCH_CHECK(h);
    }
    h->packed_dirty = false;
  }
  if (!training && h->eval_dirty) {
    for (size_t l = 0; l < h->net.convs.size(); ++l) {
      ConvLayer& c = h->net.convs[l];
      c.fold_scale.grow(c.co * 4, c.co * 4);
      c.fold_shift.grow(c.co * 4, c.co * 4);
      fold_bn_kernel<<<nblk(c.co, 128), 128, 0, h->stream>>>(h->params + c.b_off, h->bnstat + c.mm_off, h->bnstat + c.mv_off,
                                                              h->cfg.bn_eps, c.fold_scale, c.fold_shift, c.co);
      LAUNCH_CHECK(h);
      // 16-bit inference runs conv1 on the tensor cores (conv1_tc.cuh) from a core-matrix-ordered operand; training and the
      // fp32 mode run it on the CUDA-core kernel straight from the HWIO weights
      if (l == 0 && et != ET_F32 && conv1_tc_supported(c.k, c.rate, c.ci, c.co)) {
        const size_t bytes = (size_t)C1_SLOTS * c.co * 8 * 2;
        c.w_fprop.grow(bytes, bytes);
        if (et == ET_F16) pack_conv1<__half>(h, h->params + c.w_off, c.w_fprop, c.ci, c.co);
        else pack_conv1<__nv_bfloat16>(h, h->params + c.w_off, c.w_fprop, c.ci, c.co);
      }
    }
    h->eval_dirty = false;
  }
}

// ------------------------------------------------------------------------------------------------
// one convolution, any precision
// ------------------------------------------------------------------------------------------------
struct ActBuf { void* p; int cs; int co; };   // pointer, channel stride, channel offset

// the shape of one convolution outside a network (the unit-test entry points), SAME-padded as build_net pads a layer
static ConvLayer conv_shape(int k, int rate, int ci, int co) {
  ConvLayer c;
  c.k = k; c.rate = rate; c.ci = ci; c.co = co;
  c.pad_b = (k - 1) * rate / 2; c.pad_a = (k - 1) * rate - c.pad_b;
  return c;
}

static void prof_begin(Handle* h, cudaEvent_t* a, cudaEvent_t* b) {
  if (!h->time_convs) return;
  if (h->capturing) {
    h->capturing->events.emplace_back(new_event(cudaEventDefault), new_event(cudaEventDefault));
    *a = h->capturing->events.back().first;
    *b = h->capturing->events.back().second;
    CUDA_CHECK(cudaEventRecordWithFlags(*a, h->stream, cudaEventRecordExternal));
    return;
  }
  if (h->conv_events_used == h->conv_events.size())
    h->conv_events.emplace_back(new_event(cudaEventDefault), new_event(cudaEventDefault));
  *a = h->conv_events[h->conv_events_used].first;
  *b = h->conv_events[h->conv_events_used].second;
  h->conv_events_used++;
  CUDA_CHECK(cudaEventRecord(*a, h->stream));
}
static void prof_end(Handle* h, cudaEvent_t b) {
  if (!h->time_convs) return;
  if (h->capturing) { CUDA_CHECK(cudaEventRecordWithFlags(b, h->stream, cudaEventRecordExternal)); return; }
  CUDA_CHECK(cudaEventRecord(b, h->stream));
}

// generic conv over activation type TA.  w_simt: HWIO fp32 [k*k*ci][co]; w_tc: packed [co][k*k*ci].
template <typename TA>
static void run_conv(Handle* h, const ActBuf& in, int ci, const float* w_simt, const void* w_tc, const ActBuf& out, int co,
                     int B, int crop, int k, int rate, int pad_b, const float* scale, const float* shift, int act,
                     const BnFinish* stats = nullptr) {
  if (ElemTag<TA>::v == ET_F32) {
    launch_conv_simt<TA, TA>(h, (const TA*)in.p, in.cs, in.co, ci, w_simt, (TA*)out.p, out.cs, out.co, co, B, crop, k, rate,
                             pad_b, scale, shift, act);
    return;
  }
  cudaEvent_t ea = nullptr, eb = nullptr;
  prof_begin(h, &ea, &eb);
  // tensor-core path; N > 256 is split into equal column tiles
  int nsplit = 1;
  while (co / nsplit > 256 || (co % nsplit) != 0 || ((co / nsplit) % 32) != 0) {
    ++nsplit;
    DRS_CHECK(nsplit <= 8, "cannot tile N=%d", co);
  }
  DRS_CHECK(!stats || nsplit == 1, "fused BN statistics need a single N tile (Co=%d)", co);
  const int nt = co / nsplit;
  for (int s = 0; s < nsplit; ++s) {
    ConvTcArgs a;
    a.in = in.p; a.in_cstride = in.cs; a.in_coff = in.co; a.ci = ci;
    a.w = (const char*)w_tc + (size_t)s * nt * k * k * ci * 2;
    a.out = out.p; a.out_cstride = out.cs; a.out_coff = out.co + s * nt; a.co = nt;
    a.B = B; a.crop = crop; a.k = k; a.rate = rate; a.pad_b = pad_b;
    a.scale = scale + s * nt; a.shift = shift + s * nt; a.act = act;
    a.etype = ElemTag<TA>::v;
    a.stats = stats;
    launch_conv_tc(h, a);
  }
  prof_end(h, eb);
  h->conv_flops += 2.0 * (double)B * crop * crop * k * k * ci * co;
  h->conv_launches += nsplit;
}

// conv1 on the tensor cores (conv1_tc.cuh) for the shapes conv1_tc_supported accepts, in 16-bit: the fp32 input [M, ci] padded
// to 8 channels and rounded into x8 (pad_cast8_kernel), then the 25-tap kernel from the filter pack_conv1 packed into wpack.
// The inference forward, the training forward and drs_debug_conv all run conv1 through here.  `on_x8` runs between the two
// launches (the training forward builds conv1's im2col matrix from x8 there).  `timed`: the launch counts as one of the
// convolutions of the per-convolution profile (inference; the training profile covers the conv_tc and wgrad_tc kernels).
template <typename TA>
static void conv1_tc_forward(Handle* h, const float* x32, int ci, TA* x8, const void* wpack, const ActBuf& out, int co, int B, int crop,
                             const float* scale, const float* shift, int act, const BnFinish* stats, bool timed,
                             const std::function<void()>& on_x8 = nullptr) {
  const int64_t M = (int64_t)B * crop * crop;
  launch_pdl(h, pad_cast8_kernel<TA>, dim3(nblk(M, 256)), dim3(256), 0, x32, x8, ci, M);
  LAUNCH_CHECK(h);
  if (on_x8) on_x8();
  cudaEvent_t ea = nullptr, eb = nullptr;
  if (timed) prof_begin(h, &ea, &eb);
  Conv1TcArgs a;
  a.x8 = x8; a.wpack = wpack; a.out = out.p; a.out_cstride = out.cs; a.out_coff = out.co; a.co = co;
  a.B = B; a.crop = crop; a.scale = scale; a.shift = shift; a.act = act; a.etype = ElemTag<TA>::v;
  a.stats = stats;
  launch_conv1_tc(h, a);
  if (!timed) return;
  prof_end(h, eb);
  h->conv_flops += 2.0 * (double)M * 25 * ci * co;   // algorithmic FLOPs: the real input channels
  h->conv_launches += 1;
}

// DRS_DEBUG_KEEP=1: an fp32 copy of a layer's tensor, registered as the activation tap `name` (the inference forward's
// feature buffers rotate, and the training step's buffers are reused, so a tap of the buffer itself would not survive)
template <typename T>
static void debug_keep(Handle* h, const std::string& name, const T* ptr, int cs, int co, int C, int64_t M) {
  if (!h->debug_keep) return;
  h->keep.emplace_back(M * C * 4);
  float* buf = h->keep.back();
  slice_to_f32_kernel<T><<<nblk(M * C, 256), 256, 0, h->stream>>>(ptr, cs, co, C, M, buf);
  LAUNCH_CHECK(h);
  h->taps[name] = {buf, ET_F32, C, 0, C, M};
}
static void debug_keep_reset(Handle* h) {
  h->debug_keep = getenv("DRS_DEBUG_KEEP") != nullptr;
  if (h->keep.empty()) return;
  cudaStreamSynchronize(h->stream);
  h->keep.clear();
}

// ------------------------------------------------------------------------------------------------
// inference forward (eval-mode BN folded into the conv epilogue)
// ------------------------------------------------------------------------------------------------
// Every buffer the inference forward takes from the arena, in one place (see TrainWs in drs_train.cuh)
template <typename TA>
struct EvalWs {
  TA* bufs[3] = {nullptr, nullptr, nullptr};   // feature buffers (dense nets: one concatenated buffer)
  float* logits = nullptr;                     // when the caller passes no buffer
  float* se = nullptr;                         // SE gate scratch of the widest gate: sums, means, gate, hidden
  TA* x8 = nullptr;                            // conv1 on the tensor cores: input padded to 8 channels

  void layout(const Handle* h, WsAlloc& a, int B, int crop) {
    const NetDesc& n = h->net;
    const int64_t M = (int64_t)B * crop * crop;
    for (int i = 0; i < (n.dense ? 1 : 3); ++i) bufs[i] = a.take<TA>((size_t)M * n.feat_stride * sizeof(TA));
    logits = a.take<float>((size_t)M * n.classes * 4);
    size_t se_floats = 0;
    for (auto& sb : n.se) se_floats = std::max(se_floats, (size_t)B * (3 * sb.c + sb.r));
    if (se_floats) se = a.take<float>(se_floats * 4);
    const ConvLayer& c0 = n.convs[0];
    if (ElemTag<TA>::v != ET_F32 && conv1_tc_supported(c0.k, c0.rate, c0.ci, c0.co)) x8 = a.take<TA>((size_t)M * 8 * sizeof(TA));
  }
};

// the bytes workspace layout W takes from the arena: a counting run of W::layout
template <typename W>
static size_t layout_bytes(const Handle* h, int B, int crop) {
  WsAlloc count;
  W().layout(h, count, B, crop);
  return count.used;
}
static size_t eval_arena_bytes(const Handle* h, int B, int crop) {
  switch (act_type(h)) {
    case ET_F32: return layout_bytes<EvalWs<float>>(h, B, crop);
    case ET_F16: return layout_bytes<EvalWs<__half>>(h, B, crop);
    default: return layout_bytes<EvalWs<__nv_bfloat16>>(h, B, crop);
  }
}

template <typename TA>
static void forward_eval_t(Handle* h, const float* x_dev, int B, int crop, float* logits_dev, uint8_t* pred_dev) {
  NetDesc& n = h->net;
  const int64_t M = (int64_t)B * crop * crop;
  refresh_packed(h, false);
  const int fs = n.feat_stride;
  ensure_arena(h, layout_bytes<EvalWs<TA>>(h, B, crop));
  h->arena->reset();
  EvalWs<TA> ws;
  {
    WsAlloc carve{h->arena};
    ws.layout(h, carve, B, crop);
  }
  float* logits = logits_dev ? logits_dev : ws.logits;
  h->taps.clear();
  debug_keep_reset(h);

  ActBuf cur{nullptr, 0, 0};
  int xi = 0;   // index of the buffer holding the current input (non-dense)
  int sq_s = 0, sq_c = 0;   // squeeze modules: buffers of the squeeze output S and of the concatenated module output
  for (size_t l = 0; l < n.convs.size(); ++l) {
    ConvLayer& c = n.convs[l];
    ActBuf out;
    const int sq_part = (n.squeeze && l >= 1) ? (int)((l - 1) % 3) : -1;    // 0: _s1, 1: _s2_1, 2: _s2_2 (isprs:726-742)
    if (n.dense) out = {ws.bufs[0], fs, c.out_coff};
    else if (sq_part == 0) { sq_s = (xi + 1) % 3; sq_c = (xi + 2) % 3; out = {ws.bufs[sq_s], fs, 0}; }
    else if (sq_part >= 1) { cur = {ws.bufs[sq_s], fs, 0}; out = {ws.bufs[sq_c], fs, c.out_coff}; }
    else out = {ws.bufs[(xi + 1) % 3], fs, 0};
    if (l == 0 && ws.x8 && c.w_fprop) {
      conv1_tc_forward<TA>(h, x_dev, c.ci, ws.x8, c.w_fprop, out, c.co, B, crop, c.fold_scale, c.fold_shift, n.act, nullptr, true);
    } else if (l == 0) {
      launch_conv_simt<float, TA>(h, x_dev, n.channels, 0, n.channels, h->params + c.w_off, (TA*)out.p, out.cs, out.co, c.co,
                                  B, crop, c.k, c.rate, c.pad_b, c.fold_scale, c.fold_shift, n.act);
    } else {
      run_conv<TA>(h, cur, c.ci, h->params + c.w_off, c.w_fprop, out, c.co, B, crop, c.k, c.rate, c.pad_b, c.fold_scale,
                   c.fold_shift, n.act);
    }
    if (n.pool && l + 1 == n.convs.size() && c.co == n.cls_in && pool_classifier_fused_supported<TA>(c.co)) {
      // last layer: pool + classifier in one pass, the pooled activations are never stored (no activation tap for this layer)
      launch_maxpool3_classifier<TA>(h, (const TA*)out.p, out.cs, out.co, c.co, B, crop, h->params + n.cls_w_off,
                                     h->params + n.cls_b_off, n.classes, logits, pred_dev);
      return;
    } else if (n.pool) {
      ActBuf pout{ws.bufs[(xi + 2) % 3], fs, 0};
      launch_maxpool3_fwd<TA>(h, (const TA*)out.p, out.cs, out.co, (TA*)pout.p, pout.cs, pout.co, nullptr, c.co, B, crop);
      cur = pout;
      xi = (xi + 2) % 3;
    } else if (c.post == 1) {
      ActBuf pout{ws.bufs[(xi + 2) % 3], fs, 0};
      launch_avgpool_fwd<TA>(h, (const TA*)out.p, out.cs, out.co, (TA*)pout.p, pout.cs, pout.co, c.co, B, crop, c.post_k);
      cur = pout;
      xi = (xi + 2) % 3;
    } else if (c.post == 2) {
      // squeeze-and-excitation gate, in place (per-image statistics: the result depends on the patch, as in the reference)
      const SeBlock& sb = n.se[c.se];
      float* sum = ws.se;
      float* sv = sum + (size_t)B * sb.c;
      float* ev = sv + (size_t)B * sb.c;
      float* hv = ev + (size_t)B * sb.c;
      se_sum_kernel<TA, 0><<<dim3(B, (unsigned)ceil_div(sb.c, 64)), 256, 0, h->stream>>>((const TA*)out.p, out.cs, out.co, nullptr, 0, 0, sb.c,
                                                                                      crop * crop, sum);
      LAUNCH_CHECK(h);
      se_fc_fwd_kernel<<<B, 256, 0, h->stream>>>(sum, 1.0f / (float)(crop * crop), h->params + sb.w1_off, h->params + sb.b1_off,
                                                h->params + sb.w2_off, h->params + sb.b2_off, sb.c, sb.r, sv, hv, ev);
      LAUNCH_CHECK(h);
      se_scale_fwd_kernel<TA><<<nblk(M * (c.co / 8), 256), 256, 0, h->stream>>>((const TA*)out.p, out.cs, out.co, ev, (TA*)out.p, out.cs, out.co,
                                                                              c.co, M, crop * crop);
      LAUNCH_CHECK(h);
      cur = out;
      xi = (xi + 1) % 3;
    } else if (sq_part >= 0) {
      if (sq_part == 0) cur = out;                       // S: read by the two expand convolutions
      else if (sq_part == 2) { cur = {ws.bufs[sq_c], fs, 0}; xi = sq_c; }    // the module's concatenated output
    } else if (n.dense) {
      cur = {ws.bufs[0], fs, 0};
    } else {
      cur = out;
      xi = (xi + 1) % 3;
    }
    // a layer that writes a channel slice of a shared buffer (dense concat, the two expand convolutions of a squeeze module)
    // is tapped at that slice; any other layer at its finished output, after the pool or gate
    const ActBuf tap = (n.dense || sq_part >= 1) ? out : cur;
    h->taps[c.scope] = {tap.p, ElemTag<TA>::v, fs, tap.co, c.co, M};
    debug_keep<TA>(h, c.scope, (const TA*)tap.p, fs, tap.co, c.co, M);     // a later layer reuses this buffer
  }
  launch_classifier_fwd<TA>(h, (const TA*)cur.p, cur.cs, cur.co, n.cls_in, h->params + n.cls_w_off, h->params + n.cls_b_off, n.classes,
                            logits, pred_dev, M);
}

static void forward_eval(Handle* h, const float* x_dev, int B, int crop, float* logits_dev, uint8_t* pred_dev) {
  DRS_CHECK(B >= 1 && crop >= 3 && crop <= 256, "forward: bad B=%d crop=%d", B, crop);
  DRS_CHECK((int64_t)B * crop * crop < (int64_t)1 << 30, "forward: too many pixels in one call");
  switch (act_type(h)) {
    case ET_F32: forward_eval_t<float>(h, x_dev, B, crop, logits_dev, pred_dev); break;
    case ET_F16: forward_eval_t<__half>(h, x_dev, B, crop, logits_dev, pred_dev); break;
    default: forward_eval_t<__nv_bfloat16>(h, x_dev, B, crop, logits_dev, pred_dev); break;
  }
}

__global__ void widen_u8_i64_kernel(const uint8_t* __restrict__ in, long long* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}

extern "C" int drs_forward_dev(drs_handle_t h, const float* x_dev, int32_t B, int32_t crop, float* logits_dev, uint8_t* pred_dev) {
  API_BEGIN
  DRS_CHECK(h && x_dev, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  forward_eval(h, x_dev, B, crop, logits_dev, pred_dev);
  API_END
}

extern "C" int drs_forward_host(drs_handle_t h, const float* x_host, int32_t B, int32_t crop, float* logits_host, int64_t* pred_host) {
  API_BEGIN
  DRS_CHECK(h && x_host, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop * crop;
  const int C = h->net.channels, K = h->net.classes;
  const size_t xb = (size_t)M * C * 4, lb = (size_t)M * K * 4;
  ensure_dstage(h, xb + lb + (size_t)M * 9 + 4096);
  char* d = h->dstage;
  float* x_dev = (float*)d;
  float* lg_dev = (float*)(d + round_up(xb, 256));
  long long* p64 = (long long*)((char*)lg_dev + round_up(lb, 256));
  uint8_t* p8 = (uint8_t*)(p64 + M);
  CUDA_CHECK(cudaMemcpyAsync(x_dev, x_host, xb, cudaMemcpyHostToDevice, h->stream));
  forward_eval(h, x_dev, B, crop, lg_dev, p8);
  if (logits_host) CUDA_CHECK(cudaMemcpyAsync(logits_host, lg_dev, lb, cudaMemcpyDeviceToHost, h->stream));
  if (pred_host) {
    widen_u8_i64_kernel<<<nblk(M, 256), 256, 0, h->stream>>>(p8, p64, M);
    LAUNCH_CHECK(h);
    CUDA_CHECK(cudaMemcpyAsync(pred_host, p64, (size_t)M * 8, cudaMemcpyDeviceToHost, h->stream));
  }
  int rc = drs_synchronize(h);
  if (rc) return rc;
  API_END
}

#include "drs_train.cuh"
#include "drs_scene_api.cuh"
