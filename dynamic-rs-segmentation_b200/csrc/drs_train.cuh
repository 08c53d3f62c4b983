// One training step == sess.run([optimizer, loss, pred_up], is_training=True)
// (/root/reference/isprs_dilated_random.py:1750-1752; graph 1683-1690).  Included by drs_api.cu.
#pragma once

__global__ void pack_extras_kernel(float* __restrict__ dst, const float* __restrict__ loss, const unsigned int* __restrict__ cm, int ncm) {
  const int i = threadIdx.x;
  if (i == 0) dst[0] = loss[0];
  if (i < ncm) dst[1 + i] = (float)cm[i];
}
__global__ void unpack_extras_kernel(const float* __restrict__ src, float* __restrict__ loss, unsigned int* __restrict__ cm, int ncm) {
  const int i = threadIdx.x;
  if (i == 0) loss[0] = src[0];
  if (i < ncm) cm[i] = (unsigned int)(src[1 + i] + 0.5f);
}
__global__ void add2_kernel(const float* __restrict__ a, float* __restrict__ out) { pdl_sync(); out[2] = a[0] + a[1]; }

// blocks per SM of the classifier's filter-gradient kernel (its K-round shared-memory epilogue wants long-lived blocks)
constexpr int CLS_W_BLOCKS_PER_SM = 2;
constexpr int WGRAD_MAX_SPLITS = 48;     // pixel splits of a CUDA-core filter gradient: its partials hold 48 filters

// blocks of the BN statistics kernels: one wave of resident blocks
static inline int bn_blocks(const Handle* h, int64_t M) {
  return (int)std::min<int64_t>(ceil_div(M, 128), (int64_t)h->sm_count * DRS_BN_MINBLK);
}

// squeeze-and-excitation scratch per gate: channel sums, means, hidden, gate, d(gate), d(mean), per-image parameter partials
struct SeBuf { float *sum, *s, *hid, *e, *de, *ds, *part; };

// Every buffer the training step takes from the arena.  layout() is the one description of them: run against a counting
// WsAlloc it sizes the arena (train_arena_bytes), run against the arena it carves them.
template <typename TA>
struct TrainWs {
  std::vector<TA*> Z, Xn, Apre, Gg;   // per layer: conv output, output buffer, activation in front of a post-op, output gradient (squeeze)
  std::vector<uint8_t*> idx;          // per layer: max-pool winner codes
  std::vector<SeBuf> seb;
  TA *F = nullptr, *GF = nullptr;     // dense nets: the concatenated features and their gradient
  TA *T, *DZb[2], *G0, *G1;           // DZ: two buffers, the wgrad of layer l overlaps the backward of layer l-1
  float *logits, *dlogits;
  uint8_t *labels_u8, *pred;          // pred: when the caller passes no buffer
  float *part_bn, *part_ce, *part_cls, *part_clsb, *part_w, *part_l2;
  size_t part_w_cap;                  // floats
  TA *x8 = nullptr, *xcol = nullptr;  // conv1 on the tensor cores: input padded to 8 channels; im2col matrix of its filter gradient
  int nb_ce, nb_cls, cls_rows, nb_opt;

  void layout(const Handle* h, WsAlloc& a, int B, int crop) {
    const NetDesc& n = h->net;
    const int L = (int)n.convs.size(), K = n.classes;
    const int64_t M = (int64_t)B * crop * crop;
    const size_t es = sizeof(TA);
    int maxc = n.cls_in;
    size_t max_w = 0;
    for (auto& c : n.convs) {
      maxc = std::max(maxc, std::max(c.co, c.ci));
      max_w = std::max(max_w, (size_t)c.k * c.k * c.ci * c.co);
    }
    Z.assign(L, nullptr); Xn.assign(L, nullptr); Apre.assign(L, nullptr); Gg.assign(L, nullptr); idx.assign(L, nullptr);
    for (int l = 0; l < L; ++l) {
      const ConvLayer& c = n.convs[l];
      Z[l] = a.take<TA>(M * c.co * es);
      if (n.pool) idx[l] = a.take<uint8_t>(M * c.co);
      // output buffer: a layer's own, or (squeeze modules) the buffer led by layer out_group that it writes a channel slice of
      const bool leads = c.out_group < 0 || c.out_group == l;
      if (!n.dense) Xn[l] = leads ? a.take<TA>(M * std::max(c.co, c.out_cs) * es) : Xn[c.out_group];
      if (c.post) Apre[l] = a.take<TA>(M * c.co * es);
      if (n.squeeze) Gg[l] = leads ? a.take<TA>(M * std::max(c.co, c.out_cs) * es) : Gg[c.out_group];
    }
    seb.assign(n.se.size(), SeBuf{});
    for (size_t i = 0; i < n.se.size(); ++i) {
      const SeBlock& sb = n.se[i];
      float* base = a.take<float>(((size_t)B * (5 * sb.c + sb.r) + (size_t)B * (2 * sb.c * sb.r + sb.r + sb.c)) * 4);
      if (!base) continue;
      SeBuf& q = seb[i];
      q.sum = base; q.s = base + (size_t)B * sb.c; q.e = q.s + (size_t)B * sb.c;
      q.de = q.e + (size_t)B * sb.c; q.ds = q.de + (size_t)B * sb.c; q.hid = q.ds + (size_t)B * sb.c;
      q.part = q.hid + (size_t)B * sb.r;
    }
    if (n.dense) {
      F = a.take<TA>(M * n.feat_stride * es);
      GF = a.take<TA>(M * n.feat_stride * es);
    }
    T = a.take<TA>(M * maxc * es);
    DZb[0] = a.take<TA>(M * maxc * es);
    DZb[1] = a.take<TA>(M * maxc * es);
    G0 = a.take<TA>(M * maxc * es);
    G1 = a.take<TA>(M * maxc * es);
    logits = a.take<float>(M * K * 4);
    dlogits = a.take<float>(M * K * 4);
    labels_u8 = a.take<uint8_t>(M);
    pred = a.take<uint8_t>(M);
    nb_ce = (int)ceil_div(M, CE_THREADS);
    nb_cls = (int)std::min<int64_t>(ceil_div(M, 128), (int64_t)h->sm_count * CLS_W_BLOCKS_PER_SM);
    cls_rows = (int)ceil_div(M, nb_cls);
    nb_opt = (int)ceil_div(n.n_trainable, 256);
    part_w_cap = max_w * WGRAD_MAX_SPLITS;
    part_bn = a.take<float>((size_t)bn_blocks(h, M) * 2 * 256 * 4);
    part_ce = a.take<float>((size_t)nb_ce * 4);
    part_cls = a.take<float>((size_t)nb_cls * n.cls_in * K * 4);
    part_clsb = a.take<float>((size_t)nb_cls * K * 4);
    part_w = a.take<float>(part_w_cap * 4);
    part_l2 = a.take<float>((size_t)nb_opt * 4);
    const ConvLayer& c0 = n.convs[0];
    // conv1's filter gradient on the tensor cores needs the (bf16) im2col matrix of the input: built next to the forward
    if (ElemTag<TA>::v == ET_BF16 && conv1_tc_supported(c0.k, c0.rate, c0.ci, c0.co)) {
      x8 = a.take<TA>(M * 8 * es);
      if (25 * c0.ci <= 128 && wgrad_tc_supported(128, c0.co) && !getenv("DRS_NO_WGRAD_CONV1_TC")) xcol = a.take<TA>(M * 128 * es);
    }
  }
};

static size_t train_arena_bytes(const Handle* h, int B, int crop) {
  return act_type(h) == ET_F32 ? layout_bytes<TrainWs<float>>(h, B, crop) : layout_bytes<TrainWs<__nv_bfloat16>>(h, B, crop);
}

// One layer from its raw convolution output Z to its output, as the normalise and backward-to-dZ phases see it
template <typename TA>
struct NormLayer {
  int B, crop, co, act;
  bool pool;
  int post, post_k;          // ConvLayer::post / post_k
  const SeBlock* se;         // post == 2: the gate and its scratch
  SeBuf* seb;
  TA* Z;
  uint8_t* idx;              // pool: winner codes
  TA* Apre;                  // post-op: the activation in front of it
  ActBuf out;                // the output view the layer writes (pool: [M, co])
  float *mean, *istd;        // batch statistics
  float *mov_mean, *mov_var; // moving statistics the forward updates
  double bn_count;           // pixels behind the batch statistics (all ranks with SyncBN)
  float* part_bn;            // [bn_blocks][2][256] partials
  int64_t M() const { return (int64_t)B * crop * crop; }
};

// what the last block of a forward-statistics kernel does with the grid-wide sums (BnFinish); with SyncBN it only stores them
template <typename TA>
static BnFinish bn_forward_finish(const Handle* h, const NormLayer<TA>& q) {
  BnFinish f{h->bn_acc, 1048576.0, h->bn_counter, h->sums, nullptr, nullptr, nullptr, nullptr, q.bn_count, h->cfg.bn_eps,
             h->cfg.bn_decay, h->cfg.bn_unbiased_ema};
  if (!h->sync_bn) { f.mean = q.mean; f.inv_std = q.istd; f.mov_mean = q.mov_mean; f.mov_var = q.mov_var; }
  return f;
}

// Forward normalise: the batch statistics unless the convolution's epilogue reduced them (stats_fused), the SyncBN reduce,
// then normalise + activation + (max pool | average pool | SE gate).  Pooling nets: one kernel pools the raw conv output and
// normalises the winner.
template <typename TA>
static void forward_normalise(Handle* h, const NormLayer<TA>& q, bool stats_fused) {
  const int64_t M = q.M();
  if (!stats_fused) {
    const int nb = bn_blocks(h, M);
    launch_pdl(h, bn_partial_kernel<TA, TA, 0>, dim3(nb), dim3(BN_THREADS), 0, q.Z, q.co, 0, nullptr, 0, 0, nullptr, nullptr, 0,
               q.part_bn, q.co, M, (int)ceil_div(M, nb), bn_forward_finish(h, q));
    LAUNCH_CHECK(h);
  }
  if (h->sync_bn) {
    do_allreduce(h, h->sums, 2 * q.co);
    launch_pdl(h, bn_finalize_kernel, dim3(nblk(q.co, 128)), dim3(128), 0, h->sums, q.mean, q.istd, q.mov_mean, q.mov_var, q.co,
               q.bn_count, h->cfg.bn_eps, h->cfg.bn_decay, h->cfg.bn_unbiased_ema);
    LAUNCH_CHECK(h);
  }
  if (q.pool) {
    launch_maxpool3_fwd<TA>(h, q.Z, q.co, 0, (TA*)q.out.p, q.co, 0, q.idx, q.co, q.B, q.crop, q.mean, q.istd, q.act);
    return;
  }
  const ActBuf a = q.post ? ActBuf{q.Apre, q.co, 0} : q.out;        // a post-op keeps the activation in front of it
  launch_pdl(h, bn_apply_kernel<TA>, dim3(bne_grid(M, h->sm_count)), dim3(BNE_THREADS), 0, q.Z, q.co, 0, q.mean, q.istd, q.act,
             (TA*)a.p, a.cs, a.co, q.co, M);
  LAUNCH_CHECK(h);
  if (q.post == 1) {
    launch_avgpool_fwd<TA>(h, q.Apre, q.co, 0, (TA*)q.out.p, q.out.cs, q.out.co, q.co, q.B, q.crop, q.post_k);
  } else if (q.post == 2) {
    // squeeze-and-excitation (isprs:682-697): per-image channel means -> FC -> ReLU -> FC -> sigmoid -> gate
    const SeBlock& sb = *q.se;
    const SeBuf& s = *q.seb;
    const int px = q.crop * q.crop;
    se_sum_kernel<TA, 0><<<dim3(q.B, (unsigned)ceil_div(sb.c, 64)), 256, 0, h->stream>>>(q.Apre, q.co, 0, nullptr, 0, 0, sb.c, px, s.sum);
    LAUNCH_CHECK(h);
    se_fc_fwd_kernel<<<q.B, 256, 0, h->stream>>>(s.sum, 1.0f / (float)px, h->params + sb.w1_off, h->params + sb.b1_off,
                                                h->params + sb.w2_off, h->params + sb.b2_off, sb.c, sb.r, s.s, s.hid, s.e);
    LAUNCH_CHECK(h);
    se_scale_fwd_kernel<TA><<<nblk(M * (q.co / 8), 256), 256, 0, h->stream>>>(q.Apre, q.co, 0, s.e, (TA*)q.out.p, q.out.cs, q.out.co,
                                                                            q.co, M, px);
    LAUNCH_CHECK(h);
  }
}

// Pooling layers in bf16 take the backward in two passes instead of four: the BN-backward sums on the pooled side (window
// gradients and pooled activations: bn_partial_kernel MODE 2), then ONE kernel scatters the window gradients to their
// winners and applies the BN backward to the finished fp32 row; the pool's input gradient is never stored, so DRS_DEBUG_KEEP
// records no "da:" tap for these layers.
template <typename TA>
static bool fused_pool_bn_backward(const NormLayer<TA>& q) {
  return q.pool && q.post == 0 && ElemTag<TA>::v == ET_BF16 && q.co <= 512 && pool_lean_enabled() &&
         !getenv("DRS_NO_FUSED_POOL_APPLY");
}

// Backward from the gradient of the layer output (dOut) to dZ: pool or post-op backward (into T), the BN-backward sums, their
// SyncBN reduce, the wait for the filter gradient that last read the dz buffer (wgrad_done; null: none), then the
// BN-backward apply.  Returns the gradient in front of the BN backward, or a null view when the fused path never stores it.
template <typename TA>
static ActBuf backward_to_dz(Handle* h, const NormLayer<TA>& q, const ActBuf& dOut, TA* T, TA* dz, cudaEvent_t wgrad_done) {
  const int64_t M = q.M();
  const int nb = bn_blocks(h, M), rows = (int)ceil_div(M, nb);
  const BnFinish finb{h->bn_acc, 1099511627776.0, h->bn_counter, h->sums, nullptr, nullptr, nullptr, nullptr, q.bn_count, 0.0f, 0.0f, 0};
  auto wait_wgrad = [&]() {
    if (!wgrad_done) return;
    CUDA_CHECK(cudaStreamWaitEvent(h->stream, wgrad_done, 0));
    h->pdl_prev = false;                 // the next kernel also depends on another stream
  };
  if (fused_pool_bn_backward(q)) {
    launch_pdl(h, bn_partial_kernel<TA, TA, 2>, dim3(nb), dim3(BN_THREADS), 0, (const TA*)q.out.p, q.co, 0, (const TA*)dOut.p, dOut.cs,
               dOut.co, (const float*)q.mean, (const float*)q.istd, q.act, q.part_bn, q.co, M, rows, finb);
    LAUNCH_CHECK(h);
    if (h->sync_bn) do_allreduce(h, h->sums, 2 * q.co);
    wait_wgrad();
    launch_maxpool3_bwd_apply(h, (const __nv_bfloat16*)dOut.p, dOut.cs, dOut.co, q.idx, (__nv_bfloat16*)dz, q.co, 0, q.co, q.B, q.crop,
                              (const __nv_bfloat16*)q.Z, q.mean, q.istd, h->sums, 1.0 / q.bn_count, q.act);
    return ActBuf{nullptr, 0, 0};
  }
  ActBuf dA = dOut;
  if (q.pool) {
    launch_maxpool3_bwd<TA>(h, (const TA*)dOut.p, dOut.cs, dOut.co, q.idx, T, q.co, 0, q.co, q.B, q.crop);
    dA = ActBuf{T, q.co, 0};
  }
  if (q.post == 1) {
    launch_avgpool_bwd<TA>(h, (const TA*)dOut.p, dOut.cs, dOut.co, T, q.co, 0, q.co, q.B, q.crop, q.post_k);
    dA = ActBuf{T, q.co, 0};
  } else if (q.post == 2) {
    // gate backward: dA = dOut * e + ds,  ds from d(gate) = sum_px dOut * A through sigmoid, FC2, ReLU, FC1 and the mean;
    // the parameter gradients are per-image partials reduced in fixed order
    const SeBlock& sb = *q.se;
    const SeBuf& s = *q.seb;
    const int px = q.crop * q.crop;
    se_sum_kernel<TA, 1><<<dim3(q.B, (unsigned)ceil_div(sb.c, 64)), 256, 0, h->stream>>>((const TA*)dOut.p, dOut.cs, dOut.co, q.Apre, q.co,
                                                                                        0, sb.c, px, s.de);
    LAUNCH_CHECK(h);
    se_fc_bwd_kernel<<<q.B, 256, 0, h->stream>>>(s.de, s.s, s.hid, s.e, h->params + sb.w1_off, h->params + sb.w2_off, sb.c, sb.r,
                                                1.0f / (float)px, s.ds, s.part);
    LAUNCH_CHECK(h);
    const int64_t np = (int64_t)2 * sb.c * sb.r + sb.r + sb.c;       // W1, b1, W2, b2 are contiguous in the flat buffer
    launch_pdl(h, reduce_partials_kernel, dim3(reduce_partials_grid(np)), dim3(RP_COLS * RP_LANES), 0, s.part, h->grads + sb.w1_off, np,
               q.B, (int64_t)0);
    LAUNCH_CHECK(h);
    se_scale_bwd_kernel<TA><<<nblk(M * (q.co / 8), 256), 256, 0, h->stream>>>((const TA*)dOut.p, dOut.cs, dOut.co, s.e, s.ds, T, q.co, 0,
                                                                            q.co, M, px);
    LAUNCH_CHECK(h);
    dA = ActBuf{T, q.co, 0};
  }
  launch_pdl(h, bn_partial_kernel<TA, TA, 1>, dim3(nb), dim3(BN_THREADS), 0, (const TA*)q.Z, q.co, 0, (const TA*)dA.p, dA.cs, dA.co,
             (const float*)q.mean, (const float*)q.istd, q.act, q.part_bn, q.co, M, rows, finb);
  LAUNCH_CHECK(h);
  if (h->sync_bn) do_allreduce(h, h->sums, 2 * q.co);
  wait_wgrad();
  launch_pdl(h, bn_bwd_apply_kernel<TA, TA>, dim3(bne_grid(M, h->sm_count)), dim3(BNE_THREADS), 0, (const TA*)q.Z, q.co, 0, (const TA*)dA.p,
             dA.cs, dA.co, (const float*)q.mean, (const float*)q.istd, (const float*)h->sums, 1.0 / q.bn_count, q.act, dz, q.co, 0, q.co, M);
  LAUNCH_CHECK(h);
  return dA;
}

// Filter gradient of one convolution (no bias gradient: it is identically zero behind a BN without beta, sum_m dZ = 0).
// conv1 runs from its im2col matrix (xcol) on the tensor cores, or from the fp32 network input (x32) on the CUDA cores; any
// other layer runs from its input view `x` on the tensor cores when the shape allows, else on the CUDA cores.
template <typename TA>
static void filter_gradient(Handle* h, const ConvLayer& c, const ActBuf& x, const float* x32, const TA* xcol, const TA* dz, int B,
                            int crop, float* dw, float* part, size_t part_cap) {
  if (xcol) {
    WgradTcArgs wa;
    wa.x = xcol; wa.in_cstride = 128; wa.in_coff = 0; wa.ci = 128;
    wa.dy = dz; wa.dy_cstride = c.co; wa.dy_coff = 0; wa.co = c.co;
    wa.B = B; wa.crop = crop; wa.k = 1; wa.rate = 1; wa.pad_b = 0;
    wa.dw = dw; wa.part = part; wa.part_capacity = part_cap;
    wa.out_rows = c.k * c.k * c.ci;
    launch_wgrad_tc(h, wa);
  } else if (x32) {
    // conv1: K = 25*C <= 125 rows only -> parallelism must come from many short pixel splits
    // (fp32 mode keeps the generic kernel: its summation order is what the fp32 parity tests pin)
    const bool fast1 = ElemTag<TA>::v != ET_F32 &&
                       launch_wgrad_conv1<TA>(h, x32, c.ci, dz, c.co, 0, c.co, dw, part, part_cap, B, crop, c.k, c.rate);
    if (!fast1) {
      const int splits = (int)std::min<int64_t>((int64_t)part_cap / ((int64_t)c.k * c.k * c.ci * c.co), 4 * h->sm_count);
      launch_wgrad_simt<float, TA>(h, x32, c.ci, 0, c.ci, dz, c.co, 0, c.co, dw, part, splits, B, crop, c.k, c.rate, c.pad_b, 256);
    }
  } else if (ElemTag<TA>::v == ET_BF16 && wgrad_tc_supported(c.ci, c.co)) {
    WgradTcArgs wa;
    wa.x = x.p; wa.in_cstride = x.cs; wa.in_coff = x.co; wa.ci = c.ci;
    wa.dy = dz; wa.dy_cstride = c.co; wa.dy_coff = 0; wa.co = c.co;
    wa.B = B; wa.crop = crop; wa.k = c.k; wa.rate = c.rate; wa.pad_b = c.pad_b;
    wa.dw = dw; wa.part = part; wa.part_capacity = part_cap;
    cudaEvent_t ea = nullptr, eb = nullptr;
    prof_begin(h, &ea, &eb);
    launch_wgrad_tc(h, wa);
    prof_end(h, eb);
    h->conv_flops += 2.0 * (double)B * crop * crop * c.k * c.k * c.ci * c.co;
    h->conv_launches += 1;
  } else {
    launch_wgrad_simt<TA, TA>(h, (const TA*)x.p, x.cs, x.co, c.ci, dz, c.co, 0, c.co, dw, part, WGRAD_MAX_SPLITS, B, crop, c.k, c.rate,
                              c.pad_b);
  }
}

// Data gradient of one convolution: dilated convolution of dZ with the tap-flipped, Ci/Co-transposed filter (w_dgrad, as
// refresh_packed builds it) and the before/after padding swapped, written to `dx`, or -- given a [M, ci] scratch `tmp` --
// added to it
template <typename TA>
static void data_gradient(Handle* h, const ConvLayer& c, const void* w_dgrad, TA* dz, const ActBuf& dx, TA* tmp, int B, int crop) {
  const ActBuf dzb{dz, c.co, 0};
  const ActBuf out = tmp ? ActBuf{tmp, c.ci, 0} : dx;
  run_conv<TA>(h, dzb, c.co, (const float*)w_dgrad, w_dgrad, out, c.ci, B, crop, c.k, c.rate, c.pad_a, h->ones, h->zeros, ACT_NONE);
  if (!tmp) return;
  const int64_t M = (int64_t)B * crop * crop;
  launch_pdl(h, add_slice_kernel<TA>, dim3(nblk(M * (c.ci / 8), 256)), dim3(256), 0, (TA*)dx.p, dx.cs, dx.co, tmp, c.ci, 0, c.ci, M);
  LAUNCH_CHECK(h);
}

template <typename TA>
static void train_step_t(Handle* h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                         const uint8_t* acc_mask_dev, int B, int crop, float* loss_host, uint8_t* pred_out_dev,
                         uint32_t* cm_out_dev) {
  NetDesc& n = h->net;
  const int L = (int)n.convs.size();
  const int K = n.classes;
  const int64_t M = (int64_t)B * crop * crop;
  refresh_packed(h, true);

  ensure_arena(h, layout_bytes<TrainWs<TA>>(h, B, crop));
  h->arena->reset();
  TrainWs<TA> ws;
  {
    WsAlloc carve{h->arena};
    ws.layout(h, carve, B, crop);
  }
  uint8_t* pred = pred_out_dev ? pred_out_dev : ws.pred;
  h->taps.clear();
  debug_keep_reset(h);

  CUDA_CHECK(cudaMemsetAsync(h->grads, 0, (n.n_trainable + 1024) * 4, h->stream));
  h->pdl_on = true;                    // (cleared at the end of the step; see PdlScope)
  h->pdl_prev = false;
  struct PdlScope { Handle* h; ~PdlScope() { h->pdl_on = false; h->pdl_prev = false; } } pdl_scope{h};
  const double bn_count = (double)M * (h->sync_bn ? h->world : 1);

  // ---------------------------------------------------------------- forward (train-mode BN)
  auto input_of = [&](int l) -> ActBuf {
    if (l == 0) return ActBuf{(void*)x_dev, n.channels, 0};
    if (n.dense) return ActBuf{ws.F, n.feat_stride, 0};
    const ConvLayer& c = n.convs[l];
    if (c.in_group >= 0) return ActBuf{ws.Xn[c.in_group], c.in_cs, 0};      // squeeze modules: explicit routing
    return ActBuf{ws.Xn[l - 1], n.convs[l - 1].co, 0};
  };
  auto output_of = [&](int l) -> ActBuf {                                  // the view of its output buffer layer l writes
    const ConvLayer& c = n.convs[l];
    if (n.dense) return ActBuf{ws.F, n.feat_stride, c.out_coff};
    return ActBuf{ws.Xn[l], c.out_cs > 0 ? c.out_cs : c.co, c.out_cs > 0 ? c.out_coff : 0};
  };
  auto norm_layer = [&](int l) -> NormLayer<TA> {
    const ConvLayer& c = n.convs[l];
    return NormLayer<TA>{B, crop, c.co, n.act, n.pool, c.post, c.post_k, c.post == 2 ? &n.se[c.se] : nullptr,
                         c.post == 2 ? &ws.seb[c.se] : nullptr, ws.Z[l], ws.idx[l], ws.Apre[l], output_of(l), h->mean + c.mm_off,
                         h->inv_std + c.mm_off, h->bnstat + c.mm_off, h->bnstat + c.mv_off, bn_count, ws.part_bn};
  };
  for (int l = 0; l < L; ++l) {
    ConvLayer& c = n.convs[l];
    const NormLayer<TA> q = norm_layer(l);
    // conv + bias (raw): scale = 1, shift = bias, no activation   (isprs:710-713)
    // batch statistics (biased variance), moving-average update          (isprs:658-660): reduced inside the tensor-core
    // kernel's epilogue; conv1 and the fp32 mode (CUDA-core convolutions) use the separate statistics kernel
    const BnFinish fin = bn_forward_finish(h, q);
    const bool fused_stats = (l > 0 || ws.x8) && ElemTag<TA>::v != ET_F32;
    if (l == 0 && ws.x8) {
      // conv1 on the tensor cores as in inference (conv1_tc.cuh): input and filter rounded to bf16 like every other layer's
      // operands; the filter is re-packed every step (13 K elements).  The filter gradient keeps the fp32 input.
      const size_t wbytes = (size_t)C1_SLOTS * c.co * 8 * 2;
      c.w_fprop.grow(wbytes, wbytes);
      pack_conv1<TA>(h, h->params + c.w_off, c.w_fprop, c.ci, c.co);
      auto build_xcol = [&]() {
        if (!ws.xcol) return;
        // the im2col matrix is only needed at the very end of the backward: built on the side stream, under the forward
        const bool side = !h->time_convs && !getenv("DRS_NO_OVERLAP");
        if (side) CUDA_CHECK(cudaEventRecord(h->ev_x8, h->stream));
        StreamScope on_side(h, side, h->side_stream);
        if (side) CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_x8, 0));
        launch_pdl(h, im2col_conv1_kernel<TA>, dim3(nblk(M * 16, 256)), dim3(256), 0, ws.x8, ws.xcol, c.ci, crop, M);
        LAUNCH_CHECK(h);
      };
      conv1_tc_forward<TA>(h, x_dev, c.ci, ws.x8, c.w_fprop, ActBuf{ws.Z[l], c.co, 0}, c.co, B, crop, h->ones, h->params + c.b_off,
                           ACT_NONE, fused_stats ? &fin : nullptr, false, build_xcol);
    } else if (l == 0) {
      launch_conv_simt<float, TA>(h, x_dev, n.channels, 0, n.channels, h->params + c.w_off, ws.Z[l], c.co, 0, c.co, B, crop, c.k,
                                  c.rate, c.pad_b, h->ones, h->params + c.b_off, ACT_NONE);
    } else {
      run_conv<TA>(h, input_of(l), c.ci, h->params + c.w_off, c.w_fprop, ActBuf{ws.Z[l], c.co, 0}, c.co, B, crop, c.k, c.rate, c.pad_b,
                   h->ones, h->params + c.b_off, ACT_NONE, fused_stats ? &fin : nullptr);
    }
    debug_keep<TA>(h, "z:" + c.scope, ws.Z[l], c.co, 0, c.co, M);
    forward_normalise(h, q, fused_stats);
    // the layer outputs need no copy: the backward reads them but writes only T, the dZ buffers and the gradient buffers
    h->taps[c.scope] = {q.out.p, ElemTag<TA>::v, q.out.cs, q.out.co, c.co, M};
    // nor does the activation in front of an average pool or SE gate
    if (h->debug_keep && c.post) h->taps["pre:" + c.scope] = {ws.Apre[l], ElemTag<TA>::v, c.co, 0, c.co, M};
  }
  ActBuf feat = n.dense ? ActBuf{ws.F, n.feat_stride, 0}
                        : ActBuf{ws.Xn[L - 1], n.convs[L - 1].out_cs > 0 ? n.convs[L - 1].out_cs : n.convs[L - 1].co, 0};
  launch_classifier_fwd<TA>(h, (const TA*)feat.p, feat.cs, feat.co, n.cls_in, h->params + n.cls_w_off, h->params + n.cls_b_off, K,
                            ws.logits, pred, M);

  // ---------------------------------------------------------------- loss (isprs:1089-1099, contest:881-901)
  // the number of pixels in the mean stays on the device (h->loss_dev[3]); contest's mask count needs no host round trip
  if (mask_dev || h->ignore_label >= 0) {
    CUDA_CHECK(cudaMemsetAsync(h->count_dev, 0, 4, h->stream));
    h->pdl_prev = false;
    launch_pdl(h, mask_count_kernel, dim3((unsigned)std::min<int64_t>(ceil_div(M, 256), 1024)), dim3(256), 0, mask_dev, y_dev, h->ignore_label, M, h->count_dev);
    LAUNCH_CHECK(h);
    launch_pdl(h, set_count_kernel, dim3(1), dim3(1), 0, h->loss_dev + 3, h->count_dev, 0.0f);
    LAUNCH_CHECK(h);
    if (h->world > 1) do_allreduce(h, h->loss_dev + 3, 1);
  } else {
    launch_pdl(h, set_count_kernel, dim3(1), dim3(1), 0, h->loss_dev + 3, nullptr, (float)((double)M * h->world));
    LAUNCH_CHECK(h);
  }
  launch_pdl(h, ce_fwd_bwd_kernel, dim3(ws.nb_ce), dim3(CE_THREADS), 0, ws.logits, y_dev, mask_dev, K, M, h->loss_dev + 3, ws.dlogits,
             ws.part_ce, ws.labels_u8, h->ignore_label);
  LAUNCH_CHECK(h);
  launch_pdl(h, sum_fixed_kernel, dim3(1), dim3(256), 0, ws.part_ce, ws.nb_ce, h->loss_dev, 1.0f, h->loss_dev + 3);
  LAUNCH_CHECK(h);
  if (h->debug_keep) {                 // neither is written again in the step
    h->taps["logits"] = {ws.logits, ET_F32, K, 0, K, M};
    h->taps["dlogits"] = {ws.dlogits, ET_F32, K, 0, K, M};
  }
  // fused calc_accuracy_by_crop (isprs:510-531)
  CUDA_CHECK(cudaMemsetAsync(h->cm_dev, 0, (K * K + 1) * 4, h->stream));
  h->pdl_prev = false;
  launch_pdl(h, confusion_kernel, dim3((unsigned)std::min<int64_t>(ceil_div(M, 256), (int64_t)h->sm_count * 4)), dim3(256), 0, ws.labels_u8,
             pred, acc_mask_dev ? acc_mask_dev : mask_dev, M, K, h->ignore_label, h->cm_dev);
  LAUNCH_CHECK(h);

  // ---------------------------------------------------------------- backward
  // Data parallel: the gradients of the last layers are complete long before the backward ends (they are computed first)
  // and hold most of the bytes (conv4..conv6 + classifier = 83 % of Dilated6Pooling), so that bucket -- with the loss
  // numerator and the confusion counts behind it -- is summed over ranks on a third stream while the backward of the
  // earlier layers runs; only the small front part of the buffer is exchanged at the end.
  const int l_split = (h->world > 1 && !h->time_convs && !getenv("DRS_NO_BUCKETS") && L >= 4) ? L - 3 : -1;
  // classifier: dW, db, dX
  launch_pdl(h, classifier_bwd_weight_kernel<TA>, dim3(ws.nb_cls), dim3(CLSW_THREADS), 0, (const TA*)feat.p, feat.cs, feat.co, n.cls_in,
             ws.dlogits, K, ws.part_cls, ws.part_clsb, M, ws.cls_rows);
  LAUNCH_CHECK(h);
  launch_pdl(h, reduce_partials_kernel, dim3(reduce_partials_grid((int64_t)n.cls_in * K)), dim3(reduce_partials_block((int64_t)n.cls_in * K, ws.nb_cls)), 0,
             ws.part_cls, h->grads + n.cls_w_off, (int64_t)n.cls_in * K, ws.nb_cls, (int64_t)0);
  LAUNCH_CHECK(h);
  launch_pdl(h, reduce_partials_kernel, dim3(reduce_partials_grid(K)), dim3(RP_COLS * RP_LANES), 0, ws.part_clsb, h->grads + n.cls_b_off, K,
             ws.nb_cls, (int64_t)0);
  LAUNCH_CHECK(h);
  if (l_split >= 0) {
    pack_extras_kernel<<<1, 128, 0, h->stream>>>(h->grads + n.n_trainable, h->loss_dev, h->cm_dev, K * K + 1);
    LAUNCH_CHECK(h);
    CUDA_CHECK(cudaEventRecord(h->ev_bucket_ready, h->stream));      // classifier gradients + extras are in the buffer
  }
  // squeeze net: one gradient buffer per output buffer (Gg), because a squeeze convolution's output feeds two layers
  TA* Gcur = n.dense ? ws.GF : (n.squeeze ? ws.Gg[L - 1] : ws.G0);
  TA* Gnext = ws.G1;
  const int gcs0 = n.dense ? n.feat_stride : n.cls_in;
  std::vector<char> grad_written(L, 0);        // squeeze: has the gradient buffer led by layer g been written in this step?
  {
    const int cvc = n.cls_in / 8;
    if (cvc <= 256 && ElemTag<TA>::v != ET_F32) {
      const int rows = 256 / cvc;
      // few, long-lived blocks (two per SM): a thread first loads its 8 x K weights (48 scalar loads), which must be amortised
      int blocks = (int)std::min<int64_t>(ceil_div(M, 2 * rows), (int64_t)h->sm_count * 2);
      launch_pdl(h, classifier_bwd_data_reg_kernel<TA>, dim3(blocks), dim3(256), 0, ws.dlogits, h->params + n.cls_w_off, K, Gcur, gcs0, 0, n.cls_in, M);
    } else {
      int blocks = (int)std::min<int64_t>(ceil_div(M * (n.cls_in / 8), 256), (int64_t)h->sm_count * 16);
      classifier_bwd_data_kernel<TA><<<blocks, 256, n.cls_in * K * 4, h->stream>>>(ws.dlogits, h->params + n.cls_w_off, K, Gcur, gcs0, 0, n.cls_in, M);
    }
    LAUNCH_CHECK(h);
  }
  int gcs = gcs0;   // channel stride of Gcur (non-dense)
  for (int l = L - 1; l >= 0; --l) {
    ConvLayer& c = n.convs[l];
    ActBuf dOut = n.dense ? ActBuf{ws.GF, n.feat_stride, c.out_coff}
                : n.squeeze ? ActBuf{ws.Gg[l], c.out_cs > 0 ? c.out_cs : c.co, c.out_cs > 0 ? c.out_coff : 0}
                            : ActBuf{Gcur, gcs, 0};
    // The filter gradient of layer l is off the critical path (only the optimizer needs it): it runs on a side stream and
    // overlaps the HBM-bound kernels of layer l-1's backward.  dZ is double-buffered; before a buffer is rewritten the
    // main stream waits for the wgrad that read it two layers ago.
    TA* DZ = ws.DZb[l & 1];
    // (a copy: Gcur / GF / Gg are rewritten later in the step)
    debug_keep<TA>(h, "dout:" + c.scope, (const TA*)dOut.p, dOut.cs, dOut.co, c.co, M);
    const ActBuf dA = backward_to_dz(h, norm_layer(l), dOut, ws.T, DZ, l + 2 <= L - 1 ? h->ev_wgrad[l & 1].get() : nullptr);
    if (dA.p) debug_keep<TA>(h, "da:" + c.scope, (const TA*)dA.p, dA.cs, dA.co, c.co, M);
    debug_keep<TA>(h, "dz:" + c.scope, DZ, c.co, 0, c.co, M);
    CUDA_CHECK(cudaEventRecord(h->ev_dz[l & 1], h->stream));
    // (per-launch kernel timing with events needs the launches serialised: no overlap while profiling)
    const bool overlap = !h->time_convs && !getenv("DRS_NO_OVERLAP");
    {
      StreamScope on_side(h, overlap, h->side_stream);
      if (overlap) CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_dz[l & 1], 0));
      filter_gradient<TA>(h, c, input_of(l), l == 0 ? x_dev : nullptr, l == 0 ? ws.xcol : nullptr, DZ, B, crop, h->grads + c.w_off,
                          ws.part_w, ws.part_w_cap);
      CUDA_CHECK(cudaEventRecord(h->ev_wgrad[l & 1], h->stream));
      if (l == l_split) {
        // h->stream is the stream the filter gradients run on (in order: layers L-1..l_split are all complete behind it)
        CUDA_CHECK(cudaStreamWaitEvent(h->comm_stream, h->ev_wgrad[l & 1], 0));
        CUDA_CHECK(cudaStreamWaitEvent(h->comm_stream, h->ev_bucket_ready, 0));
        do_allreduce(h, h->grads + c.w_off, n.n_trainable + 2 + K * K - c.w_off, h->comm_stream);
        CUDA_CHECK(cudaEventRecord(h->ev_bucket_done, h->comm_stream));
      }
    }
    if (!overlap) h->pdl_prev = false;           // the event records went to the main stream
    // dgrad into the gradient of the input buffer
    if (l > 0) {
      if (n.dense) {
        data_gradient<TA>(h, c, c.w_dgrad, DZ, ActBuf{ws.GF, n.feat_stride, 0}, ws.G0, B, crop);
      } else if (n.squeeze) {
        // gradient of the input buffer (led by layer `ig`): the first consumer processed writes it, the second adds
        const int ig = c.in_group >= 0 ? c.in_group : l - 1;
        data_gradient<TA>(h, c, c.w_dgrad, DZ, ActBuf{ws.Gg[ig], c.ci, 0}, grad_written[ig] ? ws.G0 : nullptr, B, crop);
        grad_written[ig] = 1;
      } else {
        data_gradient<TA>(h, c, c.w_dgrad, DZ, ActBuf{Gnext, c.ci, 0}, nullptr, B, crop);
        std::swap(Gcur, Gnext);
        gcs = c.ci;
      }
    }
  }

  // join: every filter gradient is complete before the exchange / the optimizer (the side stream is in order, so the
  // two most recent events cover all layers)
  CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_wgrad[0], 0));
  if (L > 1) CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_wgrad[1], 0));
  h->pdl_prev = false;

  // ---------------------------------------------------------------- exchange + update
  if (h->world > 1) {
    if (l_split >= 0) {
      do_allreduce(h, h->grads, n.convs[l_split].w_off);             // conv1 .. conv(l_split): the small front part
      CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->ev_bucket_done, 0));
    } else {
      pack_extras_kernel<<<1, 128, 0, h->stream>>>(h->grads + n.n_trainable, h->loss_dev, h->cm_dev, K * K + 1);
      LAUNCH_CHECK(h);
      do_allreduce(h, h->grads, n.n_trainable + 2 + K * K);
    }
    unpack_extras_kernel<<<1, 128, 0, h->stream>>>(h->grads + n.n_trainable, h->loss_dev, h->cm_dev, K * K + 1);
    LAUNCH_CHECK(h);
  }
  const float lr = h->cfg.lr_initial * powf(h->cfg.decay_rate, (float)(h->global_step / (h->cfg.decay_steps > 0 ? h->cfg.decay_steps : 1)));
  launch_pdl(h, momentum_update_kernel, dim3(ws.nb_opt), dim3(256), 0, h->params, h->grads, h->moms, n.n_trainable, h->is_weight,
             h->cfg.weight_decay, lr, h->cfg.momentum, 1.0f, ws.part_l2);
  LAUNCH_CHECK(h);
  launch_pdl(h, sum_fixed_kernel, dim3(1), dim3(256), 0, ws.part_l2, ws.nb_opt, h->loss_dev + 1, 0.5f * h->cfg.weight_decay, nullptr);
  LAUNCH_CHECK(h);
  launch_pdl(h, add2_kernel, dim3(1), dim3(1), 0, h->loss_dev, h->loss_dev);
  LAUNCH_CHECK(h);
  h->global_step++;
  h->packed_dirty = true;
  h->eval_dirty = true;
  if (cm_out_dev) CUDA_CHECK(cudaMemcpyAsync(cm_out_dev, h->cm_dev, (K * K + 1) * 4, cudaMemcpyDeviceToDevice, h->stream));
  if (loss_host) {
    CUDA_CHECK(cudaMemcpyAsync(loss_host, h->loss_dev + 2, 4, cudaMemcpyDeviceToHost, h->stream));
    int rc = drs_synchronize(h);
    if (rc) throw DrsError{rc};
  }
}

static void train_step_dispatch(Handle* h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                                const uint8_t* acc_mask_dev, int B, int crop, uint8_t* pred_dev, uint32_t* cm_dev) {
  switch (act_type(h)) {
    case ET_F32: train_step_t<float>(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, nullptr, pred_dev, cm_dev); break;
    case ET_BF16: train_step_t<__nv_bfloat16>(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, nullptr, pred_dev, cm_dev); break;
    default:
      DRS_FAIL("train_step: precision F16 is inference-only (gradients underflow in fp16); create the handle with DRS_PREC_BF16 or DRS_PREC_FP32");
  }
}

static void train_step(Handle* h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                       const uint8_t* acc_mask_dev, int B, int crop, float* loss_host, uint8_t* pred_dev, uint32_t* cm_dev,
                       bool capture_only = false) {
  DRS_CHECK(B >= 1 && crop >= 3 && crop <= 256, "train_step: bad B=%d crop=%d", B, crop);
  TrainGraph* replay = nullptr;
  // (the legacy default stream cannot be captured)
  // (data parallel: capturable only when the exchange is the in-library NCCL call, not a host callback)
  const bool graphable = h->use_graphs && (h->world <= 1 || h->nccl) && !getenv("DRS_DEBUG_KEEP") &&
                         h->cfg.precision != DRS_PREC_F16 && h->stream != nullptr;
  if (!graphable) {
    if (capture_only) return;
    train_step_dispatch(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, pred_dev, cm_dev);
  } else {
    ensure_arena(h, train_arena_bytes(h, B, crop));        // before the key: a re-allocation bumps arena_epoch
    const float lr = h->cfg.lr_initial * powf(h->cfg.decay_rate, (float)(h->global_step / (h->cfg.decay_steps > 0 ? h->cfg.decay_steps : 1)));
    TrainGraphKey key;
    memset(&key, 0, sizeof(key));
    key.B = B; key.crop = crop; key.ignore_label = h->ignore_label; key.profiling = h->time_convs ? 1 : 0;
    key.x = x_dev; key.y = y_dev; key.mask = mask_dev; key.acc_mask = acc_mask_dev; key.pred = pred_dev; key.cm = cm_dev;
    memcpy(&key.lr_bits, &lr, 4);
    key.arena_epoch = h->arena_epoch;
    auto it = h->graphs.find(key);
    if (it != h->graphs.end()) {
      replay = &it->second;
      h->launches += replay->launches;
      h->conv_flops += replay->conv_flops;
      h->conv_launches += replay->conv_launches;
      h->global_step++;
    } else {
      // capture (nothing executes while capturing), then launch like any later replay
      TrainGraph g;
      const int64_t l0 = h->launches, cl0 = h->conv_launches;
      const double f0 = h->conv_flops;
      h->packed_dirty = true;                        // the operand repack must be part of every replay
      CUDA_CHECK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
      h->capturing = &g;
      cudaGraph_t graph = nullptr;
      try {
        train_step_dispatch(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, pred_dev, cm_dev);
      } catch (...) {
        h->capturing = nullptr;
        cudaStreamEndCapture(h->stream, &graph);
        if (graph) cudaGraphDestroy(graph);
        throw;
      }
      h->capturing = nullptr;
      CUDA_CHECK(cudaStreamEndCapture(h->stream, &graph));
      cudaGraphExec_t exec = nullptr;
      cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      CUDA_CHECK(e);
      g.exec = GraphExec(exec);
      CUDA_CHECK(cudaGraphUpload(g.exec, h->stream));   // pay the device-side set-up now, not at the first replay
      g.launches = h->launches - l0;
      g.conv_launches = h->conv_launches - cl0;
      g.conv_flops = h->conv_flops - f0;
      auto ins = h->graphs.emplace(key, std::move(g));
      replay = &ins.first->second;
      if (capture_only) {                            // drs_train_prepare: undo the host-side bookkeeping of the dry capture
        h->launches = l0;
        h->conv_launches = cl0;
        h->conv_flops = f0;
        h->global_step--;
        return;
      }
    }
    CUDA_CHECK(cudaGraphLaunch(replay->exec, h->stream));
    h->packed_dirty = true;
    h->eval_dirty = true;
  }
  if (loss_host) CUDA_CHECK(cudaMemcpyAsync(loss_host, h->loss_dev + 2, 4, cudaMemcpyDeviceToHost, h->stream));
  if (loss_host || (replay && h->time_convs)) {
    int rc = drs_synchronize(h);
    if (rc) throw DrsError{rc};
  }
  if (replay && h->time_convs) {
    for (auto& pr : replay->events) {
      float ms = 0.0f;
      CUDA_CHECK(cudaEventElapsedTime(&ms, pr.first, pr.second));
      h->conv_ms_acc += ms;
    }
  }
}

extern "C" int drs_train_step_dev(drs_handle_t h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                                  const uint8_t* acc_mask_dev, int32_t B, int32_t crop, float* loss_out_host, uint8_t* pred_dev,
                                  uint32_t* cm_dev) {
  API_BEGIN
  DRS_CHECK(h && x_dev && y_dev, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  train_step(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, loss_out_host, pred_dev, cm_dev);
  API_END
}

// ------------------------------------------------------------------------------------------------
// unit-test entries for the backward pieces of the step (tests/test_gpu_parity.py): each runs the step's own phase
// functions for one layer, on caller-supplied tensors
// ------------------------------------------------------------------------------------------------
template <typename TA>
static void debug_dgrad_t(Handle* h, const float* dy32, const float* w32, int B, int crop, int k, int rate, int ci, int co, float* dx32) {
  const int64_t M = (int64_t)B * crop * crop;
  const ConvLayer c = conv_shape(k, rate, ci, co);
  TA* dy = (TA*)arena_take(h, M * co * sizeof(TA));
  TA* dx = (TA*)arena_take(h, M * ci * sizeof(TA));
  void* wd = arena_take(h, (int64_t)k * k * ci * co * 4);
  cast_kernel<float, TA><<<nblk(M * co, 256), 256, 0, h->stream>>>(dy32, dy, M * co);
  LAUNCH_CHECK(h);
  repack_filter(h, w32, wd, k * k, ci, co, ElemTag<TA>::v == ET_F32 ? 2 : 1, ElemTag<TA>::v);
  data_gradient<TA>(h, c, wd, dy, ActBuf{dx, ci, 0}, nullptr, B, crop);
  cast_kernel<TA, float><<<nblk(M * ci, 256), 256, 0, h->stream>>>(dx, dx32, M * ci);
  LAUNCH_CHECK(h);
}

extern "C" int drs_debug_dgrad(drs_handle_t h, const float* dy_host, const float* w_host, int32_t B, int32_t crop, int32_t k,
                               int32_t rate, int32_t Ci, int32_t Co, int32_t precision, float* dx_host) {
  API_BEGIN
  DRS_CHECK(h && dy_host && w_host && dx_host, "null argument");
  DRS_CHECK(precision == DRS_PREC_FP32 || precision == DRS_PREC_BF16, "debug_dgrad: fp32 or bf16");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop * crop;
  const int64_t nw = (int64_t)k * k * Ci * Co;
  ensure_arena(h, (size_t)M * (Ci + Co) * 8 + nw * 8 + (1 << 20));
  h->arena->reset();
  float* dy32 = (float*)arena_take(h, M * Co * 4);
  float* w32 = (float*)arena_take(h, nw * 4);
  float* dx32 = (float*)arena_take(h, M * Ci * 4);
  CUDA_CHECK(cudaMemcpyAsync(dy32, dy_host, M * Co * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(w32, w_host, nw * 4, cudaMemcpyHostToDevice, h->stream));
  if (precision == DRS_PREC_FP32) debug_dgrad_t<float>(h, dy32, w32, B, crop, k, rate, Ci, Co, dx32);
  else debug_dgrad_t<__nv_bfloat16>(h, dy32, w32, B, crop, k, rate, Ci, Co, dx32);
  CUDA_CHECK(cudaMemcpyAsync(dx_host, dx32, M * Ci * 4, cudaMemcpyDeviceToHost, h->stream));
  int rc = drs_synchronize(h);
  if (rc) return rc;
  API_END
}

// One layer's normalise / activate / pool forward and its backward: z [M,C] is the raw conv output, dout the gradient with
// respect to the layer output.  Returns the layer output and dZ, through the training step's two phases.
template <typename TA>
static void debug_layer_t(Handle* h, const float* z32, const float* dout32, int B, int crop, int C, int pool, int act, float* out32,
                          float* dz32, float* mean_out, float* istd_out) {
  const int64_t M = (int64_t)B * crop * crop;
  NormLayer<TA> q{};
  q.B = B; q.crop = crop; q.co = C; q.act = act; q.pool = pool != 0;
  q.Z = (TA*)arena_take(h, M * C * sizeof(TA));
  TA* Xo = (TA*)arena_take(h, M * C * sizeof(TA));
  q.out = ActBuf{Xo, C, 0};
  TA* G = (TA*)arena_take(h, M * C * sizeof(TA));
  TA* T = (TA*)arena_take(h, M * C * sizeof(TA));
  TA* DZ = (TA*)arena_take(h, M * C * sizeof(TA));
  q.idx = (uint8_t*)arena_take(h, M * C);
  q.part_bn = (float*)arena_take(h, (size_t)bn_blocks(h, M) * 2 * 256 * 4);
  q.mean = h->mean;
  q.istd = h->inv_std;
  float* scratch_stats = (float*)arena_take(h, 4 * 512 * 4);      // moving statistics the finish step updates (discarded)
  q.mov_mean = scratch_stats;
  q.mov_var = scratch_stats + 512;
  q.bn_count = (double)M;
  CUDA_CHECK(cudaMemsetAsync(scratch_stats, 0, 4 * 512 * 4, h->stream));
  cast_kernel<float, TA><<<nblk(M * C, 256), 256, 0, h->stream>>>(z32, q.Z, M * C);
  LAUNCH_CHECK(h);
  cast_kernel<float, TA><<<nblk(M * C, 256), 256, 0, h->stream>>>(dout32, G, M * C);
  LAUNCH_CHECK(h);
  forward_normalise(h, q, false);
  backward_to_dz(h, q, ActBuf{G, C, 0}, T, DZ, nullptr);
  cast_kernel<TA, float><<<nblk(M * C, 256), 256, 0, h->stream>>>(Xo, out32, M * C);
  LAUNCH_CHECK(h);
  cast_kernel<TA, float><<<nblk(M * C, 256), 256, 0, h->stream>>>(DZ, dz32, M * C);
  LAUNCH_CHECK(h);
  CUDA_CHECK(cudaMemcpyAsync(mean_out, q.mean, C * 4, cudaMemcpyDeviceToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(istd_out, q.istd, C * 4, cudaMemcpyDeviceToDevice, h->stream));
}

extern "C" int drs_debug_layer(drs_handle_t h, const float* z_host, const float* dout_host, int32_t B, int32_t crop, int32_t C,
                               int32_t pool, int32_t act, int32_t precision, float* out_host, float* dz_host, float* mean_host,
                               float* inv_std_host) {
  API_BEGIN
  DRS_CHECK(h && z_host && dout_host && out_host && dz_host, "null argument");
  DRS_CHECK(precision == DRS_PREC_FP32 || precision == DRS_PREC_BF16, "debug_layer: fp32 or bf16");
  DRS_CHECK(C % 8 == 0 && C <= 256, "debug_layer: C=%d must be a multiple of 8, at most 256", C);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop * crop;
  ensure_arena(h, (size_t)M * C * (4 * 4 + 6 * 4 + 1) + (8 << 20));
  h->arena->reset();
  float* z32 = (float*)arena_take(h, M * C * 4);
  float* g32 = (float*)arena_take(h, M * C * 4);
  float* o32 = (float*)arena_take(h, M * C * 4);
  float* dz32 = (float*)arena_take(h, M * C * 4);
  float* ms = (float*)arena_take(h, 2 * C * 4);
  CUDA_CHECK(cudaMemcpyAsync(z32, z_host, M * C * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(g32, dout_host, M * C * 4, cudaMemcpyHostToDevice, h->stream));
  if (precision == DRS_PREC_FP32) debug_layer_t<float>(h, z32, g32, B, crop, C, pool, act, o32, dz32, ms, ms + C);
  else debug_layer_t<__nv_bfloat16>(h, z32, g32, B, crop, C, pool, act, o32, dz32, ms, ms + C);
  CUDA_CHECK(cudaMemcpyAsync(out_host, o32, M * C * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(dz_host, dz32, M * C * 4, cudaMemcpyDeviceToHost, h->stream));
  if (mean_host) CUDA_CHECK(cudaMemcpyAsync(mean_host, ms, C * 4, cudaMemcpyDeviceToHost, h->stream));
  if (inv_std_host) CUDA_CHECK(cudaMemcpyAsync(inv_std_host, ms + C, C * 4, cudaMemcpyDeviceToHost, h->stream));
  int rc = drs_synchronize(h);
  if (rc) return rc;
  API_END
}

// The same step without a host round trip: loss and confusion counts are copied into a pinned result slot behind an event
// and fetched later with drs_train_result(ticket) -- the reference's loop only needs them for the score update and the
// log lines (isprs:1754-1778), neither of which feeds the next step's draws.
extern "C" int drs_train_step_async(drs_handle_t h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                                    const uint8_t* acc_mask_dev, int32_t B, int32_t crop, uint8_t* pred_dev, int64_t* ticket_out) {
  API_BEGIN
  DRS_CHECK(h && x_dev && y_dev && ticket_out, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int K = h->net.classes;
  train_step(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, nullptr, pred_dev, nullptr);
  const int64_t t = h->next_ticket++;
  float* slot = h->result_host + (size_t)(t % Handle::RESULT_RING) * RESULT_STRIDE;
  CUDA_CHECK(cudaMemcpyAsync(slot, h->loss_dev + 2, 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(slot + 1, h->cm_dev, (K * K + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaEventRecord(h->result_ev[t % Handle::RESULT_RING], h->stream));
  *ticket_out = t;
  API_END
}

extern "C" int drs_train_result(drs_handle_t h, int64_t ticket, float* loss_out, uint32_t* cm_out) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  DRS_CHECK(ticket >= 0 && ticket < h->next_ticket && ticket >= h->next_ticket - Handle::RESULT_RING,
            "train_result: ticket %lld is not one of the last %d steps (next ticket %lld)", (long long)ticket,
            Handle::RESULT_RING, (long long)h->next_ticket);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  CUDA_CHECK(cudaEventSynchronize(h->result_ev[ticket % Handle::RESULT_RING]));
  const float* slot = h->result_host + (size_t)(ticket % Handle::RESULT_RING) * RESULT_STRIDE;
  const int K = h->net.classes;
  if (loss_out) *loss_out = slot[0];
  if (cm_out) memcpy(cm_out, slot + 1, (K * K + 1) * 4);
  API_END
}

extern "C" int drs_reserve_workspace(drs_handle_t h, int32_t B, int32_t crop_max, int32_t training) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  DRS_CHECK(B >= 1 && crop_max >= 3 && crop_max <= 256, "reserve_workspace: bad B=%d crop=%d", B, crop_max);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop_max * crop_max;
  const int C = h->net.channels, K = h->net.classes;
  const size_t eval = eval_arena_bytes(h, B, crop_max);
  ensure_arena(h, training ? std::max(train_arena_bytes(h, B, crop_max), eval) : eval);
  if (training) {
    // both device staging slots of the planned gather (drs_gather_plan_dev): worst case = every patch noisy
    const size_t need = (size_t)M * C * 8 + (size_t)B * 128 + 8192;
    for (int s = 0; s < 2; ++s) h->plan_stage[s].grow(need, need, {h->stream, h->plan_stream});
  }
  // staging of the *_host entry points (x, y, two masks, int64 + uint8 predictions, confusion counts, logits)
  ensure_dstage(h, round_up((size_t)M * C * 4, 256) + round_up((size_t)M * 4, 256) + 2 * round_up((size_t)M, 256) +
                       round_up((size_t)M * 9, 256) + round_up((size_t)M * K * 4, 256) + 8192);
  API_END
}

extern "C" int drs_train_prepare(drs_handle_t h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                                 const uint8_t* acc_mask_dev, int32_t B, int32_t crop, uint8_t* pred_dev, uint32_t* cm_dev) {
  API_BEGIN
  DRS_CHECK(h && x_dev && y_dev, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  train_step(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, nullptr, pred_dev, cm_dev, true);
  API_END
}

extern "C" int drs_train_step_host(drs_handle_t h, const float* x_host, const float* y_host, const uint8_t* mask_host,
                                   const uint8_t* acc_mask_host, int32_t B, int32_t crop, float* loss_out, int64_t* pred_host,
                                   uint32_t* cm_host) {
  API_BEGIN
  DRS_CHECK(h && x_host && y_host, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop * crop;
  const int C = h->net.channels, K = h->net.classes;
  const size_t xb = round_up((size_t)M * C * 4, 256), yb = round_up((size_t)M * 4, 256), mb = round_up((size_t)M, 256);
  ensure_dstage(h, xb + yb + 2 * mb + (size_t)M * 9 + 4096 + 1024);
  char* d = h->dstage;
  float* x_dev = (float*)d;
  float* y_dev = (float*)(d + xb);
  uint8_t* m_dev = (uint8_t*)(d + xb + yb);
  uint8_t* am_dev = (uint8_t*)(d + xb + yb + mb);
  long long* p64 = (long long*)(d + xb + yb + 2 * mb);
  uint8_t* p8 = (uint8_t*)(p64 + M);
  uint32_t* cm_dev = (uint32_t*)(d + xb + yb + 2 * mb + round_up((size_t)M * 9, 256));
  CUDA_CHECK(cudaMemcpyAsync(x_dev, x_host, (size_t)M * C * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(y_dev, y_host, (size_t)M * 4, cudaMemcpyHostToDevice, h->stream));
  if (mask_host) CUDA_CHECK(cudaMemcpyAsync(m_dev, mask_host, (size_t)M, cudaMemcpyHostToDevice, h->stream));
  if (acc_mask_host) CUDA_CHECK(cudaMemcpyAsync(am_dev, acc_mask_host, (size_t)M, cudaMemcpyHostToDevice, h->stream));
  float loss = 0.0f;
  train_step(h, x_dev, y_dev, mask_host ? m_dev : nullptr, acc_mask_host ? am_dev : nullptr, B, crop, &loss, p8, cm_dev);
  if (pred_host) {
    widen_u8_i64_kernel<<<nblk(M, 256), 256, 0, h->stream>>>(p8, p64, M);
    LAUNCH_CHECK(h);
    CUDA_CHECK(cudaMemcpyAsync(pred_host, p64, (size_t)M * 8, cudaMemcpyDeviceToHost, h->stream));
  }
  if (cm_host) CUDA_CHECK(cudaMemcpyAsync(cm_host, cm_dev, (K * K + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
  int rc = drs_synchronize(h);
  if (rc) return rc;
  if (loss_out) *loss_out = loss;
  API_END
}
