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

static size_t train_workspace_bytes(Handle* h, int B, int crop, size_t es) {
  NetDesc& n = h->net;
  const int K = n.classes;
  const int64_t M = (int64_t)B * crop * crop;
  int maxc = n.cls_in;
  for (auto& c : n.convs) maxc = std::max(maxc, std::max(c.co, c.ci));
  size_t need = 1 << 20;
  auto add = [&](size_t b) { need += round_up(b, 1024) + 1024; };
  for (auto& c : n.convs) {
    add(M * c.co * es);                       // Z
    if (n.pool) add(M * c.co);                // idx
    if (!n.dense) add(M * std::max(c.co, c.out_cs) * es);   // X_{l+1} (a squeeze module's two expand convs share one)
    if (c.post) add(M * c.co * es);           // A: the activation in front of the post-op (average pool / SE gate)
    if (n.squeeze) add(M * std::max(c.co, c.out_cs) * es);  // gradient of the layer's output buffer
  }
  if (n.dense) add(M * n.feat_stride * es * 2);   // F and GF
  for (auto& sb : n.se) add(((size_t)B * (5 * sb.c + sb.r) + (size_t)B * (2 * sb.c * sb.r + sb.r + sb.c)) * 4 + 4096);
  add(M * maxc * es);                         // T
  add(M * maxc * es * 2);                     // DZ (two buffers: wgrad of layer l overlaps the backward of layer l-1)
  add(M * maxc * es * 2);                     // G ping-pong / dense dgrad temp
  add(M * K * 4 * 2);                         // logits, dlogits
  add(M * 2);                                 // labels u8, pred
  add(M * 8 * es);                            // conv1 input padded to 8 channels (tensor-core conv1)
  add(M * 128 * es);                          // conv1 im2col matrix (tensor-core filter gradient)
  const int nb_bn = (int)std::min<int64_t>(ceil_div(M, 128), (int64_t)h->sm_count * DRS_BN_MINBLK);   // one wave of resident blocks
  const int bn_rows = (int)ceil_div(M, nb_bn);
  add((size_t)nb_bn * 2 * 256 * 4);
  const int nb_ce = (int)ceil_div(M, CE_THREADS);
  add((size_t)nb_ce * 4);
  const int nb_cls = (int)std::min<int64_t>(ceil_div(M, 128), (int64_t)h->sm_count * CLS_W_BLOCKS_PER_SM);
  const int cls_rows = (int)ceil_div(M, nb_cls);
  add((size_t)nb_cls * (n.cls_in + 1) * K * 4);
  const int max_splits = 48;
  size_t max_w = 0;
  for (auto& c : n.convs) max_w = std::max(max_w, (size_t)c.k * c.k * c.ci * c.co);
  add(max_w * 4 * max_splits);
  const int nb_opt = (int)ceil_div(n.n_trainable, 256);
  add((size_t)nb_opt * 4);
  return need;
}

template <typename TA>
static void train_step_t(Handle* h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                         const uint8_t* acc_mask_dev, int B, int crop, float* loss_host, uint8_t* pred_out_dev,
                         uint32_t* cm_out_dev) {
  NetDesc& n = h->net;
  HandleExtra* x = X(h);
  const int L = (int)n.convs.size();
  const int K = n.classes;
  const int64_t M = (int64_t)B * crop * crop;
  const size_t es = sizeof(TA);
  refresh_packed(h, true);

  // ---------------------------------------------------------------- workspace (sized by train_workspace_bytes)
  int maxc = n.cls_in;
  for (auto& c : n.convs) maxc = std::max(maxc, std::max(c.co, c.ci));
  const int nb_bn = (int)std::min<int64_t>(ceil_div(M, 128), (int64_t)h->sm_count * DRS_BN_MINBLK);   // one wave of resident blocks
  const int bn_rows = (int)ceil_div(M, nb_bn);
  const int nb_ce = (int)ceil_div(M, CE_THREADS);
  const int nb_cls = (int)std::min<int64_t>(ceil_div(M, 128), (int64_t)h->sm_count * CLS_W_BLOCKS_PER_SM);
  const int cls_rows = (int)ceil_div(M, nb_cls);
  const int max_splits = 48;
  size_t max_w = 0;
  for (auto& c : n.convs) max_w = std::max(max_w, (size_t)c.k * c.k * c.ci * c.co);
  const int nb_opt = (int)ceil_div(n.n_trainable, 256);
  ensure_arena(h, train_workspace_bytes(h, B, crop, es));
  h->arena.reset();

  std::vector<TA*> Z(L), Xn(L), Apre(L, nullptr), Gg(L, nullptr);
  std::vector<uint8_t*> idx(L, nullptr);
  TA* F = nullptr;
  TA* GF = nullptr;
  for (int l = 0; l < L; ++l) {
    ConvLayer& c = n.convs[l];
    Z[l] = (TA*)arena_take(h, M * c.co * es);
    if (n.pool) idx[l] = (uint8_t*)arena_take(h, M * c.co);
    // output buffer: a layer's own, or (squeeze modules) the buffer led by layer out_group that it writes a channel slice of
    if (!n.dense) {
      if (c.out_group < 0 || c.out_group == l) Xn[l] = (TA*)arena_take(h, M * std::max(c.co, c.out_cs) * es);
      else Xn[l] = Xn[c.out_group];
    }
    if (c.post) Apre[l] = (TA*)arena_take(h, M * c.co * es);
    if (n.squeeze) {
      if (c.out_group < 0 || c.out_group == l) Gg[l] = (TA*)arena_take(h, M * std::max(c.co, c.out_cs) * es);
      else Gg[l] = Gg[c.out_group];
    }
  }
  // squeeze-and-excitation scratch per gate: channel sums, means, hidden, gate, d(gate), d(mean), per-image parameter partials
  struct SeBuf { float *sum, *s, *hid, *e, *de, *ds, *part; };
  std::vector<SeBuf> seb(n.se.size());
  for (size_t i = 0; i < n.se.size(); ++i) {
    const SeBlock& sb = n.se[i];
    float* base = (float*)arena_take(h, ((size_t)B * (5 * sb.c + sb.r) + (size_t)B * (2 * sb.c * sb.r + sb.r + sb.c)) * 4);
    seb[i].sum = base; seb[i].s = base + (size_t)B * sb.c; seb[i].e = seb[i].s + (size_t)B * sb.c;
    seb[i].de = seb[i].e + (size_t)B * sb.c; seb[i].ds = seb[i].de + (size_t)B * sb.c; seb[i].hid = seb[i].ds + (size_t)B * sb.c;
    seb[i].part = seb[i].hid + (size_t)B * sb.r;
  }
  if (n.dense) {
    F = (TA*)arena_take(h, M * n.feat_stride * es);
    GF = (TA*)arena_take(h, M * n.feat_stride * es);
  }
  TA* T = (TA*)arena_take(h, M * maxc * es);
  TA* DZb[2] = {(TA*)arena_take(h, M * maxc * es), (TA*)arena_take(h, M * maxc * es)};
  TA* G0 = (TA*)arena_take(h, M * maxc * es);
  TA* G1 = (TA*)arena_take(h, M * maxc * es);
  float* logits = (float*)arena_take(h, M * K * 4);
  float* dlogits = (float*)arena_take(h, M * K * 4);
  uint8_t* labels_u8 = (uint8_t*)arena_take(h, M);
  uint8_t* pred = pred_out_dev ? pred_out_dev : (uint8_t*)arena_take(h, M);
  float* part_bn = (float*)arena_take(h, (size_t)nb_bn * 2 * 256 * 4);
  float* part_ce = (float*)arena_take(h, (size_t)nb_ce * 4);
  float* part_cls = (float*)arena_take(h, (size_t)nb_cls * n.cls_in * K * 4);
  float* part_clsb = (float*)arena_take(h, (size_t)nb_cls * K * 4);
  float* part_w = (float*)arena_take(h, max_w * 4 * max_splits);
  float* part_l2 = (float*)arena_take(h, (size_t)nb_opt * 4);
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
    if (n.dense) return ActBuf{F, n.feat_stride, 0};
    const ConvLayer& c = n.convs[l];
    if (c.in_group >= 0) return ActBuf{Xn[c.in_group], c.in_cs, 0};      // squeeze modules: explicit routing
    return ActBuf{Xn[l - 1], n.convs[l - 1].co, 0};
  };
  auto output_of = [&](int l) -> ActBuf {                                  // the view of its output buffer layer l writes
    const ConvLayer& c = n.convs[l];
    if (n.dense) return ActBuf{F, n.feat_stride, c.out_coff};
    return ActBuf{Xn[l], c.out_cs > 0 ? c.out_cs : c.co, c.out_cs > 0 ? c.out_coff : 0};
  };
  const bool conv1_on_tc = ElemTag<TA>::v == ET_BF16 && conv1_tc_supported(n.convs[0].k, n.convs[0].rate, n.convs[0].ci, n.convs[0].co);
  // conv1's filter gradient on the tensor cores needs the (bf16) im2col matrix of the input: built next to the forward
  const bool wgrad1_on_tc = conv1_on_tc && 25 * n.convs[0].ci <= 128 && wgrad_tc_supported(128, n.convs[0].co) && !getenv("DRS_NO_WGRAD_CONV1_TC");
  TA* xcol = nullptr;
  for (int l = 0; l < L; ++l) {
    ConvLayer& c = n.convs[l];
    ActBuf zb{Z[l], c.co, 0};
    // conv + bias (raw): scale = 1, shift = bias, no activation   (isprs:710-713)
    // batch statistics (biased variance), moving-average update          (isprs:658-660): reduced inside the tensor-core
    // kernel's epilogue; conv1 and the fp32 mode (CUDA-core convolutions) use the separate statistics kernel
    float* mean = x->mean + c.mm_off;
    float* istd = x->inv_std + c.mm_off;
    BnFinish fin{x->bn_acc, 1048576.0, x->bn_counter, x->sums, nullptr, nullptr, nullptr, nullptr, bn_count, h->cfg.bn_eps, h->cfg.bn_decay, h->cfg.bn_unbiased_ema};
    if (!h->sync_bn) { fin.mean = mean; fin.inv_std = istd; fin.mov_mean = h->bnstat + c.mm_off; fin.mov_var = h->bnstat + c.mv_off; }
    const bool fused_stats = (l > 0 || conv1_on_tc) && ElemTag<TA>::v != ET_F32;
    if (l == 0 && conv1_on_tc) {
      // conv1 on the tensor cores as in inference (conv1_tc.cuh): input and filter rounded to bf16 like every other layer's
      // operands; the filter is re-packed every step (13 K elements).  The filter gradient keeps the fp32 input.
      if (!c.w_fprop) CUDA_CHECK(cudaMalloc(&c.w_fprop, (size_t)C1_SLOTS * c.co * 8 * 2));
      launch_pdl(h, pack_conv1_kernel<TA>, dim3(nblk(C1_SLOTS * c.co * 8, 256)), dim3(256), 0, h->params + c.w_off, (TA*)c.w_fprop, c.ci, c.co);
      LAUNCH_CHECK(h);
      TA* x8 = (TA*)arena_take(h, (size_t)M * 8 * sizeof(TA));
      launch_pdl(h, pad_cast8_kernel<TA>, dim3(nblk(M, 256)), dim3(256), 0, x_dev, x8, c.ci, M);
      LAUNCH_CHECK(h);
      if (wgrad1_on_tc) {
        // the im2col matrix is only needed at the very end of the backward: built on the side stream, under the forward
        xcol = (TA*)arena_take(h, (size_t)M * 128 * sizeof(TA));
        const bool side = !h->time_convs && !getenv("DRS_NO_OVERLAP");
        cudaStream_t main_stream = h->stream;
        const bool pdl_main = h->pdl_prev;
        if (side) {
          CUDA_CHECK(cudaEventRecord(x->ev_x8, h->stream));
          h->stream = x->side_stream;
          h->pdl_prev = false;
          CUDA_CHECK(cudaStreamWaitEvent(h->stream, x->ev_x8, 0));
        }
        try {
          launch_pdl(h, im2col_conv1_kernel<TA>, dim3(nblk(M * 16, 256)), dim3(256), 0, x8, xcol, c.ci, crop, M);
          LAUNCH_CHECK(h);
        } catch (...) { h->stream = main_stream; throw; }
        if (side) { h->stream = main_stream; h->pdl_prev = pdl_main; }
      }
      Conv1TcArgs a1;
      a1.x8 = x8; a1.wpack = c.w_fprop; a1.out = Z[l]; a1.out_cstride = c.co; a1.out_coff = 0; a1.co = c.co;
      a1.B = B; a1.crop = crop; a1.scale = x->ones; a1.shift = h->params + c.b_off; a1.act = ACT_NONE; a1.etype = ElemTag<TA>::v;
      a1.stats = fused_stats ? &fin : nullptr;
      launch_conv1_tc(h, a1);
    } else if (l == 0) {
      launch_conv_simt<float, TA>(h, x_dev, n.channels, 0, n.channels, h->params + c.w_off, Z[l], c.co, 0, c.co, B, crop, c.k,
                                  c.rate, c.pad_b, x->ones, h->params + c.b_off, ACT_NONE);
    } else {
      run_conv<TA>(h, input_of(l), c.ci, h->params + c.w_off, c.w_fprop, zb, c.co, B, crop, c.k, c.rate, c.pad_b, x->ones,
                   h->params + c.b_off, ACT_NONE, fused_stats ? &fin : nullptr);
    }
    if (!fused_stats) {
      launch_pdl(h, bn_partial_kernel<TA, TA, 0>, dim3(nb_bn), dim3(BN_THREADS), 0, Z[l], c.co, 0, nullptr, 0, 0, nullptr, nullptr, 0, part_bn, c.co, M, bn_rows, fin);
      LAUNCH_CHECK(h);
    }
    if (h->sync_bn) {
      do_allreduce(h, x->sums, 2 * c.co);
      launch_pdl(h, bn_finalize_kernel, dim3(nblk(c.co, 128)), dim3(128), 0, x->sums, mean, istd, h->bnstat + c.mm_off, h->bnstat + c.mv_off, c.co,
                                                                  bn_count, h->cfg.bn_eps, h->cfg.bn_decay, h->cfg.bn_unbiased_ema);
      LAUNCH_CHECK(h);
    }
    // normalise + activation (+ pool).  Pooling nets: one kernel pools the raw conv output and normalises the winner.
    if (n.pool) {
      launch_maxpool3_fwd<TA>(h, Z[l], c.co, 0, Xn[l], c.co, 0, idx[l], c.co, B, crop, mean, istd, n.act);
    } else {
      ActBuf ab = output_of(l);
      ActBuf act_out = c.post ? ActBuf{Apre[l], c.co, 0} : ab;        // a post-op keeps the activation in front of it
      launch_pdl(h, bn_apply_kernel<TA>, dim3(bne_grid(M, h->sm_count)), dim3(BNE_THREADS), 0, Z[l], c.co, 0, mean, istd, n.act, (TA*)act_out.p, act_out.cs, act_out.co, c.co, M);
      LAUNCH_CHECK(h);
      if (c.post == 1) {
        launch_avgpool_fwd<TA>(h, Apre[l], c.co, 0, (TA*)ab.p, ab.cs, ab.co, c.co, B, crop, c.post_k);
      } else if (c.post == 2) {
        // squeeze-and-excitation (isprs:682-697): per-image channel means -> FC -> ReLU -> FC -> sigmoid -> gate
        const SeBlock& sb = n.se[c.se];
        SeBuf& q = seb[c.se];
        se_sum_kernel<TA, 0><<<dim3(B, (unsigned)ceil_div(sb.c, 64)), 256, 0, h->stream>>>(Apre[l], c.co, 0, nullptr, 0, 0, sb.c, crop * crop, q.sum);
        LAUNCH_CHECK(h);
        se_fc_fwd_kernel<<<B, 256, 0, h->stream>>>(q.sum, 1.0f / (float)(crop * crop), h->params + sb.w1_off, h->params + sb.b1_off,
                                                  h->params + sb.w2_off, h->params + sb.b2_off, sb.c, sb.r, q.s, q.hid, q.e);
        LAUNCH_CHECK(h);
        se_scale_fwd_kernel<TA><<<nblk(M * (c.co / 8), 256), 256, 0, h->stream>>>(Apre[l], c.co, 0, q.e, (TA*)ab.p, ab.cs, ab.co, c.co, M, crop * crop);
        LAUNCH_CHECK(h);
      }
    }
    {
      const ActBuf tb = output_of(l);
      h->taps[c.scope] = {tb.p, ElemTag<TA>::v, tb.cs, tb.co, c.co, M};
    }
  }
  ActBuf feat = n.dense ? ActBuf{F, n.feat_stride, 0}
                        : ActBuf{Xn[L - 1], n.convs[L - 1].out_cs > 0 ? n.convs[L - 1].out_cs : n.convs[L - 1].co, 0};
  launch_classifier_fwd<TA>(h, (const TA*)feat.p, feat.cs, feat.co, n.cls_in, h->params + n.cls_w_off, h->params + n.cls_b_off, K, logits,
                            pred, M);

  // ---------------------------------------------------------------- loss (isprs:1089-1099, contest:881-901)
  // the number of pixels in the mean stays on the device (x->loss_dev[3]); contest's mask count needs no host round trip
  if (mask_dev || h->ignore_label >= 0) {
    CUDA_CHECK(cudaMemsetAsync(x->count_dev, 0, 4, h->stream));
    h->pdl_prev = false;
    launch_pdl(h, mask_count_kernel, dim3((unsigned)std::min<int64_t>(ceil_div(M, 256), 1024)), dim3(256), 0, mask_dev, y_dev, h->ignore_label, M, x->count_dev);
    LAUNCH_CHECK(h);
    launch_pdl(h, set_count_kernel, dim3(1), dim3(1), 0, x->loss_dev + 3, x->count_dev, 0.0f);
    LAUNCH_CHECK(h);
    if (h->world > 1) do_allreduce(h, x->loss_dev + 3, 1);
  } else {
    launch_pdl(h, set_count_kernel, dim3(1), dim3(1), 0, x->loss_dev + 3, nullptr, (float)((double)M * h->world));
    LAUNCH_CHECK(h);
  }
  launch_pdl(h, ce_fwd_bwd_kernel, dim3(nb_ce), dim3(CE_THREADS), 0, logits, y_dev, mask_dev, K, M, x->loss_dev + 3, dlogits, part_ce, labels_u8, h->ignore_label);
  LAUNCH_CHECK(h);
  launch_pdl(h, sum_fixed_kernel, dim3(1), dim3(256), 0, part_ce, nb_ce, x->loss_dev, 1.0f, x->loss_dev + 3);
  LAUNCH_CHECK(h);
  // fused calc_accuracy_by_crop (isprs:510-531)
  CUDA_CHECK(cudaMemsetAsync(x->cm_dev, 0, (K * K + 1) * 4, h->stream));
  h->pdl_prev = false;
  launch_pdl(h, confusion_kernel, dim3((unsigned)std::min<int64_t>(ceil_div(M, 256), (int64_t)h->sm_count * 4)), dim3(256), 0, labels_u8, pred, acc_mask_dev ? acc_mask_dev : mask_dev, M, K, h->ignore_label, x->cm_dev);
  LAUNCH_CHECK(h);

  // ---------------------------------------------------------------- backward
  // Data parallel: the gradients of the last layers are complete long before the backward ends (they are computed first)
  // and hold most of the bytes (conv4..conv6 + classifier = 83 % of Dilated6Pooling), so that bucket -- with the loss
  // numerator and the confusion counts behind it -- is summed over ranks on a third stream while the backward of the
  // earlier layers runs; only the small front part of the buffer is exchanged at the end.
  const int l_split = (h->world > 1 && !h->time_convs && !getenv("DRS_NO_BUCKETS") && L >= 4) ? L - 3 : -1;
  // classifier: dW, db, dX
  launch_pdl(h, classifier_bwd_weight_kernel<TA>, dim3(nb_cls), dim3(CLSW_THREADS), 0, (const TA*)feat.p, feat.cs, feat.co, n.cls_in, dlogits, K, part_cls,
                                                                           part_clsb, M, cls_rows);
  LAUNCH_CHECK(h);
  launch_pdl(h, reduce_partials_kernel, dim3(reduce_partials_grid((int64_t)n.cls_in * K)), dim3(reduce_partials_block((int64_t)n.cls_in * K, nb_cls)), 0,
             part_cls, h->grads + n.cls_w_off, (int64_t)n.cls_in * K, nb_cls, (int64_t)0);
  LAUNCH_CHECK(h);
  launch_pdl(h, reduce_partials_kernel, dim3(reduce_partials_grid(K)), dim3(RP_COLS * RP_LANES), 0, part_clsb, h->grads + n.cls_b_off, K, nb_cls, (int64_t)0);
  LAUNCH_CHECK(h);
  if (l_split >= 0) {
    pack_extras_kernel<<<1, 128, 0, h->stream>>>(h->grads + n.n_trainable, x->loss_dev, x->cm_dev, K * K + 1);
    LAUNCH_CHECK(h);
    CUDA_CHECK(cudaEventRecord(x->ev_bucket_ready, h->stream));      // classifier gradients + extras are in the buffer
  }
  // squeeze net: one gradient buffer per output buffer (Gg), because a squeeze convolution's output feeds two layers
  TA* Gcur = n.dense ? GF : (n.squeeze ? Gg[L - 1] : G0);
  TA* Gnext = G1;
  const int gcs0 = n.dense ? n.feat_stride : n.cls_in;
  std::vector<char> grad_written(L, 0);        // squeeze: has the gradient buffer led by layer g been written in this step?
  {
    const int cvc = n.cls_in / 8;
    if (cvc <= 256 && ElemTag<TA>::v != ET_F32) {
      const int rows = 256 / cvc;
      // few, long-lived blocks (two per SM): a thread first loads its 8 x K weights (48 scalar loads), which must be amortised
      int blocks = (int)std::min<int64_t>(ceil_div(M, 2 * rows), (int64_t)h->sm_count * 2);
      launch_pdl(h, classifier_bwd_data_reg_kernel<TA>, dim3(blocks), dim3(256), 0, dlogits, h->params + n.cls_w_off, K, Gcur, gcs0, 0, n.cls_in, M);
    } else {
      int blocks = (int)std::min<int64_t>(ceil_div(M * (n.cls_in / 8), 256), (int64_t)h->sm_count * 16);
      classifier_bwd_data_kernel<TA><<<blocks, 256, n.cls_in * K * 4, h->stream>>>(dlogits, h->params + n.cls_w_off, K, Gcur, gcs0, 0, n.cls_in, M);
    }
    LAUNCH_CHECK(h);
  }
  int gcs = gcs0;   // channel stride of Gcur (non-dense)
  for (int l = L - 1; l >= 0; --l) {
    ConvLayer& c = n.convs[l];
    ActBuf dOut = n.dense ? ActBuf{GF, n.feat_stride, c.out_coff}
                : n.squeeze ? ActBuf{Gg[l], c.out_cs > 0 ? c.out_cs : c.co, c.out_cs > 0 ? c.out_coff : 0}
                            : ActBuf{Gcur, gcs, 0};
    ActBuf dA = dOut;
    float* mean = x->mean + c.mm_off;
    float* istd = x->inv_std + c.mm_off;
    BnFinish finb{x->bn_acc, 1099511627776.0, x->bn_counter, x->sums, nullptr, nullptr, nullptr, nullptr, bn_count, 0.0f, 0.0f, 0};
    // Pooling nets, bf16: two passes instead of four.  The BN-backward sums are taken on the pooled side (window gradients
    // and pooled activations: bn_partial_kernel MODE 2), then ONE kernel scatters the window gradients to their winners and
    // applies the BN backward to the finished fp32 row: the pool's input gradient is never written (it used to be stored as
    // bf16, read by the statistics pass and read again by bn_bwd_apply_kernel).
    const bool fused_pool_apply = n.pool && !n.dense && !n.squeeze && c.post == 0 && ElemTag<TA>::v == ET_BF16 && c.co <= 512 &&
                                  pool_lean_enabled() && !x->debug_keep && !getenv("DRS_NO_FUSED_POOL_APPLY");
    if (fused_pool_apply) {
      launch_pdl(h, bn_partial_kernel<TA, TA, 2>, dim3(nb_bn), dim3(BN_THREADS), 0, (const TA*)Xn[l], c.co, 0, (const TA*)dOut.p, dOut.cs, dOut.co,
                 (const float*)mean, (const float*)istd, n.act, part_bn, c.co, M, bn_rows, finb);
      LAUNCH_CHECK(h);
      if (h->sync_bn) do_allreduce(h, x->sums, 2 * c.co);
      TA* DZf = DZb[l & 1];
      if (l + 2 <= L - 1) {
        CUDA_CHECK(cudaStreamWaitEvent(h->stream, x->ev_wgrad[l & 1], 0));
        h->pdl_prev = false;
      }
      launch_maxpool3_bwd_apply(h, (const __nv_bfloat16*)dOut.p, dOut.cs, dOut.co, idx[l], (__nv_bfloat16*)DZf, c.co, 0, c.co, B, crop,
                                (const __nv_bfloat16*)Z[l], mean, istd, x->sums, 1.0 / bn_count, n.act);
    } else {
    if (n.pool) {
      launch_maxpool3_bwd<TA>(h, (const TA*)dOut.p, dOut.cs, dOut.co, idx[l], T, c.co, 0, c.co, B, crop);
      dA = ActBuf{T, c.co, 0};
    }
    if (c.post == 1) {
      launch_avgpool_bwd<TA>(h, (const TA*)dOut.p, dOut.cs, dOut.co, T, c.co, 0, c.co, B, crop, c.post_k);
      dA = ActBuf{T, c.co, 0};
    } else if (c.post == 2) {
      // gate backward: dA = dOut * e + ds,  ds from d(gate) = sum_px dOut * A through sigmoid, FC2, ReLU, FC1 and the mean;
      // the parameter gradients are per-image partials reduced in fixed order
      const SeBlock& sb = n.se[c.se];
      SeBuf& q = seb[c.se];
      se_sum_kernel<TA, 1><<<dim3(B, (unsigned)ceil_div(sb.c, 64)), 256, 0, h->stream>>>((const TA*)dOut.p, dOut.cs, dOut.co, Apre[l], c.co, 0, sb.c,
                                                                                      crop * crop, q.de);
      LAUNCH_CHECK(h);
      se_fc_bwd_kernel<<<B, 256, 0, h->stream>>>(q.de, q.s, q.hid, q.e, h->params + sb.w1_off, h->params + sb.w2_off, sb.c, sb.r,
                                                1.0f / (float)(crop * crop), q.ds, q.part);
      LAUNCH_CHECK(h);
      const int64_t np = (int64_t)2 * sb.c * sb.r + sb.r + sb.c;       // W1, b1, W2, b2 are contiguous in the flat buffer
      launch_pdl(h, reduce_partials_kernel, dim3(reduce_partials_grid(np)), dim3(RP_COLS * RP_LANES), 0, q.part, h->grads + sb.w1_off, np, B, (int64_t)0);
      LAUNCH_CHECK(h);
      se_scale_bwd_kernel<TA><<<nblk(M * (c.co / 8), 256), 256, 0, h->stream>>>((const TA*)dOut.p, dOut.cs, dOut.co, q.e, q.ds, T, c.co, 0, c.co, M,
                                                                              crop * crop);
      LAUNCH_CHECK(h);
      dA = ActBuf{T, c.co, 0};
    }
    launch_pdl(h, bn_partial_kernel<TA, TA, 1>, dim3(nb_bn), dim3(BN_THREADS), 0, (const TA*)Z[l], c.co, 0, (const TA*)dA.p, dA.cs, dA.co,
               (const float*)mean, (const float*)istd, n.act, part_bn, c.co, M, bn_rows, finb);
    LAUNCH_CHECK(h);
    if (h->sync_bn) do_allreduce(h, x->sums, 2 * c.co);
    // The filter gradient of layer l is off the critical path (only the optimizer needs it): it runs on a side stream and
    // overlaps the HBM-bound kernels of layer l-1's backward.  dZ is double-buffered; before a buffer is rewritten the
    // main stream waits for the wgrad that read it two layers ago.
    TA* DZ = DZb[l & 1];
    if (l + 2 <= L - 1) {
      CUDA_CHECK(cudaStreamWaitEvent(h->stream, x->ev_wgrad[l & 1], 0));
      h->pdl_prev = false;                 // the next kernel also depends on another stream
    }
    launch_pdl(h, bn_bwd_apply_kernel<TA, TA>, dim3(bne_grid(M, h->sm_count)), dim3(BNE_THREADS), 0, (const TA*)Z[l], c.co, 0, (const TA*)dA.p, dA.cs,
               dA.co, (const float*)mean, (const float*)istd, (const float*)x->sums, 1.0 / bn_count, n.act, DZ, c.co, 0, c.co, M);
    LAUNCH_CHECK(h);
    debug_keep<TA>(h, "da:" + c.scope, (const TA*)dA.p, dA.cs, dA.co, c.co, M);
    }
    TA* DZ = DZb[l & 1];
    debug_keep<TA>(h, "dz:" + c.scope, DZ, c.co, 0, c.co, M);
    CUDA_CHECK(cudaEventRecord(x->ev_dz[l & 1], h->stream));
    // wgrad (bias gradient is identically zero behind a BN without beta: sum_m dZ = 0)
    ActBuf xin = input_of(l);
    cudaStream_t main_stream = h->stream;
    // (per-launch kernel timing with events needs the launches serialised: no overlap while profiling)
    const bool overlap = !h->time_convs && !getenv("DRS_NO_OVERLAP");
    const bool pdl_main = h->pdl_prev;
    if (overlap) { h->stream = x->side_stream; h->pdl_prev = false; }
    try {
      if (overlap) CUDA_CHECK(cudaStreamWaitEvent(h->stream, x->ev_dz[l & 1], 0));
      if (l == 0 && xcol) {
        WgradTcArgs wa;
        wa.x = xcol; wa.in_cstride = 128; wa.in_coff = 0; wa.ci = 128;
        wa.dy = DZ; wa.dy_cstride = c.co; wa.dy_coff = 0; wa.co = c.co;
        wa.B = B; wa.crop = crop; wa.k = 1; wa.rate = 1; wa.pad_b = 0;
        wa.dw = h->grads + c.w_off; wa.part = part_w; wa.part_capacity = max_w * max_splits;
        wa.out_rows = c.k * c.k * c.ci;
        launch_wgrad_tc(h, wa);
      } else if (l == 0) {
        // conv1: K = 25*C <= 125 rows only -> parallelism must come from many short pixel splits
        // (fp32 mode keeps the generic kernel: its summation order is what the fp32 parity tests pin)
        const bool fast1 = ElemTag<TA>::v != ET_F32 &&
                           launch_wgrad_conv1<TA>(h, x_dev, n.channels, DZ, c.co, 0, c.co, h->grads + c.w_off, part_w, max_w * max_splits, B, crop, c.k, c.rate);
        if (!fast1) {
          const int conv1_splits = (int)std::min<int64_t>((int64_t)(max_w * max_splits) / ((int64_t)c.k * c.k * c.ci * c.co), 4 * h->sm_count);
          launch_wgrad_simt<float, TA>(h, x_dev, n.channels, 0, n.channels, DZ, c.co, 0, c.co, h->grads + c.w_off, part_w, conv1_splits, B, crop, c.k, c.rate, c.pad_b, 256);
        }
      } else if (ElemTag<TA>::v == ET_BF16 && wgrad_tc_supported(c.ci, c.co)) {
        WgradTcArgs wa;
        wa.x = xin.p; wa.in_cstride = xin.cs; wa.in_coff = xin.co; wa.ci = c.ci;
        wa.dy = DZ; wa.dy_cstride = c.co; wa.dy_coff = 0; wa.co = c.co;
        wa.B = B; wa.crop = crop; wa.k = c.k; wa.rate = c.rate; wa.pad_b = c.pad_b;
        wa.dw = h->grads + c.w_off; wa.part = part_w; wa.part_capacity = max_w * max_splits;
        cudaEvent_t ea = nullptr, eb = nullptr;
        prof_begin(h, &ea, &eb);
        launch_wgrad_tc(h, wa);
        prof_end(h, eb);
        x->conv_flops += 2.0 * (double)M * c.k * c.k * c.ci * c.co;
        x->conv_launches += 1;
      } else {
        launch_wgrad_simt<TA, TA>(h, (const TA*)xin.p, xin.cs, xin.co, c.ci, DZ, c.co, 0, c.co, h->grads + c.w_off, part_w, max_splits, B, crop, c.k, c.rate, c.pad_b);
      }
      CUDA_CHECK(cudaEventRecord(x->ev_wgrad[l & 1], h->stream));
      if (l == l_split) {
        // h->stream is the stream the filter gradients run on (in order: layers L-1..l_split are all complete behind it)
        CUDA_CHECK(cudaStreamWaitEvent(x->comm_stream, x->ev_wgrad[l & 1], 0));
        CUDA_CHECK(cudaStreamWaitEvent(x->comm_stream, x->ev_bucket_ready, 0));
        do_allreduce(h, h->grads + c.w_off, n.n_trainable + 2 + K * K - c.w_off, x->comm_stream);
        CUDA_CHECK(cudaEventRecord(x->ev_bucket_done, x->comm_stream));
      }
    } catch (...) { h->stream = main_stream; throw; }
    h->stream = main_stream;
    h->pdl_prev = overlap ? pdl_main : false;
    // dgrad: dilated conv of dZ with flipped taps, padding swapped
    if (l > 0) {
      ActBuf dzb{DZ, c.co, 0};
      if (n.dense) {
        ActBuf tmp{G0, c.ci, 0};
        run_conv<TA>(h, dzb, c.co, (const float*)c.w_dgrad, c.w_dgrad, tmp, c.ci, B, crop, c.k, c.rate, c.pad_a, x->ones, x->zeros, ACT_NONE);
        launch_pdl(h, add_slice_kernel<TA>, dim3(nblk(M * (c.ci / 8), 256)), dim3(256), 0, GF, n.feat_stride, 0, G0, c.ci, 0, c.ci, M);
        LAUNCH_CHECK(h);
      } else if (n.squeeze) {
        // gradient of the input buffer (led by layer `ig`): the first consumer processed writes it, the second adds
        const int ig = c.in_group >= 0 ? c.in_group : l - 1;
        if (!grad_written[ig]) {
          ActBuf gn{Gg[ig], c.ci, 0};
          run_conv<TA>(h, dzb, c.co, (const float*)c.w_dgrad, c.w_dgrad, gn, c.ci, B, crop, c.k, c.rate, c.pad_a, x->ones, x->zeros, ACT_NONE);
          grad_written[ig] = 1;
        } else {
          ActBuf tmp{G0, c.ci, 0};
          run_conv<TA>(h, dzb, c.co, (const float*)c.w_dgrad, c.w_dgrad, tmp, c.ci, B, crop, c.k, c.rate, c.pad_a, x->ones, x->zeros, ACT_NONE);
          launch_pdl(h, add_slice_kernel<TA>, dim3(nblk(M * (c.ci / 8), 256)), dim3(256), 0, Gg[ig], c.ci, 0, G0, c.ci, 0, c.ci, M);
          LAUNCH_CHECK(h);
        }
      } else {
        ActBuf gn{Gnext, c.ci, 0};
        run_conv<TA>(h, dzb, c.co, (const float*)c.w_dgrad, c.w_dgrad, gn, c.ci, B, crop, c.k, c.rate, c.pad_a, x->ones, x->zeros, ACT_NONE);
        std::swap(Gcur, Gnext);
        gcs = c.ci;
      }
    }
  }

  // join: every filter gradient is complete before the exchange / the optimizer (the side stream is in order, so the
  // two most recent events cover all layers)
  CUDA_CHECK(cudaStreamWaitEvent(h->stream, x->ev_wgrad[0], 0));
  if (L > 1) CUDA_CHECK(cudaStreamWaitEvent(h->stream, x->ev_wgrad[1], 0));
  h->pdl_prev = false;

  // ---------------------------------------------------------------- exchange + update
  if (h->world > 1) {
    if (l_split >= 0) {
      do_allreduce(h, h->grads, n.convs[l_split].w_off);             // conv1 .. conv(l_split): the small front part
      CUDA_CHECK(cudaStreamWaitEvent(h->stream, x->ev_bucket_done, 0));
    } else {
      pack_extras_kernel<<<1, 128, 0, h->stream>>>(h->grads + n.n_trainable, x->loss_dev, x->cm_dev, K * K + 1);
      LAUNCH_CHECK(h);
      do_allreduce(h, h->grads, n.n_trainable + 2 + K * K);
    }
    unpack_extras_kernel<<<1, 128, 0, h->stream>>>(h->grads + n.n_trainable, x->loss_dev, x->cm_dev, K * K + 1);
    LAUNCH_CHECK(h);
  }
  const float lr = h->cfg.lr_initial * powf(h->cfg.decay_rate, (float)(h->global_step / (h->cfg.decay_steps > 0 ? h->cfg.decay_steps : 1)));
  launch_pdl(h, momentum_update_kernel, dim3(nb_opt), dim3(256), 0, h->params, h->grads, h->moms, n.n_trainable, x->is_weight, h->cfg.weight_decay, lr,
                                                        h->cfg.momentum, 1.0f, part_l2);
  LAUNCH_CHECK(h);
  launch_pdl(h, sum_fixed_kernel, dim3(1), dim3(256), 0, part_l2, nb_opt, x->loss_dev + 1, 0.5f * h->cfg.weight_decay, nullptr);
  LAUNCH_CHECK(h);
  launch_pdl(h, add2_kernel, dim3(1), dim3(1), 0, x->loss_dev, x->loss_dev);
  LAUNCH_CHECK(h);
  h->global_step++;
  h->packed_dirty = true;
  h->eval_dirty = true;
  if (cm_out_dev) CUDA_CHECK(cudaMemcpyAsync(cm_out_dev, x->cm_dev, (K * K + 1) * 4, cudaMemcpyDeviceToDevice, h->stream));
  if (loss_host) {
    CUDA_CHECK(cudaMemcpyAsync(loss_host, x->loss_dev + 2, 4, cudaMemcpyDeviceToHost, h->stream));
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
  HandleExtra* x = X(h);
  const size_t es = h->cfg.precision == DRS_PREC_FP32 ? 4 : 2;
  TrainGraph* replay = nullptr;
  // (the legacy default stream cannot be captured)
  // (data parallel: capturable only when the exchange is the in-library NCCL call, not a host callback)
  const bool graphable = x->use_graphs && (h->world <= 1 || x->nccl) && !getenv("DRS_DEBUG_KEEP") &&
                         h->cfg.precision != DRS_PREC_F16 && h->stream != nullptr;
  if (!graphable) {
    if (capture_only) return;
    train_step_dispatch(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, pred_dev, cm_dev);
  } else {
    ensure_arena(h, train_workspace_bytes(h, B, crop, es));        // before the key: a re-allocation bumps arena_epoch
    const float lr = h->cfg.lr_initial * powf(h->cfg.decay_rate, (float)(h->global_step / (h->cfg.decay_steps > 0 ? h->cfg.decay_steps : 1)));
    TrainGraphKey key;
    memset(&key, 0, sizeof(key));
    key.B = B; key.crop = crop; key.ignore_label = h->ignore_label; key.profiling = h->time_convs ? 1 : 0;
    key.x = x_dev; key.y = y_dev; key.mask = mask_dev; key.acc_mask = acc_mask_dev; key.pred = pred_dev; key.cm = cm_dev;
    memcpy(&key.lr_bits, &lr, 4);
    key.arena_epoch = h->arena_epoch;
    auto it = x->graphs.find(key);
    if (it != x->graphs.end()) {
      replay = &it->second;
      h->launches += replay->launches;
      x->conv_flops += replay->conv_flops;
      x->conv_launches += replay->conv_launches;
      h->global_step++;
    } else {
      // capture (nothing executes while capturing), then launch like any later replay
      TrainGraph g;
      const int64_t l0 = h->launches, cl0 = x->conv_launches;
      const double f0 = x->conv_flops;
      h->packed_dirty = true;                        // the operand repack must be part of every replay
      CUDA_CHECK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
      x->capturing = &g;
      cudaGraph_t graph = nullptr;
      try {
        train_step_dispatch(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, pred_dev, cm_dev);
      } catch (...) {
        x->capturing = nullptr;
        cudaStreamEndCapture(h->stream, &graph);
        if (graph) cudaGraphDestroy(graph);
        throw;
      }
      x->capturing = nullptr;
      CUDA_CHECK(cudaStreamEndCapture(h->stream, &graph));
      cudaError_t e = cudaGraphInstantiate(&g.exec, graph, 0);
      cudaGraphDestroy(graph);
      CUDA_CHECK(e);
      CUDA_CHECK(cudaGraphUpload(g.exec, h->stream));   // pay the device-side set-up now, not at the first replay
      g.launches = h->launches - l0;
      g.conv_launches = x->conv_launches - cl0;
      g.conv_flops = x->conv_flops - f0;
      auto ins = x->graphs.emplace(key, g);
      replay = &ins.first->second;
      if (capture_only) {                            // drs_train_prepare: undo the host-side bookkeeping of the dry capture
        h->launches = l0;
        x->conv_launches = cl0;
        x->conv_flops = f0;
        h->global_step--;
        return;
      }
    }
    CUDA_CHECK(cudaGraphLaunch(replay->exec, h->stream));
    h->packed_dirty = true;
    h->eval_dirty = true;
  }
  if (loss_host) CUDA_CHECK(cudaMemcpyAsync(loss_host, x->loss_dev + 2, 4, cudaMemcpyDeviceToHost, h->stream));
  if (loss_host || (replay && h->time_convs)) {
    int rc = drs_synchronize(h);
    if (rc) throw DrsError{rc};
  }
  if (replay && h->time_convs) {
    for (auto& pr : replay->events) {
      float ms = 0.0f;
      CUDA_CHECK(cudaEventElapsedTime(&ms, pr.first, pr.second));
      x->conv_ms_acc += ms;
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
// unit-test entries for the backward pieces of the step (tests/test_gpu_parity.py): each runs exactly the launch sequence
// train_step_t uses for one layer, on caller-supplied tensors
// ------------------------------------------------------------------------------------------------
template <typename TA>
static void debug_dgrad_t(Handle* h, const float* dy32, const float* w32, int B, int crop, int k, int rate, int ci, int co, float* dx32) {
  const int64_t M = (int64_t)B * crop * crop;
  const int taps = k * k;
  const int64_t nw = (int64_t)taps * ci * co;
  const int pad_b = ((k - 1) * rate) / 2, pad_a = (k - 1) * rate - pad_b;
  HandleExtra* x = X(h);
  TA* dy = (TA*)arena_take(h, M * co * sizeof(TA));
  TA* dx = (TA*)arena_take(h, M * ci * sizeof(TA));
  void* wd = arena_take(h, nw * 4);
  cast_kernel<float, TA><<<nblk(M * co, 256), 256, 0, h->stream>>>(dy32, dy, M * co);
  LAUNCH_CHECK(h);
  // the dgrad operand exactly as refresh_packed builds it: taps flipped, Ci/Co transposed (kind 1 tensor cores, kind 2 fp32)
  RepackTable t;
  memset(&t, 0, sizeof(t));
  t.etype = ElemTag<TA>::v;
  t.seg[t.n++] = RepackSeg{w32, wd, taps, ci, co, ElemTag<TA>::v == ET_F32 ? 2 : 1, 0};
  t.total = nw;
  repack_kernel<<<nblk(nw, 256), 256, 0, h->stream>>>(t);
  LAUNCH_CHECK(h);
  // dgrad: dilated conv of dZ with flipped taps, before/after padding swapped (train_step_t)
  run_conv<TA>(h, ActBuf{dy, co, 0}, co, (const float*)wd, wd, ActBuf{dx, ci, 0}, ci, B, crop, k, rate, pad_a, x->ones, x->zeros, ACT_NONE);
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
  h->arena.reset();
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
// respect to the layer output.  Returns the layer output and dZ.  Same kernels, same order as train_step_t.
template <typename TA>
static void debug_layer_t(Handle* h, const float* z32, const float* dout32, int B, int crop, int C, int pool, int act, float* out32,
                          float* dz32, float* mean_out, float* istd_out) {
  const int64_t M = (int64_t)B * crop * crop;
  HandleExtra* x = X(h);
  TA* Z = (TA*)arena_take(h, M * C * sizeof(TA));
  TA* Xo = (TA*)arena_take(h, M * C * sizeof(TA));
  TA* G = (TA*)arena_take(h, M * C * sizeof(TA));
  TA* T = (TA*)arena_take(h, M * C * sizeof(TA));
  TA* DZ = (TA*)arena_take(h, M * C * sizeof(TA));
  uint8_t* idx = (uint8_t*)arena_take(h, M * C);
  const int nb_bn = (int)std::min<int64_t>(ceil_div(M, 128), (int64_t)h->sm_count * DRS_BN_MINBLK);
  const int bn_rows = (int)ceil_div(M, nb_bn);
  float* part_bn = (float*)arena_take(h, (size_t)nb_bn * 2 * 256 * 4);
  float* mean = x->mean;
  float* istd = x->inv_std;
  float* scratch_stats = (float*)arena_take(h, 4 * 512 * 4);      // moving statistics the finish step updates (discarded)
  CUDA_CHECK(cudaMemsetAsync(scratch_stats, 0, 4 * 512 * 4, h->stream));
  cast_kernel<float, TA><<<nblk(M * C, 256), 256, 0, h->stream>>>(z32, Z, M * C);
  LAUNCH_CHECK(h);
  cast_kernel<float, TA><<<nblk(M * C, 256), 256, 0, h->stream>>>(dout32, G, M * C);
  LAUNCH_CHECK(h);
  const double bn_count = (double)M;
  BnFinish fin{x->bn_acc, 1048576.0, x->bn_counter, x->sums, mean, istd, scratch_stats, scratch_stats + 512, bn_count, h->cfg.bn_eps,
               h->cfg.bn_decay, h->cfg.bn_unbiased_ema};
  bn_partial_kernel<TA, TA, 0><<<nb_bn, BN_THREADS, 0, h->stream>>>(Z, C, 0, nullptr, 0, 0, nullptr, nullptr, 0, part_bn, C, M, bn_rows, fin);
  LAUNCH_CHECK(h);
  if (pool) {
    launch_maxpool3_fwd<TA>(h, Z, C, 0, Xo, C, 0, idx, C, B, crop, mean, istd, act);
  } else {
    bn_apply_kernel<TA><<<bne_grid(M, h->sm_count), BNE_THREADS, 0, h->stream>>>(Z, C, 0, mean, istd, act, Xo, C, 0, C, M);
    LAUNCH_CHECK(h);
  }
  const TA* dA = G;
  BnFinish finb{x->bn_acc, 1099511627776.0, x->bn_counter, x->sums, nullptr, nullptr, nullptr, nullptr, bn_count, 0.0f, 0.0f, 0};
  // the training step's path for a pooling layer in bf16: sums from the pooled side, then pool backward + BN backward fused
  const bool fused = pool && ElemTag<TA>::v == ET_BF16 && pool_lean_enabled() && !getenv("DRS_NO_FUSED_POOL_APPLY");
  if (fused) {
    bn_partial_kernel<TA, TA, 2><<<nb_bn, BN_THREADS, 0, h->stream>>>(Xo, C, 0, G, C, 0, mean, istd, act, part_bn, C, M, bn_rows, finb);
    LAUNCH_CHECK(h);
    launch_maxpool3_bwd_apply(h, (const __nv_bfloat16*)G, C, 0, idx, (__nv_bfloat16*)DZ, C, 0, C, B, crop, (const __nv_bfloat16*)Z, mean, istd,
                              x->sums, 1.0 / bn_count, act);
  } else {
    if (pool) {
      launch_maxpool3_bwd<TA>(h, G, C, 0, idx, T, C, 0, C, B, crop);
      dA = T;
    }
    bn_partial_kernel<TA, TA, 1><<<nb_bn, BN_THREADS, 0, h->stream>>>(Z, C, 0, dA, C, 0, mean, istd, act, part_bn, C, M, bn_rows, finb);
    LAUNCH_CHECK(h);
    bn_bwd_apply_kernel<TA, TA><<<bne_grid(M, h->sm_count), BNE_THREADS, 0, h->stream>>>(Z, C, 0, dA, C, 0, mean, istd, x->sums, 1.0 / bn_count, act,
                                                                                   DZ, C, 0, C, M);
    LAUNCH_CHECK(h);
  }
  cast_kernel<TA, float><<<nblk(M * C, 256), 256, 0, h->stream>>>(Xo, out32, M * C);
  LAUNCH_CHECK(h);
  cast_kernel<TA, float><<<nblk(M * C, 256), 256, 0, h->stream>>>(DZ, dz32, M * C);
  LAUNCH_CHECK(h);
  CUDA_CHECK(cudaMemcpyAsync(mean_out, mean, C * 4, cudaMemcpyDeviceToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(istd_out, istd, C * 4, cudaMemcpyDeviceToDevice, h->stream));
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
  h->arena.reset();
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
  HandleExtra* x = X(h);
  const int K = h->net.classes;
  train_step(h, x_dev, y_dev, mask_dev, acc_mask_dev, B, crop, nullptr, pred_dev, nullptr);
  const int64_t t = x->next_ticket++;
  float* slot = x->result_host + (size_t)(t % HandleExtra::RESULT_RING) * RESULT_STRIDE;
  CUDA_CHECK(cudaMemcpyAsync(slot, x->loss_dev + 2, 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(slot + 1, x->cm_dev, (K * K + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaEventRecord(x->result_ev[t % HandleExtra::RESULT_RING], h->stream));
  *ticket_out = t;
  API_END
}

extern "C" int drs_train_result(drs_handle_t h, int64_t ticket, float* loss_out, uint32_t* cm_out) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  HandleExtra* x = X(h);
  DRS_CHECK(ticket >= 0 && ticket < x->next_ticket && ticket >= x->next_ticket - HandleExtra::RESULT_RING,
            "train_result: ticket %lld is not one of the last %d steps (next ticket %lld)", (long long)ticket,
            HandleExtra::RESULT_RING, (long long)x->next_ticket);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  CUDA_CHECK(cudaEventSynchronize(x->result_ev[ticket % HandleExtra::RESULT_RING]));
  const float* slot = x->result_host + (size_t)(ticket % HandleExtra::RESULT_RING) * RESULT_STRIDE;
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
  const size_t es = h->cfg.precision == DRS_PREC_FP32 ? 4 : 2;
  const int64_t M = (int64_t)B * crop_max * crop_max;
  const int C = h->net.channels, K = h->net.classes;
  ensure_arena(h, training ? std::max(train_workspace_bytes(h, B, crop_max, es), forward_eval_workspace(h, B, crop_max))
                           : forward_eval_workspace(h, B, crop_max));
  if (training) {
    // both device staging slots of the planned gather (drs_gather_plan_dev): worst case = every patch noisy
    HandleExtra* x = X(h);
    const size_t need = (size_t)M * C * 8 + (size_t)B * 128 + 8192;
    for (int s = 0; s < 2; ++s) {
      if (x->plan_stage_cap[s] >= need) continue;
      CUDA_CHECK(cudaStreamSynchronize(h->stream));
      CUDA_CHECK(cudaStreamSynchronize(x->plan_stream));
      if (x->plan_stage[s]) CUDA_CHECK(cudaFree(x->plan_stage[s]));
      x->plan_stage[s] = nullptr;
      x->plan_stage_cap[s] = 0;
      CUDA_CHECK(cudaMalloc(&x->plan_stage[s], need));
      x->plan_stage_cap[s] = need;
    }
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
  char* d = (char*)h->dstage;
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
