// Scene-resident entry points (gather, ordered accumulate + argmax, whole-scene inference, confusion)
// and the debug / profiling hooks.  Included by drs_api.cu.
#pragma once

static void scene_upload_rows(Handle* h, int32_t scene_id, const void* rows_host, int32_t H, int32_t W, int32_t C, int32_t dtype,
                              const uint8_t* labels_rows_host, int32_t row0, int32_t rows) {
  DRS_CHECK(h && rows_host, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  DRS_CHECK(scene_id >= 0 && scene_id < MAX_SCENES, "scene_id %d out of range [0,%d)", scene_id, MAX_SCENES);
  DRS_CHECK(dtype == DRS_SCENE_F64 || dtype == DRS_SCENE_F32, "bad scene dtype %d", dtype);
  DRS_CHECK(C == h->net.channels, "scene has %d channels, net expects %d", C, h->net.channels);
  DRS_CHECK(row0 >= 0 && rows >= 1 && row0 + rows <= H, "scene rows [%d,%d) outside [0,%d)", row0, row0 + rows, H);
  Scene& s = h->scenes[scene_id];
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  const size_t bytes = (size_t)rows * W * C * (dtype == DRS_SCENE_F64 ? 8 : 4);
  s.data.grow(bytes, bytes);
  CUDA_CHECK(cudaMemcpyAsync(s.data, rows_host, bytes, cudaMemcpyHostToDevice, h->stream));
  if (labels_rows_host) {
    s.labels.grow((size_t)rows * W, (size_t)rows * W);
    CUDA_CHECK(cudaMemcpyAsync(s.labels, labels_rows_host, (size_t)rows * W, cudaMemcpyHostToDevice, h->stream));
  } else {
    s.labels.reset();
  }
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  s.H = H; s.W = W; s.C = C; s.dtype = dtype; s.row0 = row0; s.rows = rows;
  h->table.s[scene_id] = SceneDesc{s.data, s.labels, H, W, C, dtype, row0, rows};
}

extern "C" int drs_scene_upload(drs_handle_t h, int32_t scene_id, const void* scene_host, int32_t H, int32_t W, int32_t C,
                                int32_t dtype, const uint8_t* labels_host) {
  API_BEGIN
  scene_upload_rows(h, scene_id, scene_host, H, W, C, dtype, labels_host, 0, H);
  API_END
}

extern "C" int drs_scene_upload_rows(drs_handle_t h, int32_t scene_id, const void* rows_host, int32_t H, int32_t W, int32_t C,
                                     int32_t dtype, const uint8_t* labels_rows_host, int32_t row0, int32_t rows) {
  API_BEGIN
  scene_upload_rows(h, scene_id, rows_host, H, W, C, dtype, labels_rows_host, row0, rows);
  API_END
}

extern "C" int drs_scene_free(drs_handle_t h, int32_t scene_id) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  auto it = h->scenes.find(scene_id);
  if (it == h->scenes.end()) return 0;
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  h->scenes.erase(it);
  memset(&h->table.s[scene_id], 0, sizeof(SceneDesc));
  API_END
}

extern "C" int drs_set_gather_fp16(drs_handle_t h, int32_t on) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  h->gather_fp16 = on ? 1 : 0;
  API_END
}

extern "C" int drs_set_normalization(drs_handle_t h, const double* mean3, const double* std3) {
  API_BEGIN
  DRS_CHECK(h && mean3 && std3, "null argument");
  for (int i = 0; i < 3; ++i) { h->norm_mean[i] = mean3[i]; h->norm_std[i] = std3[i]; }
  API_END
}

// all pointer members of gp are device pointers
static void launch_gather(Handle* h, GatherParams gp, const GatherInline* il = nullptr) {
  for (int i = 0; i < 3; ++i) { gp.mean[i] = h->norm_mean[i]; gp.stdv[i] = h->norm_std[i]; }
  gp.C = h->net.channels;
  gp.fp16_patches = h->gather_fp16;
  const int64_t n = (int64_t)gp.B * gp.crop * gp.crop * gp.C;
  if (il) {
    gather_kernel<true><<<nblk(n, 256), 256, 0, h->stream>>>(h->table, gp, *il);
  } else {
    static const GatherInline none = {};
    gather_kernel<false><<<nblk(n, 256), 256, 0, h->stream>>>(h->table, gp, none);
  }
  LAUNCH_CHECK(h);
}

static void gather_dev_impl(drs_handle_t h, const int32_t* inst_host, const uint8_t* flips_host, int32_t B, int32_t crop,
                            const double* noise_host, const uint8_t* noise_on_host, const double* over_x_host,
                            const uint8_t* over_y_host, const uint8_t* over_on_host, const double* rot_host,
                            const uint8_t* rot_on_host, float* x_out_dev, float* y_out_dev, uint8_t* amask_out_dev) {
  DRS_CHECK(h && inst_host && x_out_dev, "null argument");
  DRS_CHECK(B >= 1 && crop >= 1, "gather: empty batch (B=%d, crop=%d)", B, crop);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int C = h->net.channels;
  const int64_t pp = (int64_t)B * crop * crop;
  for (int b = 0; b < B; ++b) {
    const int sid = inst_host[b * 3], r = inst_host[b * 3 + 1], c = inst_host[b * 3 + 2];
    const bool over = over_on_host && over_on_host[b];
    if (over) continue;
    auto it = h->scenes.find(sid);
    DRS_CHECK(it != h->scenes.end(), "gather: scene %d not uploaded", sid);
    DRS_CHECK(r >= 0 && c >= 0 && r + crop <= it->second.H && c + crop <= it->second.W,
              "Error: Current PATCH size is out of the scene (scene %d, row %d, col %d, crop %d)", sid, r, c, crop);
    DRS_CHECK(r >= it->second.row0 && r + crop <= it->second.row0 + it->second.rows,
              "gather: rows [%d,%d) of scene %d are not resident (uploaded rows [%d,%d))", r, r + crop, sid, it->second.row0,
              it->second.row0 + it->second.rows);
  }
  const bool plain = !(noise_host && noise_on_host) && !(over_x_host && over_on_host) && !(rot_host && rot_on_host);
  if (plain && B <= GATHER_INLINE_MAX) {
    // common case (no host-made noise / rotation overrides): everything travels in the kernel parameters
    GatherInline il;
    memset(&il, 0, sizeof(il));
    memcpy(il.inst, inst_host, (size_t)B * 12);
    if (flips_host) memcpy(il.flips, flips_host, B);
    GatherParams gp;
    memset(&gp, 0, sizeof(gp));
    gp.x_out = x_out_dev;
    gp.y_out = y_out_dev;
    gp.amask_out = amask_out_dev;
    gp.B = B;
    gp.crop = crop;
    launch_gather(h, gp, &il);
    return;
  }
  size_t need = round_up((size_t)B * 3 * 4, 256) + 4 * round_up((size_t)B, 256) + round_up((size_t)B * 48, 256);
  if (noise_host) need += round_up((size_t)pp * C * 8, 256);
  if (over_x_host) need += round_up((size_t)pp * C * 8, 256) + round_up((size_t)pp, 256);
  ensure_dstage(h, need + 1024);
  char* d = h->dstage;
  GatherParams gp;
  memset(&gp, 0, sizeof(gp));
  auto put = [&](const void* src, size_t bytes) -> void* {
    void* dst = d;
    CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
    d += round_up(bytes, 256);
    return dst;
  };
  gp.inst = (const int32_t*)put(inst_host, (size_t)B * 12);
  if (flips_host) gp.flips = (const uint8_t*)put(flips_host, B);
  if (noise_host && noise_on_host) {
    gp.noise_on = (const uint8_t*)put(noise_on_host, B);
    gp.noise = (const double*)put(noise_host, (size_t)pp * C * 8);
  }
  if (over_x_host && over_on_host) {
    gp.over_on = (const uint8_t*)put(over_on_host, B);
    gp.over_x = (const double*)put(over_x_host, (size_t)pp * C * 8);
    if (over_y_host) gp.over_y = (const uint8_t*)put(over_y_host, (size_t)pp);
  }
  if (rot_host && rot_on_host) {
    gp.rot_on = (const uint8_t*)put(rot_on_host, B);
    gp.rot = (const double*)put(rot_host, (size_t)B * 48);
  }
  gp.x_out = x_out_dev;
  gp.y_out = y_out_dev;
  gp.amask_out = amask_out_dev;
  gp.B = B;
  gp.crop = crop;
  launch_gather(h, gp);
  // the staging buffer is reused by the next call: the copies above must have been consumed
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
}

extern "C" int drs_gather_dev(drs_handle_t h, const int32_t* inst_host, const uint8_t* flips_host, int32_t B, int32_t crop,
                              const double* noise_host, const uint8_t* noise_on_host, const double* over_x_host,
                              const uint8_t* over_y_host, const uint8_t* over_on_host, float* x_out_dev, float* y_out_dev) {
  API_BEGIN
  gather_dev_impl(h, inst_host, flips_host, B, crop, noise_host, noise_on_host, over_x_host, over_y_host, over_on_host, nullptr,
                  nullptr, x_out_dev, y_out_dev, nullptr);
  API_END
}

extern "C" int drs_gather_rot_dev(drs_handle_t h, const int32_t* inst_host, const uint8_t* flips_host, int32_t B, int32_t crop,
                                  const double* noise_host, const uint8_t* noise_on_host, const double* rot_host,
                                  const uint8_t* rot_on_host, float* x_out_dev, float* y_out_dev, uint8_t* amask_out_dev) {
  API_BEGIN
  gather_dev_impl(h, inst_host, flips_host, B, crop, noise_host, noise_on_host, nullptr, nullptr, nullptr, rot_host, rot_on_host,
                  x_out_dev, y_out_dev, amask_out_dev);
  API_END
}

// The gather of a planned batch (drs_plan_isprs_batch) without any host synchronisation: the plan's arrays (page-locked
// host memory owned by the caller, untouched until the step's result has been fetched) are copied on plan_stream into one
// of two device staging slots and the gather is ordered behind that copy with an event; a staging slot is rewritten only
// after the gather that read it two calls ago has run.
extern "C" int drs_gather_plan_dev(drs_handle_t h, const int32_t* inst_host, const uint8_t* flips_host, int32_t B, int32_t crop,
                                   const uint8_t* rot_on_host, const double* rot_host, const uint8_t* noise_on_host,
                                   const int32_t* noise_slot_host, const double* noise_host, int64_t noise_count,
                                   float* x_out_dev, float* y_out_dev, uint8_t* amask_out_dev) {
  API_BEGIN
  DRS_CHECK(h && inst_host && x_out_dev, "null argument");
  DRS_CHECK(B >= 1 && crop >= 1, "gather_plan: bad B=%d crop=%d", B, crop);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  for (int b = 0; b < B; ++b) {
    const int sid = inst_host[b * 3], r = inst_host[b * 3 + 1], c = inst_host[b * 3 + 2];
    auto it = h->scenes.find(sid);
    DRS_CHECK(it != h->scenes.end(), "gather: scene %d not uploaded", sid);
    DRS_CHECK(r >= it->second.row0 && r + crop <= it->second.row0 + it->second.rows && c >= 0 && c + crop <= it->second.W,
              "Error: Current PATCH size is out of the resident scene rows (scene %d, row %d, col %d, crop %d)", sid, r, c, crop);
  }
  const bool has_noise = noise_host && noise_on_host && noise_slot_host && noise_count > 0;
  const bool has_rot = rot_host && rot_on_host;
  const size_t small = round_up((size_t)B * 12, 256) + 3 * round_up((size_t)B, 256) + round_up((size_t)B * 4, 256) +
                       round_up((size_t)B * 48, 256);
  const size_t need = small + (has_noise ? round_up((size_t)noise_count * 8, 256) : 0) + 1024;
  const int s = (int)(h->plan_calls++ & 1);
  if (h->plan_consumed_valid[s]) CUDA_CHECK(cudaStreamWaitEvent(h->plan_stream, h->plan_consumed[s], 0));
  h->plan_stage[s].grow(need, need + (need >> 1), {h->stream, h->plan_stream});
  char* d = h->plan_stage[s];
  auto put = [&](const void* src, size_t bytes) -> void* {
    void* dst = d;
    CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->plan_stream));
    d += round_up(bytes, 256);
    return dst;
  };
  GatherParams gp;
  memset(&gp, 0, sizeof(gp));
  gp.inst = (const int32_t*)put(inst_host, (size_t)B * 12);
  if (flips_host) gp.flips = (const uint8_t*)put(flips_host, B);
  if (has_rot) {
    gp.rot_on = (const uint8_t*)put(rot_on_host, B);
    gp.rot = (const double*)put(rot_host, (size_t)B * 48);
  }
  if (has_noise) {
    gp.noise_on = (const uint8_t*)put(noise_on_host, B);
    gp.noise_slot = (const int32_t*)put(noise_slot_host, (size_t)B * 4);
    gp.noise = (const double*)put(noise_host, (size_t)noise_count * 8);
  }
  CUDA_CHECK(cudaEventRecord(h->plan_uploaded[s], h->plan_stream));
  CUDA_CHECK(cudaStreamWaitEvent(h->stream, h->plan_uploaded[s], 0));
  gp.x_out = x_out_dev;
  gp.y_out = y_out_dev;
  gp.amask_out = amask_out_dev;
  gp.B = B;
  gp.crop = crop;
  launch_gather(h, gp);
  CUDA_CHECK(cudaEventRecord(h->plan_consumed[s], h->stream));
  h->plan_consumed_valid[s] = true;
  API_END
}

// host-only: the visiting order of create_patches_per_map (no GPU needed)
extern "C" int drs_grid_positions(int32_t H, int32_t W, int32_t crop, int32_t batch, int32_t variant, int32_t* pos_out,
                                  int64_t cap_pairs, int64_t* n_out) {
  API_BEGIN
  std::vector<int32_t> pos;
  grid_positions(H, W, crop, batch, variant, pos);
  const int64_t n = (int64_t)pos.size() / 2;
  if (n_out) *n_out = n;
  if (pos_out) {
    DRS_CHECK(cap_pairs >= n, "grid_positions: capacity %lld < %lld", (long long)cap_pairs, (long long)n);
    memcpy(pos_out, pos.data(), pos.size() * 4);
  }
  API_END
}

static void build_cells(const std::vector<int32_t>& pos, int H, int W, int crop, CellTables& ct) {
  const int stride = crop / 2;
  ct.stride = stride;
  ct.nh = grid_count(H, crop, stride);
  ct.nw = grid_count(W, crop, stride);
  const int ncell = ct.nh * ct.nw;
  const int64_t P = (int64_t)pos.size() / 2;
  std::vector<int32_t> cell_of(P);
  ct.off.assign(ncell + 1, 0);
  for (int64_t p = 0; p < P; ++p) {
    const int y0 = pos[2 * p], x0 = pos[2 * p + 1];
    int i = (y0 % stride == 0 && y0 / stride < ct.nh) ? y0 / stride : -1;
    int j = (x0 % stride == 0 && x0 / stride < ct.nw) ? x0 / stride : -1;
    if (y0 == H - crop) i = ct.nh - 1;
    if (x0 == W - crop) j = ct.nw - 1;
    DRS_CHECK(i >= 0 && j >= 0, "accumulate: position (%d,%d) is not on the sliding-window lattice", y0, x0);
    cell_of[p] = i * ct.nw + j;
    ct.off[cell_of[p] + 1]++;
  }
  for (int c = 0; c < ncell; ++c) ct.off[c + 1] += ct.off[c];
  ct.seq.assign(P, 0);
  std::vector<int32_t> fill(ct.off.begin(), ct.off.end() - 1);
  for (int64_t p = 0; p < P; ++p) ct.seq[fill[cell_of[p]]++] = (int32_t)p;   // ascending visit order per cell
}

// Visit ranges [cuts[r], cuts[r+1]) accumulated by one launch each: every chunk of `chunk` visits starts a range, and a
// range ends before the visit that would give one of its pixels more than ACCUM_MAX_CONTRIB contributions.  The contest
// grid visits a cell up to 3 times on a contest-shaped scene and up to 11 times on a tall one, so a chunk may need several
// launches; the isprs grid and the coffee grid (square tiles) visit every cell once and never split a chunk.  Pixels
// between two consecutive patch borders of each axis are covered by the same patches, so the counts are kept per pair of
// such segments.
static void accum_ranges(const std::vector<int32_t>& pos, int H, int W, int crop, int chunk, std::vector<int32_t>& cuts) {
  const int P = (int)(pos.size() / 2);
  std::vector<int32_t> seg[2];                       // segment of every row / column
  int nseg[2];
  for (int a = 0; a < 2; ++a) {
    const int L = a ? W : H;
    std::vector<uint8_t> border(L + 1, 0);
    for (int p = 0; p < P; ++p) { border[pos[2 * p + a]] = 1; border[pos[2 * p + a] + crop] = 1; }
    seg[a].resize(L);
    int s = 0;
    for (int y = 0; y < L; ++y) { if (y > 0 && border[y]) ++s; seg[a][y] = s; }
    nseg[a] = s + 1;
  }
  std::vector<uint16_t> cnt((size_t)nseg[0] * nseg[1], 0);
  std::vector<int32_t> stamp((size_t)nseg[0] * nseg[1], -1);    // range whose visits cnt[] counts
  cuts.clear();
  for (int p = 0; p < P; ++p) {
    const int r0 = seg[0][pos[2 * p]], r1 = seg[0][pos[2 * p] + crop - 1];
    const int c0 = seg[1][pos[2 * p + 1]], c1 = seg[1][pos[2 * p + 1] + crop - 1];
    bool full = p % chunk == 0;
    for (int r = r0; r <= r1 && !full; ++r)
      for (int c = c0; c <= c1 && !full; ++c) {
        const size_t i = (size_t)r * nseg[1] + c;
        full = stamp[i] == (int32_t)cuts.size() - 1 && cnt[i] >= ACCUM_MAX_CONTRIB;
      }
    if (full) cuts.push_back(p);
    const int32_t range = (int32_t)cuts.size() - 1;
    for (int r = r0; r <= r1; ++r)
      for (int c = c0; c <= c1; ++c) {
        const size_t i = (size_t)r * nseg[1] + c;
        if (stamp[i] != range) { stamp[i] = range; cnt[i] = 0; }
        ++cnt[i];
      }
  }
  cuts.push_back(P);
}

static void accumulate_chunk(Handle* h, const CellTables& ct, const float* logits, const std::vector<int32_t>& pos,
                             int seq0, int seq1, int H, int W, int K, int crop, int row_begin, int row_end) {
  int y_lo = H, y_hi = 0;
  for (int s = seq0; s < seq1; ++s) {
    y_lo = std::min(y_lo, pos[2 * s]);
    y_hi = std::max(y_hi, pos[2 * s] + crop);
  }
  y_lo = std::max(y_lo, row_begin);
  y_hi = std::min(y_hi, row_end);
  if (y_hi <= y_lo) return;
  AccumParams ap;
  ap.logits = logits; ap.cell_off = h->pass.cell_off; ap.cell_seq = h->pass.cell_seq; ap.prob = h->pass.prob; ap.occur = h->pass.occur;
  ap.H = H; ap.W = W; ap.K = K; ap.crop = crop; ap.stride = ct.stride; ap.nh = ct.nh; ap.nw = ct.nw;
  ap.row_begin = row_begin; ap.row_end = row_end; ap.y_lo = y_lo; ap.y_hi = y_hi; ap.seq0 = seq0; ap.seq1 = seq1;
  ap.overflow = h->diag_dev + 15;
  dim3 grid(nblk(W, 128), (unsigned)(y_hi - y_lo));
  accumulate_kernel<<<grid, 128, 0, h->stream>>>(ap);
  LAUNCH_CHECK(h);
}

static void scene_pass_begin(Handle* h, const CellTables& ct, int rows, int W, int K) {
  float* prob = pass_buf(h, h->pass.prob, (size_t)rows * W * K * 4);
  uint32_t* occur = pass_buf(h, h->pass.occur, (size_t)rows * W * 4);
  int32_t* cell_off = pass_buf(h, h->pass.cell_off, ct.off.size() * 4);
  int32_t* cell_seq = pass_buf(h, h->pass.cell_seq, std::max<size_t>(ct.seq.size(), 1) * 4);
  CUDA_CHECK(cudaMemsetAsync(prob, 0, (size_t)rows * W * K * 4, h->stream));
  CUDA_CHECK(cudaMemsetAsync(occur, 0, (size_t)rows * W * 4, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(cell_off, ct.off.data(), ct.off.size() * 4, cudaMemcpyHostToDevice, h->stream));
  if (!ct.seq.empty()) CUDA_CHECK(cudaMemcpyAsync(cell_seq, ct.seq.data(), ct.seq.size() * 4, cudaMemcpyHostToDevice, h->stream));
}

// after the pass's stream has been synchronised
static void accum_overflow_check(Handle* h) {
  if (h->diag_host[15]) {
    h->diag_host[15] = 0;
    DRS_FAIL("accumulate: a pixel is covered by more than %d patch visits in one accumulation launch; the label map would be wrong", ACCUM_MAX_CONTRIB);
  }
}

static void scene_pass_finish(Handle* h, int rows, int W, int K, uint8_t* labels_host, double* mean_host) {
  const int64_t npix = (int64_t)rows * W;
  uint8_t* lab_dev = pass_buf(h, h->pass.labels, npix);
  double* mean_dev = mean_host ? pass_buf(h, h->pass.mean, npix * K * 8) : nullptr;
  scene_argmax_kernel<<<nblk(npix, 256), 256, 0, h->stream>>>(h->pass.prob, h->pass.occur, npix, K, lab_dev, mean_dev);
  LAUNCH_CHECK(h);
  if (labels_host) CUDA_CHECK(cudaMemcpyAsync(labels_host, lab_dev, npix, cudaMemcpyDeviceToHost, h->stream));
  if (mean_host) CUDA_CHECK(cudaMemcpyAsync(mean_host, mean_dev, npix * K * 8, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  accum_overflow_check(h);
}

extern "C" int drs_accumulate_argmax(drs_handle_t h, const float* logits_dev, const int32_t* pos_host, int32_t P, int32_t crop,
                                     int32_t K, int32_t H, int32_t W, uint8_t* labels_out_host, double* mean_out_host) {
  API_BEGIN
  DRS_CHECK(h && logits_dev && pos_host && labels_out_host, "null argument");
  DRS_CHECK(K >= 1 && K <= MAX_CLASSES, "K=%d out of range", K);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  std::vector<int32_t> pos(pos_host, pos_host + (size_t)P * 2);
  CellTables ct;
  build_cells(pos, H, W, crop, ct);
  std::vector<int32_t> cuts;
  accum_ranges(pos, H, W, crop, std::max(P, 1), cuts);
  scene_pass_begin(h, ct, H, W, K);
  for (size_t r = 0; r + 1 < cuts.size(); ++r)
    accumulate_chunk(h, ct, logits_dev + (size_t)cuts[r] * crop * crop * K, pos, cuts[r], cuts[r + 1], H, W, K, crop, 0, H);
  scene_pass_finish(h, H, W, K, labels_out_host, mean_out_host);
  API_END
}

// The chunks of a scene run on a lane of their own (stream + workspace); the ordered accumulation stays on the handle's
// stream, chunk after chunk, so per-pixel sums keep the script's visiting order.  The lane is kept in the handle between
// calls (its workspace is several GB for a Potsdam tile).
static void lane_ensure(Handle* h, size_t arena_bytes, size_t x_bytes, size_t lg_bytes) {
  if (!h->lane_ready) h->lane_ready = new_event();
  InferLane& L = h->lane;
  if (!L.stream) {
    L.stream = new_stream();
    L.fwd_done = new_event();
    L.acc_done = new_event();
  }
  L.arena.mem.grow(arena_bytes, arena_bytes, {L.stream});
  L.x.grow(x_bytes, x_bytes, {L.stream});
  L.lg.grow(lg_bytes, lg_bytes, {L.stream, h->stream});   // the accumulation of an earlier pass may still read the logits
}

// Streamed upload of a host scene during a scene pass: rows are copied on a separate stream, in ~8 MB pieces, just ahead of
// the chunk that first reads them, so the host->device transfer of a fresh tile (1.44 GB for a Potsdam tile) overlaps the
// convolutions instead of preceding them.
struct HostSceneFeed {
  const char* host = nullptr;    // [H,W,C] in the scene dtype, row-major
  size_t row_bytes = 0;
  int uploaded = 0;              // rows [0, uploaded) are enqueued
  bool recorded = false;         // up_ev has been recorded at least once during this pass
};

static void feed_rows(Handle* h, HostSceneFeed& f, const Scene& sc, int rows_needed, cudaStream_t consumer) {
  if (rows_needed > sc.H) rows_needed = sc.H;
  bool any = false;
  const int rows_per_piece = (int)std::max<size_t>(1, ((size_t)8 << 20) / f.row_bytes);
  while (f.uploaded < rows_needed) {
    const int n = std::min(rows_per_piece, rows_needed - f.uploaded);
    // Pageable source: the driver stages the piece itself (measured faster than a memcpy into our own pinned ring) and
    // returns once the source has been read; kernels already queued keep the GPU busy meanwhile.
    CUDA_CHECK(cudaMemcpyAsync((char*)sc.data.get() + (size_t)f.uploaded * f.row_bytes, f.host + (size_t)f.uploaded * f.row_bytes,
                               (size_t)n * f.row_bytes, cudaMemcpyHostToDevice, h->copy_stream));
    f.uploaded += n;
    any = true;
  }
  if (any) {
    CUDA_CHECK(cudaEventRecord(h->up_ev, h->copy_stream));
    f.recorded = true;
  }
  // The consumer waits for the latest "rows uploaded" event (copies on one stream complete in order, so it covers every
  // earlier piece).
  if (f.recorded) CUDA_CHECK(cudaStreamWaitEvent(consumer, h->up_ev, 0));
}

static void scene_infer_impl(drs_handle_t h, int32_t scene_id, int32_t crop, int32_t batch, int32_t variant, int32_t row_begin,
                             int32_t row_end, uint8_t* labels_out_host, double* mean_out_host, HostSceneFeed* feed);

extern "C" int drs_scene_infer(drs_handle_t h, int32_t scene_id, int32_t crop, int32_t batch, int32_t variant, int32_t row_begin,
                               int32_t row_end, uint8_t* labels_out_host, double* mean_out_host) {
  API_BEGIN
  scene_infer_impl(h, scene_id, crop, batch, variant, row_begin, row_end, labels_out_host, mean_out_host, nullptr);
  API_END
}

extern "C" int drs_scene_infer_host(drs_handle_t h, int32_t scene_id, const void* scene_host, int32_t H, int32_t W, int32_t C,
                                    int32_t dtype, int32_t crop, int32_t batch, int32_t variant, uint8_t* labels_out_host,
                                    double* mean_out_host) {
  API_BEGIN
  DRS_CHECK(h && scene_host && labels_out_host, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  DRS_CHECK(scene_id >= 0 && scene_id < MAX_SCENES, "scene_id %d out of range [0,%d)", scene_id, MAX_SCENES);
  DRS_CHECK(dtype == DRS_SCENE_F64 || dtype == DRS_SCENE_F32, "bad scene dtype %d", dtype);
  DRS_CHECK(C == h->net.channels, "scene has %d channels, net expects %d", C, h->net.channels);
  Scene& s = h->scenes[scene_id];
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  const size_t row_bytes = (size_t)W * C * (dtype == DRS_SCENE_F64 ? 8 : 4);
  const size_t bytes = row_bytes * H;
  s.data.grow(bytes, bytes);
  s.labels.reset();
  s.H = H; s.W = W; s.C = C; s.dtype = dtype; s.row0 = 0; s.rows = H;
  h->table.s[scene_id] = SceneDesc{s.data, s.labels, H, W, C, dtype, 0, H};
  if (!h->copy_stream) h->copy_stream = new_stream();
  if (!h->up_ev) h->up_ev = new_event();
  HostSceneFeed feed;
  feed.host = (const char*)scene_host;
  feed.row_bytes = row_bytes;
  scene_infer_impl(h, scene_id, crop, batch, variant, 0, H, labels_out_host, mean_out_host, &feed);
  API_END
}

static PassGeometry& pass_geometry(Handle* h, int scene_id, int H, int W, int crop, int batch, int variant, int row_begin, int row_end) {
  std::vector<PassGeometry>& cache = h->pass_geometry;
  const int key[8] = {scene_id, H, W, crop, batch, variant, row_begin, row_end};
  for (auto& g : cache)
    if (memcmp(g.key, key, sizeof(key)) == 0) return g;
  std::vector<int32_t> all;
  grid_positions(H, W, crop, batch, variant, all);   // throws for a crop that does not fit: nothing is cached then
  if (cache.size() >= 8) cache.erase(cache.begin());
  cache.emplace_back();
  PassGeometry& g = cache.back();
  memcpy(g.key, key, sizeof(key));
  for (size_t p = 0; p < all.size() / 2; ++p)
    if (all[2 * p] < row_end && all[2 * p] + crop > row_begin) { g.pos.push_back(all[2 * p]); g.pos.push_back(all[2 * p + 1]); }
  build_cells(g.pos, H, W, crop, g.ct);
  const size_t P = g.pos.size() / 2;
  g.inst.resize(P * 3);
  for (size_t p = 0; p < P; ++p) { g.inst[3 * p] = scene_id; g.inst[3 * p + 1] = g.pos[2 * p]; g.inst[3 * p + 2] = g.pos[2 * p + 1]; }
  return g;
}

// The geometry of a pass of `crop` over rows [row_begin, row_end) of a resident scene (row bounds already clipped), checked
// against the rows that are resident, with its accumulation ranges for the current chunk size.  Launches nothing.
static PassGeometry& scene_pass_geometry(Handle* h, const Scene& sc, int32_t scene_id, int32_t crop, int32_t batch,
                                         int32_t variant, int32_t row_begin, int32_t row_end) {
  const int H = sc.H, W = sc.W;
  // visiting order of the script, restricted to patches that touch the stripe (order preserved), with its per-cell visit
  // tables: pure functions of the geometry, memoised (a validation run visits the same scenes with the same crop again
  // and again; for a 6000x6000 tile they take several milliseconds of host time per call)
  PassGeometry& pg = pass_geometry(h, scene_id, H, W, crop, batch, variant, row_begin, row_end);
  const std::vector<int32_t>& pos = pg.pos;
  const int P = (int)(pos.size() / 2);
  for (int p = 0; p < P; ++p)
    DRS_CHECK(pos[2 * p] >= sc.row0 && pos[2 * p] + crop <= sc.row0 + sc.rows,
              "scene_infer: stripe [%d,%d) needs scene rows [%d,%d) but only [%d,%d) are resident", row_begin, row_end, pos[2 * p],
              pos[2 * p] + crop, sc.row0, sc.row0 + sc.rows);
  // chunk = a whole number of 128-pixel tiles close to a multiple of the SM count (full conv waves), ~0.75 M pixels
  const int64_t pp = (int64_t)crop * crop;
  const int waves = getenv("DRS_CHUNK_WAVES") ? std::max(1, atoi(getenv("DRS_CHUNK_WAVES"))) : 40;
  const int64_t target_tiles = (int64_t)h->sm_count * waves;
  int chunk = (int)std::max<int64_t>(1, std::min<int64_t>(P, (target_tiles * CONV_TC_BM) / pp));
  if (pg.chunk != chunk) {
    accum_ranges(pos, H, W, crop, chunk, pg.cuts);
    pg.chunk = chunk;
  }
  return pg;
}

// The loop of a scene pass: prob / occur cleared, then gather, forward and ordered accumulation of every chunk.  The caller
// turns h->pass.prob / occur into labels (scene_pass_finish, or the multi-scale softmax) on the handle's stream.
static void scene_pass_accumulate(Handle* h, const Scene& sc, const PassGeometry& pg, int32_t crop, int32_t row_begin,
                                  int32_t row_end, HostSceneFeed* feed) {
  const int H = sc.H, W = sc.W, K = h->net.classes, C = h->net.channels;
  const std::vector<int32_t>& pos = pg.pos;
  const CellTables& ct = pg.ct;
  const int P = (int)(pos.size() / 2);
  const int rows = row_end - row_begin;
  const int64_t pp = (int64_t)crop * crop;
  const int chunk = pg.chunk;
  const std::vector<int32_t>& cuts = pg.cuts;
  const cudaStream_t main_stream = h->stream;
  scene_pass_begin(h, ct, rows, W, K);
  const std::vector<int32_t>& inst = pg.inst;
  int32_t* inst_dev = pass_buf(h, h->pass.inst, std::max<size_t>(inst.size(), 1) * 4);
  CUDA_CHECK(cudaMemcpyAsync(inst_dev, inst.data(), inst.size() * 4, cudaMemcpyHostToDevice, h->stream));
  refresh_packed(h, false);                       // packed weights / folded BN once, before the lane starts
  lane_ensure(h, eval_arena_bytes(h, chunk, crop), (size_t)chunk * pp * C * 4, (size_t)chunk * pp * K * 4);
  InferLane& L = h->lane;
  CUDA_CHECK(cudaEventRecord(h->lane_ready, main_stream));
  CUDA_CHECK(cudaStreamWaitEvent(L.stream, h->lane_ready, 0));
  size_t r = 0;                                    // next accumulation range
  for (int s0 = 0; s0 < P; s0 += chunk) {
    const int nb = std::min(chunk, P - s0);
    {                                              // gather + forward of the chunk on the lane
      StreamScope on_lane(h, true, L.stream, &L.arena);
      if (s0 > 0) CUDA_CHECK(cudaStreamWaitEvent(L.stream, L.acc_done, 0));   // logits buffer of the previous chunk consumed
      if (feed) {
        // rows this chunk's patches read, plus one more chunk's worth so that the copy runs ahead of the compute
        int need = 0;
        const int s1 = std::min(P, s0 + 2 * chunk);
        for (int s = s0; s < s1; ++s) need = std::max(need, pos[2 * s] + crop);
        feed_rows(h, *feed, sc, need, L.stream);
      }
      GatherParams gp;
      memset(&gp, 0, sizeof(gp));
      gp.inst = inst_dev + (size_t)s0 * 3;
      gp.x_out = L.x;
      gp.B = nb;
      gp.crop = crop;
      launch_gather(h, gp);
      forward_eval(h, L.x, nb, crop, L.lg, nullptr);
      CUDA_CHECK(cudaEventRecord(L.fwd_done, L.stream));
    }
    CUDA_CHECK(cudaStreamWaitEvent(main_stream, L.fwd_done, 0));
    // the chunk's ranges in visit order on one stream: each pixel's sum keeps the script's order across launches
    for (; cuts[r] < s0 + nb; ++r)
      accumulate_chunk(h, ct, L.lg + (size_t)(cuts[r] - s0) * pp * K, pos, cuts[r], cuts[r + 1], H, W, K, crop, row_begin, row_end);
    CUDA_CHECK(cudaEventRecord(L.acc_done, main_stream));
  }
}

static void scene_infer_impl(drs_handle_t h, int32_t scene_id, int32_t crop, int32_t batch, int32_t variant, int32_t row_begin,
                             int32_t row_end, uint8_t* labels_out_host, double* mean_out_host, HostSceneFeed* feed) {
  // labels_out_host may be NULL: the stripe stays on the device for drs_scene_gather_labels / drs_scene_confusion
  DRS_CHECK(h, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  auto it = h->scenes.find(scene_id);
  DRS_CHECK(it != h->scenes.end(), "scene_infer: scene %d not uploaded", scene_id);
  const Scene& sc = it->second;
  const int H = sc.H, W = sc.W, K = h->net.classes;
  if (row_end <= 0 || row_end > H) row_end = H;
  if (row_begin < 0) row_begin = 0;
  DRS_CHECK(row_begin < row_end, "scene_infer: empty stripe");
  const PassGeometry& pg = scene_pass_geometry(h, sc, scene_id, crop, batch, variant, row_begin, row_end);
  const int rows = row_end - row_begin;
  const cudaStream_t main_stream = h->stream;
  auto cleanup = [&]() {
    cudaStreamSynchronize(main_stream);
    if (h->lane.stream) cudaStreamSynchronize(h->lane.stream);
  };
  try {
    scene_pass_accumulate(h, sc, pg, crop, row_begin, row_end, feed);
    scene_pass_finish(h, rows, W, K, labels_out_host, mean_out_host);
    h->last_scene = scene_id; h->last_row_begin = row_begin; h->last_rows = rows; h->last_W = W;
    if (feed) {                                      // rows no patch reads (none for the grids of the scripts) and the tail
      feed_rows(h, *feed, sc, sc.H, main_stream);
      CUDA_CHECK(cudaStreamSynchronize(h->copy_stream));
    }
  } catch (...) { cleanup(); throw; }
  cleanup();
}

// validate_test_multiscale (isprs:1347-1474): the scene pass of each crop, in the order given, each followed by the softmax of
// its mean map added to a float32 sum (multiscale_softmax_add_kernel); the last one also writes the label map.  Every crop
// is checked before the first launch, so a refused call leaves the handle as it was.
extern "C" int drs_scene_infer_multiscale(drs_handle_t h, int32_t scene_id, int32_t n_scales, const int32_t* crops_host, int32_t batch,
                                          int32_t variant, int32_t row_begin, int32_t row_end, uint8_t* labels_out_host,
                                          float* prob_sum_out_host) {
  API_BEGIN
  DRS_CHECK(h, "null argument");
  DRS_CHECK(n_scales >= 1, "scene_infer_multiscale: n_scales=%d, need at least one scale", n_scales);
  DRS_CHECK(crops_host, "scene_infer_multiscale: null crop list");
  DRS_CHECK(batch >= 1, "grid: batch must be >= 1");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  auto it = h->scenes.find(scene_id);
  DRS_CHECK(it != h->scenes.end(), "scene_infer: scene %d not uploaded", scene_id);
  const Scene& sc = it->second;
  const int H = sc.H, W = sc.W, K = h->net.classes;
  DRS_CHECK(K >= 1 && K <= MAX_CLASSES, "K=%d out of range", K);
  if (row_end <= 0 || row_end > H) row_end = H;
  if (row_begin < 0) row_begin = 0;
  DRS_CHECK(row_begin < row_end, "scene_infer: empty stripe");
  for (int s = 0; s < n_scales; ++s) {
    const int crop = crops_host[s];
    DRS_CHECK(crop / 2 >= 1 && crop <= H && crop <= W, "grid: crop %d does not fit scene %dx%d", crop, H, W);
    scene_pass_geometry(h, sc, scene_id, crop, batch, variant, row_begin, row_end);   // resident rows cover every patch
  }
  const int rows = row_end - row_begin;
  const int64_t npix = (int64_t)rows * W;
  const cudaStream_t main_stream = h->stream;
  auto cleanup = [&]() {
    cudaStreamSynchronize(main_stream);
    if (h->lane.stream) cudaStreamSynchronize(h->lane.stream);
  };
  h->last_scene = -1;                                // the label buffer is rewritten from here on
  try {
    float* sum = pass_buf(h, h->pass.prob_sum, (size_t)npix * K * 4);
    uint8_t* lab = pass_buf(h, h->pass.labels, npix);
    for (int s = 0; s < n_scales; ++s) {
      // (looked up again: the geometry cache keeps only the last few passes)
      const PassGeometry& pg = scene_pass_geometry(h, sc, scene_id, crops_host[s], batch, variant, row_begin, row_end);
      scene_pass_accumulate(h, sc, pg, crops_host[s], row_begin, row_end, nullptr);
      multiscale_softmax_add_kernel<<<nblk(npix, 256), 256, 0, h->stream>>>(h->pass.prob, h->pass.occur, npix, K, s == 0, sum,
                                                                            s == n_scales - 1 ? lab : nullptr);
      LAUNCH_CHECK(h);
    }
    if (labels_out_host) CUDA_CHECK(cudaMemcpyAsync(labels_out_host, lab, npix, cudaMemcpyDeviceToHost, h->stream));
    if (prob_sum_out_host) CUDA_CHECK(cudaMemcpyAsync(prob_sum_out_host, sum, (size_t)npix * K * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_CHECK(cudaStreamSynchronize(h->stream));
    accum_overflow_check(h);
    h->last_scene = scene_id; h->last_row_begin = row_begin; h->last_rows = rows; h->last_W = W;
  } catch (...) { cleanup(); throw; }
  cleanup();
  API_END
}

// One launch of multiscale_softmax_add_kernel on caller-given sums and counts (unit tests: the device arithmetic over any
// range of means, not only the ones a net produces).  prob [npix,K], occur [npix], acc [npix,K] in/out (ignored on input when
// first != 0); labels_out_host non-null = the last scale (argmax written).
extern "C" int drs_debug_multiscale_softmax_add(drs_handle_t h, const float* prob_host, const uint32_t* occur_host, int64_t npix,
                                                int32_t first, float* acc_inout_host, uint8_t* labels_out_host) {
  API_BEGIN
  DRS_CHECK(h && prob_host && occur_host && acc_inout_host && npix >= 1, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int K = h->net.classes;
  DevMem<float> prob(npix * K * 4), acc(npix * K * 4);
  DevMem<uint32_t> occur(npix * 4);
  DevMem<uint8_t> lab(npix);
  CUDA_CHECK(cudaMemcpyAsync(prob, prob_host, npix * K * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(occur, occur_host, npix * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(acc, acc_inout_host, npix * K * 4, cudaMemcpyHostToDevice, h->stream));
  multiscale_softmax_add_kernel<<<nblk(npix, 256), 256, 0, h->stream>>>(prob, occur, npix, K, first != 0, acc,
                                                                        labels_out_host ? lab.get() : nullptr);
  LAUNCH_CHECK(h);
  CUDA_CHECK(cudaMemcpyAsync(acc_inout_host, acc, npix * K * 4, cudaMemcpyDeviceToHost, h->stream));
  if (labels_out_host) CUDA_CHECK(cudaMemcpyAsync(labels_out_host, lab, npix, cudaMemcpyDeviceToHost, h->stream));
  int rc = drs_synchronize(h);
  if (rc) return rc;
  API_END
}

// Scene-level confusion matrix (isprs:1289-1296, contest:944-951): the label map of the last drs_scene_infer pass over
// `scene_id` (still resident) against the ground truth uploaded with the scene; pixels whose truth is `ignore_label`
// (the eroded class 6 of isprs, the unlabelled class 7 of the contest) or >= K are skipped.
extern "C" int drs_scene_confusion(drs_handle_t h, int32_t scene_id, int32_t K, int32_t ignore_label, uint32_t* cm_out_host) {
  API_BEGIN
  DRS_CHECK(h && cm_out_host, "null argument");
  DRS_CHECK(K >= 1 && K <= MAX_CLASSES, "K=%d out of range", K);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  auto it = h->scenes.find(scene_id);
  DRS_CHECK(it != h->scenes.end(), "scene_confusion: scene %d not uploaded", scene_id);
  const Scene& sc = it->second;
  DRS_CHECK(sc.labels, "scene_confusion: scene %d was uploaded without labels", scene_id);
  DRS_CHECK(h->last_scene == scene_id && h->pass.labels, "scene_confusion: no label map of scene %d is resident (run drs_scene_infer first)", scene_id);
  DRS_CHECK(h->last_W == sc.W && h->last_row_begin >= sc.row0 && h->last_row_begin + h->last_rows <= sc.row0 + sc.rows,
            "scene_confusion: label rows [%d,%d) outside the resident ground truth", h->last_row_begin, h->last_row_begin + h->last_rows);
  const int64_t n = (int64_t)h->last_rows * sc.W;
  const uint8_t* truth = sc.labels + (int64_t)(h->last_row_begin - sc.row0) * sc.W;
  CUDA_CHECK(cudaMemsetAsync(h->cm_dev, 0, (K * K + 1) * 4, h->stream));
  const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(std::max<int64_t>(n, 1), 256), (int64_t)h->sm_count * 8);
  confusion_kernel<<<blocks, 256, 0, h->stream>>>(truth, h->pass.labels, nullptr, n, K, ignore_label, h->cm_dev);
  LAUNCH_CHECK(h);
  CUDA_CHECK(cudaMemcpyAsync(cm_out_host, h->cm_dev, (K * K + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  API_END
}

extern "C" int drs_confusion_dev(drs_handle_t h, const uint8_t* truth_dev, const uint8_t* pred_dev, const uint8_t* mask_dev,
                                 int64_t n, int32_t K, int32_t ignore_label, uint32_t* cm_out_host) {
  API_BEGIN
  DRS_CHECK(h && truth_dev && pred_dev && cm_out_host, "null argument");
  DRS_CHECK(K >= 1 && K <= MAX_CLASSES, "K=%d out of range", K);
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  CUDA_CHECK(cudaMemsetAsync(h->cm_dev, 0, (K * K + 1) * 4, h->stream));
  const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(std::max<int64_t>(n, 1), 256), (int64_t)h->sm_count * 8);
  confusion_kernel<<<blocks, 256, 0, h->stream>>>(truth_dev, pred_dev, mask_dev, n, K, ignore_label, h->cm_dev);
  LAUNCH_CHECK(h);
  CUDA_CHECK(cudaMemcpyAsync(cm_out_host, h->cm_dev, (K * K + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  API_END
}

// ------------------------------------------------------------------------------------------------
// profiling + debug hooks
// ------------------------------------------------------------------------------------------------
extern "C" int drs_set_profiling(drs_handle_t h, int32_t on) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  h->time_convs = on != 0;
  h->conv_events_used = 0;
  h->conv_flops = 0;
  h->conv_launches = 0;
  h->conv_ms_acc = 0;
  API_END
}
// Sum of the device time of the tensor-core convolution launches recorded since drs_set_profiling(1)
// (CUDA events on the handle's stream), their count and their algorithmic FLOPs; resets the record.
extern "C" int drs_profile_read(drs_handle_t h, float* conv_ms, int64_t* conv_launches, double* conv_flops) {
  API_BEGIN
  DRS_CHECK(h, "null handle");
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  float total = (float)h->conv_ms_acc;
  h->conv_ms_acc = 0;
  for (size_t i = 0; i < h->conv_events_used; ++i) {
    float ms = 0.0f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, h->conv_events[i].first, h->conv_events[i].second));
    total += ms;
  }
  if (conv_ms) *conv_ms = total;
  if (conv_launches) *conv_launches = h->conv_launches;
  if (conv_flops) *conv_flops = h->conv_flops;
  h->conv_events_used = 0;
  h->conv_flops = 0;
  h->conv_launches = 0;
  API_END
}
extern "C" int drs_last_conv_ms(drs_handle_t h, float* ms_out) { return drs_profile_read(h, ms_out, nullptr, nullptr); }

extern "C" int drs_debug_activation(drs_handle_t h, const char* name, float* out_host, int64_t count) {
  API_BEGIN
  DRS_CHECK(h && name && out_host, "null argument");
  auto it = h->taps.find(name);
  DRS_CHECK(it != h->taps.end(), "no activation recorded for scope '%s'", name);
  const Handle::Tap& t = it->second;
  DRS_CHECK(count == t.pixels * t.co, "activation '%s' has %lld elements, got %lld", name, (long long)(t.pixels * t.co), (long long)count);
  DevMem<float> tmp(count * 4);
  if (t.type == ET_F32) slice_to_f32_kernel<float><<<nblk(count, 256), 256, 0, h->stream>>>((const float*)t.ptr, t.cstride, t.coff, t.co, t.pixels, tmp);
  else if (t.type == ET_F16) slice_to_f32_kernel<__half><<<nblk(count, 256), 256, 0, h->stream>>>((const __half*)t.ptr, t.cstride, t.coff, t.co, t.pixels, tmp);
  else slice_to_f32_kernel<__nv_bfloat16><<<nblk(count, 256), 256, 0, h->stream>>>((const __nv_bfloat16*)t.ptr, t.cstride, t.coff, t.co, t.pixels, tmp);
  h->launches++;
  CUDA_CHECK(cudaMemcpyAsync(out_host, tmp, count * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_CHECK(cudaStreamSynchronize(h->stream));
  API_END
}

// One convolution through the production path (unit tests): y = act(conv(x, w) * scale + shift).  16-bit precisions cast
// the input and pack the filter as refresh_packed packs a layer's; the conv1 shape (conv1_tc_supported) runs on conv1's
// tensor-core kernel like the first layer of both forwards, any other shape on the generic one.
template <typename T>
static void debug_conv_tc(Handle* h, const float* x32, const float* w32, const float* sc, const float* sh, const ConvLayer& c, int B,
                          int crop, int act, T* xa, void* wp, T* ya, float* y32) {
  const int64_t M = (int64_t)B * crop * crop;
  if (conv1_tc_supported(c.k, c.rate, c.ci, c.co)) {
    pack_conv1<T>(h, w32, wp, c.ci, c.co);
    conv1_tc_forward<T>(h, x32, c.ci, xa, wp, ActBuf{ya, c.co, 0}, c.co, B, crop, sc, sh, act, nullptr, true);
  } else {
    cast_kernel<float, T><<<nblk(M * c.ci, 256), 256, 0, h->stream>>>(x32, xa, M * c.ci);
    LAUNCH_CHECK(h);
    repack_filter(h, w32, wp, c.k * c.k, c.ci, c.co, 0, ElemTag<T>::v);
    run_conv<T>(h, ActBuf{xa, c.ci, 0}, c.ci, w32, wp, ActBuf{ya, c.co, 0}, c.co, B, crop, c.k, c.rate, c.pad_b, sc, sh, act);
  }
  cast_kernel<T, float><<<nblk(M * c.co, 256), 256, 0, h->stream>>>(ya, y32, M * c.co);
  LAUNCH_CHECK(h);
}

extern "C" int drs_debug_conv(drs_handle_t h, const float* x_host, const float* w_host, const float* scale_host, const float* shift_host,
                              int32_t B, int32_t crop, int32_t k, int32_t rate, int32_t Ci, int32_t Co, int32_t act, int32_t precision,
                              float* y_host) {
  API_BEGIN
  DRS_CHECK(h && x_host && w_host && scale_host && shift_host && y_host, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop * crop;
  const int64_t nw = (int64_t)k * k * Ci * Co;
  const ConvLayer c = conv_shape(k, rate, Ci, Co);
  DevMem<float> x32(M * Ci * 4), w32(nw * 4), sc(Co * 4), sh(Co * 4), y32(M * Co * 4);
  DevMem<void> xa, wp, ya;   // 16-bit operands; like the rest freed on return, after the synchronize
  CUDA_CHECK(cudaMemcpyAsync(x32, x_host, M * Ci * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(w32, w_host, nw * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(sc, scale_host, Co * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(sh, shift_host, Co * 4, cudaMemcpyHostToDevice, h->stream));
  if (precision == DRS_PREC_FP32) {
    run_conv<float>(h, ActBuf{x32, Ci, 0}, Ci, w32, nullptr, ActBuf{y32, Co, 0}, Co, B, crop, k, rate, c.pad_b, sc, sh, act);
  } else {
    // (conv1's kernel reads the input padded to 8 channels and a filter of C1_SLOTS x Co x 8 elements)
    xa = DevMem<void>(M * std::max(Ci, 8) * 2);
    wp = DevMem<void>(std::max<int64_t>(nw, (int64_t)C1_SLOTS * Co * 8) * 2);
    ya = DevMem<void>(M * Co * 2);
    if (precision == DRS_PREC_F16) debug_conv_tc<__half>(h, x32, w32, sc, sh, c, B, crop, act, (__half*)xa.get(), wp, (__half*)ya.get(), y32);
    else debug_conv_tc<__nv_bfloat16>(h, x32, w32, sc, sh, c, B, crop, act, (__nv_bfloat16*)xa.get(), wp, (__nv_bfloat16*)ya.get(), y32);
  }
  CUDA_CHECK(cudaMemcpyAsync(y_host, y32, M * Co * 4, cudaMemcpyDeviceToHost, h->stream));
  int rc = drs_synchronize(h);
  if (rc) return rc;
  API_END
}

// Kernel micro-benchmark (tools/conv_bench.py): `reps` back-to-back launches of one tcgen05 convolution on pseudo-random
// resident operands, timed with events on the handle's stream.  exp_mode >= 0 overrides DRS_EXP_MODE for these launches.
__global__ void bench_fill_kernel(uint16_t* __restrict__ p, int64_t n, uint32_t seed, int bf16) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t v = (uint32_t)i * 2654435761u + seed;
    v ^= v >> 15; v *= 2246822519u; v ^= v >> 13;
    const float f = ((float)(v & 0xffff) / 65536.0f - 0.5f) * 0.5f;
    p[i] = bf16 ? __bfloat16_as_ushort(__float2bfloat16(f)) : __half_as_ushort(__float2half(f));
  }
}
extern "C" int drs_bench_conv(drs_handle_t h, int32_t B, int32_t crop, int32_t k, int32_t rate, int32_t Ci, int32_t Co,
                              int32_t precision, int32_t exp_mode, int32_t reps, float* ms_out, uint32_t* instr_out) {
  API_BEGIN
  DRS_CHECK(h && ms_out && reps >= 1, "bad argument");
  DRS_CHECK(precision == DRS_PREC_F16 || precision == DRS_PREC_BF16, "bench_conv: tensor-core precisions only");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop * crop;
  const int64_t nw = (int64_t)k * k * Ci * Co;
  const int pad_b = ((k - 1) * rate) / 2;
  struct ExpModeReset { ~ExpModeReset() { g_conv_exp_mode = -1; } } exp_mode_reset;   // on every way out
  const int bf = precision == DRS_PREC_BF16;
  DevMem<uint16_t> xa(M * Ci * 2), wp(nw * 2), ya(M * Co * 2);
  DevMem<float> sc(2 * 256 * 4);
  bench_fill_kernel<<<1024, 256, 0, h->stream>>>(xa, M * Ci, 1u, bf);
  bench_fill_kernel<<<256, 256, 0, h->stream>>>(wp, nw, 2u, bf);
  {
    std::vector<float> one_zero(512, 0.0f);
    for (int i = 0; i < 256; ++i) one_zero[i] = 1.0f;
    CUDA_CHECK(cudaMemcpy(sc, one_zero.data(), 512 * 4, cudaMemcpyHostToDevice));
  }
  Event e0 = new_event(cudaEventDefault), e1 = new_event(cudaEventDefault);
  ConvTcArgs a;
  a.in = xa; a.in_cstride = Ci; a.in_coff = 0; a.ci = Ci; a.w = wp; a.out = ya; a.out_cstride = Co; a.out_coff = 0; a.co = Co;
  a.B = B; a.crop = crop; a.k = k; a.rate = rate; a.pad_b = pad_b; a.scale = sc; a.shift = sc + 256; a.act = ACT_RELU;
  a.etype = bf ? ET_BF16 : ET_F16;
  g_conv_exp_mode = exp_mode;
  launch_conv_tc(h, a);                       // warm-up (tensor maps, module load)
  CUDA_CHECK(cudaEventRecord(e0, h->stream));
  for (int r = 0; r < reps; ++r) launch_conv_tc(h, a);
  CUDA_CHECK(cudaEventRecord(e1, h->stream));
  int rc = drs_synchronize(h);
  if (rc) return rc;
  float ms = 0.0f;
  CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
  *ms_out = ms / reps;
  // instrumented launches (exp_mode bit 16): cycle counters of CTA 0's last launch
  if (instr_out) for (int i = 0; i < 10; ++i) instr_out[i] = h->diag_host[4 + i];
  API_END
}

// Filter gradient of one convolution through the training step's filter-gradient phase (unit tests)
extern "C" int drs_debug_wgrad(drs_handle_t h, const float* x_host, const float* dy_host, int32_t B, int32_t crop, int32_t k,
                               int32_t rate, int32_t Ci, int32_t Co, int32_t precision, float* dw_host) {
  API_BEGIN
  DRS_CHECK(h && x_host && dy_host && dw_host, "null argument");
  CUDA_CHECK(cudaSetDevice(h->cfg.device));
  const int64_t M = (int64_t)B * crop * crop;
  const int64_t nw = (int64_t)k * k * Ci * Co;
  const ConvLayer c = conv_shape(k, rate, Ci, Co);
  // (the tensor-core kernel runs 32-channel operands as 64: its split partials have the padded shape)
  const size_t part_cap = (size_t)k * k * ((Ci + 63) / 64 * 64) * ((Co + 63) / 64 * 64) * WGRAD_MAX_SPLITS;
  DevMem<float> x32(M * Ci * 4), dy32(M * Co * 4), dw(nw * 4), part(part_cap * 4);
  DevMem<__nv_bfloat16> xa, dya;   // bf16 operands; like the rest freed on return, after the synchronize
  CUDA_CHECK(cudaMemcpyAsync(x32, x_host, M * Ci * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_CHECK(cudaMemcpyAsync(dy32, dy_host, M * Co * 4, cudaMemcpyHostToDevice, h->stream));
  if (precision == DRS_PREC_FP32) {
    filter_gradient<float>(h, c, ActBuf{x32, Ci, 0}, nullptr, nullptr, dy32, B, crop, dw, part, part_cap);
  } else {
    DRS_CHECK(precision == DRS_PREC_BF16, "debug_wgrad: precision must be FP32 or BF16");
    xa = DevMem<__nv_bfloat16>(M * Ci * 2);
    dya = DevMem<__nv_bfloat16>(M * Co * 2);
    cast_kernel<float, __nv_bfloat16><<<nblk(M * Ci, 256), 256, 0, h->stream>>>(x32, xa, M * Ci);
    cast_kernel<float, __nv_bfloat16><<<nblk(M * Co, 256), 256, 0, h->stream>>>(dy32, dya, M * Co);
    h->launches += 2;
    filter_gradient<__nv_bfloat16>(h, c, ActBuf{xa, Ci, 0}, nullptr, nullptr, dya, B, crop, dw, part, part_cap);
  }
  CUDA_CHECK(cudaMemcpyAsync(dw_host, dw, nw * 4, cudaMemcpyDeviceToHost, h->stream));
  int rc = drs_synchronize(h);
  if (rc) return rc;
  API_END
}
