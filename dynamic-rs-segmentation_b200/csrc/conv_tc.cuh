// Dilated SAME convolution (stride 1) as an implicit GEMM on the 5th-gen tensor cores.
//
// Reference op: tf.nn.atrous_conv2d(x, W[kh,kw,Ci,Co], rate, 'SAME') + bias -> BN -> act
// (_conv_layer, /root/reference/isprs_dilated_random.py:700-723).  Also used for dgrad (a dilated
// convolution of dY with the tap-flipped, Ci/Co-transposed filter and swapped padding).
//
//   GEMM:  D[M, N] = A[M, K] * B[N, K]^T      M = B*crop*crop output pixels (NHWC raster)
//                                             N = Co,  K = kh*kw*Ci  (k index = tap*Ci + c)
//   A tile  128 pixels x BLOCK_K channels of ONE filter tap, fetched by a TMA *im2col* load:
//           128 consecutive output pixels (running across row and image boundaries), displaced by the
//           tap offset (kx*rate, ky*rate); pixels outside the image are zero-filled by the TMA unit,
//           which is exactly SAME padding (asymmetric before/after for even kernels included).
//   B tile  N x BLOCK_K slice of the packed filter matrix [Co][K] (K-major), tiled TMA load.
//   Both land in shared memory in the canonical K-major 128B-swizzled (64B when BLOCK_K=32) layout
//   that tcgen05.mma reads through shared-memory descriptors; the fp32 accumulator lives in TMEM
//   (two stages, so the epilogue of tile i overlaps the main loop of tile i+1).  For Co <= 128 a tile is a PAIR of 128-pixel
//   units: two A tiles per K block against one B slice, two accumulators per stage (ConvSched below).
//   Epilogue: tcgen05.ld -> y = act(acc*scale[c] + shift[c]) (bias / folded BN) -> fp16|bf16 ->
//   swizzled staging in shared memory -> TMA store into a channel slice of the NHWC output
//   (dense nets write straight into the concat buffer: tf.concat, isprs:921-948, costs nothing).
//
// Warp roles (256 threads, persistent, one CTA per SM; role warps stay converged, an elected lane issues):
//   warp 0 : TMA producer, im2col tiles     warp 1 : tcgen05.mma issuer
//   warp 3 : TMA producer, filter slices    warp 2 : TMEM allocator
//   warps 4..7 : epilogue (TMEM lane quadrant = warp % 4)
#pragma once
#include "drs_common.cuh"
#include "ptx_sm100.cuh"

struct ConvTcParams {
  int M_total;        // output pixels
  int crop;           // H = W
  int ksize, rate, pad_b;
  int ci, in_coff;    // channels consumed, channel offset inside the input buffer
  int co, out_coff;   // N, channel offset inside the output buffer
  int num_tiles;      // ceil(M_total / 128): 128-pixel units
  int mt;             // 1: every tile is one unit.  2 (Co <= 128): a tile is two consecutive units whose im2col tiles share ONE
                      // filter slice per K block (two accumulators), see ConvSched
  int stages;         // smem pipeline depth
  int kps;            // K blocks (BLOCK_K channels of one tap) per pipeline stage: one barrier round trip per kps blocks
  int acc_stride;     // TMEM columns of one accumulator
  int tmem_cols;      // allocated TMEM columns (power of two >= 32)
  int act;
  int smem_needed;    // bytes used from the 1024B-aligned base
  int smem_provided;  // dynamic shared memory bytes of the launch
  uint32_t idesc;
  int exp_mode;       // DRS_EXP_MODE timing experiments (results are garbage): 4 no epilogue, 5 no TMA store, 8 no loads,
                      // 9 no MMA, 10 neither and no epilogue (barrier hand-shake only)
  const float* scale; // [co]
  const float* shift; // [co]
  uint32_t* diag;     // host-mapped diagnostics
  // training forward: per-channel sum / sum of squares of the stored (rounded) outputs, reduced in the epilogue so that
  // train-mode batch norm needs no extra pass over Z (stats.acc == nullptr: off)
  BnFinish stats;
};

constexpr int CONV_TC_THREADS = 256;
constexpr int CONV_TC_BM = 128;

template <typename OutT>
__device__ __forceinline__ uint32_t pack2(float a, float b);
template <>
__device__ __forceinline__ uint32_t pack2<__half>(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
template <>
__device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// Which 128-pixel units a CTA works on, in order.  mt == 1: unit = blockIdx.x + i * gridDim.x (the round-robin sweep: at
// any moment the CTAs read neighbouring pixels, so the 9-25 re-fetches of an input pixel by the other taps hit L2).
// mt == 2: the same sweep over PAIRS of consecutive units for as many full rounds as there are, and one last round that
// hands the remaining units out as pairs and singles so that no CTA gets more than a pair (small-M training layers: 4.6
// rounds of singles become 2 rounds of pairs + 1 of singles instead of 3 rounds of pairs).  Every role of the CTA
// walks the same list.  The order in which a pixel's K blocks are accumulated never depends on the schedule.
struct ConvSched {
  int G, b, rounds, base, nd, iters, m2;
  // (grid, block) = (gridDim.x, blockIdx.x) in the kernel; host-callable so that tests/test_abi.py can enumerate the schedule
  __host__ __device__ __forceinline__ ConvSched(int num_units, int mt, int grid, int block) {
    G = grid; b = block; m2 = mt == 2;
    if (!m2) {
      rounds = b < num_units ? (num_units - b + G - 1) / G : 0;
      iters = rounds; base = 0; nd = 0;
    } else {
      rounds = num_units / (2 * G);
      base = 2 * G * rounds;
      const int r = num_units - base;
      nd = r > G ? r - G : 0;                         // pairs in the last round (CTAs 0..nd-1); the others take a single
      iters = rounds + ((r > G || b < r) ? 1 : 0);
    }
  }
  // unit index of iteration i and whether it is a pair
  __host__ __device__ __forceinline__ int unit(int i, bool& two) const {
    if (!m2) { two = false; return b + i * G; }
    if (i < rounds) { two = true; return (i * G + b) * 2; }
    if (b < nd) { two = true; return base + 2 * b; }
    two = false;
    return base + nd + b;                             // == base + 2 * nd + (b - nd)
  }
};

// BLOCK_K: channels per K step (64 -> 128B swizzle, 32 -> 64B swizzle).  EPI_C: channels per epilogue
// store box (64 -> 128B swizzle, 32 -> 64B swizzle).
template <int BLOCK_K, int EPI_C, typename OutT, bool INSTR>
__global__ void __launch_bounds__(CONV_TC_THREADS, EPI_C == 32 ? 2 : 1)   // the 32-channel epilogue runs two CTAs per SM: <= 128 registers
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const ConvTcParams p) {
  constexpr int A_BYTES = CONV_TC_BM * BLOCK_K * 2;
  constexpr int SW_BYTES = BLOCK_K * 2;                        // swizzle span of the operand tiles
  constexpr uint32_t OP_LAYOUT = (SW_BYTES == 128) ? 2u : 4u;  // SWIZZLE_128B : SWIZZLE_64B
  constexpr uint32_t OP_SBO = 8 * SW_BYTES;                    // 8 rows of one swizzle atom
  constexpr int STG_BYTES = CONV_TC_BM * EPI_C * 2;            // one epilogue staging buffer
  constexpr int MAX_STAGES = 8;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // operand tiles need 1024B alignment (swizzle atom); the launch adds slack only when it fits
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  if (pad + static_cast<uint32_t>(p.smem_needed) > static_cast<uint32_t>(p.smem_provided)) {
    if (threadIdx.x == 0 && p.diag) {
      p.diag[0] = 0xBAD00001u;
      p.diag[1] = raw_addr;
      __threadfence_system();
    }
    __trap();
  }
  const int B_BYTES = p.co * BLOCK_K * 2;
  const int a_bytes = p.mt * A_BYTES;                          // im2col tile(s) of one K block
  const int kb_bytes = a_bytes + B_BYTES;                      // one K block: im2col tile(s) + filter slice
  const ConvSched sched(p.num_tiles, p.mt, (int)gridDim.x, (int)blockIdx.x);
  const int stage_bytes = p.kps * kb_bytes;
  uint8_t* stg = smem + p.stages * stage_bytes;                // 2 staging buffers (1024B aligned)
  float* s_scale = reinterpret_cast<float*>(stg + 2 * STG_BYTES);
  float* s_shift = s_scale + 256;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_shift + 256);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* tmem_full = empty_bar + MAX_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  // Training forward: the running column sums live in registers (st0 / st1 below) and are combined through the staging
  // buffers at the very end, so the statistics cost no shared memory: with 2-4 KB of their own they pushed the operand ring
  // just under a stage boundary (N=128: 3 -> 2 stages, N=256: 4 -> 3) and the fused forward ran 10-17 us per layer slower
  // than the same-shape dgrad.
  constexpr int STAT_GROUPS = CONV_TC_BM / EPI_C;
  constexpr int STAT_MAX_CHUNKS = 256 / EPI_C;

  // warp index through a shuffle: the compiler then knows it is warp-uniform, role branches become uniform branches and the
  // descriptor / address arithmetic of the single-thread roles runs on the uniform datapath (no R2UR moves per UTMALDG / UTCHMMA)
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int taps = p.ksize * p.ksize;
  const int kb_per_tap = p.ci / BLOCK_K;
  const int num_kb = taps * kb_per_tap;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    ptx::prefetch_tensormap(&tmC);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 2);     // one arrive.expect_tx per producer warp (A tiles, B tiles)
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tmem_full[s], 1);    // one commit by the MMA issuer
      ptx::mbar_init(&tmem_empty[s], 4);   // one arrive per epilogue warp
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_holder, static_cast<uint32_t>(p.tmem_cols));
    ptx::tmem_relinquish();
  }
  // everything above is private to the CTA; from here on global memory written by the previous kernel is read
  pdl_sync();
  for (int i = threadIdx.x; i < p.co; i += CONV_TC_THREADS) {
    s_scale[i] = p.scale[i];
    s_shift[i] = p.shift[i];
  }
  ptx::tcgen05_fence_before();
  __syncthreads();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // The two single-thread roles are issue-bound (measured: every instruction in these loops shows in the kernel time
  // for Co <= 192), so they are written for a minimal dependent instruction stream: running shared-memory addresses,
  // 32-bit descriptor arithmetic, a per-K-block table instead of divisions, kps K blocks per barrier round trip.
  const uint32_t smem_base = ptx::smem_u32(smem);
  const uint32_t full0 = ptx::smem_u32(full_bar), empty0 = ptx::smem_u32(empty_bar);
  const uint32_t ring_bytes = static_cast<uint32_t>(p.stages * stage_bytes);
  const bool no_loads = p.exp_mode == 8 || p.exp_mode == 10;
  const bool no_mma = p.exp_mode == 9 || p.exp_mode == 10;
  if (warp == 0 || warp == 3) {
    // ------------------------------------------------------------------ TMA producers: warp 0 loads the im2col tiles (A),
    // warp 3 the filter slices (B); each arrives on the stage's full barrier with its own byte count (barrier count 2).
    // The whole warp runs the loop (convergent) and one *elected* lane issues: under `if (lane == 0)` ptxas cannot tell
    // that a single thread is active and wraps every UTMALDG / UTCHMMA in an ELECT + BRA.U.ANY loop fed by R2UR moves
    // (~100 cycles per instruction, measured); with elect.sync the warp-level instructions are issued directly.
    // Two warps because the issue loop itself is the bottleneck of the pipeline for Co <= 192 (~160 cycles per UTMALDG
    // with its operand set-up, measured with the INSTR twin): A and B issue in parallel on different schedulers.
    const bool is_a = warp == 0;
    const bool leader = ptx::elect_one_sync();
    uint32_t soff = 0, boff = 0, phase = 0;     // byte offset of the stage in the ring / of its barrier
    long long t_begin = 0, t_wait = 0, t_exp = 0, t_tma = 0;
    uint32_t n_stage = 0;
    if (INSTR) t_begin = clock64();
    const int cc = p.crop * p.crop;
    const int w_end = p.ksize * p.rate;
    for (int it = 0; it < sched.iters; ++it) {
      bool two;
      const int m0 = sched.unit(it, two) * CONV_TC_BM;
      const uint32_t kb_tx = is_a ? (two ? 2u * A_BYTES : static_cast<uint32_t>(A_BYTES)) : static_cast<uint32_t>(B_BYTES);
      const int n_img = m0 / cc;
      const int rem = m0 - n_img * cc;
      const int py = rem / p.crop;
      const int cw = rem - py * p.crop - p.pad_b, chh = py - p.pad_b;
      // second unit of a pair
      const int m1 = m0 + CONV_TC_BM;
      const int n_img1 = m1 / cc;
      const int rem1 = m1 - n_img1 * cc;
      const int py1 = rem1 / p.crop;
      const int cw1 = rem1 - py1 * p.crop - p.pad_b, chh1 = py1 - p.pad_b;
      int cb = p.in_coff, offw = 0, offh = 0, kcol = 0;   // channel block of the tap, tap offsets, filter-matrix column
      for (int kb0 = 0; kb0 < num_kb; kb0 += p.kps) {
        const int nk = min(p.kps, num_kb - kb0);
        long long t0 = 0, t1 = 0, t2 = 0;
        if (INSTR) t0 = clock64();
        ptx::mbar_wait_addr(empty0 + boff, phase ^ 1, p.diag, 0x100);
        if (INSTR) { t1 = clock64(); t_wait += t1 - t0; ++n_stage; }
        const uint32_t fb = full0 + boff;
        if (leader) {
          if (no_loads) ptx::mbar_arrive_addr(fb);                     // timing experiment: barrier hand-shake only
          else ptx::mbar_arrive_expect_tx_addr(fb, static_cast<uint32_t>(nk) * kb_tx);
        }
        if (INSTR) { t2 = clock64(); t_exp += t2 - t1; }
        uint32_t dst = smem_base + soff + (is_a ? 0u : static_cast<uint32_t>(a_bytes));
        if (is_a) {
          for (int j = 0; j < nk; ++j, dst += kb_bytes) {
            if (leader && !no_loads) {
              ptx::tma_load_im2col_4d_addr(dst, &tmA, fb, cb, cw, chh, n_img, static_cast<uint16_t>(offw), static_cast<uint16_t>(offh));
              if (two)
                ptx::tma_load_im2col_4d_addr(dst + A_BYTES, &tmA, fb, cb, cw1, chh1, n_img1, static_cast<uint16_t>(offw), static_cast<uint16_t>(offh));
            }
            cb += BLOCK_K;
            if (cb == p.in_coff + p.ci) {
              cb = p.in_coff;
              offw += p.rate;
              if (offw == w_end) { offw = 0; offh += p.rate; }
            }
          }
        } else {
          for (int j = 0; j < nk; ++j, dst += kb_bytes, kcol += BLOCK_K)
            if (leader && !no_loads) ptx::tma_load_2d_addr(dst, &tmB, fb, kcol, 0);
        }
        if (INSTR) t_tma += clock64() - t2;
        soff += stage_bytes;
        boff += 8;
        if (soff == ring_bytes) { soff = 0; boff = 0; phase ^= 1; }
      }
    }
    if (INSTR && is_a && leader && blockIdx.x == 0 && p.diag) {
      p.diag[4] = static_cast<uint32_t>(clock64() - t_begin);
      p.diag[5] = static_cast<uint32_t>(t_wait);
      p.diag[6] = n_stage;
      p.diag[7] = static_cast<uint32_t>(t_exp);
      p.diag[8] = static_cast<uint32_t>(t_tma);
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (convergent warp, elected lane issues)
    const bool leader = ptx::elect_one_sync();
    uint32_t soff = 0, boff = 0, phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    long long t_begin = 0, t_wait = 0, t_wait_acc = 0, t_mma = 0, t_commit = 0;
    if (INSTR) t_begin = clock64();
    // descriptor words: low = address >> 4 | LBO(16 B) << 16, high = SBO >> 4 | version | layout
    const uint32_t desc_lo0 = ((smem_base >> 4) & 0x3FFFu) | (1u << 16);
    const uint32_t desc_hi = ((OP_SBO >> 4) & 0x3FFFu) | (1u << 14) | (OP_LAYOUT << 29);
    const uint32_t kb_step = static_cast<uint32_t>(kb_bytes) >> 4;
    for (int it = 0; it < sched.iters; ++it) {
      bool two;
      (void)sched.unit(it, two);
      if (INSTR) {
        const long long t0 = clock64();
        ptx::mbar_wait(&tmem_empty[as], aphase ^ 1, p.diag, 0x200 + as);
        t_wait_acc += clock64() - t0;
      } else {
        ptx::mbar_wait(&tmem_empty[as], aphase ^ 1, p.diag, 0x200 + as);
      }
      const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * p.mt * p.acc_stride);
      uint32_t fresh = 0;                                  // 0 until the first MMA of the tile (overwrites D)
      for (int kb0 = 0; kb0 < num_kb; kb0 += p.kps) {
        const int nk = min(p.kps, num_kb - kb0);
        long long t0 = 0, t1 = 0, t2 = 0;
        if (INSTR) t0 = clock64();
        ptx::mbar_wait_addr(full0 + boff, phase, p.diag, 0x300);
        ptx::tcgen05_fence_after();
        if (INSTR) { t1 = clock64(); t_wait += t1 - t0; }
        if (leader && !no_mma) {
          uint32_t a_lo = desc_lo0 + (soff >> 4);
          for (int j = 0; j < nk; ++j, a_lo += kb_step) {
            const uint32_t b_lo = a_lo + (static_cast<uint32_t>(a_bytes) >> 4);
            ptx::umma_f16_kblock<BLOCK_K / 16>(d_tmem, a_lo, b_lo, desc_hi, p.idesc, fresh);
            if (two)      // the pair's second unit: same filter slice, its own accumulator
              ptx::umma_f16_kblock<BLOCK_K / 16>(d_tmem + p.acc_stride, a_lo + (A_BYTES >> 4), b_lo, desc_hi, p.idesc, fresh);
            fresh = 1;
          }
        }
        if (INSTR) { t2 = clock64(); t_mma += t2 - t1; }
        if (leader) ptx::umma_commit_addr(empty0 + boff);   // frees the smem slot when these MMAs retire
        if (INSTR) t_commit += clock64() - t2;
        soff += stage_bytes;
        boff += 8;
        if (soff == ring_bytes) { soff = 0; boff = 0; phase ^= 1; }
      }
      if (leader) ptx::umma_commit(&tmem_full[as]);        // accumulator complete -> epilogue
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (INSTR && leader && blockIdx.x == 0 && p.diag) {
      p.diag[9] = static_cast<uint32_t>(clock64() - t_begin);
      p.diag[10] = static_cast<uint32_t>(t_wait);
      p.diag[11] = static_cast<uint32_t>(t_mma);
      p.diag[12] = static_cast<uint32_t>(t_commit);
      p.diag[13] = static_cast<uint32_t>(t_wait_acc);
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue
    const int quad = warp & 3;
    const int row = quad * 32 + lane;            // accumulator row == pixel within the tile
    const int epi_tid = threadIdx.x - 128;
    // one elected lane of warp 4 owns the TMA stores (bulk groups are per thread: elect.sync picks the same lane for the
    // same member mask every time); elected at each site so that ptxas sees a single active thread
    constexpr int CHUNK16 = EPI_C / 8;           // 16-byte chunks per staged row
    const int sw = (EPI_C == 64) ? (row & 7) : ((row >> 1) & 3);
    const int n_chunks = p.co / EPI_C;
    int as = 0;
    uint32_t aphase = 0;
    int sbuf = 0;
    float st0[STAT_MAX_CHUNKS], st1[STAT_MAX_CHUNKS];      // this thread's (channel, row group) sums, per output chunk
#pragma unroll
    for (int q = 0; q < STAT_MAX_CHUNKS; ++q) { st0[q] = 0.0f; st1[q] = 0.0f; }
    for (int it = 0; it < sched.iters; ++it) {
      bool two;
      const int unit0 = sched.unit(it, two);
      ptx::mbar_wait(&tmem_full[as], aphase, p.diag, 0x400 + as);
      ptx::tcgen05_fence_after();
      for (int sub = 0; sub < (two ? 2 : 1); ++sub) {
      const int tile = unit0 + sub;                // 128-pixel unit of this accumulator
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>((as * p.mt + sub) * p.acc_stride);
      for (int ch = 0; ch < ((p.exp_mode == 4 || p.exp_mode == 10) ? 0 : n_chunks); ++ch) {
        uint32_t v[EPI_C];
        ptx::tmem_ld_32x32b_x32(t_row + ch * EPI_C, v);
        if (EPI_C == 64) ptx::tmem_ld_32x32b_x32(t_row + ch * EPI_C + 32, v + (EPI_C == 64 ? 32 : 0));
        ptx::tmem_wait_ld();
        // the TMA store that last read staging buffer `sbuf` (two chunks ago) must have drained
        if (warp == 4 && ptx::elect_one_sync()) ptx::tma_store_wait_read<1>();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        uint8_t* srow = stg + sbuf * STG_BYTES + row * (EPI_C * 2);
        const float* sc = s_scale + ch * EPI_C;
        const float* sh = s_shift + ch * EPI_C;
#pragma unroll
        for (int j = 0; j < CHUNK16; ++j) {
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int c0 = j * 8 + e * 2;
            float a = apply_act(fmaf(__uint_as_float(v[c0]), sc[c0], sh[c0]), p.act);
            float b = apply_act(fmaf(__uint_as_float(v[c0 + 1]), sc[c0 + 1], sh[c0 + 1]), p.act);
            o[e] = pack2<OutT>(a, b);
          }
          *reinterpret_cast<uint4*>(srow + ((j ^ sw) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        ptx::fence_proxy_async_smem();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (warp == 4 && p.exp_mode != 5 && ptx::elect_one_sync()) {
          ptx::tma_store_2d(&tmC, stg + sbuf * STG_BYTES, p.out_coff + ch * EPI_C, tile * CONV_TC_BM);
          ptx::tma_store_commit();
        }
        if (p.stats.acc) {
          // column sums of the staged (already rounded) tile: thread = (channel, row group); rows past the end of the
          // tensor (clipped by the TMA store) are skipped.  The (chunk, channel, row group) sum is owned by exactly one thread.
          constexpr int GROUPS = CONV_TC_BM / EPI_C, ROWS = EPI_C;
          const int c = epi_tid % EPI_C, grp = epi_tid / EPI_C;
          const int rows_valid = min(CONV_TC_BM, p.M_total - tile * CONV_TC_BM);
          const uint8_t* col = stg + sbuf * STG_BYTES + (c & 7) * 2;
          const int c16 = c >> 3;
          float a0 = 0.0f, a1 = 0.0f;
          const int r_end = min(rows_valid, (grp + 1) * ROWS);
          for (int r = grp * ROWS; r < r_end; ++r) {
            const int swr = (EPI_C == 64) ? (r & 7) : ((r >> 1) & 3);
            const float f = to_f32(*reinterpret_cast<const OutT*>(col + r * (EPI_C * 2) + ((c16 ^ swr) << 4)));
            a0 += f;
            a1 = fmaf(f, f, a1);
          }
#pragma unroll
          for (int q = 0; q < STAT_MAX_CHUNKS; ++q)
            if (q == ch) { st0[q] += a0; st1[q] += a1; }     // predicated: keeps the array in registers
          (void)GROUPS;
        }
        sbuf ^= 1;
      }
      }
      // all TMEM reads of this accumulator stage are complete (wait::ld above)
      ptx::tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (warp == 4 && ptx::elect_one_sync()) ptx::tma_store_wait_all();
    if (p.stats.acc) {
      // CTA partial (row groups combined in fixed order) -> 64-bit fixed point -> integer atomicAdd (order-independent);
      // the last CTA to arrive converts, finalizes mean / inv_std / moving averages and clears the accumulators.
      constexpr int GROUPS = CONV_TC_BM / EPI_C;
      // the staging buffers are free now (every TMA store has drained): [row group][2][co] floats <= 8 KB
      float* s_stat = reinterpret_cast<float*>(stg);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      {
        const int c = epi_tid % EPI_C, grp = epi_tid / EPI_C;
#pragma unroll
        for (int q = 0; q < STAT_MAX_CHUNKS; ++q)
          if (q < n_chunks) {
            s_stat[(grp * 2) * p.co + q * EPI_C + c] = st0[q];
            s_stat[(grp * 2 + 1) * p.co + q * EPI_C + c] = st1[q];
          }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int i = epi_tid; i < 2 * p.co; i += 128) {
        const int which = i / p.co, c = i - which * p.co;
        float a = 0.0f;
#pragma unroll
        for (int g = 0; g < GROUPS; ++g) a += s_stat[(g * 2 + which) * p.co + c];
        const long long q = __double2ll_rn((double)a * p.stats.fx_scale);
        atomicAdd(bn_acc_mine(p.stats) + i, static_cast<unsigned long long>(q));
      }
      __threadfence();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      uint32_t* s_flag = reinterpret_cast<uint32_t*>(s_stat);       // s_stat is dead now (the barrier above ordered its reads)
      if (epi_tid == 0) *s_flag = (atomicAdd(p.stats.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (*s_flag) {
        __threadfence();
        const double inv_scale = 1.0 / p.stats.fx_scale;
        const int C = p.co;
        for (int i = epi_tid; i < C; i += 128) {
          const double a = (double)bn_acc_take(p.stats, i) * inv_scale;
          const double b = (double)bn_acc_take(p.stats, C + i) * inv_scale;
          p.stats.sums[i] = (float)a;
          p.stats.sums[C + i] = (float)b;
          if (p.stats.mean) {
            const double mu = (double)(float)a / p.stats.count;
            double var = (double)(float)b / p.stats.count - mu * mu;
            if (var < 0.0) var = 0.0;
            p.stats.mean[i] = (float)mu;
            p.stats.inv_std[i] = (float)(1.0 / sqrt(var + (double)p.stats.eps));
            const double var_ema = p.stats.unbiased_ema ? var * (p.stats.count / fmax(p.stats.count - 1.0, 1.0)) : var;
            p.stats.mov_mean[i] = p.stats.decay * p.stats.mov_mean[i] + (1.0f - p.stats.decay) * (float)mu;
            p.stats.mov_var[i] = p.stats.decay * p.stats.mov_var[i] + (1.0f - p.stats.decay) * (float)var_ema;
          }
        }
        if (epi_tid == 0) *p.stats.counter = 0u;
      }
    }
  }

  ptx::tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tcgen05_fence_after();
    ptx::tmem_dealloc(tmem_base, static_cast<uint32_t>(p.tmem_cols));
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct ConvTcArgs {
  const void* in;      // NHWC [B,crop,crop,in_cstride] fp16/bf16
  int in_cstride, in_coff, ci;
  const void* w;       // packed [co][k*k*ci] fp16/bf16
  void* out;           // NHWC [B*crop*crop, out_cstride]
  int out_cstride, out_coff, co;
  int B, crop, k, rate, pad_b;
  const float* scale;
  const float* shift;
  int act;
  int etype;           // ET_F16 / ET_BF16 (operands and output)
  const BnFinish* stats = nullptr;   // training forward: reduce the BN statistics of the output in the epilogue
};

static inline CUtensorMapDataType tm_dtype(int etype) {
  return etype == ET_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
}

static void encode_tiled_2d(Handle* h, CUtensorMap* tm, int etype, const void* base, uint64_t inner, uint64_t outer,
                            uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer, int swizzle_bytes) {
  const TmKey key{{1, (uint64_t)(uintptr_t)base, inner, outer, row_stride_bytes, ((uint64_t)box_inner << 32) | box_outer,
                   ((uint64_t)etype << 32) | (uint32_t)swizzle_bytes, 0}};
  auto it = h->tm_cache.find(key);
  if (it != h->tm_cache.end()) { *tm = it->second; return; }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                        : swizzle_bytes == 64  ? CU_TENSOR_MAP_SWIZZLE_64B
                        : swizzle_bytes == 32  ? CU_TENSOR_MAP_SWIZZLE_32B
                                               : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = h->encodeTiled(tm, tm_dtype(etype), 2, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DRS_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d): inner=%llu outer=%llu stride=%llu box=%ux%u", (int)r,
            (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)row_stride_bytes, box_inner,
            box_outer);
  if (h->tm_cache.size() > 4096) h->tm_cache.clear();
  h->tm_cache[key] = *tm;
}

// NHWC activation tensor seen as (C, W, H, N); the bounding box of base pixels is the output raster.
static void encode_im2col(Handle* h, CUtensorMap* tm, int etype, const void* base, int cstride, int crop, int B,
                          int pad_b, int channels_per_pixel, int pixels_per_column, int swizzle_bytes) {
  const TmKey key{{2, (uint64_t)(uintptr_t)base, (uint64_t)cstride, ((uint64_t)crop << 32) | (uint32_t)B, (uint64_t)(uint32_t)pad_b,
                   ((uint64_t)channels_per_pixel << 32) | (uint32_t)pixels_per_column,
                   ((uint64_t)etype << 32) | (uint32_t)swizzle_bytes, 0}};
  auto it = h->tm_cache.find(key);
  if (it != h->tm_cache.end()) { *tm = it->second; return; }
  cuuint64_t dims[4] = {(cuuint64_t)cstride, (cuuint64_t)crop, (cuuint64_t)crop, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)cstride * 2, (cuuint64_t)cstride * 2 * crop, (cuuint64_t)cstride * 2 * crop * crop};
  // SAME, stride 1: lower = -pad_before; upper = pad_after - (k-1)*rate = -pad_before  (W, H order)
  int lower[2] = {-pad_b, -pad_b};
  int upper[2] = {-pad_b, -pad_b};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                        : swizzle_bytes == 64  ? CU_TENSOR_MAP_SWIZZLE_64B
                        : swizzle_bytes == 32  ? CU_TENSOR_MAP_SWIZZLE_32B
                                               : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = h->encodeIm2col(tm, tm_dtype(etype), 4, const_cast<void*>(base), dims, strides, lower, upper,
                               (cuuint32_t)channels_per_pixel, (cuuint32_t)pixels_per_column, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DRS_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeIm2col failed (%d): C=%d crop=%d B=%d pad=%d cpp=%d", (int)r, cstride,
            crop, B, pad_b, channels_per_pixel);
  // Known driver issue (<= 13.1) for small tensors in im2col mode; same workaround the CUTLASS headers apply.
  if (h->driver_version <= 13010) {
    size_t bytes = (size_t)cstride * 2 * crop * crop * B;
    if (bytes < 131072) reinterpret_cast<uint64_t*>(tm)[1] &= ~(1ull << 21);
  }
  if (h->tm_cache.size() > 4096) h->tm_cache.clear();
  h->tm_cache[key] = *tm;
}

static int g_conv_exp_mode = -1;   // drs_bench_conv override of DRS_EXP_MODE
#ifndef CONV_TC_KPS2_MAX_CO
#define CONV_TC_KPS2_MAX_CO 128      // two K blocks per stage for Co <= this
#endif

// two CTAs per SM for the small-N layers.  Measured per 0.76 M-pixel chunk (profiles/r2_conv_two_cta.txt): N=32 161 -> 119 us,
// N=64 208 -> 190 / 138 -> 130 / 253 -> 237 us; at N=128 the halved shared memory leaves only two 32 KB K blocks in flight
// per CTA and it loses (184 -> 199, 341 -> 371 us).
static inline bool conv_tc_two_cta(int co) { return co <= 64; }

template <int BLOCK_K, int EPI_C, typename OutT>
static void launch_conv_tc_t(Handle* h, const ConvTcArgs& a) {
  alignas(64) CUtensorMap tmA, tmB, tmC;
  const int64_t M = (int64_t)a.B * a.crop * a.crop;
  const int taps = a.k * a.k;
  const int sw_op = BLOCK_K * 2;
  // experiment word: bits 0-7 timing mode, bits 12-15 K blocks per stage (0 = default), bit 16 instrumented twin,
  // bits 20-21 tile pairing (1 = single units, 2 = pairs)
  const int exp_word = g_conv_exp_mode >= 0 ? g_conv_exp_mode : (getenv("DRS_EXP_MODE") ? atoi(getenv("DRS_EXP_MODE")) : 0);
  const int exp_mode = exp_word & 0xff;
  const bool instr = ((exp_word >> 16) & 1) != 0;
  const int taps_kb = taps * (a.ci / BLOCK_K);
  int kps = ((exp_word >> 12) & 0xf) ? ((exp_word >> 12) & 0xf) : (a.co <= CONV_TC_KPS2_MAX_CO ? 2 : 1);
  if (kps > taps_kb) kps = taps_kb;
  encode_im2col(h, &tmA, a.etype, a.in, a.in_cstride, a.crop, a.B, a.pad_b, BLOCK_K, CONV_TC_BM, sw_op);
  encode_tiled_2d(h, &tmB, a.etype, a.w, (uint64_t)taps * a.ci, (uint64_t)a.co, (uint64_t)taps * a.ci * 2, BLOCK_K,
                  (uint32_t)a.co, sw_op);
  encode_tiled_2d(h, &tmC, a.etype, a.out, (uint64_t)a.out_cstride, (uint64_t)M, (uint64_t)a.out_cstride * 2, EPI_C,
                  CONV_TC_BM, EPI_C * 2);

  ConvTcParams p;
  p.M_total = (int)M;
  p.crop = a.crop;
  p.ksize = a.k;
  p.rate = a.rate;
  p.pad_b = a.pad_b;
  p.ci = a.ci;
  p.in_coff = a.in_coff;
  p.co = a.co;
  p.out_coff = a.out_coff;
  p.num_tiles = (int)ceil_div(M, CONV_TC_BM);
  p.acc_stride = a.co <= 32 ? 32 : a.co <= 64 ? 64 : a.co <= 128 ? 128 : 256;
  p.act = a.act;
  p.idesc = make_idesc_f16(128, a.co, a.etype == ET_BF16, a.etype == ET_BF16, 0, 0);
  p.scale = a.scale;
  p.shift = a.shift;
  p.diag = h->diag_dev;
  p.exp_mode = exp_mode;
  if (a.stats) p.stats = *a.stats; else memset(&p.stats, 0, sizeof(p.stats));

  // Pairs of 128-pixel units on one filter slice (mt = 2) for Co <= 128.  These layers are bound by the bytes an SM takes in
  // per MMA (an im2col K block is 16 KB of A plus Co*128 B of B for 128*64*Co MACs); two units per filter slice cut them from
  // 24 to 20 KB per unit (Co = 64) and from 32 to 24 KB (Co = 128).  Needs 4 * acc_stride <= 512 TMEM columns, hence not
  // above 128.  Experiment bits 20-21: 1 = force single units, 2 = force pairs.
  const int m2_force = (exp_word >> 20) & 3;
  const int mt = (a.co <= 128 && M > CONV_TC_BM && (m2_force == 0 || m2_force == 2)) ? 2 : 1;
  if (mt == 2 && !((exp_word >> 12) & 0xf)) kps = 1;                 // a pair is already two im2col tiles per barrier round
  if (kps > taps_kb) kps = taps_kb;
  const int kb_bytes = mt * CONV_TC_BM * BLOCK_K * 2 + a.co * BLOCK_K * 2;
  const int fixed = 2 * CONV_TC_BM * EPI_C * 2 + 2 * 256 * 4 + (2 * 8 + 4) * 8 + 16;   // (statistics: registers, no smem)
  // Co <= 64: two CTAs per SM.  One CTA's two single-thread roles (TMA issue, MMA issue) need ~600 cycles per stage whatever
  // the layer, against 256 (N=64) / 512 (N=128) cycles of tensor work: a second resident CTA, with its own producers, issuer
  // and accumulators, fills the tensor pipe in the gaps.  Needs <= 128 registers (the EPI_C=32 instantiation: 106), half
  // the shared memory (113 KB) and half the TMEM (2 x 128 columns) per CTA.
  const bool two_cta = conv_tc_two_cta(a.co) && EPI_C == 32;
  const int budget = two_cta ? 113 * 1024 : 227 * 1024;
  if ((budget - fixed) / (kps * kb_bytes) < 2) kps = 1;
  const int stage_bytes = kps * kb_bytes;
  int stages = (budget - fixed) / stage_bytes;
  // at most 8 K blocks in flight: small layers then leave room for a second CTA on the SM (the filter-gradient kernel
  // of the side stream in training; without it a batch-64 crop-25 DenseDilated6 step is 20 % slower)
  if (stages > 8 / (kps * mt)) stages = std::max(2, 8 / (kps * mt));
  DRS_CHECK(stages >= 2, "conv_tc: tile does not fit shared memory (co=%d)", a.co);
  p.stages = stages;
  p.kps = kps;
  p.mt = mt;
  p.tmem_cols = 2 * mt * p.acc_stride;
  p.smem_needed = fixed + stages * stage_bytes;
  const int smem_bytes = p.smem_needed + 1024 <= budget ? p.smem_needed + 1024 : budget;
  p.smem_provided = smem_bytes;

  const int max_ctas = two_cta ? 2 * h->sm_count : h->sm_count;
  int grid = p.num_tiles < max_ctas ? p.num_tiles : max_ctas;
  if (instr && BLOCK_K == 64 && EPI_C == 64) {
    // instrumented twin (clock64 around every barrier wait of CTA 0, written to the diagnostic words): bench only
    auto kern = conv_tc_kernel<64, 64, OutT, true>;
    static bool attr_set_i = false;
    if (!attr_set_i) {
      CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, budget));
      attr_set_i = true;
    }
    kern<<<grid, CONV_TC_THREADS, smem_bytes, h->stream>>>(tmA, tmB, tmC, p);
  } else {
    auto kern = conv_tc_kernel<BLOCK_K, EPI_C, OutT, false>;
    static bool attr_set = false;
    if (!attr_set) {
      CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      attr_set = true;
    }
    launch_pdl(h, kern, dim3(grid), dim3(CONV_TC_THREADS), (size_t)smem_bytes, tmA, tmB, tmC, p);
  }
  LAUNCH_CHECK(h);
}

// Dispatch on K-step width and epilogue box; requirements are checked loudly.
static void launch_conv_tc(Handle* h, const ConvTcArgs& a) {
  DRS_CHECK(a.ci % 32 == 0, "conv_tc: Ci=%d must be a multiple of 32", a.ci);
  DRS_CHECK(a.co % 32 == 0 && a.co >= 32 && a.co <= 256, "conv_tc: Co=%d must be a multiple of 32 in [32,256]", a.co);
  DRS_CHECK(a.in_cstride % 8 == 0 && a.out_cstride % 8 == 0, "conv_tc: channel strides must be multiples of 8");
  DRS_CHECK(a.in_coff % 8 == 0 && a.out_coff % 8 == 0, "conv_tc: channel offsets must be multiples of 8");
  const bool k64 = (a.ci % 64 == 0);
  const bool e64 = (a.co % 64 == 0) && !conv_tc_two_cta(a.co);     // two CTAs per SM use the 32-channel epilogue box
  if (a.etype == ET_F16) {
    if (k64 && e64) launch_conv_tc_t<64, 64, __half>(h, a);
    else if (k64) launch_conv_tc_t<64, 32, __half>(h, a);
    else if (e64) launch_conv_tc_t<32, 64, __half>(h, a);
    else launch_conv_tc_t<32, 32, __half>(h, a);
  } else {
    if (k64 && e64) launch_conv_tc_t<64, 64, __nv_bfloat16>(h, a);
    else if (k64) launch_conv_tc_t<64, 32, __nv_bfloat16>(h, a);
    else if (e64) launch_conv_tc_t<32, 64, __nv_bfloat16>(h, a);
    else launch_conv_tc_t<32, 32, __nv_bfloat16>(h, a);
  }
}
