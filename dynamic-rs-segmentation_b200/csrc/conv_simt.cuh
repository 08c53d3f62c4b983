// CUDA-core fp32 implicit-GEMM convolutions with a fixed reduction order ("exact-order" mode,
// DRS_PREC_FP32) and the layers that do not belong on the tensor cores: conv1 (Ci = 3..5, K = 75..125,
// HBM-bound) in every precision.  Reference op: _conv_layer, isprs:700-723.
#pragma once
#include "drs_common.cuh"

constexpr int SIMT_BM = 64, SIMT_BN = 64, SIMT_BK = 16, SIMT_THREADS = 256;

// out[m, co] = act( (sum_{tap,c} in[pix(m)+tap][c] * w[(tap*ci+c)*co_total + co]) * scale[co] + shift[co] )
// w is HWIO flattened ([k*k*ci][co_total]) -- exactly the TF variable layout, no packing needed.
template <typename TIn, typename TOut>
__global__ void __launch_bounds__(SIMT_THREADS)
conv_simt_kernel(const TIn* __restrict__ in, int in_cstride, int in_coff, int ci, const float* __restrict__ w,
                 TOut* __restrict__ out, int out_cstride, int out_coff, int co, int M, int crop, int ksize, int rate,
                 int pad_b, const float* __restrict__ scale, const float* __restrict__ shift, int act) {
  __shared__ float As[SIMT_BK][SIMT_BM + 4];
  __shared__ float Bs[SIMT_BK][SIMT_BN + 4];
  const int t = threadIdx.x;
  const int m0 = blockIdx.x * SIMT_BM;
  const int n0 = blockIdx.y * SIMT_BN;
  const int Ktot = ksize * ksize * ci;
  const int cc = crop * crop;

  // A-load slots: kk_local = t % 16, pixels (t / 16) + 16 * i
  const int a_kk = t & 15;
  int a_n[4], a_y[4], a_x[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + (t >> 4) + 16 * i;
    if (m < M) {
      a_n[i] = m / cc;
      int r = m - a_n[i] * cc;
      a_y[i] = r / crop;
      a_x[i] = r - a_y[i] * crop;
    } else {
      a_n[i] = -1;
      a_y[i] = a_x[i] = 0;
    }
  }
  const int b_co = t & 63;
  const int b_kk = t >> 6;

  const int tx = t & 15, ty = t >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

  for (int k0 = 0; k0 < Ktot; k0 += SIMT_BK) {
    {
      const int kk = k0 + a_kk;
      int tap = 0, c = 0, dy = 0, dx = 0;
      const bool kvalid = kk < Ktot;
      if (kvalid) {
        tap = kk / ci;
        c = kk - tap * ci;
        const int ky = tap / ksize, kx = tap - ky * ksize;
        dy = ky * rate - pad_b;
        dx = kx * rate - pad_b;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float v = 0.0f;
        if (kvalid && a_n[i] >= 0) {
          const int iy = a_y[i] + dy, ix = a_x[i] + dx;
          if (iy >= 0 && iy < crop && ix >= 0 && ix < crop)
            v = to_f32(in[((int64_t)(a_n[i] * crop + iy) * crop + ix) * in_cstride + in_coff + c]);
        }
        As[a_kk][(t >> 4) + 16 * i] = v;
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kk = k0 + b_kk + 4 * i;
      float v = 0.0f;
      if (kk < Ktot && n0 + b_co < co) v = w[(int64_t)kk * co + n0 + b_co];
      Bs[b_kk + 4 * i][b_co] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SIMT_BK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= co) continue;
      const float v = apply_act(fmaf(acc[i][j], scale[n], shift[n]), act);
      out[(int64_t)m * out_cstride + out_coff + n] = from_f32<TOut>(v);
    }
  }
}

template <typename TIn, typename TOut>
static void launch_conv_simt(Handle* h, const TIn* in, int in_cstride, int in_coff, int ci, const float* w, TOut* out,
                             int out_cstride, int out_coff, int co, int B, int crop, int k, int rate, int pad_b,
                             const float* scale, const float* shift, int act) {
  const int64_t M = (int64_t)B * crop * crop;
  dim3 grid((unsigned)ceil_div(M, SIMT_BM), (unsigned)ceil_div(co, SIMT_BN));
  conv_simt_kernel<TIn, TOut><<<grid, SIMT_THREADS, 0, h->stream>>>(in, in_cstride, in_coff, ci, w, out, out_cstride,
                                                                    out_coff, co, (int)M, crop, k, rate, pad_b, scale,
                                                                    shift, act);
  LAUNCH_CHECK(h);
}

// ------------------------------------------------------------------------------------------------
// wgrad (fp32, fixed order): dW[kk][co] = sum_m A[m][kk] * dY[m][co], split over pixel ranges.
// part[s][kk][co] for split s; reduced in split order by reduce_partials_kernel.
// ------------------------------------------------------------------------------------------------
template <typename TIn, typename TG>
__global__ void __launch_bounds__(SIMT_THREADS)
wgrad_simt_kernel(const TIn* __restrict__ in, int in_cstride, int in_coff, int ci, const TG* __restrict__ dy,
                  int dy_cstride, int dy_coff, int co, float* __restrict__ part, int M, int crop, int ksize, int rate,
                  int pad_b, int m_per_split) {
  __shared__ float As[SIMT_BK][SIMT_BM + 4];   // [m][kk]
  __shared__ float Bs[SIMT_BK][SIMT_BN + 4];   // [m][co]
  const int t = threadIdx.x;
  const int k0 = blockIdx.x * SIMT_BM;
  const int n0 = blockIdx.y * SIMT_BN;
  const int split = blockIdx.z;
  const int Ktot = ksize * ksize * ci;
  const int cc = crop * crop;
  const int m_begin = split * m_per_split;
  const int m_end = min(M, m_begin + m_per_split);

  const int a_kk = k0 + (t & 63);
  int c = 0, dyo = 0, dxo = 0;
  const bool kvalid = a_kk < Ktot;
  if (kvalid) {
    const int tap = a_kk / ci;
    c = a_kk - tap * ci;
    const int ky = tap / ksize, kx = tap - ky * ksize;
    dyo = ky * rate - pad_b;
    dxo = kx * rate - pad_b;
  }
  const int tx = t & 15, ty = t >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

  for (int mb = m_begin; mb < m_end; mb += SIMT_BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int ml = (t >> 6) + 4 * i;
      const int m = mb + ml;
      float va = 0.0f, vb = 0.0f;
      if (m < m_end) {
        if (kvalid) {
          const int n = m / cc;
          const int r = m - n * cc;
          const int y = r / crop, x = r - y * crop;
          const int iy = y + dyo, ix = x + dxo;
          if (iy >= 0 && iy < crop && ix >= 0 && ix < crop)
            va = to_f32(in[((int64_t)(n * crop + iy) * crop + ix) * in_cstride + in_coff + c]);
        }
        if (n0 + (t & 63) < co) vb = to_f32(dy[(int64_t)m * dy_cstride + dy_coff + n0 + (t & 63)]);
      }
      As[ml][t & 63] = va;
      Bs[ml][t & 63] = vb;
    }
    __syncthreads();
#pragma unroll
    for (int mm = 0; mm < SIMT_BK; ++mm) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[mm][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[mm][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int kk = k0 + ty * 4 + i;
    if (kk >= Ktot) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= co) continue;
      part[((int64_t)split * Ktot + kk) * co + n] = acc[i][j];
    }
  }
}

// out[i] = sum_{s=0..S-1} part[s][i].  Block = 32 float4 columns x 8 split lanes: lane j adds splits j, j+8, ... in order,
// the 8 lane sums are combined in lane order through shared memory -> a fixed summation tree (deterministic) with 8x
// the memory parallelism of a serial loop.  n is a multiple of 4 for every caller (Co % 4 == 0) except the classifier's
// bias row, which takes the scalar path.
constexpr int RP_COLS = 32, RP_LANES = 8, RP_MAX_LANES = 32;
__global__ void __launch_bounds__(RP_COLS * RP_MAX_LANES)
reduce_partials_kernel(const float* __restrict__ part, float* __restrict__ out, int64_t n, int S, int64_t stride = 0) {
  pdl_sync();
  if (stride == 0) stride = n;                         // distance between two splits (> n: only the first n entries are wanted)
  __shared__ float4 s_acc[RP_MAX_LANES][RP_COLS];
  const int lanes = blockDim.x / RP_COLS;              // 8, or 32 for a narrow result with many splits (reduce_partials_block)
  const int tx = threadIdx.x % RP_COLS, ty = threadIdx.x / RP_COLS;
  if ((n & 3) != 0) {                                  // tiny scalar case: one warp per column, fixed shuffle tree
    const int lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * lanes + (threadIdx.x >> 5);
    float a = 0.0f;
    if (i < n)
      for (int k = lane; k < S; k += 32) a += part[(int64_t)k * stride + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (i < n && lane == 0) out[i] = a;
    return;
  }
  const int64_t i4 = ((int64_t)blockIdx.x * RP_COLS + tx) * 4;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i4 < n) {
#pragma unroll 4
    for (int k = ty; k < S; k += lanes) {
      const float4 v = __ldcs(reinterpret_cast<const float4*>(part + (int64_t)k * stride + i4));
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
  }
  s_acc[ty][tx] = a;
  __syncthreads();
  if (ty == 0 && i4 < n) {
    for (int j = 1; j < lanes; ++j) {
      const float4 v = s_acc[j][tx];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    *reinterpret_cast<float4*>(out + i4) = a;
  }
}
// threads per block: a narrow result reduced over many splits (the classifier's 592 block partials of 1536 values) is a
// latency chain of S / lanes dependent rounds in a dozen blocks -> 32 split lanes instead of 8
static inline unsigned reduce_partials_block(int64_t n, int S) {
  return (unsigned)(RP_COLS * ((n <= 16384 && S > 64 && (n & 3) == 0) ? RP_MAX_LANES : RP_LANES));
}
static inline unsigned reduce_partials_grid(int64_t n) {
  return (unsigned)((n & 3) ? ceil_div(n, RP_LANES) : ceil_div(n, 4 * RP_COLS));
}

template <typename TIn, typename TG>
static void launch_wgrad_simt(Handle* h, const TIn* in, int in_cstride, int in_coff, int ci, const TG* dy,
                              int dy_cstride, int dy_coff, int co, float* dw, float* part, int max_splits, int B,
                              int crop, int k, int rate, int pad_b, int m_per_split_target = 2048) {
  const int64_t M = (int64_t)B * crop * crop;
  const int Ktot = k * k * ci;
  int splits = (int)ceil_div(M, m_per_split_target);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  int m_per = (int)round_up(ceil_div(M, splits), SIMT_BK);
  splits = (int)ceil_div(M, m_per);
  dim3 grid((unsigned)ceil_div(Ktot, SIMT_BM), (unsigned)ceil_div(co, SIMT_BN), (unsigned)splits);
  wgrad_simt_kernel<TIn, TG><<<grid, SIMT_THREADS, 0, h->stream>>>(in, in_cstride, in_coff, ci, dy, dy_cstride, dy_coff,
                                                                   co, part, (int)M, crop, k, rate, pad_b, m_per);
  LAUNCH_CHECK(h);
  const int64_t n = (int64_t)Ktot * co;
  reduce_partials_kernel<<<reduce_partials_grid(n), RP_COLS * RP_LANES, 0, h->stream>>>(part, dw, n, splits);
  LAUNCH_CHECK(h);
}

// ------------------------------------------------------------------------------------------------
// conv1 filter gradient (5x5, rate 1, Ci = C <= 8 image channels, Co = 64; isprs:767 / 1687): K = 25*C rows only, so the
// generic tiled kernel above runs at a few % of anything.  Here a CTA owns (image, band of rows): the band of the fp32
// input patch with its 2-pixel zero halo and the band's dZ rows sit in shared memory, thread = (output channel, tap group of <= 7 taps) keeps
// 7 x C accumulators in registers and walks the band's pixels: one dZ load and 7 broadcast LDS.128 per pixel.
// Partials part[cta][tap*C + c][co] are reduced in CTA order by reduce_partials_kernel (deterministic).
// ------------------------------------------------------------------------------------------------
template <typename TG, int CP>
__global__ void __launch_bounds__(256)
wgrad_conv1_kernel(const float* __restrict__ x, int C, const TG* __restrict__ dy, int dy_cs, int dy_co, float* __restrict__ part,
                   int crop, int bands, int rows_per_band) {
  extern __shared__ __align__(16) float xs[];          // [(rows + 4)][crop + 4][CP]
  const int img = blockIdx.x / bands, band = blockIdx.x - img * bands;
  const int y0 = band * rows_per_band, y1 = min(crop, y0 + rows_per_band);
  const int W = crop + 4;
  const int tid = threadIdx.x;
  for (int i = tid; i < (y1 - y0 + 4) * W; i += 256) {
    const int ry = i / W, rx = i - ry * W;
    const int gy = y0 - 2 + ry, gx = rx - 2;
    const bool in = gy >= 0 && gy < crop && gx >= 0 && gx < crop;
    const float* src = x + ((int64_t)(img * crop + gy) * crop + gx) * C;
#pragma unroll
    for (int c = 0; c < CP; ++c) xs[i * CP + c] = (in && c < C) ? src[c] : 0.0f;
  }
  // the band's dZ rows, staged with 16-byte loads (a per-pixel global load in the loop below would be latency-bound)
  TG* dzs = reinterpret_cast<TG*>(xs + (size_t)(rows_per_band + 4) * W * CP);
  {
    constexpr int V = 16 / sizeof(TG);                 // elements per 16-byte vector
    const int per_px = 64 / V;
    const int npx = (y1 - y0) * crop;
    const TG* src = dy + (int64_t)(img * crop + y0) * crop * dy_cs + dy_co;
    for (int i = tid; i < npx * per_px; i += 256) {
      const int px = i / per_px, v = i - px * per_px;
      *reinterpret_cast<uint4*>(dzs + px * 64 + v * V) = *reinterpret_cast<const uint4*>(src + (int64_t)px * dy_cs + v * V);
    }
  }
  __syncthreads();
  const int co = tid & 63, tg = tid >> 6;
  int off[7];
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const int tap = min(tg + 4 * j, 24);
    off[j] = ((tap / 5) * W + (tap % 5)) * CP;
  }
  float acc[7][CP];
#pragma unroll
  for (int j = 0; j < 7; ++j)
#pragma unroll
    for (int c = 0; c < CP; ++c) acc[j][c] = 0.0f;
  for (int y = y0; y < y1; ++y) {
    const TG* dyp = dzs + (y - y0) * crop * 64 + co;
    const float* row = xs + (y - y0) * W * CP;
#pragma unroll 2
    for (int xx = 0; xx < crop; ++xx) {
      const float dz = to_f32(dyp[xx * 64]);
      const float* p = row + xx * CP;
#pragma unroll
      for (int j = 0; j < 7; ++j) {
#pragma unroll
        for (int q = 0; q < CP / 4; ++q) {
          const float4 v = *reinterpret_cast<const float4*>(p + off[j] + 4 * q);
          acc[j][4 * q + 0] = fmaf(v.x, dz, acc[j][4 * q + 0]);
          acc[j][4 * q + 1] = fmaf(v.y, dz, acc[j][4 * q + 1]);
          acc[j][4 * q + 2] = fmaf(v.z, dz, acc[j][4 * q + 2]);
          acc[j][4 * q + 3] = fmaf(v.w, dz, acc[j][4 * q + 3]);
        }
      }
    }
  }
  float* dst = part + (int64_t)blockIdx.x * 25 * C * 64;
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const int tap = tg + 4 * j;
    if (tap < 25) {
#pragma unroll
      for (int c = 0; c < CP; ++c)
        if (c < C) dst[(tap * C + c) * 64 + co] = acc[j][c];
    }
  }
}

// returns false when the shape is not the conv1 shape (caller falls back to the generic kernel)
template <typename TG>
static bool launch_wgrad_conv1(Handle* h, const float* x, int C, const TG* dy, int dy_cs, int dy_co, int co, float* dw, float* part,
                               size_t part_capacity, int B, int crop, int k, int rate) {
  if (k != 5 || rate != 1 || co != 64 || C < 1 || C > 8) return false;
  const int CP = C <= 4 ? 4 : 8;
  int bands = (int)std::min<int64_t>(std::max<int64_t>(1, ceil_div((int64_t)h->sm_count * 2, B)), std::max(1, crop / 4));
  int rows = (int)ceil_div(crop, bands);
  bands = (int)ceil_div(crop, rows);
  const int64_t n = (int64_t)25 * C * 64;
  while (bands > 1 && (size_t)B * bands * n > part_capacity) {
    rows *= 2;
    bands = (int)ceil_div(crop, rows);
  }
  if ((size_t)B * bands * n > part_capacity) return false;
  const size_t smem = (size_t)(rows + 4) * (crop + 4) * CP * 4 + (size_t)rows * crop * 64 * sizeof(TG);
  if (smem > 200 * 1024) return false;
  if (CP == 4) {
    auto kern = wgrad_conv1_kernel<TG, 4>;
    static size_t attr4 = 0;
    if (smem > 48 * 1024 && smem > attr4) { CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); attr4 = 200 * 1024; }
    kern<<<B * bands, 256, smem, h->stream>>>(x, C, dy, dy_cs, dy_co, part, crop, bands, rows);
  } else {
    auto kern = wgrad_conv1_kernel<TG, 8>;
    static size_t attr8 = 0;
    if (smem > 48 * 1024 && smem > attr8) { CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); attr8 = 200 * 1024; }
    kern<<<B * bands, 256, smem, h->stream>>>(x, C, dy, dy_cs, dy_co, part, crop, bands, rows);
  }
  LAUNCH_CHECK(h);
  reduce_partials_kernel<<<reduce_partials_grid(n), RP_COLS * RP_LANES, 0, h->stream>>>(part, dw, n, B * bands);
  LAUNCH_CHECK(h);
  return true;
}
