// HBM-bound layers of the path: 3x3 stride-1 SAME max-pool (fwd/bwd), batch-norm without gamma/beta
// (statistics, apply, backward), 1x1 classifier (fwd/bwd), softmax cross-entropy (+grad, argmax),
// momentum update.  All reductions are two-stage with a fixed order (no float atomics), so every
// result is run-to-run deterministic.  Activations are NHWC with a channel stride/offset so that the
// dense net's concat (isprs:921-948) is a view, never a copy.
#pragma once
#include <algorithm>

#include "drs_common.cuh"

// resident blocks per SM the HBM-side training kernels are compiled for (register cap = 65536 / (256 * n)); A/B knobs
#ifndef DRS_BN_MINBLK
#define DRS_BN_MINBLK 2      // resident blocks per SM the statistics kernel is compiled for (register cap 65536 / (256 * n))
#endif
#ifndef DRS_BNE_MINBLK
#define DRS_BNE_MINBLK 1
#endif
#ifndef DRS_POOL_MINBLK
#define DRS_POOL_MINBLK 1
#endif

template <typename T>
struct alignas(16) Vec8 {
  T v[8];
};

// ------------------------------------------------------------------------------------------------
// _max_pool(kernel 3x3, stride 1, SAME)  isprs:745-750.  Padding never wins (window clipped).
// idx (optional, training): position 0..8 of the first maximum in row-major window order.
// ------------------------------------------------------------------------------------------------
// Column-sliding formulation: a thread owns (image, column x, 8 channels) and walks down a segment of rows keeping
// the horizontal 3-max of the two previous rows in registers, so every input element is loaded 3 times (from L1)
// instead of 9.  Adjacent threads cover adjacent channel groups, then adjacent columns: each row access of a warp is
// one contiguous run.
template <typename T>
__device__ __forceinline__ void pool_row_max(const T* __restrict__ in, int in_cs, int64_t pix_row0, int x, int crop, int y,
                                             float (&v)[8], int (&d)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) { v[e] = -INFINITY; d[e] = 0; }
  if (y < 0 || y >= crop) return;
#pragma unroll
  for (int dx = -1; dx <= 1; ++dx) {
    const int xx = x + dx;
    if (xx < 0 || xx >= crop) continue;
    const Vec8<T> q = *reinterpret_cast<const Vec8<T>*>(in + (pix_row0 + (int64_t)y * crop + xx) * in_cs);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float f = to_f32(q.v[e]);
      if (f > v[e]) { v[e] = f; d[e] = dx + 1; }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
maxpool3_fwd_kernel(const T* __restrict__ in, int in_cs, int in_co, T* __restrict__ out, int out_cs, int out_co,
                    uint8_t* __restrict__ idx, int C, int B, int crop, int seg, int nseg, const float* __restrict__ bn_mean,
                    const float* __restrict__ bn_inv_std, int act) {
  const int cv = C >> 3;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)B * nseg * crop * cv) return;
  const int cg = (int)(gid % cv);
  int64_t t = gid / cv;
  const int x = (int)(t % crop);
  t /= crop;
  const int sg = (int)(t % nseg);
  const int b = (int)(t / nseg);
  const int y0 = sg * seg, y1 = min(crop, y0 + seg);
  const int64_t img0 = (int64_t)b * crop * crop;
  const T* inp = in + in_co + cg * 8;
  float r0[8], r1[8], r2[8];
  int d0[8], d1[8], d2[8];
  // Training forward of the pooling nets: max-pool commutes with the (strictly increasing) normalise + LeakyReLU, so the
  // pool runs on the raw conv output and act((max - mean) * inv_std) is applied to the winner only.
  float mu[8], is[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { mu[e] = bn_mean[cg * 8 + e]; is[e] = bn_inv_std[cg * 8 + e]; }
  pool_row_max<T>(inp, in_cs, img0, x, crop, y0 - 1, r0, d0);
  pool_row_max<T>(inp, in_cs, img0, x, crop, y0, r1, d1);
  for (int y = y0; y < y1; ++y) {
    pool_row_max<T>(inp, in_cs, img0, x, crop, y + 1, r2, d2);
    Vec8<T> o;
    int code[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      // rows in order dy = -1, 0, +1; a later row wins only when strictly greater (first maximum, row-major)
      float best = r0[e];
      int c = d0[e];
      if (r1[e] > best) { best = r1[e]; c = 3 + d1[e]; }
      if (r2[e] > best) { best = r2[e]; c = 6 + d2[e]; }
      best = apply_act((best - mu[e]) * is[e], act);
      o.v[e] = from_f32<T>(best);
      code[e] = c;
    }
    const int64_t m = img0 + (int64_t)y * crop + x;
    *reinterpret_cast<Vec8<T>*>(out + m * out_cs + out_co + cg * 8) = o;
    uint2 pk;
    pk.x = code[0] | (code[1] << 8) | (code[2] << 16) | (code[3] << 24);
    pk.y = code[4] | (code[5] << 8) | (code[6] << 16) | (code[7] << 24);
    *reinterpret_cast<uint2*>(idx + m * C + cg * 8) = pk;
#pragma unroll
    for (int e = 0; e < 8; ++e) { r0[e] = r1[e]; r1[e] = r2[e]; d0[e] = d1[e]; d1[e] = d2[e]; }
  }
}

// Inference variant (no winner codes, no fused normalisation): the 16-bit types are reduced with packed 2-wide max
// instructions and never converted, which takes the kernel from issue-bound to memory-bound.
__device__ __forceinline__ void vmax8(Vec8<float>& a, const Vec8<float>& b) {
#pragma unroll
  for (int e = 0; e < 8; ++e) a.v[e] = fmaxf(a.v[e], b.v[e]);
}
__device__ __forceinline__ void vmax8(Vec8<__half>& a, const Vec8<__half>& b) {
  __half2* pa = reinterpret_cast<__half2*>(a.v);
  const __half2* pb = reinterpret_cast<const __half2*>(b.v);
#pragma unroll
  for (int e = 0; e < 4; ++e) pa[e] = __hmax2(pa[e], pb[e]);
}
__device__ __forceinline__ void vmax8(Vec8<__nv_bfloat16>& a, const Vec8<__nv_bfloat16>& b) {
  __nv_bfloat162* pa = reinterpret_cast<__nv_bfloat162*>(a.v);
  const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(b.v);
#pragma unroll
  for (int e = 0; e < 4; ++e) pa[e] = __hmax2(pa[e], pb[e]);
}

// Two columns per thread, next row's loads in flight.  The reads are latency-bound: with one column per thread a thread
// has one row of loads outstanding and two of its three 16-byte loads hit L1 (the neighbours' centres), so only 16 unique
// bytes per thread are on their way from DRAM at any time.  Here a thread owns columns (x0, x0+1): four loads per row for
// two outputs (x0-1, x0, x0+1, x0+2), three packed maxima for the two horizontal results (the centre pair's maximum is
// shared), and the loads of row y+2 are issued before row y+1 is reduced.  Measured against the one-column kernel: the
// seven pools of a 0.76 M-pixel Dilated8Pooling chunk 722 -> ~600 us (5.2 TB/s of read + write traffic, 80 % of the
// measured HBM peak), the scene pass -3 % (profiles/r2c_conv_pairs_uniform_ab.txt, section 7).  Same bits: max is exact.
template <typename T>
__global__ void __launch_bounds__(256)
maxpool3_fwd_packed2_kernel(const T* __restrict__ in, int in_cs, int in_co, T* __restrict__ out, int out_cs, int out_co, int C,
                            int B, int crop, int seg, int nseg) {
  const int cv = C >> 3;
  const int xp_n = (crop + 1) >> 1;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)B * nseg * xp_n * cv) return;
  const int cg = (int)(gid % cv);
  int64_t t = gid / cv;
  const int x0 = (int)(t % xp_n) * 2;
  t /= xp_n;
  const int sg = (int)(t % nseg);
  const int b = (int)(t / nseg);
  const int y0 = sg * seg, y1 = min(crop, y0 + seg);
  const bool has1 = x0 + 1 < crop;
  // element offsets of the four columns relative to the centre x0 (missing neighbours point at a valid column: max is idempotent)
  const int o_l = x0 > 0 ? -in_cs : 0;
  const int o_1 = has1 ? in_cs : 0;
  const int o_r = x0 + 2 < crop ? 2 * in_cs : o_1;
  const int64_t rs = (int64_t)crop * in_cs;
  const T* q = in + in_co + cg * 8 + ((int64_t)b * crop * crop + (int64_t)y0 * crop + x0) * in_cs;   // centre of the next row to load
  T* po = out + out_co + cg * 8 + ((int64_t)b * crop * crop + (int64_t)y0 * crop + x0) * out_cs;
  const int64_t os = (int64_t)crop * out_cs;
  Vec8<T> nl, n0, n1, nr;                      // raw loads of the next row
  Vec8<T> a0, a1, b0, b1, c0, c1;              // horizontal maxima of rows y-1, y, y+1 for the two columns
  auto load = [&](const T* c) {
    n0 = *reinterpret_cast<const Vec8<T>*>(c);
    nl = *reinterpret_cast<const Vec8<T>*>(c + o_l);
    n1 = *reinterpret_cast<const Vec8<T>*>(c + o_1);
    nr = *reinterpret_cast<const Vec8<T>*>(c + o_r);
  };
  auto reduce = [&](Vec8<T>& h0, Vec8<T>& h1) {
    Vec8<T> m = n0;
    vmax8(m, n1);
    h0 = m; vmax8(h0, nl);
    h1 = m; vmax8(h1, nr);
  };
  bool va = y0 > 0;
  if (va) { load(q - rs); reduce(a0, a1); }
  load(q);
  reduce(b0, b1);
  q += rs;
  bool vn = y0 + 1 < crop;
  if (vn) load(q);
  for (int y = y0; y < y1; ++y) {
    const bool vc = vn;
    if (vc) reduce(c0, c1);
    q += rs;
    vn = y + 2 < crop && y + 1 < y1;
    if (vn) load(q);
    Vec8<T> r0 = b0, r1 = b1;
    if (va) { vmax8(r0, a0); vmax8(r1, a1); }
    if (vc) { vmax8(r0, c0); vmax8(r1, c1); }
    *reinterpret_cast<Vec8<T>*>(po) = r0;
    if (has1) *reinterpret_cast<Vec8<T>*>(po + out_cs) = r1;
    po += os;
    a0 = b0; a1 = b1; va = true;
    b0 = c0; b1 = c1;
  }
}

// Training variant for bf16 (winner codes + fused normalise/activation) on packed 2-wide compare / max / select: a third
// of the instructions of the scalar float version, same first-maximum semantics (strictly-greater replaces, row-major).
// Software-pipelined: the three 16-byte loads of window row y+2 are issued before the arithmetic of row y+1 starts, so a
// thread always has a row of loads in flight (consuming each row's loads immediately is latency-bound: 48 % issue
// utilisation at 17 % DRAM under ncu).  Out-of-image positions load as -inf, which never wins a strictly-greater compare.
struct PoolRawRow { uint4 q[3]; };
__device__ __forceinline__ void pool_load_raw(const __nv_bfloat16* __restrict__ in, int in_cs, int64_t pix_row0, int x, int crop,
                                              int y, PoolRawRow& r) {
  const unsigned ninf2 = 0xFF80FF80u;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int xx = x + j - 1;
    if (y >= 0 && y < crop && xx >= 0 && xx < crop)
      r.q[j] = *reinterpret_cast<const uint4*>(in + (pix_row0 + (int64_t)y * crop + xx) * in_cs);
    else
      r.q[j] = make_uint4(ninf2, ninf2, ninf2, ninf2);
  }
}
__device__ __forceinline__ void pool_hmax_raw(const PoolRawRow& r, __nv_bfloat162 (&rv)[4], unsigned (&ri)[4]) {
  const unsigned ninf2 = 0xFF80FF80u;
#pragma unroll
  for (int w = 0; w < 4; ++w) { rv[w] = *reinterpret_cast<const __nv_bfloat162*>(&ninf2); ri[w] = 0u; }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const __nv_bfloat162* q = reinterpret_cast<const __nv_bfloat162*>(&r.q[j]);
    const unsigned code2 = (unsigned)j * 0x00010001u;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const unsigned m = __hgt2_mask(q[w], rv[w]);
      rv[w] = __hmax2(rv[w], q[w]);
      ri[w] = (ri[w] & ~m) | (code2 & m);
    }
  }
}

__global__ void __launch_bounds__(256, DRS_POOL_MINBLK)
maxpool3_fwd_train_bf16_pipelined_kernel(const __nv_bfloat16* __restrict__ in, int in_cs, int in_co, __nv_bfloat16* __restrict__ out,
                                         int out_cs, int out_co, uint8_t* __restrict__ idx, int C, int B, int crop, int seg, int nseg,
                                         const float* __restrict__ bn_mean, const float* __restrict__ bn_inv_std, int act) {
  const int cv = C >> 3;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)B * nseg * crop * cv) return;
  const int cg = (int)(gid % cv);
  int64_t t = gid / cv;
  const int x = (int)(t % crop);
  t /= crop;
  const int sg = (int)(t % nseg);
  const int b = (int)(t / nseg);
  const int y0 = sg * seg, y1 = min(crop, y0 + seg);
  const int64_t img0 = (int64_t)b * crop * crop;
  const __nv_bfloat16* inp = in + in_co + cg * 8;
  float mu[8], is[8];
  if (bn_mean) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { mu[e] = bn_mean[cg * 8 + e]; is[e] = bn_inv_std[cg * 8 + e]; }
  }
  __nv_bfloat162 v0[4], v1[4], v2[4];
  unsigned i0[4], i1[4], i2[4];
  PoolRawRow ra, rb, cur, nxt;
  pool_load_raw(inp, in_cs, img0, x, crop, y0 - 1, ra);
  pool_load_raw(inp, in_cs, img0, x, crop, y0, rb);
  pool_load_raw(inp, in_cs, img0, x, crop, y0 + 1, cur);
  pool_hmax_raw(ra, v0, i0);
  pool_hmax_raw(rb, v1, i1);
  for (int y = y0; y < y1; ++y) {
    pool_load_raw(inp, in_cs, img0, x, crop, y + 2, nxt);       // in flight while row y+1 is reduced and row y is written
    pool_hmax_raw(cur, v2, i2);
    uint4 o;
    unsigned code[4];
    unsigned* ow = reinterpret_cast<unsigned*>(&o);
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      __nv_bfloat162 best = v0[w];
      unsigned bi = i0[w];
      unsigned m = __hgt2_mask(v1[w], best);
      best = __hmax2(best, v1[w]);
      bi = (bi & ~m) | ((i1[w] + 0x00030003u) & m);
      m = __hgt2_mask(v2[w], best);
      best = __hmax2(best, v2[w]);
      bi = (bi & ~m) | ((i2[w] + 0x00060006u) & m);
      code[w] = bi;
      if (bn_mean) {
        const float lo = apply_act((__low2float(best) - mu[2 * w]) * is[2 * w], act);
        const float hi = apply_act((__high2float(best) - mu[2 * w + 1]) * is[2 * w + 1], act);
        best = __floats2bfloat162_rn(lo, hi);
      }
      ow[w] = *reinterpret_cast<unsigned*>(&best);
    }
    const int64_t m = img0 + (int64_t)y * crop + x;
    *reinterpret_cast<uint4*>(out + m * out_cs + out_co + cg * 8) = o;
    uint2 pk;
    pk.x = __byte_perm(code[0], code[1], 0x6420);      // low byte of every 16-bit lane
    pk.y = __byte_perm(code[2], code[3], 0x6420);
    *reinterpret_cast<uint2*>(idx + m * C + cg * 8) = pk;
#pragma unroll
    for (int w = 0; w < 4; ++w) { v0[w] = v1[w]; v1[w] = v2[w]; i0[w] = i1[w]; i1[w] = i2[w]; }
    cur = nxt;
  }
}

// dIn for bf16, column-sliding like the forward: a thread owns (image, column x, 8 channels) and walks down the rows with
// the winner codes and output gradients of the three window rows it needs held in registers (3x fewer loads than a
// gather per pixel).  Byte-wise code compare, byte mask -> 16-bit lane mask, masked values widened to fp32 by shifts.
struct PoolBwdRow {
  uint2 code[3];     // winner codes of windows (yo, x-1), (yo, x), (yo, x+1); 0xFF.. = window outside the image
  uint4 g[3];        // their output gradients
};
__device__ __forceinline__ void pool_bwd_load(const __nv_bfloat16* __restrict__ dout, int do_cs, const uint8_t* __restrict__ idx,
                                              int C, int64_t img0, int x, int crop, int yo, PoolBwdRow& r) {
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int xo = x + j - 1;
    if (yo >= 0 && yo < crop && xo >= 0 && xo < crop) {
      const int64_t mo = img0 + (int64_t)yo * crop + xo;
      r.code[j] = *reinterpret_cast<const uint2*>(idx + mo * C);
      r.g[j] = *reinterpret_cast<const uint4*>(dout + mo * do_cs);
    } else {
      r.code[j] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);   // never equals a code 0..8
      r.g[j] = make_uint4(0u, 0u, 0u, 0u);
    }
  }
}
__device__ __forceinline__ void pool_bwd_acc(const PoolBwdRow& r, int dy, float (&acc)[8]) {
  // window row yo = y - dy; window column xo = x - dx is r.*[1 - dx]; the input pixel is the window's element (dy, dx)
#pragma unroll
  for (int dx = -1; dx <= 1; ++dx) {
    const int j = 1 - dx;
    const unsigned code4 = (unsigned)((dy + 1) * 3 + (dx + 1)) * 0x01010101u;
    const unsigned ex = __vcmpeq4(r.code[j].x, code4), ey = __vcmpeq4(r.code[j].y, code4);
    const unsigned gw[4] = {r.g[j].x & __byte_perm(ex, 0, 0x1100), r.g[j].y & __byte_perm(ex, 0, 0x3322),
                            r.g[j].z & __byte_perm(ey, 0, 0x1100), r.g[j].w & __byte_perm(ey, 0, 0x3322)};
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      acc[2 * w] += __uint_as_float(gw[w] << 16);
      acc[2 * w + 1] += __uint_as_float(gw[w] & 0xFFFF0000u);
    }
  }
}

__global__ void __launch_bounds__(256, DRS_POOL_MINBLK)
maxpool3_bwd_bf16_kernel(const __nv_bfloat16* __restrict__ dout, int do_cs, int do_co, const uint8_t* __restrict__ idx,
                         __nv_bfloat16* __restrict__ din, int di_cs, int di_co, int C, int B, int crop, int seg, int nseg) {
  const int cv = C >> 3;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)B * nseg * crop * cv) return;
  const int cg = (int)(gid % cv);
  int64_t t = gid / cv;
  const int x = (int)(t % crop);
  t /= crop;
  const int sg = (int)(t % nseg);
  const int b = (int)(t / nseg);
  const int y0 = sg * seg, y1 = min(crop, y0 + seg);
  const int64_t img0 = (int64_t)b * crop * crop;
  const __nv_bfloat16* dp = dout + do_co + cg * 8;
  const uint8_t* ip = idx + cg * 8;
  PoolBwdRow ra, rb, rc;                 // window rows y-1, y, y+1
  pool_bwd_load(dp, do_cs, ip, C, img0, x, crop, y0 - 1, ra);
  pool_bwd_load(dp, do_cs, ip, C, img0, x, crop, y0, rb);
  for (int y = y0; y < y1; ++y) {
    pool_bwd_load(dp, do_cs, ip, C, img0, x, crop, y + 1, rc);
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.0f;
    // same summation order as the gather formulation: dy = -1 (window row y+1), 0, +1 (window row y-1); dx = -1, 0, +1
    pool_bwd_acc(rc, -1, acc);
    pool_bwd_acc(rb, 0, acc);
    pool_bwd_acc(ra, 1, acc);
    uint4 o;
    unsigned* ow = reinterpret_cast<unsigned*>(&o);
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const __nv_bfloat162 p = __floats2bfloat162_rn(acc[2 * w], acc[2 * w + 1]);
      ow[w] = *reinterpret_cast<const unsigned*>(&p);
    }
    *reinterpret_cast<uint4*>(din + (img0 + (int64_t)y * crop + x) * di_cs + di_co + cg * 8) = o;
    ra = rb;
    rb = rc;
  }
}

#include "pool_train.cuh"

static bool pool_lean_enabled() {
  static const bool on = !getenv("DRS_POOL_OLD");
  return on;
}

// idx != nullptr: training (winner codes, normalise + activation of the winner with bn_mean / bn_inv_std / act);
// otherwise inference (plain max).
template <typename T>
static void launch_maxpool3_fwd(Handle* h, const T* in, int in_cs, int in_co, T* out, int out_cs, int out_co, uint8_t* idx, int C,
                                int B, int crop, const float* bn_mean = nullptr, const float* bn_inv_std = nullptr, int act = 0) {
  const int64_t base = (int64_t)B * crop * (C / 8);
  int nseg = (int)std::min<int64_t>(std::max<int64_t>(1, ceil_div((int64_t)h->sm_count * 2048, base)), std::max(1, crop / 4));
  const int seg = (int)ceil_div(crop, nseg);
  nseg = (int)ceil_div(crop, seg);
  const int64_t total = base * nseg;
  const unsigned nb = (unsigned)ceil_div(total, 256);
  if (idx && ElemTag<T>::v == ET_BF16 && pool_lean_enabled()) {
    auto k = act == ACT_RELU ? pool_lean::fwd_kernel<ACT_RELU> : act == ACT_LRELU ? pool_lean::fwd_kernel<ACT_LRELU> : pool_lean::fwd_kernel<ACT_NONE>;
    launch_pdl(h, k, dim3(nb), dim3(256), 0, (const __nv_bfloat16*)in, in_cs, in_co, (__nv_bfloat16*)out, out_cs, out_co, idx, C, B, crop, seg, nseg, bn_mean, bn_inv_std);
  } else if (idx && ElemTag<T>::v == ET_BF16)
    maxpool3_fwd_train_bf16_pipelined_kernel<<<nb, 256, 0, h->stream>>>((const __nv_bfloat16*)in, in_cs, in_co, (__nv_bfloat16*)out, out_cs, out_co, idx, C, B, crop, seg, nseg, bn_mean, bn_inv_std, act);
  else if (idx) maxpool3_fwd_kernel<T><<<nb, 256, 0, h->stream>>>(in, in_cs, in_co, out, out_cs, out_co, idx, C, B, crop, seg, nseg, bn_mean, bn_inv_std, act);
  else {
    const int64_t base2 = (int64_t)B * ((crop + 1) / 2) * (C / 8);
    int nseg2 = (int)std::min<int64_t>(std::max<int64_t>(1, ceil_div((int64_t)h->sm_count * 2048, base2)), std::max(1, crop / 4));
    const int seg2 = (int)ceil_div(crop, nseg2);
    nseg2 = (int)ceil_div(crop, seg2);
    maxpool3_fwd_packed2_kernel<T><<<(unsigned)ceil_div(base2 * nseg2, 256), 256, 0, h->stream>>>(in, in_cs, in_co, out, out_cs, out_co, C, B, crop, seg2, nseg2);
  }
  LAUNCH_CHECK(h);
}

// dIn[q] = sum over the (<=9) windows o that contain q and whose recorded maximum is q, of dOut[o]
template <typename T>
__global__ void maxpool3_bwd_kernel(const T* __restrict__ dout, int do_cs, int do_co, const uint8_t* __restrict__ idx,
                                    T* __restrict__ din, int di_cs, int di_co, int C, int64_t M, int crop) {
  const int cv = C >> 3;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= M * cv) return;
  const int64_t m = gid / cv;
  const int c0 = (int)(gid - m * cv) << 3;
  const int cc = crop * crop;
  const int r = (int)(m % cc);
  const int y = r / crop, x = r - y * crop;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.0f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int yo = y - dy;            // output window centre such that q = o + (dy, dx)
    if (yo < 0 || yo >= crop) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int xo = x - dx;
      if (xo < 0 || xo >= crop) continue;
      const int64_t mo = m - dy * crop - dx;
      const uint2 pk = *reinterpret_cast<const uint2*>(idx + mo * C + c0);
      const Vec8<T> g = *reinterpret_cast<const Vec8<T>*>(dout + mo * do_cs + do_co + c0);
      const int code = (dy + 1) * 3 + (dx + 1);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int id = ((e < 4 ? pk.x : pk.y) >> ((e & 3) * 8)) & 0xff;
        if (id == code) acc[e] += to_f32(g.v[e]);
      }
    }
  }
  Vec8<T> o;
#pragma unroll
  for (int e = 0; e < 8; ++e) o.v[e] = from_f32<T>(acc[e]);
  *reinterpret_cast<Vec8<T>*>(din + m * di_cs + di_co + c0) = o;
}

template <typename T>
static void launch_maxpool3_bwd(Handle* h, const T* dout, int do_cs, int do_co, const uint8_t* idx, T* din, int di_cs, int di_co,
                                int C, int B, int crop) {
  const int64_t M = (int64_t)B * crop * crop;
  if (ElemTag<T>::v == ET_BF16) {
    const int64_t base = (int64_t)B * crop * (C / 8);
    int nseg = (int)std::min<int64_t>(std::max<int64_t>(1, ceil_div((int64_t)h->sm_count * 2048, base)), std::max(1, crop / 4));
    const int seg = (int)ceil_div(crop, nseg);
    nseg = (int)ceil_div(crop, seg);
    const unsigned nb = (unsigned)ceil_div(base * nseg, 256);
    if (pool_lean_enabled())
      launch_pdl(h, pool_lean::bwd_kernel, dim3(nb), dim3(256), 0, (const __nv_bfloat16*)dout, do_cs, do_co, idx, (__nv_bfloat16*)din,
                 di_cs, di_co, C, B, crop, seg, nseg);
    else
      maxpool3_bwd_bf16_kernel<<<nb, 256, 0, h->stream>>>((const __nv_bfloat16*)dout, do_cs, do_co, idx, (__nv_bfloat16*)din, di_cs,
                                                          di_co, C, B, crop, seg, nseg);
  } else {
    maxpool3_bwd_kernel<T><<<(unsigned)ceil_div(M * (C / 8), 256), 256, 0, h->stream>>>(dout, do_cs, do_co, idx, din, di_cs, di_co, C, M, crop);
  }
  LAUNCH_CHECK(h);
}

// pool backward + batch-norm backward of the layer below in one pass (bf16 training, pool_train.cuh)
static void launch_maxpool3_bwd_apply(Handle* h, const __nv_bfloat16* dout, int do_cs, int do_co, const uint8_t* idx, __nv_bfloat16* dz,
                                      int dz_cs, int dz_co, int C, int B, int crop, const __nv_bfloat16* z, const float* mean,
                                      const float* inv_std, const float* sums, double inv_count, int act) {
  const int64_t base = (int64_t)B * crop * (C / 8);
  int nseg = (int)std::min<int64_t>(std::max<int64_t>(1, ceil_div((int64_t)h->sm_count * 2048, base)), std::max(1, crop / 4));
  const int seg = (int)ceil_div(crop, nseg);
  nseg = (int)ceil_div(crop, seg);
  const unsigned nb = (unsigned)ceil_div(base * nseg, 256);
  auto k = act == ACT_RELU ? pool_lean::bwd_apply_kernel<ACT_RELU>
           : act == ACT_LRELU ? pool_lean::bwd_apply_kernel<ACT_LRELU> : pool_lean::bwd_apply_kernel<ACT_NONE>;
  launch_pdl(h, k, dim3(nb), dim3(256), (size_t)4 * C * sizeof(float), dout, do_cs, do_co, idx, dz, dz_cs, dz_co, C, B, crop, seg, nseg, z, mean,
             inv_std, sums, inv_count);
  LAUNCH_CHECK(h);
}

// ------------------------------------------------------------------------------------------------
// _batch_norm (isprs:655-663): tf.contrib.layers.batch_norm(center=False, scale=False)
// ------------------------------------------------------------------------------------------------
constexpr int BN_THREADS = 256;


// part[blk][0][c] = sum_m a, part[blk][1][c] = sum_m a*b over the block's contiguous slab of rows.
//   MODE 0 (forward statistics):  a = z,            b = z
//   MODE 1 (backward sums):       a = g = dA*act'(xh), b = xh        (xh = (z-mean)*inv_std)
//   MODE 2 (backward sums through a max-pool, from the pooled side): see bn_partial_row
// Thread = (channel group of 8, row lane): 16-byte loads, per-thread fp32 partials, then a fixed-order reduction over the
// row lanes in shared memory.  The row -> (block, lane) assignment is static, so the result is run-to-run identical.
template <typename TZ, typename TG, int MODE>
__device__ __forceinline__ void bn_partial_row(const Vec8<TZ>& zv, const Vec8<TG>& gv, const float (&mu)[8], const float (&is)[8],
                                               int act, float (&s0)[8], float (&s1)[8]) {
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    if (MODE == 0) {
      const float f = to_f32(zv.v[e]);
      s0[e] += f;
      s1[e] = fmaf(f, f, s1[e]);
    } else if (MODE == 1) {
      const float xh = (to_f32(zv.v[e]) - mu[e]) * is[e];
      float g = to_f32(gv.v[e]);
      if (act == ACT_RELU) g = xh > 0.0f ? g : 0.0f;
      else if (act == ACT_LRELU) g = xh > 0.0f ? g : 0.1f * g;
      s0[e] += g;
      s1[e] = fmaf(g, xh, s1[e]);
    } else {
      // MODE 2, pooling nets: zv is the pooled ACTIVATION act(xh of the window's winner), gv the window's gradient.  The
      // winner's normalised value is recovered through the inverse activation (exact for ReLU where it matters -- the
      // negative side has no gradient; within the activation's bf16 rounding for LeakyReLU).
      const float av = to_f32(zv.v[e]);
      float g = to_f32(gv.v[e]);
      float xh = av;
      if (act == ACT_RELU) g = av > 0.0f ? g : 0.0f;
      else if (act == ACT_LRELU) { xh = av > 0.0f ? av : av * 10.0f; g = av > 0.0f ? g : 0.1f * g; }
      s0[e] += g;
      s1[e] = fmaf(g, xh, s1[e]);
    }
  }
}

constexpr int BN_UNROLL = 4;     // rows in flight per thread (8 x 16-byte loads in the backward mode)
template <typename TZ, typename TG, int MODE>
__global__ void __launch_bounds__(BN_THREADS, DRS_BN_MINBLK)
bn_partial_kernel(const TZ* __restrict__ z, int z_cs, int z_co, const TG* __restrict__ dA, int g_cs, int g_co,
                  const float* __restrict__ mean, const float* __restrict__ inv_std, int act, float* __restrict__ part, int C,
                  int64_t M, int rows_per_block, BnFinish fin) {
  // [round slot][thread]: the 16 per-thread sums go through shared memory four at a time.  The whole set at once was 16.4 KB
  // of static shared memory, and next to a resident wgrad_tc CTA (up to 216 KB, on the side stream) that does not fit: the
  // statistics pass then waited for the filter gradient instead of running beside it (CUPTI timeline: 28 us holes).
  __shared__ float s_red[4][BN_THREADS + 1];
  pdl_sync();
  const int cv = C >> 3;
  const int lanes_r = BN_THREADS / cv;
  const int cg = threadIdx.x % cv, rl = threadIdx.x / cv;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = min(M, r0 + rows_per_block);
  float s0[8], s1[8], mu[8], is[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { s0[e] = 0.0f; s1[e] = 0.0f; mu[e] = 0.0f; is[e] = 1.0f; }
  if (rl < lanes_r) {
    if (MODE == 1) {
#pragma unroll
      for (int e = 0; e < 8; ++e) { mu[e] = mean[cg * 8 + e]; is[e] = inv_std[cg * 8 + e]; }
    }
    const TZ* zp = z + z_co + cg * 8;
    const TG* gp = MODE >= 1 ? dA + g_co + cg * 8 : nullptr;
    int64_t m = r0 + rl;
    // BN_UNROLL rows per iteration: every load is issued before the first one is consumed
    for (; m + (int64_t)(BN_UNROLL - 1) * lanes_r < r1; m += (int64_t)BN_UNROLL * lanes_r) {
      Vec8<TZ> zv[BN_UNROLL];
      Vec8<TG> gv[BN_UNROLL];
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        zv[u] = *reinterpret_cast<const Vec8<TZ>*>(zp + (m + (int64_t)u * lanes_r) * z_cs);
        if (MODE >= 1) gv[u] = *reinterpret_cast<const Vec8<TG>*>(gp + (m + (int64_t)u * lanes_r) * g_cs);
      }
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) bn_partial_row<TZ, TG, MODE>(zv[u], gv[u], mu, is, act, s0, s1);
    }
    for (; m < r1; m += lanes_r) {
      const Vec8<TZ> zv = *reinterpret_cast<const Vec8<TZ>*>(zp + m * z_cs);
      Vec8<TG> gv;
      if (MODE >= 1) gv = *reinterpret_cast<const Vec8<TG>*>(gp + m * g_cs);
      bn_partial_row<TZ, TG, MODE>(zv, gv, mu, is, act, s0, s1);
    }
  }
  // Block partial (fixed order) -> 64-bit fixed point -> integer atomicAdd: integer addition is associative, so the grid-wide
  // sum does not depend on the order in which blocks arrive (deterministic without a serial reduction pass).
#pragma unroll
  for (int rd = 0; rd < 4; ++rd) {                       // round rd: elements 2rd, 2rd+1 of both sums
    if (rd) __syncthreads();
    s_red[0][threadIdx.x] = s0[2 * rd];
    s_red[1][threadIdx.x] = s0[2 * rd + 1];
    s_red[2][threadIdx.x] = s1[2 * rd];
    s_red[3][threadIdx.x] = s1[2 * rd + 1];
    __syncthreads();
    for (int i = threadIdx.x; i < 4 * cv; i += BN_THREADS) {
      const int j = i / cv, g = i - j * cv;              // consecutive threads -> consecutive channel groups (no conflicts)
      const int which = j >> 1, e = 2 * rd + (j & 1);
      float a = 0.0f;
      for (int r = 0; r < lanes_r; ++r) a += s_red[j][r * cv + g];
      const long long q = __double2ll_rn((double)a * fin.fx_scale);
      atomicAdd(bn_acc_mine(fin) + which * C + g * 8 + e, static_cast<unsigned long long>(q));
    }
  }
  // ---- the last block to finish converts the sums, finalizes and clears the accumulators for the next launch
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(fin.counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const double inv_scale = 1.0 / fin.fx_scale;
  for (int i = threadIdx.x; i < C; i += BN_THREADS) {
    const double a = (double)bn_acc_take(fin, i) * inv_scale;
    const double b = (double)bn_acc_take(fin, C + i) * inv_scale;
    fin.sums[i] = (float)a;
    fin.sums[C + i] = (float)b;
    if (fin.mean) {
      const double mu = (double)(float)a / fin.count;
      double var = (double)(float)b / fin.count - mu * mu;
      if (var < 0.0) var = 0.0;
      fin.mean[i] = (float)mu;
      fin.inv_std[i] = (float)(1.0 / sqrt(var + (double)fin.eps));
      const double var_ema = fin.unbiased_ema ? var * (fin.count / fmax(fin.count - 1.0, 1.0)) : var;
      fin.mov_mean[i] = fin.decay * fin.mov_mean[i] + (1.0f - fin.decay) * (float)mu;
      fin.mov_var[i] = fin.decay * fin.mov_var[i] + (1.0f - fin.decay) * (float)var_ema;
    }
  }
  if (threadIdx.x == 0) *fin.counter = 0u;                   // ready for the next launch on this stream
}

// mean / inv_std from (possibly all-reduced) sums; moving-average update (decay 0.999, isprs:658 defaults)
__global__ void bn_finalize_kernel(const float* __restrict__ sums, float* __restrict__ mean, float* __restrict__ inv_std,
                                   float* __restrict__ mov_mean, float* __restrict__ mov_var, int C, double count,
                                   float eps, float decay, int unbiased_ema) {
  pdl_sync();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mu = (double)sums[c] / count;
  double var = (double)sums[C + c] / count - mu * mu;
  if (var < 0.0) var = 0.0;
  mean[c] = (float)mu;
  inv_std[c] = (float)(1.0 / sqrt(var + (double)eps));
  const double var_ema = unbiased_ema ? var * (count / fmax(count - 1.0, 1.0)) : var;
  mov_mean[c] = decay * mov_mean[c] + (1.0f - decay) * (float)mu;
  mov_var[c] = decay * mov_var[c] + (1.0f - decay) * (float)var_ema;
}

// Row-slab layout shared by the two element-wise BN kernels: thread = (channel group of 8, row lane); a block walks
// its rows with the per-channel constants (mean, inv_std, reduced sums) held in registers.
constexpr int BNE_THREADS = 256;
static inline int bne_grid(int64_t M, int sm_count) { return (int)std::min<int64_t>(ceil_div(M, 64), (int64_t)sm_count * 8); }

// out = act((z - mean) * inv_std)     (training-mode normalise + activation)
template <typename T>
__global__ void __launch_bounds__(BNE_THREADS)
bn_apply_kernel(const T* __restrict__ z, int z_cs, int z_co, const float* __restrict__ mean, const float* __restrict__ inv_std,
                int act, T* __restrict__ out, int o_cs, int o_co, int C, int64_t M) {
  pdl_sync();
  const int cv = C >> 3;
  const int lanes_r = BNE_THREADS / cv;
  const int cg = threadIdx.x % cv, rl = threadIdx.x / cv;
  if (rl >= lanes_r) return;
  float mu[8], is[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { mu[e] = mean[cg * 8 + e]; is[e] = inv_std[cg * 8 + e]; }
  for (int64_t m = (int64_t)blockIdx.x * lanes_r + rl; m < M; m += (int64_t)gridDim.x * lanes_r) {
    const Vec8<T> v = *reinterpret_cast<const Vec8<T>*>(z + m * z_cs + z_co + cg * 8);
    Vec8<T> o;
#pragma unroll
    for (int e = 0; e < 8; ++e) o.v[e] = from_f32<T>(apply_act((to_f32(v.v[e]) - mu[e]) * is[e], act));
    *reinterpret_cast<Vec8<T>*>(out + m * o_cs + o_co + cg * 8) = o;
  }
}

// dZ = inv_std * (g - s0/M - xh * s1/M),  g = dA * act'(xh)      (no gamma/beta: SURVEY F5)
template <typename TZ, typename TG>
__global__ void __launch_bounds__(BNE_THREADS, DRS_BNE_MINBLK)
bn_bwd_apply_kernel(const TZ* __restrict__ z, int z_cs, int z_co, const TG* __restrict__ dA, int g_cs, int g_co,
                    const float* __restrict__ mean, const float* __restrict__ inv_std, const float* __restrict__ sums,
                    double inv_count, int act, TG* __restrict__ dZ, int d_cs, int d_co, int C, int64_t M) {
  pdl_sync();
  const int cv = C >> 3;
  const int lanes_r = BNE_THREADS / cv;
  const int cg = threadIdx.x % cv, rl = threadIdx.x / cv;
  if (rl >= lanes_r) return;
  float mu[8], is[8], m0[8], m1[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = cg * 8 + e;
    mu[e] = mean[c];
    is[e] = inv_std[c];
    m0[e] = (float)((double)sums[c] * inv_count);
    m1[e] = (float)((double)sums[C + c] * inv_count);
  }
  // two rows per iteration (four 16-byte loads in flight per thread)
  const int64_t step = (int64_t)gridDim.x * lanes_r;
  for (int64_t m = (int64_t)blockIdx.x * lanes_r + rl; m < M; m += 2 * step) {
    const int64_t m2 = m + step;
    const bool two = m2 < M;
    const Vec8<TZ> zv = *reinterpret_cast<const Vec8<TZ>*>(z + m * z_cs + z_co + cg * 8);
    const Vec8<TG> gv = *reinterpret_cast<const Vec8<TG>*>(dA + m * g_cs + g_co + cg * 8);
    Vec8<TZ> zw = zv;
    Vec8<TG> gw = gv;
    if (two) {
      zw = *reinterpret_cast<const Vec8<TZ>*>(z + m2 * z_cs + z_co + cg * 8);
      gw = *reinterpret_cast<const Vec8<TG>*>(dA + m2 * g_cs + g_co + cg * 8);
    }
    Vec8<TG> o, o2;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float xh = (to_f32(zv.v[e]) - mu[e]) * is[e];
      float g = to_f32(gv.v[e]);
      if (act == ACT_RELU) g = xh > 0.0f ? g : 0.0f;
      else if (act == ACT_LRELU) g = xh > 0.0f ? g : 0.1f * g;
      o.v[e] = from_f32<TG>(is[e] * (g - m0[e] - xh * m1[e]));
      const float xh2 = (to_f32(zw.v[e]) - mu[e]) * is[e];
      float g2 = to_f32(gw.v[e]);
      if (act == ACT_RELU) g2 = xh2 > 0.0f ? g2 : 0.0f;
      else if (act == ACT_LRELU) g2 = xh2 > 0.0f ? g2 : 0.1f * g2;
      o2.v[e] = from_f32<TG>(is[e] * (g2 - m0[e] - xh2 * m1[e]));
    }
    *reinterpret_cast<Vec8<TG>*>(dZ + m * d_cs + d_co + cg * 8) = o;
    if (two) *reinterpret_cast<Vec8<TG>*>(dZ + m2 * d_cs + d_co + cg * 8) = o2;
  }
}

// dst[:, coff:coff+C] += src (dense-net gradient accumulation into the concat gradient buffer)
template <typename T>
__global__ void add_slice_kernel(T* __restrict__ dst, int d_cs, int d_co, const T* __restrict__ src, int s_cs, int s_co,
                                 int C, int64_t M) {
  pdl_sync();
  const int cv = C >> 3;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= M * cv) return;
  const int64_t m = gid / cv;
  const int c0 = (int)(gid - m * cv) << 3;
  Vec8<T> a = *reinterpret_cast<const Vec8<T>*>(dst + m * d_cs + d_co + c0);
  const Vec8<T> b = *reinterpret_cast<const Vec8<T>*>(src + m * s_cs + s_co + c0);
#pragma unroll
  for (int e = 0; e < 8; ++e) a.v[e] = from_f32<T>(to_f32(a.v[e]) + to_f32(b.v[e]));
  *reinterpret_cast<Vec8<T>*>(dst + m * d_cs + d_co + c0) = a;
}

// ------------------------------------------------------------------------------------------------
// conv_classifier (1x1, Ci -> K, bias, no BN/act)  isprs:779-786  + tf.argmax(logits, 3) isprs:1690
// One warp per pixel: lanes stride the channels (coalesced), shuffle-reduce K partial sums.
// ------------------------------------------------------------------------------------------------
// Tile kernel: a block stages [CLS_TILE pixels x Ci] in shared memory with coalesced 16-byte loads (128B-swizzled
// rows, so that the row-per-thread reads below are conflict-free), then thread r owns pixel r: Ci*K FMAs against
// weights broadcast from shared memory, first-maximum argmax, one K-float row of logits out.  No shuffles.
template <typename T, int CLS_TILE>
__global__ void __launch_bounds__(CLS_TILE)
classifier_fwd_kernel(const T* __restrict__ x, int x_cs, int x_co, int Ci, const float* __restrict__ w,
                      const float* __restrict__ b, int K, float* __restrict__ logits, uint8_t* __restrict__ pred, int64_t M) {
  pdl_sync();
  extern __shared__ __align__(16) uint8_t cls_smem[];
  float* s_w = reinterpret_cast<float*>(cls_smem);                 // [Ci][8] (K padded to 8)
  uint8_t* s_x = cls_smem + (size_t)Ci * 8 * sizeof(float);        // [CLS_TILE][Ci] elements, 16-byte chunks swizzled
  const int tid = threadIdx.x;
  for (int i = tid; i < Ci * 8; i += CLS_TILE) {
    const int c = i >> 3, k = i & 7;
    s_w[i] = k < K ? w[c * K + k] : 0.0f;
  }
  constexpr int EPC = 16 / sizeof(T);      // elements per 16-byte chunk
  const int chunks = Ci / EPC;
  const size_t row_bytes = (size_t)Ci * sizeof(T);
  float bias[MAX_CLASSES];
#pragma unroll
  for (int k = 0; k < MAX_CLASSES; ++k) bias[k] = k < K ? b[k] : 0.0f;
  for (int64_t m0 = (int64_t)blockIdx.x * CLS_TILE; m0 < M; m0 += (int64_t)gridDim.x * CLS_TILE) {
    __syncthreads();                                            // previous tile fully consumed (and s_w visible)
    const int rows = (int)min((int64_t)CLS_TILE, M - m0);
    // asynchronous 16-byte global->shared copies: every chunk of the tile is in flight at once (a register-staged
    // loop would keep one load per thread outstanding and leave the kernel latency-bound)
    for (int i = tid; i < rows * chunks; i += CLS_TILE) {
      const int r = i / chunks, ch = i - r * chunks;
      const int sw = (ch & ~7) | ((ch & 7) ^ (r & 7));
      const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(s_x + r * row_bytes + (size_t)sw * 16));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(x + (m0 + r) * x_cs + x_co + ch * EPC) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    if (tid < rows) {
      float acc[MAX_CLASSES];
#pragma unroll
      for (int k = 0; k < MAX_CLASSES; ++k) acc[k] = 0.0f;
      const uint8_t* rowp = s_x + tid * row_bytes;
      for (int ch = 0; ch < chunks; ++ch) {
        const int sw = (ch & ~7) | ((ch & 7) ^ (tid & 7));
        const uint4 raw = *reinterpret_cast<const uint4*>(rowp + (size_t)sw * 16);
        const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
        for (int j = 0; j < EPC; ++j) {
          const float f = to_f32(e[j]);
          const float4 w0 = *reinterpret_cast<const float4*>(s_w + (ch * EPC + j) * 8);
          const float4 w1 = *reinterpret_cast<const float4*>(s_w + (ch * EPC + j) * 8 + 4);
          acc[0] = fmaf(f, w0.x, acc[0]); acc[1] = fmaf(f, w0.y, acc[1]); acc[2] = fmaf(f, w0.z, acc[2]); acc[3] = fmaf(f, w0.w, acc[3]);
          acc[4] = fmaf(f, w1.x, acc[4]); acc[5] = fmaf(f, w1.y, acc[5]); acc[6] = fmaf(f, w1.z, acc[6]); acc[7] = fmaf(f, w1.w, acc[7]);
        }
      }
      const int64_t m = m0 + tid;
      float best = -INFINITY;
      int bi = 0;
#pragma unroll
      for (int k = 0; k < MAX_CLASSES; ++k) {
        if (k < K) {
          const float v = acc[k] + bias[k];
          if (logits) logits[m * K + k] = v;
          if (v > best) { best = v; bi = k; }      // first maximum (Appendix B.7)
        }
      }
      if (pred) pred[m] = (uint8_t)bi;
    }
  }
}
template <typename T, int TILE>
static void launch_classifier_fwd_t(Handle* h, const T* x, int x_cs, int x_co, int Ci, const float* w, const float* b, int K,
                                    float* logits, uint8_t* pred, int64_t M, size_t smem) {
  auto kern = classifier_fwd_kernel<T, TILE>;
  static bool attr_set = false;
  if (!attr_set) {
    CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (size_t)(220 * 1024) / (smem + 1024)));
  const int blocks = (int)std::min<int64_t>(ceil_div(M, TILE), (int64_t)h->sm_count * per_sm);
  kern<<<blocks, TILE, smem, h->stream>>>(x, x_cs, x_co, Ci, w, b, K, logits, pred, M);
  LAUNCH_CHECK(h);
}
template <typename T>
static void launch_classifier_fwd(Handle* h, const T* x, int x_cs, int x_co, int Ci, const float* w, const float* b, int K,
                                  float* logits, uint8_t* pred, int64_t M) {
  DRS_CHECK(Ci % 64 == 0, "classifier: Ci=%d must be a multiple of 64", Ci);
  auto smem_of = [&](int tile) { return (size_t)Ci * 8 * 4 + (size_t)tile * Ci * sizeof(T); };
  if (smem_of(128) <= 112 * 1024) launch_classifier_fwd_t<T, 128>(h, x, x_cs, x_co, Ci, w, b, K, logits, pred, M, smem_of(128));
  else if (smem_of(64) <= 112 * 1024 || smem_of(128) > 220 * 1024) launch_classifier_fwd_t<T, 64>(h, x, x_cs, x_co, Ci, w, b, K, logits, pred, M, smem_of(64));
  else launch_classifier_fwd_t<T, 128>(h, x, x_cs, x_co, Ci, w, b, K, logits, pred, M, smem_of(128));
}

// Inference: the LAST 3x3 max-pool and the classifier (1x1 convolution Ci -> K, isprs:779-786) in one pass.  The pooled
// activations of the last layer feed nothing but the classifier, so they are neither written nor read back: the kernel
// reads the last convolution's output once (M*Ci*2 B) and writes M*K logits.  A thread owns (image, row segment, two
// columns, 8 channels) and walks down its rows, so the CV = Ci/8 lanes that hold one pixel are neighbours in a warp: each
// lane multiplies its 8 pooled channels (exactly the values the unfused kernel would have stored) with its 8 x K weights
// held in registers, and the K partial sums are combined by a transposing butterfly (4 + 2 + 1 shuffles halve the number of classes a lane carries, the remaining steps add one
// value), after which the lanes with (lane % (CV/8)) == 0 hold one class each.  The order of the additions is the same for
// every pixel wherever it sits, so patch-wise and scene-wise inference and every stripe agree bit for bit.
// K partial class sums per lane -> one class per lane (see the kernel's header comment); every lane of the CV-lane group calls it
template <int CV>
__device__ __forceinline__ float cls_butterfly(const float (&acc)[8], unsigned gmask, bool up0, bool up1, bool up2) {
  float a4[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float send = up0 ? acc[i] : acc[i + 4];
    const float keep = up0 ? acc[i + 4] : acc[i];
    a4[i] = keep + __shfl_xor_sync(gmask, send, CV / 2);
  }
  float a2[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float send = up1 ? a4[i] : a4[i + 2];
    const float keep = up1 ? a4[i + 2] : a4[i];
    a2[i] = keep + __shfl_xor_sync(gmask, send, CV / 4);
  }
  const float send = up2 ? a2[0] : a2[1];
  const float keep = up2 ? a2[1] : a2[0];
  float v = keep + __shfl_xor_sync(gmask, send, CV / 8);
#pragma unroll
  for (int off = CV / 16; off >= 1; off >>= 1) v += __shfl_xor_sync(gmask, v, off);
  return v;
}
// first maximum over the classes (Appendix B.7): the smaller index wins a tie; result valid in every lane of the group
template <int CV>
__device__ __forceinline__ int cls_argmax(float v, int cls, int K, unsigned gmask) {
  float bv = cls < K ? v : -INFINITY;
  int bi = cls;
#pragma unroll
  for (int off = CV / 2; off >= CV / 8; off >>= 1) {
    const float ov = __shfl_xor_sync(gmask, bv, off);
    const int oi = __shfl_xor_sync(gmask, bi, off);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  return bi;
}

// Two columns per thread like maxpool3_fwd_packed2_kernel (the reads are latency-bound: what counts is how many unique bytes
// a thread has on their way), the 8 x K weights in registers serve both pixels.
template <typename T, int CV, int KC>
__global__ void __launch_bounds__(256)
maxpool3_classifier_kernel(const T* __restrict__ in, int in_cs, int in_co, int B, int crop, int seg, int nseg,
                           const float* __restrict__ w, const float* __restrict__ bias, int K, float* __restrict__ logits,
                           uint8_t* __restrict__ pred) {
  static_assert(CV == 8 || CV == 16 || CV == 32, "Ci must be 64, 128 or 256");
  static_assert(KC <= 8, "the butterfly carries 8 classes");
  const int xp_n = (crop + 1) >> 1;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)B * nseg * xp_n * CV) return;              // whole groups of CV lanes leave together
  const int lane = threadIdx.x & 31;
  const unsigned gmask = CV == 32 ? 0xffffffffu : (((1u << CV) - 1u) << (lane & ~(CV - 1)));
  const int g = lane & (CV - 1);
  const int cg = (int)(gid % CV);
  int64_t t = gid / CV;
  const int x0 = (int)(t % xp_n) * 2;
  t /= xp_n;
  const int sg = (int)(t % nseg);
  const int b = (int)(t / nseg);
  const int y0 = sg * seg, y1 = min(crop, y0 + seg);
  const bool has1 = x0 + 1 < crop;
  float wr[8][KC];
#pragma unroll
  for (int e = 0; e < 8; ++e)
#pragma unroll
    for (int k = 0; k < KC; ++k) wr[e][k] = k < K ? w[(cg * 8 + e) * K + k] : 0.0f;
  const bool up0 = (g & (CV / 2)) != 0, up1 = (g & (CV / 4)) != 0, up2 = (g & (CV / 8)) != 0;
  const int cls = (up0 ? 4 : 0) + (up1 ? 2 : 0) + (up2 ? 1 : 0);
  const bool writer = (g & (CV / 8 - 1)) == 0 && cls < K;
  const float my_bias = cls < K ? bias[cls] : 0.0f;
  const int o_l = x0 > 0 ? -in_cs : 0;
  const int o_1 = has1 ? in_cs : 0;
  const int o_r = x0 + 2 < crop ? 2 * in_cs : o_1;
  const int64_t rs = (int64_t)crop * in_cs;
  const int64_t pix0 = (int64_t)b * crop * crop + (int64_t)y0 * crop + x0;
  const T* q = in + in_co + cg * 8 + pix0 * in_cs;               // centre of the next row to load
  float* lp = logits + pix0 * K + cls;
  uint8_t* pp = pred ? pred + pix0 : nullptr;
  Vec8<T> nl, n0, n1, nr;                      // raw loads of the next row
  Vec8<T> a0, a1, b0, b1, c0, c1;              // horizontal maxima of rows y-1, y, y+1 for the two columns
  auto load = [&](const T* c) {
    n0 = *reinterpret_cast<const Vec8<T>*>(c);
    nl = *reinterpret_cast<const Vec8<T>*>(c + o_l);
    n1 = *reinterpret_cast<const Vec8<T>*>(c + o_1);
    nr = *reinterpret_cast<const Vec8<T>*>(c + o_r);
  };
  auto reduce = [&](Vec8<T>& h0, Vec8<T>& h1) {
    Vec8<T> m = n0;
    vmax8(m, n1);
    h0 = m; vmax8(h0, nl);
    h1 = m; vmax8(h1, nr);
  };
  bool va = y0 > 0;
  if (va) { load(q - rs); reduce(a0, a1); }
  load(q);
  reduce(b0, b1);
  q += rs;
  bool vn = y0 + 1 < crop;
  if (vn) load(q);
  for (int y = y0; y < y1; ++y) {
    const bool vc = vn;
    if (vc) reduce(c0, c1);
    q += rs;
    vn = y + 2 < crop && y + 1 < y1;
    if (vn) load(q);
    Vec8<T> r0 = b0, r1 = b1;
    if (va) { vmax8(r0, a0); vmax8(r1, a1); }
    if (vc) { vmax8(r0, c0); vmax8(r1, c1); }
#pragma unroll
    for (int px = 0; px < 2; ++px) {
      // (the second column of an odd-width image's last pair computes on a copy of the first and stores nothing;
      //  the shuffles need every lane of the group either way)
      const Vec8<T>& o = px == 0 ? r0 : r1;
      float acc[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = 0.0f;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float f = to_f32(o.v[e]);
#pragma unroll
        for (int k = 0; k < KC; ++k) acc[k] = fmaf(f, wr[e][k], acc[k]);
      }
      const float v = cls_butterfly<CV>(acc, gmask, up0, up1, up2) + my_bias;
      const bool live = px == 0 || has1;
      if (writer && live) lp[px * K] = v;
      if (pp) {
        const int bi = cls_argmax<CV>(v, cls, K, gmask);
        if (g == 0 && live) pp[px] = (uint8_t)bi;
      }
    }
    lp += crop * K;
    if (pp) pp += crop;
    a0 = b0; a1 = b1; va = true;
    b0 = c0; b1 = c1;
  }
}

template <typename T>
static inline bool pool_classifier_fused_supported(int Ci) {
  return ElemTag<T>::v != ET_F32 && (Ci == 64 || Ci == 128 || Ci == 256);
}
template <typename T>
static void launch_maxpool3_classifier(Handle* h, const T* in, int in_cs, int in_co, int Ci, int B, int crop, const float* w,
                                       const float* b, int K, float* logits, uint8_t* pred) {
  DRS_CHECK(K <= MAX_CLASSES, "classifier: K=%d exceeds %d", K, MAX_CLASSES);
  const int64_t base = (int64_t)B * ((crop + 1) / 2) * (Ci / 8);       // a thread owns two columns
  int nseg = (int)std::min<int64_t>(std::max<int64_t>(1, ceil_div((int64_t)h->sm_count * 2048, base)), std::max(1, crop / 4));
  const int seg = (int)ceil_div(crop, nseg);
  nseg = (int)ceil_div(crop, seg);
  const unsigned nb = (unsigned)ceil_div(base * nseg, 256);
#define DRS_PCLS(CVV, KCC) maxpool3_classifier_kernel<T, CVV, KCC><<<nb, 256, 0, h->stream>>>(in, in_cs, in_co, B, crop, seg, nseg, w, b, K, logits, pred)
#define DRS_PCLS_K(CVV) do { if (K <= 2) DRS_PCLS(CVV, 2); else if (K <= 6) DRS_PCLS(CVV, 6); else DRS_PCLS(CVV, 8); } while (0)
  if (Ci == 256) DRS_PCLS_K(32);
  else if (Ci == 128) DRS_PCLS_K(16);
  else DRS_PCLS_K(8);
#undef DRS_PCLS_K
#undef DRS_PCLS
  LAUNCH_CHECK(h);
}

// dX[m][c] = sum_k dl[m][k] * W[c][k].  Weights are kept transposed in shared memory ([k][Ci]) so that a warp's
// 16-byte reads of 8 consecutive channels per lane are contiguous (no bank conflicts).
template <typename TG>
__global__ void classifier_bwd_data_kernel(const float* __restrict__ dl, const float* __restrict__ w, int K,
                                           TG* __restrict__ dx, int dx_cs, int dx_co, int Ci, int64_t M) {
  extern __shared__ __align__(16) float s_wt[];   // [K][Ci]
  for (int i = threadIdx.x; i < Ci * K; i += blockDim.x) {
    const int c = i / K, k = i - c * K;
    s_wt[k * Ci + c] = w[i];
  }
  __syncthreads();
  const int cv = Ci >> 3;
  for (int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; gid < M * cv;
       gid += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = gid / cv;
    const int c0 = (int)(gid - m * cv) << 3;
    float s[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) s[e] = 0.0f;
#pragma unroll
    for (int k = 0; k < MAX_CLASSES; ++k) {
      if (k < K) {
        const float g = dl[m * K + k];
        const float4 w0 = *reinterpret_cast<const float4*>(s_wt + k * Ci + c0);
        const float4 w1 = *reinterpret_cast<const float4*>(s_wt + k * Ci + c0 + 4);
        s[0] = fmaf(g, w0.x, s[0]); s[1] = fmaf(g, w0.y, s[1]); s[2] = fmaf(g, w0.z, s[2]); s[3] = fmaf(g, w0.w, s[3]);
        s[4] = fmaf(g, w1.x, s[4]); s[5] = fmaf(g, w1.y, s[5]); s[6] = fmaf(g, w1.z, s[6]); s[7] = fmaf(g, w1.w, s[7]);
      }
    }
    Vec8<TG> o;
#pragma unroll
    for (int e = 0; e < 8; ++e) o.v[e] = from_f32<TG>(s[e]);
    *reinterpret_cast<Vec8<TG>*>(dx + m * dx_cs + dx_co + c0) = o;
  }
}

// Same product with the thread's 8 x K weights in registers (a thread keeps its channel group for the whole kernel; Ci/8 <= 256,
// threads beyond the last whole row of channel groups retire): no shared-memory traffic in the loop -- the shared-memory version above is bound by its 12 LDS.128 per
// 16 bytes written (measured 1 TB/s).  Two pixels per iteration.
template <typename TG>
__global__ void __launch_bounds__(256)
classifier_bwd_data_reg_kernel(const float* __restrict__ dl, const float* __restrict__ w, int K, TG* __restrict__ dx, int dx_cs,
                               int dx_co, int Ci, int64_t M) {
  pdl_sync();
  const int cv = Ci >> 3;
  const int rows = 256 / cv;
  const int cg = threadIdx.x % cv, rl = threadIdx.x / cv;
  if (rl >= rows) return;                  // cv does not divide 256 (DenseDilated6: 448 channels = 56 groups): spare threads
  float wr[8][MAX_CLASSES];
#pragma unroll
  for (int e = 0; e < 8; ++e)
#pragma unroll
    for (int k = 0; k < MAX_CLASSES; ++k) wr[e][k] = k < K ? w[(cg * 8 + e) * K + k] : 0.0f;
  const int64_t step = (int64_t)gridDim.x * rows;
  for (int64_t m = (int64_t)blockIdx.x * rows + rl; m < M; m += 2 * step) {
    const int64_t m2 = m + step;
    const bool two = m2 < M;
    float g[MAX_CLASSES], g2[MAX_CLASSES];
#pragma unroll
    for (int k = 0; k < MAX_CLASSES; ++k) {
      g[k] = k < K ? dl[m * K + k] : 0.0f;
      g2[k] = (k < K && two) ? dl[m2 * K + k] : 0.0f;
    }
    Vec8<TG> o, o2;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float a = 0.0f, b = 0.0f;
#pragma unroll
      for (int k = 0; k < MAX_CLASSES; ++k) {       // k ascending: same summation order as the shared-memory version
        a = fmaf(g[k], wr[e][k], a);
        b = fmaf(g2[k], wr[e][k], b);
      }
      o.v[e] = from_f32<TG>(a);
      o2.v[e] = from_f32<TG>(b);
    }
    *reinterpret_cast<Vec8<TG>*>(dx + m * dx_cs + dx_co + cg * 8) = o;
    if (two) *reinterpret_cast<Vec8<TG>*>(dx + m2 * dx_cs + dx_co + cg * 8) = o2;
  }
}

// part[blk][c][k] = sum over the block's slab of rows of x[m][c]*dl[m][k];  part_b[blk][k] = sum dl[m][k].
// Thread = (channel group of 8, row lane) with 16-byte loads; fixed-order shared-memory reduction over the row lanes.
constexpr int CLSW_THREADS = 256;
template <typename T>
__global__ void __launch_bounds__(CLSW_THREADS)
classifier_bwd_weight_kernel(const T* __restrict__ x, int x_cs, int x_co, int Ci, const float* __restrict__ dl, int K,
                             float* __restrict__ part, float* __restrict__ part_b, int64_t M, int rows_per_block) {
  pdl_sync();
  __shared__ float s_red[CLSW_THREADS * 8];
  __shared__ float s_bias[CLSW_THREADS][MAX_CLASSES];
  const int cv = Ci >> 3;
  const int lanes_r = CLSW_THREADS / cv;
  const int cg = threadIdx.x % cv, rl = threadIdx.x / cv;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = min(M, r0 + rows_per_block);
  float acc[8][MAX_CLASSES], accb[MAX_CLASSES];
#pragma unroll
  for (int k = 0; k < MAX_CLASSES; ++k) {
    accb[k] = 0.0f;
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e][k] = 0.0f;
  }
  if (rl < lanes_r) {
    // two rows per iteration (both 16-byte loads and both dl rows in flight); rows are added in ascending order as before
    for (int64_t m = r0 + rl; m < r1; m += 2 * lanes_r) {
      const int64_t m2 = m + lanes_r;
      const bool two = m2 < r1;
      const Vec8<T> v = *reinterpret_cast<const Vec8<T>*>(x + m * x_cs + x_co + cg * 8);
      Vec8<T> v2 = v;
      if (two) v2 = *reinterpret_cast<const Vec8<T>*>(x + m2 * x_cs + x_co + cg * 8);
      float g[MAX_CLASSES], g2[MAX_CLASSES];
#pragma unroll
      for (int k = 0; k < MAX_CLASSES; ++k) {
        g[k] = k < K ? dl[m * K + k] : 0.0f;
        g2[k] = (k < K && two) ? dl[m2 * K + k] : 0.0f;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float f = to_f32(v.v[e]);
#pragma unroll
        for (int k = 0; k < MAX_CLASSES; ++k) acc[e][k] = fmaf(f, g[k], acc[e][k]);
      }
#pragma unroll
      for (int k = 0; k < MAX_CLASSES; ++k) accb[k] += g[k];
      if (two) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float f = to_f32(v2.v[e]);
#pragma unroll
          for (int k = 0; k < MAX_CLASSES; ++k) acc[e][k] = fmaf(f, g2[k], acc[e][k]);
        }
#pragma unroll
        for (int k = 0; k < MAX_CLASSES; ++k) accb[k] += g2[k];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < MAX_CLASSES; ++k) s_bias[threadIdx.x][k] = accb[k];
#pragma unroll
  for (int k = 0; k < MAX_CLASSES; ++k) {
    if (k < K) {                       // uniform across the block
      __syncthreads();
#pragma unroll
      for (int e = 0; e < 8; ++e) s_red[threadIdx.x * 8 + e] = acc[e][k];
      __syncthreads();
      for (int c = threadIdx.x; c < Ci; c += CLSW_THREADS) {
        const int g = c >> 3, e = c & 7;
        float a = 0.0f;
        for (int r = 0; r < lanes_r; ++r) a += s_red[(r * cv + g) * 8 + e];
        part[((int64_t)blockIdx.x * Ci + c) * K + k] = a;
      }
    }
  }
  if (threadIdx.x < K) {
    float a = 0.0f;
    for (int r = 0; r < lanes_r; ++r) a += s_bias[r * cv][threadIdx.x];   // thread (cg 0, row lane r)
    part_b[(int64_t)blockIdx.x * K + threadIdx.x] = a;
  }
}

// ------------------------------------------------------------------------------------------------
// loss_def (isprs:1089-1099, contest:881-901): per-pixel softmax cross-entropy, mean over (masked) pixels.
// One thread per pixel; block partial sums in fixed order.  dlogits = (softmax - onehot) * mask * inv_count.
// labels are the float class ids the scripts feed (isprs:1654, cast at 1091).
// ------------------------------------------------------------------------------------------------
constexpr int CE_THREADS = 256;
__global__ void __launch_bounds__(CE_THREADS)
ce_fwd_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ labels_f, const uint8_t* __restrict__ mask,
                  int K, int64_t M, const float* __restrict__ count_ptr, float* __restrict__ dlogits,
                  float* __restrict__ part_loss, uint8_t* __restrict__ labels_u8, int ignore_label) {
  pdl_sync();
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const float cnt = *count_ptr;                       // number of pixels in the mean (device scalar: no host round trip)
  const float inv_count = cnt > 0.0f ? 1.0f / cnt : 0.0f;
  float loss = 0.0f;
  if (m < M) {
    float z[MAX_CLASSES];
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < MAX_CLASSES; ++k) {
      z[k] = k < K ? logits[m * K + k] : -INFINITY;
      mx = fmaxf(mx, z[k]);
    }
    float se = 0.0f;
#pragma unroll
    for (int k = 0; k < MAX_CLASSES; ++k)
      if (k < K) se += expf(z[k] - mx);
    const float lse = mx + logf(se);
    const int y = (int)labels_f[m];
    if (labels_u8) labels_u8[m] = (uint8_t)y;
    const bool on = mask ? (mask[m] != 0) : (y != ignore_label);
    if (on && y >= 0 && y < K) loss = lse - z[y];
    if (dlogits) {
#pragma unroll
      for (int k = 0; k < MAX_CLASSES; ++k)
        if (k < K) {
          const float pk = expf(z[k] - lse);
          dlogits[m * K + k] = on ? (pk - (k == y ? 1.0f : 0.0f)) * inv_count : 0.0f;
        }
    }
  }
  __shared__ float s_red[CE_THREADS];
  s_red[threadIdx.x] = loss;
  __syncthreads();
  for (int o = CE_THREADS / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part_loss[blockIdx.x] = s_red[0];
}

// count of mask != 0 (contest): block partials -> single value
__global__ void mask_count_kernel(const uint8_t* __restrict__ mask, const float* __restrict__ labels_f, int ignore_label,
                                  int64_t M, unsigned int* __restrict__ out) {
  pdl_sync();
  unsigned int c = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x)
    c += mask ? (mask[i] != 0) : ((int)labels_f[i] != ignore_label);
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);   // integer: order-independent
}

// out[0] = sum of n floats in fixed order (single block)
__global__ void sum_fixed_kernel(const float* __restrict__ in, int n, float* __restrict__ out, float scale,
                                 const float* __restrict__ divide_by) {
  pdl_sync();
  __shared__ double s[256];
  double a = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) a += (double)in[i];
  s[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double v = s[0] * (double)scale;
    if (divide_by) v = *divide_by > 0.0f ? v * (double)(1.0f / *divide_by) : 0.0;
    out[0] = (float)v;
  }
}
// count of unmasked pixels as the float the loss kernels read
__global__ void set_count_kernel(float* __restrict__ out, const unsigned int* __restrict__ cnt, float fixed) {
  pdl_sync();
  out[0] = cnt ? (float)cnt[0] : fixed;
}

// ------------------------------------------------------------------------------------------------
// calc_accuracy_by_crop (isprs:510-531) / scene confusion (isprs:1289-1296): K x K counts + #correct
// ------------------------------------------------------------------------------------------------
__global__ void confusion_kernel(const uint8_t* __restrict__ truth, const uint8_t* __restrict__ pred,
                                 const uint8_t* __restrict__ mask, int64_t n, int K, int ignore_label,
                                 unsigned int* __restrict__ cm /* K*K+1 */) {
  pdl_sync();
  __shared__ unsigned int s_cm[MAX_CLASSES * MAX_CLASSES + 1];
  for (int i = threadIdx.x; i < K * K + 1; i += blockDim.x) s_cm[i] = 0;
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (mask && !mask[i]) continue;
    const int t = truth[i], p = pred[i];
    if (t == ignore_label || t >= K || p >= K) continue;
    atomicAdd(&s_cm[t * K + p], 1u);
    if (t == p) atomicAdd(&s_cm[K * K], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < K * K + 1; i += blockDim.x)
    if (s_cm[i]) atomicAdd(&cm[i], s_cm[i]);
}

// ------------------------------------------------------------------------------------------------
// MomentumOptimizer (isprs:1685-1687): accum = mom*accum + g ; var -= lr*accum   (Appendix B.6)
// g already contains the CE gradient; the L2 term wd*W is added here for `weights` variables, and the
// loss term wd*sum(W^2)/2 (isprs:640-652) is reduced per block from the pre-update weights.
// ------------------------------------------------------------------------------------------------
__global__ void momentum_update_kernel(float* __restrict__ w, float* __restrict__ g, float* __restrict__ a, int64_t n,
                                       const uint8_t* __restrict__ is_weight, float wd, float lr, float mom,
                                       float grad_scale, float* __restrict__ part_l2) {
  pdl_sync();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float l2 = 0.0f;
  if (i < n) {
    const float wv = w[i];
    float gv = g[i] * grad_scale;
    if (is_weight[i]) {
      gv = fmaf(wd, wv, gv);
      l2 = wv * wv;
    }
    g[i] = gv;                       // total gradient (kept for drs_get_gradient)
    const float av = fmaf(mom, a[i], gv);
    a[i] = av;
    w[i] = wv - lr * av;
  }
  __shared__ float s_red[256];
  s_red[threadIdx.x] = l2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part_l2[blockIdx.x] = s_red[0];
}

// eval-mode BN folded into the conv epilogue: y = act(conv*scale + shift),
// scale = rsqrt(mv+eps), shift = (bias - mm)*scale        (Appendix B.3)
__global__ void fold_bn_kernel(const float* __restrict__ bias, const float* __restrict__ mm, const float* __restrict__ mv,
                               float eps, float* __restrict__ scale, float* __restrict__ shift, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float s = 1.0f / sqrtf(mv[c] + eps);
  scale[c] = s;
  shift[c] = (bias[c] - mm[c]) * s;
}

template <typename TI, typename TO>
__global__ void cast_kernel(const TI* __restrict__ in, TO* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = from_f32<TO>(to_f32(in[i]));
}
// strided 2-D slice -> dense fp32 (debug taps)
template <typename T>
__global__ void slice_to_f32_kernel(const T* __restrict__ in, int cs, int co, int C, int64_t M, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * C) return;
  const int64_t m = i / C;
  const int c = (int)(i - m * C);
  out[i] = to_f32(in[m * cs + co + c]);
}
