// Training-mode 3x3 / stride 1 / SAME max-pool for bf16, forward and backward, written against the instruction count.
// Included by ops.cuh (after BnFinish).  isprs:745-750 (_max_pool), used by every pooling net of the three scripts.
//
// Both kernels of round 1 were issue-bound, not bandwidth-bound (ncu: 66-74 % issue-slot utilisation at 10-20 % DRAM): the
// forward executed 309 instructions per (pixel, 8 channels), the backward 454.  Same data flow here -- a thread owns
// (image, column x, 8 channels) and walks along the rows with the neighbouring rows in registers -- but
//   * forward: activation as a template parameter (no per-element branch), the three-row window rotates by renaming (the
//     row loop is unrolled by six = lcm of the 3-row window and the 2-deep load pipeline), the horizontal maximum starts
//     from the left neighbour instead of -inf;
//   * backward: scatter instead of gather.  Every window's gradient goes to exactly one of nine positions, three of which
//     (one per row) lie in this thread's column; the thread keeps three rows of fp32 accumulators and, per loaded window,
//     issues three packed 16-bit compares (winner code == target) whose predicate pair guards two fp32 adds.  The codes are
//     widened once per load into fp16 bit patterns 0x44cc (distinct normal numbers), so HSETP2 compares two channels per
//     instruction; no masks, no byte permutes, no shifts per tap.  Rows are walked bottom-up with the windows right to left:
//     that is the summation order of the gather kernels (dy = -1, 0, +1; dx = -1, 0, +1), so results are bit-identical.
#pragma once

namespace pool_lean {

constexpr unsigned NINF2 = 0xFF80FF80u;

template <int ACT>
__device__ __forceinline__ float act_t(float v) {
  if (ACT == ACT_RELU) return fmaxf(v, 0.0f);
  if (ACT == ACT_LRELU) return fmaxf(0.1f * v, v);
  return v;
}

struct Row3 { uint4 q[3]; };

// raw values of window row y at columns x-1, x, x+1; -inf outside the image (never wins a strictly-greater compare)
__device__ __forceinline__ void load_row(const __nv_bfloat16* __restrict__ pc, int64_t rs, int in_cs, int y, int crop, bool xl,
                                         bool xr, Row3& r) {
  const bool ok = (unsigned)y < (unsigned)crop;
  const __nv_bfloat16* p = pc + (int64_t)y * rs;
  const uint4 ninf = make_uint4(NINF2, NINF2, NINF2, NINF2);
  r.q[0] = ninf; r.q[1] = ninf; r.q[2] = ninf;
  if (ok) r.q[1] = *reinterpret_cast<const uint4*>(p);
  if (ok && xl) r.q[0] = *reinterpret_cast<const uint4*>(p - in_cs);
  if (ok && xr) r.q[2] = *reinterpret_cast<const uint4*>(p + in_cs);
}

// horizontal first-maximum of a row: value and dx index (0, 1, 2) per 16-bit lane
__device__ __forceinline__ void hmax_row(const Row3& r, __nv_bfloat162 (&rv)[4], unsigned (&ri)[4]) {
  const __nv_bfloat162* q0 = reinterpret_cast<const __nv_bfloat162*>(&r.q[0]);
  const __nv_bfloat162* q1 = reinterpret_cast<const __nv_bfloat162*>(&r.q[1]);
  const __nv_bfloat162* q2 = reinterpret_cast<const __nv_bfloat162*>(&r.q[2]);
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    unsigned m = __hgt2_mask(q1[w], q0[w]);
    __nv_bfloat162 v = __hmax2(q0[w], q1[w]);
    unsigned i = m & 0x00010001u;
    m = __hgt2_mask(q2[w], v);
    v = __hmax2(v, q2[w]);
    i = (i & ~m) | (0x00020002u & m);
    rv[w] = v;
    ri[w] = i;
  }
}

// one output row: vertical first-maximum over (va, vb, vc) = rows y-1, y, y+1, normalise + activation of the winner, stores
template <int ACT>
__device__ __forceinline__ void fwd_emit(const __nv_bfloat162 (&va)[4], const unsigned (&ia)[4], const __nv_bfloat162 (&vb)[4],
                                         const unsigned (&ib)[4], const __nv_bfloat162 (&vc)[4], const unsigned (&ic)[4],
                                         const float (&mu)[8], const float (&is)[8], __nv_bfloat16* __restrict__ po,
                                         uint8_t* __restrict__ pi) {
  uint4 o;
  unsigned code[4];
  unsigned* ow = reinterpret_cast<unsigned*>(&o);
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    unsigned m = __hgt2_mask(vb[w], va[w]);
    __nv_bfloat162 best = __hmax2(va[w], vb[w]);
    unsigned bi = (ia[w] & ~m) | ((ib[w] + 0x00030003u) & m);
    m = __hgt2_mask(vc[w], best);
    best = __hmax2(best, vc[w]);
    bi = (bi & ~m) | ((ic[w] + 0x00060006u) & m);
    code[w] = bi;
    const unsigned raw = *reinterpret_cast<const unsigned*>(&best);
    const float lo = act_t<ACT>((__uint_as_float(raw << 16) - mu[2 * w]) * is[2 * w]);
    const float hi = act_t<ACT>((__uint_as_float(raw & 0xFFFF0000u) - mu[2 * w + 1]) * is[2 * w + 1]);
    const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    ow[w] = *reinterpret_cast<const unsigned*>(&p);
  }
  *reinterpret_cast<uint4*>(po) = o;
  uint2 pk;
  pk.x = __byte_perm(code[0], code[1], 0x6420);      // low byte of every 16-bit lane
  pk.y = __byte_perm(code[2], code[3], 0x6420);
  *reinterpret_cast<uint2*>(pi) = pk;
}

template <int ACT>
__global__ void __launch_bounds__(256, DRS_POOL_MINBLK)
fwd_kernel(const __nv_bfloat16* __restrict__ in, int in_cs, int in_co, __nv_bfloat16* __restrict__ out, int out_cs, int out_co,
           uint8_t* __restrict__ idx, int C, int B, int crop, int seg, int nseg, const float* __restrict__ bn_mean,
           const float* __restrict__ bn_inv_std) {
  pdl_sync();
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
  const int64_t pix0 = (int64_t)b * crop * crop + x;                     // pixel (row 0, column x) of this image
  const bool xl = x > 0, xr = x + 1 < crop;
  const __nv_bfloat16* pc = in + pix0 * in_cs + in_co + cg * 8;
  const int64_t rs = (int64_t)crop * in_cs;
  __nv_bfloat16* po = out + (pix0 + (int64_t)y0 * crop) * out_cs + out_co + cg * 8;
  uint8_t* pi = idx + (pix0 + (int64_t)y0 * crop) * C + cg * 8;
  const int64_t os = (int64_t)crop * out_cs, cs = (int64_t)crop * C;
  float mu[8], is[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { mu[e] = bn_mean[cg * 8 + e]; is[e] = bn_inv_std[cg * 8 + e]; }
  __nv_bfloat162 v0[4], v1[4], v2[4];
  unsigned i0[4], i1[4], i2[4];
  Row3 ra, rb;
  load_row(pc, rs, in_cs, y0 - 1, crop, xl, xr, ra);
  load_row(pc, rs, in_cs, y0, crop, xl, xr, rb);
  hmax_row(ra, v0, i0);
  load_row(pc, rs, in_cs, y0 + 1, crop, xl, xr, ra);
  hmax_row(rb, v1, i1);
  // invariant at the top of a step for output row y: (A, B) hold the reduced rows y-1 and y, CUR the raw row y+1;
  // the raw row y+2 is requested into NXT before CUR is reduced, so a row of loads is always in flight
#define DRS_POOL_FWD_STEP(A_V, A_I, B_V, B_I, C_V, C_I, CUR, NXT)             \
  {                                                                            \
    load_row(pc, rs, in_cs, y + 2, crop, xl, xr, NXT);                         \
    hmax_row(CUR, C_V, C_I);                                                   \
    fwd_emit<ACT>(A_V, A_I, B_V, B_I, C_V, C_I, mu, is, po, pi);               \
    po += os; pi += cs;                                                        \
    if (++y >= y1) break;                                                      \
  }
  for (int y = y0;;) {
    DRS_POOL_FWD_STEP(v0, i0, v1, i1, v2, i2, ra, rb)
    DRS_POOL_FWD_STEP(v1, i1, v2, i2, v0, i0, rb, ra)
    DRS_POOL_FWD_STEP(v2, i2, v0, i0, v1, i1, ra, rb)
    DRS_POOL_FWD_STEP(v0, i0, v1, i1, v2, i2, rb, ra)
    DRS_POOL_FWD_STEP(v1, i1, v2, i2, v0, i0, ra, rb)
    DRS_POOL_FWD_STEP(v2, i2, v0, i0, v1, i1, rb, ra)
  }
#undef DRS_POOL_FWD_STEP
}

// ------------------------------------------------------------------------------------------------ backward
struct BwdRow {
  unsigned c16[3][4];     // winner codes of windows (yo, x-1), (yo, x), (yo, x+1), one fp16 pattern 0x44cc per channel
  uint4 g[3];             // their output gradients
};

__device__ __forceinline__ void bwd_load(const __nv_bfloat16* __restrict__ pg, int64_t gs, int do_cs, const uint8_t* __restrict__ pk,
                                         int64_t ks, int C, int yo, int crop, bool xl, bool xr, BwdRow& r) {
  const bool ok = (unsigned)yo < (unsigned)crop;
  const __nv_bfloat16* p = pg + (int64_t)yo * gs;
  const uint8_t* q = pk + (int64_t)yo * ks;
  uint2 c[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const bool okj = ok && (j == 0 ? xl : j == 2 ? xr : true);
    c[j] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);           // 0x44ff never equals a code 0x4400..0x4408
    r.g[j] = make_uint4(0u, 0u, 0u, 0u);
    if (okj) {
      c[j] = *reinterpret_cast<const uint2*>(q + (int64_t)(j - 1) * C);
      r.g[j] = *reinterpret_cast<const uint4*>(p + (int64_t)(j - 1) * do_cs);
    }
    r.c16[j][0] = __byte_perm(c[j].x, 0x44444444u, 0x4140);
    r.c16[j][1] = __byte_perm(c[j].x, 0x44444444u, 0x4342);
    r.c16[j][2] = __byte_perm(c[j].y, 0x44444444u, 0x4140);
    r.c16[j][3] = __byte_perm(c[j].y, 0x44444444u, 0x4342);
  }
}

// acc[2w], acc[2w+1] += the two channels of g word w where the window's code equals `target`
__device__ __forceinline__ void tap(const unsigned (&c16)[4], const uint4& g, unsigned target, float (&acc)[8]) {
  const unsigned gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    const float lo = __uint_as_float(gw[w] << 16), hi = __uint_as_float(gw[w] & 0xFFFF0000u);
    asm("{\n\t.reg .pred p, q;\n\t"
        "setp.eq.f16x2 p|q, %2, %3;\n\t"
        "@p add.f32 %0, %0, %4;\n\t"
        "@q add.f32 %1, %1, %5;\n\t}"
        : "+f"(acc[2 * w]), "+f"(acc[2 * w + 1])
        : "r"(c16[w]), "r"(target), "f"(lo), "f"(hi));
  }
}

// Window row yo scatters into the position rows yo-1 (UP), yo (MID), yo+1 (DOWN) of this thread's column.  The window at
// column x + j - 1 holds this column as its element dx = 1 - j, i.e. code column 2 - j; its row dy = -1 (codes 0..2) is
// position row yo-1, dy = 0 (3..5) is row yo, dy = +1 (6..8) is row yo+1.
template <bool DO_UP, bool DO_MID, bool DO_DOWN>
__device__ __forceinline__ void bwd_scatter(const BwdRow& r, float (&up)[8], float (&mid)[8], float (&down)[8]) {
#pragma unroll
  for (int j = 2; j >= 0; --j) {
    const unsigned col = (unsigned)(2 - j);
    if (DO_UP) tap(r.c16[j], r.g[j], 0x44004400u + (0u + col) * 0x00010001u, up);
    if (DO_MID) tap(r.c16[j], r.g[j], 0x44004400u + (3u + col) * 0x00010001u, mid);
    if (DO_DOWN) tap(r.c16[j], r.g[j], 0x44004400u + (6u + col) * 0x00010001u, down);
  }
}

// rounds and stores a finished row, clears its accumulators
__device__ __forceinline__ void bwd_emit(float (&acc)[8], __nv_bfloat16* __restrict__ pd) {
  uint4 o;
  unsigned* ow = reinterpret_cast<unsigned*>(&o);
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    const __nv_bfloat162 p = __floats2bfloat162_rn(acc[2 * w], acc[2 * w + 1]);
    ow[w] = *reinterpret_cast<const unsigned*>(&p);
    acc[2 * w] = 0.0f;
    acc[2 * w + 1] = 0.0f;
  }
  *reinterpret_cast<uint4*>(pd) = o;
}

__global__ void __launch_bounds__(256, DRS_POOL_MINBLK)
bwd_kernel(const __nv_bfloat16* __restrict__ dout, int do_cs, int do_co, const uint8_t* __restrict__ idx,
           __nv_bfloat16* __restrict__ din, int di_cs, int di_co, int C, int B, int crop, int seg, int nseg) {
  pdl_sync();
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
  const int64_t pix0 = (int64_t)b * crop * crop + x;
  const bool xl = x > 0, xr = x + 1 < crop;
  const __nv_bfloat16* pg = dout + pix0 * do_cs + do_co + cg * 8;
  const uint8_t* pk = idx + pix0 * C + cg * 8;
  const int64_t gs = (int64_t)crop * do_cs, ks = (int64_t)crop * C;
  __nv_bfloat16* pd = din + (pix0 + (int64_t)(y1 - 1) * crop) * di_cs + di_co + cg * 8;
  const int64_t ds = (int64_t)crop * di_cs;
  float a0[8], a1[8], a2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { a0[e] = 0.0f; a1[e] = 0.0f; a2[e] = 0.0f; }
  BwdRow r;
  // Bottom-up: position row y is complete once window rows y+1, y, y-1 have been scattered, in that order (the gather
  // kernels' dy = -1, 0, +1).  Prologue: window row y1 reaches only row y1-1 of this segment, window row y1-1 rows y1-1
  // and y1-2; contributions to rows outside [y0, y1) belong to other threads and are not computed.
  bwd_load(pg, gs, do_cs, pk, ks, C, y1, crop, xl, xr, r);
  bwd_scatter<true, false, false>(r, a0, a1, a2);
  bwd_load(pg, gs, do_cs, pk, ks, C, y1 - 1, crop, xl, xr, r);
  bwd_scatter<true, true, false>(r, a1, a0, a2);
  // step for position row y: ACC_Y = row y (window rows y+1 and y already in), ACC_1 = row y-1, ACC_2 = row y-2 (zero)
#define DRS_POOL_BWD_STEP(ACC_Y, ACC_1, ACC_2)                                                   \
  {                                                                                               \
    bwd_load(pg, gs, do_cs, pk, ks, C, y - 1, crop, xl, xr, r);                                   \
    if (y > y0) bwd_scatter<true, true, true>(r, ACC_2, ACC_1, ACC_Y);                            \
    else bwd_scatter<false, false, true>(r, ACC_2, ACC_1, ACC_Y);                                 \
    bwd_emit(ACC_Y, pd);                                                                          \
    pd -= ds;                                                                                     \
    if (--y < y0) break;                                                                          \
  }
  for (int y = y1 - 1;;) {
    DRS_POOL_BWD_STEP(a0, a1, a2)
    DRS_POOL_BWD_STEP(a1, a2, a0)
    DRS_POOL_BWD_STEP(a2, a0, a1)
  }
#undef DRS_POOL_BWD_STEP
}

// ------------------------------------------------------------------------------------------------ backward + BN backward
// The pool backward and the batch-norm backward of the layer below in one pass: the gradient of the pool input never
// goes to memory (it was written as bf16 and read back twice, by the statistics pass and by bn_bwd_apply_kernel):
//   dZ = inv_std * (g - s0/M - xh * s1/M),   g = dIn * act'(xh),   xh = (z - mean) * inv_std
// with dIn the fp32 sum the scatter has just finished for this row.  The two sums come from bn_partial_kernel<MODE 2>,
// which needs only the window gradients and the pooled activations (every window hands its whole gradient to its winner,
// so sum_positions g = sum_windows dOut * act'(winner) and likewise for g * xh).  The four per-channel constants live in
// shared memory (registers would cost the kernel a resident block).
__device__ __forceinline__ uint4 ldg_nc_u4(const void* p) {       // asm volatile: stays where it is written
  uint4 v;
  asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 lds_f4(const float* p) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(static_cast<unsigned>(__cvta_generic_to_shared(p))));
  return v;
}
template <int ACT>
__device__ __forceinline__ void bwd_emit_apply(float (&acc)[8], __nv_bfloat16* __restrict__ pd, const __nv_bfloat16* __restrict__ pz,
                                               const float* __restrict__ s_c, int C, int c0, const uint4& zraw) {
  const unsigned* zw = reinterpret_cast<const unsigned*>(&zraw);
  uint4 o;
  unsigned* ow = reinterpret_cast<unsigned*>(&o);
#pragma unroll
  for (int hv = 0; hv < 2; ++hv) {
    // (volatile: re-read every row -- hoisted out of the row loop the 32 values would live in registers again)
    const float4 mu = lds_f4(s_c + c0 + 4 * hv);
    const float4 is = lds_f4(s_c + C + c0 + 4 * hv);
    const float4 m0 = lds_f4(s_c + 2 * C + c0 + 4 * hv);
    const float4 m1 = lds_f4(s_c + 3 * C + c0 + 4 * hv);
    const float muv[4] = {mu.x, mu.y, mu.z, mu.w}, isv[4] = {is.x, is.y, is.z, is.w};
    const float m0v[4] = {m0.x, m0.y, m0.z, m0.w}, m1v[4] = {m1.x, m1.y, m1.z, m1.w};
    float dz[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = 4 * hv + q;
      const unsigned zz = zw[e >> 1];
      const float zf = __uint_as_float((e & 1) ? (zz & 0xFFFF0000u) : (zz << 16));
      const float xh = (zf - muv[q]) * isv[q];
      float g = acc[e];
      if (ACT == ACT_RELU) g = xh > 0.0f ? g : 0.0f;
      else if (ACT == ACT_LRELU) g = xh > 0.0f ? g : 0.1f * g;
      dz[q] = isv[q] * (g - m0v[q] - xh * m1v[q]);
      acc[e] = 0.0f;
    }
    const __nv_bfloat162 p0 = __floats2bfloat162_rn(dz[0], dz[1]), p1 = __floats2bfloat162_rn(dz[2], dz[3]);
    ow[2 * hv] = *reinterpret_cast<const unsigned*>(&p0);
    ow[2 * hv + 1] = *reinterpret_cast<const unsigned*>(&p1);
  }
  *reinterpret_cast<uint4*>(pd) = o;
}

#ifndef DRS_POOL_APPLY_MINBLK
#define DRS_POOL_APPLY_MINBLK 2
#endif
template <int ACT>
__global__ void __launch_bounds__(256, DRS_POOL_APPLY_MINBLK)
bwd_apply_kernel(const __nv_bfloat16* __restrict__ dout, int do_cs, int do_co, const uint8_t* __restrict__ idx,
                 __nv_bfloat16* __restrict__ dz, int dz_cs, int dz_co, int C, int B, int crop, int seg, int nseg,
                 const __nv_bfloat16* __restrict__ z, const float* __restrict__ mean, const float* __restrict__ inv_std,
                 const float* __restrict__ sums, double inv_count) {
  extern __shared__ __align__(16) float s_c[];        // [4][C]: mean, inv_std, s0/M, s1/M
  pdl_sync();
  for (int c = threadIdx.x; c < C; c += 256) {
    s_c[c] = mean[c];
    s_c[C + c] = inv_std[c];
    s_c[2 * C + c] = (float)((double)sums[c] * inv_count);
    s_c[3 * C + c] = (float)((double)sums[C + c] * inv_count);
  }
  __syncthreads();
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
  const int64_t pix0 = (int64_t)b * crop * crop + x;
  const bool xl = x > 0, xr = x + 1 < crop;
  const __nv_bfloat16* pg = dout + pix0 * do_cs + do_co + cg * 8;
  const uint8_t* pk = idx + pix0 * C + cg * 8;
  const int64_t gs = (int64_t)crop * do_cs, ks = (int64_t)crop * C;
  __nv_bfloat16* pd = dz + (pix0 + (int64_t)(y1 - 1) * crop) * dz_cs + dz_co + cg * 8;
  const int64_t ds = (int64_t)crop * dz_cs;
  const __nv_bfloat16* pz = z + (pix0 + (int64_t)(y1 - 1) * crop) * C + cg * 8;
  const int64_t zs = (int64_t)crop * C;
  float a0[8], a1[8], a2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { a0[e] = 0.0f; a1[e] = 0.0f; a2[e] = 0.0f; }
  BwdRow r;
  bwd_load(pg, gs, do_cs, pk, ks, C, y1, crop, xl, xr, r);
  bwd_scatter<true, false, false>(r, a0, a1, a2);
  bwd_load(pg, gs, do_cs, pk, ks, C, y1 - 1, crop, xl, xr, r);
  bwd_scatter<true, true, false>(r, a1, a0, a2);
#define DRS_POOL_BWD_STEP(ACC_Y, ACC_1, ACC_2)                                                   \
  {                                                                                               \
    /* Z comes from DRAM (written in the forward): requested before the window row, consumed after the scatter */ \
    const uint4 zraw = ldg_nc_u4(pz);                                                             \
    bwd_load(pg, gs, do_cs, pk, ks, C, y - 1, crop, xl, xr, r);                                   \
    if (y > y0) bwd_scatter<true, true, true>(r, ACC_2, ACC_1, ACC_Y);                            \
    else bwd_scatter<false, false, true>(r, ACC_2, ACC_1, ACC_Y);                                 \
    bwd_emit_apply<ACT>(ACC_Y, pd, pz, s_c, C, cg * 8, zraw);                                     \
    pd -= ds;                                                                                     \
    pz -= zs;                                                                                     \
    if (--y < y0) break;                                                                          \
  }
  for (int y = y1 - 1;;) {
    DRS_POOL_BWD_STEP(a0, a1, a2)
    DRS_POOL_BWD_STEP(a1, a2, a0)
    DRS_POOL_BWD_STEP(a2, a0, a1)
  }
#undef DRS_POOL_BWD_STEP
}

}  // namespace pool_lean
