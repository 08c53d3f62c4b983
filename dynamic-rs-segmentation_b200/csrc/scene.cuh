// The NumPy loops either side of sess.run, as kernels over an HBM-resident scene:
//   patch gather (+flip, +noise, +override) + normalize_images   isprs:245-334, 74-81
//   sliding-window grid (host, integer, bit-exact)               isprs:337-400, contest:257-328, coffee:296-349
//   ordered overlap accumulation + argmax                        isprs:1261-1284
//   multi-scale softmax sum + argmax                              isprs:1380-1411
#pragma once
#include <algorithm>

#include "drs_common.cuh"
#include "np_softmax.h"

constexpr int GATHER_INLINE_MAX = 256;
// Small batches carry their instance table inside the kernel parameters: no staging copy, no host synchronisation.
struct GatherInline {
  int32_t inst[GATHER_INLINE_MAX * 3];
  uint8_t flips[GATHER_INLINE_MAX];
};

struct GatherParams {
  const int32_t* inst;        // [B,3] scene, row, col
  const uint8_t* flips;       // [B] 0 none, 1 flipud, 2 fliplr
  const double* noise;        // [B,c,c,C] or null
  const uint8_t* noise_on;    // [B] or null
  const int32_t* noise_slot;  // [B] or null: compact noise, block noise_slot[b] of `noise` belongs to patch b (-1: none)
  const double* over_x;       // [B,c,c,C] patch replacing the scene crop (host-rotated), or null
  const uint8_t* over_y;      // [B,c,c]
  const uint8_t* over_on;     // [B] or null
  const double* rot;          // [B,6] m00 m01 m10 m11 off0 off1 of scipy.ndimage.rotate's affine map (isprs:292-296), or null
  const uint8_t* rot_on;      // [B] or null
  uint8_t* amask_out;         // [B,c,c] accuracy mask (rotate(np.ones) then flip, isprs:287, 296, 308-317), or null
  float* x_out;               // [B,c,c,C]
  float* y_out;               // [B,c,c] or null
  int B, crop, C;
  int fp16_patches;           // coffee training: patches are cast to float16 BEFORE normalisation (coffee:293, SURVEY F12)
  double mean[3], stdv[3];
};

// One thread per output element.  Adjacent threads walk the channels then the columns of a scene row,
// so reads of the (H,W,C) scene are contiguous runs of crop*C elements.
template <bool INLINE>
__global__ void gather_kernel(const __grid_constant__ SceneTable tab, const GatherParams p, const __grid_constant__ GatherInline il) {
  const int64_t n = (int64_t)p.B * p.crop * p.crop * p.C;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= n) return;
  const int ch = (int)(gid % p.C);
  int64_t r = gid / p.C;
  const int j = (int)(r % p.crop);
  r /= p.crop;
  const int i = (int)(r % p.crop);
  const int b = (int)(r / p.crop);
  const int32_t* inst = INLINE ? il.inst : p.inst;
  const int sid = inst[b * 3 + 0], row0 = inst[b * 3 + 1], col0 = inst[b * 3 + 2];
  const int flip = INLINE ? il.flips[b] : (p.flips ? p.flips[b] : 0);
  const int si = flip == 1 ? p.crop - 1 - i : i;    // np.flipud (isprs:309-312)
  const int sj = flip == 2 ? p.crop - 1 - j : j;    // np.fliplr (isprs:314-317)
  const SceneDesc& sc = tab.s[sid];
  const bool over = p.over_on && p.over_on[b];
  // scipy.ndimage.rotate(order=0, reshape=False, mode='constant', cval=0): output (si, sj) <- input at
  // floor(cc + 0.5), cc = (off + si*m_0) + sj*m_1 evaluated in this order in float64 (no contraction), and the
  // constant 0 when cc < 0 or cc > crop - 1 on either axis.  Pinned against scipy for every integer angle.
  int ri = si, rj = sj;
  bool outside = false;
  if (p.rot_on && p.rot_on[b]) {
    const double* m = p.rot + (int64_t)b * 6;
    const double c0 = __dadd_rn(__dadd_rn(m[4], __dmul_rn((double)si, m[0])), __dmul_rn((double)sj, m[1]));
    const double c1 = __dadd_rn(__dadd_rn(m[5], __dmul_rn((double)si, m[2])), __dmul_rn((double)sj, m[3]));
    const double hi = (double)(p.crop - 1);
    outside = c0 < 0.0 || c0 > hi || c1 < 0.0 || c1 > hi;
    if (!outside) {
      ri = (int)floor(__dadd_rn(c0, 0.5));
      rj = (int)floor(__dadd_rn(c1, 0.5));
    }
  }
  const int64_t pidx = (((int64_t)b * p.crop + si) * p.crop + sj);
  const int64_t sidx = ((int64_t)(row0 + ri - sc.row0) * sc.W + (col0 + rj));
  float outv;
  if (sc.dtype == DRS_SCENE_F64 || over || (p.rot_on && p.rot_on[b])) {
    double v = over ? p.over_x[pidx * p.C + ch]
                    : (outside ? 0.0 : (sc.dtype == DRS_SCENE_F64 ? reinterpret_cast<const double*>(sc.data)[sidx * sc.C + ch]
                                                                  : (double)reinterpret_cast<const float*>(sc.data)[sidx * sc.C + ch]));
    if (p.noise_on && p.noise_on[b]) {                                    // isprs:301
      const int64_t nidx = p.noise_slot ? (((int64_t)p.noise_slot[b] * p.crop + si) * p.crop + sj) : pidx;
      v = v + p.noise[nidx * p.C + ch];
    }
    if (ch < 3) {                                                          // isprs:75-81 (channels 0..2 only)
      v = v - p.mean[ch];
      v = v / p.stdv[ch];
    }
    outv = (float)v;                                                       // feed_dict cast to float32
  } else if (p.fp16_patches) {
    // NumPy float16 arithmetic of the reference era: operands widened to float32, one operation, result rounded to half;
    // the float64 mean/std scalars are first cast to the array's dtype (half)
    __half hv = __float2half_rn(reinterpret_cast<const float*>(sc.data)[sidx * sc.C + ch]);
    if (ch < 3) {
      hv = __float2half_rn(__half2float(hv) - __half2float(__double2half(p.mean[ch])));
      hv = __float2half_rn(__half2float(hv) / __half2float(__double2half(p.stdv[ch])));
    }
    outv = __half2float(hv);
  } else {
    float v = reinterpret_cast<const float*>(sc.data)[sidx * sc.C + ch];
    if (ch < 3) {                                                          // float32 scene: float32 arithmetic
      v = v - (float)p.mean[ch];
      v = v / (float)p.stdv[ch];
    }
    outv = v;
  }
  p.x_out[gid] = outv;
  if (p.y_out && ch == 0) {
    const uint8_t lab = over ? p.over_y[pidx] : ((sc.labels && !outside) ? sc.labels[sidx] : 0);
    p.y_out[((int64_t)b * p.crop + i) * p.crop + j] = (float)lab;
  }
  if (p.amask_out && ch == 0) p.amask_out[((int64_t)b * p.crop + i) * p.crop + j] = outside ? 0 : 1;
}

// ------------------------------------------------------------------------------------------------
// sliding-window grid (host).  Bit-exact restatement of create_patches_per_map's index arithmetic.
// ------------------------------------------------------------------------------------------------
static inline int grid_count(int length, int crop, int stride) {
  return ((length - crop) % stride == 0) ? (length - crop) / stride + 1 : (length - crop) / stride + 2;
}

// positions (row, col) of every patch the script visits, batch after batch (isprs:1264-1267)
static void grid_positions(int H, int W, int crop, int batch, int variant, std::vector<int32_t>& pos) {
  const int stride = crop / 2;                       // isprs:1243 floor(crop/2)
  DRS_CHECK(stride >= 1 && crop <= H && crop <= W, "grid: crop %d does not fit scene %dx%d", crop, H, W);
  DRS_CHECK(batch >= 1, "grid: batch must be >= 1");
  const int th = grid_count(H, crop, stride);
  int tw = grid_count(W, crop, stride);
  int div = tw, mod = tw;
  int total_w_for_count = tw;
  if (variant == DRS_GRID_CONTEST) { div = th; mod = tw; }            // contest:275-276 (SURVEY F10)
  else if (variant == DRS_GRID_COFFEE) { div = th; mod = th; tw = th; }  // coffee:302-307
  const int64_t total = (int64_t)th * total_w_for_count;             // instaces_stride (isprs:1257)
  const int64_t nb = total % batch != 0 ? total / batch + 1 : total / batch;
  pos.clear();
  for (int64_t index = 0; index < nb; ++index) {
    int offset_h = (int)((index * batch) / div) * stride;
    int offset_w = (int)((index * batch) % mod) * stride;
    int count = 0;
    bool first = true, done = false;
    for (int j = offset_h; j < th * stride && !done; j += stride) {
      if (!first) offset_w = 0;
      for (int k = offset_w; k < tw * stride; k += stride) {
        first = false;
        int cx = j, cy = k;
        const int len_x = std::max(0, std::min(cx + crop, H) - cx);
        const int len_y = std::max(0, std::min(cy + crop, W) - cy);
        if (len_x != crop) cx -= crop - len_x;
        if (len_y != crop) cy -= crop - len_y;
        pos.push_back(cx);
        pos.push_back(cy);
        if (++count == batch) { done = true; break; }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// ordered accumulation.  The lattice of patch origins is {i*s} U {H-c} x {j*s} U {W-c}; a cell is
// visited once by the isprs grid and the coffee grid (square tiles) and any number of times by the
// contest grid (bug F10).
// cell_off/cell_seq list, per cell, the visit numbers in ascending order.  Each thread owns one pixel
// and adds its contributions in visit order, which makes the fp32 sum bit-identical to NumPy's
// sequential `prob_im[...] += logits[j]` without atomics.
// ------------------------------------------------------------------------------------------------
struct AccumParams {
  const float* logits;      // [n_chunk, c, c, K], patch `seq` lives at (seq - seq0)
  const int32_t* cell_off;  // [nh*nw + 1]
  const int32_t* cell_seq;  // visit numbers
  float* prob;              // [rows, W, K] for image rows [row_begin, row_end)
  uint32_t* occur;          // [rows, W]
  int H, W, K, crop, stride, nh, nw;
  int row_begin, row_end;   // stripe owned by this rank
  int y_lo, y_hi;           // pixel rows touched by this chunk (clipped to the stripe)
  int seq0, seq1;           // visit numbers held in `logits`
  uint32_t* overflow;       // host-mapped flag: a pixel had more contributions in one launch than the kernel can order
};
// Contributions one launch orders per pixel.  A pixel lies under at most 4 x 4 lattice cells (odd crop + shifted border
// row/col); the host splits a chunk into visit ranges that stay within this limit (drs_scene_api.cuh: accum_ranges).
constexpr int ACCUM_MAX_CONTRIB = 32;

__device__ __forceinline__ int cover_range(int y, int L, int crop, int stride, int n, int* first, int* extra) {
  // regular origins i*s for i in [0, n-2] (and n-1 when the last origin is not shifted), last origin L-crop
  const int last_origin = L - crop;
  const bool last_regular = ((n - 1) * stride == last_origin);
  const int n_reg = last_regular ? n : n - 1;
  int lo = (y - crop + stride) / stride;             // ceil((y-crop+1)/stride) for y-crop+1 > 0
  if (y - crop + 1 <= 0) lo = 0;
  int hi = y / stride;
  if (hi > n_reg - 1) hi = n_reg - 1;
  *first = lo;
  *extra = (!last_regular && y >= last_origin) ? 1 : 0;   // the shifted last row/col also covers y
  return hi - lo + 1;                                  // may be <= 0
}

__global__ void accumulate_kernel(const AccumParams p) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = p.y_lo + blockIdx.y;
  if (x >= p.W || y >= p.y_hi) return;
  int i0, iex, j0, jex;
  const int ni = cover_range(y, p.H, p.crop, p.stride, p.nh, &i0, &iex);
  const int nj = cover_range(x, p.W, p.crop, p.stride, p.nw, &j0, &jex);
  const int ti = (ni > 0 ? ni : 0) + iex, tj = (nj > 0 ? nj : 0) + jex;
  int seqs[ACCUM_MAX_CONTRIB], oy[ACCUM_MAX_CONTRIB], ox[ACCUM_MAX_CONTRIB];
  int n = 0;
  for (int a = 0; a < ti; ++a) {
    const int i = (a < ni) ? i0 + a : p.nh - 1;
    const int y0 = (i == p.nh - 1) ? p.H - p.crop : i * p.stride;
    for (int b = 0; b < tj; ++b) {
      const int j = (b < nj) ? j0 + b : p.nw - 1;
      const int x0 = (j == p.nw - 1) ? p.W - p.crop : j * p.stride;
      const int cell = i * p.nw + j;
      for (int v = p.cell_off[cell]; v < p.cell_off[cell + 1]; ++v) {
        const int s = p.cell_seq[v];
        if (s >= p.seq0 && s < p.seq1 && n >= ACCUM_MAX_CONTRIB) {
          *p.overflow = 1u;        // never dropped silently: the pass fails (scene_pass_finish)
        } else if (s >= p.seq0 && s < p.seq1) {
          // insertion keeps ascending visit order
          int k = n++;
          while (k > 0 && seqs[k - 1] > s) {
            seqs[k] = seqs[k - 1]; oy[k] = oy[k - 1]; ox[k] = ox[k - 1];
            --k;
          }
          seqs[k] = s; oy[k] = y - y0; ox[k] = x - x0;
        }
      }
    }
  }
  if (n == 0) return;
  const int64_t pix = (int64_t)(y - p.row_begin) * p.W + x;
  float acc[MAX_CLASSES];
  for (int k = 0; k < p.K; ++k) acc[k] = p.prob[pix * p.K + k];
  for (int q = 0; q < n; ++q) {
    const float* lg = p.logits + ((((int64_t)(seqs[q] - p.seq0) * p.crop + oy[q]) * p.crop + ox[q]) * p.K);
    for (int k = 0; k < p.K; ++k) acc[k] = acc[k] + lg[k];
  }
  for (int k = 0; k < p.K; ++k) p.prob[pix * p.K + k] = acc[k];
  p.occur[pix] += (uint32_t)n;
}

// occur==0 -> 1 ; mean = prob / float64(occur) ; label = first argmax   (isprs:1282-1284)
__global__ void scene_argmax_kernel(const float* __restrict__ prob, const uint32_t* __restrict__ occur, int64_t npix,
                                    int K, uint8_t* __restrict__ labels, double* __restrict__ mean_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  uint32_t oc = occur[i];
  if (oc == 0) oc = 1;
  const double d = (double)oc;
  double best = -INFINITY;
  int bi = 0;
  for (int k = 0; k < K; ++k) {
    const double v = (double)prob[i * K + k] / d;
    if (mean_out) mean_out[i * K + k] = v;
    if (v > best) { best = v; bi = k; }
  }
  labels[i] = (uint8_t)bi;
}

// validate_test_multiscale (isprs:1380-1411), per pixel after each scale's pass, in NumPy's float32 arithmetic:
//   acc += softmax(float32(prob / float64(occur)))     (occur==0 -> 1; the first scale adds to 0, which is exact)
// and on the last scale (labels non-null) label = np.argmax(acc): the first maximum, or the first NaN.
static_assert(MAX_CLASSES <= NP_SOFTMAX_MAX_K, "np_softmax_pixel holds MAX_CLASSES values");
__global__ void multiscale_softmax_add_kernel(const float* __restrict__ prob, const uint32_t* __restrict__ occur, int64_t npix,
                                              int K, int first, float* __restrict__ acc, uint8_t* __restrict__ labels) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  uint32_t oc = occur[i];
  if (oc == 0) oc = 1;
  const double d = (double)oc;
  float m[NP_SOFTMAX_MAX_K], p[NP_SOFTMAX_MAX_K];
#pragma unroll
  for (int k = 0; k < NP_SOFTMAX_MAX_K; ++k)
    if (k < K) m[k] = __double2float_rn(__ddiv_rn((double)prob[i * K + k], d));   // mean_prob[scale] = prob_im / occur_im
  np_softmax_pixel(m, K, p);
  float best = 0.0f;
  int bi = 0;
  bool nan_seen = false;
#pragma unroll
  for (int k = 0; k < NP_SOFTMAX_MAX_K; ++k)
    if (k < K) {
      const float a = __fadd_rn(first ? 0.0f : acc[i * K + k], p[k]);
      acc[i * K + k] = a;
      if (!nan_seen && (k == 0 || !(a <= best))) {
        best = a;
        bi = k;
        nan_seen = a != a;
      }
    }
  if (labels) labels[i] = (uint8_t)bi;
}
