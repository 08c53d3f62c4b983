// NumPy's float32 softmax of the multi-scale evaluation (softmax, isprs:38-43: exp, sum over the last axis, divide), restated
// operation by operation so that the device reproduces the host composition bit for bit.  One source for both sides: the
// scene pass includes it in a CUDA unit (scene.cuh), and np_softmax.cpp compiles it for the host (drs_debug_np_softmax, CPU
// tests) without FMA contraction and without fast-math.
//
// NumPy's float32 exp is not correctly rounded (up to 2 ulp off on ~39 % of inputs), so expf would not match it.  Its SIMD
// algorithm (the AVX-512F and AVX2+FMA3 paths of numpy 2.x) uses IEEE float32 operations only: rint by the magic constant,
// a two-step Cody-Waite reduction, a rational approximation of degree 5/2 and an exact scaling.  np_expf restates it; on the
// host it matched np.exp (numpy 2.3.5, AVX-512) on every one of the 4,278,190,080 finite float32 inputs, denormal results
// included.  Every operation is written as its own rounding step: on the device as the _rn intrinsics, which nvcc never
// fuses (a plain a*b+c becomes one FMA under --fmad=true, and fusing the rint into an FMA alone gave 84 mismatches).
//
// np.sum over the last axis is NumPy's pairwise_sum: K < 8 contiguous float32 values are added in order, ((e0+e1)+e2)+...,
// and K = 8 by its eight-accumulator path, ((e0+e1)+(e2+e3))+((e4+e5)+(e6+e7)).  np.divide is IEEE division.
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define NP_HD __host__ __device__ __forceinline__
#else
#define NP_HD inline
#endif

constexpr int NP_SOFTMAX_MAX_K = 8;

NP_HD float np_mul(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
NP_HD float np_add(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
NP_HD float np_fma(float a, float b, float c) {
#ifdef __CUDA_ARCH__
  return __fmaf_rn(a, b, c);
#else
  return fmaf(a, b, c);
#endif
}
NP_HD float np_div(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fdiv_rn(a, b);
#else
  return a / b;
#endif
}

// np.exp on a float32 value
NP_HD float np_expf(float x) {
  if (x != x) return x;
  if (x > 88.72283935546875f) return INFINITY;
  if (x < -103.97208404541015625f) return 0.0f;
  float q = np_mul(x, 0x1.715476p+0f);                 // x * log2(e), then rint by the magic constant
  q = np_add(np_add(q, 0x1.8p+23f), -0x1.8p+23f);
  float y = np_fma(q, -6.93145752e-1f, x);             // Cody-Waite: x - q * ln2 in two parts
  y = np_fma(q, -1.42860677e-6f, y);
  float n = np_fma(5.082762527590693718096e-04f, y, 6.757896990527504603057e-03f);
  n = np_fma(n, y, 5.114512081637298353406e-02f);
  n = np_fma(n, y, 2.473615434895520810817e-01f);
  n = np_fma(n, y, 7.257664613233124478488e-01f);
  n = np_fma(n, y, 9.999999999980870924916e-01f);
  float d = np_fma(2.159509375685829852307e-02f, y, -2.742335390411667452936e-01f);
  d = np_fma(d, y, 1.0f);
  return ldexpf(np_div(n, d), (int)q);                 // one rounding, also into the denormal range
}

// softmax(m) of one pixel's K (<= NP_SOFTMAX_MAX_K) values into p.  The loops run to the constant bound so that the device
// keeps both arrays in registers.
static_assert(NP_SOFTMAX_MAX_K == 8, "np_softmax_pixel restates np.sum for K <= 8 only");
NP_HD void np_softmax_pixel(const float* m, int K, float* p) {
  float s = 0.0f;
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int k = 0; k < NP_SOFTMAX_MAX_K; ++k)
    if (k < K) {
      p[k] = np_expf(m[k]);
      s = k == 0 ? p[k] : np_add(s, p[k]);
    }
  if (K == 8)   // pairwise_sum's unrolled block: eight partial sums (one value each here) combined as a tree
    s = np_add(np_add(np_add(p[0], p[1]), np_add(p[2], p[3])), np_add(np_add(p[4], p[5]), np_add(p[6], p[7])));
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
  for (int k = 0; k < NP_SOFTMAX_MAX_K; ++k)
    if (k < K) p[k] = np_div(p[k], s);
}
