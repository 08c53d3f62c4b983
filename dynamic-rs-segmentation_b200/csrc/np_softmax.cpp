// The multi-scale softmax of the scene pass (np_softmax.h) compiled for the host, so that CPU tests can pin the device's
// arithmetic against NumPy without a GPU.  Built without FMA contraction and without fast-math (build.py HOST_FLAGS).
#include <stdint.h>
#include <stdio.h>

#include "../../include/drs.h"
#include "np_softmax.h"

extern thread_local char g_drs_err[1024];

extern "C" int drs_debug_np_softmax(const float* in_host, int64_t n_pixels, int32_t K, float* out_host) {
  if (!in_host || !out_host || n_pixels < 0 || K < 1 || K > NP_SOFTMAX_MAX_K) {
    snprintf(g_drs_err, sizeof(g_drs_err), "debug_np_softmax: bad argument (n_pixels=%lld, K=%d, at most %d classes)",
             (long long)n_pixels, K, NP_SOFTMAX_MAX_K);
    return 1;
  }
  for (int64_t i = 0; i < n_pixels; ++i) np_softmax_pixel(in_host + i * K, K, out_host + i * K);
  return 0;
}

extern "C" int drs_debug_np_expf(const float* in_host, int64_t n, float* out_host) {
  if (!in_host || !out_host || n < 0) {
    snprintf(g_drs_err, sizeof(g_drs_err), "debug_np_expf: bad argument (n=%lld)", (long long)n);
    return 1;
  }
  for (int64_t i = 0; i < n; ++i) out_host[i] = np_expf(in_host[i]);
  return 0;
}
