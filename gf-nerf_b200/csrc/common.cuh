// Shared helpers of the gfnerf_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/gfnerf_b200.h"

namespace gf {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

inline int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return GF_ERR_CUDA;
  }
  return GF_OK;
}

#define GF_REQUIRE(cond, ...)      \
  do {                             \
    if (!(cond)) {                 \
      gf::set_error(__VA_ARGS__);  \
      return GF_ERR_INVALID;       \
    }                              \
  } while (0)

#define GF_CUDA(call)                                                   \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) {                                           \
      gf::set_error("%s: %s", #call, cudaGetErrorString(e__));          \
      return GF_ERR_CUDA;                                               \
    }                                                                   \
  } while (0)

// B200: 148 SMs.  Grids of streaming kernels are sized as a multiple of this.
int sm_count();

inline int64_t div_up(int64_t a, int64_t b) { return (a + b - 1) / b; }

// grid for a grid-stride kernel: enough CTAs for `n` items but never more than
// `waves` resident waves of `ctas_per_sm` CTAs on every SM.
inline int stride_grid(int64_t n, int block, int ctas_per_sm, int waves = 1) {
  int64_t need = div_up(n > 0 ? n : 1, block);
  int64_t cap = (int64_t)sm_count() * ctas_per_sm * waves;
  return (int)(need < cap ? need : cap);
}

// Host: the normalised fp32 Gaussian window of S3IM and SSIM, g[x] = exp(-(x - ksize/2)^2 / (2 sigma^2)) / sum, x in
// [0, ksize); the 2-D window is the outer product g[y] * g[x].  The exponent is evaluated in double and rounded once,
// the sum and the division in fp32.
inline void gaussian_window(int ksize, double sigma, float* g) {
  float gs = 0.f;
  for (int x = 0; x < ksize; x++) {
    g[x] = (float)exp(-(double)((x - ksize / 2) * (x - ksize / 2)) / (2.0 * sigma * sigma));
    gs += g[x];
  }
  for (int x = 0; x < ksize; x++) g[x] /= gs;
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

}  // namespace gf
