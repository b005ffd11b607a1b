// Field MLP, per-ray part and C-ABI entry points (sm_100a).
//
// The per-sample layers -- the two MLPNetwork stacks of the reference field (gfnerf/mlp.py:25-57, built at
// gfnerf/nerfacto_field.py:174-179, 217-227), trunc_exp(x + 1) (:499), the sigmoid head and their backward -- run
// on the tcgen05 / TMEM tensor-core kernels of mlp_tc.cu (H = 64) and mlp_tc128.cu (H = 128), which share
// mlp_tc_common.cuh with this file (the parameter blob layout, Blob<H>).  This file holds what is constant along a ray:
//
//  * the head's first layer is split: SH(dir) (tcnn SH degree 4, :152-158, 521) and the appearance embedding
//    (:530-537) are the same for every sample of a ray, so  W2[:, SH|emb] . [SH; emb] + b2  is evaluated once per
//    RAY in fp32 (ray_bias_kernel) and enters the per-sample layer as a bias row; only the 15 geo features go
//    through the per-sample MMA (K = 16 instead of 63).  The reference recomputes SH and gathers the embedding
//    for all 1024 slots of every ray;
//  * ray_bias_bwd_kernel turns d(ray_bias) back into the gradients of those W2 columns, b2 and the embedding.
//
// (Round 1 first shipped register-chained mma.sync.m16n8k16 kernels here: forward 0.73 ms, backward 2.54 ms on the
// bench workload; the tcgen05 kernels that replaced them run 0.37 ms / 1.63 ms -- profiles/.)
#include <stdlib.h>

#include "mlp_tc_common.cuh"

namespace gf {

// ---------------------------------------------------------------------------------------------
// per-ray part of the head's first layer
// ---------------------------------------------------------------------------------------------
// tcnn SphericalHarmonics degree 4 on (dir+1)/2, fp16 output (gfnerf/nerfacto_field.py:64-70, 152-158, 521)
__device__ __forceinline__ void sh4(float dx, float dy, float dz, float (&o)[16]) {
  const float x = ((dx + 1.f) * .5f) * 2.f - 1.f, y = ((dy + 1.f) * .5f) * 2.f - 1.f, z = ((dz + 1.f) * .5f) * 2.f - 1.f;
  const float xy = x * y, xz = x * z, yz = y * z, x2 = x * x, y2 = y * y, z2 = z * z;
  o[0] = 0.28209479177387814f;
  o[1] = -0.48860251190291987f * y;
  o[2] = 0.48860251190291987f * z;
  o[3] = -0.48860251190291987f * x;
  o[4] = 1.0925484305920792f * xy;
  o[5] = -1.0925484305920792f * yz;
  o[6] = 0.94617469575755997f * z2 - 0.31539156525251999f;
  o[7] = -1.0925484305920792f * xz;
  o[8] = 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
  o[9] = 0.59004358992664352f * y * (-3.0f * x2 + y2);
  o[10] = 2.8906114426405538f * xy * z;
  o[11] = 0.45704579946446572f * y * (1.0f - 5.0f * z2);
  o[12] = 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
  o[13] = 0.45704579946446572f * x * (1.0f - 5.0f * z2);
  o[14] = 1.4453057213202769f * z * (x2 - y2);
  o[15] = 0.59004358992664352f * x * (-x2 + 3.0f * y2);
#pragma unroll
  for (int i = 0; i < 16; i++) o[i] = __half2float(__float2half_rn(o[i]));
}

constexpr int kRbRays = 32;  // rays per CTA of the ray-bias kernels
constexpr int kRbIn = 48;    // SH(16) | emb(32)

// ray_bias[r][j] = b2[j] + W2[j][0:16] . SH(dir_r) + W2[j][31:63] . emb_r      (fp32)
template <int kH>
__global__ void __launch_bounds__(256)
ray_bias_kernel(int64_t n_rays, const float* __restrict__ params, const float* __restrict__ dirs,
                const float* __restrict__ emb, float* __restrict__ ray_bias) {
  constexpr int kW2 = Blob<kH>::kW2, kB2 = Blob<kH>::kB2;
  __shared__ float s_w[kH][kRbIn + 1];
  __shared__ float s_in[kRbRays][kRbIn + 1];
  for (int i = threadIdx.x; i < kH * kRbIn; i += blockDim.x) {
    const int j = i / kRbIn, k = i % kRbIn;
    s_w[j][k] = __ldg(params + kW2 + j * 63 + (k < 16 ? k : 15 + k));
  }
  const int64_t r0 = (int64_t)blockIdx.x * kRbRays;
  if (threadIdx.x < kRbRays) {
    const int64_t r = r0 + threadIdx.x;
    float o[16];
    if (r < n_rays) sh4(__ldg(dirs + 3 * r), __ldg(dirs + 3 * r + 1), __ldg(dirs + 3 * r + 2), o);
    else
      for (int i = 0; i < 16; i++) o[i] = 0.f;
    for (int i = 0; i < 16; i++) s_in[threadIdx.x][i] = o[i];
  }
  for (int i = threadIdx.x; i < kRbRays * 32; i += blockDim.x) {
    const int rr = i >> 5, k = i & 31;
    const int64_t r = r0 + rr;
    s_in[rr][16 + k] = (emb && r < n_rays) ? __ldg(emb + r * 32 + k) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kRbRays * kH; i += blockDim.x) {
    const int rr = i / kH, j = i % kH;
    const int64_t r = r0 + rr;
    if (r >= n_rays) continue;
    float acc = __ldg(params + kB2 + j);
#pragma unroll 8
    for (int k = 0; k < kRbIn; k++) acc = fmaf(s_w[j][k], s_in[rr][k], acc);
    ray_bias[r * kH + j] = acc;
  }
}

// G = d_ray_bias [R,64]:  d_b2 += sum_r G ; d_W2[:, SH|emb] += G^T [SH|emb] ; d_emb = G W2[:, emb]
template <int kH>
__global__ void __launch_bounds__(256)
ray_bias_bwd_kernel(int64_t n_rays, const float* __restrict__ params, const float* __restrict__ dirs,
                    const float* __restrict__ emb, const float* __restrict__ g_rb, float* __restrict__ d_params,
                    float* __restrict__ d_emb) {
  constexpr int kW2 = Blob<kH>::kW2, kB2 = Blob<kH>::kB2;
  __shared__ float s_g[kRbRays][kH + 1];
  __shared__ float s_in[kRbRays][kRbIn + 1];
  const int64_t r0 = (int64_t)blockIdx.x * kRbRays;
  if (threadIdx.x < kRbRays) {
    const int64_t r = r0 + threadIdx.x;
    float o[16];
    if (r < n_rays) sh4(__ldg(dirs + 3 * r), __ldg(dirs + 3 * r + 1), __ldg(dirs + 3 * r + 2), o);
    else
      for (int i = 0; i < 16; i++) o[i] = 0.f;
    for (int i = 0; i < 16; i++) s_in[threadIdx.x][i] = o[i];
  }
  for (int i = threadIdx.x; i < kRbRays * 32; i += blockDim.x) {
    const int rr = i >> 5, k = i & 31;
    const int64_t r = r0 + rr;
    s_in[rr][16 + k] = (emb && r < n_rays) ? __ldg(emb + r * 32 + k) : 0.f;
  }
  for (int i = threadIdx.x; i < kRbRays * kH; i += blockDim.x) {
    const int rr = i / kH, j = i % kH;
    const int64_t r = r0 + rr;
    s_g[rr][j] = r < n_rays ? __ldg(g_rb + r * kH + j) : 0.f;
  }
  __syncthreads();
  if (d_params) {
    // (j, k) outputs: k < 48 weight columns, k == 48 the bias
    for (int i = threadIdx.x; i < kH * (kRbIn + 1); i += blockDim.x) {
      const int j = i / (kRbIn + 1), k = i % (kRbIn + 1);
      float acc = 0.f;
      if (k < kRbIn) {
#pragma unroll 8
        for (int rr = 0; rr < kRbRays; rr++) acc = fmaf(s_g[rr][j], s_in[rr][k], acc);
        if (k >= 16 && !emb) continue;
        if (acc != 0.f) atomicAdd(d_params + kW2 + j * 63 + (k < 16 ? k : 15 + k), acc);
      } else {
#pragma unroll 8
        for (int rr = 0; rr < kRbRays; rr++) acc += s_g[rr][j];
        if (acc != 0.f) atomicAdd(d_params + kB2 + j, acc);
      }
    }
  }
  if (d_emb) {
    for (int i = threadIdx.x; i < kRbRays * 32; i += blockDim.x) {
      const int rr = i >> 5, k = i & 31;
      const int64_t r = r0 + rr;
      if (r >= n_rays) continue;
      float acc = 0.f;
#pragma unroll 8
      for (int j = 0; j < kH; j++) acc = fmaf(s_g[rr][j], __ldg(params + kW2 + j * 63 + 31 + k), acc);
      d_emb[r * 32 + k] += acc;
    }
  }
}

}  // namespace gf

using namespace gf;

int gf_launch_mlp_fwd_tc(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                         const int32_t* ray_id, const float* ray_bias, float* sigma, float* rgb, void* relu_masks,
                         cudaStream_t st);
int gf_launch_mlp_bwd_tc(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                         const int32_t* ray_id, const float* ray_bias, const void* relu_masks, const float* d_sigma,
                         const float* d_rgb, void* d_feat, float* d_params, float* d_ray_bias, float gscale,
                         cudaStream_t st);
// hidden width 128 (mlp_tc128.cu)
int gf_launch_mlp_fwd_tc128(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                            const int32_t* ray_id, const float* ray_bias, float* sigma, float* rgb, void* relu_masks,
                            cudaStream_t st);
int gf_launch_mlp_bwd_tc128(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                            const int32_t* ray_id, const float* ray_bias, const void* relu_masks, const float* d_sigma,
                            const float* d_rgb, void* d_feat, float* d_params, float* d_ray_bias, float gscale,
                            cudaStream_t st);

static inline bool width_built(int hidden) { return hidden == 64 || hidden == 128; }

extern "C" {

int64_t gf_mlp_param_count(int hidden) {
  return hidden == 64 ? (int64_t)Blob<64>::kParamCount : hidden == 128 ? (int64_t)Blob<128>::kParamCount : -1;
}

int gf_mlp_mask_words(int hidden) { return hidden == 64 ? 8 : hidden == 128 ? 16 : -1; }

int gf_mlp_ray_bias(int64_t n_rays, int hidden, const float* params, const float* ray_dirs, const float* ray_emb,
                    float* ray_bias, void* stream) {
  GF_REQUIRE(width_built(hidden), "gf_mlp_ray_bias: hidden width %d is not built (64 and 128 are)", hidden);
  GF_REQUIRE(n_rays >= 0, "gf_mlp_ray_bias: bad sizes");
  if (n_rays == 0) return GF_OK;
  GF_REQUIRE(params && ray_dirs && ray_bias, "gf_mlp_ray_bias: null pointer");
  const int grid = (int)div_up(n_rays, kRbRays);
  if (hidden == 64)
    ray_bias_kernel<64><<<grid, 256, 0, (cudaStream_t)stream>>>(n_rays, params, ray_dirs, ray_emb, ray_bias);
  else
    ray_bias_kernel<128><<<grid, 256, 0, (cudaStream_t)stream>>>(n_rays, params, ray_dirs, ray_emb, ray_bias);
  return check_launch("ray_bias_kernel");
}

int gf_mlp_ray_bias_backward(int64_t n_rays, int hidden, const float* params, const float* ray_dirs,
                             const float* ray_emb, const float* d_ray_bias, float* d_params, float* d_ray_emb,
                             void* stream) {
  GF_REQUIRE(width_built(hidden), "gf_mlp_ray_bias_backward: hidden width %d is not built (64 and 128 are)", hidden);
  GF_REQUIRE(n_rays >= 0, "gf_mlp_ray_bias_backward: bad sizes");
  if (n_rays == 0) return GF_OK;
  GF_REQUIRE(params && ray_dirs && d_ray_bias, "gf_mlp_ray_bias_backward: null pointer");
  GF_REQUIRE(!d_ray_emb || ray_emb, "gf_mlp_ray_bias_backward: d_ray_emb without ray_emb");
  const int grid = (int)div_up(n_rays, kRbRays);
  if (hidden == 64)
    ray_bias_bwd_kernel<64><<<grid, 256, 0, (cudaStream_t)stream>>>(n_rays, params, ray_dirs, ray_emb, d_ray_bias,
                                                                    d_params, d_ray_emb);
  else
    ray_bias_bwd_kernel<128><<<grid, 256, 0, (cudaStream_t)stream>>>(n_rays, params, ray_dirs, ray_emb, d_ray_bias,
                                                                     d_params, d_ray_emb);
  return check_launch("ray_bias_bwd_kernel");
}

int gf_mlp_forward(int64_t n, const int32_t* d_n_ptr, int hidden, const float* params, const void* feat_f16,
                   const int32_t* ray_id, const float* ray_bias, float* sigma, float* rgb, void* relu_masks,
                   void* stream) {
  GF_REQUIRE(width_built(hidden), "gf_mlp_forward: hidden width %d is not built (64 and 128 are)", hidden);
  GF_REQUIRE(n >= 0, "gf_mlp_forward: bad sizes");
  if (n == 0) return GF_OK;
  GF_REQUIRE(params && feat_f16 && ray_id && ray_bias && sigma && rgb, "gf_mlp_forward: null pointer");
  GF_REQUIRE((reinterpret_cast<uintptr_t>(relu_masks) & 15) == 0, "gf_mlp_forward: relu_masks must be 16-byte aligned");
  GF_REQUIRE((reinterpret_cast<uintptr_t>(ray_bias) & 15) == 0 && (reinterpret_cast<uintptr_t>(feat_f16) & 15) == 0,
             "gf_mlp_forward: ray_bias and feat must be 16-byte aligned");
  return (hidden == 64 ? gf_launch_mlp_fwd_tc : gf_launch_mlp_fwd_tc128)(n, d_n_ptr, params, feat_f16, ray_id, ray_bias,
                                                                         sigma, rgb, relu_masks, (cudaStream_t)stream);
}

int gf_mlp_backward(int64_t n, const int32_t* d_n_ptr, int hidden, const float* params, const void* feat_f16,
                    const int32_t* ray_id, const float* ray_bias, const void* relu_masks, const float* d_sigma,
                    const float* d_rgb,
                    void* d_feat_scaled_f16, float* d_params, float* d_ray_bias, float grad_scale, void* stream) {
  GF_REQUIRE(width_built(hidden), "gf_mlp_backward: hidden width %d is not built (64 and 128 are)", hidden);
  GF_REQUIRE(n >= 0 && grad_scale > 0.f, "gf_mlp_backward: bad sizes");
  if (n == 0) return GF_OK;
  GF_REQUIRE(params && feat_f16 && ray_id && ray_bias && relu_masks && d_sigma && d_rgb && d_feat_scaled_f16,
             "gf_mlp_backward: null pointer");
  GF_REQUIRE((reinterpret_cast<uintptr_t>(relu_masks) & 15) == 0, "gf_mlp_backward: relu_masks must be 16-byte aligned");
  GF_REQUIRE((d_params == nullptr) == (d_ray_bias == nullptr),
             "gf_mlp_backward: d_params and d_ray_bias go together (both NULL = frozen MLP)");
  return (hidden == 64 ? gf_launch_mlp_bwd_tc : gf_launch_mlp_bwd_tc128)(
      n, d_n_ptr, params, feat_f16, ray_id, ray_bias, relu_masks, d_sigma, d_rgb, d_feat_scaled_f16, d_params, d_ray_bias,
      grad_scale, (cudaStream_t)stream);
}

}  // extern "C"
