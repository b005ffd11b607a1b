// Alpha compositing along rays, forward and backward, one warp per ray.
//
// Replaces RaySamples.get_weights_f2nerf (reference nerfstudio/cameras/rays.py:178-200:
// alpha = 1-exp(-delta*sigma), T = exp(-exclusive cumsum), w = alpha*T, nan_to_num) and
// RGBRenderer.combine_rgb / DepthRenderer('expected') / AccumulationRenderer
// (nerfstudio/model_components/renderers.py:97-110, 269-283, 220) and their autograd.
//
// The reference runs ~11 elementwise/scan/reduce kernels over the dense [R,1024,1]
// tensors (padding included) and autograd keeps every intermediate.  Here a warp walks
// the CSR range of its ray in 32-sample chunks: delta*sigma is prefix-summed with
// shuffles (carry kept in a register), the four reductions ride along in the same pass,
// and each sample is read exactly once (28 B) -- HBM-bound streaming work.
#include "common.cuh"

namespace gf {

constexpr int kCompBlock = 256;

__device__ __forceinline__ float nan_to_num(float x) {
  if (isnan(x)) return 0.f;
  if (isinf(x)) return x > 0.f ? 3.4028234663852886e38f : -3.4028234663852886e38f;
  return x;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

__global__ void __launch_bounds__(kCompBlock)
composite_fwd_kernel(int64_t n_rays, const int* __restrict__ offsets, const float* __restrict__ sigma,
                     const float* __restrict__ delta, const float* __restrict__ rgb, const float* __restrict__ t,
                     float* __restrict__ weights, float* __restrict__ alphas, float* __restrict__ trans,
                     float* __restrict__ out_rgb, float* __restrict__ out_depth, float* __restrict__ out_acc,
                     float* __restrict__ d_tmax) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float tmax = 0.f;
  for (int64_t ray = warp0; ray < n_rays; ray += n_warps) {
    const int s0 = __ldg(offsets + ray), s1 = __ldg(offsets + ray + 1);
    float carry = 0.f;  // sum of delta*sigma over the samples before this chunk
    float ar = 0.f, ag = 0.f, ab = 0.f, ad = 0.f, aw = 0.f;
    for (int base = s0; base < s1; base += 32) {
      const int s = base + lane;
      const bool valid = s < s1;
      float dd = 0.f, ts = 0.f, cr = 0.f, cg = 0.f, cb = 0.f;
      if (valid) {
        dd = __fmul_rn(__ldg(delta + s), __ldg(sigma + s));
        if (t) ts = __ldg(t + s);
        if (rgb) {
          cr = __ldg(rgb + 3 * s);
          cg = __ldg(rgb + 3 * s + 1);
          cb = __ldg(rgb + 3 * s + 2);
        }
      }
      float incl = dd;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float y = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += y;
      }
      // exclusive prefix = the previous lane's inclusive sum: incl - dd would lose the earlier samples' sum to
      // ulp(dd) at an opaque sample and turn it into NaN at dd = inf
      const float prev = __shfl_up_sync(0xffffffffu, incl, 1);
      const float excl = carry + (lane > 0 ? prev : 0.f);
      const float alpha = 1.f - expf(-dd);
      const float T = expf(-excl);
      const float w = nan_to_num(alpha * T);
      if (valid) {
        if (weights) weights[s] = w;
        if (alphas) alphas[s] = alpha;
        if (trans) trans[s] = T;
        ar = fmaf(w, cr, ar);
        ag = fmaf(w, cg, ag);
        ab = fmaf(w, cb, ab);
        ad = fmaf(w, ts, ad);
        aw += w;
        tmax = fmaxf(tmax, ts);
      }
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    ar = warp_sum(ar);
    ag = warp_sum(ag);
    ab = warp_sum(ab);
    ad = warp_sum(ad);
    aw = warp_sum(aw);
    if (lane == 0) {
      if (out_rgb) {
        out_rgb[3 * ray] = ar;
        out_rgb[3 * ray + 1] = ag;
        out_rgb[3 * ray + 2] = ab;
      }
      if (out_depth) out_depth[ray] = ad / (aw + 1e-10f);
      if (out_acc) out_acc[ray] = aw;
    }
  }
  if (d_tmax) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, off));
    // t >= 0, so the int ordering of the bit patterns is the float ordering
    if (lane == 0 && tmax > 0.f) atomicMax(reinterpret_cast<int*>(d_tmax), __float_as_int(tmax));
  }
}

// reverse sweep: d_dd_i = gw_i * exp(-dd_i) * T_i - sum_{j>i} gw_j w_j
__global__ void __launch_bounds__(kCompBlock)
composite_bwd_kernel(int64_t n_rays, const int* __restrict__ offsets, const float* __restrict__ sigma,
                     const float* __restrict__ delta, const float* __restrict__ rgb, const float* __restrict__ trans,
                     const float* __restrict__ g_rgb, const float* __restrict__ g_acc,
                     const float* __restrict__ g_w, float* __restrict__ d_sigma, float* __restrict__ d_rgb) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t ray = warp0; ray < n_rays; ray += n_warps) {
    const int s0 = __ldg(offsets + ray), s1 = __ldg(offsets + ray + 1);
    const int cnt = s1 - s0;
    if (cnt <= 0) continue;
    const bool col = g_rgb != nullptr && rgb != nullptr;
    const float gr = col ? __ldg(g_rgb + 3 * ray) : 0.f, gg = col ? __ldg(g_rgb + 3 * ray + 1) : 0.f,
                gb = col ? __ldg(g_rgb + 3 * ray + 2) : 0.f;
    const float ga = g_acc ? __ldg(g_acc + ray) : 0.f;
    float carry = 0.f;  // sum of gw*w over the samples behind this chunk
    for (int base = s0 + ((cnt - 1) / 32) * 32; base >= s0; base -= 32) {
      const int s = base + lane;
      const bool valid = s < s1;
      float dd = 0.f, T = 0.f, cr = 0.f, cg = 0.f, cb = 0.f, dl = 0.f, gws = 0.f;
      if (valid) {
        dl = __ldg(delta + s);
        dd = __fmul_rn(dl, __ldg(sigma + s));
        T = __ldg(trans + s);
        if (col) {
          cr = __ldg(rgb + 3 * s);
          cg = __ldg(rgb + 3 * s + 1);
          cb = __ldg(rgb + 3 * s + 2);
        }
        if (g_w) gws = __ldg(g_w + s);
      }
      const float e = expf(-dd);
      const float w = (1.f - e) * T;
      const float gw = fmaf(gr, cr, fmaf(gg, cg, fmaf(gb, cb, ga))) + gws;
      const float own = valid ? gw * w : 0.f;
      float incl = own;  // inclusive suffix sum within the chunk
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float y = __shfl_down_sync(0xffffffffu, incl, off);
        if (lane + off < 32) incl += y;
      }
      // exclusive suffix = the next lane's inclusive suffix, never incl - own (see the forward)
      const float next = __shfl_down_sync(0xffffffffu, incl, 1);
      const float behind = carry + (lane < 31 ? next : 0.f);
      if (valid) {
        d_sigma[s] = (gw * e * T - behind) * dl;
        if (d_rgb) {
          d_rgb[3 * s] = w * gr;
          d_rgb[3 * s + 1] = w * gg;
          d_rgb[3 * s + 2] = w * gb;
        }
      }
      carry += __shfl_sync(0xffffffffu, incl, 0);
    }
  }
}

// CharbonnierLoss (nerfstudio/model_components/losses.py:73-84), out_norm 'b'
__global__ void charbonnier_kernel(int64_t n3, float inv_rays, const float* __restrict__ rgb,
                                   const float* __restrict__ target, float eps2, float* __restrict__ g_rgb,
                                   float* __restrict__ d_loss) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n3; i += stride) {
    const float d = rgb[i] - target[i];
    const float s = sqrtf(fmaf(d, d, eps2));
    acc += s;
    if (g_rgb) g_rgb[i] = d / s * inv_rays;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0 && d_loss) atomicAdd(d_loss, acc * inv_rays);
}

// S3IM (nerfstudio/model_components/losses.py:713-794): SSIM between two virtual images built from the ray batch
// laid out `repeat` times (index = arange ++ randperm x (repeat-1)), Gaussian window ksize x ksize (sigma 1.5), stride,
// zero padding (ksize-1)/2.  One thread per window (channel, oy, ox): gathers its ksize^2 (src, tar) pairs through the
// index list, adds  -mult/n_map * d ssim/d src  to g_src and  mult * (1 - ssim)/n_map  to the loss.
struct S3imWindow {
  float w[64];
};

__global__ void __launch_bounds__(128)
s3im_kernel(int64_t n_map, int64_t W, int64_t oh, int64_t ow, int patch_h, int ksize, int stride, int pad,
            const long long* __restrict__ index, const float* __restrict__ src, const float* __restrict__ tar,
            S3imWindow win, float mult, float* __restrict__ g_src, float* __restrict__ d_loss) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float part = 0.f;
  if (i < n_map) {
    const int64_t ox = i % ow, oy = (i / ow) % oh;
    const int c = (int)(i / (ow * oh));
    float mu1 = 0.f, mu2 = 0.f, e11 = 0.f, e22 = 0.f, e12 = 0.f;
    for (int ky = 0; ky < ksize; ky++)
      for (int kx = 0; kx < ksize; kx++) {
        const int64_t h = oy * stride - pad + ky, w = ox * stride - pad + kx;
        if (h < 0 || h >= patch_h || w < 0 || w >= W) continue;
        const long long r = __ldg(index + h * W + w);
        const float x = __ldg(src + 3 * r + c), y = __ldg(tar + 3 * r + c), wt = win.w[ky * ksize + kx];
        mu1 = fmaf(wt, x, mu1);
        mu2 = fmaf(wt, y, mu2);
        e11 = fmaf(wt * x, x, e11);
        e22 = fmaf(wt * y, y, e22);
        e12 = fmaf(wt * x, y, e12);
      }
    const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
    const float s11 = e11 - mu1 * mu1, s22 = e22 - mu2 * mu2, s12 = e12 - mu1 * mu2;
    const float A1 = 2.f * mu1 * mu2 + C1, A2 = 2.f * s12 + C2, B1 = mu1 * mu1 + mu2 * mu2 + C1, B2 = s11 + s22 + C2;
    const float inv = 1.f / (B1 * B2);
    const float ssim = A1 * A2 * inv;
    const float inv_n = 1.f / (float)n_map;
    part = mult * (1.f - ssim) * inv_n;
    if (g_src) {
      const float k = -mult * inv_n;
      for (int ky = 0; ky < ksize; ky++)
        for (int kx = 0; kx < ksize; kx++) {
          const int64_t h = oy * stride - pad + ky, w = ox * stride - pad + kx;
          if (h < 0 || h >= patch_h || w < 0 || w >= W) continue;
          const long long r = __ldg(index + h * W + w);
          const float x = __ldg(src + 3 * r + c), y = __ldg(tar + 3 * r + c), wt = win.w[ky * ksize + kx];
          const float dA1 = 2.f * mu2 * wt, dA2 = 2.f * wt * (y - mu2), dB1 = 2.f * mu1 * wt, dB2 = 2.f * wt * (x - mu1);
          const float d = (dA1 * A2 + A1 * dA2) * inv - ssim * (dB1 * B2 + B1 * dB2) * inv;
          atomicAdd(g_src + 3 * r + c, k * d);
        }
    }
  }
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0 && d_loss && part != 0.f) atomicAdd(d_loss, part);
}

}  // namespace gf

using namespace gf;

extern "C" {

int gf_composite_forward(int64_t n_rays, const int32_t* offsets, const float* sigma, const float* delta,
                         const float* rgb, const float* t, float* weights, float* alphas, float* trans,
                         float* out_rgb, float* out_depth, float* out_acc, float* d_tmax, void* stream) {
  GF_REQUIRE(n_rays >= 0, "gf_composite_forward: bad sizes");
  if (n_rays == 0) return GF_OK;
  GF_REQUIRE(offsets && sigma && delta, "gf_composite_forward: null pointer");
  GF_REQUIRE(!out_rgb || rgb, "gf_composite_forward: out_rgb without rgb");
  GF_REQUIRE(!out_depth || t, "gf_composite_forward: out_depth without t");
  const int grid = stride_grid(n_rays * 32, kCompBlock, 8, 2);
  composite_fwd_kernel<<<grid, kCompBlock, 0, (cudaStream_t)stream>>>(n_rays, offsets, sigma, delta, rgb, t, weights,
                                                                      alphas, trans, out_rgb, out_depth, out_acc,
                                                                      d_tmax);
  return check_launch("composite_fwd_kernel");
}

int gf_composite_backward(int64_t n_rays, const int32_t* offsets, const float* sigma, const float* delta,
                          const float* rgb, const float* trans, const float* g_rgb, const float* g_acc,
                          const float* g_w, float* d_sigma, float* d_rgb, void* stream) {
  GF_REQUIRE(n_rays >= 0, "gf_composite_backward: bad sizes");
  if (n_rays == 0) return GF_OK;
  GF_REQUIRE(offsets && sigma && delta && trans && d_sigma, "gf_composite_backward: null pointer");
  GF_REQUIRE(!g_rgb || rgb, "gf_composite_backward: g_rgb without rgb");
  GF_REQUIRE(!d_rgb || (g_rgb && rgb), "gf_composite_backward: d_rgb needs g_rgb and rgb");
  const int grid = stride_grid(n_rays * 32, kCompBlock, 8, 2);
  composite_bwd_kernel<<<grid, kCompBlock, 0, (cudaStream_t)stream>>>(n_rays, offsets, sigma, delta, rgb, trans,
                                                                      g_rgb, g_acc, g_w, d_sigma, d_rgb);
  return check_launch("composite_bwd_kernel");
}

int gf_charbonnier(int64_t n_rays, const float* rgb, const float* target, float eps, float* g_rgb, float* d_loss,
                   void* stream) {
  GF_REQUIRE(n_rays >= 0, "gf_charbonnier: bad sizes");
  if (n_rays == 0) return GF_OK;
  GF_REQUIRE(rgb && target, "gf_charbonnier: null pointer");
  const int64_t n3 = n_rays * 3;
  charbonnier_kernel<<<stride_grid(n3, 256, 4), 256, 0, (cudaStream_t)stream>>>(n3, 1.f / (float)n_rays, rgb, target,
                                                                                eps * eps, g_rgb, d_loss);
  return check_launch("charbonnier_kernel");
}

int gf_s3im(int64_t n_rays, int64_t n_virtual, const int64_t* index, const float* src, const float* target,
            int patch_h, int ksize, int stride, float mult, float* g_src, float* d_loss, void* stream) {
  GF_REQUIRE(n_rays >= 0 && n_virtual >= 0 && patch_h > 0 && stride > 0 && ksize >= 1 && ksize <= 8,
             "gf_s3im: bad sizes");
  GF_REQUIRE(n_virtual % patch_h == 0, "gf_s3im: n_virtual must be a multiple of the patch height");
  if (n_rays == 0 || n_virtual == 0) return GF_OK;
  GF_REQUIRE(index && src && target, "gf_s3im: null pointer");
  const int64_t W = n_virtual / patch_h;
  const int pad = (ksize - 1) / 2;
  // checked before the division, which truncates toward zero: a window one row too tall would still give oh = 1
  GF_REQUIRE(patch_h + 2 * pad >= ksize && W + 2 * pad >= ksize, "gf_s3im: the window does not fit the virtual image");
  const int64_t oh = (patch_h + 2 * pad - ksize) / stride + 1, ow = (W + 2 * pad - ksize) / stride + 1;
  // the reference's window: fp32 Gaussian, sigma 1.5, normalised, outer product (losses.py:726-734)
  S3imWindow win;
  float g1[8];
  gaussian_window(ksize, 1.5, g1);
  for (int y = 0; y < ksize; y++)
    for (int x = 0; x < ksize; x++) win.w[y * ksize + x] = g1[y] * g1[x];
  const int64_t n_map = 3 * oh * ow;
  s3im_kernel<<<(int)div_up(n_map, 128), 128, 0, (cudaStream_t)stream>>>(
      n_map, W, oh, ow, patch_h, ksize, stride, pad, (const long long*)index, src, target, win, mult, g_src, d_loss);
  return check_launch("s3im_kernel");
}

}  // extern "C"
