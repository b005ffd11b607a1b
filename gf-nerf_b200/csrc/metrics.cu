// Image-quality metrics of rendered views: per-image MSE, PSNR and SSIM with the conventions of nerfstudio's nerfacto
// evaluation (torchmetrics' PeakSignalNoiseRatio(data_range=1.0) and structural_similarity_index_measure with its
// defaults; restated in include/gfnerf_b200.h).  Four launches, no host sync, no allocation:
//   stats     one CTA per (image, chunk of kStatsChunk floats): min / max of both images, SSE in double
//   range     one CTA per image: the data range L and C1, C2 from the chunk results
//   ssim      one CTA per (image, 32 x 32 output tile): separable 11-tap moments in shared memory, SSIM per pixel and
//             channel, one double partial per tile
//   finalize  one CTA per image: psnr, ssim, mse
// The partition depends only on (B, H, W) and every sum runs in a fixed order, so results are bit-identical from run
// to run and an image gives the same bits alone or inside a batch.
#include <float.h>

#include "common.cuh"

namespace gf {
namespace {

constexpr int kStatsThreads = 256;
constexpr int64_t kStatsChunk = 16384;               // floats of one image per stats CTA (a multiple of 4)
constexpr int kWin = 11, kHalo = kWin - 1;
constexpr int kTileW = 32, kTileH = 32;              // output pixels per SSIM CTA
constexpr int kInRows = kTileH + kHalo;              // input rows staged per tile
constexpr int kBlocksPerRow = (3 * (kTileW + kHalo) + 3 + 3) / 4;   // 16-byte blocks covering a misaligned row segment
constexpr int kRowFloats = 4 * kBlocksPerRow;
constexpr int kSsimThreads = 256;
constexpr int kSsimWarps = kSsimThreads / 32;
constexpr int kRowsPerThread = kTileH / kSsimWarps;  // output rows per thread in the vertical pass
constexpr int kSmemIn = 2 * kInRows * kRowFloats * 4;
constexpr int kSmemH = 5 * kInRows * kTileW * 4;
constexpr int kSmemSsim = kSmemIn + kSmemH + kInRows * 4;
static_assert(kTileW == 32, "one lane per output column");
static_assert(kTileH % kSsimWarps == 0, "whole output rows per warp");

struct ChunkStats {
  float pmin, pmax, gmin, gmax;
  double sse;
  double unused;
};
struct ImageConsts {
  float c1, c2, range, unused;
};
struct SsimWindow {
  float w[kWin];
};

__device__ __forceinline__ double warp_sum_f64(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Sum over the CTA in a fixed order (butterfly in each warp, then warp results in index order); valid in thread 0.
template <int kWarps>
__device__ __forceinline__ double cta_sum_f64(double v, double* s_red) {
  v = warp_sum_f64(v);
  if (lane_id() == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kWarps; w++) t += s_red[w];
  return t;
}

// ---- stats ---------------------------------------------------------------------------------------------------------
// Elements [s, e) of both images; pred and gt are 16-byte aligned, so float index i is aligned iff i % 4 == 0.
__global__ void __launch_bounds__(kStatsThreads)
metrics_stats_kernel(int64_t n_img, int64_t n_chunks, const float* __restrict__ pred, const float* __restrict__ gt,
                     ChunkStats* __restrict__ out) {
  __shared__ float s_mm[4][kStatsThreads / 32];
  __shared__ double s_red[kStatsThreads / 32];
  const int64_t b = blockIdx.y, k = blockIdx.x;
  const int64_t s = b * n_img + k * kStatsChunk;
  const int64_t e = b * n_img + min(n_img, (k + 1) * kStatsChunk);
  const int64_t a4 = min((s + 3) & ~(int64_t)3, e), e4 = max(e & ~(int64_t)3, a4);
  float pmin = FLT_MAX, pmax = -FLT_MAX, gmin = FLT_MAX, gmax = -FLT_MAX;
  double sse = 0.0;
  auto visit = [&](float p, float g) {
    pmin = fminf(pmin, p), pmax = fmaxf(pmax, p), gmin = fminf(gmin, g), gmax = fmaxf(gmax, g);
    const double d = (double)p - (double)g;            // exact: the difference of two floats fits a double
    sse = fma(d, d, sse);
  };
  const float4* p4 = reinterpret_cast<const float4*>(pred);
  const float4* g4 = reinterpret_cast<const float4*>(gt);
  for (int64_t q = a4 / 4 + threadIdx.x; q < e4 / 4; q += kStatsThreads) {
    const float4 p = __ldg(p4 + q), g = __ldg(g4 + q);
    visit(p.x, g.x), visit(p.y, g.y), visit(p.z, g.z), visit(p.w, g.w);
  }
  if (threadIdx.x < 3) {                                // up to 3 floats before the first / after the last block
    const int64_t h = s + threadIdx.x, t = e4 + threadIdx.x;
    if (h < a4) visit(__ldg(pred + h), __ldg(gt + h));
    if (t < e) visit(__ldg(pred + t), __ldg(gt + t));
  }
  pmin = warp_min(pmin), pmax = warp_max(pmax), gmin = warp_min(gmin), gmax = warp_max(gmax);
  const int w = threadIdx.x >> 5;
  if (lane_id() == 0) s_mm[0][w] = pmin, s_mm[1][w] = pmax, s_mm[2][w] = gmin, s_mm[3][w] = gmax;
  sse = cta_sum_f64<kStatsThreads / 32>(sse, s_red);    // (its __syncthreads also publishes s_mm)
  if (threadIdx.x == 0) {
    ChunkStats c{FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX, sse, 0.0};
    for (int i = 0; i < kStatsThreads / 32; i++) {
      c.pmin = fminf(c.pmin, s_mm[0][i]), c.pmax = fmaxf(c.pmax, s_mm[1][i]);
      c.gmin = fminf(c.gmin, s_mm[2][i]), c.gmax = fmaxf(c.gmax, s_mm[3][i]);
    }
    out[b * n_chunks + k] = c;
  }
}

// ---- range: L = max(max p - min p, max g - min g), C1 = (0.01 L)^2, C2 = (0.03 L)^2 in fp32, as torchmetrics --------
__global__ void __launch_bounds__(256)
metrics_range_kernel(int64_t n_chunks, const ChunkStats* __restrict__ stats, ImageConsts* __restrict__ consts) {
  __shared__ float s_mm[4][8];
  const int64_t b = blockIdx.x;
  float pmin = FLT_MAX, pmax = -FLT_MAX, gmin = FLT_MAX, gmax = -FLT_MAX;
  for (int64_t k = threadIdx.x; k < n_chunks; k += 256) {
    const ChunkStats c = stats[b * n_chunks + k];
    pmin = fminf(pmin, c.pmin), pmax = fmaxf(pmax, c.pmax), gmin = fminf(gmin, c.gmin), gmax = fmaxf(gmax, c.gmax);
  }
  pmin = warp_min(pmin), pmax = warp_max(pmax), gmin = warp_min(gmin), gmax = warp_max(gmax);
  const int w = threadIdx.x >> 5;
  if (lane_id() == 0) s_mm[0][w] = pmin, s_mm[1][w] = pmax, s_mm[2][w] = gmin, s_mm[3][w] = gmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; i++) {
      s_mm[0][0] = fminf(s_mm[0][0], s_mm[0][i]), s_mm[1][0] = fmaxf(s_mm[1][0], s_mm[1][i]);
      s_mm[2][0] = fminf(s_mm[2][0], s_mm[2][i]), s_mm[3][0] = fmaxf(s_mm[3][0], s_mm[3][i]);
    }
    const float L = fmaxf(s_mm[1][0] - s_mm[0][0], s_mm[3][0] - s_mm[2][0]);
    const float a = 0.01f * L, c = 0.03f * L;
    consts[b] = ImageConsts{a * a, c * c, L, 0.f};
  }
}

// ---- SSIM over one 32 x 32 tile of the (H - 10) x (W - 10) valid-window region ---------------------------------------
// Output (oy, ox) is the window over input rows oy .. oy + 10 and columns ox .. ox + 10.  The tile's input, 42 rows of
// 42 interleaved RGB pixels of both images, is staged with 16-byte loads: a row segment starts at any float offset, so
// it is stored from its enclosing 16-byte block on (offset s_off[r] into the shared row), and the partial blocks at
// its two ends are loaded element by element, so nothing outside the segment is read.
// The moments are taken of p - p0 and g - g0, where p0, g0 are the tile's centre pixel (per channel): variances and
// the covariance do not change under a shift, E[x^2] - mu^2 cancels far less, and a constant region gives exactly 0.
__global__ void __launch_bounds__(kSsimThreads)
metrics_ssim_kernel(int64_t H, int64_t W, int64_t tiles_x, int64_t n_tiles, const float* __restrict__ pred,
                    const float* __restrict__ gt, const ImageConsts* __restrict__ consts, SsimWindow win,
                    double* __restrict__ partial) {
  extern __shared__ __align__(16) unsigned char smem[];
  float* s_in = reinterpret_cast<float*>(smem);                          // [2][kInRows][kRowFloats]
  float* s_h = reinterpret_cast<float*>(smem + kSmemIn);                 // [5][kInRows][kTileW]
  int* s_off = reinterpret_cast<int*>(smem + kSmemIn + kSmemH);          // [kInRows]
  __shared__ double s_red[kSsimWarps];
  const int64_t b = blockIdx.y, tile = blockIdx.x;
  const int64_t y0 = (tile / tiles_x) * kTileH, x0 = (tile % tiles_x) * kTileW;
  const int n_rows = (int)min((int64_t)kInRows, H - y0), n_cols = (int)min((int64_t)(kTileW + kHalo), W - x0);
  const int out_rows = n_rows - kHalo, out_cols = n_cols - kHalo;
  const ImageConsts cst = consts[b];

  // stage: item = (tensor, row, 16-byte block); consecutive threads take consecutive blocks of a row
  for (int i = threadIdx.x; i < 2 * kInRows * kBlocksPerRow; i += kSsimThreads) {
    const int q = i % kBlocksPerRow, r = (i / kBlocksPerRow) % kInRows, m = i / (kBlocksPerRow * kInRows);
    if (r >= n_rows) continue;
    const float* src = m ? gt : pred;
    const int64_t s = ((b * H + y0 + r) * W + x0) * 3, e = s + 3 * n_cols;
    const int off = (int)(s & 3);
    if (m == 0 && q == 0) s_off[r] = off;
    const int64_t f = s - off + 4 * q;                                   // first float of this block
    if (f >= e) continue;
    float* dst = s_in + (m * kInRows + r) * kRowFloats + 4 * q;
    if (f >= s && f + 4 <= e) {
      *reinterpret_cast<float4*>(dst) = __ldg(reinterpret_cast<const float4*>(src + f));
    } else {
      for (int j = 0; j < 4; j++)
        if (f + j >= s && f + j < e) dst[j] = __ldg(src + f + j);
    }
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = lane_id();
  const int rc = (n_rows - 1) / 2, cc = (n_cols - 1) / 2;
  float acc = 0.f;
  for (int c = 0; c < 3; c++) {
    const float p0 = s_in[rc * kRowFloats + s_off[rc] + 3 * cc + c];
    const float g0 = s_in[(kInRows + rc) * kRowFloats + s_off[rc] + 3 * cc + c];
    // horizontal: five 11-tap moments per (input row, output column)
    if (lane < out_cols) {
      for (int r = warp; r < n_rows; r += kSsimWarps) {
        const float* rp = s_in + r * kRowFloats + s_off[r] + 3 * lane + c;
        const float* rg = rp + kInRows * kRowFloats;
        float mp = 0.f, mg = 0.f, epp = 0.f, egg = 0.f, epg = 0.f;
#pragma unroll
        for (int t = 0; t < kWin; t++) {
          const float p = rp[3 * t] - p0, g = rg[3 * t] - g0, w = win.w[t];
          mp = fmaf(w, p, mp);
          mg = fmaf(w, g, mg);
          const float wp = w * p, wg = w * g;
          epp = fmaf(wp, p, epp);
          epg = fmaf(wp, g, epg);
          egg = fmaf(wg, g, egg);
        }
        float* h = s_h + r * kTileW + lane;
        h[0] = mp, h[kInRows * kTileW] = mg, h[2 * kInRows * kTileW] = epp, h[3 * kInRows * kTileW] = egg,
        h[4 * kInRows * kTileW] = epg;
      }
    }
    __syncthreads();
    // vertical: kRowsPerThread consecutive output rows per thread share their input rows
    const int i0 = warp * kRowsPerThread;
    if (lane < out_cols && i0 < out_rows) {
      float a[kRowsPerThread][5];
#pragma unroll
      for (int j = 0; j < kRowsPerThread; j++)
#pragma unroll
        for (int m = 0; m < 5; m++) a[j][m] = 0.f;
#pragma unroll
      for (int k = 0; k < kRowsPerThread + kHalo; k++) {
        float v[5];
        const int r = min(i0 + k, n_rows - 1);       // rows past the image feed only outputs that are dropped
#pragma unroll
        for (int m = 0; m < 5; m++) v[m] = s_h[(m * kInRows + r) * kTileW + lane];
#pragma unroll
        for (int j = 0; j < kRowsPerThread; j++) {
          if (k - j < 0 || k - j >= kWin) continue;
#pragma unroll
          for (int m = 0; m < 5; m++) a[j][m] = fmaf(win.w[k - j], v[m], a[j][m]);
        }
      }
#pragma unroll
      for (int j = 0; j < kRowsPerThread; j++) {
        if (i0 + j >= out_rows) continue;
        const float dp = a[j][0], dg = a[j][1];
        const float spp = a[j][2] - dp * dp, sgg = a[j][3] - dg * dg, spg = a[j][4] - dp * dg;
        const float mu_p = p0 + dp, mu_g = g0 + dg;
        const float num = (2.f * mu_p * mu_g + cst.c1) * (2.f * spg + cst.c2);
        const float den = (mu_p * mu_p + mu_g * mu_g + cst.c1) * (spp + sgg + cst.c2);
        acc += num / den;
      }
    }
    __syncthreads();
  }
  const double t = cta_sum_f64<kSsimWarps>((double)acc, s_red);
  if (threadIdx.x == 0) partial[b * n_tiles + tile] = t;
}

// ---- finalize: one CTA per image -----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
metrics_finalize_kernel(int64_t n_chunks, int64_t n_tiles, double n_px3, double n_win3,
                        const ChunkStats* __restrict__ stats, const double* __restrict__ partial,
                        float* __restrict__ psnr, float* __restrict__ ssim, float* __restrict__ mse) {
  __shared__ double s_red[8];
  const int64_t b = blockIdx.x;
  double sse = 0.0, ss = 0.0;
  for (int64_t k = threadIdx.x; k < n_chunks; k += 256) sse += stats[b * n_chunks + k].sse;
  for (int64_t k = threadIdx.x; k < n_tiles; k += 256) ss += partial[b * n_tiles + k];
  sse = cta_sum_f64<8>(sse, s_red);
  __syncthreads();                                       // s_red is reused
  ss = cta_sum_f64<8>(ss, s_red);
  if (threadIdx.x == 0) {
    const double m = sse / n_px3;
    mse[b] = (float)m;
    psnr[b] = (float)(10.0 * log10(1.0 / m));            // m == 0: +inf, as torchmetrics
    ssim[b] = (float)(ss / n_win3);
  }
}

struct Layout {
  int64_t n_chunks, tiles_x, n_tiles, off_consts, off_partial, bytes;
};

inline int64_t align256(int64_t x) { return (x + 255) & ~(int64_t)255; }

Layout layout(int64_t B, int64_t H, int64_t W) {
  Layout l;
  l.n_chunks = div_up(3 * H * W, kStatsChunk);
  l.tiles_x = div_up(W - kHalo, kTileW);
  l.n_tiles = l.tiles_x * div_up(H - kHalo, kTileH);
  l.off_consts = align256(B * l.n_chunks * (int64_t)sizeof(ChunkStats));
  l.off_partial = l.off_consts + align256(B * (int64_t)sizeof(ImageConsts));
  l.bytes = l.off_partial + align256(B * l.n_tiles * (int64_t)sizeof(double));
  return l;
}

int set_ssim_smem() {
  static std::atomic<bool> done_dev[64];
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  const bool track = dev >= 0 && dev < 64;
  if (!track || !done_dev[dev].load(std::memory_order_acquire)) {
    GF_CUDA(cudaFuncSetAttribute(metrics_ssim_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemSsim));
    if (track) done_dev[dev].store(true, std::memory_order_release);
  }
  return GF_OK;
}

}  // namespace
}  // namespace gf

using namespace gf;

extern "C" {

int64_t gf_image_metrics_scratch_bytes(int64_t n_images, int64_t height, int64_t width) {
  if (n_images < 1 || height < kWin || width < kWin) return -1;
  return layout(n_images, height, width).bytes;
}

int gf_image_metrics(int64_t n_images, int64_t height, int64_t width, const float* pred, const float* gt, float* psnr,
                     float* ssim, float* mse, void* scratch, int64_t scratch_bytes, void* stream) {
  GF_REQUIRE(n_images >= 1 && n_images <= 65535, "gf_image_metrics: n_images must be in [1, 65535], got %lld",
             (long long)n_images);
  GF_REQUIRE(height >= kWin && width >= kWin,
             "gf_image_metrics: images must be at least 11 x 11 (the SSIM window), got %lld x %lld",
             (long long)height, (long long)width);
  GF_REQUIRE(height <= (1 << 20) && width <= (1 << 20), "gf_image_metrics: image too large");
  GF_REQUIRE(pred && gt && psnr && ssim && mse && scratch, "gf_image_metrics: null pointer");
  GF_REQUIRE(((uintptr_t)pred | (uintptr_t)gt) % 16 == 0, "gf_image_metrics: pred and gt must be 16-byte aligned");
  GF_REQUIRE((uintptr_t)scratch % 16 == 0, "gf_image_metrics: scratch must be 16-byte aligned");
  const Layout l = layout(n_images, height, width);
  GF_REQUIRE(scratch_bytes >= l.bytes, "gf_image_metrics: scratch has %lld bytes, needs %lld",
             (long long)scratch_bytes, (long long)l.bytes);
  GF_REQUIRE(l.n_chunks < INT32_MAX && l.n_tiles < INT32_MAX, "gf_image_metrics: image too large");
  int rc = set_ssim_smem();
  if (rc) return rc;
  ChunkStats* stats = reinterpret_cast<ChunkStats*>(scratch);
  ImageConsts* consts = reinterpret_cast<ImageConsts*>((char*)scratch + l.off_consts);
  double* partial = reinterpret_cast<double*>((char*)scratch + l.off_partial);
  const cudaStream_t s = (cudaStream_t)stream;
  const dim3 g_stats((unsigned)l.n_chunks, (unsigned)n_images), g_ssim((unsigned)l.n_tiles, (unsigned)n_images);
  metrics_stats_kernel<<<g_stats, kStatsThreads, 0, s>>>(3 * height * width, l.n_chunks, pred, gt, stats);
  if ((rc = check_launch("metrics_stats_kernel"))) return rc;
  metrics_range_kernel<<<(unsigned)n_images, 256, 0, s>>>(l.n_chunks, stats, consts);
  if ((rc = check_launch("metrics_range_kernel"))) return rc;
  SsimWindow win;
  gaussian_window(kWin, 1.5, win.w);
  metrics_ssim_kernel<<<g_ssim, kSsimThreads, kSmemSsim, s>>>(height, width, l.tiles_x, l.n_tiles, pred, gt, consts,
                                                               win, partial);
  if ((rc = check_launch("metrics_ssim_kernel"))) return rc;
  metrics_finalize_kernel<<<(unsigned)n_images, 256, 0, s>>>(
      l.n_chunks, l.n_tiles, 3.0 * (double)height * (double)width,
      3.0 * (double)(height - kHalo) * (double)(width - kHalo), stats, partial, psnr, ssim, mse);
  return check_launch("metrics_finalize_kernel");
}

}  // extern "C"
