// Fused field MLP, hidden width 128 (the width the reference's shipped gf-nerf config uses: gfnerf/config.py:124-125
// hidden_dim = hidden_dim_color = 128), on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a: forward
// (plain fp16 for inference, split precision + ReLU masks for training) and backward (frozen / full).
//
// Same mapping to the hardware as the 64-wide kernel (mlp_tc.cu, read its header first; the code both share is in
// mlp_tc_common.cuh) with these differences:
//
//  * a thread (warp w, lane l) is still row 32 (w & 3) + l of the 128-sample tile and owns the column half
//    hf = w >> 2 of the hidden matrices -- now 64 columns, worked in two chunks of 32;
//  * biases are added in the epilogues from an fp32 copy in shared memory (broadcast reads) instead of by a bias MMA:
//    the [N x 16] bias tiles and the all-ones A tile of the 64-wide kernel would cost 13 KB here, which is what
//    decides between one and two resident CTAs for the split-precision forward (2 x 104 KB);
//  * TMEM columns: D 0..127 | A 128..191 | (split forward) A_lo 192..255 | (full backward) dW3' 192..335 (128 x 144,
//    column 128 = b3) | dW0' 336..383 (128 x 48, column 32 = b0) | dW2g 384..399 | dW1^T 400..415 | dW4^T 416..431 |
//    db1 432..447 and db4 448..463 (M = 64: X'^T . Gh and X'^T . Go, whose row 32 -- the all-ones feature of the X
//    tile -- is the column sum; the M side of dW1^T / dW4^T is the full 128 features of H1 / H3, so the bias cannot
//    ride along there as it does at H = 64) | S 464..479 (128 x 16 ray slots).  Forward / frozen backward allocate
//    256 columns (2 CTAs per SM), the full backward all 512 (1 CTA per SM: its [sample][feature] tiles take 133 KB);
//  * 16 ray slots per tile instead of 8 (N of an M = 128 MMA is a multiple of 16); a tile whose rays do not fit them
//    adds its d ray_bias rows with per-thread atomics;
//  * ReLU masks: uint32 [n][2][8] = per sample and column half {h1 c0, h1 c1, h2 c0, h2 c1, h3 c0, h3 c1, 0, 0}, one
//    word per 32-column chunk in the bit layout of mask_bits_of_pair.
#include "mlp_tc_common.cuh"

namespace gf {
namespace tc128 {

using namespace gf::tc;

constexpr int kH = 128;
using P = Blob<kH>;

// ---- shared memory ------------------------------------------------------------------------------------
constexpr uint32_t kOffB0 = 0;                          // N 128, K 32
constexpr uint32_t kOffB1 = kOffB0 + 128 * 32 * 2;      // N 16,  K 128
constexpr uint32_t kOffB2 = kOffB1 + 16 * 128 * 2;      // N 128, K 16 (geo columns of the head's layer 0)
constexpr uint32_t kOffB3 = kOffB2 + 128 * 16 * 2;      // N 128, K 128
constexpr uint32_t kOffB4 = kOffB3 + 128 * 128 * 2;     // N 16 (3 real rows), K 128
constexpr uint32_t kOffBias = kOffB4 + 16 * 128 * 2;    // fp32: b0 [128] | b1 [16] | b3 [128] | b4 [4]
constexpr int kBiasB0 = 0, kBiasB1 = 128, kBiasB3 = 144, kBiasB4 = 272, kBiasCount = 276;
constexpr uint32_t kOffBar = kOffBias + kBiasCount * 4;
constexpr uint32_t kOffBarW = kOffBar + 8;              // second mbarrier: completion of the weight-gradient MMAs
constexpr uint32_t kOffTmem = kOffBar + 16;
constexpr uint32_t kOffRay = kOffTmem + 8;              // int32 [128] ray of each row | [16] ray of each slot | [1] overflow flag
constexpr int kSlots = 16, kRaySlot0 = 128, kRayBad = 144;
constexpr uint32_t kSmemBase = (kOffRay + 4 * 160 + 127) / 128 * 128;
static_assert(kOffBar % 8 == 0, "mbarrier alignment");
// split forward only: the lo halves of the weight tiles of layers 0..3 (same layouts as the hi tiles)
constexpr uint32_t kOffB0L = kSmemBase;
constexpr uint32_t kOffB1L = kOffB0L + 128 * 32 * 2;
constexpr uint32_t kOffB2L = kOffB1L + 16 * 128 * 2;
constexpr uint32_t kOffB3L = kOffB2L + 128 * 16 * 2;
constexpr uint32_t kSmemSplit = kOffB3L + 128 * 128 * 2;
// [sample][feature] tiles of the full backward (feature chunk j of row r at (r / 8) * SBO + j * 128 + (r % 8) * 16)
constexpr uint32_t kSboX = 768, kSboH = 2048, kSboH2 = 2304, kSboS = 256;
constexpr uint32_t kOffX = kSmemBase;                   // [128][32 + 16]  (feature 32 = 1)
constexpr uint32_t kOffH1 = kOffX + 16 * kSboX;         // [128][128]      (G1 reuses it; the M = 64 reads of X' run into it)
constexpr uint32_t kOffH2 = kOffH1 + 16 * kSboH;        // [128][128 + 16] (feature 128 = 1; G2 reuses the first 128)
constexpr uint32_t kOffH3 = kOffH2 + 16 * kSboH2;       // [128][128]      (G3 reuses it)
constexpr uint32_t kOffHh = kOffH3 + 16 * kSboH;        // [128][16]
constexpr uint32_t kOffGo = kOffHh + 16 * kSboS;        // [128][16]
constexpr uint32_t kOffGh = kOffGo + 16 * kSboS;        // [128][16]
constexpr uint32_t kOffInd = kOffGh + 16 * kSboS;       // [128][16] ray-slot indicator (one-hot rows)
constexpr uint32_t kSmemFull = kOffInd + 16 * kSboS;
constexpr uint32_t kSmemSmall = kSmemBase;              // plain forward / frozen backward: weights only

// ---- tensor memory --------------------------------------------------------------------------------------
constexpr uint32_t kColD = 0, kColA = 128, kColAlo = 192;
constexpr uint32_t kColW3 = 192, kColW0 = 336, kColW2 = 384, kColW1 = 400, kColW4 = 416, kColB1 = 432, kColB4 = 448,
                   kColS = 464;

// fp32 parameter blob -> fp16 weight tiles (hi, and lo for the split forward), fp32 biases
template <bool SPLIT>
__device__ __forceinline__ void stage_weights(const float* __restrict__ p, unsigned char* smem) {
  for (uint32_t i = threadIdx.x; i < kOffBias / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0u;
  if (SPLIT)
    for (uint32_t i = threadIdx.x; i < (kSmemSplit - kOffB0L) / 4; i += blockDim.x)
      reinterpret_cast<uint32_t*>(smem + kOffB0L)[i] = 0u;
  __syncthreads();
  for (int i = threadIdx.x; i < kH * 32; i += blockDim.x)
    put_w<SPLIT>(smem, kOffB0, kOffB0L, 32, i >> 5, i & 31, __ldg(p + P::kW0 + i));
  for (int i = threadIdx.x; i < 16 * kH; i += blockDim.x)
    put_w<SPLIT>(smem, kOffB1, kOffB1L, kH, i / kH, i % kH, __ldg(p + P::kW1 + i));
  // geo column c (1..15) of the head's first layer multiplies h[c] = in2[15 + c]; column 0 (the density logit) is 0
  for (int i = threadIdx.x; i < kH * 15; i += blockDim.x) {
    const int j = i / 15, c = i % 15;
    put_w<SPLIT>(smem, kOffB2, kOffB2L, 16, j, 1 + c, __ldg(p + P::kW2 + j * 63 + 16 + c));
  }
  for (int i = threadIdx.x; i < kH * kH; i += blockDim.x)
    put_w<SPLIT>(smem, kOffB3, kOffB3L, kH, i / kH, i % kH, __ldg(p + P::kW3 + i));
  for (int i = threadIdx.x; i < 3 * kH; i += blockDim.x) put_b(smem, kOffB4, kH, i / kH, i % kH, __ldg(p + P::kW4 + i));
  float* sb = reinterpret_cast<float*>(smem + kOffBias);
  for (int i = threadIdx.x; i < kH; i += blockDim.x) {
    sb[kBiasB0 + i] = __ldg(p + P::kB0 + i);
    sb[kBiasB3 + i] = __ldg(p + P::kB3 + i);
    if (i < 16) sb[kBiasB1 + i] = __ldg(p + P::kB1 + i);
    if (i < 4) sb[kBiasB4 + i] = i < 3 ? __ldg(p + P::kB4 + i) : 0.f;
  }
}

// split-precision layer: D = A_hi . Bhi^T + A_hi . Blo^T (+ A_lo . Bhi^T)
template <int N, int K, bool A_LO>
__device__ __forceinline__ void issue_split(uint32_t tmem, uint32_t sBe, uint32_t off_w, uint32_t off_w_lo) {
  issue_ts<N, K>(tmem + kColD, tmem + kColA, sBe, off_w, false);
  issue_ts<N, K>(tmem + kColD, tmem + kColA, sBe, off_w_lo, true);
  if (A_LO) issue_ts<N, K>(tmem + kColD, tmem + kColAlo, sBe, off_w, true);
}
// 32 accumulator columns + fp32 bias (shared or global memory) -> ReLU -> 16 packed fp16 pairs
__device__ __forceinline__ void bias_relu_pack32(const uint32_t (&v)[32], const float* bias, uint32_t (&out)[16]) {
#pragma unroll
  for (int q = 0; q < 8; q++) {
    const float4 b = *reinterpret_cast<const float4*>(bias + 4 * q);
    out[2 * q] = pack_relu_h2(__uint_as_float(v[4 * q]) + b.x, __uint_as_float(v[4 * q + 1]) + b.y);
    out[2 * q + 1] = pack_relu_h2(__uint_as_float(v[4 * q + 2]) + b.z, __uint_as_float(v[4 * q + 3]) + b.w);
  }
}
// plain epilogue of a 128-wide layer for this thread's 64 columns: -> A operand in TMEM (+ the [sample][feature] tile)
template <bool STORE>
__device__ __forceinline__ void plain_epilogue64(uint32_t lane_addr, int hf, int r, const float* bias,
                                                 unsigned char* tile, uint32_t sbo) {
#pragma unroll
  for (int c = 0; c < 2; c++) {
    uint32_t v[32], h[16];
    tmem_ld32(lane_addr + kColD + 64 * hf + 32 * c, v);
    tmem_wait_ld();
    bias_relu_pack32(v, bias + 32 * c, h);
    tmem_st16(lane_addr + kColA + 32 * hf + 16 * c, h);
    if (STORE) store_chunks<4>(tile, sbo, r, 8 * hf + 4 * c, h);
  }
}
constexpr int min_ctas(int mode) { return mode == kBwdFull ? 1 : 2; }
constexpr int max_regs(int mode) { return mode == kBwdFull ? 232 : 128; }

template <int MODE>
__global__ void __launch_bounds__(kThreads, min_ctas(MODE)) __maxnreg__(max_regs(MODE))
mlp_tc128_kernel(int64_t n, const int32_t* __restrict__ d_n_ptr, const float* __restrict__ params,
                 const __half* __restrict__ feat, const int32_t* __restrict__ ray_id,
                 const float* __restrict__ ray_bias, float* __restrict__ sigma, float* __restrict__ rgb,
                 uint4* __restrict__ relu_masks, const float* __restrict__ d_sigma, const float* __restrict__ d_rgb,
                 __half* __restrict__ d_feat, float* __restrict__ d_params, float* __restrict__ d_ray_bias, float gscale) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr bool WGRAD = MODE == kBwdFull;
  constexpr bool BWD = MODE == kBwdFull || MODE == kBwdFrozen;
  constexpr bool SPLIT = MODE == kFwdSplit;
  constexpr uint32_t kCols = WGRAD ? 512u : 256u;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r = 32 * (warp & 3) + lane;  // row of the tile = TMEM lane
  const int hf = warp >> 2;              // column half (64 columns of the 128-wide matrices)
  const float inv_gscale = BWD ? 1.f / gscale : 1.f;
  stage_weights<SPLIT>(params, smem);
  const uint32_t bar = smem_u32(smem + kOffBar), bar_w = smem_u32(smem + kOffBarW);
  cta_alloc<kCols>(bar, bar_w, smem + kOffTmem);
  if (WGRAD) {
    // constant parts of the [sample][feature] tiles: X' features 32 (= 1) .. 47, H2' features 128 (= 1) .. 143
    if (hf == 0) {
      store_ones(smem + kOffX, kSboX, r, 4);
      store_ones(smem + kOffH2, kSboH2, r, 16);
    } else {
      *tile_chunk(smem + kOffX, kSboX, r, 5) = make_uint4(0u, 0u, 0u, 0u);
      *tile_chunk(smem + kOffH2, kSboH2, r, 17) = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  const uint32_t tmem = cta_publish(smem + kOffTmem);
  const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
  const uint32_t sBe = smem_base_enc(smem_u32(smem));
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);  // provably warp-uniform: the issue branch stays converged
  int* s_ray = reinterpret_cast<int*>(smem + kOffRay);
  const float* s_bias = reinterpret_cast<const float*>(smem + kOffBias);
  if (d_n_ptr) {
    const int64_t dn = *d_n_ptr;
    n = dn < n ? dn : n;
  }
  uint32_t phase = 0, phase_w = 0;
  bool first_tile = true;
  const int64_t n_tiles = (n + kTile - 1) / kTile;
  // this thread's inputs of the CTA's NEXT tile are loaded one tile ahead into registers
  uint4 xn0 = make_uint4(0u, 0u, 0u, 0u), xn1 = xn0;
  int rayn = -1;
  {
    const int64_t row0 = (int64_t)blockIdx.x * kTile + r;
    if (row0 < n) load_row(feat, ray_id, row0, hf, xn0, xn1, rayn);
  }
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t row = tile * kTile + r;
    const bool valid = row < n;
    const int ray = rayn;
    const uint4 x0 = xn0, x1 = xn1;
    // backward: the forward's ReLU masks of this thread's 64 columns: {h1 c0, h1 c1, h2 c0, h2 c1}, {h3 c0, h3 c1, -, -}
    uint4 mk0 = make_uint4(0u, 0u, 0u, 0u), mk1 = mk0;
    if (BWD && valid) {
      mk0 = __ldg(relu_masks + 2 * (2 * row + hf));
      mk1 = __ldg(relu_masks + 2 * (2 * row + hf) + 1);
    }
    const float* rb = ray_bias + (int64_t)(valid ? ray : 0) * kH + 64 * hf;
    // real loads instead of prefetch hints (see mlp_tc.cu): two 4-byte loads pull the thread's two 128-byte bias lines
    // into L1, and the four upstream gradients of the row go to registers now (hf == 0 consumes them)
    float up[4] = {0.f, 0.f, 0.f, 0.f};
    if (valid) {
      float touch;
      asm volatile("ld.global.nc.f32 %0, [%1];\n" : "=f"(touch) : "l"(rb));
      asm volatile("ld.global.nc.f32 %0, [%1];\n" : "=f"(touch) : "l"(rb + 32));
      if (BWD && hf == 0) {
        up[0] = __ldg(d_rgb + 3 * row);
        up[1] = __ldg(d_rgb + 3 * row + 1);
        up[2] = __ldg(d_rgb + 3 * row + 2);
        up[3] = __ldg(d_sigma + row);
      }
    }
    const int64_t nrow = row + (int64_t)gridDim.x * kTile;
    uint32_t m1[2] = {0u, 0u}, m2[2] = {0u, 0u}, m3[2] = {0u, 0u};  // split forward: ReLU masks of the two chunks
    float pre = 0.f;                                                   // density logit + 1 (hf == 0)
    // ---- input: features 16 hf .. 16 hf + 15 of this row -> A columns [8 hf, 8 hf + 8) (+ X tile) -------------
    {
      const uint32_t x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
      if (WGRAD) {
        *tile_chunk(smem + kOffX, kSboX, r, 2 * hf) = x0;
        *tile_chunk(smem + kOffX, kSboX, r, 2 * hf + 1) = x1;
        if (hf == 0) s_ray[r] = ray;
        if (tid >= 128 && tid <= 128 + kSlots) s_ray[tid] = tid == kRayBad ? 0 : -1;  // slot rays := none, flag := 0
      }
      tmem_st8(lane_addr + kColA + 8 * hf, x);
    }
    // next tile's inputs: in flight during this whole tile
    xn0 = xn1 = make_uint4(0u, 0u, 0u, 0u);
    rayn = -1;
    if (nrow < n) {
      load_row(feat, ray_id, nrow, hf, xn0, xn1, rayn);
      if (BWD && (lane & 7) == 0) {  // its upstream gradients towards L2
        if (hf == 0) prefetch_l2(d_rgb + 3 * nrow);
        else prefetch_l2(d_sigma + nrow);
      }
      if (BWD && (lane & 1) == 0) prefetch_l2(relu_masks + 2 * (2 * nrow + hf));
    }
    // ---- layer 0: h1 = relu(X . W0^T + b0) ------------------------------------------------------------------
    if (SPLIT) {   // the input features ARE fp16 (the hash encoder's output): only the weights carry a lo part
      GF_TC_SYNC_ISSUE((issue_split<128, 32, false>(tmem, sBe, kOffB0, kOffB0L)))
    } else {
      GF_TC_SYNC_ISSUE((issue_ts<128, 32>(tmem + kColD, tmem + kColA, sBe, kOffB0, false)))
    }
    GF_TC_WAIT()
    if (SPLIT) {
#pragma unroll
      for (int c = 0; c < 2; c++)
        m1[c] = split_epilogue32<true, true, false>(lane_addr + kColD + 64 * hf + 32 * c,
                                                    lane_addr + kColA + 32 * hf + 16 * c,
                                                    lane_addr + kColAlo + 32 * hf + 16 * c,
                                                    s_bias + kBiasB0 + 64 * hf + 32 * c);
    } else {
      plain_epilogue64<WGRAD>(lane_addr, hf, r, s_bias + kBiasB0 + 64 * hf, smem + kOffH1, kSboH);
      if (WGRAD && hf == 1) {
        // One-hot "ray slot" row of this sample (slot = ray - the tile's first ray; rays are non-decreasing along the
        // samples): d ray_bias of the tile's rays is then G2^T . Ind, one more weight-gradient-shaped MMA.  A tile
        // whose rays do not fit the 16 slots raises the flag and its rows add their gradients with atomics.
        const unsigned slot = (unsigned)(ray - s_ray[0]);
        uint32_t one = 0u;
        if (valid) {
          if (slot < (unsigned)kSlots) {
            one = 0x3C00u << (16 * (slot & 1));  // fp16 1.0 in the slot's half of its 32-bit word
            if (r == 0 || s_ray[r - 1] != ray) s_ray[kRaySlot0 + slot] = ray;
          } else {
            s_ray[kRayBad] = 1;
          }
        }
        const unsigned wd = slot >> 1;
        *tile_chunk(smem + kOffInd, kSboS, r, 0) =
            make_uint4(wd == 0u ? one : 0u, wd == 1u ? one : 0u, wd == 2u ? one : 0u, wd == 3u ? one : 0u);
        *tile_chunk(smem + kOffInd, kSboS, r, 1) =
            make_uint4(wd == 4u ? one : 0u, wd == 5u ? one : 0u, wd == 6u ? one : 0u, wd == 7u ? one : 0u);
      }
    }
    // ---- layer 1: h = h1 . W1^T + b1; density = exp(h0 + 1); geo features -> A (16 fp16) -----------------------
    if (SPLIT) {
      GF_TC_SYNC_ISSUE((issue_split<16, 128, true>(tmem, sBe, kOffB1, kOffB1L)))
    } else {
      GF_TC_SYNC_ISSUE((issue_ts<16, 128>(tmem + kColD, tmem + kColA, sBe, kOffB1, false)))
    }
    GF_TC_WAIT()
    if (hf == 0) {
      uint32_t v[16], a[8];
      tmem_ld16(lane_addr + kColD, v);
      tmem_wait_ld();
      float h[16];
#pragma unroll
      for (int j = 0; j < 16; j++) h[j] = __uint_as_float(v[j]) + s_bias[kBiasB1 + j];
      pre = h[0] + 1.f;
      if (!BWD && valid) sigma[row] = expf(pre);  // trunc_exp(h0 + 1), nerfacto_field.py:499
      h[0] = 0.f;                                   // column 0 of the geo tile has zero weights
      if (SPLIT) {
        uint32_t al[8];
        float hh[16];
#pragma unroll
        for (int j = 0; j < 16; j++) hh[j] = trunc11(h[j]);
#pragma unroll
        for (int j = 0; j < 8; j++) {
          a[j] = pack_h2(hh[2 * j], hh[2 * j + 1]);
          al[j] = pack_h2(h[2 * j] - hh[2 * j], h[2 * j + 1] - hh[2 * j + 1]);
        }
        tmem_st8(lane_addr + kColAlo, al);
      } else {
#pragma unroll
        for (int j = 0; j < 8; j++) a[j] = pack_h2(h[2 * j], h[2 * j + 1]);
      }
      tmem_st8(lane_addr + kColA, a);
      if (WGRAD) store_chunks<2>(smem + kOffHh, kSboS, r, 0, a);
    }
    // ---- head layer 0: h2 = relu(geo . W2g^T + ray_bias[ray]) ---------------------------------------------------
    if (SPLIT) {
      GF_TC_SYNC_ISSUE((issue_split<128, 16, true>(tmem, sBe, kOffB2, kOffB2L)))
    } else {
      GF_TC_SYNC_ISSUE((issue_ts<128, 16>(tmem + kColD, tmem + kColA, sBe, kOffB2, false)))
    }
    GF_TC_WAIT()
    if (SPLIT) {
#pragma unroll
      for (int c = 0; c < 2; c++)
        m2[c] = split_epilogue32<true, true, false>(lane_addr + kColD + 64 * hf + 32 * c,
                                                    lane_addr + kColA + 32 * hf + 16 * c,
                                                    lane_addr + kColAlo + 32 * hf + 16 * c, rb + 32 * c);
    } else {
      plain_epilogue64<WGRAD>(lane_addr, hf, r, rb, smem + kOffH2, kSboH2);
    }
    // ---- head layer 1: h3 = relu(h2 . W3^T + b3) -------------------------------------------------------------
    if (SPLIT) {
      GF_TC_SYNC_ISSUE((issue_split<128, 128, true>(tmem, sBe, kOffB3, kOffB3L)))
    } else {
      GF_TC_SYNC_ISSUE((issue_ts<128, 128>(tmem + kColD, tmem + kColA, sBe, kOffB3, false)))
    }
    GF_TC_WAIT()
    if (SPLIT) {
      // (no lo part: the output layer takes h3 as plain fp16 -- no ReLU follows it)
#pragma unroll
      for (int c = 0; c < 2; c++)
        m3[c] = split_epilogue32<true, false, false>(lane_addr + kColD + 64 * hf + 32 * c,
                                                     lane_addr + kColA + 32 * hf + 16 * c, 0u,
                                                     s_bias + kBiasB3 + 64 * hf + 32 * c);
      if (relu_masks && valid) {
        relu_masks[2 * (2 * row + hf)] = make_uint4(m1[0], m1[1], m2[0], m2[1]);
        relu_masks[2 * (2 * row + hf) + 1] = make_uint4(m3[0], m3[1], 0u, 0u);
      }
    } else {
      plain_epilogue64<WGRAD>(lane_addr, hf, r, s_bias + kBiasB3 + 64 * hf, smem + kOffH3, kSboH);
    }
    // ---- head layer 2: rgb logits = h3 . W4^T + b4 ----------------------------------------------------------
    GF_TC_SYNC_ISSUE((issue_ts<16, 128>(tmem + kColD, tmem + kColA, sBe, kOffB4, false)))
    GF_TC_WAIT()
    if (!BWD) {
      if (hf == 0) {
        uint32_t v[4];
        tmem_ld4(lane_addr + kColD, v);
        tmem_wait_ld();
        if (valid) {
          rgb[3 * row] = sigmoidf_(__uint_as_float(v[0]) + s_bias[kBiasB4]);
          rgb[3 * row + 1] = sigmoidf_(__uint_as_float(v[1]) + s_bias[kBiasB4 + 1]);
          rgb[3 * row + 2] = sigmoidf_(__uint_as_float(v[2]) + s_bias[kBiasB4 + 2]);
        }
      }
      tc_fence_before();
      continue;
    }
    // ---- g o = d rgb * s (1 - s)  (all gradients carry the factor gscale while they are fp16) ------------------
    if (hf == 0) {
      uint32_t v[4], a[8];
      tmem_ld4(lane_addr + kColD, v);
      tmem_wait_ld();
      float go[3] = {0.f, 0.f, 0.f};
      if (valid) {
#pragma unroll
        for (int c = 0; c < 3; c++) {
          const float sg = sigmoidf_(__uint_as_float(v[c]) + s_bias[kBiasB4 + c]);
          go[c] = up[c] * gscale * sg * (1.f - sg);
        }
      }
      a[0] = pack_h2(go[0], go[1]);
      a[1] = pack_h2(go[2], 0.f);
#pragma unroll
      for (int j = 2; j < 8; j++) a[j] = 0u;
      tmem_st8(lane_addr + kColA, a);
      if (WGRAD) store_chunks<2>(smem + kOffGo, kSboS, r, 0, a);
    }
    // g h3 = g o . W4 ; dW4^T += H3^T . Go ; db4 = row 32 of X'^T . Go
    GF_TC_SYNC_ISSUE2((issue_dgrad<128, 16>(tmem + kColD, tmem + kColA, sBe, kOffB4, sbo_of(kH))),
                      (issue_wgrad<128, 16>(tmem + kColW4, sBe, kOffH3, kSboH, kOffGo, kSboS, first_tile),
                       issue_wgrad<64, 16>(tmem + kColB4, sBe, kOffX, kSboX, kOffGo, kSboS, first_tile)))
    GF_TC_WAIT()
    {
      uint32_t g[2][16];
#pragma unroll
      for (int c = 0; c < 2; c++) {
        uint32_t v[32];
        tmem_ld32(lane_addr + kColD + 64 * hf + 32 * c, v);
        tmem_wait_ld();
        mask_bits_pack32(v, c == 0 ? mk1.x : mk1.y, g[c]);
        tmem_st16(lane_addr + kColA + 32 * hf + 16 * c, g[c]);
      }
      GF_TC_WAIT_W()
      if (WGRAD) {  // G3 over H3 (its readers have completed)
        store_chunks<4>(smem + kOffH3, kSboH, r, 8 * hf, g[0]);
        store_chunks<4>(smem + kOffH3, kSboH, r, 8 * hf + 4, g[1]);
      }
    }
    // g h2 = g h3 . W3 ; dW3 (+ b3 column) += G3^T . H2'
    GF_TC_SYNC_ISSUE2((issue_dgrad<128, 128>(tmem + kColD, tmem + kColA, sBe, kOffB3, sbo_of(kH))),
                      (issue_wgrad<128, 144>(tmem + kColW3, sBe, kOffH3, kSboH, kOffH2, kSboH2, first_tile)))
    GF_TC_WAIT()
    {
      uint32_t g[2][16];
#pragma unroll
      for (int c = 0; c < 2; c++) {
        uint32_t v[32];
        tmem_ld32(lane_addr + kColD + 64 * hf + 32 * c, v);
        tmem_wait_ld();
        mask_bits_pack32(v, c == 0 ? mk0.z : mk0.w, g[c]);
        tmem_st16(lane_addr + kColA + 32 * hf + 16 * c, g[c]);
      }
      if (WGRAD && valid && s_ray[kRayBad] != 0) {
        // the tile's rays did not fit the ray slots: d ray_bias[ray] += this row's g h2, element by element
        float* dst = d_ray_bias + (int64_t)ray * kH + 64 * hf;
#pragma unroll
        for (int c = 0; c < 2; c++)
#pragma unroll
          for (int q = 0; q < 16; q++) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&g[c][q]));
            if (f.x != 0.f) atomicAdd(dst + 32 * c + 2 * q, f.x * inv_gscale);
            if (f.y != 0.f) atomicAdd(dst + 32 * c + 2 * q + 1, f.y * inv_gscale);
          }
      }
      GF_TC_WAIT_W()
      if (WGRAD) {  // G2 over H2 (features 0..127; the ones column stays)
        store_chunks<4>(smem + kOffH2, kSboH2, r, 8 * hf, g[0]);
        store_chunks<4>(smem + kOffH2, kSboH2, r, 8 * hf + 4, g[1]);
      }
    }
    // g h[1:16] = g h2 . W2[:, geo] ; S[128 x 16 slots] = G2^T . Ind ; dW2[:, geo] += G2^T . Hh
    GF_TC_SYNC_ISSUE2((issue_dgrad<16, 128>(tmem + kColD, tmem + kColA, sBe, kOffB2, sbo_of(16)),
                       WGRAD ? issue_wgrad<128, 16>(tmem + kColS, sBe, kOffH2, kSboH2, kOffInd, kSboS, true) : (void)0),
                      (issue_wgrad<128, 16>(tmem + kColW2, sBe, kOffH2, kSboH2, kOffHh, kSboS, first_tile)))
    GF_TC_WAIT()
    if (WGRAD && hf == 1 && s_ray[kRayBad] == 0) {
      // d ray_bias[ray of slot s][o] += S[o][s]; M = 128 accumulator: row o = this thread's TMEM lane
      uint32_t sv[16];
      tmem_ld16(lane_addr + kColS, sv);
      tmem_wait_ld();
#pragma unroll
      for (int q = 0; q < kSlots; q++) {
        const int rr = s_ray[kRaySlot0 + q];
        const float f = __uint_as_float(sv[q]);
        if (rr >= 0 && f != 0.f) atomicAdd(d_ray_bias + (int64_t)rr * kH + r, f * inv_gscale);
      }
    }
    // ---- g h = [ d sigma * exp(clamp(h0 + 1)) | acc[1:16] ] ---------------------------------------------------
    if (hf == 0) {
      uint32_t a[8];
      grad_h16(lane_addr + kColD, valid, up[3], gscale, pre, a);
      tmem_st8(lane_addr + kColA, a);
      if (WGRAD) store_chunks<2>(smem + kOffGh, kSboS, r, 0, a);
    }
    GF_TC_WAIT_W()   // dW2's MMAs; every thread waits every phase of bar_w (the parity is tracked per thread)
    // g h1 = g h . W1 ; dW1^T += H1^T . Gh ; db1 = row 32 of X'^T . Gh
    GF_TC_SYNC_ISSUE2((issue_dgrad<128, 16>(tmem + kColD, tmem + kColA, sBe, kOffB1, sbo_of(kH))),
                      (issue_wgrad<128, 16>(tmem + kColW1, sBe, kOffH1, kSboH, kOffGh, kSboS, first_tile),
                       issue_wgrad<64, 16>(tmem + kColB1, sBe, kOffX, kSboX, kOffGh, kSboS, first_tile)))
    GF_TC_WAIT()
    {
      uint32_t g[2][16];
#pragma unroll
      for (int c = 0; c < 2; c++) {
        uint32_t v[32];
        tmem_ld32(lane_addr + kColD + 64 * hf + 32 * c, v);
        tmem_wait_ld();
        mask_bits_pack32(v, c == 0 ? mk0.x : mk0.y, g[c]);
        tmem_st16(lane_addr + kColA + 32 * hf + 16 * c, g[c]);
      }
      GF_TC_WAIT_W()
      if (WGRAD) {  // G1 over H1
        store_chunks<4>(smem + kOffH1, kSboH, r, 8 * hf, g[0]);
        store_chunks<4>(smem + kOffH1, kSboH, r, 8 * hf + 4, g[1]);
      }
    }
    // g x = g h1 . W0 ; dW0 (+ b0 column) += G1^T . X'
    GF_TC_SYNC_ISSUE2((issue_dgrad<32, 128>(tmem + kColD, tmem + kColA, sBe, kOffB0, sbo_of(32))),
                      (issue_wgrad<128, 48>(tmem + kColW0, sBe, kOffH1, kSboH, kOffX, kSboX, first_tile)))
    GF_TC_WAIT()
    // ---- d feat -------------------------------------------------------------------------------------------------
    store_d_feat(lane_addr + kColD + 16 * hf, valid, inv_gscale, d_feat, row, hf);
    GF_TC_WAIT_W()   // dW0's MMAs read the X and G1 tiles the next tile overwrites (and the flush reads the sums)
    tc_fence_before();
    first_tile = false;
  }
  if (WGRAD && !first_tile) {
    // ---- flush the weight-gradient accumulators: one atomicAdd per parameter per CTA ------------------------------
    // (every MMA has completed: the last waits covered them).  M = 128 accumulators: row = this thread's TMEM lane r
    {
      // dW3 [o = r][64 hf .. 64 hf + 63]
#pragma unroll
      for (int c = 0; c < 2; c++) {
        uint32_t v[32];
        tmem_ld32(lane_addr + kColW3 + 64 * hf + 32 * c, v);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; i++) {
          const float g = __uint_as_float(v[i]);
          if (g != 0.f) atomicAdd(d_params + P::kW3 + r * kH + 64 * hf + 32 * c + i, g * inv_gscale);
        }
      }
    }
    if (hf == 0) {
      uint32_t v[32], w[4];
      tmem_ld4(lane_addr + kColW3 + 128, w);   // b3[o] = column 128
      tmem_ld32(lane_addr + kColW0, v);        // dW0 [o][0..31]
      tmem_wait_ld();
      if (__uint_as_float(w[0]) != 0.f) atomicAdd(d_params + P::kB3 + r, __uint_as_float(w[0]) * inv_gscale);
#pragma unroll
      for (int i = 0; i < 32; i++) {
        const float g = __uint_as_float(v[i]);
        if (g != 0.f) atomicAdd(d_params + P::kW0 + r * 32 + i, g * inv_gscale);
      }
      tmem_ld4(lane_addr + kColW0 + 32, w);    // b0[o] = column 32
      tmem_wait_ld();
      if (__uint_as_float(w[0]) != 0.f) atomicAdd(d_params + P::kB0 + r, __uint_as_float(w[0]) * inv_gscale);
      // dW4^T [i = r][oo]
      tmem_ld4(lane_addr + kColW4, w);
      tmem_wait_ld();
#pragma unroll
      for (int oo = 0; oo < 3; oo++) {
        const float g = __uint_as_float(w[oo]);
        if (g != 0.f) atomicAdd(d_params + P::kW4 + oo * kH + r, g * inv_gscale);
      }
      // db1, db4: row 32 of the M = 64 accumulators = lane 0 of quadrant 2
      uint32_t u[16];
      tmem_ld16(lane_addr + kColB1, u);
      tmem_ld4(lane_addr + kColB4, w);
      tmem_wait_ld();
      if ((warp & 3) == 2 && lane == 0) {
#pragma unroll
        for (int oo = 0; oo < 16; oo++)
          if (__uint_as_float(u[oo]) != 0.f) atomicAdd(d_params + P::kB1 + oo, __uint_as_float(u[oo]) * inv_gscale);
#pragma unroll
        for (int oo = 0; oo < 3; oo++)
          if (__uint_as_float(w[oo]) != 0.f) atomicAdd(d_params + P::kB4 + oo, __uint_as_float(w[oo]) * inv_gscale);
      }
    } else {
      uint32_t w[16];
      // dW2 [o = r][geo c], c = 1..15 -> column 15 + c of W2
      tmem_ld16(lane_addr + kColW2, w);
      tmem_wait_ld();
#pragma unroll
      for (int c = 1; c < 16; c++) {
        const float g = __uint_as_float(w[c]);
        if (g != 0.f) atomicAdd(d_params + P::kW2 + r * 63 + 15 + c, g * inv_gscale);
      }
      // dW1^T [i = r][oo]
      tmem_ld16(lane_addr + kColW1, w);
      tmem_wait_ld();
#pragma unroll
      for (int oo = 0; oo < 16; oo++) {
        const float g = __uint_as_float(w[oo]);
        if (g != 0.f) atomicAdd(d_params + P::kW1 + oo * kH + r, g * inv_gscale);
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kCols);
}
}  // namespace tc128
}  // namespace gf

using namespace gf;

static_assert(tc128::kSmemFull <= 227 * 1024, "full backward smem");
static_assert(2 * (tc128::kSmemSplit + 1024) <= 228 * 1024, "two split-forward CTAs per SM");

// launched by gf_mlp_forward / gf_mlp_backward (mlp.cu) for hidden == 128
int gf_launch_mlp_fwd_tc128(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                            const int32_t* ray_id, const float* ray_bias, float* sigma, float* rgb, void* relu_masks,
                            cudaStream_t st) {
  int rc = set_smem_attrs<tc128::kH>(tc128::mlp_tc128_kernel<tc::kFwd>, tc128::mlp_tc128_kernel<tc::kBwdFrozen>,
                                     tc128::mlp_tc128_kernel<tc::kBwdFull>, tc128::mlp_tc128_kernel<tc::kFwdSplit>,
                                     {(int)tc128::kSmemSmall, (int)tc128::kSmemSmall, (int)tc128::kSmemFull,
                                      (int)tc128::kSmemSplit});
  if (rc) return rc;
  const int64_t tiles = div_up(n, tc::kTile);
  const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * 2);
  if (relu_masks) {   // training: split precision + the ReLU masks for gf_mlp_backward
    tc128::mlp_tc128_kernel<tc::kFwdSplit><<<grid, tc::kThreads, tc128::kSmemSplit, st>>>(
        n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, sigma, rgb, (uint4*)relu_masks, nullptr, nullptr,
        nullptr, nullptr, nullptr, 1.f);
    return check_launch("mlp_tc128_kernel<fwd split>");
  }
  tc128::mlp_tc128_kernel<tc::kFwd><<<grid, tc::kThreads, tc128::kSmemSmall, st>>>(
      n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, sigma, rgb, nullptr, nullptr, nullptr, nullptr,
      nullptr, nullptr, 1.f);
  return check_launch("mlp_tc128_kernel<fwd>");
}

int gf_launch_mlp_bwd_tc128(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                            const int32_t* ray_id, const float* ray_bias, const void* relu_masks, const float* d_sigma,
                            const float* d_rgb, void* d_feat, float* d_params, float* d_ray_bias, float gscale,
                            cudaStream_t st) {
  int rc = set_smem_attrs<tc128::kH>(tc128::mlp_tc128_kernel<tc::kFwd>, tc128::mlp_tc128_kernel<tc::kBwdFrozen>,
                                     tc128::mlp_tc128_kernel<tc::kBwdFull>, tc128::mlp_tc128_kernel<tc::kFwdSplit>,
                                     {(int)tc128::kSmemSmall, (int)tc128::kSmemSmall, (int)tc128::kSmemFull,
                                      (int)tc128::kSmemSplit});
  if (rc) return rc;
  const int64_t tiles = div_up(n, tc::kTile);
  if (d_params) {
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count());
    tc128::mlp_tc128_kernel<tc::kBwdFull><<<grid, tc::kThreads, tc128::kSmemFull, st>>>(
        n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, nullptr, nullptr, (uint4*)relu_masks, d_sigma,
        d_rgb, (__half*)d_feat, d_params, d_ray_bias, gscale);
  } else {  // frozen MLP (focal stage): dgrad only
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * 2);
    tc128::mlp_tc128_kernel<tc::kBwdFrozen><<<grid, tc::kThreads, tc128::kSmemSmall, st>>>(
        n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, nullptr, nullptr, (uint4*)relu_masks, d_sigma,
        d_rgb, (__half*)d_feat, nullptr, nullptr, gscale);
  }
  return check_launch("mlp_tc128_kernel<bwd>");
}
