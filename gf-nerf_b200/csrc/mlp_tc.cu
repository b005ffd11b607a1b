// Fused field MLP on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a: forward and backward.
//
// The two MLPNetwork stacks of the reference field (gfnerf/mlp.py:25-57 as built at
// gfnerf/nerfacto_field.py:174-179,217-227), trunc_exp(x + 1) (:499), the sigmoid head, and everything autograd
// does for them; SH(dir) and the appearance embedding enter as a per-ray bias of the head's first layer
// (ray_bias kernels in mlp.cu).  Mapping to the Blackwell execution model:
//
//  * a CTA of 256 threads owns a tile of 128 samples.  Thread (warp w, lane l) IS ROW 32 (w & 3) + l of every
//    activation / gradient matrix -- it owns TMEM lane r (tcgen05.ld/st shape 32x32b, warp w <-> lane quadrant
//    w & 3) -- and the column half hf = w >> 2 of the 64-wide matrices;
//  * every layer is D[128 x N] = A[128 x K] . B^T issued by ONE thread as K/16 tcgen05.mma (M = 128, kind::f16,
//    fp32 accumulate in TMEM) plus one more MMA that adds the bias: A = a constant [128 x 16] tile whose first
//    column is 1, B = [N x 16] with the bias in its first column;
//  * the A operand never touches shared memory: the epilogue of layer l (tcgen05.ld of the fp32 accumulator row,
//    fp16 pack, ReLU) writes the next layer's A straight back into TMEM with tcgen05.st and the next MMA reads it
//    from there (TS form: A K-major in TMEM, two fp16 per 32-bit column);
//  * weights are staged once per CTA into shared memory as fp16 in the canonical no-swizzle K-major core-matrix
//    layout and addressed through shared-memory matrix descriptors; the backward's dgrad layers read the SAME tiles
//    transposed through MN-major descriptors;
//  * weight gradients: the activation / gradient tiles are also written to shared memory ([sample][feature]
//    fp16, core-matrix layout) and dW = G^T . ACT is an SS-form MMA with BOTH operands MN-major (K = the 128
//    samples), accumulated over all tiles of the CTA in TMEM; bias gradients ride along as an all-ones feature
//    column of the activation tiles.  tcgen05.commit covers every MMA issued before it, so a tile buffer is free
//    again one dgrad round after the weight-gradient MMAs that read it were issued: G3 / G2 / G1 / Gh reuse the
//    H3 / H2 / H1 / Go buffers.  One atomicAdd per parameter per CTA at the end;
//  * completion: tcgen05.commit -> mbarrier; the 256 threads wait on it with try_wait.parity.
//  * SPLIT PRECISION (forward): an fp16 MLP reproduces the reference's fp32 outputs to ~1e-3, but not its ReLU
//    masks: a hidden unit whose pre-activation lies within fp16 rounding of zero flips, and every flip changes one
//    (sample, unit) gradient term by 100 % -- 1-2 % in relative L2 on every gradient that passes a ReLU (measured in
//    numpy, tests/test_mlp_gpu.py).  The forward therefore carries weights AND activations of layers 0..3 as fp16
//    pairs hi + lo (value = hi + lo to ~21 bits) and evaluates  A_hi.W_hi + A_hi.W_lo + A_lo.W_hi  (three TS-form
//    MMA groups into the same fp32 accumulator; the lo.lo term is below fp32 resolution), biases as hi + lo in two
//    columns of the bias MMA.  The ReLU masks of that forward are written out as 3 x 64 bits per sample and the
//    backward -- which recomputes the activations in plain fp16, good to 5e-4 -- applies THOSE masks (and no
//    longer keeps 48 registers of activations alive for them).  Gradients then agree with the fp32 reference to
//    ~4e-4 relative L2 instead of 1-2e-2.
//
// TMEM columns: D 0..63 | A 64..95 | (forward) A_lo 96..127 | (backward with weight gradients) dW3' 96..167 (64 x 72) | dW0' 168..207
// (64 x 40) | dW2g 208..223 (64 x 16) | dW1^T 224..239 (128 x 16) | dW4^T 240..255 (128 x 16).
// Forward / frozen-MLP backward allocate 128 columns (4 CTAs per SM), the full backward 256 (2 CTAs per SM).
//
// What this kernel does exactly as the 128-wide one (mlp_tc128.cu) -- the parameter blob layout, the MMA issue helpers,
// the issue / commit / wait macros, the split-precision epilogue, the CTA prologue, the backward's g h and d feat
// blocks, the shared-memory opt-in -- is in mlp_tc_common.cuh; this file holds the 64-wide layouts, the bias MMA and
// the kernel body.
#ifdef GF_MLP_TRACE
// profiling build only (tools/mlp_trace.py): clock64() of thread 0 / thread 128 of CTA 0 at the phase boundaries of
// its third tile, marked by GF_TR() in the kernel and in the issue / wait macros of mlp_tc_common.cuh
#define GF_TR()                                                                              \
  {                                                                                          \
    if (blockIdx.x == 0 && tile == 2 * (int64_t)gridDim.x && (tid & 127) == 0 && tr_i < 64)  \
      g_mlp_trace[tid >> 7][tr_i] = clock64();                                               \
    tr_i++;                                                                                  \
  }
#endif
#include "mlp_tc_common.cuh"

namespace gf {
namespace tc {

constexpr int kH = 64;
using P = Blob<kH>;

#ifdef GF_MLP_TRACE
__device__ unsigned long long g_mlp_trace[2][64];
#endif

// ---- shared memory ------------------------------------------------------------------------------------
constexpr uint32_t kOffB0 = 0;                        // N 64, K 32
constexpr uint32_t kOffB1 = kOffB0 + 64 * 32 * 2;     // N 16, K 64
constexpr uint32_t kOffB2 = kOffB1 + 16 * 64 * 2;     // N 64, K 16 (geo columns of the head's layer 0)
constexpr uint32_t kOffB3 = kOffB2 + 64 * 16 * 2;     // N 64, K 64
constexpr uint32_t kOffB4 = kOffB3 + 64 * 64 * 2;     // N 16 (3 real rows), K 64
constexpr uint32_t kOffBb0 = kOffB4 + 16 * 64 * 2;    // bias tiles [N][16]: column 0 = bias
constexpr uint32_t kOffBb1 = kOffBb0 + 64 * 16 * 2;
constexpr uint32_t kOffBb3 = kOffBb1 + 16 * 16 * 2;
constexpr uint32_t kOffBb4 = kOffBb3 + 64 * 16 * 2;
constexpr uint32_t kOffOnes = kOffBb4 + 16 * 16 * 2;  // A tile [128][16]: column 0 = 1
constexpr uint32_t kOffBar = kOffOnes + 128 * 16 * 2;
constexpr uint32_t kOffBarW = kOffBar + 8;            // second mbarrier: completion of the weight-gradient MMAs
constexpr uint32_t kOffTmem = kOffBar + 16;
constexpr uint32_t kOffRay = kOffTmem + 8;             // int32 ray id of each row (full backward)
// + int32 [8]: the ray of each of the tile's (up to) 8 ray slots, + int32: "a row fell outside the 8 slots"
constexpr uint32_t kSmemBase = (kOffRay + 512 + 64 + 127) / 128 * 128;
// forward only: the lo halves of the weight tiles of layers 0..3 (same layouts as the hi tiles)
constexpr uint32_t kOffB0L = kSmemBase;
constexpr uint32_t kOffB1L = kOffB0L + 64 * 32 * 2;
constexpr uint32_t kOffB2L = kOffB1L + 16 * 64 * 2;
constexpr uint32_t kOffB3L = kOffB2L + 64 * 16 * 2;
constexpr uint32_t kSmemFwd = kOffB3L + 64 * 64 * 2;
// [sample][feature] tiles of the full backward
constexpr uint32_t kSboX = 640, kSboH = 1152, kSboG = 1024, kSboS = 256;
constexpr uint32_t kOffX = kSmemBase;                  // [128][32 + 8]   SBO 640
constexpr uint32_t kOffH1 = kOffX + 16 * kSboX;        // [128][64 + 8]   SBO 1152 (G1 reuses it with SBO 1024)
constexpr uint32_t kOffH2 = kOffH1 + 16 * kSboH;
constexpr uint32_t kOffH3 = kOffH2 + 16 * kSboH;
constexpr uint32_t kOffHh = kOffH3 + 16 * kSboH;       // [128][16]       SBO 256
constexpr uint32_t kOffGo = kOffHh + 16 * kSboS;       // [128][16]       SBO 256 (Gh reuses it)
constexpr uint32_t kOffInd = kOffGo + 16 * kSboS;      // [128][8]        SBO 128: ray-slot indicator (one-hot rows)
constexpr uint32_t kSmemFull = kOffInd + 16 * 128 + 1024;  // + slack: the M = 128 reads of H3' run past its tile

// ---- tensor memory --------------------------------------------------------------------------------------
constexpr uint32_t kColD = 0, kColA = 64, kColAlo = 96;
constexpr uint32_t kColW3 = 96, kColW0 = 168, kColW2 = 208, kColW1 = 224, kColW4 = 240;

// bias b -> columns 0 (hi) and 1 (lo) of a bias tile; the all-ones A tile has ones in both columns
__device__ __forceinline__ void put_bias(unsigned char* smem, uint32_t off, int n, float b) {
  put_b(smem, off, 16, n, 0, b);
  put_b(smem, off, 16, n, 1, b - __half2float(__float2half_rn(b)));
}

// fp32 parameter blob -> fp16 weight / bias tiles, the all-ones A tile
template <bool SPLIT>
__device__ __forceinline__ void stage_weights(const float* __restrict__ p, unsigned char* smem) {
  for (uint32_t i = threadIdx.x; i < kOffBar / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0u;
  if (SPLIT)
    for (uint32_t i = threadIdx.x; i < (kSmemFwd - kOffB0L) / 4; i += blockDim.x)
      reinterpret_cast<uint32_t*>(smem + kOffB0L)[i] = 0u;
  __syncthreads();
  for (int i = threadIdx.x; i < kH * 32; i += blockDim.x)
    put_w<SPLIT>(smem, kOffB0, kOffB0L, 32, i >> 5, i & 31, __ldg(p + P::kW0 + i));
  for (int i = threadIdx.x; i < 16 * kH; i += blockDim.x)
    put_w<SPLIT>(smem, kOffB1, kOffB1L, 64, i >> 6, i & 63, __ldg(p + P::kW1 + i));
  // geo column c (1..15) of the head's first layer multiplies h[c] = in2[15 + c]; column 0 (the density logit) is 0
  for (int i = threadIdx.x; i < kH * 15; i += blockDim.x) {
    const int j = i / 15, c = i % 15;
    put_w<SPLIT>(smem, kOffB2, kOffB2L, 16, j, 1 + c, __ldg(p + P::kW2 + j * 63 + 16 + c));
  }
  for (int i = threadIdx.x; i < kH * kH; i += blockDim.x)
    put_w<SPLIT>(smem, kOffB3, kOffB3L, 64, i >> 6, i & 63, __ldg(p + P::kW3 + i));
  for (int i = threadIdx.x; i < 3 * kH; i += blockDim.x) put_b(smem, kOffB4, 64, i >> 6, i & 63, __ldg(p + P::kW4 + i));
  for (int i = threadIdx.x; i < 64; i += blockDim.x) {
    put_bias(smem, kOffBb0, i, __ldg(p + P::kB0 + i));
    put_bias(smem, kOffBb3, i, __ldg(p + P::kB3 + i));
    if (i < 16) put_bias(smem, kOffBb1, i, __ldg(p + P::kB1 + i));
    if (i < 3) put_bias(smem, kOffBb4, i, __ldg(p + P::kB4 + i));
  }
  for (int i = threadIdx.x; i < kTile; i += blockDim.x) {
    put_b(smem, kOffOnes, 16, i, 0, 1.f);
    put_b(smem, kOffOnes, 16, i, 1, 1.f);
  }
}

// bias of a forward layer: D[kColD .. +N) += the all-ones A tile . the bias tile^T (one SS-form MMA)
template <int N, bool BIAS>
__device__ __forceinline__ void issue_bias(uint32_t tmem, uint32_t sBe, uint32_t off_bias) {
  if (BIAS)
    mma_ss(tmem + kColD, smem_desc_at(sBe, kOffOnes, kLbo, sbo_of(16)), smem_desc_at(sBe, off_bias, kLbo, sbo_of(16)),
           instr_desc(kTile, N), 1u);
}
// forward layer: D[kColD .. +N) = A[kColA .. +K/2) . B^T (+ bias): K/16 TS-form MMAs + the bias MMA
// (sBe = smem_base_enc of the CTA's shared memory; all offsets are compile-time constants)
template <int N, int K, bool BIAS>
__device__ __forceinline__ void issue_fwd(uint32_t tmem, uint32_t sBe, uint32_t off_w, uint32_t off_bias) {
  issue_ts<N, K>(tmem + kColD, tmem + kColA, sBe, off_w, false);
  issue_bias<N, BIAS>(tmem, sBe, off_bias);
}
// split-precision forward layer: D = A_hi . Bhi^T + A_hi . Blo^T (+ A_lo . Bhi^T) (+ bias hi + lo)
template <int N, int K, bool BIAS, bool A_LO>
__device__ __forceinline__ void issue_fwd_split(uint32_t tmem, uint32_t sBe, uint32_t off_w, uint32_t off_w_lo,
                                                uint32_t off_bias) {
  issue_ts<N, K>(tmem + kColD, tmem + kColA, sBe, off_w, false);
  issue_ts<N, K>(tmem + kColD, tmem + kColA, sBe, off_w_lo, true);
  if (A_LO) issue_ts<N, K>(tmem + kColD, tmem + kColAlo, sBe, off_w, true);
  issue_bias<N, BIAS>(tmem, sBe, off_bias);
}

// accumulator row (fp32 bits, bias already added by the MMA) -> ReLU -> 16 packed fp16 pairs
__device__ __forceinline__ void relu_pack32(const uint32_t (&v)[32], uint32_t (&out)[16]) {
#pragma unroll
  for (int q = 0; q < 16; q++) out[q] = relu_h2(pack_h2(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])));
}
// the same with an fp32 per-row bias (the ray's bias row of the head's first layer)
__device__ __forceinline__ void bias_relu_pack32(const uint32_t (&v)[32], const float* bias, uint32_t (&out)[16]) {
#pragma unroll
  for (int q = 0; q < 8; q++) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + q);
    out[2 * q] = relu_h2(pack_h2(__uint_as_float(v[4 * q]) + b.x, __uint_as_float(v[4 * q + 1]) + b.y));
    out[2 * q + 1] = relu_h2(pack_h2(__uint_as_float(v[4 * q + 2]) + b.z, __uint_as_float(v[4 * q + 3]) + b.w));
  }
}
// gradient row masked by relu'(h) (h = the post-ReLU activation as 16 packed fp16 pairs) -> 16 packed pairs
__device__ __forceinline__ void mask_pack32(const uint32_t (&v)[32], const uint32_t (&h)[16], uint32_t (&out)[16]) {
  const __half2 zero = __float2half2_rn(0.f);
#pragma unroll
  for (int q = 0; q < 16; q++)
    out[q] = pack_h2(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])) &
             __hgt2_mask(*reinterpret_cast<const __half2*>(&h[q]), zero);
}

// relu_masks: uint4 per (sample, column half): {mask h1, mask h2, mask h3, 0} -- written by the forward (may be
// NULL: render), read by the backward
// Registers (measured on the bench's sample count, r02e): the plain forward runs 4 CTAs per SM at 64 registers; the
// split forward 3 per SM at 80 with both accumulator halves in flight (0.497 ms; 4 per SM with 36 bytes of spills:
// 0.511); the backward modes 2 per SM uncapped (126 registers, 1.08 ms; capped at 112 -- what would leave room for a
// sampler CTA underneath -- 16-36 bytes of spills cost 0.11 ms, more than the overlap gives).
constexpr int kSplitCtas = 3;   // resident CTAs per SM of the split forward
constexpr int min_ctas(int mode) { return mode == kFwd ? 4 : mode == kFwdSplit ? kSplitCtas : 2; }
constexpr int max_regs(int mode) { return mode == kFwd ? 64 : mode == kFwdSplit ? 80 : 128; }
template <int MODE>
__global__ void __launch_bounds__(kThreads, min_ctas(MODE)) __maxnreg__(max_regs(MODE))
mlp_tc_kernel(int64_t n, const int32_t* __restrict__ d_n_ptr, const float* __restrict__ params,
              const __half* __restrict__ feat, const int32_t* __restrict__ ray_id,
              const float* __restrict__ ray_bias, float* __restrict__ sigma, float* __restrict__ rgb,
              uint4* __restrict__ relu_masks, const float* __restrict__ d_sigma, const float* __restrict__ d_rgb,
              __half* __restrict__ d_feat, float* __restrict__ d_params, float* __restrict__ d_ray_bias, float gscale) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr bool WGRAD = MODE == kBwdFull;
  constexpr bool BWD = MODE == kBwdFull || MODE == kBwdFrozen;
  constexpr bool SPLIT = MODE == kFwdSplit;   // split-precision forward (see the header)
  constexpr uint32_t kCols = WGRAD ? 256u : 128u;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r = 32 * (warp & 3) + lane;  // row of the tile = TMEM lane
  const int hf = warp >> 2;              // column half
  const float inv_gscale = BWD ? 1.f / gscale : 1.f;
  stage_weights<SPLIT>(params, smem);
  const uint32_t bar = smem_u32(smem + kOffBar), bar_w = smem_u32(smem + kOffBarW);
  cta_alloc<kCols>(bar, bar_w, smem + kOffTmem);
  const uint32_t tmem = cta_publish(smem + kOffTmem);
  const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
  const uint32_t sBe = smem_base_enc(smem_u32(smem));
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);  // provably warp-uniform: the issue branch stays converged
  int* s_ray = reinterpret_cast<int*>(smem + kOffRay);
  if (d_n_ptr) {
    const int64_t dn = *d_n_ptr;
    n = dn < n ? dn : n;
  }
  uint32_t phase = 0, phase_w = 0;
  bool first_tile = true;
  const int64_t n_tiles = (n + kTile - 1) / kTile;
  // this thread's inputs of the CTA's NEXT tile are loaded one tile ahead into registers (a DRAM round trip at the
  // top of a tile would sit on the critical path of all 256 threads)
  // (backward modes: the forward runs 4 CTAs per SM at 64 registers and uses an L2 prefetch instead)
  constexpr bool kRegAhead = BWD;
  uint4 xn0 = make_uint4(0u, 0u, 0u, 0u), xn1 = xn0;
  int rayn = -1;
  if (kRegAhead) {
    const int64_t row0 = (int64_t)blockIdx.x * kTile + r;
    if (row0 < n) load_row(feat, ray_id, row0, hf, xn0, xn1, rayn);
  }
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t row = tile * kTile + r;
    const bool valid = row < n;
#ifdef GF_MLP_TRACE
    int tr_i = 0;
    GF_TR()
#endif
    int ray = rayn;
    uint4 x0 = xn0, x1 = xn1;
    // backward: the forward's ReLU masks of this thread's 32 columns (h1, h2, h3); first used half a tile from here
    uint4 mk = make_uint4(0u, 0u, 0u, 0u);
    if (BWD && valid) mk = __ldg(relu_masks + 2 * row + hf);
    if (!kRegAhead) {
      ray = -1;
      x0 = x1 = make_uint4(0u, 0u, 0u, 0u);
      if (valid) {
        const uint4* src = reinterpret_cast<const uint4*>(feat + row * 32 + 16 * hf);
        x0 = __ldg(src);
        x1 = __ldg(src + 1);
        ray = __ldg(ray_id + row);
      }
    }
    // the ray's bias row (b2 + W2[:, SH] SH(d) + W2[:, emb] emb), read in the epilogue of the head's first layer,
    // and the upstream gradients read at the turn to the backward half: towards L1 now
    const float* rb = ray_bias + (int64_t)(valid ? ray : 0) * kH + 32 * hf;
    // real loads instead of prefetch hints (r02ad: prefetch.global.L1 left the upstream-gradient loads at the turn to
    // the backward half on the critical path, ~1000 cycles of a 11 000-cycle tile; backward 1.11 -> 1.00 ms): one
    // 4-byte load pulls the thread's 128-byte bias line into L1 (its result is dead), and the four upstream
    // gradients of the row go to registers now (hf == 0 consumes them)
    float up[4] = {0.f, 0.f, 0.f, 0.f};
    if (valid) {
      float touch;
      asm volatile("ld.global.nc.f32 %0, [%1];\n" : "=f"(touch) : "l"(rb));
      if (BWD && hf == 0) {
        up[0] = __ldg(d_rgb + 3 * row);
        up[1] = __ldg(d_rgb + 3 * row + 1);
        up[2] = __ldg(d_rgb + 3 * row + 2);
        up[3] = __ldg(d_sigma + row);
      }
    }
    const int64_t nrow = row + (int64_t)gridDim.x * kTile;
    uint32_t h1p[16], h2p[16], h3p[16];  // post-ReLU activations of this thread's column half
    uint32_t m1 = 0u, m2 = 0u, m3 = 0u;  // forward: their ReLU masks
    float pre = 0.f;                      // density logit + 1 (hf == 0)
    // ---- input: features 16 hf .. 16 hf + 15 of this row -> A columns [8 hf, 8 hf + 8) (+ X tile) -------------
    {
      const uint32_t x[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
      if (WGRAD) {
        *tile_chunk(smem + kOffX, kSboX, r, 2 * hf) = x0;
        *tile_chunk(smem + kOffX, kSboX, r, 2 * hf + 1) = x1;
      }
      tmem_st8(lane_addr + kColA + 8 * hf, x);
      if (WGRAD && hf == 0) {
        store_ones(smem + kOffX, kSboX, r, 4);
        s_ray[r] = ray;
      }
      if (WGRAD && tid >= 128 && tid < 137) s_ray[tid] = tid == 136 ? 0 : -1;  // slot rays := none, bad flag := 0
    }
    // next tile's inputs: in flight during this whole tile
    xn0 = xn1 = make_uint4(0u, 0u, 0u, 0u);
    rayn = -1;
    if (nrow < n) {
      if (kRegAhead) {
        load_row(feat, ray_id, nrow, hf, xn0, xn1, rayn);
      } else {
        prefetch_l2(feat + nrow * 32 + 16 * hf);
        if ((lane & 7) == 0) prefetch_l2(ray_id + nrow);
      }
      if (BWD && (lane & 7) == 0) {  // its upstream gradients towards L2
        if (hf == 0) prefetch_l2(d_rgb + 3 * nrow);
        else prefetch_l2(d_sigma + nrow);
      }
      if (BWD && (lane & 3) == 0) prefetch_l2(relu_masks + 2 * nrow + hf);
    }
    if (SPLIT) {   // the input features ARE fp16 (the hash encoder's output): only the weights carry a lo part
      GF_TC_SYNC_ISSUE((issue_fwd_split<64, 32, true, false>(tmem, sBe, kOffB0, kOffB0L, kOffBb0)))
    } else {
      GF_TC_SYNC_ISSUE((issue_fwd<64, 32, true>(tmem, sBe, kOffB0, kOffBb0)))
    }
    GF_TC_WAIT()
    // ---- h1 = relu(acc) ----------------------------------------------------------------------------------
    if (SPLIT) {
      m1 = split_epilogue32<false, true, true>(lane_addr + kColD + 32 * hf, lane_addr + kColA + 16 * hf,
                                               lane_addr + kColAlo + 16 * hf, nullptr);
    } else {
      uint32_t v[32];
      tmem_ld32(lane_addr + kColD + 32 * hf, v);
      tmem_wait_ld();
      relu_pack32(v, h1p);
      tmem_st16(lane_addr + kColA + 16 * hf, h1p);
      if (WGRAD) {
        store_chunks<4>(smem + kOffH1, kSboH, r, 4 * hf, h1p);
        if (hf == 0) {
          store_ones(smem + kOffH1, kSboH, r, 8);
        } else {
          // One-hot "ray slot" row of this sample (slot = ray - the tile's first ray; rays are non-decreasing along
          // the samples): d ray_bias of the tile's rays is then G2^T . Ind, one more weight-gradient-shaped MMA,
          // instead of a CUDA-core reduction over the rows.  A tile whose rays do not fit 8 slots (runs of empty or
          // very short rays) raises the flag and takes the CUDA-core path below.
          const unsigned slot = (unsigned)(ray - s_ray[0]);
          uint32_t one = 0u;
          if (valid) {
            if (slot < 8u) {
              one = 0x3C00u << (16 * (slot & 1));  // fp16 1.0 in the slot's half of its 32-bit word
              if (r == 0 || s_ray[r - 1] != ray) s_ray[128 + slot] = ray;
            } else {
              s_ray[136] = 1;
            }
          }
          const unsigned wd = slot >> 1;
          *tile_chunk(smem + kOffInd, 128, r, 0) =
              make_uint4(wd == 0u ? one : 0u, wd == 1u ? one : 0u, wd == 2u ? one : 0u, wd == 3u ? one : 0u);
        }
      }
    }
    if (SPLIT) {
      GF_TC_SYNC_ISSUE((issue_fwd_split<16, 64, true, true>(tmem, sBe, kOffB1, kOffB1L, kOffBb1)))
    } else {
      GF_TC_SYNC_ISSUE((issue_fwd<16, 64, true>(tmem, sBe, kOffB1, kOffBb1)))
    }
    GF_TC_WAIT()
    // ---- h = acc; density = exp(h0 + 1); geo features -> A (16 fp16) ------------------------------------------
    if (hf == 0) {
      uint32_t v[16], a[8];
      tmem_ld16(lane_addr + kColD, v);
      tmem_wait_ld();
      pre = __uint_as_float(v[0]) + 1.f;
      if (!BWD && valid) sigma[row] = expf(pre);  // trunc_exp(h0 + 1), nerfacto_field.py:499
      if (SPLIT) {
        uint32_t al[8];
        float hh[16], hl[16];
#pragma unroll
        for (int j = 0; j < 16; j++) {
          const float x = __uint_as_float(v[j]);
          hh[j] = trunc11(x);
          hl[j] = x - hh[j];
        }
        hh[0] = hl[0] = 0.f;                                // column 0 of the geo tile has zero weights
#pragma unroll
        for (int j = 0; j < 8; j++) {
          a[j] = pack_h2(hh[2 * j], hh[2 * j + 1]);
          al[j] = pack_h2(hl[2 * j], hl[2 * j + 1]);
        }
        tmem_st8(lane_addr + kColAlo, al);
      } else {
        a[0] = pack_h2(0.f, __uint_as_float(v[1]));          // column 0 of the geo tile has zero weights
#pragma unroll
        for (int j = 1; j < 8; j++) a[j] = pack_h2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
      }
      tmem_st8(lane_addr + kColA, a);
      if (WGRAD) store_chunks<2>(smem + kOffHh, kSboS, r, 0, a);
    }
    if (SPLIT) {
      GF_TC_SYNC_ISSUE((issue_fwd_split<64, 16, false, true>(tmem, sBe, kOffB2, kOffB2L, 0u)))
    } else {
      GF_TC_SYNC_ISSUE((issue_fwd<64, 16, false>(tmem, sBe, kOffB2, 0u)))
    }
    GF_TC_WAIT()
    // ---- h2 = relu(acc + ray_bias[ray]) ----------------------------------------------------------------------
    if (SPLIT) {
      m2 = split_epilogue32<true, true, true>(lane_addr + kColD + 32 * hf, lane_addr + kColA + 16 * hf,
                                              lane_addr + kColAlo + 16 * hf, rb);
    } else {
      uint32_t v[32];
      tmem_ld32(lane_addr + kColD + 32 * hf, v);
      tmem_wait_ld();
      bias_relu_pack32(v, rb, h2p);
      tmem_st16(lane_addr + kColA + 16 * hf, h2p);
      if (WGRAD) {
        store_chunks<4>(smem + kOffH2, kSboH, r, 4 * hf, h2p);
        if (hf == 0) store_ones(smem + kOffH2, kSboH, r, 8);
      }
    }
    if (SPLIT) {
      GF_TC_SYNC_ISSUE((issue_fwd_split<64, 64, true, true>(tmem, sBe, kOffB3, kOffB3L, kOffBb3)))
    } else {
      GF_TC_SYNC_ISSUE((issue_fwd<64, 64, true>(tmem, sBe, kOffB3, kOffBb3)))
    }
    GF_TC_WAIT()
    // ---- h3 = relu(acc) ----------------------------------------------------------------------------------
    if (SPLIT) {
      // (no lo part: the output layer takes h3 as plain fp16 -- no ReLU follows it)
      m3 = split_epilogue32<false, false, true>(lane_addr + kColD + 32 * hf, lane_addr + kColA + 16 * hf, 0u, nullptr);
      if (relu_masks && valid) relu_masks[2 * row + hf] = make_uint4(m1, m2, m3, 0u);
    } else {
      uint32_t v[32];
      tmem_ld32(lane_addr + kColD + 32 * hf, v);
      tmem_wait_ld();
      relu_pack32(v, h3p);
      tmem_st16(lane_addr + kColA + 16 * hf, h3p);
      if (WGRAD) {
        store_chunks<4>(smem + kOffH3, kSboH, r, 4 * hf, h3p);
        if (hf == 0) store_ones(smem + kOffH3, kSboH, r, 8);
      }
    }
    GF_TC_SYNC_ISSUE((issue_fwd<16, 64, true>(tmem, sBe, kOffB4, kOffBb4)))
    GF_TC_WAIT()
    if (!BWD) {
      // ---- rgb = sigmoid(acc) --------------------------------------------------------------------------------
      if (hf == 0) {
        uint32_t v[4];
        tmem_ld4(lane_addr + kColD, v);
        tmem_wait_ld();
        if (valid) {
          rgb[3 * row] = sigmoidf_(__uint_as_float(v[0]));
          rgb[3 * row + 1] = sigmoidf_(__uint_as_float(v[1]));
          rgb[3 * row + 2] = sigmoidf_(__uint_as_float(v[2]));
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
          const float sg = sigmoidf_(__uint_as_float(v[c]));
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
    // g h3 = g o . W4 ; dW4^T (+ b4 row) += H3'^T . Go
    GF_TC_SYNC_ISSUE2((issue_dgrad<64, 16>(tmem + kColD, tmem + kColA, sBe, kOffB4, sbo_of(64))),
                      (issue_wgrad<128, 16>(tmem + kColW4, sBe, kOffH3, kSboH, kOffGo, kSboS, first_tile)))
    GF_TC_WAIT()
    {
      uint32_t v[32], g[16];
      tmem_ld32(lane_addr + kColD + 32 * hf, v);
      tmem_wait_ld();
      mask_bits_pack32(v, mk.z, g);
      tmem_st16(lane_addr + kColA + 16 * hf, g);
      GF_TC_WAIT_W()
      if (WGRAD) store_chunks<4>(smem + kOffH3, kSboG, r, 4 * hf, g);  // G3 over H3 (its readers have completed)
    }
    // g h2 = g h3 . W3 ; dW3 (+ b3 column) += G3^T . H2'
    GF_TC_SYNC_ISSUE2((issue_dgrad<64, 64>(tmem + kColD, tmem + kColA, sBe, kOffB3, sbo_of(64))),
                      (issue_wgrad<64, 72>(tmem + kColW3, sBe, kOffH3, kSboG, kOffH2, kSboH, first_tile)))
    GF_TC_WAIT()
    {
      uint32_t v[32], g[16];
      tmem_ld32(lane_addr + kColD + 32 * hf, v);
      tmem_wait_ld();
      mask_bits_pack32(v, mk.y, g);
      tmem_st16(lane_addr + kColA + 16 * hf, g);
      GF_TC_WAIT_W()
      if (WGRAD) store_chunks<4>(smem + kOffH2, kSboG, r, 4 * hf, g);  // G2 over H2
    }
    // g h[1:16] = g h2 . W2[:, geo] ; dW2[:, geo] += G2^T . Hh
    // (+ per-slot column sums of g h2 into the free accumulator columns 16..23: S[64 x 8] = G2^T . Ind)
    GF_TC_SYNC_ISSUE2((issue_dgrad<16, 64>(tmem + kColD, tmem + kColA, sBe, kOffB2, sbo_of(16)),
                       WGRAD ? issue_wgrad<64, 8>(tmem + kColD + 16, sBe, kOffH2, kSboG, kOffInd, 128, true) : (void)0),
                      (issue_wgrad<64, 16>(tmem + kColW2, sBe, kOffH2, kSboG, kOffHh, kSboS, first_tile)))
    const bool slots_ok = WGRAD && s_ray[136] == 0;
    if (WGRAD && !slots_ok) {
      // d ray_bias[ray] += column sums of g h2 over the rows of that ray (rows of a ray are contiguous), from the
      // G2 tile the MMAs are reading too.  Warp w sums rows 16 w .. 16 w + 15: lane = (row group of 4, chunk of 8
      // columns); 4 rows in fp16 pairs, then across the row groups with shuffles, fp32 from there.
      const int s0 = 16 * warp;
      if (s_ray[s0] == s_ray[s0 + 15]) {  // one ray (or all rows past the end): the common case
        const int j = lane & 7, rg = lane >> 3;
        __half2 acc[4];
        {
          const uint4 u = *tile_chunk(smem + kOffH2, kSboG, s0 + 4 * rg, j);
          acc[0] = *reinterpret_cast<const __half2*>(&u.x);
          acc[1] = *reinterpret_cast<const __half2*>(&u.y);
          acc[2] = *reinterpret_cast<const __half2*>(&u.z);
          acc[3] = *reinterpret_cast<const __half2*>(&u.w);
        }
#pragma unroll
        for (int k = 1; k < 4; k++) {
          const uint4 u = *tile_chunk(smem + kOffH2, kSboG, s0 + 4 * rg + k, j);
          acc[0] = __hadd2(acc[0], *reinterpret_cast<const __half2*>(&u.x));
          acc[1] = __hadd2(acc[1], *reinterpret_cast<const __half2*>(&u.y));
          acc[2] = __hadd2(acc[2], *reinterpret_cast<const __half2*>(&u.z));
          acc[3] = __hadd2(acc[3], *reinterpret_cast<const __half2*>(&u.w));
        }
        float f[8];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const float2 t = __half22float2(acc[k]);
          f[2 * k] = t.x;
          f[2 * k + 1] = t.y;
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {
          f[k] += __shfl_xor_sync(0xffffffffu, f[k], 8);
          f[k] += __shfl_xor_sync(0xffffffffu, f[k], 16);
        }
        const int rr = s_ray[s0];
        if (rg == 0 && rr >= 0) {
          float* dst = d_ray_bias + (int64_t)rr * kH + 8 * j;
#pragma unroll
          for (int k = 0; k < 8; k++)
            if (f[k] != 0.f) atomicAdd(dst + k, f[k] * inv_gscale);
        }
      } else {  // a ray boundary inside these 16 rows: lane = column pair, serial over the rows
        const unsigned char* g2 = smem + kOffH2 + (lane >> 2) * 128 + (lane & 3) * 4;
        float a0 = 0.f, a1 = 0.f;
        int cur = -1;
        for (int s2 = s0; s2 < s0 + 16; s2++) {
          const int rr = s_ray[s2];
          if (rr != cur) {
            if (cur >= 0) {
              atomicAdd(d_ray_bias + (int64_t)cur * kH + 2 * lane, a0 * inv_gscale);
              atomicAdd(d_ray_bias + (int64_t)cur * kH + 2 * lane + 1, a1 * inv_gscale);
            }
            cur = rr;
            a0 = a1 = 0.f;
          }
          const float2 t = __half22float2(*reinterpret_cast<const __half2*>(g2 + (s2 >> 3) * kSboG + (s2 & 7) * 16));
          a0 += t.x;
          a1 += t.y;
        }
        if (cur >= 0) {
          atomicAdd(d_ray_bias + (int64_t)cur * kH + 2 * lane, a0 * inv_gscale);
          atomicAdd(d_ray_bias + (int64_t)cur * kH + 2 * lane + 1, a1 * inv_gscale);
        }
      }
    }
    GF_TC_WAIT()
    if (slots_ok && hf == 1) {
      // d ray_bias[ray of slot s][o] += S[o][s]; M = 64 accumulator: row o = 16 (warp & 3) + lane, lane < 16
      uint32_t sv[8];
      tmem_ld8(lane_addr + kColD + 16, sv);
      tmem_wait_ld();
      if (lane < 16) {
        const int o = 16 * (warp & 3) + lane;
#pragma unroll
        for (int q = 0; q < 8; q++) {
          const int rr = s_ray[128 + q];
          const float f = __uint_as_float(sv[q]);
          if (rr >= 0 && f != 0.f) atomicAdd(d_ray_bias + (int64_t)rr * kH + o, f * inv_gscale);
        }
      }
    }
    // ---- g h = [ d sigma * exp(clamp(h0 + 1)) | acc[1:16] ] ---------------------------------------------------
    if (hf == 0) {
      uint32_t a[8];
      grad_h16(lane_addr + kColD, valid, up[3], gscale, pre, a);
      tmem_st8(lane_addr + kColA, a);
      if (WGRAD) store_chunks<2>(smem + kOffGo, kSboS, r, 0, a);  // Gh over Go (read by round 1's dW4 only)
    }
    GF_TC_WAIT_W()   // dW2's MMAs; every thread waits every phase of bar_w (the parity is tracked per thread)
    // g h1 = g h . W1 ; dW1^T (+ b1 row) += H1'^T . Gh
    GF_TC_SYNC_ISSUE2((issue_dgrad<64, 16>(tmem + kColD, tmem + kColA, sBe, kOffB1, sbo_of(64))),
                      (issue_wgrad<128, 16>(tmem + kColW1, sBe, kOffH1, kSboH, kOffGo, kSboS, first_tile)))
    GF_TC_WAIT()
    {
      uint32_t v[32], g[16];
      tmem_ld32(lane_addr + kColD + 32 * hf, v);
      tmem_wait_ld();
      mask_bits_pack32(v, mk.x, g);
      tmem_st16(lane_addr + kColA + 16 * hf, g);
      GF_TC_WAIT_W()
      if (WGRAD) store_chunks<4>(smem + kOffH1, kSboG, r, 4 * hf, g);  // G1 over H1
    }
    // g x = g h1 . W0 ; dW0 (+ b0 column) += G1^T . X'
    GF_TC_SYNC_ISSUE2((issue_dgrad<32, 64>(tmem + kColD, tmem + kColA, sBe, kOffB0, sbo_of(32))),
                      (issue_wgrad<64, 40>(tmem + kColW0, sBe, kOffH1, kSboG, kOffX, kSboX, first_tile)))
    GF_TC_WAIT()
    // ---- d feat -------------------------------------------------------------------------------------------------
    store_d_feat(lane_addr + kColD + 16 * hf, valid, inv_gscale, d_feat, row, hf);
    GF_TC_WAIT_W()   // dW0's MMAs read the X and G1 tiles the next tile overwrites (and the flush reads the sums)
    tc_fence_before();
    first_tile = false;
  }
  if (WGRAD && !first_tile) {
    // ---- flush the weight-gradient accumulators: one atomicAdd per parameter per CTA ------------------------------
    // (every MMA has completed: the last GF_TC_WAIT covered them)
    if (hf == 0) {
      // M = 64 accumulators live in lanes 0..15 of every 32-lane quadrant: row o = 16 (warp & 3) + lane (lane < 16)
      const int o = 16 * (warp & 3) + lane;
      const bool own = lane < 16;
      uint32_t v[32];
      // dW3 [o][0..63], b3[o] = column 64
#pragma unroll
      for (int part = 0; part < 2; part++) {
        tmem_ld32(lane_addr + kColW3 + 32 * part, v);
        tmem_wait_ld();
        if (own)
#pragma unroll
          for (int i = 0; i < 32; i++) {
            const float g = __uint_as_float(v[i]);
            if (g != 0.f) atomicAdd(d_params + P::kW3 + o * kH + 32 * part + i, g * inv_gscale);
          }
      }
      {
        uint32_t w[8];
        tmem_ld8(lane_addr + kColW3 + 64, w);
        tmem_wait_ld();
        if (own && __uint_as_float(w[0]) != 0.f) atomicAdd(d_params + P::kB3 + o, __uint_as_float(w[0]) * inv_gscale);
      }
      // dW0 [o][0..31], b0[o] = column 32
      tmem_ld32(lane_addr + kColW0, v);
      tmem_wait_ld();
      if (own)
#pragma unroll
        for (int i = 0; i < 32; i++) {
          const float g = __uint_as_float(v[i]);
          if (g != 0.f) atomicAdd(d_params + P::kW0 + o * 32 + i, g * inv_gscale);
        }
      {
        uint32_t w[8];
        tmem_ld8(lane_addr + kColW0 + 32, w);
        tmem_wait_ld();
        if (own && __uint_as_float(w[0]) != 0.f) atomicAdd(d_params + P::kB0 + o, __uint_as_float(w[0]) * inv_gscale);
      }
      // dW2 [o][geo c], c = 1..15 -> column 15 + c of W2
      {
        uint32_t w[16];
        tmem_ld16(lane_addr + kColW2, w);
        tmem_wait_ld();
        if (own)
#pragma unroll
          for (int c = 1; c < 16; c++) {
            const float g = __uint_as_float(w[c]);
            if (g != 0.f) atomicAdd(d_params + P::kW2 + o * 63 + 15 + c, g * inv_gscale);
          }
      }
      // dW1^T, dW4^T: M = 128, lane = input feature i (rows 0..63), row 64 = the bias
      {
        uint32_t w[16];
        tmem_ld16(lane_addr + kColW1, w);
        tmem_wait_ld();
        const int i = r;
        if (i <= 64)
#pragma unroll
          for (int oo = 0; oo < 16; oo++) {
            const float g = __uint_as_float(w[oo]);
            if (g != 0.f) atomicAdd(i < 64 ? d_params + P::kW1 + oo * kH + i : d_params + P::kB1 + oo, g * inv_gscale);
          }
        tmem_ld16(lane_addr + kColW4, w);
        tmem_wait_ld();
        if (i <= 64)
#pragma unroll
          for (int oo = 0; oo < 3; oo++) {
            const float g = __uint_as_float(w[oo]);
            if (g != 0.f) atomicAdd(i < 64 ? d_params + P::kW4 + oo * kH + i : d_params + P::kB4 + oo, g * inv_gscale);
          }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kCols);
}
}  // namespace tc
}  // namespace gf

#ifdef GF_MLP_TRACE
extern "C" int gf_debug_mlp_trace(unsigned long long* host128) {
  return cudaMemcpyFromSymbol(host128, gf::tc::g_mlp_trace, sizeof(unsigned long long) * 128) == cudaSuccess ? 0 : 1;
}
#endif

using namespace gf;

// Shared-memory request per mode.  It also caps residency so that the CTAs of one SM never ask for more than its
// 512 TMEM columns (a CTA beyond that would sit in tcgen05.alloc until another one exits):
// 128-column modes: 52 KB -> at most 4 CTAs per SM; full backward: ~102 KB (its tiles) -> 2 CTAs per SM.
static constexpr int kSmemSmall = 52 * 1024;
static_assert(tc::kSmemFwd <= kSmemSmall, "forward smem");

// launched by gf_mlp_forward / gf_mlp_backward (mlp.cu)
int gf_launch_mlp_fwd_tc(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                         const int32_t* ray_id, const float* ray_bias, float* sigma, float* rgb, void* relu_masks,
                         cudaStream_t st) {
  int rc = set_smem_attrs<tc::kH>(tc::mlp_tc_kernel<tc::kFwd>, tc::mlp_tc_kernel<tc::kBwdFrozen>,
                                  tc::mlp_tc_kernel<tc::kBwdFull>, tc::mlp_tc_kernel<tc::kFwdSplit>,
                                  {kSmemSmall, kSmemSmall, (int)tc::kSmemFull, kSmemSmall});
  if (rc) return rc;
  const int64_t tiles = div_up(n, tc::kTile);
  if (relu_masks) {   // training: split precision + the ReLU masks for gf_mlp_backward
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * tc::kSplitCtas);
    tc::mlp_tc_kernel<tc::kFwdSplit><<<grid, tc::kThreads, kSmemSmall, st>>>(
        n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, sigma, rgb, (uint4*)relu_masks, nullptr, nullptr,
        nullptr, nullptr, nullptr, 1.f);
    return check_launch("mlp_tc_kernel<fwd split>");
  }
  const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * 4);
  tc::mlp_tc_kernel<tc::kFwd><<<grid, tc::kThreads, kSmemSmall, st>>>(
      n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, sigma, rgb, nullptr, nullptr, nullptr, nullptr,
      nullptr, nullptr, 1.f);
  return check_launch("mlp_tc_kernel<fwd>");
}

int gf_launch_mlp_bwd_tc(int64_t n, const int32_t* d_n_ptr, const float* params, const void* feat_f16,
                         const int32_t* ray_id, const float* ray_bias, const void* relu_masks, const float* d_sigma,
                         const float* d_rgb, void* d_feat, float* d_params, float* d_ray_bias, float gscale,
                         cudaStream_t st) {
  int rc = set_smem_attrs<tc::kH>(tc::mlp_tc_kernel<tc::kFwd>, tc::mlp_tc_kernel<tc::kBwdFrozen>,
                                  tc::mlp_tc_kernel<tc::kBwdFull>, tc::mlp_tc_kernel<tc::kFwdSplit>,
                                  {kSmemSmall, kSmemSmall, (int)tc::kSmemFull, kSmemSmall});
  if (rc) return rc;
  const int64_t tiles = div_up(n, tc::kTile);
  if (d_params) {
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * 2);
    tc::mlp_tc_kernel<tc::kBwdFull><<<grid, tc::kThreads, tc::kSmemFull, st>>>(
        n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, nullptr, nullptr, (uint4*)relu_masks, d_sigma,
        d_rgb, (__half*)d_feat, d_params, d_ray_bias, gscale);
  } else {  // frozen MLP (focal stage): dgrad only
    const int grid = (int)std::min<int64_t>(tiles, (int64_t)sm_count() * 2);
    tc::mlp_tc_kernel<tc::kBwdFrozen><<<grid, tc::kThreads, kSmemSmall, st>>>(
        n, d_n_ptr, params, (const __half*)feat_f16, ray_id, ray_bias, nullptr, nullptr, (uint4*)relu_masks, d_sigma,
        d_rgb, (__half*)d_feat, nullptr, nullptr, gscale);
  }
  return check_launch("mlp_tc_kernel<bwd>");
}
