// What the tcgen05 field-MLP kernels (mlp_tc.cu: H = 64, mlp_tc128.cu: H = 128) share: the parameter blob layout,
// fp16 packing, the ReLU-mask bit layout, the no-swizzle core-matrix tile addressing of weights and [sample][feature]
// tiles, the MMA issue helpers and issue / commit / wait macros, the split-precision epilogue, the CTA prologue, the
// backward's density-gradient and d-feat blocks, and the shared-memory opt-in of the launchers.
#pragma once
#include <atomic>

#include "common.cuh"
#include "tcgen05.cuh"

namespace gf {

// parameter blob offsets (torch nn.Linear layout), see include/gfnerf_b200.h
template <int H>
struct Blob {
  static constexpr int kW0 = 0, kB0 = kW0 + H * 32, kW1 = kB0 + H, kB1 = kW1 + 16 * H, kW2 = kB1 + 16,
                       kB2 = kW2 + H * 63, kW3 = kB2 + H, kB3 = kW3 + H * H, kW4 = kB3 + H, kB4 = kW4 + 3 * H,
                       kParamCount = kB4 + 3;
};

namespace tc {

constexpr int kTile = 128;  // samples per CTA tile = MMA M
constexpr int kThreads = 256;

// kFwd: plain fp16 forward (inference: no gradients, no masks).  kFwdSplit: the split-precision training forward that
// also writes the ReLU masks the backward modes consume.
enum Mode { kFwd = 0, kBwdFrozen = 1, kBwdFull = 2, kFwdSplit = 3 };

// B operands: [N rows][K] fp16, K-major, no swizzle: element (n, k) at
//   (n / 8) * SBO + (k / 8) * 128 + (n % 8) * 16 + (k % 8) * 2,   SBO = (K / 8) * 128
constexpr uint32_t kLbo = 128;
constexpr uint32_t sbo_of(int K) { return (uint32_t)(K / 8) * 128u; }

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t relu_h2(uint32_t v) {
  __half2 h = __hmax2(*reinterpret_cast<__half2*>(&v), __float2half2_rn(0.f));
  return *reinterpret_cast<uint32_t*>(&h);
}
// two fp32 -> packed fp16 pair with ReLU in the conversion (cvt.rn.relu.f16x2.f32: first source = upper half)
__device__ __forceinline__ uint32_t pack_relu_h2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;\n" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
// fp32 -> fp16 hi + fp16 lo: hi = the value truncated to 11 significant bits (exact in fp16), lo = the rest
__device__ __forceinline__ float trunc11(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }
// bits of the ReLU-mask word for the pair (2q, 2q+1) of a thread's 32 columns: chosen so that the backward expands
// them to a half2 AND-mask with one shift + one PRMT in sign-replicating mode (mask_bits_pack32)
__host__ __device__ constexpr uint32_t mask_bits_of_pair(int q) {
  return q < 8 ? ((1u << (7 - q)) | (1u << (23 - q))) : ((1u << (15 - (q - 8))) | (1u << (31 - (q - 8))));
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }

__device__ __forceinline__ void put_b(unsigned char* smem, uint32_t off, int K, int n, int k, float v) {
  *reinterpret_cast<__half*>(smem + off + (n >> 3) * sbo_of(K) + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2) =
      __float2half_rn(v);
}
// v -> fp16 hi tile (and, SPLIT, the fp16 remainder into the lo tile at off_lo)
template <bool SPLIT>
__device__ __forceinline__ void put_w(unsigned char* smem, uint32_t off, uint32_t off_lo, int K, int n, int k, float v) {
  put_b(smem, off, K, n, k, v);
  if (SPLIT) put_b(smem, off_lo, K, n, k, v - __half2float(__float2half_rn(v)));
}


// 16-byte chunk j (features 8 j .. 8 j + 7) of row r of a [sample][feature] tile
__device__ __forceinline__ uint4* tile_chunk(unsigned char* buf, uint32_t sbo, int r, int j) {
  return reinterpret_cast<uint4*>(buf + (r >> 3) * sbo + j * 128 + (r & 7) * 16);
}
template <int NCH>
__device__ __forceinline__ void store_chunks(unsigned char* buf, uint32_t sbo, int r, int j0, const uint32_t* a) {
#pragma unroll
  for (int q = 0; q < NCH; q++)
    *tile_chunk(buf, sbo, r, j0 + q) = make_uint4(a[4 * q], a[4 * q + 1], a[4 * q + 2], a[4 * q + 3]);
}
__device__ __forceinline__ void store_ones(unsigned char* buf, uint32_t sbo, int r, int j) {
  *tile_chunk(buf, sbo, r, j) = make_uint4(0x00003C00u, 0u, 0u, 0u);  // feature 8 j = 1.0, the rest 0
}

// this thread's inputs of a row: its 16 features (16 hf .. 16 hf + 15, fp16) and the row's ray
__device__ __forceinline__ void load_row(const __half* feat, const int32_t* ray_id, int64_t row, int hf, uint4& x0,
                                         uint4& x1, int& ray) {
  const uint4* src = reinterpret_cast<const uint4*>(feat + row * 32 + 16 * hf);
  x0 = __ldg(src);
  x1 = __ldg(src + 1);
  ray = __ldg(ray_id + row);
}

// ---- MMA issue (one thread) --------------------------------------------------------------------------------------
// D[d .. +N) (+)= A[a .. +K/2) (TMEM, fp16 pairs) . B^T, B = [N][K] K-major tile at off_w: K/16 TS-form MMAs
template <int N, int K>
__device__ __forceinline__ void issue_ts(uint32_t d, uint32_t a, uint32_t sBe, uint32_t off_w, bool accumulate) {
  constexpr uint32_t idesc = instr_desc(kTile, N);
#pragma unroll
  for (int k = 0; k < K / 16; k++)
    mma_ts(d, a + 8 * k, smem_desc_at(sBe, off_w + 2 * k * kLbo, kLbo, sbo_of(K)), idesc, (k > 0 || accumulate) ? 1u : 0u);
}
// dgrad layer: D[128 x N] = G[128 x K] (TMEM at a) . W[K x N], W = the forward tile [K = out][N = in] read MN-major
template <int N, int K>
__device__ __forceinline__ void issue_dgrad(uint32_t d, uint32_t a, uint32_t sBe, uint32_t off_w, uint32_t sbo_fwd) {
  constexpr uint32_t idesc = instr_desc(kTile, N, 0, 1);
#pragma unroll
  for (int k = 0; k < K / 16; k++)
    mma_ts(d, a + 8 * k, smem_desc_at(sBe, off_w + 2 * k * sbo_fwd, sbo_fwd, 128), idesc, k > 0);
}
// wgrad: D[M x N] (+)= P^T . Q over the tile's 128 samples; P, Q = [sample][feature] tiles (SBO sp / sq), MN-major
template <int M, int N>
__device__ __forceinline__ void issue_wgrad(uint32_t d_tmem, uint32_t sBe, uint32_t off_p, uint32_t sp, uint32_t off_q,
                                            uint32_t sq, bool first_tile) {
  constexpr uint32_t idesc = instr_desc(M, N, 1, 1);
#pragma unroll
  for (int k = 0; k < kTile / 16; k++)
    mma_ss(d_tmem, smem_desc_at(sBe, off_p + 2 * k * sp, sp, 128), smem_desc_at(sBe, off_q + 2 * k * sq, sq, 128), idesc,
           (k > 0 || !first_tile) ? 1u : 0u);
}

// GF_TR(): a phase mark of mlp_tc.cu's profiling build (it defines the macro under GF_MLP_TRACE); nothing otherwise
#ifndef GF_TR
#define GF_TR()
#endif

// The macros below use the kernel's locals warp_u (warp-uniform warp index), bar / phase (dgrad completion) and, in
// the backward, WGRAD, bar_w / phase_w (weight-gradient completion).
// publish this thread's TMEM / shared-memory writes, let one thread issue the MMAs, wait for their completion
#define GF_TC_SYNC_ISSUE(ISSUE) \
  GF_TR()                       \
  tmem_wait_st();               \
  tc_fence_before();            \
  fence_proxy_async();          \
  __syncthreads();              \
  GF_TR()                       \
  if (warp_u == 0) {            \
    if (elect_one()) {          \
      tc_fence_after();         \
      ISSUE;                    \
      mma_commit(bar);          \
    }                           \
    __syncwarp();               \
  }                             \
  GF_TR()
#define GF_TC_WAIT()     \
  mbar_wait(bar, phase); \
  phase ^= 1;            \
  tc_fence_after();      \
  GF_TR()
// backward round: the dgrad MMAs (whose result the epilogue needs) and the weight-gradient MMAs (which only have to
// finish before their shared-memory operands are overwritten) are committed to different barriers, so the
// weight-gradient MMAs run underneath the epilogue's tcgen05.ld / pack / tcgen05.st
#define GF_TC_SYNC_ISSUE2(ISSUE_D, ISSUE_W) \
  GF_TR()                                   \
  tmem_wait_st();                           \
  tc_fence_before();                        \
  fence_proxy_async();                      \
  __syncthreads();                          \
  GF_TR()                                   \
  if (warp_u == 0) {                        \
    if (elect_one()) {                      \
      tc_fence_after();                     \
      ISSUE_D;                              \
      mma_commit(bar);                      \
      if (WGRAD) {                          \
        ISSUE_W;                            \
        mma_commit(bar_w);                  \
      }                                     \
    }                                       \
    __syncwarp();                           \
  }                                         \
  GF_TR()
#define GF_TC_WAIT_W()         \
  if (WGRAD) {                 \
    mbar_wait(bar_w, phase_w); \
    phase_w ^= 1;              \
  }                            \
  GF_TR()

// ---- epilogues ---------------------------------------------------------------------------------------------------
// split-precision epilogue of one 32-column chunk: accumulator at d_addr (+ an fp32 bias row: through the read-only
// cache if BIAS_LDG, else a plain load, which may be from shared memory) -> ReLU -> fp16 hi (and lo) pairs written
// back to TMEM at a_addr (alo_addr) as the next layer's A operand(s); returns the chunk's ReLU-mask word.  Both
// 16-column halves are loaded before the first wait.
template <bool WITH_BIAS, bool WITH_LO, bool BIAS_LDG>
__device__ __forceinline__ uint32_t split_epilogue32(uint32_t d_addr, uint32_t a_addr, uint32_t alo_addr,
                                                     const float* bias) {
  const __half2 zero = __float2half2_rn(0.f);
  uint32_t m = 0u;
  uint32_t vv[2][16];
  tmem_ld16(d_addr, vv[0]);
  tmem_ld16(d_addr + 16, vv[1]);
  tmem_wait_ld();
#pragma unroll
  for (int part = 0; part < 2; part++) {
    uint32_t hi[8], lo[8];
    const uint32_t (&v)[16] = vv[part];
#pragma unroll
    for (int q4 = 0; q4 < 4; q4++) {
      float x[4] = {__uint_as_float(v[4 * q4]), __uint_as_float(v[4 * q4 + 1]), __uint_as_float(v[4 * q4 + 2]),
                    __uint_as_float(v[4 * q4 + 3])};
      if (WITH_BIAS) {   // (an unconditional "+ 0.f" would not fold: -0.f + 0.f)
        const float4* b4 = reinterpret_cast<const float4*>(bias + 16 * part + 4 * q4);
        const float4 b = BIAS_LDG ? __ldg(b4) : *b4;
        x[0] += b.x;
        x[1] += b.y;
        x[2] += b.z;
        x[3] += b.w;
      }
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const float a = x[2 * e], c = x[2 * e + 1];
        if (WITH_LO) {
          const float ah = trunc11(a), ch = trunc11(c);
          hi[2 * q4 + e] = pack_relu_h2(ah, ch);
          // the remainder has the sign of the value: the conversion's ReLU zeroes it together with the hi part
          lo[2 * q4 + e] = pack_relu_h2(a - ah, c - ch);
        } else {
          hi[2 * q4 + e] = pack_relu_h2(a, c);   // no lo part wanted: plain round-to-nearest fp16
        }
        m |= __hgt2_mask(*reinterpret_cast<const __half2*>(&hi[2 * q4 + e]), zero) &
             mask_bits_of_pair(8 * part + 2 * q4 + e);
      }
    }
    tmem_st8(a_addr + 8 * part, hi);
    if (WITH_LO) tmem_st8(alo_addr + 8 * part, lo);
  }
  return m;
}

// gradient row masked by the forward's ReLU-mask word -> 16 packed pairs.  Pair q < 8: its two bits sit at 7 - q and
// 23 - q, so after a left shift by q they are the sign bits of bytes 0 and 2, which PRMT (selector nibble | 8 =
// replicate the byte's sign) spreads over the two halves; pairs 8..15 use bytes 1 and 3.
__device__ __forceinline__ void mask_bits_pack32(const uint32_t (&v)[32], uint32_t mask, uint32_t (&out)[16]) {
#pragma unroll
  for (int q = 0; q < 16; q++) {
    uint32_t sel;   // (__byte_perm only takes 3-bit selectors; the sign-replicate bit needs the PTX form)
    asm("prmt.b32 %0, %1, %2, %3;\n" : "=r"(sel) : "r"(mask << (q & 7)), "r"(0u), "r"(q < 8 ? 0xAA88u : 0xBB99u));
    out[q] = pack_h2(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])) & sel;
  }
}

// g h = [ d sigma * exp(clamp(h0 + 1)) | acc[1:16] ] as 8 packed pairs: the density column through trunc_exp, the
// geo columns' dgrad from the accumulator at d_addr
__device__ __forceinline__ void grad_h16(uint32_t d_addr, bool valid, float d_sigma, float gscale, float pre,
                                         uint32_t (&a)[8]) {
  uint32_t v[16];
  tmem_ld16(d_addr, v);
  tmem_wait_ld();
  // _TruncExp.backward: g * exp(clamp(x, -15, 15))  (nerfstudio/field_components/activations.py:33-36)
  const float g0 = valid ? d_sigma * gscale * expf(fminf(fmaxf(pre, -15.f), 15.f)) : 0.f;
  a[0] = pack_h2(g0, __uint_as_float(v[1]));
#pragma unroll
  for (int j = 1; j < 8; j++) a[j] = pack_h2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
}

// d feat of this thread's 16 features of the row (accumulator at d_addr), handed to the hash backward as
// fp16(g * 128) (Hash3DAnchored_cuda.cu:209)
__device__ __forceinline__ void store_d_feat(uint32_t d_addr, bool valid, float inv_gscale, __half* d_feat, int64_t row,
                                             int hf) {
  uint32_t v[16];
  tmem_ld16(d_addr, v);
  tmem_wait_ld();
  if (valid) {
    const float sc = GF_GRAD_SCALE * inv_gscale;
    uint4* dst = reinterpret_cast<uint4*>(d_feat + row * 32 + 16 * hf);
#pragma unroll
    for (int q = 0; q < 2; q++)
      dst[q] = make_uint4(pack_h2(__uint_as_float(v[8 * q]) * sc, __uint_as_float(v[8 * q + 1]) * sc),
                          pack_h2(__uint_as_float(v[8 * q + 2]) * sc, __uint_as_float(v[8 * q + 3]) * sc),
                          pack_h2(__uint_as_float(v[8 * q + 4]) * sc, __uint_as_float(v[8 * q + 5]) * sc),
                          pack_h2(__uint_as_float(v[8 * q + 6]) * sc, __uint_as_float(v[8 * q + 7]) * sc));
  }
}

// ---- CTA prologue ------------------------------------------------------------------------------------------------
// Tile-independent set-up once the weights are in shared memory, in two steps so that constant parts of the
// [sample][feature] tiles can be written in between: cta_alloc inits the two mbarriers (dgrad and weight-gradient MMA
// completion) and lets warp 0 allocate kCols TMEM columns; cta_publish makes the shared-memory writes visible to the
// MMA and returns the TMEM base address.
template <uint32_t kCols>
__device__ __forceinline__ void cta_alloc(uint32_t bar, uint32_t bar_w, unsigned char* tmem_slot) {
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    mbar_init(bar_w, 1);
    fence_mbar_init();
  }
  if (threadIdx.x < 32) {
    __syncwarp();
    tmem_alloc(smem_u32(tmem_slot), kCols);
  }
}
__device__ __forceinline__ uint32_t cta_publish(const unsigned char* tmem_slot) {
  fence_proxy_async();  // the tiles were written through the generic proxy; the MMA reads them through the async proxy
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return *reinterpret_cast<const volatile uint32_t*>(tmem_slot);
}

}  // namespace tc

// ---- host: shared-memory opt-in ------------------------------------------------------------------------------------
// Raises the dynamic shared-memory limit of the four instantiations of the width-H kernel, given in Mode order, to
// smem[mode].  The opt-in is per device (context), and one process may drive several: it is remembered per device
// ordinal.
template <int H, class Kernel>
int set_smem_attrs(Kernel fwd, Kernel bwd_frozen, Kernel bwd_full, Kernel fwd_split, const int (&smem)[4]) {
  const Kernel kernels[4] = {fwd, bwd_frozen, bwd_full, fwd_split};
  static std::atomic<bool> done_dev[64];
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  const bool track = dev >= 0 && dev < 64;
  if (!track || !done_dev[dev].load(std::memory_order_acquire)) {
    for (int m = 0; m < 4; m++)
      GF_CUDA(cudaFuncSetAttribute(kernels[m], cudaFuncAttributeMaxDynamicSharedMemorySize, smem[m]));
    if (track) done_dev[dev].store(true, std::memory_order_release);
  }
  return GF_OK;
}

}  // namespace gf
