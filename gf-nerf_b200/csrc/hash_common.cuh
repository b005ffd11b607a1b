// Device helpers of the Hash3DAnchored encode (cell / corner rows / weights, and one level of the backward scatter)
// used by the kernels of hash3d.cu.  Arithmetic follows the oracle's FMA convention exactly (oracle/gf_oracle.c);
// line references are to the reference's field/Hash3DAnchored_cuda.cu.
#pragma once
#include "common.cuh"

namespace gf {

// First table ROW of level l.  The reference's kernels offset the table pointer by feat_local_idx[l] = l * local_size
// (Hash3DAnchored.cpp:66-70) while that pointer is a pointer to SCALARS (`T* feat_pool`, Hash3DAnchored_cuda.cu:38,
// :105), and then index it with pos * N_CHANNELS + k: level l's window therefore starts at row l * local_size / 2 and
// is local_size rows long -- consecutive levels overlap by half a window and rows >= 8.5 * local_size are never
// touched.  Found by running the reference's own kernel bodies on the host (oracle/ref_driver.cpp); reproduced here
// because a table trained by the reference is only meaningful under this addressing.  local_size is even (the
// reference rounds it to a multiple of 16); the C-ABI rejects odd sizes.
__host__ __device__ __forceinline__ int64_t level_base_row(int l, uint32_t local_size) {
  return ((int64_t)l * (int64_t)local_size) >> 1;
}

template <bool POW2>
__device__ __forceinline__ uint32_t wrap(uint32_t h, uint32_t local_size) {
  if (POW2) return h & (local_size - 1u);
  return h % local_size;
}

struct Cell {
  uint32_t px, py, pz;
  float a, b, c;
};

// :26-46  pt*mul + bias, floor, fractional part.  bias == nullptr: an all-zero bias pool (what the reference always
// has, Hash3DAnchored.cpp:57-62), same arithmetic without the three loads.
__device__ __forceinline__ Cell cell_of(float x, float y, float z, float mul, const float* __restrict__ bias) {
  float p0 = __fmaf_rn(x, mul, bias ? __ldg(bias + 0) : 0.f);
  float p1 = __fmaf_rn(y, mul, bias ? __ldg(bias + 1) : 0.f);
  float p2 = __fmaf_rn(z, mul, bias ? __ldg(bias + 2) : 0.f);
  float f0 = floorf(p0), f1 = floorf(p1), f2 = floorf(p2);
  Cell c;
  c.px = __float2uint_rz(f0);  // saturating, negative/NaN -> 0
  c.py = __float2uint_rz(f1);
  c.pz = __float2uint_rz(f2);
  c.a = __fsub_rn(p0, f0);
  c.b = __fsub_rn(p1, f1);
  c.c = __fsub_rn(p2, f2);
  return c;
}

// :48-55 corner rows, order 000,001,010,011,100,101,110,111 (bits x,y,z)
template <bool POW2>
__device__ __forceinline__ void corners(const Cell& c, uint32_t pa, uint32_t pb, uint32_t pc, uint32_t local_size,
                                        uint32_t (&pos)[8]) {
  uint32_t x0 = c.px * pa, x1 = (c.px + 1u) * pa;
  uint32_t y0 = c.py * pb, y1 = (c.py + 1u) * pb;
  uint32_t z0 = c.pz * pc, z1 = (c.pz + 1u) * pc;
  pos[0] = wrap<POW2>(x0 ^ y0 ^ z0, local_size);
  pos[1] = wrap<POW2>(x0 ^ y0 ^ z1, local_size);
  pos[2] = wrap<POW2>(x0 ^ y1 ^ z0, local_size);
  pos[3] = wrap<POW2>(x0 ^ y1 ^ z1, local_size);
  pos[4] = wrap<POW2>(x1 ^ y0 ^ z0, local_size);
  pos[5] = wrap<POW2>(x1 ^ y0 ^ z1, local_size);
  pos[6] = wrap<POW2>(x1 ^ y1 ^ z0, local_size);
  pos[7] = wrap<POW2>(x1 ^ y1 ^ z1, local_size);
}

// :58-69 trilinear weights, products left to right
__device__ __forceinline__ void weights(const Cell& c, float (&w)[8]) {
  float ia = __fsub_rn(1.f, c.a), ib = __fsub_rn(1.f, c.b), ic = __fsub_rn(1.f, c.c);
  float iaib = __fmul_rn(ia, ib), iab = __fmul_rn(ia, c.b), aib = __fmul_rn(c.a, ib), ab = __fmul_rn(c.a, c.b);
  w[0] = __fmul_rn(iaib, ic);
  w[1] = __fmul_rn(iaib, c.c);
  w[2] = __fmul_rn(iab, ic);
  w[3] = __fmul_rn(iab, c.c);
  w[4] = __fmul_rn(aib, ic);
  w[5] = __fmul_rn(aib, c.c);
  w[6] = __fmul_rn(ab, ic);
  w[7] = __fmul_rn(ab, c.c);
}

// ---- backward scatter ---------------------------------------------------------------------------------------
// Shared-memory staging of the run reduction: one row per lane = 8 x {half2 contribution, u32 table row} (the
// contributions ARE fp16 values, :148-151), padded to 18 words: the 8-byte row writes of a half-warp and the 8-byte
// column reads of its two lane quarters each cover the 32 banks exactly once.  (r02y: 12 + 24 shared-memory
// wavefronts per warp and level with float2 contributions and separate rows -> 16 + 16.)
constexpr int kScatterRowWords = 18;
constexpr int kScatterWarpWords = 32 * kScatterRowWords;
// longest run of lanes the segmented shuffle reduction takes; longer runs go through shared memory
constexpr int kScatterShuffleMaxRun = 4;

// `keep` of a lane that issues reductions: a sum of +0 / -0 is skipped, it would not change the table
constexpr uint32_t kScatterKeep = 0x7fffffffu;

// red.global.add.v2.f32 of (s0, s1) (times 1 / GF_GRAD_SCALE when UNSCALE) to tab[row] unless (s0 | s1) & keep is
// zero; keep is kScatterKeep or 0 (a lane that writes nothing).  ptxas branches around a predicated reduction
// whatever the source form, so the cost per corner is one LOP3 for the predicate, one IMAD.WIDE for the address and
// the branch; the row is a 32-bit index into the level's 64-bit base.
template <bool UNSCALE>
__device__ __forceinline__ void red_add_f32x2(float2* tab, uint32_t row, float s0, float s1, uint32_t keep) {
  if ((__float_as_uint(s0) | __float_as_uint(s1)) & keep) {
    constexpr float out_scale = 1.f / GF_GRAD_SCALE;
    if (UNSCALE) {
      s0 = __fmul_rn(s0, out_scale);
      s1 = __fmul_rn(s1, out_scale);
    }
    // not atomicAdd: its unused result can still compile to an ATOM that returns the old value
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(tab + row), "f"(s0), "f"(s1) : "memory");
  }
}

// One level of the backward scatter for the 32 consecutive samples held by a warp (:81-155): recompute cell / corner
// rows / weights, quantise the 8 x 2 contributions like the reference (fp16(g * 128) times w, each product rounded to
// fp16, one F2FP per corner), then add them to the fp32 gradient table.  Lanes that fall into the same cell of the
// same volume (contiguous runs along the ray) are summed first; three warp-uniform paths by the longest run:
//   1        every lane issues its own 8 predicated vector reductions;
//   2..4     segmented shuffle reduction (1-2 steps, kScatterShuffleMaxRun), the run's first lane issues the reductions;
//   > 4      the contributions and rows go through shared memory and lane (corner d = lane & 7, quarter q = lane >> 3)
//            walks the 8 rows of its quarter in lane order, flushing its fp32 partial sum at every run boundary:
//            8 loads + 16 adds per lane whatever the run structure (a 5-step shuffle tree costs 80 + 80).
// gh: this sample's two gradients of the level as fp16(g * 128).  vol_head: lane 0, or the previous lane's sample is
// in another volume (the same at every level, so the caller shuffles it once).  Must be called by all 32 lanes.
// UNSCALE: the sums are divided by GF_GRAD_SCALE (:238); false leaves the table at the x128 scale for a caller that
// folds the division into its optimizer step (exact either way: a power of two).
template <bool POW2, bool HAS_BIAS, bool UNSCALE>
__device__ __forceinline__ void hash_scatter_level(int l, float x, float y, float z, int vol, bool vol_head, __half2 gh,
                                                   int lane, int32_t n_volumes, uint32_t local_size,
                                                   const int32_t* __restrict__ prim_pool,
                                                   const float* __restrict__ bias_pool, float scale,
                                                   float* __restrict__ grad_table, float* __restrict__ s_warp) {
  // every product of a zero gradient is zero and no reduction of this level would be issued
  if (!__any_sync(0xffffffffu, *reinterpret_cast<const uint32_t*>(&gh) & 0x7fff7fffu)) return;
  const int tr = (l * n_volumes + vol) * 3;
  const Cell c = cell_of(x, y, z, scale, HAS_BIAS ? bias_pool + tr : nullptr);
  const uint32_t pa = (uint32_t)__ldg(prim_pool + tr), pb = (uint32_t)__ldg(prim_pool + tr + 1),
                 pc = (uint32_t)__ldg(prim_pool + tr + 2);
  uint32_t pos[8];
  corners<POW2>(c, pa, pb, pc, local_size, pos);
  float w[8];
  weights(c, w);
  const float g0 = __low2float(gh), g1 = __high2float(gh);
  // gh is zero for a lane past the end; a zero gradient gives zero products, which are never written (:147)
  uint32_t cq[8];  // (__half)(g0 * w), (__half)(g1 * w) :148-151
#pragma unroll
  for (int d = 0; d < 8; d++) {
    const __half2 h = __floats2half2_rn(__fmul_rn(g0, w[d]), __fmul_rn(g1, w[d]));
    cq[d] = *reinterpret_cast<const uint32_t*>(&h);
  }
  // the level's first row as one 64-bit register: the opaque move keeps nvcc from folding the 64-bit base row into
  // every corner's address (4 instructions per reduction instead of one IMAD.WIDE.U32 of the 32-bit row)
  float2* tab = reinterpret_cast<float2*>(grad_table) + level_base_row(l, local_size);
  asm("mov.b64 %0, %0;" : "+l"(tab));
  const uint32_t ppx = __shfl_up_sync(0xffffffffu, c.px, 1), ppy = __shfl_up_sync(0xffffffffu, c.py, 1),
                 ppz = __shfl_up_sync(0xffffffffu, c.pz, 1);
  const bool head = vol_head || ppx != c.px || ppy != c.py || ppz != c.pz;
  const uint32_t heads = __ballot_sync(0xffffffffu, head);
  const uint32_t above = lane == 31 ? 0u : (heads & (0xffffffffu << (lane + 1)));
  const int end = above ? (__ffs(above) - 1) : 32;
  const int maxrun = (int)__reduce_max_sync(0xffffffffu, head ? (unsigned)(end - lane) : 0u);
  if (maxrun > kScatterShuffleMaxRun) {  // warp-uniform
    uint2* row = reinterpret_cast<uint2*>(s_warp + lane * kScatterRowWords);
#pragma unroll
    for (int d = 0; d < 8; d++) row[d] = make_uint2(cq[d], pos[d]);
    __syncwarp();
    const int d = lane & 7, j0 = lane & 24;
    // bit k: lane j0 + k is the last of its run or of its quarter
    const uint32_t stops = ((heads >> 1) | 0x80808080u) >> j0;
    float a0, a1;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const uint2 e = reinterpret_cast<const uint2*>(s_warp + (j0 + k) * kScatterRowWords)[d];
      const float2 v = __half22float2(*reinterpret_cast<const __half2*>(&e.x));
      a0 = k == 0 ? v.x : a0 + v.x;  // (not 0 + v: a -0 differs only in a zero sum, which is never written)
      a1 = k == 0 ? v.y : a1 + v.y;
      const bool stop = (stops >> k) & 1u;
      red_add_f32x2<UNSCALE>(tab, e.y, a0, a1, stop ? kScatterKeep : 0u);
      a0 = stop ? 0.f : a0;
      a1 = stop ? 0.f : a1;
    }
    __syncwarp();  // the rows are rewritten by the next level
    return;
  }
  float c0[8], c1[8];
#pragma unroll
  for (int d = 0; d < 8; d++) {
    const float2 v = __half22float2(*reinterpret_cast<const __half2*>(&cq[d]));
    c0[d] = v.x;
    c1[d] = v.y;
  }
  uint32_t keep = kScatterKeep;  // contributions of dead lanes are already zero
  if (maxrun > 1) {
    // two steps with fixed offsets: no loop whose trip count ptxas cannot prove uniform
    static_assert(kScatterShuffleMaxRun == 4, "offsets 1 and 2 cover runs of up to 4 lanes");
    auto step = [&](int off) {
      const bool take = lane + off < end;
#pragma unroll
      for (int d = 0; d < 8; d++) {
        const float o0 = __shfl_down_sync(0xffffffffu, c0[d], off);
        const float o1 = __shfl_down_sync(0xffffffffu, c1[d], off);
        if (take) {
          c0[d] += o0;
          c1[d] += o1;
        }
      }
    };
    step(1);
    if (maxrun > 2) step(2);
    keep = (heads >> lane) & 1u ? kScatterKeep : 0u;
  }
#pragma unroll
  for (int d = 0; d < 8; d++) red_add_f32x2<UNSCALE>(tab, pos[d], c0[d], c1[d], keep);
}

}  // namespace gf
