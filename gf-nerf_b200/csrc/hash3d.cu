// Hash3DAnchored encode: forward gather and backward scatter for sm_100a.
//
// Replaces Hash3DAnchoredForwardKernel / Hash3DAnchoredBackwardKernel and the
// host glue of Hash3DAnchoredFunction (reference gfnerf/bindings/field/
// Hash3DAnchored_cuda.cu:11-79, 81-155, 160-239).
//
// Design (DESIGN.md "hash encode"):
//  * one thread per sample walks all 16 levels, so the point, its anchor and the
//    per-(level,volume) primes are read once instead of 16x, and the 32 outputs
//    leave as four 16-byte stores of the fp16 values the reference computes anyway;
//  * lanes of a warp hold CONSECUTIVE samples of one ray (the sampler's compact
//    layout), so on coarse levels the 32 lanes of a gather hit the same few
//    32-byte sectors and the LSU coalesces them;
//  * the table is an fp16 shadow that is only re-cast when feat_pool changes,
//    not on every forward as the reference does (:185);
//  * backward: lanes that fall into the same grid cell (contiguous runs along the
//    ray) are summed first -- by a 1-2 step segmented shuffle reduction for short
//    runs, through shared memory for long ones -- and the run issues its 8
//    vectorised fp32 reductions (red.global.add.v2.f32) once (hash_common.cuh);
//    a level whose 32 quantised gradients are all zero is left after one vote.
//
// Arithmetic follows the oracle's FMA convention exactly (oracle/gf_oracle.c).
#include "common.cuh"
#include "hash_common.cuh"

namespace gf {

__global__ void level_scales_kernel(float* out) {
  int l = threadIdx.x;
  if (l < GF_N_LEVELS)  // the reference's expression, evaluated by the device's exp2f (:28)
    out[l] = exp2f((10.f - 3.f) * float(l) / float(GF_N_LEVELS - 1) + 3.f);
}

__global__ void cast_table_kernel(const float4* __restrict__ in, uint2* __restrict__ out, int64_t n4) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = __ldg(in + i);
    __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&lo);
    o.y = *reinterpret_cast<uint32_t*>(&hi);
    out[i] = o;
  }
}

__global__ void cast_table_tail_kernel(const float* __restrict__ in, __half* __restrict__ out, int64_t from, int64_t n) {
  int64_t i = from + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2half_rn(in[i]);
}

constexpr int kHashBlock = 256;
// Two register / scheduling variants of the forward gather (r02u, bench samples), chosen by hash_forward_impl:
//   PREFETCH = false  48 registers, 5 CTAs per SM: the most warps in flight -- best when the table does not fit the
//                     L2 and the gather waits on HBM (log2T = 23: 1.79 ms against 2.15 for the other one);
//   PREFETCH = true   the 32 gathers of a four-level group are all issued before the first is consumed, 79 registers,
//                     3 CTAs per SM -- best while the reachable rows fit the L2 and the kernel is bound by the L1 -> L2
//                     request path, not by DRAM latency (log2T = 19: 0.949 ms against 0.985; log2T = 21, 71 MB of
//                     rows: 0.970 against 1.338).
// The table a sample reads.  `OneTable`: every sample the same (hash_fwd_kernel).  `RoutedTables`: sample i takes
// table ray_table[ray_id[i]] of a device descriptor array (hash_fwd_routed_kernel); an id outside [0, n_tables)
// selects none, and the sample's base row is passed through.
struct OneTable {
  const __half2* __restrict__ feat;
  const int32_t* __restrict__ prim_pool;
  const float* __restrict__ bias_pool;
  __device__ __forceinline__ bool operator()(int64_t, const __half2*& f, const int32_t*& p, const float*& b) const {
    f = feat;
    p = prim_pool;
    b = bias_pool;
    return true;
  }
};

struct RoutedTables {
  const gf_hash_table_ref* __restrict__ tables;
  int32_t n_tables;
  const int32_t* __restrict__ ray_id;
  const int32_t* __restrict__ ray_table;
  __device__ __forceinline__ bool operator()(int64_t i, const __half2*& f, const int32_t*& p, const float*& b) const {
    const int32_t t = __ldg(ray_table + __ldg(ray_id + i));
    if ((uint32_t)t >= (uint32_t)n_tables) return false;
    f = reinterpret_cast<const __half2*>(__ldg(reinterpret_cast<const unsigned long long*>(&tables[t].feat_f16)));
    p = reinterpret_cast<const int32_t*>(__ldg(reinterpret_cast<const unsigned long long*>(&tables[t].prim_pool)));
    b = reinterpret_cast<const float*>(__ldg(reinterpret_cast<const unsigned long long*>(&tables[t].bias_pool)));
    return true;
  }
};

// The forward gather of hash_fwd_kernel and hash_fwd_routed_kernel: one thread per sample, all 16 levels.
template <bool POW2, typename AnchorT, bool OUT16, bool OUT32, bool PREFETCH, typename Tables>
__device__ __forceinline__ void hash_fwd_body(int64_t n, const int32_t* __restrict__ d_n_ptr, int32_t n_volumes,
                                              uint32_t local_size, const Tables& table,
                                              const float* __restrict__ scales, const float* __restrict__ pts,
                                              const AnchorT* __restrict__ anchors, uint4* __restrict__ out16,
                                              float4* __restrict__ out32, const uint4* __restrict__ base16) {
  if (d_n_ptr) {
    int64_t dn = *d_n_ptr;
    n = dn < n ? dn : n;
  }
  __shared__ float s_scale[GF_N_LEVELS];
  if (threadIdx.x < GF_N_LEVELS) s_scale[threadIdx.x] = __ldg(scales + threadIdx.x);
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const __half2* feat;
    const int32_t* prim_pool;
    const float* bias_pool;
    if (!table(i, feat, prim_pool, bias_pool)) {   // routed, no table: the base row unchanged
      if ((const void*)out16 != (const void*)base16) {
#pragma unroll
        for (int q = 0; q < GF_N_LEVELS / 4; q++) out16[i * 4 + q] = __ldg(base16 + i * 4 + q);
      }
      continue;
    }
    const float x = __ldg(pts + 3 * i), y = __ldg(pts + 3 * i + 1), z = __ldg(pts + 3 * i + 2);
    const int vol = (int)anchors[i];
#pragma unroll 1
    for (int q = 0; q < GF_N_LEVELS / 4; q++) {
      uint32_t packed[4];
      // this level's cell and the fp16 table rows of its eight corners
      auto gather = [&](int l, Cell& c, __half2 (&f)[8]) {
        const int tr = (l * n_volumes + vol) * 3;
        c = cell_of(x, y, z, s_scale[l], bias_pool ? bias_pool + tr : nullptr);
        const uint32_t pa = (uint32_t)__ldg(prim_pool + tr), pb = (uint32_t)__ldg(prim_pool + tr + 1),
                       pc = (uint32_t)__ldg(prim_pool + tr + 2);
        uint32_t pos[8];
        corners<POW2>(c, pa, pb, pc, local_size, pos);
        const __half2* tab = feat + level_base_row(l, local_size);
#pragma unroll
        for (int d = 0; d < 8; d++) f[d] = __ldg(tab + pos[d]);
      };
      // trilinear blend in fp32, rounded to fp16 (:58-77)
      auto blend = [](const Cell& c, const __half2 (&f)[8]) {
        float w[8];
        weights(c, w);
        // nvcc's contraction of w000*f000 + w001*f001 + ... (:73-77)
        float t0 = __fmul_rn(w[1], __low2float(f[1]));
        float t1 = __fmul_rn(w[1], __high2float(f[1]));
        t0 = __fmaf_rn(w[0], __low2float(f[0]), t0);
        t1 = __fmaf_rn(w[0], __high2float(f[0]), t1);
#pragma unroll
        for (int d = 2; d < 8; d++) {
          t0 = __fmaf_rn(w[d], __low2float(f[d]), t0);
          t1 = __fmaf_rn(w[d], __high2float(f[d]), t1);
        }
        const __half2 o = __floats2half2_rn(t0, t1);
        return *reinterpret_cast<const uint32_t*>(&o);
      };
      if (PREFETCH) {   // all 32 gathers of the group in flight before the first blend
        Cell cc[4];
        __half2 ff[4][8];
#pragma unroll
        for (int j = 0; j < 4; j++) gather(4 * q + j, cc[j], ff[j]);
#pragma unroll
        for (int j = 0; j < 4; j++) packed[j] = blend(cc[j], ff[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; j++) {
          Cell c;
          __half2 f[8];
          gather(4 * q + j, c, f);
          packed[j] = blend(c, f);
        }
      }
      if (base16) {  // focal stage: residual on top of the global encoder's features (nerfacto_field.py:477-489)
        const uint4 b = __ldg(base16 + i * 4 + q);
        const uint32_t bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; j++) {
          __half2 o = __hadd2(*reinterpret_cast<const __half2*>(&bb[j]), *reinterpret_cast<__half2*>(&packed[j]));
          packed[j] = *reinterpret_cast<uint32_t*>(&o);
        }
      }
      if (OUT16) out16[i * 4 + q] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
      if (OUT32) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
          __half2 h0 = *reinterpret_cast<__half2*>(&packed[2 * h]);
          __half2 h1 = *reinterpret_cast<__half2*>(&packed[2 * h + 1]);
          out32[i * 8 + 2 * q + h] = make_float4(__low2float(h0), __high2float(h0), __low2float(h1), __high2float(h1));
        }
      }
    }
  }
}

template <bool POW2, typename AnchorT, bool OUT16, bool OUT32, bool PREFETCH>
__global__ void __launch_bounds__(kHashBlock, PREFETCH ? 3 : 5)
hash_fwd_kernel(int64_t n, const int32_t* __restrict__ d_n_ptr, int32_t n_volumes, uint32_t local_size,
                const __half2* __restrict__ feat, const int32_t* __restrict__ prim_pool,
                const float* __restrict__ bias_pool, const float* __restrict__ scales,
                const float* __restrict__ pts, const AnchorT* __restrict__ anchors,
                uint4* __restrict__ out16, float4* __restrict__ out32, const uint4* __restrict__ base16) {
  hash_fwd_body<POW2, AnchorT, OUT16, OUT32, PREFETCH>(n, d_n_ptr, n_volumes, local_size,
                                                       OneTable{feat, prim_pool, bias_pool}, scales, pts, anchors,
                                                       out16, out32, base16);
}

// Residual gather with a table per sample (gf_hash_forward_residual_routed): fp16 output on top of base16 only.
// Same register budget and occupancy as hash_fwd_kernel's variant of the same PREFETCH.
template <bool POW2, typename AnchorT, bool PREFETCH>
__global__ void __launch_bounds__(kHashBlock, PREFETCH ? 3 : 5)
hash_fwd_routed_kernel(int64_t n, const int32_t* __restrict__ d_n_ptr, int32_t n_volumes, uint32_t local_size,
                       int32_t n_tables, const gf_hash_table_ref* __restrict__ tables,
                       const float* __restrict__ scales, const float* __restrict__ pts,
                       const AnchorT* __restrict__ anchors, const int32_t* __restrict__ ray_id,
                       const int32_t* __restrict__ ray_table, uint4* out16, const uint4* base16) {
  hash_fwd_body<POW2, AnchorT, true, false, PREFETCH>(n, d_n_ptr, n_volumes, local_size,
                                                      RoutedTables{tables, n_tables, ray_id, ray_table}, scales, pts,
                                                      anchors, out16, nullptr, base16);
}

// The table a sample's gradient goes to.  `OneGradTable`: every sample the same (hash_bwd_kernel).  `RoutedGradTables`:
// sample i takes table ray_table[ray_id[i]] of a device descriptor array (hash_bwd_routed_kernel); an id outside
// [0, n_tables) contributes nothing (the lane is treated like one past the end, with table 0's pools for its
// unused cell, and a run key of its own).  `key` is the table id that, with the volume, starts a new run.
struct OneGradTable {
  static constexpr bool kRouted = false;
  const int32_t* __restrict__ prim_pool;
  const float* __restrict__ bias_pool;
  float* __restrict__ grad_table;
  __device__ __forceinline__ bool operator()(int64_t, bool, const int32_t*& p, const float*& b, float*& g,
                                             int32_t&) const {
    p = prim_pool;
    b = bias_pool;
    g = grad_table;
    return true;
  }
};

struct RoutedGradTables {
  static constexpr bool kRouted = true;
  const gf_hash_grad_ref* __restrict__ tables;
  int32_t n_tables;
  const int32_t* __restrict__ ray_id;
  const int32_t* __restrict__ ray_table;
  __device__ __forceinline__ bool operator()(int64_t i, bool valid, const int32_t*& p, const float*& b, float*& g,
                                             int32_t& key) const {
    const int32_t t = valid ? __ldg(ray_table + __ldg(ray_id + i)) : -1;
    const bool ok = (uint32_t)t < (uint32_t)n_tables;
    key = ok ? t : -1;
    const gf_hash_grad_ref* r = tables + (ok ? t : 0);
    p = reinterpret_cast<const int32_t*>(__ldg(reinterpret_cast<const unsigned long long*>(&r->prim_pool)));
    b = reinterpret_cast<const float*>(__ldg(reinterpret_cast<const unsigned long long*>(&r->bias_pool)));
    g = reinterpret_cast<float*>(__ldg(reinterpret_cast<const unsigned long long*>(&r->grad_table)));
    return ok;
  }
};

// The backward scatter of hash_bwd_kernel and hash_bwd_routed_kernel: a warp per 32 consecutive samples, all levels.
template <bool POW2, typename AnchorT, bool GRAD_F16, bool HAS_BIAS, bool UNSCALE, typename Tables>
__device__ __forceinline__ void hash_bwd_body(int64_t n, const int32_t* __restrict__ d_n_ptr, int32_t n_volumes,
                                              uint32_t local_size, const Tables& tables,
                                              const float* __restrict__ scales, const float* __restrict__ pts,
                                              const AnchorT* __restrict__ anchors, const void* __restrict__ grad_in_v,
                                              int level_begin, int level_end) {
  if (d_n_ptr) {
    int64_t dn = *d_n_ptr;
    n = dn < n ? dn : n;
  }
  __shared__ float s_scale[GF_N_LEVELS];
  __shared__ __align__(16) float s_stage[(kHashBlock / 32) * kScatterWarpWords];
  // GRAD_F16: the warp's 32 gradient rows (64 bytes each, 2 KB contiguous) are fetched with four coalesced 16-byte
  // loads per lane and transposed through shared memory (row stride 17 words: the per-level reads are conflict-free).
  // Reading element (row, level) straight from global memory costs one 32-lane load at a 64-byte stride per level:
  // 16 L1 wavefronts x 16 levels per warp, 14 % of the LSU data pipe that bounds this kernel in steady state (r02x)
  constexpr int kGradRowWords = GF_N_LEVELS + 1;
  __shared__ uint32_t s_grad[GRAD_F16 ? (kHashBlock / 32) * 32 * kGradRowWords : 1];
  if (threadIdx.x < GF_N_LEVELS) s_scale[threadIdx.x] = __ldg(scales + threadIdx.x);
  __syncthreads();
  const int lane = lane_id();
  // (the mask restates the kernels' launch bounds, which the compiler no longer applies here after inlining)
  uint32_t* sg = s_grad + (GRAD_F16 ? ((threadIdx.x & (kHashBlock - 1)) >> 5) * 32 * kGradRowWords : 0);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  // warp-uniform trip count: every lane of a warp runs the same iterations
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + threadIdx.x - lane; base < n; base += stride) {
    const int64_t i = base + lane;
    const int32_t* prim_pool;
    const float* bias_pool;
    float* grad_table;
    int32_t key = 0;
    const bool valid = tables(i, i < n, prim_pool, bias_pool, grad_table, key) && i < n;
    float x = 0.f, y = 0.f, z = 0.f;
    int vol = 0;
    if (valid) {
      x = __ldg(pts + 3 * i);
      y = __ldg(pts + 3 * i + 1);
      z = __ldg(pts + 3 * i + 2);
      vol = (int)anchors[i];
    }
    const int pvol = __shfl_up_sync(0xffffffffu, vol, 1);  // by all 32 lanes: not inside the || below
    bool vol_head = lane == 0 || pvol != vol;
    if (Tables::kRouted) {  // a run also ends where the table changes
      const int32_t pkey = __shfl_up_sync(0xffffffffu, key, 1);   // by all 32 lanes, like pvol
      vol_head = vol_head || pkey != key;
    }
    if (GRAD_F16) {
      __syncwarp();  // the previous batch's readers are done with sg
      const uint4* src = reinterpret_cast<const uint4*>(grad_in_v) + base * (GF_N_LEVELS / 4);
#pragma unroll
      for (int k = 0; k < GF_N_LEVELS / 4; k++) {
        const int c = lane + 32 * k, row = c >> 2, part = c & 3;
        const uint4 v = base + row < n ? __ldg(src + c) : make_uint4(0u, 0u, 0u, 0u);
        uint32_t* dst = sg + row * kGradRowWords + part * 4;
        dst[0] = v.x;
        dst[1] = v.y;
        dst[2] = v.z;
        dst[3] = v.w;
      }
      __syncwarp();
    }
#pragma unroll 1
    for (int l = level_begin; l < level_end; l++) {
      // this level's two gradients, quantised like the reference: fp16(g*128)  (:209)
      __half2 gh = __float2half2_rn(0.f);
      if (GRAD_F16) {
        gh = *reinterpret_cast<const __half2*>(sg + lane * kGradRowWords + l);   // (rows past the end were zero-filled)
        if (Tables::kRouted && !valid) gh = __float2half2_rn(0.f);            // (a sample routed to no table)
      } else if (valid) {
        {
          const float2 v = __ldg(reinterpret_cast<const float2*>(grad_in_v) + i * GF_N_LEVELS + l);
          gh = __floats2half2_rn(__fmul_rn(v.x, GF_GRAD_SCALE), __fmul_rn(v.y, GF_GRAD_SCALE));
        }
      }
      hash_scatter_level<POW2, HAS_BIAS, UNSCALE, Tables::kRouted>(
          l, x, y, z, vol, vol_head, gh, lane, n_volumes, local_size, prim_pool, bias_pool, s_scale[l], grad_table,
          s_stage + (threadIdx.x >> 5) * kScatterWarpWords);
    }
  }
}

template <bool POW2, typename AnchorT, bool GRAD_F16, bool HAS_BIAS, bool UNSCALE>
__global__ void __launch_bounds__(kHashBlock, 4)   // 64 registers: four CTAs per SM (three at 72 cost 4 %, r02z)
hash_bwd_kernel(int64_t n, const int32_t* __restrict__ d_n_ptr, int32_t n_volumes, uint32_t local_size,
                const int32_t* __restrict__ prim_pool, const float* __restrict__ bias_pool,
                const float* __restrict__ scales, const float* __restrict__ pts,
                const AnchorT* __restrict__ anchors, const void* __restrict__ grad_in_v,
                float* __restrict__ grad_table, int level_begin, int level_end) {
  hash_bwd_body<POW2, AnchorT, GRAD_F16, HAS_BIAS, UNSCALE>(n, d_n_ptr, n_volumes, local_size,
                                                            OneGradTable{prim_pool, bias_pool, grad_table}, scales,
                                                            pts, anchors, grad_in_v, level_begin, level_end);
}

// Scatter with a gradient table per sample (gf_hash_backward_routed), all 16 levels.  A table's bias pool is read
// when its descriptor has one (a per-lane test instead of the HAS_BIAS instantiation).
// Registers: the three per-lane table pointers fit the 64 of four CTAs per SM when the table stays at the x128 scale
// Registers: with the three per-lane table pointers, the variant that leaves the table at the x128 scale (the engine's
// call) spills at the 64 registers of four CTAs per SM (ptxas keeps the unscaled variant's multiplier in a register
// and schedules differently), so it runs three at up to 80; the unscaled variant fits 64 and keeps four.
template <bool POW2, typename AnchorT, bool GRAD_F16, bool UNSCALE>
__global__ void __launch_bounds__(kHashBlock, UNSCALE ? 4 : 3)
hash_bwd_routed_kernel(int64_t n, const int32_t* __restrict__ d_n_ptr, int32_t n_volumes, uint32_t local_size,
                       int32_t n_tables, const gf_hash_grad_ref* __restrict__ tables,
                       const float* __restrict__ scales, const float* __restrict__ pts,
                       const AnchorT* __restrict__ anchors, const int32_t* __restrict__ ray_id,
                       const int32_t* __restrict__ ray_table, const void* __restrict__ grad_in_v) {
  hash_bwd_body<POW2, AnchorT, GRAD_F16, false, UNSCALE>(n, d_n_ptr, n_volumes, local_size,
                                                         RoutedGradTables{tables, n_tables, ray_id, ray_table}, scales,
                                                         pts, anchors, grad_in_v, 0, GF_N_LEVELS);
}

// table row of every corner, int32 [n,16,8] -- the parity probe for "bit-exact hash indices"
template <bool POW2, typename AnchorT>
__global__ void __launch_bounds__(kHashBlock)
hash_rows_kernel(int64_t n, int32_t n_volumes, uint32_t local_size, const int32_t* __restrict__ prim_pool,
                 const float* __restrict__ bias_pool, const float* __restrict__ scales,
                 const float* __restrict__ pts, const AnchorT* __restrict__ anchors, int32_t* __restrict__ rows) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float x = __ldg(pts + 3 * i), y = __ldg(pts + 3 * i + 1), z = __ldg(pts + 3 * i + 2);
    const int vol = (int)anchors[i];
    for (int l = 0; l < GF_N_LEVELS; l++) {
      const int tr = (l * n_volumes + vol) * 3;
      const Cell c = cell_of(x, y, z, __ldg(scales + l), bias_pool ? bias_pool + tr : nullptr);
      uint32_t pos[8];
      corners<POW2>(c, (uint32_t)__ldg(prim_pool + tr), (uint32_t)__ldg(prim_pool + tr + 1),
                    (uint32_t)__ldg(prim_pool + tr + 2), local_size, pos);
#pragma unroll
      for (int d = 0; d < 8; d++) rows[(i * GF_N_LEVELS + l) * 8 + d] = (int32_t)(level_base_row(l, local_size) + pos[d]);
    }
  }
}

static bool is_pow2(int64_t v) { return v > 0 && (v & (v - 1)) == 0; }

}  // namespace gf

using namespace gf;

extern "C" {

int gf_hash_level_scales(float* d_scales16, float* h_copy16, void* stream) {
  GF_REQUIRE(d_scales16 != nullptr, "gf_hash_level_scales: null output");
  cudaStream_t st = (cudaStream_t)stream;
  level_scales_kernel<<<1, 32, 0, st>>>(d_scales16);
  int rc = check_launch("level_scales_kernel");
  if (rc) return rc;
  if (h_copy16) {
    GF_CUDA(cudaMemcpyAsync(h_copy16, d_scales16, sizeof(float) * GF_N_LEVELS, cudaMemcpyDeviceToHost, st));
    GF_CUDA(cudaStreamSynchronize(st));
  }
  return GF_OK;
}

int gf_hash_cast_table(const float* feat_f32, void* feat_f16, int64_t n_elems, void* stream) {
  GF_REQUIRE(feat_f32 && feat_f16 && n_elems >= 0, "gf_hash_cast_table: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t n4 = n_elems / 4;
  if (n4 > 0) {
    cast_table_kernel<<<stride_grid(n4, 256, 8, 4), 256, 0, st>>>((const float4*)feat_f32, (uint2*)feat_f16, n4);
    int rc = check_launch("cast_table_kernel");
    if (rc) return rc;
  }
  if (n4 * 4 < n_elems) {
    cast_table_tail_kernel<<<1, 32, 0, st>>>(feat_f32, (__half*)feat_f16, n4 * 4, n_elems);
    return check_launch("cast_table_tail_kernel");
  }
  return GF_OK;
}

static int hash_forward_impl(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                             const void* feat_f16, const int32_t* prim_pool, const float* bias_pool,
                             const float* level_scales, const float* pts, const void* anchors, int anchor_i64,
                             void* out_f16, float* out_f32, const void* base_f16, void* stream) {
  GF_REQUIRE(n >= 0 && n_volumes > 0 && local_size > 0 && local_size <= 0x7fffffffLL && local_size % 2 == 0,
             "gf_hash_forward: bad sizes n=%lld n_volumes=%d local_size=%lld (must be even)", (long long)n, n_volumes,
             (long long)local_size);
  GF_REQUIRE((int64_t)n_volumes * GF_N_LEVELS * 3 <= 0x7fffffffLL, "gf_hash_forward: n_volumes too large");
  GF_REQUIRE(out_f16 || out_f32, "gf_hash_forward: no output buffer");
  if (n == 0) return GF_OK;
  GF_REQUIRE(feat_f16 && prim_pool && level_scales && pts && anchors, "gf_hash_forward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = stride_grid(n, kHashBlock, 8, 4);
  const bool p2 = is_pow2(local_size);
  // the rows the levels can reach (8.5 * local_size, 4 bytes each) against the 126 MB L2: which variant (see the kernel)
  const bool l2_resident = (int64_t)local_size * 34 <= (int64_t)100 << 20;
#define GF_FWD_V(P2, AT, O16, O32, PF)                                                                        \
  hash_fwd_kernel<P2, AT, O16, O32, PF><<<grid, kHashBlock, 0, st>>>(                                         \
      n, d_n_ptr, n_volumes, (uint32_t)local_size, (const __half2*)feat_f16, prim_pool, bias_pool,            \
      level_scales, pts, (const AT*)anchors, (uint4*)out_f16, (float4*)out_f32, (const uint4*)base_f16)
#define GF_FWD(P2, AT, O16, O32)                    \
  do {                                              \
    if (l2_resident) GF_FWD_V(P2, AT, O16, O32, true); \
    else GF_FWD_V(P2, AT, O16, O32, false);         \
  } while (0)
#define GF_FWD_O(P2, AT)                                     \
  do {                                                       \
    if (out_f16 && out_f32) GF_FWD(P2, AT, true, true);      \
    else if (out_f16) GF_FWD(P2, AT, true, false);           \
    else GF_FWD(P2, AT, false, true);                        \
  } while (0)
  if (p2) {
    if (anchor_i64) GF_FWD_O(true, int64_t); else GF_FWD_O(true, int32_t);
  } else {
    if (anchor_i64) GF_FWD_O(false, int64_t); else GF_FWD_O(false, int32_t);
  }
#undef GF_FWD_O
#undef GF_FWD
#undef GF_FWD_V
  return check_launch("hash_fwd_kernel");
}

int gf_hash_forward(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                    const void* feat_f16, const int32_t* prim_pool, const float* bias_pool,
                    const float* level_scales, const float* pts, const void* anchors, int anchor_i64,
                    void* out_f16, float* out_f32, void* stream) {
  return hash_forward_impl(n, d_n_ptr, n_volumes, local_size, feat_f16, prim_pool, bias_pool, level_scales, pts,
                           anchors, anchor_i64, out_f16, out_f32, nullptr, stream);
}

int gf_hash_forward_residual(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                             const void* feat_f16, const int32_t* prim_pool, const float* bias_pool,
                             const float* level_scales, const float* pts, const void* anchors, int anchor_i64,
                             const void* base_f16, void* out_f16, void* stream) {
  GF_REQUIRE(base_f16 && out_f16, "gf_hash_forward_residual: null base / output");
  return hash_forward_impl(n, d_n_ptr, n_volumes, local_size, feat_f16, prim_pool, bias_pool, level_scales, pts,
                           anchors, anchor_i64, out_f16, nullptr, base_f16, stream);
}

int gf_hash_forward_residual_routed(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                                    int32_t n_tables, const gf_hash_table_ref* d_tables, const float* level_scales,
                                    const float* pts, const void* anchors, int anchor_i64, const int32_t* ray_id,
                                    const int32_t* ray_table, const void* base_f16, void* out_f16, void* stream) {
  GF_REQUIRE(n >= 0 && n_volumes > 0 && local_size > 0 && local_size <= 0x7fffffffLL && local_size % 2 == 0,
             "gf_hash_forward_residual_routed: bad sizes n=%lld n_volumes=%d local_size=%lld (must be even)",
             (long long)n, n_volumes, (long long)local_size);
  GF_REQUIRE((int64_t)n_volumes * GF_N_LEVELS * 3 <= 0x7fffffffLL, "gf_hash_forward_residual_routed: n_volumes too large");
  GF_REQUIRE(n_tables > 0, "gf_hash_forward_residual_routed: n_tables = %d (must be > 0)", n_tables);
  GF_REQUIRE(d_tables && ray_id && ray_table && base_f16 && out_f16,
             "gf_hash_forward_residual_routed: null table descriptors / ray_id / ray_table / base / output");
  if (n == 0) return GF_OK;
  GF_REQUIRE(level_scales && pts && anchors, "gf_hash_forward_residual_routed: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = stride_grid(n, kHashBlock, 8, 4);
  const bool p2 = is_pow2(local_size);
  const bool l2_resident = (int64_t)local_size * 34 <= (int64_t)100 << 20;   // as hash_forward_impl
#define GF_FWD_R(P2, AT, PF)                                                                                    \
  hash_fwd_routed_kernel<P2, AT, PF><<<grid, kHashBlock, 0, st>>>(                                              \
      n, d_n_ptr, n_volumes, (uint32_t)local_size, n_tables, d_tables, level_scales, pts, (const AT*)anchors,   \
      ray_id, ray_table, (uint4*)out_f16, (const uint4*)base_f16)
#define GF_FWD_RA(P2, AT)                        \
  do {                                           \
    if (l2_resident) GF_FWD_R(P2, AT, true);     \
    else GF_FWD_R(P2, AT, false);                \
  } while (0)
  if (p2) {
    if (anchor_i64) GF_FWD_RA(true, int64_t); else GF_FWD_RA(true, int32_t);
  } else {
    if (anchor_i64) GF_FWD_RA(false, int64_t); else GF_FWD_RA(false, int32_t);
  }
#undef GF_FWD_RA
#undef GF_FWD_R
  return check_launch("hash_fwd_routed_kernel");
}

int gf_hash_backward(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                     const int32_t* prim_pool, const float* bias_pool, const float* level_scales,
                     const float* pts, const void* anchors, int anchor_i64, const void* grad_in,
                     int grad_in_is_scaled_f16, float* grad_table, void* stream) {
  return gf_hash_backward_levels(n, d_n_ptr, n_volumes, local_size, prim_pool, bias_pool, level_scales, pts, anchors,
                                 anchor_i64, grad_in, grad_in_is_scaled_f16, grad_table, 0, GF_N_LEVELS, stream);
}

int gf_hash_backward_levels(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                            const int32_t* prim_pool, const float* bias_pool, const float* level_scales,
                            const float* pts, const void* anchors, int anchor_i64, const void* grad_in,
                            int grad_in_is_scaled_f16, float* grad_table, int level_begin, int level_end,
                            void* stream) {
  GF_REQUIRE(n >= 0 && n_volumes > 0 && local_size > 0 && local_size <= 0x7fffffffLL && local_size % 2 == 0,
             "gf_hash_backward: bad sizes n=%lld n_volumes=%d local_size=%lld (must be even)", (long long)n, n_volumes,
             (long long)local_size);
  GF_REQUIRE(0 <= level_begin && level_begin <= level_end && level_end <= GF_N_LEVELS,
             "gf_hash_backward: bad level range [%d, %d)", level_begin, level_end);
  if (level_begin == level_end) return GF_OK;
  if (n == 0) return GF_OK;
  GF_REQUIRE(prim_pool && level_scales && pts && anchors && grad_in && grad_table, "gf_hash_backward: null pointer");
  GF_REQUIRE((reinterpret_cast<uintptr_t>(grad_in) & 15) == 0, "gf_hash_backward: grad_in must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = stride_grid(n, kHashBlock, 4, 4);
  const bool p2 = is_pow2(local_size);
  const bool g16 = (grad_in_is_scaled_f16 & 1) != 0, unscale = (grad_in_is_scaled_f16 & 2) == 0;
#define GF_BWD(P2, AT, G16, HB, US)                                                                              \
  hash_bwd_kernel<P2, AT, G16, HB, US><<<grid, kHashBlock, 0, st>>>(n, d_n_ptr, n_volumes, (uint32_t)local_size, \
                                                                    prim_pool, bias_pool, level_scales, pts,     \
                                                                    (const AT*)anchors, grad_in, grad_table,     \
                                                                    level_begin, level_end)
#define GF_BWD_U(P2, AT, G16, HB)                  \
  do {                                             \
    if (unscale) GF_BWD(P2, AT, G16, HB, true);    \
    else GF_BWD(P2, AT, G16, HB, false);           \
  } while (0)
#define GF_BWD_B(P2, AT, G16)                      \
  do {                                             \
    if (bias_pool) GF_BWD_U(P2, AT, G16, true);    \
    else GF_BWD_U(P2, AT, G16, false);             \
  } while (0)
#define GF_BWD_G(P2, AT)                           \
  do {                                             \
    if (g16) GF_BWD_B(P2, AT, true);               \
    else GF_BWD_B(P2, AT, false);                  \
  } while (0)
  if (p2) {
    if (anchor_i64) GF_BWD_G(true, int64_t); else GF_BWD_G(true, int32_t);
  } else {
    if (anchor_i64) GF_BWD_G(false, int64_t); else GF_BWD_G(false, int32_t);
  }
#undef GF_BWD_G
#undef GF_BWD_B
#undef GF_BWD_U
#undef GF_BWD
  return check_launch("hash_bwd_kernel");
}

int gf_hash_backward_routed(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                            int32_t n_tables, const gf_hash_grad_ref* d_tables, const float* level_scales,
                            const float* pts, const void* anchors, int anchor_i64, const int32_t* ray_id,
                            const int32_t* ray_table, const void* grad_in, int grad_in_is_scaled_f16, void* stream) {
  GF_REQUIRE(n >= 0 && n_volumes > 0 && local_size > 0 && local_size <= 0x7fffffffLL && local_size % 2 == 0,
             "gf_hash_backward_routed: bad sizes n=%lld n_volumes=%d local_size=%lld (must be even)", (long long)n,
             n_volumes, (long long)local_size);
  GF_REQUIRE(n_tables > 0, "gf_hash_backward_routed: n_tables = %d (must be > 0)", n_tables);
  GF_REQUIRE(d_tables && ray_id && ray_table, "gf_hash_backward_routed: null table descriptors / ray_id / ray_table");
  if (n == 0) return GF_OK;
  GF_REQUIRE(level_scales && pts && anchors && grad_in, "gf_hash_backward_routed: null pointer");
  GF_REQUIRE((reinterpret_cast<uintptr_t>(grad_in) & 15) == 0,
             "gf_hash_backward_routed: grad_in must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = stride_grid(n, kHashBlock, 4, 4);
  const bool p2 = is_pow2(local_size);
  const bool g16 = (grad_in_is_scaled_f16 & 1) != 0, unscale = (grad_in_is_scaled_f16 & 2) == 0;
#define GF_BWD_R(P2, AT, G16, US)                                                                               \
  hash_bwd_routed_kernel<P2, AT, G16, US><<<grid, kHashBlock, 0, st>>>(                                         \
      n, d_n_ptr, n_volumes, (uint32_t)local_size, n_tables, d_tables, level_scales, pts, (const AT*)anchors,   \
      ray_id, ray_table, grad_in)
#define GF_BWD_RU(P2, AT, G16)                      \
  do {                                              \
    if (unscale) GF_BWD_R(P2, AT, G16, true);       \
    else GF_BWD_R(P2, AT, G16, false);              \
  } while (0)
#define GF_BWD_RG(P2, AT)                           \
  do {                                              \
    if (g16) GF_BWD_RU(P2, AT, true);               \
    else GF_BWD_RU(P2, AT, false);                  \
  } while (0)
  if (p2) {
    if (anchor_i64) GF_BWD_RG(true, int64_t); else GF_BWD_RG(true, int32_t);
  } else {
    if (anchor_i64) GF_BWD_RG(false, int64_t); else GF_BWD_RG(false, int32_t);
  }
#undef GF_BWD_RG
#undef GF_BWD_RU
#undef GF_BWD_R
  return check_launch("hash_bwd_routed_kernel");
}

int gf_hash_corner_rows(int64_t n, int32_t n_volumes, int64_t local_size, const int32_t* prim_pool,
                        const float* bias_pool, const float* level_scales, const float* pts,
                        const void* anchors, int anchor_i64, int32_t* rows, void* stream) {
  GF_REQUIRE(n >= 0 && n_volumes > 0 && local_size > 0 && local_size * GF_N_LEVELS <= 0x7fffffffLL &&
                 local_size % 2 == 0,
             "gf_hash_corner_rows: bad sizes (local_size must be even)");
  if (n == 0) return GF_OK;
  GF_REQUIRE(prim_pool && level_scales && pts && anchors && rows, "gf_hash_corner_rows: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = stride_grid(n, kHashBlock, 8, 4);
  const bool p2 = is_pow2(local_size);
#define GF_ROWS(P2, AT)                                                                                    \
  hash_rows_kernel<P2, AT><<<grid, kHashBlock, 0, st>>>(n, n_volumes, (uint32_t)local_size, prim_pool,     \
                                                        bias_pool, level_scales, pts, (const AT*)anchors, rows)
  if (p2) {
    if (anchor_i64) GF_ROWS(true, int64_t); else GF_ROWS(true, int32_t);
  } else {
    if (anchor_i64) GF_ROWS(false, int64_t); else GF_ROWS(false, int32_t);
  }
#undef GF_ROWS
  return check_launch("hash_rows_kernel");
}

}  // extern "C"
