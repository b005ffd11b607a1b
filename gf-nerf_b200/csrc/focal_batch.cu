// Focal-stage batch source on the device: error-weighted pixel draws over a sum tree of the error map.
//
// The draw has the distribution of ErrorPixelSampler.sample_method (pixel_samplers.py): per "job" (one 2^24-pixel
// chunk of the weighted part, the weighted remainder, or a uniform part) `count` distinct flat pixel numbers in the
// order of successive sampling (what torch.multinomial(replacement=False) draws).  Draws are made WITH replacement and
// the first occurrence of each pixel, in draw order, is kept: the accepted sequence is the prefix of one iid sequence,
// so the result is exactly successive sampling.  Rounds draw again for the pixels still missing, with more draws per
// round while duplicates dominate; a job that is complete makes the later rounds' kernels return at once.
//
// Sum tree over the flat map (fp64 sums, int32 non-zero counts, one array of each, levels stored one after another):
//   level 0: tiles of 1024 pixels (one warp: lane l sums pixels [32 l, 32 l + 32) in order, then a warp scan),
//   levels 1, 2: 32 children each, level 3: 16 children = one node per 2^24-pixel chunk.
// Every node is (re)computed from its children by the same warp scan, in a fixed order, and a descent renormalises
// each level by the same scan, so a rebuild gives the same bits and the level probabilities telescope to w / sum w.
#include <curand_kernel.h>

#include "common.cuh"

namespace gf {

namespace {

constexpr int kTile = 1024;          // pixels per tile
constexpr unsigned kFull = 0xffffffffu;

// job table: int64 fields per job (built by pixel_samplers.FocalBatchSource)
enum { J_LO, J_HI, J_COUNT, J_WEIGHTED, J_CHUNK, J_CAND_OFF, J_CAND_CAP, J_OUT_OFF, J_TAB_OFF, J_TAB_CAP, J_FIELDS };

struct TreeLayout {
  int64_t n, n0, n1, n2, n3, o1, o2, o3;
};

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

inline TreeLayout tree_layout(int64_t n) {
  TreeLayout L;
  L.n = n;
  L.n0 = ceil_div(n, kTile);
  L.n1 = ceil_div(L.n0, 32);
  L.n2 = ceil_div(L.n1, 32);
  L.n3 = ceil_div(L.n2, 16);
  L.o1 = L.n0;
  L.o2 = L.o1 + L.n1;
  L.o3 = L.o2 + L.n2;
  return L;
}

__device__ __forceinline__ double warp_incl_scan(double v) {
  const int lane = lane_id();
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double t = __shfl_up_sync(kFull, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// lane's 32 pixels of tile t, summed in order; c = how many are > 0
__device__ __forceinline__ void lane_pixels(const float* __restrict__ map, int64_t n, int64_t t, double& s, int& c) {
  const int64_t base = t * kTile + 32 * lane_id();
  s = 0.0;
  c = 0;
  if (base + 32 <= n) {
    const float4* p = reinterpret_cast<const float4*>(map + base);
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const float4 v = __ldg(p + q);
      s += (double)v.x; s += (double)v.y; s += (double)v.z; s += (double)v.w;
      c += (v.x > 0.f) + (v.y > 0.f) + (v.z > 0.f) + (v.w > 0.f);
    }
  } else {
    for (int64_t i = base; i < base + 32 && i < n; i++) {
      const float w = __ldg(map + i);
      s += (double)w;
      c += w > 0.f;
    }
  }
}

// flat pixel of an (image, y, x) row, with torch's single wrap of negative indices; -1 if out of range
__device__ __forceinline__ int64_t row_pixel(const int64_t* __restrict__ idx, int64_t i, int64_t n_images,
                                             int64_t height, int64_t width) {
  int64_t c = idx[3 * i], y = idx[3 * i + 1], x = idx[3 * i + 2];
  if (c < 0) c += n_images;
  if (y < 0) y += height;
  if (x < 0) x += width;
  if (c < 0 || c >= n_images || y < 0 || y >= height || x < 0 || x >= width) return -1;
  return (c * height + y) * width + x;
}

// One warp per node.  rows == NULL: node = item of `level`; else the node of `level` above row item's pixel.
__global__ void __launch_bounds__(256)
sumtree_node_kernel(int level, int64_t n_items, const int64_t* __restrict__ rows, int64_t n_images, int64_t height,
                    int64_t width, const float* __restrict__ map, TreeLayout L, double* __restrict__ sums,
                    int* __restrict__ counts) {
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int lane = lane_id();
  for (int64_t it = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; it < n_items; it += n_warps) {
    int64_t node = it;
    if (rows) {
      const int64_t f = row_pixel(rows, it, n_images, height, width);
      if (f < 0) continue;                                        // skipped (and flagged) by the map update
      node = (f / kTile) >> (level == 3 ? 14 : 5 * level);
    }
    double s;
    int c;
    if (level == 0) {
      lane_pixels(map, L.n, node, s, c);
    } else {
      const int fan = level == 3 ? 16 : 32;
      const int64_t child_off = level == 1 ? 0 : (level == 2 ? L.o1 : L.o2);
      const int64_t n_child = level == 1 ? L.n0 : (level == 2 ? L.n1 : L.n2);
      const int64_t ch = node * fan + lane;
      const bool ok = lane < fan && ch < n_child;
      s = ok ? sums[child_off + ch] : 0.0;
      c = ok ? counts[child_off + ch] : 0;
    }
    const double tot = __shfl_sync(kFull, warp_incl_scan(s), 31);
    c = __reduce_add_sync(kFull, c);
    if (lane == 0) {
      const int64_t off = level == 0 ? 0 : (level == 1 ? L.o1 : (level == 2 ? L.o2 : L.o3));
      sums[off + node] = tot;
      counts[off + node] = c;
    }
  }
}

// Warp: child in [first, first + cnt) with probability v / sum v, by the scan the tree was built with; -1 if no
// child has mass.  t = u * total can round up to total: then the last child with mass is taken.
__device__ __forceinline__ int64_t pick_child(const double* __restrict__ s, int64_t first, int64_t cnt, double u) {
  const int lane = lane_id();
  const double v = lane < cnt ? s[first + lane] : 0.0;
  const double incl = warp_incl_scan(v);
  const double t = u * __shfl_sync(kFull, incl, 31);
  unsigned hit = __ballot_sync(kFull, incl > t && v > 0.0);
  if (hit) return first + __ffs(hit) - 1;
  hit = __ballot_sync(kFull, v > 0.0);
  return hit ? first + 31 - __clz(hit) : -1;
}

// Warp: pixel of tile `tile` with probability w / tile sum; -1 if the tile has no mass
__device__ int64_t pick_pixel(const float* __restrict__ map, int64_t n, int64_t tile, double u) {
  const int lane = lane_id();
  double s;
  int c;
  lane_pixels(map, n, tile, s, c);
  const double incl = warp_incl_scan(s);
  double excl = __shfl_up_sync(kFull, incl, 1);
  if (lane == 0) excl = 0.0;
  const double t = u * __shfl_sync(kFull, incl, 31);
  unsigned hit = __ballot_sync(kFull, incl > t && s > 0.0);
  const bool exact = hit != 0;
  if (!hit) hit = __ballot_sync(kFull, s > 0.0);
  if (!hit) return -1;
  const int sel = exact ? __ffs(hit) - 1 : 31 - __clz(hit);
  int64_t pix = -1;
  if (lane == sel) {
    const double r = exact ? t - excl : INFINITY;              // residual inside this lane's 32 pixels
    const int64_t base = tile * kTile + 32 * lane;
    double acc = 0.0;
    for (int64_t i = base; i < base + 32 && i < n; i++) {
      const float w = __ldg(map + i);
      acc += (double)w;
      if (w > 0.f) {
        pix = i;
        if (acc > r) break;
      }
    }
  }
  return __shfl_sync(kFull, pix, sel);
}

__device__ __forceinline__ double unit53(unsigned a, unsigned b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// draws a job makes in `round`: the missing count, doubled each round (duplicates dominate when the mass is
// concentrated on few pixels), at most the job's candidate capacity
__device__ __forceinline__ int64_t round_draws(int64_t need, int64_t cap, int round) {
  const int sh = round < 20 ? round : 20;
  const int64_t m = need << sh;
  return m < cap ? m : cap;
}

__global__ void focal_init_kernel(int64_t n_jobs, int* __restrict__ have, int* __restrict__ pending) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_jobs) have[i] = 0;
  if (i == 0) *pending = (int)n_jobs;
}

// One warp per candidate slot: a fresh Philox stream per (step round counter, slot), four 53-bit uniforms per draw.
__global__ void __launch_bounds__(256)
focal_draw_kernel(int round, const int64_t* __restrict__ jobs, const int* __restrict__ slot_job, int64_t total_cap,
                  const int* __restrict__ have, const int* __restrict__ pending, const int64_t* __restrict__ rng,
                  const float* __restrict__ map, const double* __restrict__ sums, TreeLayout L,
                  int64_t* __restrict__ cand) {
  if (*pending == 0) return;
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const unsigned long long seed = (unsigned long long)rng[0], sub = (unsigned long long)rng[1] + round;
  for (int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < total_cap; s += n_warps) {
    const int j = slot_job[s];
    const int64_t* J = jobs + (int64_t)J_FIELDS * j;
    const int64_t count = J[J_COUNT], h = have[j];
    if (h >= count || s - J[J_CAND_OFF] >= round_draws(count - h, J[J_CAND_CAP], round)) continue;
    curandStatePhilox4_32_10_t st;
    curand_init(seed, sub, (unsigned long long)s * 8, &st);
    const uint4 a = curand4(&st), b = curand4(&st);
    const int64_t lo = J[J_LO], hi = J[J_HI];
    int64_t pix;
    if (!J[J_WEIGHTED]) {
      const int64_t k = (int64_t)(unit53(a.x, a.y) * (double)(hi - lo));
      pix = lo + (k < hi - lo ? k : hi - lo - 1);
    } else {
      const int64_t c = J[J_CHUNK];
      int64_t p = pick_child(sums + L.o2, 16 * c, min((int64_t)16, L.n2 - 16 * c), unit53(a.x, a.y));
      if (p >= 0) p = pick_child(sums + L.o1, 32 * p, min((int64_t)32, L.n1 - 32 * p), unit53(a.z, a.w));
      if (p >= 0) p = pick_child(sums, 32 * p, min((int64_t)32, L.n0 - 32 * p), unit53(b.x, b.y));
      pix = p >= 0 ? pick_pixel(map, L.n, p, unit53(b.z, b.w)) : -1;
    }
    if (lane_id() == 0) cand[s] = pix;
  }
}

__device__ __forceinline__ uint32_t hash_slot(int64_t key, int64_t mask) {
  uint64_t x = (uint64_t)key * 0x9E3779B97F4A7C15ull;
  return (uint32_t)((x ^ (x >> 29)) & (uint64_t)mask);
}

// One CTA per job: keep the first occurrence of each pixel (in draw order: position = round * cap + slot) that no
// earlier round accepted, append the first `need` of them in draw order.
__global__ void __launch_bounds__(1024)
focal_accept_kernel(int round, const int64_t* __restrict__ jobs, int* __restrict__ have, int* __restrict__ pending,
                    const int64_t* __restrict__ cand, unsigned long long* __restrict__ tab_keys,
                    int* __restrict__ tab_pos, const double* __restrict__ sums, const int* __restrict__ counts,
                    TreeLayout L, int64_t* __restrict__ sel, int* __restrict__ err) {
  __shared__ int s_warp[32];
  __shared__ int s_total;
  const int j = blockIdx.x, tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
  const int64_t* J = jobs + (int64_t)J_FIELDS * j;
  const int64_t count = J[J_COUNT], h = have[j];
  if (h >= count) return;
  const int64_t lo = J[J_LO], cand_cap = J[J_CAND_CAP], out = J[J_OUT_OFF] + h;
  const int64_t mask = J[J_TAB_CAP] - 1;
  unsigned long long* keys = tab_keys + J[J_TAB_OFF];
  int* pos = tab_pos + J[J_TAB_OFF];
  const int64_t* cj = cand + J[J_CAND_OFF];
  if (round == 0) {
    for (int64_t i = tid; i <= mask; i += blockDim.x) {
      keys[i] = ~0ull;
      pos[i] = INT_MAX;
    }
    if (J[J_WEIGHTED]) {
      // torch.multinomial's errors: a non-finite sum ("invalid multinomial distribution") and fewer non-zero
      // categories than samples ("not enough non-negative category")
      const double tot = sums[L.o3 + J[J_CHUNK]];
      const int bad = !isfinite(tot) ? 2 : (counts[L.o3 + J[J_CHUNK]] < count ? 1 : 0);
      if (bad) {
        for (int64_t i = tid; i < count; i += blockDim.x) sel[out + i] = lo;   // in range; the flag reports it
        if (tid == 0) {
          atomicOr(err, bad);
          have[j] = (int)count;
          atomicSub(pending, 1);
        }
        return;
      }
    }
    __syncthreads();
  }
  const int64_t need = count - h, m = round_draws(need, cand_cap, round);
  const int base_pos = round * (int)cand_cap;
  for (int64_t k = tid; k < m; k += blockDim.x) {
    const int64_t key = cj[k];
    if (key < 0) continue;
    for (uint32_t e = hash_slot(key, mask);; e = (e + 1) & (uint32_t)mask) {
      const unsigned long long prev = atomicCAS(keys + e, ~0ull, (unsigned long long)key);
      if (prev == ~0ull || prev == (unsigned long long)key) {
        atomicMin(pos + e, base_pos + (int)k);
        break;
      }
    }
  }
  __syncthreads();
  int64_t run = 0;
  for (int64_t k0 = 0; k0 < m; k0 += blockDim.x) {
    const int64_t k = k0 + tid;
    int64_t key = -1;
    bool fresh = false;
    if (k < m && (key = cj[k]) >= 0) {
      uint32_t e = hash_slot(key, mask);
      while (keys[e] != (unsigned long long)key) e = (e + 1) & (uint32_t)mask;
      fresh = pos[e] == base_pos + (int)k;
    }
    const unsigned bal = __ballot_sync(kFull, fresh);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
      const int v = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
      int incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += t;
      }
      s_warp[lane] = incl - v;
      if (lane == 31) s_total = incl;
    }
    __syncthreads();
    const int64_t r = run + s_warp[warp] + __popc(bal & ((1u << lane) - 1u));
    if (fresh && r < need) sel[out + r] = key;
    run += s_total;
    __syncthreads();
  }
  if (tid == 0) {
    const int64_t got = run < need ? run : need;
    have[j] = (int)(h + got);
    if (got == need) atomicSub(pending, 1);
  }
}

// One thread per batch row: (slot, y, x), the absolute and relative camera indices, the pixel's colour and the pixel
// centre for the ray generator.  Also closes the step: an unfinished job is flagged, the Philox counter advances.
__global__ void __launch_bounds__(256)
focal_gather_kernel(int64_t n_rows, const int64_t* __restrict__ sel, int64_t n_jobs, const int64_t* __restrict__ jobs,
                    const int* __restrict__ have, int64_t height, int64_t width, const float* __restrict__ images,
                    const int64_t* __restrict__ image_idx, const int64_t* __restrict__ rel_idx,
                    int64_t* __restrict__ slot_out, int64_t* __restrict__ idx_out, int64_t* __restrict__ rel_out,
                    float* __restrict__ rgb_out, float* __restrict__ coords_out, int64_t* __restrict__ cam_out,
                    int64_t* __restrict__ rng, int rounds, int* __restrict__ err) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_jobs && have[i] < jobs[(int64_t)J_FIELDS * i + J_COUNT]) atomicOr(err, 4);
  if (i == 0) rng[1] += rounds;
  if (i >= n_rows) return;
  const int64_t f = sel[i];
  const int64_t slot = f / (height * width), y = (f / width) % height, x = f % width;
  const int64_t cam = image_idx[slot];
  slot_out[3 * i] = slot;
  slot_out[3 * i + 1] = y;
  slot_out[3 * i + 2] = x;
  idx_out[3 * i] = cam;
  idx_out[3 * i + 1] = y;
  idx_out[3 * i + 2] = x;
  rel_out[i] = rel_idx[slot];
  cam_out[i] = cam;
  rgb_out[3 * i] = images[3 * f];
  rgb_out[3 * i + 1] = images[3 * f + 1];
  rgb_out[3 * i + 2] = images[3 * f + 2];
  coords_out[2 * i] = __fadd_rn((float)y, 0.5f);
  coords_out[2 * i + 1] = __fadd_rn((float)x, 0.5f);
}

int launch_levels(int64_t n_items, const int64_t* rows, int64_t n_images, int64_t height, int64_t width,
                  const float* map, const TreeLayout& L, double* sums, int* counts, cudaStream_t st) {
  for (int level = 0; level < 4; level++) {
    const int64_t items = rows ? n_items : (level == 0 ? L.n0 : level == 1 ? L.n1 : level == 2 ? L.n2 : L.n3);
    sumtree_node_kernel<<<stride_grid(items * 32, 256, 8, 4), 256, 0, st>>>(level, items, rows, n_images, height,
                                                                            width, map, L, sums, counts);
    const int rc = check_launch("sumtree_node_kernel");
    if (rc != GF_OK) return rc;
  }
  return GF_OK;
}

}  // namespace

}  // namespace gf

using namespace gf;

extern "C" int64_t gf_sumtree_nodes(int64_t n_pixels) {
  if (n_pixels <= 0) return 0;
  const TreeLayout L = tree_layout(n_pixels);
  return L.o3 + L.n3;
}

extern "C" int gf_sumtree_build(int64_t n_pixels, const float* error_map, double* sums, int32_t* counts,
                                void* stream) {
  GF_REQUIRE(n_pixels > 0 && n_pixels < ((int64_t)1 << 40), "gf_sumtree_build: bad size %lld", (long long)n_pixels);
  GF_REQUIRE(error_map && sums && counts, "gf_sumtree_build: null pointer");
  GF_REQUIRE(((uintptr_t)error_map & 15) == 0, "gf_sumtree_build: error_map must be 16-byte aligned");
  return launch_levels(0, nullptr, 0, 0, 0, error_map, tree_layout(n_pixels), sums, counts, (cudaStream_t)stream);
}

extern "C" int gf_sumtree_refresh(int64_t n_rows, const int64_t* indices, int64_t n_images, int64_t height,
                                  int64_t width, const float* error_map, double* sums, int32_t* counts, void* stream) {
  GF_REQUIRE(n_rows >= 0 && n_images > 0 && height > 0 && width > 0, "gf_sumtree_refresh: bad sizes");
  if (n_rows == 0) return GF_OK;
  GF_REQUIRE(indices && error_map && sums && counts, "gf_sumtree_refresh: null pointer");
  GF_REQUIRE(((uintptr_t)error_map & 15) == 0, "gf_sumtree_refresh: error_map must be 16-byte aligned");
  return launch_levels(n_rows, indices, n_images, height, width, error_map, tree_layout(n_images * height * width),
                       sums, counts, (cudaStream_t)stream);
}

extern "C" int gf_focal_draw(int64_t n_images, int64_t height, int64_t width, const float* error_map,
                             const double* sums, const int32_t* counts, int64_t n_jobs, const int64_t* jobs,
                             const int32_t* slot_job, int64_t total_cap, int64_t* cand, uint64_t* tab_keys,
                             int32_t* tab_pos, int32_t* work, int64_t* rng, int32_t rounds, int64_t n_rows,
                             int64_t* sel, const float* images, const int64_t* image_idx, const int64_t* rel_idx,
                             int64_t* slot_out, int64_t* idx_out, int64_t* rel_out, float* rgb_out,
                             float* coords_out, int64_t* cam_out, int32_t* err, void* stream) {
  GF_REQUIRE(n_images > 0 && height > 0 && width > 0 && n_jobs > 0 && n_jobs < (1 << 20) && total_cap > 0 &&
                 rounds > 0 && rounds <= 64 && n_rows > 0,
             "gf_focal_draw: bad sizes map=[%lld,%lld,%lld] jobs=%lld cap=%lld rounds=%d rows=%lld",
             (long long)n_images, (long long)height, (long long)width, (long long)n_jobs, (long long)total_cap,
             (int)rounds, (long long)n_rows);
  GF_REQUIRE(error_map && sums && counts && jobs && slot_job && cand && tab_keys && tab_pos && work && rng && sel &&
                 images && image_idx && rel_idx && slot_out && idx_out && rel_out && rgb_out && coords_out &&
                 cam_out && err,
             "gf_focal_draw: null pointer");
  GF_REQUIRE(((uintptr_t)error_map & 15) == 0, "gf_focal_draw: error_map must be 16-byte aligned");
  GF_REQUIRE(total_cap * rounds < INT_MAX, "gf_focal_draw: %lld candidates x %d rounds overflow the draw order",
             (long long)total_cap, (int)rounds);
  const cudaStream_t st = (cudaStream_t)stream;
  const TreeLayout L = tree_layout(n_images * height * width);
  int* have = work;
  int* pending = work + n_jobs;
  focal_init_kernel<<<(int)ceil_div(n_jobs, 256), 256, 0, st>>>(n_jobs, have, pending);
  int rc = check_launch("focal_init_kernel");
  const int draw_grid = stride_grid(total_cap * 32, 256, 8, 2);
  for (int r = 0; r < rounds && rc == GF_OK; r++) {
    focal_draw_kernel<<<draw_grid, 256, 0, st>>>(r, jobs, slot_job, total_cap, have, pending, rng, error_map, sums, L,
                                                 cand);
    rc = check_launch("focal_draw_kernel");
    if (rc != GF_OK) break;
    focal_accept_kernel<<<(int)n_jobs, 1024, 0, st>>>(r, jobs, have, pending, cand,
                                                      reinterpret_cast<unsigned long long*>(tab_keys), tab_pos, sums,
                                                      counts, L, sel, err);
    rc = check_launch("focal_accept_kernel");
  }
  if (rc != GF_OK) return rc;
  const int64_t n_thr = n_rows > n_jobs ? n_rows : n_jobs;
  focal_gather_kernel<<<(int)ceil_div(n_thr, 256), 256, 0, st>>>(n_rows, sel, n_jobs, jobs, have, height, width,
                                                                  images, image_idx, rel_idx, slot_out, idx_out,
                                                                  rel_out, rgb_out, coords_out, cam_out, rng, rounds,
                                                                  err);
  return check_launch("focal_gather_kernel");
}
