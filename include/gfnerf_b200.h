/*
 * gfnerf_b200.h -- C-ABI of the B200-native GF-NeRF per-ray hot path.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes (device
 * pointers unless the parameter name starts with `h_`), takes the CUDA stream
 * as an opaque `void*` (a `cudaStream_t`; NULL = legacy default stream) and
 * returns 0 on success or a negative gf_status.  After a failure
 * `gf_last_error()` returns a thread-local, NUL-terminated description.
 * Nothing here includes torch or CUDA headers, so the reference's binding
 * layer (TORCH_LIBRARY custom classes, see INTEGRATION.md) or any other FFI
 * (ctypes, cgo, JNI) can bind it directly.
 *
 * Each group cites the reference interface it replaces (paths relative to the
 * reference checkout, gfnerf/bindings/...).
 */
#ifndef GFNERF_B200_H
#define GFNERF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GF_N_LEVELS 16          /* field/Hash3DAnchored.h:18 N_LEVELS   */
#define GF_N_CHANNELS 2         /* field/Hash3DAnchored.h:17 N_CHANNELS */
#define GF_HASH_DIM 32          /* N_LEVELS * N_CHANNELS                */
#define GF_MAX_SAMPLE_PER_RAY 1024   /* PtsSampler/PersSampler_cuda.cu:9  */
#define GF_MAX_OCT_PER_RAY 1024      /* PtsSampler/PersSampler_cuda.cu:8  */
#define GF_TREE_NODE_BYTES 128  /* sizeof(TreeNode),  PtsSampler/PersSampler.h:40-49 */
#define GF_TRANS_INFO_BYTES 576 /* sizeof(TransInfo), PtsSampler/PersSampler.h:31-38 */
#define GF_N_PROS 12            /* PtsSampler/PersSampler.h:15 */
#define GF_GRAD_SCALE 128.0f    /* field/Hash3DAnchored_cuda.cu:209 grad_scale */

typedef enum {
  GF_OK = 0,
  GF_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, unsupported width) */
  GF_ERR_CUDA = -2,      /* a CUDA runtime call or launch failed; see gf_last_error()      */
  GF_ERR_UNSUPPORTED = -3
} gf_status;

/* ---- library ---------------------------------------------------------- */
const char* gf_last_error(void);
/* "gfnerf_b200 <semver> sm_100a" */
const char* gf_version(void);
/* number of kernel launches issued by this library in this process (all threads) */
int64_t gf_launch_count(void);

/* ---- Hash3DAnchored ---------------------------------------------------
 * Replaces Hash3DAnchoredForwardKernel / Hash3DAnchoredBackwardKernel and the
 * host glue Hash3DAnchoredFunction::{forward,backward}
 * (field/Hash3DAnchored_cuda.cu:11-79, 81-155, 160-239).
 *
 * Layouts (all row-major, contiguous):
 *   feat_f16   __half [n_levels*local_size, 2]   fp16 shadow of feat_pool.  Level l reads / scatters rows
 *              [l*local_size/2, l*local_size/2 + local_size): the reference adds feat_local_idx[l] = l*local_size
 *              (Hash3DAnchored.cpp:66-70) to a pointer to SCALARS (Hash3DAnchored_cuda.cu:38, :105), so consecutive
 *              levels overlap by half a window and rows >= 8.5*local_size are never touched.  Reproduced (a table
 *              trained by the reference only means something under this addressing); local_size must be even.
 *   prim_pool  int32  [16, n_volumes, 3]
 *   bias_pool  float  [16*n_volumes, 3], or NULL = all zeros (what the reference always has,
 *              Hash3DAnchored.cpp:57-62: rand_bias is never set) -- same arithmetic, three loads fewer per level
 *   pts        float  [n, 3]   (already (warp+1.5)/3, nerfacto_field.py:431)
 *   anchors    int64 [n] (anchor_i64=1, the reference dtype) or int32 [n]
 *   level_scales float[16] device table, see gf_hash_level_scales
 *   n may also come from device memory: if d_n_ptr != NULL the kernels use
 *   min(n, *d_n_ptr) points, so a producer on the same stream can hand over a
 *   data-dependent count without a host sync.
 */

/* Fills a device table with s_l = exp2f(7*l/15 + 3) evaluated ON THE DEVICE with
 * the reference's expression (Hash3DAnchored_cuda.cu:28).  h_copy (16 floats,
 * host, optional) receives the same values after a stream sync. */
int gf_hash_level_scales(float* d_scales16, float* h_copy16, void* stream);

/* feat_pool fp32 -> fp16 shadow (Hash3DAnchored_cuda.cu:185 `.to(kFloat16)`) */
int gf_hash_cast_table(const float* feat_f32, void* feat_f16, int64_t n_elems, void* stream);

/* out_f16: __half [n,32] (may be NULL), out_f32: float [n,32] (may be NULL);
 * both hold the fp16-rounded value the reference returns (:73-77,195). */
int gf_hash_forward(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                    const void* feat_f16, const int32_t* prim_pool, const float* bias_pool,
                    const float* level_scales,
                    const float* pts, const void* anchors, int anchor_i64,
                    void* out_f16, float* out_f32, void* stream);

/* Focal (block) stage: out_f16 = base_f16 + encode(pts) in fp16, the residual sub-encoder's features added to the
 * frozen global encoder's at the hash-feature level (gfnerf/nerfacto_field.py:477-489).  base_f16 / out_f16:
 * __half [n,32]; they may alias. */
int gf_hash_forward_residual(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                             const void* feat_f16, const int32_t* prim_pool, const float* bias_pool,
                             const float* level_scales, const float* pts, const void* anchors, int anchor_i64,
                             const void* base_f16, void* out_f16, void* stream);

/* grad_in: fp32 [n,32] dL/dout (unscaled; grad_in_is_scaled_f16=0) -- the kernel
 * applies the reference's x128 -> fp16 quantisation (:209) -- or __half [n,32]
 * already scaled by 128 (grad_in_is_scaled_f16=1, produced by gf_mlp_backward).
 * grad_table: float [n_levels*local_size, 2]; ACCUMULATED into (caller zeroes it),
 * in units of dL/dfeat (the /128 of :238 is applied per contribution).
 * grad_in_is_scaled_f16 is a bit set: bit 0 as above; bit 1 (value 2) leaves the table at
 * the x128 scale -- a caller that folds the division into its optimizer step
 * (gf_adam_step's grad_div) saves two multiplies per corner; exact, 128 is a power of two. */
int gf_hash_backward(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                     const int32_t* prim_pool, const float* bias_pool, const float* level_scales,
                     const float* pts, const void* anchors, int anchor_i64,
                     const void* grad_in, int grad_in_is_scaled_f16,
                     float* grad_table, void* stream);

/* The same for the levels [level_begin, level_end) only (rows level * local_size ... of grad_table): data-parallel
 * training scatters the table gradient in level groups and starts each group's all-reduce while the next group is
 * being scattered. */
int gf_hash_backward_levels(int64_t n, const int32_t* d_n_ptr, int32_t n_volumes, int64_t local_size,
                            const int32_t* prim_pool, const float* bias_pool, const float* level_scales,
                            const float* pts, const void* anchors, int anchor_i64,
                            const void* grad_in, int grad_in_is_scaled_f16,
                            float* grad_table, int level_begin, int level_end, void* stream);

/* Parity probe: rows int32 [n,16,8] = table row (level offset included) of the 8 corners of
 * every (point, level), order 000,001,...,111 (:48-55).  Not on the hot path. */
int gf_hash_corner_rows(int64_t n, int32_t n_volumes, int64_t local_size, const int32_t* prim_pool,
                        const float* bias_pool, const float* level_scales, const float* pts,
                        const void* anchors, int anchor_i64, int32_t* rows, void* stream);

/* ---- PersSampler -------------------------------------------------------
 * Replaces FindRayOctreeIntersectionKernel<false/true>, RayMarchKernel<false/true>
 * and PersSampler::GetSamples (PtsSampler/PersSampler_cuda.cu:53-152, 190-318,
 * 321-477).  tree_nodes / pers_trans are the reference's state blobs
 * (128 B TreeNode, 576 B TransInfo; PersSampler.h:31-49), search_order is the
 * uint8[64] table of PersSampler.cpp:137-151.
 *
 * One fused pass per ray (traverse + march), no host sync.  Outputs are written
 * for sample k of ray r at slot r*1024+k ("dense", the reference layout
 * [R,1024,...]); untouched slots are NOT written, so the caller zero-fills the
 * dense tensors when it needs the reference's padding (:437-444).
 */
typedef struct {
  float* world_pts;      /* [R,1024,3] or NULL */
  float* warp_pts;       /* [R,1024,3] */
  float* dirs;           /* [R,1024,3] or NULL */
  float* dists;          /* [R,1024]   */
  float* ts;             /* [R,1024]   */
  int64_t* anchors_i64;  /* [R,1024,3] (trans_idx, node_idx, block_idx) or NULL */
  int32_t* anchors_i32;  /* [R,1024,2] (trans_idx, node_idx)            or NULL */
  int64_t* pts_idx_start_end; /* [R,2] start = exclusive prefix of counts, or NULL */
  int32_t* counts;       /* [R] samples per ray (always written) */
  float* first_oct_dis;  /* [R] */
  int32_t* n_oct;        /* [R] leaves intersected per ray, or NULL */
  void* packed;          /* [R,1024] 32-byte records {warp x, y, z, unused | t, dist, trans_idx, node_idx}
                            (two float4, ints stored bit-wise) for gf_sampler_compact, or NULL */
} gf_sampler_out;

int gf_sampler_get_samples(int64_t n_rays, const float* rays_o, const float* rays_d_unit,
                           const float* noise /* [1024 + n_rays + 10] already x fineness */,
                           const void* tree_nodes, int64_t n_nodes,
                           const void* pers_trans, int64_t n_trans,
                           const uint8_t* search_order,
                           float global_near, float sample_l, int scale_by_dis,
                           int64_t max_oct_intersect_per_ray,
                           const gf_sampler_out* out, void* stream);

/* exclusive prefix sum of counts[R] -> offsets[R+1] (offsets[R] = total), int32;
 * also writes *d_total. Single launch, no host sync. */
int gf_sampler_scan_counts(int64_t n_rays, const int32_t* counts, int32_t* offsets,
                           int32_t* d_total, void* stream);

/* packed records [R,1024] -> CSR (sample s of ray r at offsets[r]+k); outputs:
 * pts01 = (warp+1.5)/3 float[V,3] (nerfacto_field.py:431), anchor = trans_idx int32[V],
 * node int32[V], t float[V], delta float[V], ray_id int32[V]. */
int gf_sampler_compact(int64_t n_rays, const int32_t* counts, const int32_t* offsets,
                       const void* packed,
                       float* c_pts01, int32_t* c_anchor, int32_t* c_node, float* c_t,
                       float* c_delta, int32_t* c_ray, void* stream);

/* MarkVistNodeKernel + the stat update + MarkInvalidNodes of
 * PersSampler::UpdateOctNodes (PersSampler_cuda.cu:518-655), compact layout.
 * weight_stats/alpha_stats/visit_cnt: int64 [n_nodes] state, updated in place;
 * tree_nodes blob updated in place (trans_idx := -1 for pruned leaves).
 * scratch: int64 [3*n_nodes] (adders + mark), overwritten. */
int gf_sampler_update_oct_nodes(int64_t n_rays, const int32_t* counts, const int32_t* offsets,
                                const int32_t* c_node, const float* weights, const float* alphas,
                                void* tree_nodes, int64_t n_nodes,
                                int64_t* weight_stats, int64_t* alpha_stats, int64_t* visit_cnt,
                                int64_t* scratch, void* stream);

/* The two halves of gf_sampler_update_oct_nodes, for data-parallel training: every rank votes on its own rays
 * (gf_sampler_vote fills scratch = {weight adders, alpha adders, visited mark} and atomicMax'es visit_cnt), the
 * ranks MAX-reduce scratch and visit_cnt (the votes are atomicMax'es in the reference, so the max over ranks is
 * what one process voting on all rays would have produced), then every rank applies the same votes
 * (gf_sampler_apply_votes) and the replicated octrees stay identical. */
int gf_sampler_vote(int64_t n_rays, const int32_t* counts, const int32_t* offsets, const int32_t* c_node,
                    const float* weights, const float* alphas, int64_t n_nodes, int64_t* visit_cnt,
                    int64_t* scratch, void* stream);
int gf_sampler_apply_votes(void* tree_nodes, int64_t n_nodes, int64_t* weight_stats, int64_t* alpha_stats,
                           const int64_t* scratch, void* stream);

/* PersOctree::PersOctree / ConstructTreeNode / GetVisiCams / DistanceSummary / ConstructTrans
 * (PtsSampler/PersSampler.cpp:12-26, 45-152, 516-831) -- HOST code, as in the reference: builds the octree over the
 * camera rig (c2w f32 [n,3,4], intri f32 [n,3,3], bound f32 [n,2] = near, far; host pointers) down to max_depth, with
 * the perspective-warp transform of every valid leaf.  bbox_side_len = 2^(bbox_levels - 1); n_rand_pts sample points
 * per leaf for the PCA (reference: 32^3); visi_res_w = width of the visibility pixel grid (reference: 128).
 * The result stays behind *handle; *n_nodes / *n_trans give the blob sizes (128 B / 576 B each, PersSampler.h:31-49).
 * gf_octree_build_fetch copies the blobs out (either pointer may be NULL) and frees the handle. */
int gf_octree_build(int64_t max_depth, float bbox_side_len, float split_dist_thres, const float* c2w, const float* intri,
                    const float* bound, int64_t n_cams, uint32_t seed, int64_t n_rand_pts, int64_t visi_res_w,
                    void** handle, int64_t* n_nodes, int64_t* n_trans);
int gf_octree_build_fetch(void* handle, void* tree_nodes_out, void* pers_trans_out);
/* uint8 [64]: children in front-to-back order for each of the 8 ray octants (PersSampler.cpp:137-151) */
int gf_octree_search_order(uint8_t* out64);

/* PersOctree::ProcOctree (PtsSampler/PersSampler.cpp:154-417) -- HOST code, like the reference's (which copies the
 * node blob to the CPU, rebuilds it and uploads it again): all pointers are host pointers, no stream.
 * compact: drop leaves with trans_idx < 0 from their parents, turn childless interior nodes into leaves (repeat),
 * splice out single-child chains, keep interior nodes and valid leaves in their old order.  subdivide: depth-first
 * renumbering in which every leaf with visit_cnt > 4 (or every leaf, brute_force) becomes an interior node followed
 * by its eight new leaf children (same trans_idx, statistics inherited, the parent's reset to 1000).
 * nodes_in: n_in TreeNode blobs (128 B each, PersSampler.h:31-40); *_stats_in / visit_cnt_in: int64 [n_in].
 * nodes_out == NULL: size query, only *n_out is written.  Otherwise `capacity` nodes of room in nodes_out /
 * weight_stats_out / alpha_stats_out (int64); visit counts restart at 0 in the reference, so none are returned. */
int gf_octree_proc(const void* nodes_in, int64_t n_in, const int64_t* weight_stats_in, const int64_t* alpha_stats_in,
                   const int64_t* visit_cnt_in, int compact, int subdivide, int brute_force, void* nodes_out,
                   int64_t* weight_stats_out, int64_t* alpha_stats_out, int64_t capacity, int64_t* n_out);

/* The same ProcOctree ON THE DEVICE (csrc/octree_device.cu): every pointer is a device pointer, one single-CTA kernel
 * on `stream`, byte-identical output to gf_octree_proc (which stays as the host-side checker), and the node blob never
 * leaves HBM -- the reference's ProcOctree is a D2H copy + host rebuild + H2D copy every compact_freq steps and twice
 * per subdivision milestone (PersSampler.cpp:154-417).  nodes_out / *_stats_out: room for `capacity` nodes (worst
 * case 9 * n_in with subdivide, n_in without); scratch: gf_octree_proc_device_scratch_bytes(n_in) bytes, 16-byte
 * aligned.  *d_n_out (device int64) = nodes written.  *d_error (device int32, OR-ed): 1 = the root was pruned,
 * 2 = a removed node is still linked (compact = 0 on a pruned tree; the reference CHECK-fails), 4 = capacity too
 * small (*d_n_out = nodes needed).  The host reads d_n_out / d_error when it needs them (8 + 4 bytes). */
int64_t gf_octree_proc_device_scratch_bytes(int64_t n_in);
int gf_octree_proc_device(const void* nodes_in, int64_t n_in, const int64_t* weight_stats_in,
                          const int64_t* alpha_stats_in, const int64_t* visit_cnt_in, int compact, int subdivide,
                          int brute_force, void* nodes_out, int64_t* weight_stats_out, int64_t* alpha_stats_out,
                          int64_t capacity, void* scratch, int64_t scratch_bytes, int64_t* d_n_out, int32_t* d_error,
                          void* stream);

/* PersOctree::MarkInvisibleNodes (MarkInvisibleNodesKernel + CheckVisible, PersSampler_cuda.cu:680-742; run at the
 * subdivision milestones, :657-677): every node whose bounding sphere (radius 0.707 * side_len) no camera sees gets
 * trans_idx = -1, in place in the device node blob.  w2c f32 [n_cams,3,4], intri f32 [n_cams,3,3], bounds f32
 * [n_cams,2] (device).  Same bits as the reference's kernel built by nvcc (arithmetic order: csrc/octree_device.cu). */
int gf_octree_mark_invisible(void* tree_nodes, int64_t n_nodes, const float* w2c, const float* intri,
                             const float* bounds, int64_t n_cams, void* stream);

/* SetBlockIdxsNearestKernel (PersSampler_cuda.cu:746-766), the device half of PersOctree::UpdateBlockIdxs (:767-798;
 * the caller compacts afterwards): block_idx of every node = index of the nearest of `centers` f32 [n_blocks,3]
 * (device), the first of equal minima, -1 if none is closer than 1e9; in place in the device node blob. */
int gf_octree_set_block_idxs(void* tree_nodes, int64_t n_nodes, const float* centers, int64_t n_blocks, void* stream);

/* PersSampler::GetPointsAnchors (GetRaysTreeNodesIntersectsKernel + GetTreeNodeIdxFromTsKernel, :799-853, 924-980;
 * the proposal-sampler variant, cold): anchors i64 [n_rays, n_pts_per_ray] = index of the LEAF whose slab interval
 * along the ray contains t_cur (= (t_start + t_end) / 2, f32 [n_rays, n_pts_per_ray]), -1 if none; a sample exactly
 * on a face shared by two leaves gets the larger index (the reference's stores race there). */
int gf_sampler_points_anchors(int64_t n_rays, int64_t n_pts_per_ray, const float* rays_o, const float* rays_d,
                              const float* t_cur, const void* tree_nodes, int64_t n_nodes, int64_t* anchors,
                              void* stream);

/* PersOctree::ConstructEdgePool (PersSampler.cpp:833-893), HOST code: the faces shared by neighbouring valid leaves
 * as 64-byte EdgePool records (PersSampler.h:50-56).  edges_out == NULL: size query. */
int gf_octree_edge_pool(const void* nodes_in, int64_t n_nodes, void* edges_out, int64_t capacity, int64_t* n_out);
/* GetEdgeSamplesKernel (:479-495): point edge_idx[i] / edge_coords[i] (f32 [n,2] in [-1,1]^2) of the edge pool
 * (device copy), warped by the transforms of both leaves: out_pts f32 [n,2,3], out_idx i64 [n,2] (trans indices).
 * The random draws (:498-499) stay with the caller. */
int gf_sampler_edge_samples(int64_t n_pts, const void* edge_pool, int64_t n_edges, const void* pers_trans,
                            const int64_t* edge_idx, const float* edge_coords, float* out_pts, int64_t* out_idx,
                            void* stream);

/* QueryFrameTransform for arbitrary points (TransQueryFrameKernel, :854-922) */
int gf_sampler_trans_query_frame(int64_t n_pts, const void* tree_nodes, int64_t n_nodes,
                                 const void* pers_trans, const int64_t* anchors,
                                 const float* world_pts, float* warp_pts, void* stream);

/* ---- compositing --------------------------------------------------------
 * Replaces RaySamples.get_weights_f2nerf (nerfstudio/cameras/rays.py:178-200)
 * and RGBRenderer.combine_rgb / DepthRenderer('expected') / AccumulationRenderer
 * (nerfstudio/model_components/renderers.py:97-110, 269-283, 220), one warp per
 * ray, shuffle scan.  Samples of ray r are [offsets[r], offsets[r+1]).
 * Per-sample outputs (weights, alphas, trans) may be NULL.
 * depth is the UNCLIPPED expected depth sum(w t)/(sum(w)+1e-10); the caller
 * applies the global clip of renderers.py:281 with t_max = gf_composite's
 * d_tmax output (max t over valid samples; min is 0 because of padding).
 */
int gf_composite_forward(int64_t n_rays, const int32_t* offsets,
                         const float* sigma, const float* delta, const float* rgb /*[V,3]*/,
                         const float* t,
                         float* weights, float* alphas, float* trans,
                         float* out_rgb /*[R,3]*/, float* out_depth /*[R]*/, float* out_acc /*[R]*/,
                         float* d_tmax /* [1], atomicMax'ed; caller zeroes */, void* stream);

/* rgb / t / out_rgb / out_depth / out_acc may be NULL in gf_composite_forward (weights only).
 *
 * Backward: d_sigma[V] (and d_rgb[V,3] if not NULL) from any of: g_rgb [R,3] (gradient of
 * out_rgb; needs rgb), g_acc [R] (gradient of out_acc), g_w [V] (gradient flowing into the
 * per-sample weights themselves, the operator-API path where the renderers are torch ops).
 * trans[V] is the transmittance the forward wrote. */
int gf_composite_backward(int64_t n_rays, const int32_t* offsets,
                          const float* sigma, const float* delta, const float* rgb,
                          const float* trans, const float* g_rgb, const float* g_acc, const float* g_w,
                          float* d_sigma, float* d_rgb, void* stream);

/* ---- fused field MLP ----------------------------------------------------
 * Replaces MLPNetwork x2 (gfnerf/mlp.py:25-57 as built at
 * gfnerf/nerfacto_field.py:174-179,217-227), trunc_exp(x+1) (:499),
 * the tcnn SH degree-4 direction encoding (:152-158,521), the appearance
 * embedding lookup (:530-537) and the concat (:540-547).
 * fp16 tensor-core math, fp32 accumulate.  Hidden width H = 64 (nerfstudio's default, csrc/mlp_tc.cu) or H = 128 (the
 * reference's shipped gf-nerf config, gfnerf/config.py:124-125; csrc/mlp_tc128.cu); both stacks have the same width.
 *
 * params: one fp32 blob, torch nn.Linear layout (weight [out,in] row-major, then bias):
 *   base.0: W[H,32] b[H] ; base.1: W[16,H] b[16]
 *   head.0: W[H,63] b[H] ; head.1: W[H,H] b[H] ; head.2: W[3,H] b[3]
 * (gf_mlp_param_count(H) floats).  Head input order: SH(16) | geo(15) | emb(32).
 */
int64_t gf_mlp_param_count(int hidden);   /* -1 if the width is not built */
/* 32-bit words of ReLU masks per sample that gf_mlp_forward writes and gf_mlp_backward reads: 8 (H = 64), 16 (H = 128);
 * -1 if the width is not built */
int gf_mlp_mask_words(int hidden);

/* Per-RAY part of the head's first layer (fp32):
 *   ray_bias[r][j] = b2[j] + W2[j][0:16] . SH4(dir_r) + W2[j][31:63] . emb_r
 * SH4 = tcnn SphericalHarmonics degree 4 on (dir+1)/2, fp16-rounded (nerfacto_field.py:64-70,
 * 152-158, 521); emb_r = embedding_appearance(rel_camera_index of ray r) (:530-537), NULL = zeros.
 * ray_dirs [R,3] unit, ray_emb [R,32], ray_bias [R,H]. */
int gf_mlp_ray_bias(int64_t n_rays, int hidden, const float* params, const float* ray_dirs,
                    const float* ray_emb, float* ray_bias, void* stream);

/* feat_f16 __half [n,32] (the hash encoding), ray_id int32 [n] -> sigma [n] = exp(h0 + 1),
 * rgb [n,3] = sigmoid(head).
 * relu_masks == NULL (inference): plain fp16 weights / activations, fp32 accumulate (outputs within ~1e-3 of the
 * reference's fp32 nn.Linear stack, gfnerf/mlp.py:45-57).
 * relu_masks != NULL (training): uint32 [n][gf_mlp_mask_words(H)] = [n][2][H / 16], 16-byte aligned.  Split precision: weights and hidden activations
 * are carried as fp16 pairs hi + lo (three tensor-core products per layer), so pre-activations -- and with them the
 * ReLU masks -- agree with the fp32 reference far inside fp16 rounding (outputs within ~1e-4).  Written per sample
 * and per column half of the hidden layers, one word per 32 columns: H = 64 {mask of base.0's ReLU, of head.0's, of
 * head.1's, 0}, H = 128 {base.0 x2, head.0 x2, head.1 x2, 0, 0}; bit layout private to the library
 * (csrc/mlp_tc_common.cuh mask_bits_of_pair).  gf_mlp_backward consumes it. */
int gf_mlp_forward(int64_t n, const int32_t* d_n_ptr, int hidden, const float* params,
                   const void* feat_f16, const int32_t* ray_id, const float* ray_bias,
                   float* sigma, float* rgb, void* relu_masks, void* stream);

/* d_sigma [n], d_rgb [n,3] -> d_feat_scaled_f16 __half [n,32] (= dL/dfeat * 128, the reference's
 * grad_in, Hash3DAnchored_cuda.cu:209), d_params fp32 [param_count] ACCUMULATED (all of it except
 * the SH / emb columns of W2 and b2), d_ray_bias fp32 [R,H] ACCUMULATED (caller zeroes).
 * d_params == d_ray_bias == NULL: frozen MLP (focal stage), only d_feat is produced.
 * Hidden activations are recomputed (plain fp16); the ReLU masks are the forward's (relu_masks, required): a
 * recomputed fp16 mask flips ~1e-3 of the units near zero, which alone costs 1-2 % of every gradient in L2.
 * grad_scale: internal loss scale of the fp16 gradient
 * fragments (a power of two near 1/|d_rgb|, e.g. the ray count); results are unscaled. */
int gf_mlp_backward(int64_t n, const int32_t* d_n_ptr, int hidden, const float* params,
                    const void* feat_f16, const int32_t* ray_id, const float* ray_bias,
                    const void* relu_masks, const float* d_sigma, const float* d_rgb,
                    void* d_feat_scaled_f16, float* d_params, float* d_ray_bias, float grad_scale,
                    void* stream);

/* d_ray_bias [R,H] -> d_params (SH / emb columns of W2, b2; ACCUMULATED; may be NULL) and
 * d_ray_emb [R,32] (ACCUMULATED; may be NULL). */
int gf_mlp_ray_bias_backward(int64_t n_rays, int hidden, const float* params, const float* ray_dirs,
                             const float* ray_emb, const float* d_ray_bias, float* d_params,
                             float* d_ray_emb, void* stream);

/* ---- loss + optimiser tail ------------------------------------------------
 * CharbonnierLoss (nerfstudio/model_components/losses.py:73-84, eps 1e-6,
 * out_norm 'b'): loss = sum(sqrt((x-y)^2+eps^2))/R.  Writes g_rgb = dL/drgb and
 * accumulates the loss into d_loss[0] (caller zeroes).
 */
int gf_charbonnier(int64_t n_rays, const float* rgb, const float* target, float eps,
                   float* g_rgb, float* d_loss, void* stream);

/* S3IM (nerfstudio/model_components/losses.py:713-794; gf-nerf: ksize 4, stride 4, repeat 10, patch_h 32,
 * gfnerf/nerfacto.py:186-197): 1 - SSIM between the rendered and target colours laid out as a virtual image
 * [3, patch_h, n_virtual / patch_h] through index (int64 [n_virtual] = arange(R) followed by repeat-1 random
 * permutations of the rays).  ACCUMULATES mult * loss into d_loss[0] and mult * dloss/dsrc into g_src [R,3]
 * (either may be NULL), so it composes with gf_charbonnier on the same buffers. */
int gf_s3im(int64_t n_rays, int64_t n_virtual, const int64_t* index, const float* src, const float* target,
            int patch_h, int ksize, int stride, float mult, float* g_src, float* d_loss, void* stream);

/* ---- image-quality metrics of a rendered view (csrc/metrics.cu) -----------------------------------------------
 * nerfstudio's Model.get_image_metrics_and_images for nerfacto (nerfstudio/models/nerfacto.py): torchmetrics'
 * PeakSignalNoiseRatio(data_range=1.0) and functional structural_similarity_index_measure with its defaults, one
 * call per image.  pred, gt: float [n_images, height, width, 3], contiguous, interleaved RGB, rows in the pixel
 * order of the render loop (row-major), both 16-byte aligned.  Outputs float [n_images] each:
 *   mse[b]  = sum (p - g)^2 / (3 H W), summed in double;
 *   psnr[b] = 10 log10(1 / mse[b]); +inf when mse is 0;
 *   ssim[b] = mean over the 3 (H - 10) (W - 10) (channel, y, x) whose 11 x 11 window lies inside the image (the
 *             region torchmetrics keeps after its reflect pad and crop) of
 *             ((2 mu_p mu_g + C1)(2 s_pg + C2)) / ((mu_p^2 + mu_g^2 + C1)(s_p^2 + s_g^2 + C2)),
 *             window = outer product of the normalised Gaussian of size 11, sigma 1.5; C1 = (0.01 L)^2,
 *             C2 = (0.03 L)^2 with L = max(max p - min p, max g - min g) over image b.  Two constant images give
 *             L = 0 and NaN, as the formula does.
 * scratch: gf_image_metrics_scratch_bytes(n_images, height, width) bytes, 16-byte aligned (-1: sizes invalid).
 * Requires n_images >= 1 and height, width >= 11.  No host sync and no allocation: the call can be captured in a
 * CUDA graph.  The work partition depends only on the sizes, so the results are bit-identical from run to run and the
 * same for an image alone or inside a batch. */
int64_t gf_image_metrics_scratch_bytes(int64_t n_images, int64_t height, int64_t width);
int gf_image_metrics(int64_t n_images, int64_t height, int64_t width, const float* pred, const float* gt,
                     float* psnr, float* ssim, float* mse, void* scratch, int64_t scratch_bytes, void* stream);

/* torch.optim.Adam (no amsgrad, no weight decay) as configured at
 * gfnerf/config.py:132-135 / Hash3DAnchored.cpp:146-150.  step >= 1.
 * If shadow_f16 != NULL it is refreshed with the updated parameters.
 * grad is divided by grad_div first (world size for the DDP mean) and zeroed if
 * zero_grad != 0. */
int gf_adam_step(int64_t n, float* param, float* grad, float* exp_avg, float* exp_avg_sq,
                 void* shadow_f16, float lr, float beta1, float beta2, float eps,
                 int64_t step, float grad_div, int zero_grad, void* stream);

/* The trainer's NaN-gradient guard (nerfstudio/engine/trainer.py:416-426: scan every parameter's gradient, skip the
 * optimizer step if any is NaN) without its per-parameter host syncs: gf_grad_nan_scan ORs 1 into *flag (device
 * int32, caller zeroes) if grad holds a NaN; gf_adam_step_guarded is gf_adam_step that leaves param / moments
 * untouched (and only zero-fills the gradient) when *skip_flag != 0. */
int gf_grad_nan_scan(int64_t n, const float* grad, int32_t* flag, void* stream);
int gf_adam_step_guarded(int64_t n, float* param, float* grad, float* exp_avg, float* exp_avg_sq,
                         void* shadow_f16, float lr, float beta1, float beta2, float eps,
                         int64_t step, float grad_div, int zero_grad, const int32_t* skip_flag, void* stream);
/* gf_adam_step_guarded whose step count lives on the device: the bias corrections use *d_step + 1 and *d_step is
 * advanced only when the step was applied -- a step skipped by the NaN guard does not exist for the optimizer, as in
 * the reference, which skips optimizer.step() altogether (trainer.py:416-426).  d_step: device int64, starts at 0. */
int gf_adam_step_counted(int64_t n, float* param, float* grad, float* exp_avg, float* exp_avg_sq,
                         void* shadow_f16, float lr, float beta1, float beta2, float eps,
                         int64_t* d_step, float grad_div, int zero_grad, const int32_t* skip_flag, void* stream);

/* ---- data-parallel exchange over NVLink peer memory (SURVEY 8e; csrc/peer.cu) ----------------------------------
 * Replaces the DDP gradient all-reduce + replicated optimizer step of the reference's multi-GPU setup
 * (gfnerf/gf_pipeline.py:136-138, nerfstudio/engine/optimizers.py:125-137) for one node: one process per GPU, every
 * rank's exchange buffers mapped into every other rank (CUDA IPC).
 *
 * gf_peer_alloc / free: a zero-filled device allocation that can be exported (cudaMalloc; sub-blocks of a caching
 * allocator cannot).  gf_peer_export: its 64-byte IPC handle.  gf_peer_import / close: map / unmap a peer's handle
 * (peer access is enabled lazily). */
int gf_peer_alloc(int64_t bytes, void** dptr);
int gf_peer_free(void* dptr);
int gf_peer_export(const void* dptr, void* handle64);
int gf_peer_import(const void* handle64, void** dptr);
int gf_peer_close(void* dptr);
/* Cross-GPU barrier as one single-CTA kernel on `stream`.  flag_ptrs: host array [world] of device pointers, entry r =
 * rank r's uint32[world] flag array (peer-mapped, zero at start).  epoch: 1, 2, 3, ... -- the same on every rank, one
 * flag array per barrier site.  d_local_flag (may be NULL): this rank's int32 flag; d_any_flag (may be NULL) receives
 * the OR over all ranks.  A wait longer than ~2 s sets *d_error (int32, may be NULL) instead of hanging. */
int gf_peer_barrier(int world, int rank, uint32_t epoch, void* const* flag_ptrs, const int32_t* d_local_flag,
                    int32_t* d_any_flag, int32_t* d_error, void* stream);
/* dst[i] = max over ranks r of src_ptrs[r][i], int64 [n]: all-reduce(MAX) of the octree votes (the adders / marks of
 * MarkVistNodeKernel and the visit counts, PersSampler_cuda.cu:518-574) as peer loads, between gf_sampler_vote and
 * gf_sampler_apply_votes.  The caller orders it behind a gf_peer_barrier ("every rank's votes are complete") and
 * alternates between two vote buffers per rank, so no second barrier is needed. */
int gf_peer_max_i64(int world, int64_t n, void* const* src_ptrs, int64_t* dst, void* stream);

/* Reduce-scatter + Adam + all-gather of one flat fp32 parameter array of n elements in ONE kernel: for the elements
 * [lo, hi) this rank owns (multiples of 4), sum grad_ptrs[0..world) (host array of device pointers to every rank's
 * gradient array, summed in rank order -- bit-identical whoever computes it), divide by grad_div, apply torch.optim.Adam
 * (as gf_adam_step_counted: bias corrections from *d_step + 1, *d_step advanced unless skipped) to param / exp_avg /
 * exp_avg_sq, and -- if shadow_ptrs != NULL -- store the updated elements as fp16 into EVERY rank's shadow array.
 * Gradients are left untouched (peers may still be reading them): the caller zeroes them after the closing barrier.
 * *skip_flag != 0: nothing is updated. */
int gf_peer_reduce_adam(int world, int64_t n, int64_t lo, int64_t hi, void* const* grad_ptrs, float* param,
                        float* exp_avg, float* exp_avg_sq, void* const* shadow_ptrs, float lr, float beta1,
                        float beta2, float eps, int64_t* d_step, float grad_div, const int32_t* skip_flag,
                        void* stream);

/* ---- ray generation (SURVEY 8f rank 4: the step before the path) --------
 * Cameras.generate_rays for PERSPECTIVE cameras without distortion (nerfstudio/cameras/cameras.py:583-727, with
 * GF-NeRF's lookat_directions :704,723): cam_idx int64 [n], coords_yx f32 [n,2] = pixel (y, x) as the pixel samplers
 * give them (index + 0.5); c2w f32 [n_cams,3,4]; fx, fy, cx, cy f32 [n_cams].  Outputs f32: origins [n,3] = c2w[:, 3],
 * directions [n,3] (unit), lookat [n,3] = c2w[:, 2], pixel_area [n] = dx * dy from the one-pixel-offset directions,
 * dir_norm [n] (metadata["directions_norm"]); lookat / pixel_area / dir_norm may be NULL. */
int gf_generate_rays(int64_t n_rays, const int64_t* cam_idx, const float* coords_yx, const float* c2w,
                     const float* fx, const float* fy, const float* cx, const float* cy, int64_t n_cams,
                     float* origins, float* directions, float* lookat, float* pixel_area, float* dir_norm,
                     void* stream);

/* ---- error-map feedback of the focal stage (SURVEY 8f rank 4) -------------
 * gfnerf/gf_pipeline.py:180-185 + TrainDataloader._update_error_map (nerfstudio/data/utils/dataloaders.py:140-142):
 * error[i] = sum over the 3 channels of |gt - pred|; error_map[indices[i,0], indices[i,1], indices[i,2]] = error[i].
 * indices int64 [n,3] = (image slot in the cached batch, y, x) as the pixel sampler drew them; error_map f32
 * [n_images, height, width] (the reference's trailing singleton channel is a view of the same memory).
 * error_out f32 [n] (may be NULL) also receives the per-ray error.  An index out of range (after one wrap of a
 * negative index, as torch does) writes nothing and sets *bad_index_flag (device int32, may be NULL, caller zeroes)
 * -- torch raises IndexError there; the host wrapper turns the flag into the same error. */
int gf_error_map_update(int64_t n_rays, const int64_t* indices, const float* pred_rgb, const float* gt_rgb,
                        int64_t n_images, int64_t height, int64_t width, float* error_map, float* error_out,
                        int32_t* bad_index_flag, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GFNERF_B200_H */
