"""ctypes binding of the C-ABI library (include/gfnerf_b200.h).

This is the only way the Python host layer reaches the CUDA kernels.  There is no
CPU fallback: if libgfnerf_b200.so is missing or a call fails, this raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgfnerf_b200.so")

_lib = None

_vp, _i64, _i32, _f32, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_int


class SamplerOut(C.Structure):
    """gf_sampler_out of include/gfnerf_b200.h"""
    _fields_ = [(n, _vp) for n in ("world_pts", "warp_pts", "dirs", "dists", "ts", "anchors_i64", "anchors_i32",
                                   "pts_idx_start_end", "counts", "first_oct_dis", "n_oct", "packed")]


_SIGS = {
    "gf_hash_level_scales": [_vp, _vp, _vp],
    "gf_hash_cast_table": [_vp, _vp, _i64, _vp],
    "gf_hash_forward": [_i64, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp],
    "gf_hash_forward_residual": [_i64, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp],
    "gf_hash_backward": [_i64, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _int, _vp, _int, _vp, _vp],
    "gf_hash_backward_levels": [_i64, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _int, _vp, _int, _vp, _int, _int, _vp],
    "gf_hash_corner_rows": [_i64, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _int, _vp, _vp],
    "gf_sampler_get_samples": [_i64, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _f32, _f32, _int, _i64,
                               C.POINTER(SamplerOut), _vp],
    "gf_sampler_scan_counts": [_i64, _vp, _vp, _vp, _vp],
    "gf_sampler_compact": [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "gf_sampler_update_oct_nodes": [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp],
    "gf_sampler_vote": [_i64, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp],
    "gf_sampler_apply_votes": [_vp, _i64, _vp, _vp, _vp, _vp],
    "gf_octree_build": [_i64, _f32, _f32, _vp, _vp, _vp, _i64, C.c_uint32, _i64, _i64, _vp, _vp, _vp],
    "gf_octree_build_fetch": [_vp, _vp, _vp],
    "gf_octree_search_order": [_vp],
    "gf_octree_proc": [_vp, _i64, _vp, _vp, _vp, _int, _int, _int, _vp, _vp, _vp, _i64, _vp],
    "gf_octree_proc_device": [_vp, _i64, _vp, _vp, _vp, _int, _int, _int, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp],
    "gf_octree_mark_invisible": [_vp, _i64, _vp, _vp, _vp, _i64, _vp],
    "gf_octree_set_block_idxs": [_vp, _i64, _vp, _i64, _vp],
    "gf_sampler_points_anchors": [_i64, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp],
    "gf_octree_edge_pool": [_vp, _i64, _vp, _i64, _vp],
    "gf_sampler_edge_samples": [_i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp],
    "gf_sampler_trans_query_frame": [_i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp],
    "gf_generate_rays": [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp],
    "gf_error_map_update": [_i64, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp],
    "gf_composite_forward": [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "gf_composite_backward": [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "gf_mlp_ray_bias": [_i64, _int, _vp, _vp, _vp, _vp, _vp],
    "gf_mlp_forward": [_i64, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "gf_mlp_backward": [_i64, _vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp],
    "gf_mlp_ray_bias_backward": [_i64, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "gf_s3im": [_i64, _i64, _vp, _vp, _vp, _int, _int, _int, _f32, _vp, _vp, _vp],
    "gf_charbonnier": [_i64, _vp, _vp, _f32, _vp, _vp, _vp],
    "gf_grad_nan_scan": [_i64, _vp, _vp, _vp],
    "gf_adam_step_guarded": [_i64, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _i64, _f32, _int, _vp, _vp],
    "gf_peer_alloc": [_i64, _vp],
    "gf_peer_free": [_vp],
    "gf_peer_export": [_vp, _vp],
    "gf_peer_import": [_vp, _vp],
    "gf_peer_close": [_vp],
    "gf_peer_barrier": [_int, _int, C.c_uint32, _vp, _vp, _vp, _vp, _vp],
    "gf_peer_max_i64": [_int, _i64, _vp, _vp, _vp],
    "gf_peer_reduce_adam": [_int, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _vp, _f32, _vp, _vp],
    "gf_adam_step_counted": [_i64, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _vp, _f32, _int, _vp, _vp],
    "gf_adam_step": [_i64, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _i64, _f32, _int, _vp],
}

EXPORTS = ["gf_last_error", "gf_version", "gf_launch_count", "gf_mlp_param_count", "gf_mlp_mask_words",
           "gf_octree_proc_device_scratch_bytes"] + sorted(_SIGS)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python gf-nerf_b200/build.py` "
                "(there is no CPU or PyTorch fallback for the GF-NeRF hot path)")
        L = C.CDLL(LIB_PATH)
        L.gf_last_error.restype = C.c_char_p
        L.gf_version.restype = C.c_char_p
        L.gf_launch_count.restype = C.c_int64
        for name, sig in list(_SIGS.items()) + [("gf_mlp_param_count", [_int]), ("gf_mlp_mask_words", [_int]),
                                                   ("gf_octree_proc_device_scratch_bytes", [_i64])]:
            try:
                fn = getattr(L, name)
            except AttributeError as e:  # a stale build: fail loudly, never fall back
                raise RuntimeError(f"{LIB_PATH} does not export {name}; rebuild with "
                                   "`python gf-nerf_b200/build.py --force`") from e
            fn.argtypes = sig
            fn.restype = C.c_int64 if name in ("gf_mlp_param_count", "gf_octree_proc_device_scratch_bytes") else _int
        _lib = L
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RuntimeError(f"gfnerf_b200 {what} failed ({rc}): {lib().gf_last_error().decode()}")


def ptr(t):
    """device (or host) address of a tensor, None -> NULL"""
    if t is None:
        return None
    assert t.is_contiguous(), "gfnerf_b200 kernels need contiguous tensors"
    return t.data_ptr()


def cur_stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("gfnerf_b200: tensor is not on a CUDA device (there is no CPU path)")


def launch_count() -> int:
    return int(lib().gf_launch_count())
