"""Image-quality metrics of rendered views on the device: PSNR, SSIM and MSE per image in one kernel sequence
(`gf_image_metrics`, csrc/metrics.cu).  The conventions are those of nerfstudio's nerfacto evaluation -- torchmetrics'
`PeakSignalNoiseRatio(data_range=1.0)` and functional `structural_similarity_index_measure` with its defaults, one
call per image; see include/gfnerf_b200.h.  `evaluate_views` is the held-out evaluation loop around them."""
import time
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib


def image_metrics(pred: torch.Tensor, gt: torch.Tensor) -> Dict[str, torch.Tensor]:
    """pred, gt: fp32 CUDA tensors [H, W, 3] or [B, H, W, 3] (interleaved RGB, rows in render order, H, W >= 11).
    Returns {"psnr", "ssim", "mse"}: fp32 device tensors [B] ([1] for a single image).  Launches on the current stream
    and does not synchronise."""
    if not isinstance(pred, torch.Tensor) or not isinstance(gt, torch.Tensor):
        raise RuntimeError("image_metrics: pred and gt must be tensors")
    _lib.require_cuda(pred, gt)
    if pred.dtype != torch.float32 or gt.dtype != torch.float32:
        raise RuntimeError(f"image_metrics: pred and gt must be float32, got {pred.dtype} and {gt.dtype}")
    if pred.shape != gt.shape or pred.dim() not in (3, 4) or pred.shape[-1] != 3:
        raise RuntimeError(f"image_metrics: pred and gt must both be [H,W,3] or [B,H,W,3], got {tuple(pred.shape)} "
                           f"and {tuple(gt.shape)}")
    if pred.device != gt.device:
        raise RuntimeError(f"image_metrics: pred is on {pred.device}, gt on {gt.device}")
    B, H, W = (1, *pred.shape[:2]) if pred.dim() == 3 else tuple(pred.shape[:3])
    pred, gt = (_aligned(t.detach()) for t in (pred, gt))
    with torch.cuda.device(pred.device):
        n_scratch = int(_lib.lib().gf_image_metrics_scratch_bytes(B, H, W))
        scratch = torch.empty(max(n_scratch, 0), dtype=torch.uint8, device=pred.device)
        out = torch.empty((3, B), dtype=torch.float32, device=pred.device)
        _lib.check(_lib.lib().gf_image_metrics(B, H, W, _lib.ptr(pred), _lib.ptr(gt), _lib.ptr(out[0]),
                                               _lib.ptr(out[1]), _lib.ptr(out[2]), _lib.ptr(scratch), n_scratch,
                                               _lib.cur_stream()), "gf_image_metrics")
    return {"psnr": out[0], "ssim": out[1], "mse": out[2]}


def _aligned(t: torch.Tensor) -> torch.Tensor:
    """contiguous and 16-byte aligned (the kernels load 16-byte blocks); a view into the middle of a tensor is copied"""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def evaluate_views(model, cameras, images, camera_indices: Optional[Sequence[int]] = None, route_blocks: bool = False
                   ) -> Tuple[Dict[str, float], List[Dict[str, float]]]:
    """The body of nerfstudio's `Pipeline.get_average_eval_image_metrics` (nerfstudio/pipelines/base_pipeline.py)
    without the datamanager.  `cameras`: a `Cameras` with `width` and `height` set; `images`: one ground truth per
    evaluated camera, [H, W, 3] fp32, on the device or the host; `camera_indices`: the cameras to evaluate (default:
    all, in order).  Per view: the frame's rays (`gf_generate_rays`) as an [H, W] bundle ->
    `model.get_outputs_for_camera_ray_bundle` -> `model.get_image_metrics_and_images`, plus `num_rays_per_sec`
    = H * W / wall time and `fps` = 1 / wall time, host clock from the render to the metrics' `.item()`.  The bundle
    has no `rel_camera_indices`: the model picks the appearance embedding by its nearest-camera rule, as the
    reference's evaluation does.  route_blocks: passed to `get_outputs_for_camera_ray_bundle` (a focal-stage model
    evaluated with every chunk's own block table).  Returns (averages: the mean of every key plus `psnr_std` and `ssim_std`, the
    unbiased std of torch.std_mean as nerfstudio reports it; per_image: one dict per view)."""
    from .rays import RayBundle
    idx = list(range(len(cameras))) if camera_indices is None else [int(i) for i in camera_indices]
    if len(images) != len(idx):
        raise RuntimeError(f"evaluate_views: {len(images)} images for {len(idx)} cameras")
    H, W = int(cameras.height), int(cameras.width)
    per_image = []
    for i, gt in zip(idx, images):
        if tuple(gt.shape) != (H, W, 3):
            raise RuntimeError(f"evaluate_views: ground truth of camera {i} is {tuple(gt.shape)}, the camera renders "
                               f"({H}, {W}, 3)")
        rays = cameras.generate_frame_rays(i)
        bundle = RayBundle(origins=rays.origins.view(H, W, 3), directions=rays.directions.view(H, W, 3),
                           lookat_directions=rays.lookat_directions.view(H, W, 3),
                           pixel_area=rays.pixel_area.view(H, W, 1), camera_indices=rays.camera_indices.view(H, W, 1),
                           metadata=rays.metadata)
        torch.cuda.synchronize(rays.origins.device)
        t0 = time.perf_counter()
        outputs = model.get_outputs_for_camera_ray_bundle(bundle, route_blocks=route_blocks)
        metrics, _ = model.get_image_metrics_and_images(outputs, {"image": gt})
        dt = time.perf_counter() - t0
        metrics["num_rays_per_sec"] = H * W / dt
        metrics["fps"] = 1.0 / dt
        per_image.append(metrics)
    averages = {}
    for key in per_image[0] if per_image else ():
        vals = torch.tensor([m[key] for m in per_image], dtype=torch.float64)
        if key in ("psnr", "ssim"):
            std, mean = torch.std_mean(vals)
            averages[key], averages[key + "_std"] = float(mean), float(std)
        else:
            averages[key] = float(vals.mean())
    return averages, per_image
