"""Image-quality metrics of rendered views on the device: PSNR, SSIM and MSE per image in one kernel sequence
(`gf_image_metrics`, csrc/metrics.cu).  The conventions are those of nerfstudio's nerfacto evaluation -- torchmetrics'
`PeakSignalNoiseRatio(data_range=1.0)` and functional `structural_similarity_index_measure` with its defaults, one
call per image; see include/gfnerf_b200.h."""
from typing import Dict

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
