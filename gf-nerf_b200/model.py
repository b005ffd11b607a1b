"""`GFNeRFModel.get_outputs` through the operator API (reference gfnerf/nerfacto.py:522-619): sampler ->
field -> get_weights_f2nerf -> RGB / depth / accumulation renderers -> octree feedback, on the reference's dense
`[R,1024,...]` tensors.  This is the drop-in path for callers that keep nerfstudio's Trainer / autograd / optimizers;
`engine.GFNeRFEngine` is the same computation fused end to end on the compact layout (what bench.py times).
"""
from typing import Dict, Tuple

import torch
from torch import nn

from .field import FieldHeadNames, GFNeRFField
from .metrics import image_metrics
from .perssampler import PersSampler
from .rays import RayBundle
from .renderers import AccumulationRenderer, DepthRenderer, RGBRenderer


class GFNeRFModel(nn.Module):
    def __init__(self, persampler: PersSampler, field: GFNeRFField, scale_factor: float = 1.0,
                 background_color="last_sample"):
        super().__init__()
        self.persampler, self.field, self.scale_factor = persampler, field, float(scale_factor)
        self.field.persampler = persampler
        self.renderer_rgb = RGBRenderer(background_color=background_color)
        self.renderer_accumulation = AccumulationRenderer()
        self.renderer_depth = DepthRenderer(method="expected")     # gfnerf/nerfacto.py:288

    def get_outputs(self, ray_bundle: RayBundle) -> Dict[str, torch.Tensor]:
        ray_samples = self.persampler(ray_bundle)
        field_outputs = self.field(ray_samples)
        weights, alphas, trans = ray_samples.get_weights_f2nerf(field_outputs[FieldHeadNames.DENSITY])
        rgb = self.renderer_rgb(rgb=field_outputs[FieldHeadNames.RGB], weights=weights)
        depth = self.renderer_depth(weights=weights, ray_samples=ray_samples) / self.scale_factor
        accumulation = self.renderer_accumulation(weights=weights)
        oct_depth = ray_samples.f2samples.first_oct_dis[:, 0, :] / self.scale_factor
        outputs = {"rgb": rgb, "accumulation": accumulation, "depth": depth, "oct_depth": oct_depth}
        if self.training and ray_bundle.steps is not None:          # nerfacto.py:598-616
            cur_step = int(ray_bundle.steps.reshape(-1)[0].item())
            self.persampler.update_ray_march(cur_step)
            self.persampler.update_mode(0)
            if self.field.cur_stage == "init_stage":
                self.persampler.update_oct_nodes(sampled_anchors=ray_samples.f2samples.sampled_anchors,
                                                 pts_idx_bounds=ray_samples.f2samples.pts_idx_start_end,
                                                 sampled_weights=weights.detach(), sampled_alpha=alphas,
                                                 iter_step=cur_step)
            else:
                self.persampler.update_mode(1)
        return outputs

    forward = get_outputs

    def get_image_metrics_and_images(self, outputs: Dict[str, torch.Tensor],
                                     batch: Dict[str, torch.Tensor]) -> Tuple[Dict[str, float], Dict[str, torch.Tensor]]:
        """nerfstudio's `get_image_metrics_and_images` (nerfstudio/models/nerfacto.py) on `gf_image_metrics`:
        outputs["rgb"] and batch["image"] are one view [H, W, 3] (RGB; batch["image"] is moved to the rendered
        image's device).  Returns metrics_dict = {"psnr": float, "ssim": float} and images_dict = {"img": ground truth
        and rendering side by side, [H, 2W, 3]}.

        LPIPS is not computed: its network weights are not part of this package, so the "lpips" key is absent -- a
        caller that needs it keeps the reference's own method.  The accumulation and depth panels of nerfstudio's
        images_dict are not produced either."""
        rgb = outputs["rgb"]
        gt = batch["image"].to(rgb.device)
        m = image_metrics(rgb, gt)
        metrics_dict = {"psnr": float(m["psnr"].item()), "ssim": float(m["ssim"].item())}
        images_dict = {"img": torch.cat([gt, rgb], dim=1)}
        return metrics_dict, images_dict
