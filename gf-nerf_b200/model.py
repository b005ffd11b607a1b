"""`GFNeRFModel.get_outputs` through the operator API (reference gfnerf/nerfacto.py:522-619): sampler ->
field -> get_weights_f2nerf -> RGB / depth / accumulation renderers -> octree feedback, on the reference's dense
`[R,1024,...]` tensors.  This is the drop-in path for callers that keep nerfstudio's Trainer / autograd / optimizers;
`engine.GFNeRFEngine` is the same computation fused end to end on the compact layout (what bench.py times).
`get_outputs_for_camera_ray_bundle` renders whole views of the modules' parameters through that fused path.
"""
import os
from typing import Dict, Tuple

import torch
from torch import nn

from . import _lib
from .engine import FusedRenderer
from .field import FieldHeadNames, GFNeRFField
from .hash_3d_anchored import Hash3DAnchoredCore
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
        self._fused = None        # FusedRenderer of get_outputs_for_camera_ray_bundle, made at its first call

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

    # rays per get_outputs call in the reference's evaluation (eval_num_rays_per_chunk, gfnerf/config.py:109); the
    # appearance embedding of a view is chosen per chunk of this many rays
    EVAL_NUM_RAYS_PER_CHUNK = 2048

    @torch.no_grad()
    def get_outputs_for_camera_ray_bundle(self, camera_ray_bundle: RayBundle, chunk: int = 32768,
                                          route_blocks: bool = False) -> Dict[str, torch.Tensor]:
        """nerfstudio's `Model.get_outputs_for_camera_ray_bundle` (nerfstudio/models/base_model.py:166-190) on the fused
        kernels: `get_outputs` in eval mode over a whole view, `chunk` rays per fused render with no host sync in
        between.  origins / directions are [H, W, 3] (any leading shape works); returns {"rgb": [H,W,3],
        "accumulation", "depth", "oct_depth": [H,W,1]}.

        The parameters are the modules' as they are at the call: the global table, the MLP blob, the appearance
        embedding and, in the block stage, the residual table `base_encoding_{i}` of `field.active_block_idxs_test`.
        The fp16 table copies and the MLP blob are refreshed once per call; nothing is copied into an engine and no
        optimizer state is made.  Rays take the embedding row of `rel_camera_indices` if the bundle has them, else
        the one of the training camera nearest to the first origin of their 2048-ray chunk, as the reference's
        `PersSampler.generate_ray_samples` chooses it for each `get_outputs` call of its evaluation loop.  The octree
        is not updated and `self.training` is left as it is; the march noise follows the sampler's mode.

        route_blocks (block stage only): every 2048-ray chunk adds the residual table of ITS block instead of the one
        of `active_block_idxs_test` -- the block of the training camera nearest to the chunk's first origin, as the
        reference's `generate_ray_samples` / `update_active_blocks(cur_split_dataset_idx)` choose it: the camera's
        `cameras_labels` entry, else its index bucket.  The block follows the origins even when the bundle has
        `rel_camera_indices`.  A block table that is not resident is loaded from `base_dir` (`load_table`) and stays
        resident; one that is neither resident nor saved raises FileNotFoundError before anything is rendered.  The
        fused chunks keep their size whatever the routes: the table is chosen per ray on the device."""
        f, rb = self.field, camera_ray_bundle
        if route_blocks and f.cur_stage != "block_stage":
            raise ValueError("get_outputs_for_camera_ray_bundle: route_blocks needs the block stage "
                             f"(the field is in {f.cur_stage})")
        shape = tuple(rb.origins.shape[:-1])
        _lib.require_cuda(rb.origins, rb.directions)
        o = rb.origins.reshape(-1, 3).contiguous().float()
        d = rb.directions.reshape(-1, 3).contiguous().float()
        n = o.shape[0]
        r = self._fused
        if r is None or r.sampler is not self.persampler.sampler or r.hidden != f.hidden_dim:
            r = self._fused = FusedRenderer(self.persampler.sampler, f.hidden_dim)
        r.enc, r.res, r.res_tables = f.base_encoding_init.hash_3d, None, None
        ray_table, tables = None, []
        if route_blocks:
            ray_table, blocks = self._route_blocks(o)
            tables = [getattr(f, f"base_encoding_{b}").hash_3d for b in blocks]
        elif f.cur_stage == "block_stage":
            if len(f.active_block_idxs_test) != 1:
                raise RuntimeError(f"get_outputs_for_camera_ray_bundle: the block stage renders one block table, "
                                   f"active_block_idxs_test is {f.active_block_idxs_test}")
            r.res = getattr(f, f"base_encoding_{f.active_block_idxs_test[0]}").hash_3d
        for enc in [r.enc, r.res] + tables:
            if enc is not None:
                enc.shadow(force=True)
                enc._bias()          # the all-zero test of the bias pool (a host read) before the chunk loop
        if tables:
            r.res_tables = (tables, Hash3DAnchoredCore.table_refs(tables, r.device, recast=False))
        blob = torch.cat([f.base_network.flat_params(), f.mlp_head.flat_params()]).float()
        if r.mlp is None or r.mlp.numel() != blob.numel():
            # the MLP kernels load a 16-byte vector tail past the blob (as for GFNeRFEngine.mlp)
            r.mlp = torch.zeros((blob.numel() + 3) // 4 * 4, device=r.device)[:blob.numel()]
        r.mlp.copy_(blob)
        r.emb, cam = None, None
        if f.use_appearance_embedding:
            r.emb = f.embedding_appearance.embedding.weight.detach()
            if rb.rel_camera_indices is not None:
                cam = rb.rel_camera_indices.reshape(n, -1)[:, 0].to(device=r.device, dtype=torch.int64)
            else:
                cam = self._nearest_cameras(o)
        rgb, depth, acc, first = r.render_rays(o, d, cam, chunk=chunk, first_oct_dis=True, ray_table=ray_table)
        return {"rgb": rgb.view(*shape, 3), "accumulation": acc.view(*shape, 1),
                "depth": (depth / self.scale_factor).view(*shape, 1),
                "oct_depth": (first / self.scale_factor).view(*shape, 1)}

    def _nearest_cameras(self, origins: torch.Tensor) -> torch.Tensor:
        """int64 [N]: per ray, the training camera nearest to the first origin of its EVAL_NUM_RAYS_PER_CHUNK-ray chunk,
        with the distance and argmin of `PersSampler.get_nearest_split_dataset*`; on the device, no host read."""
        return self._per_ray(self._chunk_nearest(origins), origins.shape[0]).to(origins.device)

    def _chunk_nearest(self, origins: torch.Tensor) -> torch.Tensor:
        """int64 [chunks]: the training camera nearest to the first origin of each EVAL_NUM_RAYS_PER_CHUNK-ray chunk"""
        c2w = self.persampler.c2w
        firsts = origins[::self.EVAL_NUM_RAYS_PER_CHUNK].to(c2w.device)                # [chunks, 3]
        dists = torch.linalg.norm(c2w[None, :, 0:3, -1] - firsts[:, None, :], dim=2)   # [chunks, cameras]
        return torch.argmin(dists, dim=1)

    def _per_ray(self, per_chunk: torch.Tensor, n: int) -> torch.Tensor:
        k = self.EVAL_NUM_RAYS_PER_CHUNK
        return per_chunk.view(-1, 1).expand(-1, k).reshape(-1)[:n]

    def _route_blocks(self, origins: torch.Tensor):
        """(ray_table int32 [N], blocks): every ray's entry in `blocks`, the sorted block indices the view needs.  The
        block of a chunk is `get_nearest_split_dataset*`'s: cameras_labels[nearest], or without labels
        min(nearest // max(n_cams // n_split_dataset, 1), n_split_dataset - 1).  One host read (the block set); every
        block's table is made resident here, or FileNotFoundError is raised before anything is launched."""
        ps, f = self.persampler, self.field
        nearest = self._chunk_nearest(origins)
        if ps.cameras_labels is not None:
            block = ps.cameras_labels.reshape(-1).to(nearest.device)[nearest].to(torch.int64)
        else:
            per = max(ps.c2w.shape[0] // ps.n_split_dataset, 1)
            block = torch.clamp(nearest // per, max=ps.n_split_dataset - 1)
        uniq = torch.unique(block)                                     # sorted
        blocks = [int(b) for b in uniq.tolist()]                       # the call's one host read of the routes
        missing = [b for b in blocks if not hasattr(f, f"base_encoding_{b}")]
        for b in missing:
            path = str(f.encodings_ckpt_dir / f"base_encoding_{b}.ckpt")
            if not os.path.exists(path):
                raise FileNotFoundError(f"block {b} has neither a resident table nor a saved one: {path}")
        for b in missing:             # swapped out: brought back like update_active_blocks' eval branch does
            f.load_table(b, strict=True)
            getattr(f, f"base_encoding_{b}").set_require_grad(False)
        slot = torch.searchsorted(uniq, block).to(torch.int32)
        ray_table = self._per_ray(slot, origins.shape[0]).to(origins.device).contiguous()
        return ray_table, blocks

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
