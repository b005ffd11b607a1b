"""Fused per-ray hot path: one training / render step over a ray batch, compact (CSR) layout.

This is what `GFNeRFModel.get_outputs` + loss + backward + optimizer step amount to for the path of
SURVEY.md section 8 (reference gfnerf/nerfacto.py:522-619, gfnerf/gf_pipeline.py:146-186,
nerfstudio/engine/trainer.py:382-443), with every stage a kernel of the C-ABI library and no host
synchronisation inside the step:

  sample (traverse + march) -> scan -> compact -> hash encode -> ray bias -> MLP -> composite
  -> Charbonnier -> composite bwd -> MLP bwd -> ray-bias bwd -> hash scatter
  -> [NCCL all-reduce of table / MLP / embedding gradients] -> Adam (table + fp16 shadow, MLP, embedding)
  -> octree vote.

The reference evaluates all R*1024 padded slots; here only the V valid samples exist.  Results per
valid sample are identical (padding contributes weight 0 in the reference because its delta is 0).
"""
import contextlib
import os
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib
from .ddp import FlatBucket, GradSync, table_reduce_ranges
from .hash_3d_anchored import Hash3DAnchoredCore
from .perssampler import CompactSamples, PersSamplerCore

HIDDEN = 64
GRAD_SCALE = 128.0   # GF_GRAD_SCALE, field/Hash3DAnchored_cuda.cu:209
APPEARANCE_DIM = 32


def mlp_param_count(hidden: int = HIDDEN) -> int:
    return int(_lib.lib().gf_mlp_param_count(hidden))


def init_mlp_params(hidden: int = HIDDEN, generator: torch.Generator = None, device="cpu") -> torch.Tensor:
    """torch nn.Linear default init (kaiming_uniform(a=sqrt(5)) = U(-1/sqrt(in), 1/sqrt(in)) for weight and
    bias), in the blob order of include/gfnerf_b200.h -- what MLPNetwork (gfnerf/mlp.py:35-43) constructs."""
    parts = []
    for out_f, in_f in ((hidden, 32), (16, hidden), (hidden, 63), (hidden, hidden), (3, hidden)):
        bound = 1.0 / np.sqrt(in_f)
        parts.append((torch.rand(out_f * in_f, generator=generator) * 2 - 1) * bound)
        parts.append((torch.rand(out_f, generator=generator) * 2 - 1) * bound)
    return torch.cat(parts).float().to(device).contiguous()


class _Adam:
    """State of gf_adam_step for one flat fp32 tensor."""

    def __init__(self, param: torch.Tensor, lr: float, eps: float = 1e-15, betas=(0.9, 0.999), grad=None,
                 grad_scale: float = 1.0, n_active: Optional[int] = None):
        self.param, self.lr, self.eps, self.betas = param, lr, eps, betas
        # n_active: the leading elements the step sweeps.  For a hash table that is the 8.5 * T rows its levels can
        # reach (level_base_row): the rows beyond never receive a gradient, so their moments stay 0 and dense Adam
        # leaves them where they are (update = lr * 0 / (sqrt(0) + eps)) -- skipping them is exact, not an approximation
        self.n_active = int(param.numel() if n_active is None else n_active)
        # `grad` holds grad_scale x the gradient (a power of two: the hash tables stay at the reference's x128 scale,
        # Hash3DAnchored_cuda.cu:209, and the division rides along with the optimizer's 1 / world)
        self.grad_scale = float(grad_scale)
        self.grad = torch.zeros_like(param) if grad is None else grad
        # (moments with room for a vector tail: the peer exchange kernel works in 16-byte units)
        n4 = (param.numel() + 3) // 4 * 4
        self.m = torch.zeros(n4, dtype=param.dtype, device=param.device)[:param.numel()].view_as(param)
        self.v = torch.zeros(n4, dtype=param.dtype, device=param.device)[:param.numel()].view_as(param)
        # the step count lives on the device: a step skipped by the NaN guard must not advance the bias correction
        # (the reference skips optimizer.step() altogether, trainer.py:416-426)
        self.d_step = torch.zeros(1, dtype=torch.int64, device=param.device)

    @property
    def t(self) -> int:
        """steps applied so far (host sync; for tests / checkpoints)"""
        return int(self.d_step.item())

    def unscaled_grad(self) -> torch.Tensor:
        """The gradient in units of dL/dparam (a copy when grad_scale != 1; exact, the scale is a power of two)."""
        return self.grad if self.grad_scale == 1.0 else self.grad / self.grad_scale

    def step(self, shadow=None, grad_div=1.0, lr=None, skip_flag=None):
        """skip_flag: device int32 set by gf_grad_nan_scan -- non-zero leaves the parameters untouched (the trainer's
        NaN guard, trainer.py:416-426) and does not count as a step"""
        _lib.check(_lib.lib().gf_adam_step_counted(
            self.n_active, _lib.ptr(self.param), _lib.ptr(self.grad), _lib.ptr(self.m), _lib.ptr(self.v),
            _lib.ptr(shadow), float(self.lr if lr is None else lr), self.betas[0], self.betas[1], self.eps,
            _lib.ptr(self.d_step), float(grad_div) * self.grad_scale, 1, _lib.ptr(skip_flag), _lib.cur_stream()),
            "gf_adam_step_counted")


@dataclass
class StepOutputs:
    rgb: torch.Tensor            # [R,3]
    depth: torch.Tensor          # [R]
    accumulation: torch.Tensor   # [R]
    loss: Optional[torch.Tensor]  # [1] or None
    n_samples: torch.Tensor      # int32 [1] (device)
    block_losses: Optional[torch.Tensor] = None   # [K]: each block's loss (several focal blocks); loss is their sum


class FusedRenderer:
    """The forward-only render body on the fused kernels -- compact sampling with the next chunk sampled ahead, hash
    encode (+ the focal stage's residual table), ray bias, MLP, composite, the eval clamp -- over one parameter
    source: `sampler`, `enc` (Hash3DAnchoredCore), `res` (residual Hash3DAnchoredCore or None), `mlp` (the flat MLP
    blob, with room for a 16-byte vector tail past its end) and `emb` (appearance embedding [n_images, 32] or None).
    `res_tables` = (cores, refs) instead of `res`: several residual tables, each ray taking the one its `ray_table`
    entry names (`Hash3DAnchoredCore.launch_forward_residual_routed`; refs from `Hash3DAnchoredCore.table_refs`).
    `GFNeRFEngine` renders its own parameters through it; `GFNeRFModel.get_outputs_for_camera_ray_bundle` points a
    renderer of its own at the modules' parameters (model.py)."""

    def __init__(self, sampler: PersSamplerCore, hidden: int = HIDDEN):
        self.sampler = sampler
        self.device = sampler.device
        self.hidden = hidden
        self.mask_words = int(_lib.lib().gf_mlp_mask_words(hidden))
        if self.mask_words < 0:
            raise ValueError(f"gfnerf_b200: hidden width {hidden} is not built (64 and 128 are)")
        self.enc = self.res = self.mlp = self.emb = self.res_tables = None
        self._ws = {}

    # GF_NVTX=1: every stage of the step is an NVTX range ("gf/<stage>", SURVEY 8d) -- what `ncu --nvtx --nvtx-include
    # "gf/hash_fwd/"` / an nsys timeline filter on.  Off by default: two extra host calls per stage.
    NVTX = os.environ.get("GF_NVTX", "0") == "1"

    @contextlib.contextmanager
    def _stage(self, name):
        ev = getattr(self, "_events", None)
        if ev is None and not self.NVTX:
            yield
            return
        if self.NVTX:
            torch.cuda.nvtx.range_push("gf/" + name)
        if ev is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        try:
            yield
        finally:
            if ev is not None:
                e1.record()
                ev.append((name, e0, e1))
            if self.NVTX:
                torch.cuda.nvtx.range_pop()


    def _buf(self, name, shape, dtype, zero=False):
        n = int(np.prod(shape))
        t = self._ws.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._ws[name] = t
        t = t[:n].view(*shape)
        if zero:
            t.zero_()
        return t

    # ---- forward pieces --------------------------------------------------------------------
    def _field_forward(self, cs: CompactSamples, ray_emb, train: bool = False, ray_table=None):
        """train: also keep the forward's ReLU masks (`relu_masks` workspace) for gf_mlp_backward.  ray_table: int32
        [n_rays], each ray's index into `res_tables` (used only when `res_tables` is set)"""
        L, st = _lib.lib(), _lib.cur_stream()
        cap, R = cs.pts01.shape[0], cs.n_rays
        feat = self._buf("feat", (cap, 32), torch.float16)
        sigma = self._buf("sigma", (cap,), torch.float32)
        rgb = self._buf("rgb", (cap, 3), torch.float32)
        ray_bias = self._buf("ray_bias", (R, self.hidden), torch.float32)
        masks = self._buf("relu_masks", (cap, self.mask_words), torch.int32) if train else None
        with self._stage("hash_fwd"):
            self.enc.launch_forward(cs.pts01, cs.anchor, out_f16=feat, d_n_ptr=cs.total, recast=False)
            if self.res_tables is not None:
                if ray_table is None:
                    raise ValueError("gfnerf_b200: several residual tables are set, but no per-ray ray_table")
                cores, refs = self.res_tables
                Hash3DAnchoredCore.launch_forward_residual_routed(cores, cs.pts01, cs.anchor, feat, cs.ray_id, ray_table,
                                                                  d_n_ptr=cs.total, refs=refs)
            elif self.res is not None:
                self.res.launch_forward_residual(cs.pts01, cs.anchor, feat, d_n_ptr=cs.total, recast=False)
        with self._stage("ray_bias"):
            _lib.check(L.gf_mlp_ray_bias(R, self.hidden, _lib.ptr(self.mlp), _lib.ptr(cs.rays_d),
                                         _lib.ptr(ray_emb), _lib.ptr(ray_bias), st), "gf_mlp_ray_bias")
        with self._stage("mlp_fwd"):
            _lib.check(L.gf_mlp_forward(cap, _lib.ptr(cs.total), self.hidden, _lib.ptr(self.mlp), _lib.ptr(feat),
                                        _lib.ptr(cs.ray_id), _lib.ptr(ray_bias), _lib.ptr(sigma), _lib.ptr(rgb),
                                        _lib.ptr(masks), st), "gf_mlp_forward")
        return feat, sigma, rgb, ray_bias

    def _composite(self, cs: CompactSamples, sigma, rgb, keep: bool):
        L, st = _lib.lib(), _lib.cur_stream()
        cap, R = cs.pts01.shape[0], cs.n_rays
        weights = self._buf("weights", (cap,), torch.float32) if keep else None
        alphas = self._buf("alphas", (cap,), torch.float32) if keep else None
        trans = self._buf("trans", (cap,), torch.float32) if keep else None
        out_rgb = torch.empty((R, 3), dtype=torch.float32, device=self.device)
        depth = torch.empty(R, dtype=torch.float32, device=self.device)
        acc = torch.empty(R, dtype=torch.float32, device=self.device)
        tmax = torch.zeros(1, dtype=torch.float32, device=self.device)
        with self._stage("composite_fwd"):
            _lib.check(L.gf_composite_forward(R, _lib.ptr(cs.offsets), _lib.ptr(sigma), _lib.ptr(cs.delta),
                                              _lib.ptr(rgb), _lib.ptr(cs.t), _lib.ptr(weights), _lib.ptr(alphas),
                                              _lib.ptr(trans), _lib.ptr(out_rgb), _lib.ptr(depth), _lib.ptr(acc),
                                              _lib.ptr(tmax), st), "gf_composite_forward")
        # DepthRenderer clips to the global [t.min(), t.max()] of the DENSE tensor, whose min is the padding's 0
        # (nerfstudio/model_components/renderers.py:281)
        depth = torch.minimum(torch.clamp_min(depth, 0.0), tmax)
        return out_rgb, depth, acc, weights, alphas, trans

    def _ray_emb(self, rel_camera_indices):
        if self.emb is None or rel_camera_indices is None:
            return None
        return self.emb.index_select(0, rel_camera_indices.to(torch.int64)).contiguous()

    # ---- public API ------------------------------------------------------------------------
    @torch.no_grad()
    def render(self, rays_o, rays_d, rel_camera_indices=None, noise=None, next_rays=None) -> StepOutputs:
        """Forward-only (eval) pass: GFNeRFModel.get_outputs without the training feedback.  next_rays: the rays of
        the next call, sampled on the side stream underneath this call's encode / MLP / composite (`_presample`;
        nothing changes the octree in between)."""
        return self._render(rays_o, rays_d, rel_camera_indices, noise, next_rays)[0]

    def _render(self, rays_o, rays_d, rel_camera_indices=None, noise=None, next_rays=None, ray_table=None):
        """`render`, also returning the chunk's CompactSamples (valid until the sampler reuses its slot)"""
        with torch.cuda.device(self.device):
            cs = self._take_presampled(rays_o, rays_d) if noise is None else None
            if cs is None:
                cs = self.sampler.sample_compact(rays_o, rays_d, noise=noise, slot=getattr(self, "_cs_slot", 0))
            self.flush()
            if next_rays is not None:
                self._presample(next_rays[0], next_rays[1])
            _, sigma, rgb, _ = self._field_forward(cs, self._ray_emb(rel_camera_indices), ray_table=ray_table)
            out_rgb, depth, acc, _, _, _ = self._composite(cs, sigma, rgb, keep=False)
            # RGBRenderer in eval mode: nan_to_num + clamp (renderers.py:131-137)
            out_rgb = torch.nan_to_num(out_rgb).clamp_(0.0, 1.0)
        return StepOutputs(out_rgb, depth, acc, None, cs.total), cs

    @torch.no_grad()
    def render_rays(self, rays_o, rays_d, ray_cam=None, chunk: int = 32768, sample_ahead: bool = True,
                    first_oct_dis: bool = False, ray_table=None):
        """Render of N rays in chunks of `chunk` with no host sync inside, the next chunk sampled underneath the
        current one.  ray_cam: int64 [N], the row of `emb` each ray takes (None: no appearance embedding).  ray_table:
        int32 [N], the entry of `res_tables` each ray takes (with `res_tables` only).  Returns rgb [N,3], depth [N],
        acc [N] and, with `first_oct_dis`, the sampler's first_oct_dis [N] (else None)."""
        N = rays_o.shape[0]
        rgb = torch.empty((N, 3), dtype=torch.float32, device=self.device)
        depth = torch.empty(N, dtype=torch.float32, device=self.device)
        acc = torch.empty(N, dtype=torch.float32, device=self.device)
        first = torch.empty(N, dtype=torch.float32, device=self.device) if first_oct_dis else None
        for a in range(0, N, chunk):
            b = min(a + chunk, N)
            nxt = (rays_o[b:b + chunk], rays_d[b:b + chunk]) if (b < N and sample_ahead) else None
            out, cs = self._render(rays_o[a:b], rays_d[a:b], None if ray_cam is None else ray_cam[a:b], next_rays=nxt,
                                   ray_table=None if ray_table is None else ray_table[a:b])
            rgb[a:b], depth[a:b], acc[a:b] = out.rgb, out.depth, out.accumulation
            if first is not None:
                # copied before the chunk after next is sampled into the same slot (that sampling waits on this stream)
                first[a:b] = cs.first_oct_dis
        return rgb, depth, acc, first

    # ---- sampling one batch ahead ----------------------------------------------------------------------------
    def _presample(self, rays_o, rays_d, vote=None, after=None):
        """Launches the ray sampling of the NEXT batch on a side stream, ordered after everything issued so far on the
        current stream (in particular this step's octree vote, the only thing the sampler depends on).  The sampler
        is a latency-bound kernel that leaves most issue slots of an SM idle; the backward kernels of the current
        batch run underneath it.  Results are identical to sampling at the start of the next step."""
        if not hasattr(self, "_pre_stream"):
            # GF_PRESAMPLE_PRIO=-1: the side stream's CTAs are scheduled ahead of the main stream's (A/B knob)
            self._pre_stream = torch.cuda.Stream(device=self.device, priority=int(os.environ.get("GF_PRESAMPLE_PRIO", "0")))
            self._pre = None
            self._cs_slot = 0
        cur = torch.cuda.current_stream(self.device)
        slot = self._cs_slot ^ 1
        # `after`: an event recorded where the side stream's inputs were complete (the forward).  Waiting on the
        # whole current stream instead would also wait for whatever was launched since -- the MLP backward this work
        # is meant to run underneath.
        if after is not None:
            self._pre_stream.wait_event(after)
        else:
            self._pre_stream.wait_stream(cur)
        hook, self.sampler.stage_hook = getattr(self.sampler, "stage_hook", None), None   # events are per stream
        with torch.cuda.stream(self._pre_stream):
            if vote is not None:
                # the octree feedback of the current batch (and, data parallel, its MAX all-reduce with the rank
                # skew it absorbs) only gates the NEXT sampling: off the stream that runs the backward pass
                vcs, weights, alphas, step = vote
                self.sampler.update_oct_nodes_compact(vcs, weights, alphas, step)
                self.sampler.UpdateRayMarch(step)
            cs = self.sampler.sample_compact(rays_o, rays_d, slot=slot)
            done = self._pre_stream.record_event()
        self.sampler.stage_hook = hook
        self._pre = (rays_o.data_ptr(), rays_d.data_ptr(), tuple(rays_o.shape), cs, done, slot)

    def _take_presampled(self, rays_o, rays_d):
        pre, self._pre = getattr(self, "_pre", None), None
        if pre is None:
            return None
        torch.cuda.current_stream(self.device).wait_event(pre[4])    # also orders the workspace reuse
        if pre[:3] != (rays_o.data_ptr(), rays_d.data_ptr(), tuple(rays_o.shape)):
            return None                                              # another batch came: sample it now
        self._cs_slot = pre[5]
        return pre[3]

    def flush(self):
        """Orders the current stream after a sampling issued ahead on the side stream."""
        pre = getattr(self, "_pre", None)
        if pre is not None:
            torch.cuda.current_stream(self.device).wait_event(pre[4])


class GFNeRFEngine(FusedRenderer):
    """Global-stage model state (hash table, MLPs, appearance embedding) + the fused step."""

    # Levels per scatter launch / all-reduce message when world > 1.  16 = one scatter, one all-reduce after it (of the
    # 8.5 * local_size rows the reference's level addressing can reach, 36 MB at log2T = 19; see level_base_row).
    # Smaller groups start reducing while the rest is still being scattered, but on 8 B200s NCCL's CTAs next to the
    # issue-bound scatter cost more than the hidden transfer saves: 5.70 ms/step with groups of 4, 5.57 with 8,
    # 5.46 with 16 (GF_LEVEL_GROUP to experiment).
    LEVEL_GROUP = int(os.environ.get("GF_LEVEL_GROUP", "16"))

    def __init__(self, sampler: PersSamplerCore, log2_table_size: int = 19, num_images: int = 1, hidden: int = HIDDEN,
                 use_appearance_embedding: bool = True, lr_table: float = 1e-2, lr_mlp: float = 1e-2,
                 seed: int = 0, dist_group=None, nan_guard: bool = True, s3im_loss_mult: float = 0.0,
                 s3im_kernel_size: int = 4, s3im_stride: int = 4, s3im_repeat_time: int = 10,
                 s3im_patch_height: int = 32):
        super().__init__(sampler, hidden)
        self.nan_guard = bool(nan_guard)    # skip the optimizer step on a NaN gradient (trainer.py:416-426)
        # S3IM on top of the Charbonnier loss (gfnerf/nerfacto.py:186-197, 686-688); 0 = off
        self.s3im = (float(s3im_loss_mult), int(s3im_kernel_size), int(s3im_stride), int(s3im_repeat_time),
                     int(s3im_patch_height))
        self.last_nan_flag = None
        gen = torch.Generator().manual_seed(seed)
        # n_volumes: the reference sizes the prime pool by the number of tree nodes (gfnerf/nerfacto.py:267)
        # while indexing it with trans_idx (< number of transforms); any bound >= n_trans is equivalent.
        self.n_volumes = max(int(sampler.n_volumes_), 1)
        self.enc = Hash3DAnchoredCore(log2_table_size, self.n_volumes, device=self.device, generator=gen)
        self.enc.feat_pool_.requires_grad_(False)
        self.enc.Reset(generator=gen)   # U(-0.01, 0.01), gfnerf/nerfacto_field.py:200; reproducible from `seed`
        mlp0 = init_mlp_params(hidden, gen, self.device)
        self.mlp = torch.zeros((mlp0.numel() + 3) // 4 * 4, device=self.device)[:mlp0.numel()]   # room for a vector tail
        self.mlp.copy_(mlp0)
        self.emb = (torch.randn(num_images, APPEARANCE_DIM, generator=gen).to(self.device)
                    if use_appearance_embedding else None)
        self.opt_table = _Adam(self.enc.feat_pool_.detach().view(-1), lr_table, grad_scale=GRAD_SCALE,
                               n_active=self.enc.used_rows_ * 2)
        # MLP + embedding gradients live in one flat bucket: one collective for both
        small = FlatBucket([self.mlp.shape] + ([self.emb.shape] if self.emb is not None else []), device=self.device)
        self.opt_mlp = _Adam(self.mlp, lr_mlp, grad=small.views[0])
        self.opt_emb = _Adam(self.emb.view(-1), lr_mlp, grad=small.views[1].view(-1)) if self.emb is not None else None
        self._small = small
        self._small_grads = small.flat
        self.sync = GradSync(dist_group, self.device)
        self.world = self.sync.world
        self.peer = None
        if self.world > 1 and self.device.type == "cuda" and os.environ.get("GF_PEER_EXCHANGE", "1") != "0":
            self._setup_peer_exchange(dist_group)
        if self.world > 1:
            # identical initial parameters on every replica, whatever seed each rank was built with (what DDP's
            # constructor does; ranks seeded seed + rank -- ddp.rank_seed -- would otherwise average gradients of
            # different tables forever)
            self.sync.broadcast_([self.enc.feat_pool_.data, self.enc.prim_pool_, self.enc.bias_pool_, self.mlp]
                                 + ([self.emb] if self.emb is not None else []))
            sampler.vote_reduce = self._peer_vote_max if self.peer is not None else self.sync.max_
        self.enc.shadow(force=True)
        self.step_count = 0
        self._deferred = None   # lr_scale of an optimizer step whose gradient reduce is still in flight
        self.stage = "init_stage"
        self.opt_res = None     # focal stage: Adam of this GPU's residual sub-encoder `res`
        # focal stage with several blocks (start_block_stage(blocks=...)): their ids, residual cores and Adams
        self.blocks = self.res_blocks = self.opt_res_blocks = None

    # ---- focal (block) stage: reference gfnerf/nerfacto_field.py:458-489, gfnerf/nerfacto.py:432-488 ------------
    def start_block_stage(self, log2_table_size: int = None, lr: float = 5e-3, seed: int = 1, blocks=None):
        """Freezes the global table, both MLPs and the appearance embedding and adds a zero-initialised residual
        sub-encoder whose features are summed with the global encoder's before the (frozen) MLP.  The residual tables
        are private to this rank, so the focal stage has NO gradient exchange at all.

        blocks = [b0, ..., bK-1]: this rank trains K blocks at once, table k seeded `seed + k` (the table a single-block
        engine started with `seed + k` has).  A training batch is then K equal contiguous segments of rays, segment k
        belonging to blocks[k]; each block's step is what a single-block engine computes on its segment.  Renders
        take a per-ray `ray_table` (index into `blocks`).  Without `blocks`: one residual table `res`."""
        if blocks is not None:
            blocks = [int(b) for b in blocks]
            if not blocks or len(set(blocks)) != len(blocks) or min(blocks) < 0:
                raise ValueError(f"gfnerf_b200: block ids must be distinct and >= 0, got {blocks}")
        self.flush()
        log2_table_size = int(np.log2(self.enc.local_size_)) if log2_table_size is None else int(log2_table_size)

        def block_table(seed_):
            res = Hash3DAnchoredCore(log2_table_size, self.n_volumes, device=self.device,
                                     generator=torch.Generator().manual_seed(seed_))
            res.feat_pool_.requires_grad_(False)
            res.Zero()
            res.shadow(force=True)
            opt = _Adam(res.feat_pool_.detach().view(-1), lr, grad_scale=GRAD_SCALE,   # sub-encoder lr, gfnerf/nerfacto.py:483
                        n_active=res.used_rows_ * 2)
            return res, opt

        self.res = self.opt_res = self.res_tables = None
        self.blocks = self.res_blocks = self.opt_res_blocks = None
        if blocks is None:
            self.res, self.opt_res = block_table(seed)
        else:
            made = [block_table(seed + k) for k in range(len(blocks))]
            self.blocks = blocks
            self.res_blocks = [m[0] for m in made]
            self.opt_res_blocks = [m[1] for m in made]
            self._block_refs()
        self.stage = "block_stage"
        self.sampler.UpdateMode(1)                                        # nerfacto.py:614-616

    def _block_refs(self):
        """Descriptor arrays of the block tables for the routed gather and scatter (again after a pool was replaced)"""
        self.res_tables = (self.res_blocks, Hash3DAnchoredCore.table_refs(self.res_blocks, self.device, recast=False))
        self._grad_refs = Hash3DAnchoredCore.grad_refs(self.res_blocks, [o.grad for o in self.opt_res_blocks],
                                                       self.device)
        self._block_ray_tables = {}

    def block_ray_table(self, n_rays: int) -> torch.Tensor:
        """int32 [n_rays]: the training batch's route, K contiguous segments of n_rays / K rays, segment k to table k"""
        K = len(self.blocks)
        if n_rays % K:
            raise ValueError(f"gfnerf_b200: a batch of {n_rays} rays does not split into {K} equal block segments")
        rt = self._block_ray_tables.get(n_rays)
        if rt is None:
            rt = torch.arange(K, dtype=torch.int32, device=self.device).repeat_interleave(n_rays // K)
            self._block_ray_tables[n_rays] = rt
        return rt

    def end_block_stage(self):
        self.res = self.opt_res = self.res_tables = None
        self.blocks = self.res_blocks = self.opt_res_blocks = None
        self.stage = "init_stage"
        self.sampler.UpdateMode(0)

    # ---- parameters in / out of the operator-API modules ------------------------------------------------------------
    # GFNeRFField / GFNeRFModel carry the reference's state-dict keys (field.py), so this is also the way a checkpoint
    # of the reference gets into the fused engine and back: load_state_dict on the modules, then `from_model`.
    @classmethod
    def from_model(cls, model, **kw) -> "GFNeRFEngine":
        """Fused engine over the sampler and the parameters of a `GFNeRFModel` (model.py): same octree object (the
        model's `persampler.sampler`), table size, width and embedding as its field; parameters copied (`load_model`)."""
        f = model.field
        eng = cls(model.persampler.sampler, log2_table_size=f.log2_table_size, num_images=f.num_images,
                  hidden=f.hidden_dim, use_appearance_embedding=f.use_appearance_embedding, **kw)
        eng.load_model(model)
        return eng

    def load_model(self, model, reset_optimizer: bool = True):
        """Adopt the global table (+ primes / bias pool), both MLPs and the appearance embedding of a GFNeRFField (or of
        a GFNeRFModel's field).  The Adam moments restart unless `reset_optimizer` is False (a checkpoint of the
        reference keeps its optimizer state with the trainer, not with the model)."""
        f = getattr(model, "field", model)
        if int(f.hidden_dim) != self.hidden:
            raise ValueError(f"gfnerf_b200: the field is {f.hidden_dim} wide, the engine {self.hidden}")
        src = f.base_encoding_init.hash_3d
        if tuple(src.feat_pool_.shape) != tuple(self.enc.feat_pool_.shape):
            raise ValueError(f"gfnerf_b200: table of {tuple(src.feat_pool_.shape)} rows x channels into an engine built "
                             f"for {tuple(self.enc.feat_pool_.shape)}")
        if (self.emb is None) != (not f.use_appearance_embedding):
            raise ValueError("gfnerf_b200: field and engine disagree on use_appearance_embedding")
        self.flush()
        self.enc.LoadStates([t.detach() for t in src.States()], 0)
        self.n_volumes = self.enc.n_volumes_
        blob = torch.cat([f.base_network.flat_params(), f.mlp_head.flat_params()]).detach().float()
        if blob.numel() != self.mlp.numel():
            raise ValueError(f"gfnerf_b200: {blob.numel()} MLP parameters, the fused kernel takes {self.mlp.numel()}")
        self.mlp.copy_(blob)
        if self.emb is not None:
            w = f.embedding_appearance.embedding.weight.detach()
            if tuple(w.shape) != tuple(self.emb.shape):
                raise ValueError(f"gfnerf_b200: embedding {tuple(w.shape)} into an engine built for {tuple(self.emb.shape)}")
            self.emb.copy_(w)
        if reset_optimizer:
            for opt in (self.opt_table, self.opt_mlp, self.opt_emb):
                if opt is not None:
                    opt.m.zero_(), opt.v.zero_(), opt.d_step.zero_()
        self.enc.shadow(force=True)

    def store_model(self, model, block: Optional[int] = None):
        """The inverse of `load_model`: the engine's current parameters into the field's modules (whose `state_dict()`
        is the reference's checkpoint layout).  block = b (block stage only): the residual table `res` also goes into
        the field's `base_encoding_{b}`, which is created if the field has none -- how the blocks of a focal run
        are gathered into one model (each rank stores its blocks, then `field.save_table(b)`).  With several blocks
        (start_block_stage(blocks=...)) b must be one of them, and its table is the one stored."""
        f = getattr(model, "field", model)
        if int(f.hidden_dim) != self.hidden:
            raise ValueError(f"gfnerf_b200: the field is {f.hidden_dim} wide, the engine {self.hidden}")
        res = None
        if block is not None:
            if self.stage != "block_stage" or (self.res is None and self.blocks is None):
                raise ValueError(f"gfnerf_b200: store_model(block={block}) needs the block stage; the engine is in "
                                 f"{self.stage}")
            if self.blocks is not None:
                if int(block) not in self.blocks:
                    raise ValueError(f"gfnerf_b200: block {block} is not one of this engine's blocks {self.blocks}")
                res = self.res_blocks[self.blocks.index(int(block))]
            else:
                res = self.res
            if int(f.log2_table_size) != int(np.log2(res.local_size_)):
                raise ValueError(f"gfnerf_b200: the field's block tables are 2^{f.log2_table_size} rows per level, "
                                 f"the engine's residual table 2^{int(np.log2(res.local_size_))}")
        self.flush()
        self.sync_master_params()       # peer exchange: every rank only keeps ITS fp32 rows current
        f.base_encoding_init.load_states([t.detach() for t in self.enc.States()], 0)
        o = 0
        with torch.no_grad():
            for lin in f.base_network.linears() + f.mlp_head.linears():
                for p in (lin.weight, lin.bias):
                    p.copy_(self.mlp[o:o + p.numel()].view_as(p))
                    o += p.numel()
            if self.emb is not None:
                f.embedding_appearance.embedding.weight.copy_(self.emb)
        assert o == self.mlp.numel()
        if block is not None:
            name = f"base_encoding_{int(block)}"
            if not hasattr(f, name):
                f.add_table(int(block))
            getattr(f, name).load_states([t.detach() for t in res.States()], 0)

    # ---- resume ---------------------------------------------------------------------------------------------------------
    def checkpoint(self) -> dict:
        """Everything a resumed run of the fused engine needs, as host tensors / scalars (`torch.save`-able): parameters,
        Adam moments and step counts, the octree blobs with their vote statistics, the march schedule.  (The reference
        keeps model, optimizer and scheduler state in the trainer's checkpoint, nerfstudio/engine/trainer.py:455-489, and
        drops the vote statistics: `PersSampler::LoadStates` restarts them at 1000, PersSampler.cpp:1010-1013.)  Data
        parallel: call on every rank (the owners' table rows are collected first); the result is the same everywhere."""
        self.flush()
        self.sync_master_params()
        cpu = lambda t: None if t is None else t.detach().to("cpu", copy=True)

        def adam(opt):
            # (the moments beyond n_active belong to table rows no level can reach: they stay zero, `_Adam`)
            return None if opt is None else {"m": cpu(opt.m.view(-1)[:opt.n_active]), "v": cpu(opt.v.view(-1)[:opt.n_active]),
                                             "t": opt.t, "n_active": opt.n_active}

        s = self.sampler
        s.flush_stats()
        out = {"version": 1, "hidden": self.hidden, "step_count": self.step_count, "stage": self.stage,
               "table": [cpu(t) for t in self.enc.States()], "mlp": cpu(self.mlp), "emb": cpu(self.emb),
               "adam": {"table": adam(self.opt_table), "mlp": adam(self.opt_mlp), "emb": adam(self.opt_emb)},
               "sampler": {"states": [cpu(t) for t in s.States()], "weight_stats": cpu(s.tree_weight_stats_),
                           "alpha_stats": cpu(s.tree_alpha_stats_), "ray_march_fineness": s.ray_march_fineness_,
                           "sampled_oct_per_ray": s.sampled_oct_per_ray_, "mode": s.mode_}}
        if self.res is not None:
            out["res_table"] = [cpu(t) for t in self.res.States()]
            out["adam"]["res"] = adam(self.opt_res)
            out["res_lr"] = self.opt_res.lr
        if self.blocks is not None:
            out["res_blocks"] = list(self.blocks)
            out["res_block_tables"] = [[cpu(t) for t in c.States()] for c in self.res_blocks]
            out["adam"]["res_blocks"] = [adam(o) for o in self.opt_res_blocks]
            out["res_lr"] = self.opt_res_blocks[0].lr
        return out

    def restore(self, ckpt: dict) -> None:
        """Inverse of `checkpoint()` on an engine built with the same table size, width and embedding shape."""
        if ckpt.get("version") != 1 or int(ckpt["hidden"]) != self.hidden:
            raise ValueError("gfnerf_b200: not a checkpoint of this engine (version / hidden width)")
        if tuple(ckpt["table"][0].shape) != tuple(self.enc.feat_pool_.shape) or tuple(ckpt["mlp"].shape) != tuple(self.mlp.shape):
            raise ValueError("gfnerf_b200: the checkpoint's table / MLP shapes are not this engine's")
        if (ckpt["emb"] is None) != (self.emb is None) or (self.emb is not None and ckpt["emb"].shape != self.emb.shape):
            raise ValueError("gfnerf_b200: the checkpoint's appearance embedding is not this engine's")
        self.flush()
        self._pre = None                       # samples taken ahead belong to the octree that is being replaced

        def adam(opt, st):
            n = int(st["n_active"])
            if n != opt.n_active:
                raise ValueError("gfnerf_b200: optimizer state of another table size")
            opt.m.view(-1)[:n].copy_(st["m"].view(-1))
            opt.v.view(-1)[:n].copy_(st["v"].view(-1))
            opt.d_step.fill_(int(st["t"]))
            opt.grad.zero_()

        self.enc.LoadStates(ckpt["table"], 0)
        self.n_volumes = self.enc.n_volumes_
        self.mlp.copy_(ckpt["mlp"])
        adam(self.opt_table, ckpt["adam"]["table"])
        adam(self.opt_mlp, ckpt["adam"]["mlp"])
        if self.emb is not None:
            self.emb.copy_(ckpt["emb"])
            adam(self.opt_emb, ckpt["adam"]["emb"])
        self.enc.shadow(force=True)
        s, ss = self.sampler, ckpt["sampler"]
        s.LoadStates(ss["states"], 0)
        s.tree_weight_stats_ = ss["weight_stats"].to(s.device).contiguous()
        s.tree_alpha_stats_ = ss["alpha_stats"].to(s.device).contiguous()
        s.ray_march_fineness_ = float(ss["ray_march_fineness"])
        s.sampled_oct_per_ray_ = float(ss["sampled_oct_per_ray"])
        s.UpdateMode(int(ss["mode"]))
        s._octree_stale = True                 # the host mirror picks the statistics up when somebody asks for it
        self.step_count = int(ckpt["step_count"])
        if ckpt["stage"] == "block_stage" and "res_blocks" in ckpt:
            tables = ckpt["res_block_tables"]
            self.start_block_stage(log2_table_size=int(np.log2(tables[0][0].shape[0] // 16)),
                                   lr=float(ckpt["res_lr"]), blocks=ckpt["res_blocks"])
            for c, o, t, st in zip(self.res_blocks, self.opt_res_blocks, tables, ckpt["adam"]["res_blocks"]):
                c.LoadStates(t, 0)
                c.shadow(force=True)
                adam(o, st)
            self._block_refs()                 # LoadStates replaced the prime pools
        elif ckpt["stage"] == "block_stage":
            self.start_block_stage(log2_table_size=int(np.log2(ckpt["res_table"][0].shape[0] // 16)),
                                   lr=float(ckpt["res_lr"]))
            self.res.LoadStates(ckpt["res_table"], 0)
            self.res.shadow(force=True)
            adam(self.opt_res, ckpt["adam"]["res"])
        elif self.stage == "block_stage":
            self.end_block_stage()

    @torch.no_grad()
    def render_image(self, rays_o, rays_d, rel_camera_index: int = 0, chunk: int = 32768, sample_ahead: bool = True):
        """Full-image render in chunks: Model.get_outputs_for_camera_ray_bundle (nerfstudio/models/base_model.py:
        166-190, eval_num_rays_per_chunk = 2048 in the reference, gfnerf/config.py:109; here the chunk is as large
        as the workspace allows and there is no host sync inside it).  Returns rgb [N,3], depth [N], acc [N]."""
        cam = None
        if self.emb is not None:
            cam = torch.full((rays_o.shape[0],), int(rel_camera_index), dtype=torch.int64, device=self.device)
        return self.render_rays(rays_o, rays_d, cam, chunk, sample_ahead)[:3]

    # ---- per-stage device timing (bench / profiling only) -----------------------------------
    def enable_timers(self, on: bool = True):
        """Brackets every stage with CUDA events on the launching stream; read with `stage_times()`."""
        self._events = [] if on else None
        self.sampler.stage_hook = self._stage if on else None

    def stage_times(self, reset: bool = True):
        """-> {stage: (total ms, calls)} of everything recorded since the last reset (synchronises)."""
        torch.cuda.synchronize(self.device)
        out = {}
        for name, e0, e1 in self._events or []:
            t, c = out.get(name, (0.0, 0))
            out[name] = (t + e0.elapsed_time(e1), c + 1)
        if reset and self._events is not None:
            self._events = []
        return out

    # ---- workspace -----------------------------------------------------------------------
    # ---- data-parallel exchange over NVLink peer memory (csrc/peer.cu) ------------------------------------------
    def _setup_peer_exchange(self, group):
        """Move the buffers the ranks exchange -- table gradient, fp16 gather table, small-gradient bucket -- into
        peer-mapped memory.  Falls back to the NCCL all-reduce path (saying so) if the node cannot map peers."""
        from .peer import PeerExchange
        import torch.distributed as dist
        ok = torch.ones(1, dtype=torch.int32, device=self.device)
        try:
            # votes: two alternating buffers of 4 int64 per octree node (3 adders / marks + the visit count), with room
            # for the tree to grow through the subdivision milestones
            self._vote_cap = 4 * max(16 * int(self.sampler.n_nodes), 1 << 17)
            peer = PeerExchange(group, self.device, {
                "table_grad": 4 * self.opt_table.param.numel(), "shadow": 2 * self.enc.feat_pool_.numel(),
                "small": 4 * self._small.flat.numel(), "votes": 2 * 8 * self._vote_cap})
        except RuntimeError as e:
            peer, ok[0] = None, 0
            import sys
            sys.stderr.write(f"gfnerf_b200: peer-memory exchange unavailable ({e}); using NCCL all-reduce\n")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)     # all ranks or none
        if int(ok.item()) == 0:
            return
        self.peer = peer
        self.opt_table.grad = peer.tensor("table_grad", torch.float32, tuple(self.opt_table.param.shape))
        self.enc._shadow = peer.tensor("shadow", torch.float16, tuple(self.enc.feat_pool_.shape))
        self.enc._shadow_key = None
        self._small.rebind(peer.tensor("small", torch.float32, (self._small.flat.numel(),)))
        self._small_grads = self._small.flat
        self.opt_mlp.grad = self._small.views[0]
        if self.opt_emb is not None:
            self.opt_emb.grad = self._small.views[1].view(-1)
        n4 = (self.opt_table.n_active + 3) // 4
        chunk4 = (n4 + self.world - 1) // self.world
        r = self.sync.rank
        self._peer_own = (min(r * chunk4 * 4, self.opt_table.n_active), min((r + 1) * chunk4 * 4, self.opt_table.n_active))
        self._peer_chunk = chunk4 * 4

    def _peer_exchange(self, lr_scale: float):
        """reduce-scatter + Adam + all-gather of the table, all-reduce + Adam of the small parameters, between two
        cross-GPU barriers, all on the current stream (see csrc/peer.cu)."""
        L, st, peer, W = _lib.lib(), _lib.cur_stream(), self.peer, self.world
        with self._stage("exchange"):
            flag = self._nan_flag([self._small_grads, self.opt_table.grad[:self.opt_table.n_active]])   # this rank's
            ep = peer.next_epoch()
            peer.barrier("in", ep, local_flag=flag, want_any=flag is not None)
            skip = peer.any_flag if flag is not None else None
            self.last_nan_flag = skip

            def run(opt, lo, hi, grad_ptrs, shadow_ptrs, lr):
                n = (opt.param.numel() + 3) // 4 * 4 if shadow_ptrs is None else opt.n_active
                _lib.check(L.gf_peer_reduce_adam(
                    W, n, lo, hi if hi is not None else n, grad_ptrs, _lib.ptr(opt.param), _lib.ptr(opt.m),
                    _lib.ptr(opt.v), shadow_ptrs, float(lr), opt.betas[0], opt.betas[1], opt.eps, _lib.ptr(opt.d_step),
                    float(W) * opt.grad_scale, _lib.ptr(skip), st), "gf_peer_reduce_adam")

            run(self.opt_table, self._peer_own[0], self._peer_own[1], peer.ptrs("table_grad"), peer.ptrs("shadow"),
                self.opt_table.lr * lr_scale)
            run(self.opt_mlp, 0, None, peer.ptrs("small", 4 * self._small.offsets[0]), None, self.opt_mlp.lr * lr_scale)
            if self.opt_emb is not None:
                run(self.opt_emb, 0, None, peer.ptrs("small", 4 * self._small.offsets[1]), None,
                    self.opt_emb.lr * lr_scale)
            peer.barrier("out", ep)
            # every rank has read my gradients: zero them for the next step
            self.opt_table.grad[:self.opt_table.n_active].zero_()
            self._small_grads.zero_()
        self.enc.mark_shadow_fresh()

    def _peer_vote_max(self, buffers):
        """all-reduce(MAX) of the octree votes over peer memory, in stream order on the current (sampling-ahead) stream:
        stage this rank's votes in one of two alternating peer buffers, one cross-GPU barrier, then every rank takes the
        maximum over all ranks' buffers with peer loads (csrc/peer.cu gf_peer_max_i64).  Two buffers, so the barrier of
        step k + 1 is what guarantees that every peer has finished reading the buffer this rank rewrites at k + 2."""
        total = sum(int(b.numel()) for b in buffers)
        if total > self._vote_cap:          # the octree outgrew the buffers (same decision on every rank): NCCL
            return self.sync.max_(buffers)
        L, peer = _lib.lib(), self.peer
        peer.vote_epoch += 1
        slot = peer.vote_epoch & 1
        stage = peer.tensor("votes", torch.int64, (2, self._vote_cap))[slot]
        off = 0
        for b in buffers:
            n = int(b.numel())
            stage[off:off + n].copy_(b.view(-1))
            off += n
        peer.barrier("vote", peer.vote_epoch)
        off = 0
        for b in buffers:
            n = int(b.numel())
            _lib.check(L.gf_peer_max_i64(self.world, n, peer.ptrs("votes", 8 * (slot * self._vote_cap + off)),
                                         _lib.ptr(b), _lib.cur_stream()), "gf_peer_max_i64")
            off += n

    def sync_master_params(self):
        """Peer exchange only: every rank keeps the fp32 master copy (and Adam moments) of ITS rows of the table up to
        date -- the forward reads the fp16 gather table, which is complete everywhere.  Before reading `feat_pool_`
        (checkpoint, inspection) collect the owners' rows; not on the step path."""
        if self.peer is None:
            return
        import torch.distributed as dist
        self.flush()
        n, chunk = self.opt_table.n_active, self._peer_chunk
        for t in (self.opt_table.param, self.opt_table.m, self.opt_table.v):
            mine = torch.zeros(chunk, dtype=t.dtype, device=t.device)
            lo, hi = self._peer_own
            mine[:hi - lo] = t[lo:hi]
            allr = torch.empty(chunk * self.world, dtype=t.dtype, device=t.device)
            dist.all_gather_into_tensor(allr, mine, group=self.sync.group)
            t[:n] = allr[:n]

    @torch.no_grad()
    def train_step(self, rays_o, rays_d, target_rgb, rel_camera_indices=None, noise=None, lr_scale: float = 1.0,
                   update_octree: bool = True, optimizer_step: bool = True, next_rays=None) -> StepOutputs:
        """next_rays = (rays_o, rays_d) of the batch the NEXT call will be given: their sampling is started as soon
        as this step's octree vote has been issued and overlaps this step's backward pass (`_presample`).

        Several focal blocks (start_block_stage(blocks=...)): the batch is K equal contiguous segments, segment k
        belonging to blocks[k].  The loss terms are computed per segment (S3IM's permutations stay inside it) and
        returned in `block_losses`; `loss` is their sum.  One routed scatter takes every sample to its block's
        gradient table, and each block has its own NaN guard and Adam step."""
        L = _lib.lib()
        multi = self.stage == "block_stage" and self.blocks is not None
        K = len(self.blocks) if multi else 1
        ray_table = self.block_ray_table(rays_o.shape[0]) if multi else None
        with torch.cuda.device(self.device):
            st = _lib.cur_stream()
            step = self.step_count
            cs = self._take_presampled(rays_o, rays_d) if noise is None else None
            if cs is None:
                cs = self.sampler.sample_compact(rays_o, rays_d, noise=noise, slot=getattr(self, "_cs_slot", 0))
            self.flush()   # a deferred optimizer step of the previous iteration lands here
            cap, R = cs.pts01.shape[0], cs.n_rays
            ray_emb = self._ray_emb(rel_camera_indices)
            feat, sigma, rgb, ray_bias = self._field_forward(cs, ray_emb, train=True, ray_table=ray_table)
            out_rgb, depth, acc, weights, alphas, trans = self._composite(cs, sigma, rgb, keep=True)
            # loss (CharbonnierLoss, nerfstudio/model_components/losses.py:73-84)
            g_rgb = self._buf("g_rgb", (R, 3), torch.float32)
            target = target_rgb.contiguous().float()
            Rb = R // K
            losses = torch.zeros(K, dtype=torch.float32, device=self.device)   # K = 1: the step's loss
            with self._stage("loss"):
                for k in range(K):
                    _lib.check(L.gf_charbonnier(Rb, _lib.ptr(out_rgb[k * Rb:]), _lib.ptr(target[k * Rb:]), 1e-6,
                                                _lib.ptr(g_rgb[k * Rb:]), _lib.ptr(losses[k:]), st), "gf_charbonnier")
            mult, ks, stride, repeat, patch_h = self.s3im
            if mult > 0.0 and (Rb * repeat) % patch_h == 0:
                # S3IM.forward (losses.py:779-794): the batch once in order, then repeat-1 random permutations
                perms = torch.rand((K, repeat - 1, Rb), device=self.device).argsort(dim=2)
                for k in range(K):
                    index = torch.cat([torch.arange(Rb, device=self.device).view(1, Rb), perms[k]]).reshape(-1).contiguous()
                    with self._stage("loss"):
                        _lib.check(L.gf_s3im(Rb, index.numel(), _lib.ptr(index), _lib.ptr(out_rgb[k * Rb:]),
                                             _lib.ptr(target[k * Rb:]), patch_h, ks, stride, mult,
                                             _lib.ptr(g_rgb[k * Rb:]), _lib.ptr(losses[k:]), st), "gf_s3im")
            loss = losses.sum().view(1) if multi else losses
            # training feedback (gfnerf/nerfacto.py:598-616).  It only needs the forward's weights, so it is issued
            # here: its (tiny) MAX all-reduce over ranks must not queue behind the gradient all-reduce below
            vote = None
            if update_octree and self.stage == "init_stage":   # the octree is only updated in the init stage (:605)
                if next_rays is not None:
                    vote = (cs, weights, alphas, step)        # issued with the next batch's sampling, see _presample
                else:
                    with self._stage("octree_vote"):
                        self.sampler.update_oct_nodes_compact(cs, weights, alphas, step)
                        self.sampler.UpdateRayMarch(step)
            presample_late = next_rays is not None and getattr(self, "presample_after_mlp", True)
            fwd_done = torch.cuda.current_stream(self.device).record_event() if presample_late else None
            if next_rays is not None and not presample_late:
                self._presample(next_rays[0], next_rays[1], vote, after=fwd_done)
            # backward
            d_sigma = self._buf("d_sigma", (cap,), torch.float32)
            d_rgb = self._buf("d_rgb", (cap, 3), torch.float32)
            with self._stage("composite_bwd"):
                _lib.check(L.gf_composite_backward(R, _lib.ptr(cs.offsets), _lib.ptr(sigma), _lib.ptr(cs.delta),
                                                   _lib.ptr(rgb), _lib.ptr(trans), _lib.ptr(g_rgb), None, None,
                                                   _lib.ptr(d_sigma), _lib.ptr(d_rgb), st), "gf_composite_backward")
            d_feat = self._buf("d_feat", (cap, 32), torch.float16)
            grad_scale = float(2 ** int(np.ceil(np.log2(max(Rb, 1)))))   # (per block: the single-block d_feat bits)
            block = self.stage == "block_stage"
            d_ray_bias = None if block else self._buf("d_ray_bias", (R, self.hidden), torch.float32, zero=True)
            with self._stage("mlp_bwd"):   # block stage: frozen MLP, only d_feat
                _lib.check(L.gf_mlp_backward(cap, _lib.ptr(cs.total), self.hidden, _lib.ptr(self.mlp), _lib.ptr(feat),
                                             _lib.ptr(cs.ray_id), _lib.ptr(ray_bias),
                                             _lib.ptr(self._buf("relu_masks", (cap, self.mask_words), torch.int32)),
                                             _lib.ptr(d_sigma), _lib.ptr(d_rgb), _lib.ptr(d_feat),
                                             None if block else _lib.ptr(self.opt_mlp.grad),
                                             _lib.ptr(d_ray_bias), grad_scale, st), "gf_mlp_backward")
            if presample_late:
                # issued behind the MLP backward: that kernel is resident first (2 CTAs / SM, tensor pipe + epilogue,
                # ~25 % of the issue slots) and the sampler's CTAs fill the registers it leaves free
                self._presample(next_rays[0], next_rays[1], vote, after=fwd_done)
            if multi:
                with self._stage("hash_bwd"):
                    Hash3DAnchoredCore.launch_backward_routed(self.res_blocks, cs.pts01, cs.anchor, d_feat, True,
                                                              cs.ray_id, ray_table, refs=self._grad_refs,
                                                              d_n_ptr=cs.total, keep_x128=True)
                if optimizer_step:
                    with self._stage("adam_table"):
                        flags = self._nan_flags([o.grad[:o.n_active] for o in self.opt_res_blocks])
                        for k, (res, opt) in enumerate(zip(self.res_blocks, self.opt_res_blocks)):
                            opt.step(shadow=res._shadow, lr=opt.lr * lr_scale,
                                     skip_flag=None if flags is None else flags[k:k + 1])
                            res.mark_shadow_fresh()
            elif block:
                with self._stage("hash_bwd"):
                    self.res.launch_backward(cs.pts01, cs.anchor, d_feat, True, self.opt_res.grad.view(-1, 2),
                                             d_n_ptr=cs.total, keep_x128=True)
                if optimizer_step:
                    with self._stage("adam_table"):
                        self.opt_res.step(shadow=self.res._shadow, lr=self.opt_res.lr * lr_scale,
                                          skip_flag=self._nan_flag([self.opt_res.grad[:self.opt_res.n_active]]))
                    self.res.mark_shadow_fresh()
            else:
                d_ray_emb = (self._buf("d_ray_emb", (R, APPEARANCE_DIM), torch.float32, zero=True)
                             if ray_emb is not None else None)
                with self._stage("ray_bias_bwd"):
                    _lib.check(L.gf_mlp_ray_bias_backward(R, self.hidden, _lib.ptr(self.mlp), _lib.ptr(cs.rays_d),
                                                          _lib.ptr(ray_emb), _lib.ptr(d_ray_bias),
                                                          _lib.ptr(self.opt_mlp.grad), _lib.ptr(d_ray_emb), st),
                               "gf_mlp_ray_bias_backward")
                    if d_ray_emb is not None:
                        self.opt_emb.grad.view(-1, APPEARANCE_DIM).index_add_(0, rel_camera_indices.to(torch.int64),
                                                                              d_ray_emb)
                g_table = self.opt_table.grad.view(-1, 2)
                if self.peer is not None and optimizer_step:
                    with self._stage("hash_bwd"):
                        self.enc.launch_backward(cs.pts01, cs.anchor, d_feat, True, g_table, d_n_ptr=cs.total,
                                                 keep_x128=True)
                    self._peer_exchange(lr_scale)
                elif self.world > 1 and optimizer_step:
                    # data parallel: the small bucket's all-reduce starts now and runs under the scatter; the table is
                    # scattered and all-reduced in LEVEL_GROUP-level groups.  Level l owns rows [l*T/2, l*T/2 + T)
                    # (level_base_row: windows overlap by half), so once levels < l1 are scattered the rows below
                    # l1*T/2 are final; the last group takes the rest of the reachable rows.
                    self.sync.start_sum([self._small_grads])
                    with self._stage("hash_bwd"):
                        for l0, l1, r0, r1 in table_reduce_ranges(self.enc.local_size_, self.LEVEL_GROUP):
                            self.enc.launch_backward(cs.pts01, cs.anchor, d_feat, True, g_table, d_n_ptr=cs.total,
                                                     keep_x128=True, levels=(l0, l1))
                            self.sync.start_sum([g_table[r0:r1]])
                    self._deferred = lr_scale
                else:
                    with self._stage("hash_bwd"):
                        self.enc.launch_backward(cs.pts01, cs.anchor, d_feat, True, g_table, d_n_ptr=cs.total,
                                                 keep_x128=True)
                    if optimizer_step:
                        self._reduce_and_step(lr_scale)
            self.step_count += 1
        return StepOutputs(out_rgb, depth, acc, loss, cs.total, losses if multi else None)

    # ---- host-buffer entry point ------------------------------------------------------------------------------
    @torch.no_grad()
    def train_step_host(self, rays_o, rays_d, target_rgb, rel_camera_indices=None, next_rays=None, **kw) -> StepOutputs:
        """`train_step` for HOST tensors (pinned for true asynchrony), the call a data loader makes: the batch goes
        host -> device on a copy stream into one of three staging slots, so the copy of batch k + 1 overlaps the
        compute of batch k (three, not two: the slot batch k + 1 is staged into was last read by step k - 2, so the copy
        never waits for the step in flight -- with two slots every step started one H2D latency after the previous one
        had drained); the step's loss comes back device -> host asynchronously into a pinned ring
        (`read_losses()`), so the host never blocks inside the training loop (the reference blocks five times per
        step on .item(), SURVEY.md section 1).  next_rays = the NEXT call's (rays_o, rays_d) host tensors: they are
        staged now and sampled underneath this step's backward pass (`train_step(next_rays=...)`)."""
        dev = self.device
        if not hasattr(self, "_h2d"):
            self._h2d = dict(stream=torch.cuda.Stream(device=dev), d2h=torch.cuda.Stream(device=dev), slot=0,
                             free=[None] * 3, bufs=[{}, {}, {}], losses=[], pinned=None, staged_rays=[None] * 3)
        h = self._h2d
        slot = h["slot"]
        h["slot"] = (slot + 1) % 3
        cur = torch.cuda.current_stream(dev)

        def stage(slot_, name, src):
            buf = h["bufs"][slot_].get(name)
            if buf is None or buf.shape != src.shape or buf.dtype != src.dtype:
                buf = torch.empty(src.shape, dtype=src.dtype, device=dev)
                h["bufs"][slot_][name] = buf
            buf.copy_(src, non_blocking=True)
            return buf

        names = ("o", "d", "t", "c")
        host = (rays_o, rays_d, target_rgb, rel_camera_indices)
        # rays already staged by the previous call's next_rays?
        pre = h["staged_rays"][slot]
        have_rays = pre is not None and pre == (rays_o.data_ptr(), rays_d.data_ptr(), tuple(rays_o.shape))
        h["staged_rays"][slot] = None
        staged = []
        with torch.cuda.stream(h["stream"]):
            if h["free"][slot] is not None:    # the step that last read this slot (three calls ago) has finished
                h["stream"].wait_event(h["free"][slot])
            for name, src in zip(names, host):
                if src is None:
                    staged.append(None)
                elif have_rays and name in ("o", "d"):
                    staged.append(h["bufs"][slot][name])
                else:
                    staged.append(stage(slot, name, src))
            nxt = None
            if next_rays is not None:
                nslot = (slot + 1) % 3
                if h["free"][nslot] is not None:
                    h["stream"].wait_event(h["free"][nslot])
                nxt = (stage(nslot, "o", next_rays[0]), stage(nslot, "d", next_rays[1]))
                h["staged_rays"][nslot] = (next_rays[0].data_ptr(), next_rays[1].data_ptr(), tuple(next_rays[0].shape))
            ready = h["stream"].record_event()
        cur.wait_event(ready)
        out = self.train_step(staged[0], staged[1], staged[2], staged[3], next_rays=nxt, **kw)
        done = cur.record_event()
        h["free"][slot] = done
        # the loss goes home on its own stream, behind the step: the step's stream is not held up by a 4-byte DMA, and
        # the pinned ring is allocated once (a pinned allocation per step is a cudaHostAlloc per step)
        k = len(h["losses"])
        ring = h["pinned"]
        if ring is None or k >= ring.numel():
            new = torch.empty(max(1024, 2 * (k + 1)), dtype=torch.float32).pin_memory()
            if ring is not None:
                for ev in h["losses"]:
                    ev.synchronize()
                new[:k] = ring[:k]
            h["pinned"] = ring = new
        with torch.cuda.stream(h["d2h"]):
            h["d2h"].wait_event(done)
            ring[k:k + 1].copy_(out.loss, non_blocking=True)
            out.loss.record_stream(h["d2h"])
            h["losses"].append(h["d2h"].record_event())
        return out

    def read_losses(self):
        """Losses of the `train_step_host` calls since the last read (waits for their device -> host copies)."""
        h = getattr(self, "_h2d", None)
        if h is None:
            return []
        vals = []
        for k, ev in enumerate(h["losses"]):
            ev.synchronize()
            vals.append(float(h["pinned"][k]))
        h["losses"] = []
        return vals

    def _reduce_and_step(self, lr_scale: float):
        """DDP semantics (mean over ranks) for ALL parameters -- including the hash table, which the reference's
        DDP wrapper silently skips because feat_pool is not a registered nn.Parameter (SURVEY.md section 5).
        With more than one rank the all-reduce is launched on the comm stream and the Adam step is DEFERRED to the
        point where the parameters are next needed: the start of the next iteration's forward (`flush`).  With
        `next_rays` the next batch's sampling has moved underneath the backward pass, so there the reduce is exposed
        (DESIGN.md section 6)."""
        if self.world > 1:   # (train_step pipelines this per level group; this is the one-shot form)
            # rows past used_rows_ never receive a gradient on any rank (level_base_row): nothing to exchange there
            self.sync.start_sum([self._small_grads, self.opt_table.grad.view(-1, 2)[:self.enc.used_rows_]])
            self._deferred = lr_scale
        else:
            self._apply_adam(lr_scale)

    def flush(self):
        """Completes a deferred optimizer step (call before reading parameters, checkpointing or timing)."""
        super().flush()       # an octree vote / sampling issued ahead on the side stream
        if self._deferred is not None:
            self.sync.wait()
            self._apply_adam(self._deferred)
            self._deferred = None

    def _nan_flag(self, grads):
        """device flag = any NaN in the (already all-reduced) gradients; None when the guard is off"""
        if not self.nan_guard:
            return None
        flag = self._buf("nan_flag", (1,), torch.int32, zero=True)
        L, st = _lib.lib(), _lib.cur_stream()
        for g in grads:
            _lib.check(L.gf_grad_nan_scan(g.numel(), _lib.ptr(g), _lib.ptr(flag), st), "gf_grad_nan_scan")
        self.last_nan_flag = flag
        return flag

    def _nan_flags(self, grads):
        """device int32 [len(grads)]: flag k = any NaN in grads[k] (one guard per focal block); None when the guard is
        off"""
        if not self.nan_guard:
            return None
        flags = self._buf("nan_flags", (len(grads),), torch.int32, zero=True)
        L, st = _lib.lib(), _lib.cur_stream()
        for k, g in enumerate(grads):
            _lib.check(L.gf_grad_nan_scan(g.numel(), _lib.ptr(g), _lib.ptr(flags[k:]), st), "gf_grad_nan_scan")
        self.last_nan_flag = flags
        return flags

    def _apply_adam(self, lr_scale: float):
        div = float(self.world)
        with self._stage("adam_small"):
            flag = self._nan_flag([self._small_grads, self.opt_table.grad[:self.opt_table.n_active]])
            self.opt_mlp.step(grad_div=div, lr=self.opt_mlp.lr * lr_scale, skip_flag=flag)
            if self.opt_emb is not None:
                self.opt_emb.step(grad_div=div, lr=self.opt_emb.lr * lr_scale, skip_flag=flag)
        with self._stage("adam_table"):
            self.opt_table.step(shadow=self.enc._shadow, grad_div=div, lr=self.opt_table.lr * lr_scale, skip_flag=flag)
        self.enc.mark_shadow_fresh()
