"""Error-map importance sampling of training pixels for the focal (block) stage -- SURVEY.md 8(f) rank 4, the step
before ray generation -- and the error-map feedback after the forward pass.

Mirrors `ErrorPixelSampler` (nerfstudio/data/pixel_samplers.py:594-760, tensor-batch path) and
`TrainDataloader._update_error_map` (nerfstudio/data/utils/dataloaders.py:140-142) as called from
gfnerf/gf_pipeline.py:180-185: same method names, argument meaning and batch keys.

What is different, on purpose:
  * the batch (images, error map) is expected to be resident in HBM; nothing here moves it;
  * the 80 % uniform draw is done on the batch's device (`uniform_without_replacement`) instead of Python's
    `random.sample` over `range(n_pixels)` (6.5 k Python-level draws per step);
  * the `nonzero(error_map >= 0)` table the reference builds every step (n_pixels x 3 int64: 50 MB for 2 M pixels)
    is replaced by unravelling the flat pixel number, which is what that table holds whenever no entry is negative;
    with negative entries the reference's table is shorter than the flat weights it is indexed by -- that quirk is
    reproduced through the same `nonzero` call so behaviour (including the IndexError) is unchanged;
  * the error feedback is one kernel (`gf_error_map_update`, csrc/rays.cu) instead of abs / sum / index_put.

The weighted 20 % draw is `torch.multinomial` without replacement in chunks of 2^24, exactly as the reference:
which pixels come out is defined by torch's generator, so parity here is distributional (tests/test_pixel_samplers.py).
"""
from typing import Dict, Optional

import torch

from . import _lib

MULTINOMIAL_CHUNK = 2 ** 24      # torch.multinomial's category limit; pixel_samplers.py:647


def uniform_without_replacement(n: int, k: int, device, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """k distinct integers of [0, n), uniformly, in draw order (the reference: `random.sample(range(n), k)`).
    Draw k, re-draw the (rare) duplicates until none is left; expected rounds ~ 1 + k^2 / (2 n)."""
    if k < 0 or k > n:
        raise ValueError("Sample larger than population or is negative")        # random.sample's own error
    if k == 0:
        return torch.empty(0, dtype=torch.int64, device=device)
    if 2 * k > n:                                                              # dense case: a permutation is cheaper
        return torch.randperm(n, device=device, generator=generator)[:k]
    idx = torch.randint(n, (k,), device=device, generator=generator)
    while True:
        s, order = idx.sort(stable=True)
        dup_sorted = torch.zeros(k, dtype=torch.bool, device=device)
        dup_sorted[1:] = s[1:] == s[:-1]
        n_dup = int(dup_sorted.sum())
        if n_dup == 0:
            return idx
        idx[order[dup_sorted]] = torch.randint(n, (n_dup,), device=device, generator=generator)


class ErrorPixelSampler:
    """Samples pixel batches from an image batch: `weighted_choice_ratio` of them in proportion to the error map,
    the rest uniformly."""

    def __init__(self, num_rays_per_batch: int, keep_full_image: bool = False,
                 generator: Optional[torch.Generator] = None, **kwargs) -> None:
        self.kwargs = kwargs
        self.num_rays_per_batch = num_rays_per_batch
        self.keep_full_image = keep_full_image
        self.weighted_choice_ratio = 0.2                                       # pixel_samplers.py:606
        self.generator = generator

    def set_num_rays_per_batch(self, num_rays_per_batch: int):
        self.num_rays_per_batch = num_rays_per_batch

    def weighted_choice_multinomial(self, dist: torch.Tensor, size: int, device) -> torch.Tensor:
        """`size` flat pixel numbers drawn without replacement in proportion to `dist` (pixel_samplers.py:634-669):
        one multinomial if n < 2^24; else size // n_chunks from every full 2^24-chunk (each normalised on its own)
        and the size % n_chunks remainder from the tail chunk, or uniformly if n is a multiple of n_chunks."""
        n = dist.shape[0]
        n_chunks = n // MULTINOMIAL_CHUNK
        g = self.generator
        if n_chunks == 0:
            return torch.multinomial(dist, size, False, generator=g).to(device).long()
        picks = []
        for i in range(n_chunks):
            lo = i * MULTINOMIAL_CHUNK
            picks.append(torch.multinomial(dist[lo:lo + MULTINOMIAL_CHUNK], size // n_chunks, False, generator=g) + lo)
        rest = size % n_chunks
        if rest:
            if n % n_chunks != 0:
                lo = n_chunks * MULTINOMIAL_CHUNK
                picks.append(torch.multinomial(dist[lo:], rest, False, generator=g) + lo)
            else:
                picks.append(uniform_without_replacement(n, rest, dist.device, g))
        out = torch.cat(picks, dim=0).long().to(device)
        assert out.shape[0] == size
        return out

    def sample_method(self, batch_size: int, num_images: int, image_height: int, image_width: int,
                      error_map: torch.Tensor, device="cpu") -> torch.Tensor:
        """int64 [batch_size, 3] = (image slot, y, x): first int(batch_size * ratio) error-weighted rows, then the
        uniform ones (pixel_samplers.py:672-716)."""
        if error_map.dim() == 4:
            error_map = error_map.squeeze(-1)                                  # (n_image, h, w)
        weights = error_map.reshape(-1)
        n_pixels = weights.shape[0]
        n_weighted = int(batch_size * self.weighted_choice_ratio)
        chosen = torch.cat((self.weighted_choice_multinomial(weights, n_weighted, device),
                            uniform_without_replacement(n_pixels, batch_size - n_weighted, weights.device,
                                                        self.generator).to(device)), dim=0)
        if bool((weights >= 0).all()):
            h, w = error_map.shape[1], error_map.shape[2]
            indices = torch.stack((chosen // (h * w), (chosen // w) % h, chosen % w), dim=-1)
        else:                                                                  # the reference's table, quirk included
            indices = torch.nonzero(error_map >= 0.0, as_tuple=False).to(device)[chosen]
        assert indices.shape[0] == batch_size
        return indices.long()

    def collate_image_dataset_batch(self, batch: Dict, num_rays_per_batch: int, keep_full_image: bool = False):
        """Gathers every per-pixel entry of `batch` at the sampled pixels (pixel_samplers.py:718-757).  Returned keys:
        the batch's own per-pixel keys (`image`, `error_map`, masks ...), `indices` (column 0 = absolute camera
        index, `image_idx[slot]`), `rel_camera_indices`, and `full_image` if asked for."""
        device = batch["image"].device
        num_images, image_height, image_width, _ = batch["image"].shape
        indices = self.sample_method(num_rays_per_batch, num_images, image_height, image_width,
                                     error_map=batch["error_map"], device=device)
        c, y, x = indices[:, 0], indices[:, 1], indices[:, 2]
        out = {k: v[c, y, x] for k, v in batch.items() if k not in ("image_idx", "rel_camera_idx") and v is not None}
        assert out["image"].shape == (num_rays_per_batch, 3), out["image"].shape
        out["slot_indices"] = indices.clone()              # (slot, y, x): what update_error_map needs (see there)
        indices = indices.clone()
        indices[:, 0] = batch["image_idx"].to(device)[c]
        out["indices"] = indices
        out["rel_camera_indices"] = batch["rel_camera_idx"].to(device)[c]
        if keep_full_image:
            out["full_image"] = batch["image"]
        return out

    def sample(self, image_batch: Dict):
        if isinstance(image_batch["image"], torch.Tensor):
            return self.collate_image_dataset_batch(image_batch, self.num_rays_per_batch,
                                                    keep_full_image=self.keep_full_image)
        raise ValueError("image_batch['image'] must be a torch.Tensor (the list path of the reference, "
                         "pixel_samplers.py:759-829, calls sample_method with arguments it does not take)")


def update_error_map(error_map: torch.Tensor, ray_indices: torch.Tensor, pred_rgb: torch.Tensor,
                     gt_rgb: torch.Tensor, return_error: bool = False, check_indices: bool = True):
    """error_map[ray_indices[:,0], ray_indices[:,1], ray_indices[:,2]] = sum_c |gt - pred|, in place, one kernel.

    The reference passes `batch["indices"]`, whose column 0 is the ABSOLUTE camera index, and indexes the cached
    batch's error map (ordered by slot) with it (gf_pipeline.py:185, dataloaders.py:142): right only when the cached
    batch holds every image in dataset order, which is the configuration GF-NeRF trains in.  This function indexes
    with whatever it is given, like the reference; `ErrorPixelSampler` also returns `slot_indices` for callers whose
    cached batch is a subset.

    `check_indices` reads the kernel's out-of-range flag back (one 4-byte D2H, which waits for the forward that
    produced `pred_rgb`) to raise torch's IndexError; a training loop that trusts its sampler passes False and the
    bad rows are simply skipped."""
    _lib.require_cuda(error_map, ray_indices, pred_rgb, gt_rgb)
    if error_map.dtype != torch.float32 or not error_map.is_contiguous():
        raise RuntimeError("update_error_map: error_map must be a contiguous f32 tensor [n,h,w] or [n,h,w,1]")
    if error_map.dim() == 4 and error_map.shape[-1] == 1:
        n_img, h, w = error_map.shape[:3]
    elif error_map.dim() == 3:
        n_img, h, w = error_map.shape
    else:
        raise RuntimeError("update_error_map: error_map must be [n,h,w] or [n,h,w,1]")
    n = ray_indices.shape[0]
    if ray_indices.shape != (n, 3) or pred_rgb.shape != (n, 3) or gt_rgb.shape != (n, 3):
        raise RuntimeError("update_error_map: ray_indices i64 [n,3], pred_rgb / gt_rgb f32 [n,3]")
    idx = ray_indices.to(torch.int64).contiguous()
    pred, gt = pred_rgb.detach().float().contiguous(), gt_rgb.detach().float().contiguous()
    err = torch.empty(n, dtype=torch.float32, device=error_map.device) if return_error else None
    bad = torch.zeros(1, dtype=torch.int32, device=error_map.device)
    with torch.cuda.device(error_map.device):
        _lib.check(_lib.lib().gf_error_map_update(n, _lib.ptr(idx), _lib.ptr(pred), _lib.ptr(gt), n_img, h, w,
                                                  _lib.ptr(error_map), _lib.ptr(err), _lib.ptr(bad),
                                                  _lib.cur_stream()), "gf_error_map_update")
    if check_indices and int(bad.item()):
        raise IndexError("update_error_map: ray index out of range for the error map")   # torch raises here too
    return err


class FocalBatchSource:
    """Training batches of the focal (block) stage drawn on the device: `ErrorPixelSampler.sample_method`'s
    distribution with work in proportion to the batch, not to the error map, and no host read between steps.

    Unlike `ErrorPixelSampler`, which nerfstudio's datamanager calls with whatever image batch it holds, this source
    OWNS `error_map`: it keeps a sum tree of it (fp64 sums and non-zero counts over 1024-pixel tiles, up to one total
    per 2^24-pixel chunk) that `update` keeps current.  A caller that writes `error_map` in any other way calls
    `rebuild()` before the next draw.

    * weighted part: int(R * weighted_choice_ratio) distinct pixels in proportion to the map, drawn without replacement
      (successive sampling, as torch.multinomial), with the reference's chunk rule (`weighted_choice_multinomial`);
    * uniform part: the other rows, distinct and uniform, independent of the weighted part (the two may overlap);
    * rows are (slot, y, x), weighted first, as `sample_method` returns them.

    Draws are made with replacement and the first occurrence of each pixel is kept, in rounds on the device
    (`max_rounds` launches at most; the rounds after the last job is complete return at once).  The pseudo-random
    state (Philox seed and counter) lives on the device, so `next_batch` + `update` can be captured in a CUDA graph and
    every replay draws new pixels.  What torch would raise inside the draw is recorded in a device flag instead, and
    `check()` raises it: a chunk with fewer non-zero pixels than it must draw, a non-finite chunk sum, a job still
    incomplete after `max_rounds` rounds (an error map whose mass sits on far fewer pixels than the batch draws), and
    an out-of-range row given to `update`."""

    _ERRORS = ((1, "a 2^24-pixel chunk of the error map has fewer non-zero pixels than it must draw "
                   "(torch.multinomial: not enough non-negative category to sample)"),
               (2, "the error map holds a non-finite value (torch.multinomial: invalid multinomial distribution)"),
               (4, "a draw did not complete within max_rounds rounds: the error map's mass sits on too few pixels"))
    _CAND_FACTOR = 8            # candidate slots per pixel a job draws: the last rounds draw up to 8x what is missing

    def __init__(self, images: torch.Tensor, error_map: torch.Tensor, cameras, image_idx: torch.Tensor,
                 rel_camera_idx: torch.Tensor, num_rays_per_batch: int = 8192, weighted_choice_ratio: float = 0.2,
                 seed: int = 0, max_rounds: int = 16):
        _lib.require_cuda(images, error_map, image_idx, rel_camera_idx)
        if images.dim() != 4 or images.shape[-1] != 3 or images.dtype != torch.float32 or not images.is_contiguous():
            raise RuntimeError("FocalBatchSource: images must be a contiguous f32 tensor [n,h,w,3]")
        n_img, h, w = images.shape[:3]
        if error_map.dtype != torch.float32 or not error_map.is_contiguous() or \
                tuple(error_map.shape) not in ((n_img, h, w, 1), (n_img, h, w)):
            raise RuntimeError("FocalBatchSource: error_map must be a contiguous f32 tensor [n,h,w,1] like images")
        if error_map.device != images.device or error_map.data_ptr() % 16:
            raise RuntimeError("FocalBatchSource: error_map must be 16-byte aligned, on the images' device")
        if image_idx.shape != (n_img,) or rel_camera_idx.shape != (n_img,):
            raise RuntimeError("FocalBatchSource: image_idx and rel_camera_idx hold one entry per image [n]")
        dev = images.device
        self.device, self.images, self.error_map, self.cameras = dev, images, error_map, cameras
        self.shape = (n_img, h, w)
        self.image_idx = image_idx.to(dev, torch.int64).contiguous()
        self.rel_camera_idx = rel_camera_idx.to(dev, torch.int64).contiguous()
        n = n_img * h * w
        R = int(num_rays_per_batch)
        n_w = int(R * weighted_choice_ratio)
        if n == 0:
            raise RuntimeError("FocalBatchSource: empty image set")
        if R <= 0 or not 0 <= n_w <= R:
            raise ValueError("FocalBatchSource: num_rays_per_batch > 0 and 0 <= weighted_choice_ratio <= 1")
        if not 0 < max_rounds <= 64:
            raise ValueError("FocalBatchSource: max_rounds in [1, 64]")
        self.num_rays_per_batch, self.n_weighted, self.max_rounds = R, n_w, int(max_rounds)

        # the reference's rule (weighted_choice_multinomial, sample_method): (lo, hi, count, weighted, tree chunk)
        C = MULTINOMIAL_CHUNK
        n_chunks = n // C
        jobs = []
        if n_chunks == 0:
            jobs.append((0, n, n_w, 1, 0))
        else:
            jobs += [(i * C, (i + 1) * C, n_w // n_chunks, 1, i) for i in range(n_chunks)]
            rest = n_w % n_chunks
            if rest:
                jobs.append((n_chunks * C, n, rest, 1, n_chunks) if n % n_chunks else (0, n, rest, 0, 0))
        jobs.append((0, n, R - n_w, 0, 0))
        jobs = [j for j in jobs if j[2] > 0]
        for lo, hi, cnt, weighted, _ in jobs:
            if not weighted and cnt > hi - lo:
                raise ValueError("Sample larger than population or is negative")   # random.sample's own error
        table, slot_job, cand_off, out_off, tab_off = [], [], 0, 0, 0
        for j, (lo, hi, cnt, weighted, chunk) in enumerate(jobs):
            cand_cap = self._CAND_FACTOR * cnt + 64
            tab_cap = 1 << (2 * (cnt + cand_cap) - 1).bit_length()
            table.append((lo, hi, cnt, weighted, chunk, cand_off, cand_cap, out_off, tab_off, tab_cap))
            slot_job.append(torch.full((cand_cap,), j, dtype=torch.int32))
            cand_off, out_off, tab_off = cand_off + cand_cap, out_off + cnt, tab_off + tab_cap
        if cand_off * self.max_rounds >= 2 ** 31:
            raise ValueError("FocalBatchSource: batch too large for max_rounds")
        self._jobs = torch.tensor(table, dtype=torch.int64, device=dev)
        self._slot_job = torch.cat(slot_job).to(dev)
        self._cand = torch.empty(cand_off, dtype=torch.int64, device=dev)
        self._tab_keys = torch.empty(tab_off, dtype=torch.int64, device=dev)
        self._tab_pos = torch.empty(tab_off, dtype=torch.int32, device=dev)
        self._work = torch.zeros(len(table) + 1, dtype=torch.int32, device=dev)
        self._rng = torch.tensor([int(seed), 0], dtype=torch.int64, device=dev)
        self._sel = torch.zeros(R, dtype=torch.int64, device=dev)
        self._err = torch.zeros(2, dtype=torch.int32, device=dev)      # draw errors, update's out-of-range rows
        nodes = int(_lib.lib().gf_sumtree_nodes(n))
        self.sums = torch.empty(nodes, dtype=torch.float64, device=dev)
        self.counts = torch.empty(nodes, dtype=torch.int32, device=dev)
        f = lambda *s, dt=torch.float32: torch.empty(s, dtype=dt, device=dev)
        self._coords, self._cam = f(R, 2), f(R, dt=torch.int64)
        self._batch = {"origins": f(R, 3), "directions": f(R, 3), "rgb": f(R, 3),
                       "rel_camera_indices": f(R, dt=torch.int64), "slot_indices": f(R, 3, dt=torch.int64),
                       "indices": f(R, 3, dt=torch.int64)}

        # one host read: the map's range (aminmax: NaN propagates) and the camera indices' range
        mn, mx, c_lo, c_hi = torch.cat([torch.stack(torch.aminmax(self.error_map)).double(),
                                        torch.stack(torch.aminmax(self.image_idx)).double()]).tolist()
        if not (mn >= 0.0 and mx < float("inf")):
            raise ValueError("FocalBatchSource: the error map has a negative or non-finite entry")
        if c_lo < 0 or c_hi >= len(cameras):
            raise RuntimeError("FocalBatchSource: image_idx out of range of the cameras")
        self.rebuild()

    def rebuild(self) -> None:
        """Recomputes the whole sum tree from `error_map` (after the caller wrote the map directly)."""
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().gf_sumtree_build(self.error_map.numel(), _lib.ptr(self.error_map), _lib.ptr(self.sums),
                                                   _lib.ptr(self.counts), _lib.cur_stream()), "gf_sumtree_build")

    def next_batch(self) -> Dict[str, torch.Tensor]:
        """Draws the next batch.  Returns the same dict of fixed buffers every call (overwritten by the next call):
        origins, directions [R,3] (Cameras.generate_rays of the pixel centres), rgb [R,3] = images[slot, y, x],
        rel_camera_indices [R], slot_indices [R,3] = (slot, y, x) and indices [R,3] = (image_idx[slot], y, x)."""
        b, cams, n_img, h, w = self._batch, self.cameras, *self.shape
        L = _lib.lib()
        with torch.cuda.device(self.device):
            s = _lib.cur_stream()
            _lib.check(L.gf_focal_draw(
                n_img, h, w, _lib.ptr(self.error_map), _lib.ptr(self.sums), _lib.ptr(self.counts), self._jobs.shape[0],
                _lib.ptr(self._jobs), _lib.ptr(self._slot_job), self._cand.numel(), _lib.ptr(self._cand),
                _lib.ptr(self._tab_keys), _lib.ptr(self._tab_pos), _lib.ptr(self._work), _lib.ptr(self._rng),
                self.max_rounds, self.num_rays_per_batch, _lib.ptr(self._sel), _lib.ptr(self.images),
                _lib.ptr(self.image_idx), _lib.ptr(self.rel_camera_idx), _lib.ptr(b["slot_indices"]),
                _lib.ptr(b["indices"]), _lib.ptr(b["rel_camera_indices"]), _lib.ptr(b["rgb"]), _lib.ptr(self._coords),
                _lib.ptr(self._cam), _lib.ptr(self._err), s), "gf_focal_draw")
            _lib.check(L.gf_generate_rays(
                self.num_rays_per_batch, _lib.ptr(self._cam), _lib.ptr(self._coords), _lib.ptr(cams.camera_to_worlds),
                _lib.ptr(cams.fx), _lib.ptr(cams.fy), _lib.ptr(cams.cx), _lib.ptr(cams.cy), len(cams),
                _lib.ptr(b["origins"]), _lib.ptr(b["directions"]), None, None, None, s), "gf_generate_rays")
        return b

    def update(self, slot_indices: torch.Tensor, pred_rgb: torch.Tensor, gt_rgb: Optional[torch.Tensor] = None):
        """error_map[slot, y, x] = sum_c |gt - pred| (the arithmetic of `update_error_map`), then the sum tree above
        the written pixels is recomputed from the map.  `gt_rgb` defaults to the last batch's rgb, which is right when
        `slot_indices` are that batch's rows.  A pixel named twice holds one of its rows' errors.  Out-of-range rows
        are skipped and flagged for `check()`."""
        _lib.require_cuda(slot_indices, pred_rgb, gt_rgb)
        gt = self._batch["rgb"] if gt_rgb is None else gt_rgb.detach().float().contiguous()
        n = slot_indices.shape[0]
        if slot_indices.shape != (n, 3) or pred_rgb.shape != (n, 3) or gt.shape != (n, 3):
            raise RuntimeError("FocalBatchSource.update: slot_indices i64 [n,3], pred_rgb / gt_rgb f32 [n,3]")
        idx = slot_indices.to(torch.int64).contiguous()
        pred = pred_rgb.detach().float().contiguous()
        n_img, h, w = self.shape
        L = _lib.lib()
        with torch.cuda.device(self.device):
            s = _lib.cur_stream()
            _lib.check(L.gf_error_map_update(n, _lib.ptr(idx), _lib.ptr(pred), _lib.ptr(gt), n_img, h, w,
                                             _lib.ptr(self.error_map), None, _lib.ptr(self._err[1:]), s),
                       "gf_error_map_update")
            _lib.check(L.gf_sumtree_refresh(n, _lib.ptr(idx), n_img, h, w, _lib.ptr(self.error_map),
                                            _lib.ptr(self.sums), _lib.ptr(self.counts), s), "gf_sumtree_refresh")

    def check(self) -> None:
        """Raises what the draws and updates since the last check flagged (one device read), and clears the flags:
        RuntimeError for a draw error, IndexError for an out-of-range `update` row."""
        draw, bad_row = self._err.tolist()
        if not (draw or bad_row):
            return
        self._err.zero_()
        if draw:
            raise RuntimeError("FocalBatchSource: " + "; ".join(m for bit, m in self._ERRORS if draw & bit))
        raise IndexError("FocalBatchSource.update: row index out of range for the error map")
