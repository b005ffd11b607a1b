"""Hash3DAnchored: host-side mirror of the reference operator.

`Hash3DAnchoredCore` mirrors the C++ class behind `torch.classes.my_classes.Hash3DAnchored`
(reference gfnerf/bindings/field/Hash3DAnchored.cpp:17-200, bindings.cpp:300-357): same
constructor arguments, method names, state tensors and their order.
`Hash3DAnchored` mirrors the nn.Module shell (reference gfnerf/hash_3d_anchored.py:17-139).
The arithmetic runs in gf_hash_forward / gf_hash_backward of the C-ABI library; there is
no fallback.
"""
from typing import Any, Iterator, List, Mapping

import numpy as np
import torch
from torch import nn

from . import _lib

N_LEVELS = 16
N_CHANNELS = 2


def _is_prime_u32(x: np.ndarray) -> np.ndarray:
    """Deterministic Miller-Rabin (bases 2, 7, 61) for x < 2^32, vectorised.

    The reference uses trial division (Hash3DAnchored.cpp:32-37); the predicate is the same.
    """
    x = x.astype(np.uint64)
    res = np.ones(x.shape, bool)
    res &= (x > 3) & (x % 2 == 1)
    d = x - 1
    s = np.zeros_like(x)
    while True:
        even = (d % 2 == 0) & (d > 0)
        if not even.any():
            break
        d = np.where(even, d // 2, d)
        s = s + even.astype(np.uint64)
    for a in (2, 7, 61):
        # y = a^d mod x  (x < 2^30 here, so products fit in uint64)
        y = np.ones_like(x)
        base = np.full_like(x, a) % x
        e = d.copy()
        while (e > 0).any():
            odd = (e % 2 == 1)
            y = np.where(odd, (y * base) % x, y)
            base = (base * base) % x
            e = e // 2
        ok = (y == 1) | (y == x - 1)
        smax = int(s.max()) if s.size else 0
        for r in range(1, smax):
            y = (y * y) % x
            ok |= (y == x - 1) & (r < s)
        res &= ok | (x == a)
    return res


def draw_primes(count: int, generator: torch.Generator = None) -> torch.Tensor:
    """`count` random primes in [2^28, 2^30), the reference's rejection loop (Hash3DAnchored.cpp:39-52)."""
    lo, hi = 1 << 28, 1 << 30
    out = np.empty(0, np.int64)
    while out.size < count:
        need = count - out.size
        cand = torch.randint(lo, hi, (need * 24 + 64,), dtype=torch.int64, generator=generator).numpy()
        out = np.concatenate([out, cand[_is_prime_u32(cand)]])
    return torch.from_numpy(out[:count].astype(np.int32))


class _AnchoredQueryFn(torch.autograd.Function):
    """Hash3DAnchoredFunction (Hash3DAnchored_cuda.cu:160-239).

    Unlike the reference, the query points / anchors are saved on the autograd node, not on
    the encoder object, so two forwards before a backward do not corrupt each other.
    """

    @staticmethod
    def forward(ctx, feat_pool, core, points, anchors):
        _lib.require_cuda(feat_pool, points, anchors)
        n = points.shape[0]
        out = torch.empty((n, N_LEVELS * N_CHANNELS), dtype=torch.float32, device=points.device)
        core.launch_forward(points, anchors, out_f16=None, out_f32=out)
        ctx.core = core
        ctx.save_for_backward(points, anchors)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        core = ctx.core
        points, anchors = ctx.saved_tensors
        grad_table = torch.zeros((core.pool_size_, N_CHANNELS), dtype=torch.float32, device=points.device)
        core.launch_backward(points, anchors, grad_out.contiguous(), False, grad_table)
        return grad_table, None, None, None


class Hash3DAnchoredCore:
    """State + launches of one anchored hash grid (reference class Hash3DAnchored)."""

    def __init__(self, log2_table_size: int, n_volume: int, learn_rate: float = 1e-1, device=None,
                 generator: torch.Generator = None):
        if not torch.cuda.is_available():
            raise RuntimeError("Hash3DAnchored needs a CUDA device: the B200 kernels have no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.learn_rate_ = float(learn_rate)
        self.pool_size_ = (1 << int(log2_table_size)) * N_LEVELS
        self.n_volumes_ = int(n_volume)
        # Hash3DAnchored.cpp:26  (rand*.2 - 1) * 1e-4 ; Reset() overrides it in the field
        self.feat_pool_ = ((torch.rand((self.pool_size_, N_CHANNELS), device=self.device) * .2 - 1.) * 1e-4)
        self.feat_pool_.requires_grad_(True)
        self.prim_pool_ = draw_primes(3 * N_LEVELS * self.n_volumes_, generator).reshape(
            N_LEVELS, self.n_volumes_, 3).contiguous().to(self.device)
        # rand_bias is read uninitialised in the reference (Hash3DAnchored.h:55); treated as false
        self.bias_pool_ = torch.zeros((N_LEVELS * self.n_volumes_, 3), dtype=torch.float32, device=self.device)
        local_size = self.pool_size_ // N_LEVELS
        local_size = (local_size >> 4) << 4
        self.local_size_ = local_size
        self.feat_local_size_ = torch.full((N_LEVELS,), local_size, dtype=torch.int32, device=self.device)
        # Hash3DAnchored.cpp:66-70.  NB the reference's kernels add this offset to a pointer to SCALARS
        # (Hash3DAnchored_cuda.cu:38, :105), so level l's window starts at ROW l * local_size / 2: consecutive levels
        # overlap by half a window and only the first 8.5 * local_size rows of feat_pool are ever read or given a
        # gradient (csrc/hash_common.cuh level_base_row; pinned by tests/test_ref_kernels.py).
        self.feat_local_idx_ = (torch.cumsum(self.feat_local_size_, 0) - local_size).to(torch.int32)
        self.used_rows_ = (N_LEVELS - 1) * local_size // 2 + local_size
        self.level_scales_ = torch.empty(N_LEVELS, dtype=torch.float32, device=self.device)
        self.level_scales_host = np.zeros(N_LEVELS, np.float32)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().gf_hash_level_scales(_lib.ptr(self.level_scales_),
                                                       self.level_scales_host.ctypes.data, _lib.cur_stream()),
                       "gf_hash_level_scales")
        self._shadow = None       # fp16 copy of feat_pool_
        self._shadow_key = None   # (data_ptr, _version) the shadow was cast from

    # ---- launches -------------------------------------------------------
    def shadow(self, force: bool = False) -> torch.Tensor:
        """fp16 table.  The operator API re-casts on every forward like the reference (:185, 15 us at
        log2T=19); the fused engine owns the optimiser step, refreshes the shadow inside its Adam
        kernel and calls mark_shadow_fresh(), so it never pays for the cast."""
        fp = self.feat_pool_
        key = (fp.data_ptr(), fp._version)
        if force or self._shadow is None or self._shadow.shape != fp.shape or self._shadow_key != key:
            if self._shadow is None or self._shadow.shape != fp.shape:
                self._shadow = torch.empty(fp.shape, dtype=torch.float16, device=fp.device)
            _lib.check(_lib.lib().gf_hash_cast_table(_lib.ptr(fp.detach()), _lib.ptr(self._shadow), fp.numel(),
                                                     _lib.cur_stream()), "gf_hash_cast_table")
            self._shadow_key = key
        return self._shadow

    def mark_shadow_fresh(self):
        """Called by the fused Adam step, which writes the shadow itself."""
        self._shadow_key = (self.feat_pool_.data_ptr(), self.feat_pool_._version)

    def _bias(self):
        """bias_pool for the kernels: None (= zeros, no loads) while the pool is all zero, which it always is in the
        reference; checked once per pool (a host sync) and again after LoadStates"""
        key = (self.bias_pool_.data_ptr(), self.bias_pool_._version)
        if getattr(self, "_bias_key", None) != key:
            self._bias_zero = not bool(self.bias_pool_.any())
            self._bias_key = key
        return None if self._bias_zero else self.bias_pool_

    def launch_forward(self, points, anchors, out_f16=None, out_f32=None, d_n_ptr=None, recast=True):
        assert points.dtype == torch.float32 and points.is_contiguous()
        assert anchors.dtype in (torch.int64, torch.int32) and anchors.is_contiguous()
        with torch.cuda.device(points.device):
            _lib.check(_lib.lib().gf_hash_forward(
                points.shape[0], _lib.ptr(d_n_ptr), self.n_volumes_, self.local_size_,
                _lib.ptr(self.shadow(force=recast)),
                _lib.ptr(self.prim_pool_), _lib.ptr(self._bias()), _lib.ptr(self.level_scales_),
                _lib.ptr(points), _lib.ptr(anchors), int(anchors.dtype == torch.int64),
                _lib.ptr(out_f16), _lib.ptr(out_f32), _lib.cur_stream()), "gf_hash_forward")

    def launch_forward_residual(self, points, anchors, base_f16, out_f16=None, d_n_ptr=None, recast=True):
        """out_f16 = base_f16 + encode(points) (focal-stage residual, nerfacto_field.py:477-489); in place by default"""
        out_f16 = base_f16 if out_f16 is None else out_f16
        with torch.cuda.device(points.device):
            _lib.check(_lib.lib().gf_hash_forward_residual(
                points.shape[0], _lib.ptr(d_n_ptr), self.n_volumes_, self.local_size_,
                _lib.ptr(self.shadow(force=recast)), _lib.ptr(self.prim_pool_), _lib.ptr(self._bias()),
                _lib.ptr(self.level_scales_), _lib.ptr(points), _lib.ptr(anchors), int(anchors.dtype == torch.int64),
                _lib.ptr(base_f16), _lib.ptr(out_f16), _lib.cur_stream()), "gf_hash_forward_residual")

    @staticmethod
    def table_refs(cores, device, recast=True) -> torch.Tensor:
        """The gf_hash_table_ref array of `cores` on `device` (int64 [K, 3]: fp16 shadow, prime pool, bias pool or 0),
        for `launch_forward_residual_routed`.  The shadows are refreshed first (recast); the array holds their
        addresses, so it is valid until one of the tables is reallocated.  The bias-pool tests may read the host."""
        cores = list(cores)
        if not cores:
            raise ValueError("Hash3DAnchored routed gather: no tables")
        c0 = cores[0]
        for c in cores[1:]:
            if c.local_size_ != c0.local_size_ or c.n_volumes_ != c0.n_volumes_:
                raise ValueError(f"Hash3DAnchored routed gather: tables of local_size / n_volumes {c.local_size_} / "
                                 f"{c.n_volumes_} and {c0.local_size_} / {c0.n_volumes_}; all must agree")
        rows = [[c.shadow(force=recast).data_ptr(), c.prim_pool_.data_ptr(), _lib.ptr(c._bias()) or 0] for c in cores]
        # an ordinary host-to-device copy, ordered on the current stream
        return torch.tensor(rows, dtype=torch.int64).to(device, non_blocking=True)

    @staticmethod
    def launch_forward_residual_routed(cores, points, anchors, base_f16, ray_id, ray_table, out_f16=None, d_n_ptr=None,
                                       refs=None, recast=True):
        """out_f16 = base_f16 + cores[ray_table[ray_id[i]]].encode(points[i]) per sample, bit for bit what
        `launch_forward_residual` of that table computes; a table id outside [0, len(cores)) leaves the base row.
        ray_id int32 [n], ray_table int32 [n_rays] (device).  refs: `table_refs(cores, ...)` made once by a caller that
        launches many times (else built here, one host-to-device copy)."""
        out_f16 = base_f16 if out_f16 is None else out_f16
        assert ray_id.dtype == torch.int32 and ray_table.dtype == torch.int32
        if refs is None:
            refs = Hash3DAnchoredCore.table_refs(cores, points.device, recast=recast)
        c0 = cores[0]
        with torch.cuda.device(points.device):
            _lib.check(_lib.lib().gf_hash_forward_residual_routed(
                points.shape[0], _lib.ptr(d_n_ptr), c0.n_volumes_, c0.local_size_, len(cores), _lib.ptr(refs),
                _lib.ptr(c0.level_scales_), _lib.ptr(points), _lib.ptr(anchors), int(anchors.dtype == torch.int64),
                _lib.ptr(ray_id), _lib.ptr(ray_table), _lib.ptr(base_f16), _lib.ptr(out_f16), _lib.cur_stream()),
                "gf_hash_forward_residual_routed")

    @staticmethod
    def grad_refs(cores, grads, device) -> torch.Tensor:
        """The gf_hash_grad_ref array of `cores` on `device` (int64 [K, 3]: prime pool, bias pool or 0, gradient
        table), for `launch_backward_routed`.  grads[k]: fp32 [pool_size, 2] gradient table of cores[k].  It holds
        addresses: valid until a pool or gradient table is reallocated.  The bias-pool tests may read the host."""
        cores, grads = list(cores), list(grads)
        if not cores or len(cores) != len(grads):
            raise ValueError(f"Hash3DAnchored routed scatter: {len(cores)} tables and {len(grads)} gradient tables")
        c0 = cores[0]
        for c, g in zip(cores, grads):
            if c.local_size_ != c0.local_size_ or c.n_volumes_ != c0.n_volumes_:
                raise ValueError(f"Hash3DAnchored routed scatter: tables of local_size / n_volumes {c.local_size_} / "
                                 f"{c.n_volumes_} and {c0.local_size_} / {c0.n_volumes_}; all must agree")
            if g.dtype != torch.float32 or not g.is_contiguous() or g.numel() != c.pool_size_ * N_CHANNELS:
                raise ValueError("Hash3DAnchored routed scatter: each gradient table is a contiguous fp32 tensor of "
                                 "its table's size")
        rows = [[c.prim_pool_.data_ptr(), _lib.ptr(c._bias()) or 0, g.data_ptr()] for c, g in zip(cores, grads)]
        return torch.tensor(rows, dtype=torch.int64).to(device, non_blocking=True)

    @staticmethod
    def launch_backward_routed(cores, points, anchors, grad_in, grad_is_scaled_f16, ray_id, ray_table, grads=None,
                               refs=None, d_n_ptr=None, keep_x128=False):
        """`launch_backward` with one gradient table per sample: sample i accumulates into grads[ray_table[ray_id[i]]]
        with that table's pools, what `launch_backward` of cores[k] into grads[k] computes for it; a table id outside
        [0, len(cores)) contributes nothing.  refs: `grad_refs(cores, grads, ...)` made once by a caller that launches
        many times (else built here from `grads`, one host-to-device copy)."""
        assert ray_id.dtype == torch.int32 and ray_table.dtype == torch.int32
        if refs is None:
            refs = Hash3DAnchoredCore.grad_refs(cores, grads, points.device)
        c0 = cores[0]
        with torch.cuda.device(points.device):
            _lib.check(_lib.lib().gf_hash_backward_routed(
                points.shape[0], _lib.ptr(d_n_ptr), c0.n_volumes_, c0.local_size_, len(cores), _lib.ptr(refs),
                _lib.ptr(c0.level_scales_), _lib.ptr(points), _lib.ptr(anchors), int(anchors.dtype == torch.int64),
                _lib.ptr(ray_id), _lib.ptr(ray_table), _lib.ptr(grad_in),
                int(bool(grad_is_scaled_f16)) | (2 if keep_x128 else 0), _lib.cur_stream()), "gf_hash_backward_routed")

    def launch_backward(self, points, anchors, grad_in, grad_is_scaled_f16, grad_table, d_n_ptr=None,
                        keep_x128=False, levels=(0, 16)):
        """keep_x128: leave grad_table at the reference's x128 gradient scale (Hash3DAnchored_cuda.cu:209) for a
        caller that divides in its optimizer step (the fused engine: `_Adam.grad_scale`)."""
        with torch.cuda.device(points.device):
            _lib.check(_lib.lib().gf_hash_backward_levels(
                points.shape[0], _lib.ptr(d_n_ptr), self.n_volumes_, self.local_size_, _lib.ptr(self.prim_pool_),
                _lib.ptr(self._bias()), _lib.ptr(self.level_scales_), _lib.ptr(points), _lib.ptr(anchors),
                int(anchors.dtype == torch.int64), _lib.ptr(grad_in), int(bool(grad_is_scaled_f16)) | (2 if keep_x128 else 0),
                _lib.ptr(grad_table), int(levels[0]), int(levels[1]), _lib.cur_stream()), "gf_hash_backward")

    # ---- reference method surface (bindings.cpp:300-357) ----------------
    def AnchoredQuery(self, points: torch.Tensor, anchors: torch.Tensor) -> torch.Tensor:
        points = points.contiguous()
        anchors = anchors.contiguous()
        if self.feat_pool_.requires_grad and torch.is_grad_enabled():
            return _AnchoredQueryFn.apply(self.feat_pool_, self, points, anchors)
        _lib.require_cuda(points, anchors)
        out = torch.empty((points.shape[0], N_LEVELS * N_CHANNELS), dtype=torch.float32, device=points.device)
        self.launch_forward(points, anchors, out_f32=out)
        return out

    def GetParams(self) -> List[torch.Tensor]:
        return [self.feat_pool_]

    def States(self) -> List[torch.Tensor]:
        return [self.feat_pool_.data, self.prim_pool_.data, self.bias_pool_.data,
                torch.full((1,), self.n_volumes_, dtype=torch.int32)]

    def LoadStates(self, states: List[torch.Tensor], idx: int) -> int:
        self.feat_pool_.data.copy_(states[idx]); idx += 1
        self.prim_pool_ = states[idx].clone().to(self.device).contiguous(); idx += 1   # the size may change
        bias = states[idx]; idx += 1
        if tuple(bias.shape) == tuple(self.bias_pool_.shape):
            self.bias_pool_.data.copy_(bias)
        else:
            # a checkpoint written with another n_volumes: the reference's `bias_pool_.data().copy_()` (:116) throws
            # here although it lets prim_pool change size one line above; the pool follows the checkpoint instead
            self.bias_pool_ = bias.detach().clone().to(self.device, torch.float32).contiguous()
        self.n_volumes_ = int(states[idx].item()); idx += 1
        if (tuple(self.prim_pool_.shape) != (N_LEVELS, self.n_volumes_, 3)
                or tuple(self.bias_pool_.shape) != (N_LEVELS * self.n_volumes_, 3)):
            raise ValueError(f"Hash3DAnchored.LoadStates: prime pool {tuple(self.prim_pool_.shape)} / bias pool "
                             f"{tuple(self.bias_pool_.shape)} do not belong to n_volumes = {self.n_volumes_}")
        # `.data.copy_()` does not bump `_version`: drop both cached decisions (fp16 shadow, all-zero bias) by hand
        self._shadow_key = None
        self._bias_key = None
        return idx

    def Reset(self, generator: torch.Generator = None) -> None:
        """U(-0.01, 0.01) (Hash3DAnchored.cpp Reset).  `generator` (a CPU generator) makes the table reproducible
        from a seed -- the draw then happens on the host and is copied; without it the device's global RNG is used
        like the reference does."""
        if generator is None:
            self.feat_pool_.data.uniform_(-1e-2, 1e-2)
        else:
            host = torch.empty(self.feat_pool_.shape, dtype=torch.float32).uniform_(-1e-2, 1e-2, generator=generator)
            self.feat_pool_.data.copy_(host)
        self._shadow_key = None

    def Zero(self) -> None:
        self.feat_pool_.data.zero_()
        self._shadow_key = None

    def SetFeatPoolRequireGrad(self, require_grad: bool) -> None:
        self.feat_pool_.requires_grad_(require_grad)

    def to(self, device: str) -> None:
        # Hash3DAnchored.cpp:180-200: "cpu" parks the table on the host, anything else is cuda
        if device == "cpu":
            self.feat_pool_ = self.feat_pool_.to("cpu")
        else:
            self.feat_pool_ = self.feat_pool_.to(self.device)
        self._shadow_key = None

    def ReleaseResources(self) -> None:
        empty = torch.empty(0, dtype=torch.float32)
        self.feat_pool_ = empty
        self.prim_pool_ = empty
        self.bias_pool_ = empty
        self._shadow = None
        self._shadow_key = None
        torch.cuda.empty_cache()


class Hash3DAnchored(nn.Module):
    """Drop-in for reference gfnerf/hash_3d_anchored.py:17-139 (same methods, same state-dict keys)."""

    def __init__(self, log2_table_size: int, n_volumes: int, generator: torch.Generator = None) -> None:
        super().__init__()
        self.hash_3d = Hash3DAnchoredCore(log2_table_size, n_volumes, 1e-1, generator=generator)
        self.register_parameter("feat_pool", None)
        self.register_buffer("prime_pool", None)
        self.register_buffer("bias_pool", None)
        self.register_buffer("n_volumes", None)
        self.hook_handles = [self._register_state_dict_hook(self.state_dict_hook)]

    def unregister_hooks(self):
        for h in self.hook_handles:
            h.remove()

    def state_dict_hook(self, *args):
        destination, prefix = args[1], args[2]
        feat_pool_, prime_pool_, bias_pool_, n_volume_ = self.states()
        destination[prefix + "feat_pool"] = feat_pool_
        destination[prefix + "prime_pool"] = prime_pool_
        destination[prefix + "bias_pool"] = bias_pool_
        destination[prefix + "n_volumes"] = n_volume_
        return destination

    def forward(self, input):
        points, anchors = input
        assert len(anchors.shape) == 1
        assert points.shape[1] == 3
        assert len(points.shape) == 2
        assert anchors.dtype == torch.int64
        return self.anchored_query(points, anchors)

    def parameters(self, recurse: bool = True) -> Iterator[nn.Parameter]:
        for p in self.hash_3d.GetParams():
            yield p

    def anchored_query(self, points, anchors):
        return self.hash_3d.AnchoredQuery(points, anchors)

    def load_state_dict(self, state_dict: Mapping[str, Any], strict: bool = True, prefix=''):
        pre = "" if prefix == '' else f"{prefix}."
        keys = [pre + k for k in ("feat_pool", "prime_pool", "bias_pool", "n_volumes")]
        states = [state_dict[k] for k in keys]
        for k in keys:
            del state_dict[k]
        self.load_states(states, idx=0)
        return None

    def set_require_grad(self, require_grad):
        assert type(require_grad) == bool
        self.hash_3d.SetFeatPoolRequireGrad(require_grad)

    def to(self, device):
        assert type(device) == str
        self.hash_3d.to(device)

    def load_states(self, states, idx: int) -> int:
        return self.hash_3d.LoadStates(states, idx)

    def states(self):
        return self.hash_3d.States()

    def get_params(self):
        return self.hash_3d.GetParams()

    def reset(self) -> None:
        self.hash_3d.Reset()

    def zero(self) -> None:
        self.hash_3d.Zero()

    def release_resources(self) -> None:
        self.hash_3d.ReleaseResources()
