"""gf_composite_forward / gf_composite_backward, gf_s3im and gf_charbonnier against float64 torch restatements of the
reference (nerfstudio/cameras/rays.py:178-200 get_weights_f2nerf; model_components/renderers.py:97-110, 220, 269-283;
model_components/losses.py:73-84 CharbonnierLoss, 713-794 S3IM and its SSIM) where the kernels can go wrong: opaque
samples (delta * sigma up to +inf) at every position of a 32-sample chunk, NaN densities, empty and transparent rays,
the chunk boundaries, more rays than one grid wave, every optional pointer; overlapping, partial and repeated S3IM
windows; the Charbonnier grid-stride loop.

Compositing tolerance.  The kernels keep every sum in fp32, so they are held to what fp32 attains, not to a flat rtol.
With u = 2^-24 and excl the exclusive prefix sum of delta * sigma in front of a sample,
    |dT| <= C u (1 + excl) T + FLOOR,   |d alpha| <= C u,   |dw| <= |d alpha| T + alpha |dT| + FLOOR,
and the bounds of the renderers' sums and of the gradients follow from these by the triangle inequality (`bounds`).
C = 64 covers the depth of the chunked scan (5 shuffle levels plus one carry addition per chunk: 37 for a 1024-sample
ray) and the roundings of exp and the products.  The reference's formula evaluated in fp32 torch meets the same bounds
(`test_fp32_reference_meets_the_bound`).  An exclusive prefix taken as (inclusive - own term) does not: at an opaque
sample it loses the earlier sum to ulp(delta * sigma), and at delta * sigma = inf it is NaN.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import oracle as orc
from tests.test_composite_gpu import ragged

U = 2.0 ** -24
C = 64
FLOOR = 1e-30
SURFACE_DD = (10.0, 1e2, 1e3, 1e4, 1e6, math.inf)
SURFACE_AT = (0, 1, 31, 32, 1023)          # lanes 0, 1, 31 of the first chunk, lane 0 of the second, the last of 1024
CHUNK_LENGTHS = (1, 2, 31, 32, 33, 63, 64, 65, 1023, 1024)
FWD_OUTPUTS = ("weights", "alphas", "trans", "rgb", "depth", "acc", "tmax")

gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ fixtures
def _smooth(rng, n):
    """sigma, delta, rgb of ordinary samples (delta * sigma mostly well below 1)"""
    return np.exp(rng.normal(0, 2, size=n)), rng.uniform(1e-3, 5e-2, size=n), rng.rand(n, 3)


def _pack(rays):
    """[(sigma, delta, rgb)] per ray -> CSR offsets and float32 samples; t = 0.1 + the running sum of delta"""
    counts = np.array([len(r[0]) for r in rays], np.int64)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    cat = lambda i, shape: (np.concatenate([r[i] for r in rays]) if counts.sum() else np.zeros(shape))
    t = [0.1 + np.cumsum(r[1]) for r in rays]
    return dict(offsets=offsets, sigma=cat(0, (0,)).astype(np.float32), delta=cat(1, (0,)).astype(np.float32),
                rgb=cat(2, (0, 3)).astype(np.float32).reshape(-1, 3),
                t=(np.concatenate(t) if counts.sum() else np.zeros(0)).astype(np.float32))


def surface_rays(dds=SURFACE_DD, repeats=3, seed=0):
    """Rays with one opaque sample of delta * sigma = dd at position `at`, behind a prefix sum of 0.5 - 5 (none at
    position 0) and followed by 0 - 69 ordinary samples (none after position 1023 of a 1024-sample ray).
    -> (batch, [(ray, at, dd)])"""
    rng = np.random.RandomState(seed)
    rays, where = [], []
    for dd in dds:
        for at in SURFACE_AT:
            for _ in range(repeats):
                n = 1024 if at == 1023 else at + 1 + rng.randint(0, 70)
                sigma, delta, rgb = _smooth(rng, n)
                if at > 0:
                    share = rng.rand(at) + 0.05
                    sigma[:at] = rng.uniform(0.5, 5.0) * share / share.sum() / delta[:at]
                sigma[at] = dd / delta[at]
                where.append((len(rays), at, dd))
                rays.append((sigma, delta, rgb))
    return _pack(rays), where


def chunk_rays(seed=1):
    """three rays of every length in CHUNK_LENGTHS: thin, medium and dense media"""
    rng = np.random.RandomState(seed)
    rays = []
    for n in CHUNK_LENGTHS:
        for scale in (1e-3, 1.0, 30.0):
            sigma, delta, rgb = _smooth(rng, n)
            rays.append((sigma * scale, delta, rgb))
    return _pack(rays)


def degenerate_rays(seed=2):
    """empty rays first, in the middle and last; sigma = 0 rays; delta = 0 samples among ordinary ones"""
    rng = np.random.RandomState(seed)
    empty = (np.zeros(0), np.zeros(0), np.zeros((0, 3)))
    rays = [empty, empty]
    for n in (1, 5, 40):
        _, delta, rgb = _smooth(rng, n)
        rays.append((np.zeros(n), delta, rgb))                 # transparent: acc 0, depth 0
    rays.append(empty)
    for n in (3, 37, 70):
        sigma, delta, rgb = _smooth(rng, n)
        delta[rng.rand(n) < 0.3] = 0.0
        delta[0] = 0.0
        rays.append((sigma * 20, delta, rgb))
    rays += [empty, empty]
    return _pack(rays)


def nan_rays(seed=3):
    """a NaN density at sample 0, 5 and 33 of three rays, ordinary rays around them -> (batch, NaN rays)"""
    rng = np.random.RandomState(seed)
    rays, bad = [], []
    for at in (None, 0, None, 5, 33, None):
        sigma, delta, rgb = _smooth(rng, 50)
        if at is not None:
            sigma[at] = np.nan
            bad.append(len(rays))
        rays.append((sigma, delta, rgb))
    return _pack(rays), bad


def ragged_batch(R, max_len, seed):
    offsets, sigma, delta, rgb, t = ragged(R, max_len, seed)
    return dict(offsets=offsets, sigma=sigma, delta=delta, rgb=rgb, t=t)


def grads_for(b, seed, which=("g_rgb", "g_acc")):
    rng = np.random.RandomState(seed)
    R, V = b["offsets"].shape[0] - 1, b["sigma"].shape[0]
    shapes = dict(g_rgb=(R, 3), g_acc=(R,), g_w=(V,))
    return {k: rng.normal(size=shapes[k]).astype(np.float32) for k in which}


# ------------------------------------------------------------------------------------------------ reference
def reference(b, g_rgb=None, g_acc=None, g_w=None, dtype=torch.float64, device="cpu"):
    """get_weights_f2nerf + RGB / expected-depth / accumulation renderers on the dense [R, S] layout the reference
    uses (padding: delta 0, t 0), and autograd of sum(out_rgb g_rgb) + sum(acc g_acc) + sum(weights g_w).
    Per-sample outputs come back in CSR order; also `excl`, the exclusive prefix sum of delta * sigma."""
    offsets = b["offsets"]
    counts = np.diff(offsets)
    R, S = counts.shape[0], max(int(counts.max(initial=0)), 1)
    idx = torch.from_numpy(np.flatnonzero(np.arange(S)[None, :] < counts[:, None])).to(device)
    f = lambda a: torch.from_numpy(np.asarray(a)).to(device, dtype)
    sg = f(b["sigma"]).requires_grad_()
    cl = f(b["rgb"]).requires_grad_()
    dense = lambda v: torch.zeros((R * S,) + tuple(v.shape[1:]), dtype=dtype, device=device).index_copy(
        0, idx, v).view((R, S) + tuple(v.shape[1:]))
    dd = dense(f(b["delta"])) * dense(sg)                                   # rays.py:188-200
    alphas = 1 - torch.exp(-dd)
    excl = torch.cat([torch.zeros((R, 1), dtype=dtype, device=device), torch.cumsum(dd[:, :-1], dim=1)], dim=1)
    trans = torch.exp(-excl)
    w = torch.nan_to_num(alphas * trans)
    out_rgb = (w[..., None] * dense(cl)).sum(1)                             # renderers.py:97-110
    acc = w.sum(1)                                                          # :220
    depth = (w * dense(f(b["t"]))).sum(1) / (acc + 1e-10)                   # :269-280, before the clip
    flat = lambda x: x.reshape(-1)[idx]
    out = dict(weights=flat(w), alphas=flat(alphas), trans=flat(trans), excl=flat(excl), rgb=out_rgb, depth=depth,
               acc=acc)
    terms = []
    if g_rgb is not None:
        terms.append((out_rgb * f(g_rgb)).sum())
    if g_acc is not None:
        terms.append((acc * f(g_acc)).sum())
    if g_w is not None:
        terms.append((flat(w) * f(g_w)).sum())
    if terms:
        sum(terms).backward()
        out["d_sigma"], out["d_rgb"] = sg.grad, cl.grad
    return {k: v.detach().cpu().double() for k, v in out.items() if v is not None}


def _ray_ids(offsets):
    return torch.from_numpy(np.repeat(np.arange(offsets.shape[0] - 1), np.diff(offsets)))


def _suffix_excl(offsets, v):
    """per sample, the sum of v over the later samples of its ray"""
    counts = np.diff(offsets)
    R, S = counts.shape[0], max(int(counts.max(initial=0)), 1)
    idx = torch.from_numpy(np.flatnonzero(np.arange(S)[None, :] < counts[:, None]))
    d = torch.zeros(R * S, dtype=v.dtype).index_copy(0, idx, v).view(R, S)
    incl = d.flip(1).cumsum(1).flip(1)
    return torch.cat([incl[:, 1:], torch.zeros((R, 1), dtype=v.dtype)], dim=1).reshape(-1)[idx]


def bounds(b, ref, g_rgb=None, g_acc=None, g_w=None):
    """|fp32 value - float64 value| bounds of every output of `reference` (module docstring); NaN-free"""
    nz = lambda x: torch.nan_to_num(x, nan=0.0)
    T, a, w, excl = nz(ref["trans"]), nz(ref["alphas"]), nz(ref["weights"]), ref["excl"]
    offsets = b["offsets"]
    R, rid = offsets.shape[0] - 1, _ray_ids(offsets)
    seg = lambda v: torch.zeros((R,) + tuple(v.shape[1:]), dtype=torch.float64).index_add_(0, rid, v)
    c = torch.from_numpy(b["rgb"]).double().abs()
    t = torch.from_numpy(b["t"]).double().abs()
    bT = C * U * torch.where(T > 0, (1 + excl) * T, 0.0) + FLOOR
    bA = torch.full_like(T, C * U)
    bW = bA * T + a * bT + FLOOR
    out = dict(trans=bT, alphas=bA, weights=bW)
    out["rgb"] = seg(bW[:, None] * c) + C * U * seg(w[:, None] * c) + FLOOR
    out["acc"] = seg(bW) + C * U * seg(w) + FLOOR
    den = ref["acc"] + 1e-10
    out["depth"] = (seg(bW * t) + C * U * seg(w * t)) / den + ref["depth"].abs() * out["acc"] / den \
        + C * U * ref["depth"].abs() + FLOOR
    if g_rgb is None and g_acc is None and g_w is None:
        return out
    # d_sigma_i = (gw_i e_i T_i - sum_{j>i} gw_j w_j) delta_i,  gw_i = g_rgb . c_i + g_acc + g_w_i,  e_i = exp(-dd_i)
    G = torch.zeros_like(T)
    if g_rgb is not None:
        G += (torch.from_numpy(g_rgb).double().abs()[rid] * c).sum(1)
    if g_acc is not None:
        G += torch.from_numpy(g_acc).double().abs()[rid]
    if g_w is not None:
        G += torch.from_numpy(g_w).double().abs()
    delta = torch.from_numpy(b["delta"]).double()
    dd = nz(delta * torch.from_numpy(b["sigma"]).double())
    e = torch.exp(-dd)
    bE = C * U * torch.where(e > 0, (1 + dd) * e, 0.0)
    out["d_sigma"] = delta * (G * (bE * T + e * bT + C * U * e * T) + _suffix_excl(offsets, G * (bW + C * U * w))) \
        + FLOOR
    if g_rgb is not None:
        out["d_rgb"] = (bW + C * U * w)[:, None] * torch.from_numpy(g_rgb).double().abs()[rid] + FLOOR
    return out


def close(name, got, want, bound):
    """NaN exactly where the reference has NaN; elsewhere equal (inf) or within the bound"""
    got = got.detach().double().cpu().reshape(want.shape)
    assert torch.equal(torch.isnan(got), torch.isnan(want)), \
        f"{name}: NaN at {torch.isnan(got).nonzero()[:8].tolist()}, reference NaN at {torch.isnan(want).nonzero()[:8].tolist()}"
    err = torch.where(torch.isnan(want) | (got == want), 0.0, (got - want).abs())
    bad = ~(err <= bound)
    if bad.any():
        ratio = torch.where(bad, err / bound, 0.0)
        i = int(torch.argmax(ratio.reshape(-1)))
        raise AssertionError(f"{name}: {int(bad.sum())} of {bad.numel()} values outside the fp32 bound; worst at "
                             f"{np.unravel_index(i, tuple(bad.shape))}: got {got.reshape(-1)[i].item()!r}, reference "
                             f"{want.reshape(-1)[i].item()!r}, bound {bound.reshape(-1)[i].item():.3g}")


# ------------------------------------------------------------------------------------------------ kernel calls
def _dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_forward(b, outs=FWD_OUTPUTS, tmax0=0.0, t=None):
    """gf_composite_forward; outputs not in `outs` are NULL, the others start as NaN (tmax as tmax0)"""
    from gfnerf_b200 import _lib
    R, V = b["offsets"].shape[0] - 1, b["sigma"].shape[0]
    shapes = dict(weights=(V,), alphas=(V,), trans=(V,), rgb=(R, 3), depth=(R,), acc=(R,), tmax=(1,))
    o = {k: torch.full(shapes[k], tmax0 if k == "tmax" else math.nan, device="cuda") for k in outs}
    P = lambda k: _lib.ptr(o.get(k))
    dv = {k: _dev(b[k]) for k in ("offsets", "sigma", "delta", "rgb")}
    tt = _dev(b["t"] if t is None else t)
    _lib.check(_lib.lib().gf_composite_forward(R, _lib.ptr(dv["offsets"]), _lib.ptr(dv["sigma"]),
                                               _lib.ptr(dv["delta"]), _lib.ptr(dv["rgb"]), _lib.ptr(tt), P("weights"),
                                               P("alphas"), P("trans"), P("rgb"), P("depth"), P("acc"), P("tmax"),
                                               _lib.cur_stream()), "gf_composite_forward")
    torch.cuda.synchronize()
    return o


def run_backward(b, trans, g_rgb=None, g_acc=None, g_w=None, want_d_rgb=True):
    """gf_composite_backward with the given gradients (rgb passed exactly when g_rgb is) -> (d_sigma, d_rgb)"""
    from gfnerf_b200 import _lib
    R, V = b["offsets"].shape[0] - 1, b["sigma"].shape[0]
    d_sigma = torch.full((V,), math.nan, device="cuda")
    d_rgb = torch.full((V, 3), math.nan, device="cuda") if (want_d_rgb and g_rgb is not None) else None
    dv = {k: _dev(b[k]) for k in ("offsets", "sigma", "delta")}
    rgb = _dev(b["rgb"]) if g_rgb is not None else None
    g = [_dev(x) for x in (g_rgb, g_acc, g_w)]
    _lib.check(_lib.lib().gf_composite_backward(R, _lib.ptr(dv["offsets"]), _lib.ptr(dv["sigma"]),
                                                _lib.ptr(dv["delta"]), _lib.ptr(rgb), _lib.ptr(trans),
                                                *[_lib.ptr(x) for x in g], _lib.ptr(d_sigma), _lib.ptr(d_rgb),
                                                _lib.cur_stream()), "gf_composite_backward")
    torch.cuda.synchronize()
    return d_sigma, d_rgb


def check_forward(b, got, ref=None, bnd=None):
    ref = reference(b) if ref is None else ref
    bnd = bounds(b, ref) if bnd is None else bnd
    for k in ("weights", "alphas", "trans", "rgb", "depth", "acc"):
        close(k, got[k], ref[k], bnd[k])
    return ref


def check_backward(b, trans, **g):
    ref = reference(b, **g)
    bnd = bounds(b, ref, **g)
    d_sigma, d_rgb = run_backward(b, trans, **g)
    close("d_sigma", d_sigma, ref["d_sigma"], bnd["d_sigma"])
    if g.get("g_rgb") is not None:
        close("d_rgb", d_rgb, ref["d_rgb"], bnd["d_rgb"])
    return d_sigma


# ------------------------------------------------------------------------------------------------ compositing
@gpu
@pytest.mark.parametrize("dd", SURFACE_DD)
def test_opaque_surface(dd):
    b, _ = surface_rays(dds=(dd,))
    got = run_forward(b)
    check_forward(b, got)
    g = grads_for(b, 5)
    check_backward(b, got["trans"], g_rgb=g["g_rgb"])
    check_backward(b, got["trans"], g_acc=g["g_acc"])


@gpu
def test_infinite_density():
    """sigma = inf: alpha 1 and weight T_i at the sample, T 0 behind it, finite gradients equal to autograd's"""
    b, where = surface_rays(dds=(math.inf,))
    got = run_forward(b)
    ref = check_forward(b, got)
    assert torch.isfinite(got["trans"]).all()
    s = torch.tensor([int(b["offsets"][ray]) + at for ray, at, _ in where])
    assert torch.equal(got["alphas"].cpu()[s], torch.ones(len(s)))
    assert torch.equal(got["weights"].cpu()[s], got["trans"].cpu()[s])
    close("weight = T_i", got["weights"].cpu()[s], ref["trans"][s], bounds(b, ref)["trans"][s])
    g = grads_for(b, 6, ("g_rgb", "g_acc", "g_w"))
    d_sigma = check_backward(b, got["trans"], **g)
    assert torch.isfinite(d_sigma).all()


@gpu
def test_nan_density():
    """NaN where the reference has NaN (alpha at the sample, T behind it), weight 0 from the sample on; the ray's
    d_sigma holds a NaN (so the NaN-gradient guard skips the step, as it does in torch); other rays unaffected"""
    b, bad = nan_rays()
    got = run_forward(b)
    ref = check_forward(b, got)
    offsets = b["offsets"]
    for ray in bad:
        w = got["weights"].cpu()[offsets[ray]:offsets[ray + 1]]
        first = int(torch.isnan(ref["alphas"][offsets[ray]:offsets[ray + 1]]).nonzero()[0])
        assert torch.all(w[first:] == 0)
    g = grads_for(b, 7)
    ref = reference(b, **g)
    d_sigma, _ = run_backward(b, got["trans"], **g)
    d_sigma = d_sigma.cpu().double()
    good = np.ones(len(offsets) - 1, bool)
    good[bad] = False
    keep = torch.from_numpy(good[_ray_ids(offsets).numpy()])
    for ray in bad:
        assert torch.isnan(d_sigma[offsets[ray]:offsets[ray + 1]]).any()
        assert torch.isnan(ref["d_sigma"][offsets[ray]:offsets[ray + 1]]).any()
    bnd = bounds(b, ref, **g)
    close("d_sigma (rays without NaN)", d_sigma[keep], ref["d_sigma"][keep], bnd["d_sigma"][keep])


@gpu
def test_transparent_and_degenerate_rays():
    b = degenerate_rays()
    got = run_forward(b)
    check_forward(b, got)
    counts = np.diff(b["offsets"])
    R = counts.shape[0]
    empty = torch.from_numpy(counts == 0)
    assert torch.equal(got["rgb"].cpu()[empty], torch.zeros(int(empty.sum()), 3))
    for k in ("depth", "acc"):
        assert torch.equal(got[k].cpu()[empty], torch.zeros(int(empty.sum()))), k
    transparent = [r for r in range(R) if counts[r] and not b["sigma"][b["offsets"][r]:b["offsets"][r + 1]].any()]
    assert len(transparent) == 3
    for k in ("acc", "depth"):
        assert torch.equal(got[k].cpu()[transparent], torch.zeros(3)), k
    zero_delta = torch.from_numpy(b["delta"] == 0)
    assert torch.equal(got["weights"].cpu()[zero_delta], torch.zeros(int(zero_delta.sum())))
    g = grads_for(b, 8, ("g_rgb", "g_acc", "g_w"))
    d_sigma = check_backward(b, got["trans"], **g)
    assert torch.equal(d_sigma.cpu()[zero_delta], torch.zeros(int(zero_delta.sum())))


@gpu
def test_chunk_boundaries():
    b = chunk_rays()
    got = run_forward(b)
    check_forward(b, got)
    check_backward(b, got["trans"], **grads_for(b, 9, ("g_rgb", "g_acc", "g_w")))


@gpu
def test_more_rays_than_one_grid_wave():
    """The grid holds SMs x 16 CTAs of 8 warps; every warp also serves rays n_warps, 2 n_warps, ... later"""
    n_warps = torch.cuda.get_device_properties(0).multi_processor_count * 16 * 8
    R = int(2.5 * n_warps) + 17
    rng = np.random.RandomState(10)
    rays = [_smooth(rng, n) for n in rng.randint(0, 41, size=R)]
    b = _pack(rays)
    far = n_warps + 5                                  # a ray of a warp's second pass, with samples
    while b["offsets"][far + 1] == b["offsets"][far]:
        far += 1
    b["t"][b["offsets"][far + 1] - 1] = 1000.0
    got = run_forward(b)
    check_forward(b, got)
    assert float(got["tmax"]) == 1000.0 == b["t"].max()
    assert float(run_forward(b, tmax0=2000.0)["tmax"]) == 2000.0       # a larger preset value is kept
    zeros = np.zeros_like(b["t"])
    assert float(run_forward(b, tmax0=0.0, t=zeros)["tmax"]) == 0.0   # t all 0: d_tmax untouched
    assert float(run_forward(b, tmax0=0.5, t=zeros)["tmax"]) == 0.5
    check_backward(b, got["trans"], **grads_for(b, 11, ("g_rgb", "g_acc")))


@gpu
@pytest.mark.parametrize("null", FWD_OUTPUTS)
def test_forward_null_output_leaves_the_others_bit_identical(null):
    b = ragged_batch(500, 200, 12)
    full = run_forward(b)
    part = run_forward(b, outs=tuple(k for k in FWD_OUTPUTS if k != null))
    for k, v in part.items():
        assert torch.equal(v, full[k]), k


@gpu
@pytest.mark.parametrize("which", [("g_rgb",), ("g_acc",), ("g_w",), ("g_rgb", "g_acc"), ("g_rgb", "g_w"),
                                   ("g_acc", "g_w"), ("g_rgb", "g_acc", "g_w")])
def test_backward_every_gradient_subset(which):
    b = ragged_batch(300, 150, 13)
    got = run_forward(b)
    g = grads_for(b, 14, which)
    d_sigma = check_backward(b, got["trans"], **g)
    if "g_rgb" in which:            # d_rgb = NULL gives the same d_sigma bit for bit
        assert torch.equal(run_backward(b, got["trans"], want_d_rgb=False, **g)[0], d_sigma)


def test_backward_rejects_colour_gradient_without_colours():
    """argument checks run before any CUDA call (no GPU needed); the pointers are never dereferenced"""
    from gfnerf_b200 import _lib
    L = _lib.lib()
    p = 256
    # g_rgb without rgb would silently drop the colour gradient
    assert L.gf_composite_backward(1, p, p, p, None, p, p, None, None, p, None, None) == -1
    assert b"g_rgb without rgb" in L.gf_last_error()
    assert L.gf_composite_backward(1, p, p, p, p, p, None, p, None, p, p, None) == -1     # d_rgb without g_rgb
    assert b"d_rgb needs" in L.gf_last_error()


@gpu
def test_fp32_reference_meets_the_bound():
    """the bounds are ones the reference's own formula attains in fp32 torch on the GPU (forward and autograd)"""
    for b in (surface_rays(dds=SURFACE_DD, repeats=1)[0], chunk_rays(), degenerate_rays(), ragged_batch(300, 1024, 0)):
        g = grads_for(b, 15, ("g_rgb", "g_acc", "g_w"))
        ref = reference(b, **g)
        r32 = reference(b, dtype=torch.float32, device="cuda", **g)
        bnd = bounds(b, ref, **g)
        for k in ("weights", "alphas", "trans", "rgb", "depth", "acc", "d_sigma", "d_rgb"):
            close(f"fp32 torch {k}", r32[k], ref[k], bnd[k])


def test_reference_restatement_matches_oracle():
    """CPU: the float64 restatement against the C oracle (fp64 prefix sums, rays.py / renderers.py) on ragged data,
    within the same bounds; and the fixtures hold every placement the GPU tests rely on"""
    b = ragged_batch(200, 1024, 0)
    g = grads_for(b, 16)
    ref = reference(b, **g)
    bnd = bounds(b, ref, **g)
    o = orc.composite_forward(b["offsets"], b["sigma"], b["delta"], b["rgb"], b["t"])
    for k in ("weights", "alphas", "trans", "rgb", "depth", "acc"):
        close(f"oracle {k}", torch.from_numpy(o[k]), ref[k], bnd[k])
    d_sigma, d_rgb = orc.composite_backward(b["offsets"], b["sigma"], b["delta"], b["rgb"], g["g_rgb"], g["g_acc"])
    close("oracle d_sigma", torch.from_numpy(d_sigma), ref["d_sigma"], bnd["d_sigma"])
    close("oracle d_rgb", torch.from_numpy(d_rgb), ref["d_rgb"], bnd["d_rgb"])

    b, where = surface_rays()
    dd = b["delta"].astype(np.float64) * b["sigma"].astype(np.float64)
    seen = set()
    for ray, at, want in where:
        s0 = int(b["offsets"][ray])
        assert b["offsets"][ray + 1] - s0 > at
        got = dd[s0 + at]
        assert got == want if math.isinf(want) else abs(got - want) <= 1e-6 * want
        assert at == 0 or 0.5 - 1e-5 <= dd[s0:s0 + at].sum() <= 5 + 1e-5
        seen.add((at, want))
    assert seen == {(at, x) for at in SURFACE_AT for x in SURFACE_DD}
    assert {int(b["offsets"][r + 1] - b["offsets"][r]) for r, at, _ in where if at == 1023} == {1024}
    counts = np.diff(chunk_rays()["offsets"])
    assert sorted(set(counts.tolist())) == list(CHUNK_LENGTHS)
    counts = np.diff(degenerate_rays()["offsets"])
    assert counts[0] == 0 and counts[-1] == 0 and (counts[1:-1] == 0).any()
    assert (degenerate_rays()["delta"] == 0).any()


# ------------------------------------------------------------------------------------------------ S3IM
def s3im_window(ksize):
    """the reference's window (losses.py:726-734): fp32 Gaussian, sigma 1.5, normalised in fp32, outer product"""
    g = torch.tensor([math.exp(-(x - ksize // 2) ** 2 / float(2 * 1.5 ** 2)) for x in range(ksize)],
                     dtype=torch.float32)
    g = g / g.sum()
    return (g[:, None] @ g[None, :]).double()


def _ssim_map(mu1, mu2, e11, e22, e12):
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    s11, s22, s12 = e11 - mu1 * mu1, e22 - mu2 * mu2, e12 - mu1 * mu2
    return ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 * mu1 + mu2 * mu2 + C1) * (s11 + s22 + C2))


def s3im_reference(src, tar, index, patch_h, ksize, stride):
    """float64 S3IM.forward (losses.py:779-794): 1 - SSIM of the virtual images [1, 3, patch_h, n / patch_h] with a
    depthwise conv2d, stride and zero padding (ksize - 1) // 2.  -> (loss, dloss/dsrc, loss bound): the bound lets
    each of the five window sums carry (ksize^2 + 8) u of the sum of its terms' magnitudes and propagates that through
    SSIM's partial derivatives, plus the roundings of the SSIM formula and of the sum over windows."""
    x0 = torch.from_numpy(src).double().requires_grad_()
    idx = torch.from_numpy(index)
    img = lambda v: v[idx].t().reshape(1, 3, patch_h, -1)
    win = s3im_window(ksize).expand(3, 1, ksize, ksize)
    conv = lambda a: F.conv2d(a, win, padding=(ksize - 1) // 2, groups=3, stride=stride)
    x, y = img(x0), img(torch.from_numpy(tar).double())
    sums = [conv(x), conv(y), conv(x * x), conv(y * y), conv(x * y)]
    ssim = _ssim_map(*sums)
    loss = 1 - ssim.mean()
    loss.backward()
    q = [s.detach().requires_grad_() for s in sums]
    s = _ssim_map(*q)
    s.sum().backward()
    xd = x.detach()
    mu1, mu2 = q[0].detach(), q[1].detach()
    mag = [conv(xd.abs()), conv(y.abs()), conv(xd * xd) + mu1 * mu1, conv(y * y) + mu2 * mu2,
           conv((xd * y).abs()) + (mu1 * mu2).abs()]
    d_ssim = (ksize * ksize + 8) * U * sum(qi.grad.abs() * m for qi, m in zip(q, mag)) + 8 * U * s.detach().abs()
    bound = float(d_ssim.mean() + C * U * (1 - s.detach()).abs().mean()) + FLOOR
    return float(loss.detach()), x0.grad.numpy(), bound


def run_s3im(src, tar, index, patch_h, ksize, stride, mult=1.0, g0=None, loss0=0.0):
    from gfnerf_b200 import _lib
    R = src.shape[0]
    g = _dev(np.zeros_like(src) if g0 is None else g0)
    loss = torch.full((1,), loss0, device="cuda")
    s, t, i = _dev(src), _dev(tar), _dev(index)
    _lib.check(_lib.lib().gf_s3im(R, index.size, _lib.ptr(i), _lib.ptr(s), _lib.ptr(t), patch_h, ksize, stride, mult,
                                  _lib.ptr(g), _lib.ptr(loss), _lib.cur_stream()), "gf_s3im")
    return float(loss), g.cpu().numpy()


def s3im_case(R, repeat, seed):
    rng = np.random.RandomState(seed)
    src = rng.uniform(0, 1, size=(R, 3)).astype(np.float32)
    tar = np.clip(src + rng.normal(0, 0.1, size=(R, 3)), 0, 1).astype(np.float32)
    index = np.concatenate([np.arange(R)] + [rng.permutation(R) for _ in range(repeat - 1)]).astype(np.int64)
    return src, tar, index


# (patch_h, repeat, R / patch_h): virtual widths 13, 21, 30, 50, 11 -- most leave the last window partial
S3IM_LAYOUTS = ((8, 1, 13), (32, 3, 7), (64, 10, 3), (8, 10, 5), (32, 1, 11))


def check_s3im(got_loss, got_g, loss, g, bound, mult=1.0, rel=1e-4):
    assert abs(got_loss - mult * loss) <= abs(mult) * bound, (got_loss, mult * loss, abs(mult) * bound)
    tol = rel * abs(mult) * np.abs(g).max()      # fp32 variance terms cancel: 1e-4 of the largest gradient
    err = np.abs(got_g - mult * g)
    assert err.max() <= tol, (float(err.max()), tol, np.unravel_index(err.argmax(), err.shape))


@gpu
@pytest.mark.parametrize("stride", (1, 2, 3, 5))
@pytest.mark.parametrize("ksize", (1, 2, 3, 4, 5, 7, 8))
def test_s3im_matches_float64_reference(ksize, stride):
    for n, (patch_h, repeat, q) in enumerate(S3IM_LAYOUTS):
        src, tar, index = s3im_case(patch_h * q, repeat, seed=100 * ksize + 10 * stride + n)
        loss, g, bound = s3im_reference(src, tar, index, patch_h, ksize, stride)
        got_loss, got_g = run_s3im(src, tar, index, patch_h, ksize, stride)
        check_s3im(got_loss, got_g, loss, g, bound)


@gpu
def test_s3im_accumulates_with_its_multiplier():
    src, tar, index = s3im_case(32 * 9, 10, seed=20)
    loss, g, bound = s3im_reference(src, tar, index, 32, 4, 2)
    # an existing gradient of the S3IM gradient's scale (a larger one would round the sum beyond the tolerance)
    g0 = (np.random.RandomState(21).normal(size=src.shape) * np.abs(g).max()).astype(np.float32)
    got_loss, got_g = run_s3im(src, tar, index, 32, 4, 2, mult=0.5, g0=g0, loss0=0.375)
    check_s3im(got_loss - 0.375, got_g - g0, loss, g, bound + 2 * C * U, mult=0.5)


@gpu
def test_s3im_constant_images():
    R, repeat, patch_h = 32 * 6, 3, 32
    index = s3im_case(R, repeat, seed=22)[2]
    for ksize, stride in ((4, 4), (3, 1), (8, 2)):
        same = np.full((R, 3), 0.4, np.float32)
        got_loss, got_g = run_s3im(same, same, index, patch_h, ksize, stride)
        assert abs(got_loss) <= 16 * U and np.abs(got_g).max() <= 1e-7      # SSIM 1, a maximum: loss and gradient 0
        src, tar = np.full((R, 3), 0.3, np.float32), np.full((R, 3), 0.7, np.float32)
        loss, g, bound = s3im_reference(src, tar, index, patch_h, ksize, stride)
        # windows of (nearly) zero variance: the fp32 variance terms are rounding noise next to C2 = 9e-4, which
        # costs the gradient about 1e-4 of its largest value (fp32 torch: 1.1e-4 at ksize 8, stride 2)
        check_s3im(*run_s3im(src, tar, index, patch_h, ksize, stride), loss, g, bound, rel=1e-3)


def test_s3im_rejects_bad_shapes():
    """argument checks run before any CUDA call (no GPU needed)"""
    from gfnerf_b200 import _lib
    L = _lib.lib()
    p = 256
    # the last three: 1 + 2 * 3 < 8 rows or columns; with stride 2 or 3, (1 + 6 - 8) / stride truncates to 0 and
    # would pass as one output row
    for ksize, stride, n_virtual, patch_h, what in ((0, 1, 64, 8, b"bad sizes"), (9, 1, 64, 8, b"bad sizes"),
                                                    (4, 0, 64, 8, b"bad sizes"), (4, 4, 60, 8, b"multiple"),
                                                    (8, 1, 64, 1, b"does not fit"), (8, 2, 64, 1, b"does not fit"),
                                                    (8, 3, 64, 64, b"does not fit")):
        assert L.gf_s3im(8, n_virtual, p, p, p, patch_h, ksize, stride, 1.0, p, p, None) == -1, (ksize, stride)
        assert what in L.gf_last_error(), L.gf_last_error()


# ------------------------------------------------------------------------------------------------ Charbonnier
@gpu
@pytest.mark.parametrize("R", (1, 33, 8192, 200_000))
def test_charbonnier_matches_float64(R):
    from gfnerf_b200 import _lib
    rng = np.random.RandomState(R)
    pred = rng.uniform(0, 1, size=(R, 3)).astype(np.float32)
    target = rng.uniform(0, 1, size=(R, 3)).astype(np.float32)
    same = rng.rand(R) < 0.2
    same[0] = True
    target[same] = pred[same]                                  # zero residual: sqrt(eps^2) and a zero gradient
    eps = 1e-6
    d = pred.astype(np.float64) - target
    s = np.sqrt(d * d + eps * eps)
    loss, g = s.sum() / R, d / s / R
    g_rgb, got = torch.full((R, 3), math.nan, device="cuda"), torch.zeros(1, device="cuda")
    p, t = _dev(pred), _dev(target)
    _lib.check(_lib.lib().gf_charbonnier(R, _lib.ptr(p), _lib.ptr(t), eps, _lib.ptr(g_rgb),
                                         _lib.ptr(got), _lib.cur_stream()), "gf_charbonnier")
    g_rgb = g_rgb.cpu().numpy().astype(np.float64)
    assert np.array_equal(g_rgb[same], np.zeros((int(same.sum()), 3)))
    assert np.all(np.abs(g_rgb - g) <= 8 * U * np.abs(g) + FLOOR)
    # the sum: a few terms per thread, 5 shuffle levels, then one atomicAdd per warp of the 4-CTAs-per-SM grid
    n3 = 3 * R
    threads = min(-(-n3 // 256), torch.cuda.get_device_properties(0).multi_processor_count * 4) * 256
    adds = -(-n3 // threads) + 5 + threads // 32 + 8
    assert abs(float(got) - loss) <= adds * U * loss, (float(got), loss)
