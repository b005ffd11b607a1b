"""GPU parity: gf_hash_* (through the C-ABI) against the CPU oracle on the same seeded inputs.

Bar: bit-exact corner rows and bit-exact forward values (both follow the same FMA convention);
gradients within 1e-5 relative of the exactly-summed oracle (fp32 atomics, order-dependent).
"""
import re

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import oracle as orc
from tests.helpers import hash_inputs

pytestmark = pytest.mark.gpu


def make_core(feat, prim, bias, log2T):
    from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
    core = Hash3DAnchoredCore(log2T, prim.shape[1])
    core.feat_pool_.data.copy_(torch.from_numpy(feat))
    core.prim_pool_ = torch.from_numpy(prim.astype(np.int32)).cuda().contiguous()
    core.bias_pool_ = torch.from_numpy(bias).cuda().contiguous()
    return core


def test_device_level_scales_reported():
    from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
    core = Hash3DAnchoredCore(8, 1)
    host = orc.hash_level_scales()
    dev = core.level_scales_host
    # the device's exp2f is an approximation (ex2.approx + range handling): allow 2 ulp, report equality
    np.testing.assert_allclose(dev, host, rtol=3e-7)
    print("device exp2f level scales bit-equal to host:", bool(np.array_equal(dev, host)))


def fwd_prefetch_args(prof):
    """the PREFETCH template argument (the last one) of every hash_fwd_kernel instantiation a profile recorded"""
    return {m.group(1) for e in prof.key_averages() for m in re.finditer(r"hash_fwd_kernel<[^>]*, (\w+)>", e.key)}


# the last three: the table sizes of BASELINE.json configs[1] (global stage, log2T = 19), configs[3] (focal stage, 21) and
# configs[4] (render, 23) -- value-level parity at the sizes the bench runs, on as many points as the oracle does in
# seconds, and both gather variants: the prefetching one while the reachable rows fit the L2 (up to 21), the other at 23
@pytest.mark.parametrize("n,n_vol,log2T,along", [(4096, 5, 12, True), (10000, 37, 15, False), (33, 1, 4, True),
                                                 (16384, 37, 19, True), (8192, 37, 21, True), (4096, 37, 23, False)])
def test_corner_rows_and_forward_bit_exact(n, n_vol, log2T, along):
    from gfnerf_b200 import _lib
    feat, prim, bias, pts, anchors = hash_inputs(n, n_vol, log2T, seed=n, along_rays=along)
    core = make_core(feat, prim, bias, log2T)
    scales = core.level_scales_host
    ref_out, ref_idx = orc.hash_forward(feat, prim, bias, pts, anchors, scales, want_idx=True)
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anchors).cuda()
    rows = torch.empty((n, 16, 8), dtype=torch.int32, device="cuda")
    _lib.check(_lib.lib().gf_hash_corner_rows(n, n_vol, core.local_size_, _lib.ptr(core.prim_pool_),
                                              _lib.ptr(core.bias_pool_), _lib.ptr(core.level_scales_), _lib.ptr(tp),
                                              _lib.ptr(ta), 1, _lib.ptr(rows), _lib.cur_stream()))
    assert np.array_equal(rows.cpu().numpy(), ref_idx)
    # int32 anchors + fp16 output + device-side count
    out16 = torch.zeros((n, 32), dtype=torch.float16, device="cuda")
    n_dev = torch.tensor([n - 7], dtype=torch.int32, device="cuda")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = core.AnchoredQuery(tp, ta)
        core.launch_forward(tp, ta.to(torch.int32), out_f16=out16, d_n_ptr=n_dev)
        torch.cuda.synchronize()
    assert fwd_prefetch_args(prof) == {"false" if log2T == 23 else "true"}
    assert np.array_equal(out.detach().cpu().numpy(), ref_out)
    got = out16.float().cpu().numpy()
    assert np.array_equal(got[: n - 7], ref_out[: n - 7])
    assert not got[n - 7:].any()


def test_non_pow2_table():
    from gfnerf_b200 import _lib
    rng = np.random.RandomState(4)
    local = 48 * 16
    n, n_vol = 2000, 3
    _, prim, bias, pts, anchors = hash_inputs(n, n_vol, 10, seed=9)
    feat = rng.uniform(-1, 1, size=(16 * local, 2)).astype(np.float32)
    scales_d = torch.empty(16, device="cuda")
    scales_h = np.zeros(16, np.float32)
    _lib.check(_lib.lib().gf_hash_level_scales(_lib.ptr(scales_d), scales_h.ctypes.data, _lib.cur_stream()))
    ref = orc.hash_forward(feat, prim, bias, pts, anchors, scales_h)
    f16 = torch.from_numpy(feat).cuda().half().contiguous()
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anchors).cuda()
    tprim, tbias = torch.from_numpy(prim.astype(np.int32)).cuda().contiguous(), torch.from_numpy(bias).cuda()
    out = torch.empty((n, 32), device="cuda")
    _lib.check(_lib.lib().gf_hash_forward(n, None, n_vol, local, _lib.ptr(f16), _lib.ptr(tprim), _lib.ptr(tbias),
                                          _lib.ptr(scales_d), _lib.ptr(tp), _lib.ptr(ta), 1, None, _lib.ptr(out),
                                          _lib.cur_stream()))
    assert np.array_equal(out.cpu().numpy(), ref)


@pytest.mark.parametrize("n,n_vol,log2T,along", [(4096, 5, 12, True), (20000, 11, 14, False), (31, 2, 6, True),
                                                 (16384, 37, 19, True), (8192, 37, 21, False)])   # configs[1] / [3] table sizes
def test_backward_matches_oracle(n, n_vol, log2T, along):
    feat, prim, bias, pts, anchors = hash_inputs(n, n_vol, log2T, seed=n + 1, along_rays=along)
    core = make_core(feat, prim, bias, log2T)
    rng = np.random.RandomState(n)
    g = (rng.normal(size=(n, 32)) * 1e-3).astype(np.float32)
    g[rng.rand(n, 32) < 0.2] = 0
    ref = orc.hash_backward(core.local_size_, prim, bias, pts, anchors, g, core.level_scales_host)
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anchors).cuda()
    out = core.AnchoredQuery(tp, ta)
    out.backward(torch.from_numpy(g).cuda())
    got = core.feat_pool_.grad.double().cpu().numpy()
    scale = np.abs(ref).max()
    # 1e-5 relative (north star) on every row, with an absolute floor for rows that cancel
    assert np.all(np.abs(got - ref) <= 1e-5 * np.abs(ref) + 1e-6 * scale)
    assert np.array_equal(got == 0, ref == 0)
    # pre-scaled fp16 gradient input (what gf_mlp_backward hands over) gives the same table
    g16 = (torch.from_numpy(g).cuda() * 128).half().contiguous()
    gt = torch.zeros_like(core.feat_pool_)
    core.launch_backward(tp, ta.to(torch.int32), g16, True, gt)
    assert np.all(np.abs(gt.double().cpu().numpy() - ref) <= 1e-5 * np.abs(ref) + 1e-6 * scale)
    # level groups (data-parallel training scatters and all-reduces the table group by group): same table
    gt.zero_()
    for l0 in range(0, 16, 4):
        core.launch_backward(tp, ta.to(torch.int32), g16, True, gt, levels=(l0, l0 + 4))
    assert np.all(np.abs(gt.double().cpu().numpy() - ref) <= 1e-5 * np.abs(ref) + 1e-6 * scale)
    # table left at the reference's x128 scale (the fused engine folds the division into Adam): same sums, x128
    gt.zero_()
    core.launch_backward(tp, ta.to(torch.int32), g16, True, gt, keep_x128=True)
    assert np.all(np.abs(gt.double().cpu().numpy() / 128 - ref) <= 1e-5 * np.abs(ref) + 1e-6 * scale)


def test_module_surface_and_state_roundtrip():
    from gfnerf_b200 import Hash3DAnchored
    enc = Hash3DAnchored(10, 3)
    enc.reset()
    pts = torch.rand(100, 3, device="cuda") * 0.6 + 0.2
    anc = torch.randint(0, 3, (100,), device="cuda")
    a = enc([pts, anc])
    sd = enc.state_dict(prefix="field.base_encoding_init.")
    assert set(k.split(".")[-1] for k in sd) >= {"feat_pool", "prime_pool", "bias_pool", "n_volumes"}
    enc2 = Hash3DAnchored(10, 3)
    enc2.load_state_dict({k: v.clone() for k, v in sd.items()}, prefix="field.base_encoding_init")
    b = enc2([pts, anc])
    assert torch.equal(a, b)
    assert list(enc.parameters())[0] is enc.get_params()[0]
    enc.zero()
    assert float(enc([pts, anc]).abs().max()) == 0.0
    # two forwards before one backward: gradients of both reach the table (reference hazard fixed)
    enc.reset()
    y1, y2 = enc([pts, anc]), enc([pts * 0.9, anc])
    (y1.sum() + y2.sum()).backward()
    assert enc.get_params()[0].grad.abs().sum() > 0


def test_full_size_properties():
    """BASELINE config 2 size (log2T=19, 2^20 points): linearity in the table and adjointness."""
    from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
    torch.manual_seed(0)
    n, n_vol = 1 << 20, 64
    core = Hash3DAnchoredCore(19, n_vol)
    core.Reset()
    # fp16-exact, fp16-normal table entries: then x2 is exact through the fp16 shadow
    q = core.feat_pool_.data.half().float()
    core.feat_pool_.data.copy_(torch.where(q.abs() < 2.0 ** -13, torch.full_like(q, 2.0 ** -13), q))
    pts = (torch.rand(n, 3, device="cuda") * 0.66 + 0.17).contiguous()
    anc = torch.randint(0, n_vol, (n,), device="cuda")
    y = core.AnchoredQuery(pts, anc)
    g = torch.randn_like(y) * 1e-3
    y.backward(g)
    # <J^T g, table16> ~= <g, J table16>
    t16 = core.feat_pool_.detach().half().double()
    lhs = float((core.feat_pool_.grad.double() * t16).sum())
    rhs = float((g.double() * y.detach().double()).sum())
    # Both sides are sums of ~3e7 random-sign terms g_i * y_i, so |rhs| itself is only ~ the L2 norm of the terms and
    # a tolerance relative to |rhs| is a ratio of two Gaussians (it failed one time in six by chance).  The honest
    # scale is that L2 norm: the fp16 quantisations (gradient x128 -> fp16, every w * g product -> fp16, y -> fp16)
    # put ~1e-3 of it between the two sides; a backward that scattered into other rows than the forward read would put
    # ~1.4 x of it there.
    l2 = float((g.double() * y.detach().double()).pow(2).sum().sqrt())
    assert abs(lhs - rhs) <= 0.02 * l2, (lhs, rhs, l2)
    # scaling the table by 2 (exact in fp16) scales the encoding by 2 exactly
    core.feat_pool_.data.mul_(2)
    y2 = core.AnchoredQuery(pts, anc)
    # (exact except where the fp16 result is subnormal: allow one subnormal step)
    assert float((y2.detach() - y.detach() * 2).abs().max()) <= 2.0 ** -23


def test_bias_pool_paths():
    """A non-zero bias pool (the reference allocates one but never fills it, Hash3DAnchored.cpp:57-62) against the
    oracle, and NULL == an all-zero pool bit for bit."""
    n, n_vol, log2T = 3000, 4, 11
    feat, prim, bias, pts, anchors = hash_inputs(n, n_vol, log2T, seed=21)
    rng = np.random.RandomState(1)
    bias_nz = rng.uniform(0, 1, size=bias.shape).astype(np.float32)
    for b in (bias_nz, bias):
        core = make_core(feat, prim, b, log2T)
        tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anchors).cuda()
        out = torch.empty((n, 32), device="cuda")
        core.launch_forward(tp, ta, out_f32=out)
        ref = orc.hash_forward(feat, prim, b, pts, anchors, core.level_scales_host)
        assert np.array_equal(out.cpu().numpy(), ref)
        assert (core._bias() is None) == (not b.any())
        g = (rng.normal(size=(n, 32)) * 1e-3).astype(np.float32)
        gref = orc.hash_backward(core.local_size_, prim, b, pts, anchors, g, core.level_scales_host)
        gt = torch.zeros_like(core.feat_pool_)
        core.launch_backward(tp, ta, torch.from_numpy(g).cuda(), False, gt)
        assert np.all(np.abs(gt.double().cpu().numpy() - gref) <= 1e-5 * np.abs(gref) + 1e-6 * np.abs(gref).max())
    # explicit zero pool pointer vs NULL through the C-ABI
    from gfnerf_b200 import _lib
    core = make_core(feat, prim, bias, log2T)
    o1, o2 = torch.empty((n, 32), device="cuda"), torch.empty((n, 32), device="cuda")
    for o, bp in ((o1, core.bias_pool_), (o2, None)):
        _lib.check(_lib.lib().gf_hash_forward(n, None, n_vol, core.local_size_, _lib.ptr(core.shadow()),
                                              _lib.ptr(core.prim_pool_), _lib.ptr(bp), _lib.ptr(core.level_scales_),
                                              _lib.ptr(tp), _lib.ptr(ta), 1, None, _lib.ptr(o), _lib.cur_stream()))
    assert torch.equal(o1, o2)
