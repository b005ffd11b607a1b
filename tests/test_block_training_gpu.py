"""Several focal-stage blocks trained in one step: the routed residual hash scatter `gf_hash_backward_routed` (what
`gf_hash_backward_levels` computes with each sample's table) and `GFNeRFEngine.start_block_stage(blocks=...)`, whose
step must be, block for block, what a single-block engine computes on the block's segment of the batch.

Scatter sums are compared bit for bit in the exact-sum regime of test_kernel_variants_gpu.py (every contribution a
multiple of 2^-31 and every row's sum|c| below 2^-7, so any summation order gives the same fp32 value), and within twice
the (k - 1) 2^-24 sum|c| reorder bound outside it.  The argument checks at the top need no GPU."""
import ctypes

import numpy as np
import pytest
import torch

from tests.helpers import hash_inputs, load_rig, make_sampler

EXACT_LIMIT = 2.0 ** -7


# ---- argument checks (no GPU) -----------------------------------------------------------------------------------------
def test_routed_scatter_rejections():
    from gfnerf_b200 import _lib
    L = _lib.lib()
    p = ctypes.c_void_p(4096)

    def call(n_tables=2, tables=p, ray_id=p, ray_table=p, grad=p, n=10, local=16, pts=p):
        return L.gf_hash_backward_routed(n, None, 1, local, n_tables, tables, p, pts, p, 0, ray_id, ray_table, grad, 1,
                                         None)

    for kw in (dict(n_tables=0), dict(n_tables=-3), dict(tables=None), dict(ray_id=None), dict(ray_table=None),
               dict(n_tables=0, n=0), dict(tables=None, n=0), dict(grad=None), dict(pts=None), dict(local=15),
               dict(grad=ctypes.c_void_p(4096 + 8))):
        assert call(**kw) == -1, kw
        assert b"gf_hash_backward_routed" in L.gf_last_error(), kw


# ---- the kernel -------------------------------------------------------------------------------------------------------
def _scales():
    from gfnerf_b200 import _lib
    s = torch.empty(16, device="cuda")
    _lib.check(_lib.lib().gf_hash_level_scales(_lib.ptr(s), None, _lib.cur_stream()))
    return s


def _tables(k, local, n_vol, seed, bias_at=None):
    """k (prime pool, bias pool or None, zeroed gradient table) triples of 16 * local rows"""
    rng = np.random.RandomState(seed)
    out = []
    for j in range(k):
        _, prim, _, _, _ = hash_inputs(8, n_vol, 10, seed=seed + 31 * j)
        bias = (torch.from_numpy(rng.uniform(-1, 1, size=(16 * n_vol, 3)).astype(np.float32)).cuda()
                if j == bias_at else None)
        out.append((torch.from_numpy(prim.astype(np.int32)).cuda().contiguous(), bias,
                    torch.zeros((16 * local, 2), device="cuda")))
    return out


def _refs(tables):
    return torch.tensor([[p.data_ptr(), 0 if b is None else b.data_ptr(), g.data_ptr()] for p, b, g in tables],
                        dtype=torch.int64).cuda()


def _per_table(tables, n_vol, local, scales, pts, anc, grad, flags, ray_id, ray_table, n=None):
    """gf_hash_backward_levels of each table on the samples routed to it (the first n samples)"""
    from gfnerf_b200 import _lib
    L = _lib.lib()
    n = pts.shape[0] if n is None else n
    t = ray_table.long()[ray_id[:n].long()]
    for k, (prim, bias, g) in enumerate(tables):
        idx = (t == k).nonzero().squeeze(1)
        if idx.numel() == 0:
            continue
        p, a, gi = pts[idx].contiguous(), anc[idx].contiguous(), grad[idx].contiguous()
        _lib.check(L.gf_hash_backward_levels(idx.numel(), None, n_vol, local, _lib.ptr(prim), _lib.ptr(bias),
                                             _lib.ptr(scales), _lib.ptr(p), _lib.ptr(a), int(a.dtype == torch.int64),
                                             _lib.ptr(gi), flags, _lib.ptr(g), 0, 16, _lib.cur_stream()),
                   "gf_hash_backward_levels")
    torch.cuda.synchronize()


def _routed(tables, n_vol, local, scales, pts, anc, grad, flags, ray_id, ray_table, n=None, d_n=None):
    from gfnerf_b200 import _lib
    refs = _refs(tables)
    n = pts.shape[0] if n is None else n
    _lib.check(_lib.lib().gf_hash_backward_routed(
        n, _lib.ptr(d_n), n_vol, local, len(tables), _lib.ptr(refs), _lib.ptr(scales), _lib.ptr(pts), _lib.ptr(anc),
        int(anc.dtype == torch.int64), _lib.ptr(ray_id), _lib.ptr(ray_table), _lib.ptr(grad), flags,
        _lib.cur_stream()), "gf_hash_backward_routed")
    torch.cuda.synchronize()


def _rays_of(n, seed, mean_len=12):
    """ray_id int32 [n] in the sampler's compact layout: consecutive samples of a ray, runs of 1..2*mean_len"""
    rng = np.random.RandomState(seed)
    lens = rng.randint(1, 2 * mean_len, size=n)
    rid = np.repeat(np.arange(n), lens)[:n]
    return torch.from_numpy(rid.astype(np.int32)).cuda(), int(rid[-1]) + 1


def _routes(n_rays, k, seed):
    rng = np.random.RandomState(seed)
    per_ray = rng.randint(-1, k + 1, size=n_rays)                     # -1 and k: no table
    segments = np.minimum(np.arange(n_rays) * k // n_rays, k - 1)      # the engine's layout: K contiguous segments
    return {"per_ray": per_ray, "segments": segments}


def _grad_in(n, g16, scale, seed):
    """fp32 dL/dfeat [n,32], or the fp16 x128 form gf_mlp_backward writes"""
    g = torch.empty((n, 32), device="cuda").uniform_(-scale, scale, generator=torch.Generator("cuda").manual_seed(seed))
    return (g * 128).half().contiguous() if g16 else g


def _flags(g16, x128):
    return int(g16) | (2 if x128 else 0)


def _cmp_exact(tables, ref_tables, what):
    for j, ((_, _, g), (_, _, r)) in enumerate(zip(tables, ref_tables)):
        bad = (g != r).any(1).nonzero().squeeze(1)
        assert bad.numel() == 0, f"{what}: table {j}: {bad.numel()} rows differ, first {bad[:4].tolist()}"


@pytest.mark.gpu
@pytest.mark.parametrize("log2T,local_pow2", [(19, True), (23, True), (19, False)])
def test_routed_scatter_bit_exact(log2T, local_pow2):
    """exact-sum regime: bit for bit the per-table scatter, for K = 1, 3, 8, random and segment routes, both gradient
    forms with and without x128, both anchor types, a table with a bias pool"""
    n, n_vol = 20000, 7
    local = (1 << log2T) if local_pow2 else (3 << (log2T - 2))
    _, _, _, pts, anc = hash_inputs(n, n_vol, 12, seed=log2T)
    tp = torch.from_numpy(pts).cuda()
    scales = _scales()
    ray_id, n_rays = _rays_of(n, seed=2, mean_len=6)
    # |g| <= 2^-22 with n samples: no row's sum|c| can reach n * 2^-22 < 2^-7
    assert n * 2.0 ** -22 < EXACT_LIMIT
    written = 0
    for k in (1, 3, 8):
        for name, rt in _routes(n_rays, k, seed=k).items():
            ray_table = torch.from_numpy(rt.astype(np.int32)).cuda()
            for g16 in (True, False):
                for x128 in (True, False):
                    anc_dt = torch.int64 if (k + g16 + x128) % 2 else torch.int32
                    ta = torch.from_numpy(anc).cuda().to(anc_dt)
                    grad = _grad_in(n, g16, 2.0 ** -22, seed=k * 7 + g16 * 2 + x128)
                    got = _tables(k, local, n_vol, seed=log2T + k, bias_at=k - 1)
                    ref = _tables(k, local, n_vol, seed=log2T + k, bias_at=k - 1)
                    _routed(got, n_vol, local, scales, tp, ta, grad, _flags(g16, x128), ray_id, ray_table)
                    _per_table(ref, n_vol, local, scales, tp, ta, grad, _flags(g16, x128), ray_id, ray_table)
                    _cmp_exact(got, ref, (k, name, g16, x128, anc_dt))
                    written += sum(int((g != 0).any(1).sum()) for _, _, g in got)
    assert written > 100000


@pytest.mark.gpu
def test_routed_scatter_counts():
    """a device-side count below n, and n = 0"""
    n, n_vol, k, local = 9000, 5, 3, 1 << 14
    _, _, _, pts, anc = hash_inputs(n, n_vol, 10, seed=3)
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anc).cuda().to(torch.int32)
    scales = _scales()
    ray_id, n_rays = _rays_of(n, seed=7)
    ray_table = torch.from_numpy(np.random.RandomState(5).randint(-1, k + 1, size=n_rays).astype(np.int32)).cuda()
    grad = _grad_in(n, True, 2.0 ** -22, seed=1)
    m = n - 1234
    got, ref = _tables(k, local, n_vol, seed=1), _tables(k, local, n_vol, seed=1)
    _routed(got, n_vol, local, scales, tp, ta, grad, 1, ray_id, ray_table,
            d_n=torch.tensor([m], dtype=torch.int32, device="cuda"))
    _per_table(ref, n_vol, local, scales, tp, ta, grad, 1, ray_id, ray_table, n=m)
    _cmp_exact(got, ref, "d_n_ptr")
    assert any(bool(g.any()) for _, _, g in got)
    got = _tables(k, local, n_vol, seed=1)
    _routed(got, n_vol, local, scales, tp, ta, grad, 1, ray_id, ray_table, n=0)
    assert not any(bool(g.any()) for _, _, g in got)


@pytest.mark.gpu
@pytest.mark.parametrize("run", [2, 3, 4, 5, 8, 13])
def test_same_cell_different_tables(run):
    """adjacent lanes with the same point and anchor but another table: the run key includes the table.  Runs of 2-4
    lanes take the shuffle reduction, longer ones the shared-memory walker; a key without the table sums a whole warp
    into one lane's table and fails here."""
    n_vol, k, local = 3, 3, 1 << 14
    n = 32 * 64
    rng = np.random.RandomState(run)
    # every warp: one point and anchor for all 32 lanes; tables change every `run` lanes (cycling, so a table also
    # comes back after another one)
    pts = np.repeat(rng.uniform(0.2, 0.8, size=(n // 32, 3)), 32, axis=0).astype(np.float32)
    anc = np.repeat(rng.randint(0, n_vol, size=n // 32), 32).astype(np.int64)
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anc).cuda()
    ray_id = torch.arange(n, dtype=torch.int32, device="cuda")
    lane = np.arange(n) % 32
    ray_table = torch.from_numpy(((lane // run + np.arange(n) // 32) % k).astype(np.int32)).cuda()
    scales = _scales()
    for g16 in (True, False):
        grad = _grad_in(n, g16, 2.0 ** -22, seed=run)
        got, ref = _tables(k, local, n_vol, seed=4), _tables(k, local, n_vol, seed=4)
        _routed(got, n_vol, local, scales, tp, ta, grad, _flags(g16, True), ray_id, ray_table)
        _per_table(ref, n_vol, local, scales, tp, ta, grad, _flags(g16, True), ray_id, ray_table)
        _cmp_exact(got, ref, (run, g16))
        assert all(bool(g.any()) for _, _, g in got)


@pytest.mark.gpu
def test_routed_scatter_reorder_bound():
    """|g| ~ 1e-3, outside the exact regime: both sides are within (k - 1) 2^-24 sum|c| of the exact row sum"""
    from gfnerf_b200 import _lib
    n, n_vol, k, log2T = 60000, 7, 3, 16
    local = 1 << log2T
    _, _, _, pts, anc = hash_inputs(n, n_vol, 12, seed=8)
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anc).cuda()
    scales = _scales()
    ray_id, n_rays = _rays_of(n, seed=9, mean_len=8)
    ray_table = torch.from_numpy(_routes(n_rays, k, seed=3)["per_ray"].astype(np.int32)).cuda()
    grad = _grad_in(n, False, 1e-3, seed=5)
    got, ref = _tables(k, local, n_vol, seed=6, bias_at=1), _tables(k, local, n_vol, seed=6, bias_at=1)
    _routed(got, n_vol, local, scales, tp, ta, grad, 0, ray_id, ray_table)
    _per_table(ref, n_vol, local, scales, tp, ta, grad, 0, ray_id, ray_table)
    # sum|c| per row: the same scatter of |g| (fp16 rounding is symmetric, so |c| = c of |g|), and k per row from
    # the corner rows of the samples routed to each table
    absg = grad.abs().contiguous()
    sabs = _tables(k, local, n_vol, seed=6, bias_at=1)
    _per_table(sabs, n_vol, local, scales, tp, ta, absg, 0, ray_id, ray_table)
    t = ray_table.long()[ray_id.long()]
    beyond = 0
    for j, ((prim, bias, g), (_, _, r), (_, _, s)) in enumerate(zip(got, ref, sabs)):
        idx = (t == j).nonzero().squeeze(1)
        rows = torch.empty((idx.numel(), 16, 8), dtype=torch.int32, device="cuda")
        a = ta[idx].contiguous()
        _lib.check(_lib.lib().gf_hash_corner_rows(idx.numel(), n_vol, local, _lib.ptr(prim), _lib.ptr(bias),
                                                  _lib.ptr(scales), _lib.ptr(tp[idx].contiguous()), _lib.ptr(a), 1,
                                                  _lib.ptr(rows), _lib.cur_stream()), "gf_hash_corner_rows")
        k_row = torch.bincount(rows.view(-1).long(), minlength=16 * local).double()[:, None]
        bound = 2 * (k_row - 1).clamp_min(0) * 2.0 ** -24 * s.double() * 1.01
        err = (g.double() - r.double()).abs()
        assert bool((err <= bound).all()), f"table {j}: worst excess {float((err - bound).max())}"
        assert not bool(g[k_row[:, 0] == 0].any())
        beyond += int((s.double() > EXACT_LIMIT).sum())
    assert beyond > 10                                # the test is outside the exact regime


# ---- the engine -------------------------------------------------------------------------------------------------------
def _engine(rig, hidden=64, seed=5, blocks=None, s3im=0.0, res_init=None):
    from gfnerf_b200.engine import GFNeRFEngine
    eng = GFNeRFEngine(make_sampler(rig, mode=1), log2_table_size=14, num_images=rig["c2w"].shape[0], hidden=hidden,
                       seed=3, s3im_loss_mult=s3im)
    init = torch.rand(eng.enc.feat_pool_.shape, generator=torch.Generator().manual_seed(11)) * 0.2 - 0.1
    eng.enc.feat_pool_.data.copy_(init)
    eng.enc.shadow(force=True)
    eng.start_block_stage(log2_table_size=14, seed=seed, blocks=blocks)
    if res_init is not None:                           # non-zero residual tables, so the forward reads them
        cores = eng.res_blocks if blocks is not None else [eng.res]
        for j, c in enumerate(cores):
            c.feat_pool_.data.copy_(res_init(j))
            c.shadow(force=True)
    return eng


def _res_init(offset):
    return lambda j: torch.rand((16 << 14, 2), generator=torch.Generator().manual_seed(100 + offset + j)) * 0.1 - 0.05


def _batch(rig, R, seed):
    from gfnerf_b200.persoctree import rig_rays
    o, d, cam = rig_rays(rig["c2w"], rig["intri"], R, seed=seed)
    target = torch.rand((R, 3), generator=torch.Generator().manual_seed(seed)).cuda()
    return torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), target, torch.from_numpy(cam).cuda()


def _close_tables(a, b, what):
    """two gradient tables summed in another order (the kernel tests check the reorder bound itself): within 1e-4 of
    the element and of the table's largest magnitude (rows where large terms cancel keep their absolute error)"""
    tol = 1e-4 * (torch.maximum(a.abs(), b.abs()) + float(b.abs().max()))
    assert bool(((a - b).abs() <= tol).all()), f"{what}: worst {float(((a - b).abs() - tol).max())}"


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [64, 128])
def test_first_step_matches_single_block_engines(hidden):
    K, Rb = 3, 512
    blocks = [4, 0, 7]
    rig = load_rig("rig8")
    multi = _engine(rig, hidden, blocks=blocks, res_init=_res_init(0))
    singles = [_engine(rig, hidden, seed=5 + k, res_init=lambda j, k=k: _res_init(k)(0)) for k in range(K)]
    for k in range(K):
        assert torch.equal(multi.res_blocks[k].prim_pool_, singles[k].res.prim_pool_)   # table k seeded seed + k
    o, d, t, cam = _batch(rig, K * Rb, seed=21)
    out = multi.train_step(o, d, t, cam, optimizer_step=False)
    assert out.block_losses.shape == (K,) and torch.equal(out.loss, out.block_losses.sum().view(1))
    V = int(out.n_samples.item())
    d_feat = multi._ws["d_feat"][:V * 32].view(V, 32).clone()
    feat = multi._ws["feat"][:V * 32].view(V, 32).clone()
    off = 0
    for k, s in enumerate(singles):
        seg = slice(k * Rb, (k + 1) * Rb)
        so = s.train_step(o[seg], d[seg], t[seg], cam[seg], optimizer_step=False)
        assert torch.equal(out.rgb[seg], so.rgb) and torch.equal(out.depth[seg], so.depth)
        assert torch.equal(out.accumulation[seg], so.accumulation)
        torch.testing.assert_close(out.block_losses[k:k + 1], so.loss, rtol=1e-6, atol=0)
        v = int(so.n_samples.item())
        # the features and the per-sample gradients the scatter receives: the same bits
        assert torch.equal(feat[off:off + v].view(torch.int16), s._ws["feat"][:v * 32].view(v, 32).view(torch.int16))
        assert torch.equal(d_feat[off:off + v].view(torch.int16),
                           s._ws["d_feat"][:v * 32].view(v, 32).view(torch.int16))
        off += v
        ga, gb = multi.opt_res_blocks[k].grad, s.opt_res.grad
        assert bool(gb.any())
        _close_tables(ga, gb, f"block {k} gradient")
    assert off == V


@pytest.mark.gpu
def test_focal_loop_with_batch_sources():
    """K FocalBatchSources feed one K-block engine and, with the same seeds, K single-block engines: 20 steps within
    the gates of test_focal_loop_matches_the_error_pixel_sampler_path"""
    from gfnerf_b200 import pixel_samplers as ps
    from gfnerf_b200.cameras import Cameras
    dev = torch.device("cuda:0")
    rig = load_rig("rig8")
    n_cam = rig["c2w"].shape[0]
    intri = torch.from_numpy(rig["intri"])
    cams = Cameras(torch.from_numpy(rig["c2w"]).to(dev), intri[:, 0, 0], intri[:, 1, 1], intri[:, 0, 2],
                   intri[:, 1, 2], width=1920, height=1080)
    K, Rb = 2, 1024
    g = torch.Generator(device=dev).manual_seed(0)
    slots = [torch.arange(k, n_cam, 16, device=dev) for k in range(K)]   # 4 images of each block
    images = [torch.rand(s.numel(), 1080, 1920, 3, device=dev, generator=g) for s in slots]
    errs = [torch.rand(s.numel(), 1080, 1920, 1, device=dev, generator=g) for s in slots]

    def sources():
        return [ps.FocalBatchSource(images[k], errs[k].clone(), cams, slots[k], slots[k], num_rays_per_batch=Rb,
                                    seed=40 + k) for k in range(K)]

    src_m, src_s = sources(), sources()
    multi = _engine(rig, blocks=[1, 2])
    singles = [_engine(rig, seed=5 + k) for k in range(K)]
    lm, ls = [], []
    for step in range(20):
        bm = [s.next_batch() for s in src_m]
        bs = [s.next_batch() for s in src_s]
        cat = {key: torch.cat([b[key] for b in bm]) for key in ("origins", "directions", "rgb", "rel_camera_indices")}
        out = multi.train_step(cat["origins"], cat["directions"], cat["rgb"], cat["rel_camera_indices"])
        lm.append(out.block_losses.clone())
        row = []
        for k in range(K):
            assert torch.equal(bs[k]["slot_indices"], bm[k]["slot_indices"])
            so = singles[k].train_step(bs[k]["origins"], bs[k]["directions"], bs[k]["rgb"], bs[k]["rel_camera_indices"])
            row.append(so.loss.clone())
            rgb_k = out.rgb[k * Rb:(k + 1) * Rb]
            src_m[k].update(bm[k]["slot_indices"], rgb_k)
            src_s[k].update(bs[k]["slot_indices"], rgb_k)                # the same feedback: the same next batches
        ls.append(torch.cat(row))
    for s in src_m + src_s:
        s.check()
    multi.flush()
    assert torch.allclose(torch.stack(lm), torch.stack(ls), rtol=1e-3, atol=0)
    for k in range(K):
        ra, rb = multi.res_blocks[k].feat_pool_.detach(), singles[k].res.feat_pool_.detach()
        assert bool(ra.any())
        assert float((ra - rb).abs().mean()) <= 1e-3 * float(ra.abs().mean())
        assert multi.opt_res_blocks[k].t == singles[k].opt_res.t == 20


@pytest.mark.gpu
def test_blocks_are_independent_with_s3im():
    K, Rb, j = 3, 512, 1
    rig = load_rig("rig8")
    o, d, t, cam = _batch(rig, K * Rb, seed=5)

    def run(target):
        eng = _engine(rig, blocks=[0, 1, 2], s3im=1.0, res_init=_res_init(0))
        assert eng.s3im == (1.0, 4, 4, 10, 32)
        torch.manual_seed(123)
        out = eng.train_step(o, d, target, cam, optimizer_step=False)
        return eng, out

    ea, oa = run(t)
    t2 = t.clone()
    t2[j * Rb:(j + 1) * Rb] = torch.rand((Rb, 3), generator=torch.Generator().manual_seed(9)).cuda()
    eb, ob = run(t2)
    assert not torch.equal(oa.block_losses[j], ob.block_losses[j])
    for k in range(K):
        if k == j:
            continue
        torch.testing.assert_close(oa.block_losses[k], ob.block_losses[k], rtol=1e-6, atol=0)
        _close_tables(ea.opt_res_blocks[k].grad, eb.opt_res_blocks[k].grad, f"block {k}")
    # a NaN in block j's targets: only block j skips its step
    t3 = t.clone()
    t3[j * Rb + 7, 1] = float("nan")
    eng = _engine(rig, blocks=[0, 1, 2], s3im=1.0, res_init=_res_init(0))
    before = [c.feat_pool_.detach().clone() for c in eng.res_blocks]
    out = eng.train_step(o, d, t3, cam)
    eng.flush()
    assert bool(torch.isnan(out.block_losses[j])) and bool(torch.isfinite(out.block_losses[[0, 2]]).all())
    for k in range(K):
        now = eng.res_blocks[k].feat_pool_.detach()
        if k == j:
            assert torch.equal(now, before[k]) and eng.opt_res_blocks[k].t == 0
        else:
            assert not torch.equal(now, before[k]) and eng.opt_res_blocks[k].t == 1
    assert [bool(x) for x in eng.last_nan_flag.tolist()] == [False, True, False]


@pytest.mark.gpu
def test_store_blocks_and_routed_model_render(tmp_path):
    """store_model(block=b) for every block, then the model's route_blocks=True render == the engine's render_rays
    with the same per-ray tables"""
    from gfnerf_b200.engine import GFNeRFEngine
    from tests.test_eval_views_gpu import make_cameras, make_model, view_bundle
    rig = load_rig("rig8")
    model = make_model(rig)
    f, ps = model.field, model.persampler
    eng = GFNeRFEngine.from_model(model)
    blocks = [2, 0, 1]
    eng.start_block_stage(seed=20, blocks=blocks)
    with pytest.raises(ValueError):
        eng.render_image(torch.zeros(4, 3, device="cuda"), torch.ones(4, 3, device="cuda"))   # no per-ray tables
    for it in range(4):
        o, d, t, cam = _batch(rig, 3 * 512, seed=60 + it)
        eng.train_step(o, d, t, cam)
    for b in blocks:
        eng.store_model(model, block=b)
    with pytest.raises(ValueError):
        eng.store_model(model, block=5)
    n_cam = ps.c2w.shape[0]
    labels = (torch.arange(n_cam) % 3).view(-1, 1)
    ps.cameras_labels = labels.cuda()
    f.set_stage("block_stage", active_block=0)
    model.eval()
    cams = make_cameras(rig)
    for k in (3, 4, 5):
        rb = view_bundle(cams, k)
        got = model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)
        n = rb.origins.shape[0] * rb.origins.shape[1]
        table = torch.full((n,), blocks.index(int(labels[k, 0])), dtype=torch.int32, device="cuda")
        cam = torch.full((n,), k, dtype=torch.int64, device="cuda")
        rgb, depth, acc, _ = eng.render_rays(rb.origins.reshape(-1, 3).contiguous(),
                                             rb.directions.reshape(-1, 3).contiguous(), cam, ray_table=table)
        assert float(acc.max()) > 0.5
        assert torch.equal(got["rgb"].reshape(-1, 3), rgb)
        assert torch.equal(got["depth"].reshape(-1), depth)
        assert torch.equal(got["accumulation"].reshape(-1), acc)


@pytest.mark.gpu
def test_checkpoint_resumes_like_the_uninterrupted_run():
    rig = load_rig("rig8")
    batches = [_batch(rig, 2 * 512, seed=80 + i) for i in range(8)]
    a = _engine(rig, blocks=[3, 1])
    for b in batches[:4]:
        a.train_step(*b)
    ck = a.checkpoint()
    assert ck["res_blocks"] == [3, 1] and "res_table" not in ck
    for b in batches[4:]:
        a.train_step(*b)
    r = _engine(rig, blocks=None, seed=99)               # another stage layout: restore rebuilds the blocks
    r.restore(ck)
    assert r.blocks == [3, 1] and r.res is None
    for b in batches[4:]:
        r.train_step(*b)
    a.flush()
    r.flush()
    for k in range(2):
        assert r.opt_res_blocks[k].t == a.opt_res_blocks[k].t == 8
        x, y = a.res_blocks[k].feat_pool_.detach(), r.res_blocks[k].feat_pool_.detach()
        assert float((x - y).abs().mean()) <= 1e-3 * float(x.abs().mean())
    single = _engine(rig)
    sck = single.checkpoint()
    assert "res_blocks" not in sck and "res_table" in sck


@pytest.mark.gpu
def test_no_host_sync_per_step():
    rig = load_rig("rig8")
    eng = _engine(rig, blocks=[0, 1])
    b = _batch(rig, 2 * 512, seed=3)
    eng.train_step(*b)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(2):
            eng.train_step(*b)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    eng.flush()


@pytest.mark.gpu
def test_rejections():
    rig = load_rig("rig8")
    eng = _engine(rig)
    for bad in ([1, 1], [-1, 2], []):
        with pytest.raises(ValueError):
            eng.start_block_stage(blocks=bad)
    eng.start_block_stage(blocks=[0, 1, 2])
    b = _batch(rig, 1000, seed=1)
    with pytest.raises(ValueError):
        eng.train_step(*b)                               # 1000 rays do not split into 3 segments
    eng.end_block_stage()
    assert eng.blocks is None and eng.res_tables is None and eng.res is None
