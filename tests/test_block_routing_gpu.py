"""Focal-stage evaluation across all blocks: the routed residual gather `gf_hash_forward_residual_routed` (bit for bit
what `gf_hash_forward_residual` computes with each sample's table), `GFNeRFModel.get_outputs_for_camera_ray_bundle(
route_blocks=True)` against the reference's per-chunk block routing (eval mode, `generate_ray_samples` ->
`field.update_active_blocks(cur_split_dataset_idx)` -> `get_outputs` on every 2048-ray chunk), and the engine's
`store_model(model, block=b)` round trip.  The argument checks at the top need no GPU."""
import ctypes
import os
import warnings

import numpy as np
import pytest
import torch

from tests.helpers import hash_inputs, load_rig

TOL = dict(rtol=1e-4, atol=1e-5)          # test_eval_views_gpu.py's tolerance against the dense path
KEYS = ("rgb", "accumulation", "depth", "oct_depth")
W, H = 64, 48
K = 4                                     # blocks of the model tests


# ---- argument checks (no GPU) -----------------------------------------------------------------------------------------
def test_routed_gather_rejections():
    from gfnerf_b200 import _lib
    L = _lib.lib()
    p = ctypes.c_void_p(4096)

    def call(n_tables=2, tables=p, ray_id=p, ray_table=p, n=10):
        return L.gf_hash_forward_residual_routed(n, None, 1, 16, n_tables, tables, p, p, p, 0, ray_id, ray_table, p, p,
                                                 None)

    for kw in (dict(n_tables=0), dict(n_tables=-3), dict(tables=None), dict(ray_id=None), dict(ray_table=None),
               dict(n_tables=0, n=0), dict(tables=None, n=0)):
        assert call(**kw) == -1, kw
        assert b"gf_hash_forward_residual_routed" in L.gf_last_error(), kw
    assert L.gf_hash_forward_residual_routed(10, None, 1, 15, 2, p, p, p, p, 0, p, p, p, p, None) == -1   # odd size
    assert b"gf_hash_forward_residual_routed" in L.gf_last_error()


# ---- the kernel -------------------------------------------------------------------------------------------------------
def _i16(t):
    return t.view(torch.int16)


def _rays_of(n, seed, mean_len=12):
    """ray_id int32 [n] in the sampler's compact layout: consecutive samples of a ray, runs of 1..2*mean_len"""
    rng = np.random.RandomState(seed)
    lens = rng.randint(1, 2 * mean_len, size=n)
    rid = np.repeat(np.arange(n), lens)[:n]
    return torch.from_numpy(rid.astype(np.int32)).cuda(), int(rid[-1]) + 1


def _reference(tables, n_vol, local, scales, pts, anc, base, ray_id, ray_table):
    """gf_hash_forward_residual of each table on the samples routed to it; base rows elsewhere"""
    from gfnerf_b200 import _lib
    L = _lib.lib()
    out = base.clone()
    t = ray_table.long()[ray_id.long()]
    for k, (f16, prim, bias) in enumerate(tables):
        idx = (t == k).nonzero().squeeze(1)
        if idx.numel() == 0:
            continue
        p, a, b = pts[idx].contiguous(), anc[idx].contiguous(), base[idx].contiguous()
        o = torch.empty_like(b)
        _lib.check(L.gf_hash_forward_residual(idx.numel(), None, n_vol, local, _lib.ptr(f16), _lib.ptr(prim),
                                              _lib.ptr(bias), _lib.ptr(scales), _lib.ptr(p), _lib.ptr(a),
                                              int(a.dtype == torch.int64), _lib.ptr(b), _lib.ptr(o),
                                              _lib.cur_stream()), "gf_hash_forward_residual")
        out[idx] = o
    return out


def _routed(tables, n_vol, local, scales, pts, anc, base, out, ray_id, ray_table, n=None, d_n=None):
    from gfnerf_b200 import _lib
    refs = torch.tensor([[f.data_ptr(), p.data_ptr(), 0 if b is None else b.data_ptr()] for f, p, b in tables],
                        dtype=torch.int64).cuda()
    n = pts.shape[0] if n is None else n
    _lib.check(_lib.lib().gf_hash_forward_residual_routed(
        n, _lib.ptr(d_n), n_vol, local, len(tables), _lib.ptr(refs), _lib.ptr(scales), _lib.ptr(pts), _lib.ptr(anc),
        int(anc.dtype == torch.int64), _lib.ptr(ray_id), _lib.ptr(ray_table), _lib.ptr(base), _lib.ptr(out),
        _lib.cur_stream()), "gf_hash_forward_residual_routed")
    torch.cuda.synchronize()


def _cores(k, log2T, n_vol, seed):
    from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
    gen = torch.Generator().manual_seed(seed)
    cores = []
    for j in range(k):
        c = Hash3DAnchoredCore(log2T, n_vol, generator=gen)
        c.feat_pool_.data.uniform_(-0.3, 0.3)
        cores.append(c)
    return cores


def _route_cases(n_rays, k, seed):
    rng = np.random.RandomState(seed)
    per_ray = rng.randint(-1, k + 1, size=n_rays)                     # changes inside a warp; -1 and k are bad ids
    runs = (np.arange(n_rays) // 2048) % (k + 1)                       # 2048-ray runs, the last id of the cycle bad
    runs = np.where(runs == k, -1, runs)
    return {"per_ray": per_ray, "runs": runs}


@pytest.mark.gpu
@pytest.mark.parametrize("log2T", [19, 23])
def test_routed_gather_bit_exact(log2T):
    """both variants (prefetching while the rows fit the L2, the other beyond) against the per-table gather"""
    n_vol, k = 37, 3 if log2T == 19 else 2
    n = 60000
    _, _, _, pts, anc = hash_inputs(n, n_vol, 12, seed=log2T)
    cores = _cores(k, log2T, n_vol, seed=log2T)
    cores[-1].bias_pool_.uniform_(-0.5, 0.5)                            # a table with a bias pool next to zero ones
    tables = [(c.shadow(force=True), c.prim_pool_, c._bias()) for c in cores]
    assert tables[-1][2] is not None and tables[0][2] is None
    local, scales = cores[0].local_size_, cores[0].level_scales_
    tp = torch.from_numpy(pts).cuda()
    ray_id, n_rays = _rays_of(n, seed=1, mean_len=3)
    assert n_rays > 2 * 2048
    base = (torch.rand((n, 32), device="cuda") - 0.5).half()
    for anc_dt in (torch.int64, torch.int32):
        ta = torch.from_numpy(anc).cuda().to(anc_dt)
        for name, rt in _route_cases(n_rays, k, seed=log2T).items():
            ray_table = torch.from_numpy(rt.astype(np.int32)).cuda()
            ref = _reference(tables, n_vol, local, scales, tp, ta, base, ray_id, ray_table)
            out = torch.full_like(base, 7.0)
            _routed(tables, n_vol, local, scales, tp, ta, base, out, ray_id, ray_table)
            assert torch.equal(_i16(out), _i16(ref)), (name, anc_dt)
            bad = ((ray_table.long()[ray_id.long()] < 0) | (ray_table.long()[ray_id.long()] >= k))
            assert 0 < int(bad.sum()) < n and torch.equal(_i16(out[bad]), _i16(base[bad]))
            # in place (out aliases base), as the renderer calls it
            inplace = base.clone()
            _routed(tables, n_vol, local, scales, tp, ta, inplace, inplace, ray_id, ray_table)
            assert torch.equal(_i16(inplace), _i16(ref)), (name, anc_dt)


# run in a process of its own: a profiler session in this process has been seen to leave the next test module's
# sessions (tests/test_hash_gpu.py) without kernel records
_VARIANTS = """
import json, re, sys
import torch
from torch.profiler import ProfilerActivity, profile
from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
from tests.helpers import hash_inputs
seen = {}
for log2T in (19, 23):
    cores = [Hash3DAnchoredCore(log2T, 5, generator=torch.Generator().manual_seed(j)) for j in range(2)]
    _, _, _, pts, anc = hash_inputs(4096, 5, 12, seed=1)
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anc).cuda()
    rid = torch.arange(4096, dtype=torch.int32, device="cuda") // 8
    table = (torch.arange(512, dtype=torch.int32, device="cuda") % 2).contiguous()
    base = torch.zeros((4096, 32), dtype=torch.float16, device="cuda")
    refs = Hash3DAnchoredCore.table_refs(cores, "cuda")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        Hash3DAnchoredCore.launch_forward_residual_routed(cores, tp, ta, base, rid, table, refs=refs)
        torch.cuda.synchronize()
    seen[log2T] = sorted({m.group(1) for e in prof.key_averages()
                          for m in re.finditer(r"hash_fwd_routed_kernel<[^>]*, (\\w+)>", e.key)})
print(json.dumps(seen))
"""


@pytest.mark.gpu
def test_routed_variants_ran():
    """the prefetching variant at log2T 19 (the reachable rows fit the L2), the other at 23, as for the plain gather"""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-c", _VARIANTS], cwd=root, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    seen = json.loads(r.stdout.strip().splitlines()[-1])
    assert seen == {"19": ["true"], "23": ["false"]}, seen


@pytest.mark.gpu
def test_routed_gather_counts_and_non_pow2():
    """device-side count below n (rows past it untouched), n = 0, and a table size that is no power of two through
    the raw C-ABI"""
    from gfnerf_b200 import _lib
    n, n_vol, k = 9000, 5, 3
    local = 48 * 16
    _, _, _, pts, anc = hash_inputs(n, n_vol, 10, seed=3)
    rng = np.random.RandomState(5)
    scales = torch.empty(16, device="cuda")
    _lib.check(_lib.lib().gf_hash_level_scales(_lib.ptr(scales), None, _lib.cur_stream()))
    tables = []
    for j in range(k):
        _, prim, _, _, _ = hash_inputs(8, n_vol, 10, seed=20 + j)
        f16 = torch.from_numpy(rng.uniform(-1, 1, size=(16 * local, 2)).astype(np.float32)).cuda().half()
        bias = torch.from_numpy(rng.uniform(-1, 1, size=(16 * n_vol, 3)).astype(np.float32)).cuda() if j == 1 else None
        tables.append((f16.contiguous(), torch.from_numpy(prim.astype(np.int32)).cuda().contiguous(), bias))
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anc).cuda().to(torch.int32)
    ray_id, n_rays = _rays_of(n, seed=7)
    ray_table = torch.from_numpy(rng.randint(-1, k + 1, size=n_rays).astype(np.int32)).cuda()
    base = (torch.rand((n, 32), device="cuda") - 0.5).half()
    ref = _reference(tables, n_vol, local, scales, tp, ta, base, ray_id, ray_table)
    out = torch.full_like(base, 7.0)
    _routed(tables, n_vol, local, scales, tp, ta, base, out, ray_id, ray_table)
    assert torch.equal(_i16(out), _i16(ref))
    m = n - 1234
    out = torch.full_like(base, 7.0)
    _routed(tables, n_vol, local, scales, tp, ta, base, out, ray_id, ray_table,
            d_n=torch.tensor([m], dtype=torch.int32, device="cuda"))
    assert torch.equal(_i16(out[:m]), _i16(ref[:m])) and bool((out[m:] == 7.0).all())
    out = torch.full_like(base, 7.0)
    _routed(tables, n_vol, local, scales, tp, ta, base, out, ray_id, ray_table, n=0)
    assert bool((out == 7.0).all())


@pytest.mark.gpu
def test_core_method_matches_and_checks_sizes():
    from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
    n, n_vol = 5000, 7
    cores = _cores(3, 14, n_vol, seed=2)
    _, _, _, pts, anc = hash_inputs(n, n_vol, 12, seed=4)
    tp, ta = torch.from_numpy(pts).cuda(), torch.from_numpy(anc).cuda()
    ray_id, n_rays = _rays_of(n, seed=3)
    ray_table = torch.randint(0, 3, (n_rays,), dtype=torch.int32, device="cuda")
    base = (torch.rand((n, 32), device="cuda") - 0.5).half()
    got = base.clone()
    Hash3DAnchoredCore.launch_forward_residual_routed(cores, tp, ta, got, ray_id, ray_table)
    tables = [(c.shadow(), c.prim_pool_, c._bias()) for c in cores]
    ref = _reference(tables, n_vol, cores[0].local_size_, cores[0].level_scales_, tp, ta, base, ray_id, ray_table)
    assert torch.equal(_i16(got), _i16(ref))
    with pytest.raises(ValueError):
        Hash3DAnchoredCore.table_refs(cores + _cores(1, 15, n_vol, seed=9), "cuda")
    with pytest.raises(ValueError):
        Hash3DAnchoredCore.table_refs(cores + _cores(1, 14, n_vol + 1, seed=9), "cuda")


# ---- the model against the reference's per-chunk routing -------------------------------------------------------------
def make_block_model(tmp_path, hidden=64, emb=True, labels=True, log2T=14, seed=0):
    from pathlib import Path
    from tests.test_eval_views_gpu import make_model
    rig = load_rig("rig8")
    model = make_model(rig, hidden=hidden, emb=emb, log2T=log2T, seed=seed)
    f, ps = model.field, model.persampler
    f.n_blocks = K
    f.encodings_ckpt_dir = Path(tmp_path) / "encodings_ckpt"
    gen = torch.Generator(device="cuda").manual_seed(seed + 11)
    for b in range(K):
        f.add_table(b)
        pool = getattr(f, f"base_encoding_{b}").hash_3d.feat_pool_
        pool.data.copy_(torch.rand(pool.shape, generator=gen, device="cuda") * 0.6 - 0.3)
    f.set_stage("block_stage", active_block=0)
    if labels:   # K strips along x of the camera centres
        x = ps.c2w[:, 0, 3]
        ps.cameras_labels = (torch.argsort(torch.argsort(x)) * K // x.numel()).view(-1, 1).to(torch.int64)
    else:
        ps.n_split_dataset = K
    return rig, model


def block_of(model, cam):
    ps = model.persampler
    if ps.cameras_labels is not None:
        return int(ps.cameras_labels.reshape(-1)[cam])
    return min(cam // max(ps.c2w.shape[0] // ps.n_split_dataset, 1), ps.n_split_dataset - 1)


def routed_oracle(model, rb):
    """the reference's evaluation with routing: eval mode, then per 2048-ray chunk generate_ray_samples ->
    update_active_blocks(cur_split_dataset_idx) -> get_outputs"""
    import gfnerf_b200 as gf
    model.eval()
    shape = tuple(rb.origins.shape[:-1])
    flat = lambda t: None if t is None else t.reshape(int(np.prod(shape)), -1)
    o, d, cam, rel = flat(rb.origins), flat(rb.directions), flat(rb.camera_indices), flat(rb.rel_camera_indices)
    outs, used = [], []
    with torch.no_grad():
        for a in range(0, o.shape[0], 2048):
            sl = slice(a, a + 2048)
            sub = gf.RayBundle(origins=o[sl], directions=d[sl], camera_indices=cam[sl],
                               rel_camera_indices=None if rel is None else rel[sl])
            b = model.persampler.generate_ray_samples(sub).cur_split_dataset_idx
            model.field.update_active_blocks(b)
            used.append(b)
            outs.append(model.get_outputs(sub))
    return {k: torch.cat([x[k] for x in outs]).view(*shape, -1) for k in KEYS}, used


def mosaic(cams, cam_ids, rows=37, rel=False):
    """views of several cameras stacked, each after the first shifted by `rows` rows, so the camera -- and with it
    the block -- changes inside 2048-ray chunks and inside the fused chunks"""
    import gfnerf_b200 as gf
    from tests.test_eval_views_gpu import view_bundle
    parts = [view_bundle(cams, c) for c in cam_ids]
    o = torch.cat([p.origins for p in parts])[rows:]
    d = torch.cat([p.directions for p in parts])[rows:]
    ci = torch.cat([p.camera_indices for p in parts])[rows:]
    r = None
    if rel:
        r = (torch.arange(ci.numel(), device="cuda") * 7 % len(cams)).view(ci.shape)
    return gf.RayBundle(origins=o, directions=d, camera_indices=ci, rel_camera_indices=r)


def pick_cameras(model, n_cams):
    """one camera of every block, in a shuffled block order"""
    by = {}
    for c in range(n_cams):
        by.setdefault(block_of(model, c), c)
    return [by[b] for b in (2, 0, 3, 1) if b in by]


def assert_close(got, ref):
    for k in KEYS:
        assert got[k].shape == ref[k].shape, k
        assert torch.allclose(got[k], ref[k], **TOL), (k, float((got[k] - ref[k]).abs().max()))


def assert_equal(a, b):
    for k in KEYS:
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [64, 128])
@pytest.mark.parametrize("emb", [True, False])
@pytest.mark.parametrize("labels", [True, False])
def test_routed_matches_reference_routing(tmp_path, hidden, emb, labels):
    from tests.test_eval_views_gpu import make_cameras
    rig, model = make_block_model(tmp_path, hidden=hidden, emb=emb, labels=labels)
    cams = make_cameras(rig)
    ids = pick_cameras(model, len(cams))
    assert len(ids) == K
    rb = mosaic(cams, ids)
    ref, used = routed_oracle(model, rb)
    assert len(set(used)) >= 3, used                 # the bundle really crosses blocks
    f = model.field
    swapped = [b for b in range(K) if not hasattr(f, f"base_encoding_{b}")]
    assert swapped                                   # the oracle swapped tables out to disk: the render loads them
    got = model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)
    assert all(hasattr(f, f"base_encoding_{b}") for b in set(used))
    assert float(got["accumulation"].max()) > 0.5
    assert_close(got, ref)
    small = model.get_outputs_for_camera_ray_bundle(rb, chunk=1000, route_blocks=True)
    assert_equal(small, got)
    # one table for the whole bundle gives another image: the routing is what the oracle matched
    f.active_block_idxs_test = [used[0]]
    one = model.get_outputs_for_camera_ray_bundle(rb)
    assert not torch.allclose(one["rgb"], ref["rgb"], **TOL)


@pytest.mark.gpu
def test_blocks_follow_origins_with_rel_camera_indices(tmp_path):
    from tests.test_eval_views_gpu import make_cameras
    rig, model = make_block_model(tmp_path)
    cams = make_cameras(rig)
    rb = mosaic(cams, pick_cameras(model, len(cams)), rel=True)
    ref, used = routed_oracle(model, rb)
    assert len(set(used)) >= 3, used
    got = model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)
    assert_close(got, ref)
    assert_equal(model.get_outputs_for_camera_ray_bundle(rb, chunk=1000, route_blocks=True), got)


@pytest.mark.gpu
def test_single_block_routing_equals_active_block(tmp_path):
    from tests.test_eval_views_gpu import make_cameras
    rig, model = make_block_model(tmp_path)
    cams = make_cameras(rig)
    rb = mosaic(cams, [3, 17, 30])
    f, ps = model.field, model.persampler
    for b in (1, 3):
        ps.cameras_labels = torch.full_like(ps.cameras_labels, b)
        routed = model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)
        f.active_block_idxs_test = [b]
        assert_equal(routed, model.get_outputs_for_camera_ray_bundle(rb))


@pytest.mark.gpu
def test_missing_table_raises_before_any_launch(tmp_path):
    from gfnerf_b200 import _lib
    from tests.test_eval_views_gpu import make_cameras, view_bundle
    rig, model = make_block_model(tmp_path)
    cams = make_cameras(rig)
    f = model.field
    cam = pick_cameras(model, len(cams))[1]
    b = block_of(model, cam)
    f.del_table(b)                                   # neither resident nor saved
    rb = view_bundle(cams, cam)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with pytest.raises(FileNotFoundError):
        model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)
    assert _lib.launch_count() == n0


@pytest.mark.gpu
def test_init_stage_rejects_routing(tmp_path):
    from tests.test_eval_views_gpu import make_cameras, make_model, view_bundle
    rig = load_rig("rig8")
    model = make_model(rig)
    with pytest.raises(ValueError):
        model.get_outputs_for_camera_ray_bundle(view_bundle(make_cameras(rig), 0), route_blocks=True)


@pytest.mark.gpu
def test_routed_no_sync_per_chunk_and_state_untouched(tmp_path):
    from tests.test_eval_views_gpu import make_cameras
    rig, model = make_block_model(tmp_path)
    cams = make_cameras(rig)
    rb = mosaic(cams, pick_cameras(model, len(cams)))
    n = int(np.prod(rb.origins.shape[:-1]))
    s = model.persampler.sampler
    blobs = lambda: [t.clone() for t in (s.tree_nodes_gpu_, s.pers_trans_gpu_, s.tree_weight_stats_,
                                         s.tree_alpha_stats_, s.tree_visit_cnt_)]
    keep = blobs()
    model.train()
    first = model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)   # workspaces, streams, bias tests
    assert model.training
    model.eval()

    def syncs(chunk):
        torch.cuda.synchronize()
        with warnings.catch_warnings(record=True) as rec:
            warnings.simplefilter("always")
            torch.cuda.set_sync_debug_mode("warn")
            try:
                out = model.get_outputs_for_camera_ray_bundle(rb, chunk=chunk, route_blocks=True)
            finally:
                torch.cuda.set_sync_debug_mode(0)
        return len(rec), out

    one, out_one = syncs(n)
    many, out_many = syncs(512)                      # 24 chunks
    assert many <= one, (one, many)
    assert not model.training
    assert_equal(out_one, first)
    assert_equal(out_many, first)
    assert all(torch.equal(x, y) for x, y in zip(blobs(), keep))


@pytest.mark.gpu
def test_evaluate_views_routed(tmp_path):
    import gfnerf_b200 as gf
    from tests.test_eval_views_gpu import make_cameras, view_bundle
    rig, model = make_block_model(tmp_path)
    cams = make_cameras(rig)
    views = pick_cameras(model, len(cams))[:3]
    gen = torch.Generator(device="cuda").manual_seed(5)
    gts = [torch.rand((H, W, 3), generator=gen, device="cuda") for _ in views]
    _, per_image = gf.evaluate_views(model, cams, gts, camera_indices=views, route_blocks=True)
    for c, gt, m in zip(views, gts, per_image):
        own = model.get_outputs_for_camera_ray_bundle(view_bundle(cams, c), route_blocks=True)["rgb"]
        ref = gf.image_metrics(own, gt)
        assert m["psnr"] == float(ref["psnr"].item()) and m["ssim"] == float(ref["ssim"].item())
    _, plain = gf.evaluate_views(model, cams, gts, camera_indices=views)
    assert [m["psnr"] for m in plain] != [m["psnr"] for m in per_image]


# ---- engine round trip ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_engine_store_blocks_and_routed_render(tmp_path):
    from gfnerf_b200.engine import GFNeRFEngine
    from gfnerf_b200.persoctree import rig_rays
    from tests.test_eval_views_gpu import make_cameras, make_model, view_bundle
    rig = load_rig("rig8")
    model = make_model(rig)
    f, ps = model.field, model.persampler
    eng = GFNeRFEngine.from_model(model)
    with pytest.raises(ValueError):
        eng.store_model(model, block=0)              # init stage: there is no residual table
    stored = {}
    for b in (0, 1):
        eng.start_block_stage(seed=20 + b)
        for it in range(4):
            o, d, cam = rig_rays(rig["c2w"], rig["intri"], 1024, seed=60 + 10 * b + it)
            target = torch.rand((1024, 3), generator=torch.Generator().manual_seed(it)).cuda()
            eng.train_step(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), target, torch.from_numpy(cam).cuda())
        eng.store_model(model, block=b)
        assert bool(eng.res.feat_pool_.any())
        stored[b] = [t.detach().cpu().clone() for t in eng.res.States()]
        got = getattr(f, f"base_encoding_{b}").states()
        assert all(torch.equal(x.cpu(), y) for x, y in zip(got, stored[b]))
    for b in (0, 1):                                 # block 0 survived block 1's phase
        got = getattr(f, f"base_encoding_{b}").states()
        assert all(torch.equal(x.cpu(), y) for x, y in zip(got, stored[b]))
    # a training camera labelled 1: its view routed through the model == the engine's render with block 1 active
    k = 5
    labels = torch.zeros((ps.c2w.shape[0], 1), dtype=torch.int64)
    labels[k] = 1
    ps.cameras_labels = labels.cuda()
    f.set_stage("block_stage", active_block=0)
    model.eval()
    cams = make_cameras(rig)
    rb = view_bundle(cams, k)
    got = model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)
    rgb, depth, acc = eng.render_image(rb.origins.reshape(-1, 3).contiguous(), rb.directions.reshape(-1, 3).contiguous(),
                                       rel_camera_index=k)
    assert float(acc.max()) > 0.5
    assert torch.equal(got["rgb"].reshape(-1, 3), rgb)
    assert torch.equal(got["depth"].reshape(-1), depth)
    assert torch.equal(got["accumulation"].reshape(-1), acc)
    # and the tables travel through base_dir like the ranks of a focal run hand them over
    f.encodings_ckpt_dir = tmp_path / "encodings_ckpt"
    for b in (0, 1):
        f.save_table(b)
        f.del_table(b)
    again = model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True)
    assert_equal(again, got)
