"""GPU: whole-view rendering of the operator-API modules on the fused kernels
(`GFNeRFModel.get_outputs_for_camera_ray_bundle`) against the reference's own evaluation path -- `model.eval()`, then
`model.get_outputs` on consecutive 2048-ray slices (eval_num_rays_per_chunk, gfnerf/config.py:109) -- and the
held-out evaluation loop `evaluate_views`.  rig8 in VALIDATE mode (march noise of ones), 64 x 48 views."""
import warnings

import numpy as np
import pytest
import torch

from tests.helpers import load_rig, rig_octree

pytestmark = pytest.mark.gpu

W, H = 64, 48
TOL = dict(rtol=1e-4, atol=1e-5)
KEYS = ("rgb", "accumulation", "depth", "oct_depth")


def make_model(rig, hidden=64, emb=True, log2T=14, seed=0):
    import gfnerf_b200 as gf
    torch.manual_seed(seed)
    ps = gf.PersSampler(rig["c2w"], rig["intri"], rig["bounds"], bbox_levels=10, mode=1, octree=rig_octree(rig))
    field = gf.GFNeRFField(torch.zeros(2, 3), rig["c2w"].shape[0], log2_hashmap_size=log2T, hidden_dim=hidden,
                           hidden_dim_color=hidden, use_appearance_embedding=emb,
                           n_volumes=max(ps.get_n_volumes(), 1)).cuda()
    field.base_encoding_init.hash_3d.feat_pool_.data.uniform_(-0.5, 0.5)   # opaque surfaces, realistic ray lengths
    return gf.GFNeRFModel(ps, field).cuda()


def make_cameras(rig, width=W, height=H):
    import gfnerf_b200 as gf
    K = torch.from_numpy(rig["intri"]).float()
    sx, sy = width / float(2 * K[0, 0, 2]), height / float(2 * K[0, 1, 2])
    return gf.Cameras(torch.from_numpy(rig["c2w"]).float().cuda(), K[:, 0, 0] * sx, K[:, 1, 1] * sy,
                      K[:, 0, 2] * sx, K[:, 1, 2] * sy, width=width, height=height)


def view_bundle(cams, cam_idx, rel=None):
    """the [H, W] bundle of one camera; rel: per-ray rel_camera_indices [H*W] or None"""
    import gfnerf_b200 as gf
    rb = cams.generate_frame_rays(cam_idx)
    h, w = cams.height, cams.width
    return gf.RayBundle(origins=rb.origins.view(h, w, 3), directions=rb.directions.view(h, w, 3),
                        camera_indices=rb.camera_indices.view(h, w, 1),
                        rel_camera_indices=None if rel is None else rel.view(h, w, 1))


def dense_oracle(model, rb):
    """the reference's evaluation: eval mode, get_outputs on consecutive 2048-ray slices, concatenated"""
    import gfnerf_b200 as gf
    model.eval()
    shape = tuple(rb.origins.shape[:-1])
    flat = lambda t: None if t is None else t.reshape(int(np.prod(shape)), -1)
    o, d, cam, rel = flat(rb.origins), flat(rb.directions), flat(rb.camera_indices), flat(rb.rel_camera_indices)
    outs = []
    with torch.no_grad():
        for a in range(0, o.shape[0], 2048):
            sl = slice(a, a + 2048)
            outs.append(model.get_outputs(gf.RayBundle(origins=o[sl], directions=d[sl], camera_indices=cam[sl],
                                                       rel_camera_indices=None if rel is None else rel[sl])))
    return {k: torch.cat([x[k] for x in outs]).view(*shape, -1) for k in KEYS}


def assert_close(got, ref):
    for k in KEYS:
        assert got[k].shape == ref[k].shape, k
        assert torch.allclose(got[k], ref[k], **TOL), (k, float((got[k] - ref[k]).abs().max()))


@pytest.mark.parametrize("hidden", [64, 128])
@pytest.mark.parametrize("emb", [True, False])
@pytest.mark.parametrize("with_rel", [True, False])
def test_matches_dense_oracle(hidden, emb, with_rel):
    rig = load_rig("rig8")
    model = make_model(rig, hidden=hidden, emb=emb)
    cams = make_cameras(rig)
    rel = (torch.arange(W * H, device="cuda") * 7 % len(cams)) if with_rel else None
    rb = view_bundle(cams, 5, rel)
    got = model.get_outputs_for_camera_ray_bundle(rb)
    assert got["rgb"].shape == (H, W, 3) and got["depth"].shape == (H, W, 1)
    assert float(got["accumulation"].max()) > 0.5 and float(got["oct_depth"].max()) > 0   # the view sees the scene
    assert_close(got, dense_oracle(model, rb))


def test_routing_per_reference_chunk():
    """Two cameras' rays in one bundle, switching at ray 37 * 64 = 2368 (neither a multiple of 2048 nor of the fused
    chunk): the second 2048-ray chunk starts in camera A, so all of it -- B's rays too -- takes A's embedding."""
    import gfnerf_b200 as gf
    rig = load_rig("rig8")
    model = make_model(rig)
    cams = make_cameras(rig)
    a, b = view_bundle(cams, 3), view_bundle(cams, 20)
    rows = 37
    o = torch.cat([a.origins[:rows], b.origins, a.origins[rows:]])            # [2H, W, 3]: A rows, B rows, A rows
    d = torch.cat([a.directions[:rows], b.directions, a.directions[rows:]])
    ci = torch.cat([a.camera_indices[:rows], b.camera_indices, a.camera_indices[rows:]])
    rb = gf.RayBundle(origins=o, directions=d, camera_indices=ci)
    ref = dense_oracle(model, rb)
    for chunk in (1000, 32768):
        assert_close(model.get_outputs_for_camera_ray_bundle(rb, chunk=chunk), ref)
    flat = o.reshape(-1, 3)
    per_ray = model._nearest_cameras(flat)
    firsts = [model.persampler.get_nearest_split_dataset_orig(flat[k])[1] for k in range(0, flat.shape[0], 2048)]
    assert firsts == [3, 3, 20]            # chunks start at rays 0, 2048 (camera A) and 4096 (camera B)
    assert torch.equal(per_ray, torch.tensor(firsts, device="cuda").repeat_interleave(2048)[:flat.shape[0]])
    # per-ray routing of the view's own cameras gives another image: the chunk rule is what the oracle matched
    own = rb.camera_indices.reshape(-1)
    rb_own = gf.RayBundle(origins=o, directions=d, camera_indices=ci, rel_camera_indices=own.view(-1, W, 1))
    assert not torch.allclose(model.get_outputs_for_camera_ray_bundle(rb_own)["rgb"], ref["rgb"], **TOL)


def test_block_stage():
    rig = load_rig("rig8")
    model = make_model(rig)
    cams = make_cameras(rig)
    rb = view_bundle(cams, 7)
    init = model.get_outputs_for_camera_ray_bundle(rb)
    f = model.field
    f.add_table(2)
    f.set_stage("block_stage", active_block=2)
    f.base_encoding_2.hash_3d.feat_pool_.data.uniform_(-0.3, 0.3)
    got = model.get_outputs_for_camera_ray_bundle(rb)
    assert_close(got, dense_oracle(model, rb))
    assert not torch.allclose(got["rgb"], init["rgb"], **TOL)


def test_parameters_read_at_call_time():
    import gfnerf_b200 as gf
    rig = load_rig("rig8")
    model = make_model(rig, log2T=16)
    cams = make_cameras(rig)
    rb = view_bundle(cams, 11)
    before = model.get_outputs_for_camera_ray_bundle(rb)
    f = model.field
    opt = torch.optim.Adam(list(f.parameters()), lr=1e-2)
    model.train()
    o, d, ci = rb.origins.reshape(-1, 3), rb.directions.reshape(-1, 3), rb.camera_indices.reshape(-1, 1)
    out = model.get_outputs(gf.RayBundle(origins=o[:2048], directions=d[:2048], camera_indices=ci[:2048],
                                         rel_camera_indices=ci[:2048]))
    out["rgb"].mean().backward()
    opt.step()
    model.eval()
    pool = f.base_encoding_init.hash_3d.feat_pool_
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    after = model.get_outputs_for_camera_ray_bundle(rb)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown < pool.numel() * pool.element_size(), grown     # Adam state of the table alone is twice that
    assert_close(after, dense_oracle(model, rb))
    assert not torch.allclose(after["rgb"], before["rgb"], **TOL)


def test_chunking_mode_and_octree_untouched():
    rig = load_rig("rig8")
    model = make_model(rig)
    cams = make_cameras(rig)
    rb = view_bundle(cams, 9)
    s = model.persampler.sampler
    blobs = lambda: [t.clone() for t in (s.tree_nodes_gpu_, s.pers_trans_gpu_, s.tree_weight_stats_,
                                         s.tree_alpha_stats_, s.tree_visit_cnt_)]
    keep = blobs()
    model.train()
    ref = model.get_outputs_for_camera_ray_bundle(rb)
    assert model.training
    model.eval()
    for chunk in (512, 4096):
        got = model.get_outputs_for_camera_ray_bundle(rb, chunk=chunk)
        assert not model.training
        for k in KEYS:
            assert torch.equal(got[k], ref[k]), (chunk, k)
    assert all(torch.equal(x, y) for x, y in zip(blobs(), keep))


def test_no_sync_per_chunk():
    rig = load_rig("rig8")
    model = make_model(rig)
    cams = make_cameras(rig)
    rb = view_bundle(cams, 4)
    model.get_outputs_for_camera_ray_bundle(rb)          # first call: workspaces, streams, the bias-pool test

    def syncs(chunk):
        torch.cuda.synchronize()
        with warnings.catch_warnings(record=True) as rec:
            warnings.simplefilter("always")
            torch.cuda.set_sync_debug_mode("warn")
            try:
                model.get_outputs_for_camera_ray_bundle(rb, chunk=chunk)
            finally:
                torch.cuda.set_sync_debug_mode(0)
        return len(rec)

    one, many = syncs(W * H), syncs(256)                 # 1 chunk, 12 chunks
    assert many <= one, (one, many)


# GFNeRFEngine.render / render_image as they were before the render body moved into FusedRenderer
def _render_before(eng, rays_o, rays_d, rel_camera_indices=None, next_rays=None):
    with torch.cuda.device(eng.device):
        cs = eng._take_presampled(rays_o, rays_d)
        if cs is None:
            cs = eng.sampler.sample_compact(rays_o, rays_d, noise=None, slot=getattr(eng, "_cs_slot", 0))
        eng.flush()
        if next_rays is not None:
            eng._presample(next_rays[0], next_rays[1])
        _, sigma, rgb, _ = eng._field_forward(cs, eng._ray_emb(rel_camera_indices))
        out_rgb, depth, acc, _, _, _ = eng._composite(cs, sigma, rgb, keep=False)
        out_rgb = torch.nan_to_num(out_rgb).clamp_(0.0, 1.0)
    return out_rgb, depth, acc


def _render_image_before(eng, rays_o, rays_d, rel_camera_index=0, chunk=32768, sample_ahead=True):
    N = rays_o.shape[0]
    rgb = torch.empty((N, 3), dtype=torch.float32, device=eng.device)
    depth = torch.empty(N, dtype=torch.float32, device=eng.device)
    acc = torch.empty(N, dtype=torch.float32, device=eng.device)
    cam = None
    if eng.emb is not None:
        cam = torch.full((chunk,), int(rel_camera_index), dtype=torch.int64, device=eng.device)
    for a in range(0, N, chunk):
        b = min(a + chunk, N)
        nxt = (rays_o[b:b + chunk], rays_d[b:b + chunk]) if (b < N and sample_ahead) else None
        rgb[a:b], depth[a:b], acc[a:b] = _render_before(eng, rays_o[a:b], rays_d[a:b],
                                                        None if cam is None else cam[:b - a], next_rays=nxt)
    return rgb, depth, acc


@pytest.mark.parametrize("hidden", [64, 128])
def test_engine_render_unchanged(hidden):
    from gfnerf_b200.engine import GFNeRFEngine
    from gfnerf_b200.persoctree import frame_rays
    from tests.helpers import make_sampler
    rig = load_rig("rig8")
    eng = GFNeRFEngine(make_sampler(rig, mode=1), log2_table_size=14, num_images=rig["c2w"].shape[0], seed=4,
                       hidden=hidden)
    eng.enc.feat_pool_.data.uniform_(-0.5, 0.5)
    eng.enc.shadow(force=True)
    o, d = (torch.from_numpy(x).cuda() for x in frame_rays(rig["c2w"][6], rig["intri"][6], 160, 120))
    for chunk, ahead in ((4096, True), (5000, False)):
        ref = _render_image_before(eng, o, d, 6, chunk=chunk, sample_ahead=ahead)
        got = eng.render_image(o, d, 6, chunk=chunk, sample_ahead=ahead)
        for x, y in zip(got, ref):
            assert torch.equal(x, y)
    one = eng.render(o[:3000], d[:3000], torch.full((3000,), 2, device="cuda"))
    ref = _render_before(eng, o[:3000], d[:3000], torch.full((3000,), 2, device="cuda"))
    assert all(torch.equal(x, y) for x, y in zip((one.rgb, one.depth, one.accumulation), ref))


def test_evaluate_views():
    import gfnerf_b200 as gf
    rig = load_rig("rig8")
    model = make_model(rig)
    cams = make_cameras(rig)
    views = [2, 13, 40]
    f = model.field
    # ground truth from a perturbed parameter set
    saved = [p.detach().clone() for p in f.base_network.parameters()]
    gen = torch.Generator(device="cuda").manual_seed(3)
    with torch.no_grad():
        for p in f.base_network.parameters():
            p.add_(0.05 * torch.randn(p.shape, generator=gen, device="cuda"))
    gts = [model.get_outputs_for_camera_ray_bundle(view_bundle(cams, c))["rgb"].clone() for c in views]
    with torch.no_grad():
        for p, s in zip(f.base_network.parameters(), saved):
            p.copy_(s)
    gts[1] = gts[1].cpu()                                # ground truth may live on the host
    averages, per_image = gf.evaluate_views(model, cams, gts, camera_indices=views)
    assert len(per_image) == 3
    for c, gt, m in zip(views, gts, per_image):
        own = model.get_outputs_for_camera_ray_bundle(view_bundle(cams, c))["rgb"]
        ref = gf.image_metrics(own, gt.cuda())
        assert m["psnr"] == float(ref["psnr"].item()) and m["ssim"] == float(ref["ssim"].item())
        assert 0 < m["ssim"] < 1 and np.isfinite(m["psnr"])
        assert m["num_rays_per_sec"] > 0 and m["fps"] > 0
        assert m["num_rays_per_sec"] == pytest.approx(W * H * m["fps"], rel=1e-9)
    for k in ("psnr", "ssim", "num_rays_per_sec", "fps"):
        assert averages[k] == pytest.approx(np.mean([m[k] for m in per_image]), rel=1e-12)
    for k in ("psnr", "ssim"):
        assert averages[k + "_std"] == pytest.approx(np.std([m[k] for m in per_image], ddof=1), rel=1e-9)
    with pytest.raises(RuntimeError):
        gf.evaluate_views(model, cams, [torch.zeros(H, W + 1, 3)], camera_indices=[0])
