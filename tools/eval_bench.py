"""Times whole-view evaluation renders of the operator-API modules: `GFNeRFModel.get_outputs_for_camera_ray_bundle`
(fused kernels, one call per view) against the reference-shaped loop (`model.eval()`, then `model.get_outputs` on
consecutive 2048-ray slices, eval_num_rays_per_chunk of gfnerf/config.py:109), on 1920 x 1080 views of rig20's
cameras (the 400-camera synthetic aerial rig of bench.py), at log2T 19 and 23 and hidden widths 64 and 128.  The table
is drawn from U(-0.5, 0.5) as in bench.py's render workload (opaque surfaces, realistic ray lengths); the sampler is in
VALIDATE mode.

    python tools/eval_bench.py [--views 4] [--dense-views 1] [--width 1920] [--height 1080]

Prints the card and its power limit, then per configuration: ms per view and rays/s of both paths (device-synchronised
host clock, after a warm-up view), the speed-up, and the largest difference between the two renders of the same view
per output.  A path that was not run is reported as "not measured".

    python tools/eval_bench.py --blocks K [--views 4] [--configs 19:64,19:128,21:64,21:128]

times the focal stage's evaluation across K block tables instead (`route_blocks=True`).  The model gets K residual
tables drawn from U(-0.3, 0.3), and `cameras_labels` splits rig20's cameras into K strips along x.  Per configuration:
(a) a single-camera view routed against the same view with its block set active and `route_blocks=False`, alternated;
(b) a mosaic bundle whose 2048-ray runs cycle through cameras of all K blocks, routed, against the dense 2048-ray
loop that sets `active_block_idxs_test` per chunk (tables resident, no swaps to disk), with the largest difference
between the two; (c) the routed gather alone against `gf_hash_forward_residual` on one bench batch (8192 rays of
rig20, each ray routed to its camera's block), CUDA events over many launches."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KEYS = ("rgb", "accumulation", "depth", "oct_depth")
TOL = dict(rtol=1e-4, atol=1e-5)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return torch.cuda.get_device_name() + ", power limit unknown"


def build(rig, log2T, hidden):
    import gfnerf_b200 as gf
    from tests.helpers import rig_octree
    torch.manual_seed(0)
    ps = gf.PersSampler(rig["c2w"], rig["intri"], rig["bounds"], bbox_levels=10, mode=1, octree=rig_octree(rig))
    field = gf.GFNeRFField(torch.zeros(2, 3), rig["c2w"].shape[0], log2_hashmap_size=log2T, hidden_dim=hidden,
                           hidden_dim_color=hidden, use_appearance_embedding=True,
                           n_volumes=max(ps.get_n_volumes(), 1)).cuda()
    field.base_encoding_init.hash_3d.feat_pool_.data.uniform_(-0.5, 0.5)
    model = gf.GFNeRFModel(ps, field).cuda()
    model.eval()
    return model


def cameras(rig, width, height):
    import gfnerf_b200 as gf
    K = torch.from_numpy(rig["intri"]).float()
    sx, sy = width / float(2 * K[0, 0, 2]), height / float(2 * K[0, 1, 2])
    return gf.Cameras(torch.from_numpy(rig["c2w"]).float().cuda(), K[:, 0, 0] * sx, K[:, 1, 1] * sy,
                      K[:, 0, 2] * sx, K[:, 1, 2] * sy, width=width, height=height)


def view(cams, i):
    import gfnerf_b200 as gf
    rb = cams.generate_frame_rays(i)
    h, w = cams.height, cams.width
    return gf.RayBundle(origins=rb.origins.view(h, w, 3), directions=rb.directions.view(h, w, 3),
                        camera_indices=rb.camera_indices.view(h, w, 1))


def dense(model, rb, max_rays=None):
    """the reference's loop: get_outputs on 2048-ray slices (one host sync per slice inside the field)"""
    import gfnerf_b200 as gf
    o, d, c = rb.origins.reshape(-1, 3), rb.directions.reshape(-1, 3), rb.camera_indices.reshape(-1, 1)
    n = o.shape[0] if max_rays is None else min(max_rays, o.shape[0])
    outs = []
    with torch.no_grad():
        for a in range(0, n, 2048):
            s = slice(a, min(a + 2048, n))
            outs.append(model.get_outputs(gf.RayBundle(origins=o[s], directions=d[s], camera_indices=c[s])))
    return {k: torch.cat([x[k] for x in outs]).view(*rb.origins.shape[:-1], -1) if max_rays is None else None
            for k in KEYS}


def build_blocks(rig, log2T, hidden, k):
    """build() plus k residual tables in U(-0.3, 0.3) and cameras_labels = k strips of the cameras along x"""
    model = build(rig, log2T, hidden)
    f, ps = model.field, model.persampler
    f.n_blocks = k
    gen = torch.Generator(device="cuda").manual_seed(7)
    for b in range(k):
        f.add_table(b)
        pool = getattr(f, f"base_encoding_{b}").hash_3d.feat_pool_
        pool.data.copy_(torch.rand(pool.shape, generator=gen, device="cuda") * 0.6 - 0.3)
    f.set_stage("block_stage", active_block=0)
    x = ps.c2w[:, 0, 3]
    ps.cameras_labels = (torch.argsort(torch.argsort(x)) * k // x.numel()).view(-1, 1).to(torch.int64)
    model.eval()
    return model


def mosaic(cams, cam_ids):
    """a [H, W] bundle whose consecutive 2048-ray runs come from cam_ids in turn (each run the same pixels of its
    camera's view)"""
    import gfnerf_b200 as gf
    h, w = cams.height, cams.width
    n = h * w
    run = torch.arange(n, device="cuda") // 2048
    which = torch.tensor(cam_ids, device="cuda")[run % len(cam_ids)]
    o, d = torch.empty((n, 3), device="cuda"), torch.empty((n, 3), device="cuda")
    ci = torch.empty((n, 1), dtype=torch.int64, device="cuda")
    for c in cam_ids:
        rb = cams.generate_frame_rays(c)
        m = which == c
        o[m], d[m], ci[m] = rb.origins.reshape(-1, 3)[m], rb.directions.reshape(-1, 3)[m], rb.camera_indices.reshape(-1, 1)[m]
    return gf.RayBundle(origins=o.view(h, w, 3), directions=d.view(h, w, 3), camera_indices=ci.view(h, w, 1))


def dense_routed(model, rb):
    """the reference's loop with its per-chunk block: active_block_idxs_test set per 2048-ray slice, get_outputs"""
    import gfnerf_b200 as gf
    ps, f = model.persampler, model.field
    o, d, c = rb.origins.reshape(-1, 3), rb.directions.reshape(-1, 3), rb.camera_indices.reshape(-1, 1)
    outs = []
    with torch.no_grad():
        for a in range(0, o.shape[0], 2048):
            s = slice(a, a + 2048)
            f.active_block_idxs_test = [ps.get_nearest_split_dataset(o[a])[0]]
            outs.append(model.get_outputs(gf.RayBundle(origins=o[s], directions=d[s], camera_indices=c[s])))
    return {k: torch.cat([x[k] for x in outs]).view(*rb.origins.shape[:-1], -1) for k in KEYS}


def gather_bench(model, rig, reps=200):
    """(c): ms per launch of the routed gather and of gf_hash_forward_residual on one bench batch"""
    from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
    from gfnerf_b200.persoctree import rig_rays
    f, ps = model.field, model.persampler
    o, d, cam = rig_rays(rig["c2w"], rig["intri"], 8192, seed=5)
    cs = ps.sampler.sample_compact(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda())
    V = int(cs.total.item())
    pts, anc, rid = cs.pts01[:V].contiguous(), cs.anchor[:V].contiguous(), cs.ray_id[:V].contiguous()
    cores = [getattr(f, f"base_encoding_{b}").hash_3d for b in range(f.n_blocks)]
    refs = Hash3DAnchoredCore.table_refs(cores, "cuda")
    table = ps.cameras_labels.reshape(-1)[torch.from_numpy(cam).cuda()].to(torch.int32).contiguous()
    base = torch.zeros((V, 32), dtype=torch.float16, device="cuda")
    out = torch.empty_like(base)
    runs = {"routed": lambda: Hash3DAnchoredCore.launch_forward_residual_routed(cores, pts, anc, base, rid, table,
                                                                                 out_f16=out, refs=refs),
            "single": lambda: cores[0].launch_forward_residual(pts, anc, base, out_f16=out, recast=False)}
    ms = {}
    for rnd in range(3):                                   # alternated rounds, the median kept
        for name, fn in runs.items():
            for _ in range(10):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms.setdefault(name, []).append(e0.elapsed_time(e1) / reps)
    return {"samples": V, **{f"{k}_ms": float(sorted(v)[1]) for k, v in ms.items()},
            **{f"{k}_ms_all": [round(x, 4) for x in v] for k, v in ms.items()}}


def main_blocks(a, rig, cams, dev_card):
    import numpy as np
    k = a.blocks
    n_rays = a.width * a.height
    results = []
    for cfg in a.configs.split(","):
        log2T, hidden = (int(x) for x in cfg.split(":"))
        model = build_blocks(rig, log2T, hidden, k)
        f, ps = model.field, model.persampler
        labels = ps.cameras_labels.reshape(-1).tolist()
        first_of = {}
        for c in range(10, len(labels)):
            first_of.setdefault(labels[c], c)
        cam_ids = [first_of[b] for b in range(k)]
        res = {"log2T": log2T, "hidden": hidden, "blocks": k, "width": a.width, "height": a.height}
        # (a) one camera: routed against its block set active
        ms_r, ms_a = [], []
        for i in range(a.views + 1):
            c = cam_ids[i % k]
            rb = view(cams, c)
            f.active_block_idxs_test = [labels[c]]
            got_a, t_a = timed(lambda: model.get_outputs_for_camera_ray_bundle(rb))
            got_r, t_r = timed(lambda: model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True))
            if i > 0:                                      # the first pair warms up
                ms_a.append(t_a)
                ms_r.append(t_r)
            assert torch.equal(got_a["rgb"], got_r["rgb"]), "one block routed differs from that block set active"
            del got_a, got_r
        res["a_routed_ms"], res["a_active_ms"] = float(np.median(ms_r)), float(np.median(ms_a))
        res["a_routed_ms_all"], res["a_active_ms_all"] = [round(x, 2) for x in ms_r], [round(x, 2) for x in ms_a]
        # (b) mosaic: fused routed against the dense loop with the per-chunk block
        rb = mosaic(cams, cam_ids)
        ms_m = []
        for i in range(a.views + 1):
            got, t = timed(lambda: model.get_outputs_for_camera_ray_bundle(rb, route_blocks=True))
            if i > 0:
                ms_m.append(t)
        res["b_routed_ms"] = float(np.median(ms_m))
        res["b_routed_ms_all"] = [round(x, 2) for x in ms_m]
        res["b_routed_rays_per_s"] = n_rays / (res["b_routed_ms"] * 1e-3)
        if a.dense_views > 0:
            dense_routed(model, gf_bundle_slice(rb, 16 * 2048))            # warm-up of the dense shapes
            ref, t = timed(lambda: dense_routed(model, rb))
            res["b_dense_ms"] = t
            res["b_speedup"] = t / res["b_routed_ms"]
            res["b_max_abs_diff"] = {key: float((got[key] - ref[key]).abs().max()) for key in KEYS}
            res["b_allclose_rtol1e-4_atol1e-5"] = all(bool(torch.allclose(got[key], ref[key], **TOL)) for key in KEYS)
            del ref
        else:
            res["b_dense_ms"] = res["b_speedup"] = res["b_max_abs_diff"] = "not measured"
        del got
        # (c) the gather alone
        res["c"] = gather_bench(model, rig)
        results.append(res)
        c = res["c"]
        print(f"log2T {log2T} H {hidden} K {k}: (a) one view routed {res['a_routed_ms']:.1f} ms, its block active "
              f"{res['a_active_ms']:.1f} ms; (b) mosaic routed {res['b_routed_ms']:.1f} ms"
              + (f", dense per-chunk loop {res['b_dense_ms']:.1f} ms ({res['b_speedup']:.1f}x), max |routed - dense| "
                 f"{res['b_max_abs_diff']}" if isinstance(res["b_dense_ms"], float) else ", dense not measured")
              + f"; (c) gather on {c['samples']} samples: routed {c['routed_ms']:.4f} ms, single table "
                f"{c['single_ms']:.4f} ms")
        del model
        torch.cuda.empty_cache()
    print(json.dumps({"card": dev_card, "results": results}))
    if any(r.get("b_allclose_rtol1e-4_atol1e-5") is False for r in results):
        sys.exit("eval_bench: the routed render and the dense per-chunk loop disagree")


def gf_bundle_slice(rb, n):
    import gfnerf_b200 as gf
    return gf.RayBundle(origins=rb.origins.reshape(-1, 3)[:n], directions=rb.directions.reshape(-1, 3)[:n],
                        camera_indices=rb.camera_indices.reshape(-1, 1)[:n])


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=4, help="timed fused views per configuration")
    ap.add_argument("--dense-views", type=int, default=1, help="timed dense-loop views per configuration")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--configs", default=None, help="log2T:hidden,... (default 19:64,19:128,23:64,23:128; with "
                                                    "--blocks 19:64,19:128,21:64,21:128)")
    ap.add_argument("--blocks", type=int, default=0, help="K > 0: time the focal stage's routed evaluation over K blocks")
    a = ap.parse_args()
    if a.configs is None:
        a.configs = "19:64,19:128,21:64,21:128" if a.blocks > 0 else "19:64,19:128,23:64,23:128"
    if not torch.cuda.is_available():
        sys.exit("eval_bench: needs a CUDA device")
    import numpy as np
    rig = {k: v for k, v in np.load(os.path.join(ROOT, "tests", "golden", "rig20.npz")).items()}
    cams = cameras(rig, a.width, a.height)
    n_rays = a.width * a.height
    first = 10                                     # the cameras bench.py's render workload flies along
    dev_card = card()
    print(f"card: {dev_card}")
    if a.blocks > 0:
        return main_blocks(a, rig, cams, dev_card)
    results = []
    for cfg in a.configs.split(","):
        log2T, hidden = (int(x) for x in cfg.split(":"))
        model = build(rig, log2T, hidden)
        model.get_outputs_for_camera_ray_bundle(view(cams, first))             # warm-up: workspaces, modules
        fused_ms = []
        for k in range(a.views):
            _, ms = timed(lambda: model.get_outputs_for_camera_ray_bundle(view(cams, first + k)))
            fused_ms.append(ms)
        res = {"log2T": log2T, "hidden": hidden, "width": a.width, "height": a.height,
               "fused_ms_per_view": float(np.median(fused_ms)), "fused_ms_all": [round(x, 2) for x in fused_ms]}
        res["fused_rays_per_s"] = n_rays / (res["fused_ms_per_view"] * 1e-3)
        if a.dense_views > 0:
            dense(model, view(cams, first), max_rays=16 * 2048)                 # warm-up of the dense shapes
            dense_ms, max_diff, close = [], {k: 0.0 for k in KEYS}, True
            for k in range(a.dense_views):
                rb = view(cams, first + k)
                ref, ms = timed(lambda: dense(model, rb))
                dense_ms.append(ms)
                got = model.get_outputs_for_camera_ray_bundle(rb)
                for key in KEYS:
                    max_diff[key] = max(max_diff[key], float((got[key] - ref[key]).abs().max()))
                    close = close and bool(torch.allclose(got[key], ref[key], **TOL))
                del ref, got
            res["dense_ms_per_view"] = float(np.median(dense_ms))
            res["dense_rays_per_s"] = n_rays / (res["dense_ms_per_view"] * 1e-3)
            res["speedup"] = res["dense_ms_per_view"] / res["fused_ms_per_view"]
            res["max_abs_diff"] = max_diff
            res["allclose_rtol1e-4_atol1e-5"] = close
        else:
            res["dense_ms_per_view"] = res["speedup"] = res["max_abs_diff"] = "not measured"
        results.append(res)
        dm = res["dense_ms_per_view"]
        print(f"log2T {log2T} H {hidden}: fused {res['fused_ms_per_view']:.1f} ms/view "
              f"({res['fused_rays_per_s'] / 1e6:.2f} M rays/s); dense 2048-ray loop "
              + (f"{dm:.1f} ms/view ({res['dense_rays_per_s'] / 1e6:.3f} M rays/s), speed-up {res['speedup']:.1f}x, "
                 f"max |fused - dense| {res['max_abs_diff']}, within tolerance: {res['allclose_rtol1e-4_atol1e-5']}"
                 if isinstance(dm, float) else "not measured"))
        del model
        torch.cuda.empty_cache()
    print(json.dumps({"card": dev_card, "results": results}))
    if any(r.get("allclose_rtol1e-4_atol1e-5") is False for r in results):
        sys.exit("eval_bench: the fused render and the dense loop disagree")


if __name__ == "__main__":
    main()
