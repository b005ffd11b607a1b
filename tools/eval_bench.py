"""Times whole-view evaluation renders of the operator-API modules: `GFNeRFModel.get_outputs_for_camera_ray_bundle`
(fused kernels, one call per view) against the reference-shaped loop (`model.eval()`, then `model.get_outputs` on
consecutive 2048-ray slices, eval_num_rays_per_chunk of gfnerf/config.py:109), on 1920 x 1080 views of rig20's
cameras (the 400-camera synthetic aerial rig of bench.py), at log2T 19 and 23 and hidden widths 64 and 128.  The table
is drawn from U(-0.5, 0.5) as in bench.py's render workload (opaque surfaces, realistic ray lengths); the sampler is in
VALIDATE mode.

    python tools/eval_bench.py [--views 4] [--dense-views 1] [--width 1920] [--height 1080]

Prints the card and its power limit, then per configuration: ms per view and rays/s of both paths (device-synchronised
host clock, after a warm-up view), the speed-up, and the largest difference between the two renders of the same view
per output.  A path that was not run is reported as "not measured"."""
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
    ap.add_argument("--configs", default="19:64,19:128,23:64,23:128", help="log2T:hidden,...")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("eval_bench: needs a CUDA device")
    import numpy as np
    rig = {k: v for k, v in np.load(os.path.join(ROOT, "tests", "golden", "rig20.npz")).items()}
    cams = cameras(rig, a.width, a.height)
    n_rays = a.width * a.height
    first = 10                                     # the cameras bench.py's render workload flies along
    dev_card = card()
    print(f"card: {dev_card}")
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
