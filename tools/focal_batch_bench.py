"""Times the pixel selection of a focal-stage step at a user-sized image set: `ErrorPixelSampler.sample` (one
torch.multinomial per 2^24-pixel chunk, host syncs) against `FocalBatchSource.next_batch()` + `update()` (sum tree,
no host read), and a whole focal step with the selection included, both ways.

The default set is BASELINE config 4's: 1600 images of 1920 x 1080 (3.3 G pixels: a 13.3 GB f32 error map beside
40 GB of f32 images).  Images and error map are seeded random values; the focal engine is bench.py's focal workload
(rig20 octree, frozen log2T-19 global encoder, log2T-21 residual table) at 8192 rays.

    python tools/focal_batch_bench.py [--images 1600] [--steps 20]

Prints one JSON line: the card and its power limit, the set's size, and ms per step for each variant."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return torch.cuda.get_device_name()


def per_step_ms(fn, steps, warmup=3):
    """host clock around `steps` calls that ends in a device synchronise (the torch path syncs inside anyway)"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1600)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--rays", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "focal_batch_bench needs a CUDA device"
    from gfnerf_b200 import pixel_samplers as ps
    from gfnerf_b200.cameras import Cameras
    from gfnerf_b200.engine import GFNeRFEngine
    from tests.helpers import load_rig, make_sampler

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    rig = load_rig("rig20")
    n_cam = rig["c2w"].shape[0]
    intri = torch.from_numpy(rig["intri"])
    cams = Cameras(torch.from_numpy(rig["c2w"]).to(dev), intri[:, 0, 0], intri[:, 1, 1], intri[:, 0, 2],
                   intri[:, 1, 2], width=args.width, height=args.height)
    n, h, w, R = args.images, args.height, args.width, args.rays
    g = torch.Generator(device=dev).manual_seed(0)
    images = torch.rand(n, h, w, 3, device=dev, generator=g)
    err = torch.rand(n, h, w, 1, device=dev, generator=g)
    image_idx = torch.arange(n, device=dev) % n_cam
    rel = image_idx.clone()
    batch = {"image": images, "error_map": err, "image_idx": image_idx, "rel_camera_idx": rel}
    sampler = ps.ErrorPixelSampler(R, generator=torch.Generator(device=dev).manual_seed(1))
    src = ps.FocalBatchSource(images, err, cams, image_idx, rel, num_rays_per_batch=R, seed=1)
    pred = torch.rand(R, 3, device=dev, generator=g)
    res = {"card (name, power limit)": card(), "images": n, "height": h, "width": w, "pixels": n * h * w,
           "error_map_GB": round(err.numel() * 4 / 1e9, 2), "rays": R, "steps": args.steps}

    def torch_select():
        b = sampler.sample(batch)
        ps.update_error_map(err, b["slot_indices"], pred, b["image"], check_indices=False)

    def source_select():
        b = src.next_batch()
        src.update(b["slot_indices"], pred)

    res["select_ms ErrorPixelSampler.sample + update_error_map"] = per_step_ms(torch_select, args.steps)
    res["select_ms FocalBatchSource.next_batch + update"] = per_step_ms(source_select, args.steps)
    src.rebuild()                                  # (the torch path wrote the map behind the source's back)

    smp = make_sampler(rig, mode=0, device=dev)
    smp.generator = torch.Generator(device=dev).manual_seed(1234)
    smp.ray_march_fineness_decay_end_iter_ = 0.0
    smp.ray_march_fineness_ = 1.0
    eng = GFNeRFEngine(smp, log2_table_size=19, num_images=n_cam, seed=0)
    eng.start_block_stage(log2_table_size=21, seed=100)

    def torch_step():
        b = sampler.sample(batch)
        ray = cams.generate_rays(b["indices"][:, 0], b["indices"][:, 1:].float() + 0.5)
        out = eng.train_step(ray.origins, ray.directions, b["image"], b["rel_camera_indices"])
        ps.update_error_map(err, b["slot_indices"], out.rgb, b["image"], check_indices=False)

    def source_step():
        b = src.next_batch()
        out = eng.train_step(b["origins"], b["directions"], b["rgb"], b["rel_camera_indices"])
        src.update(b["slot_indices"], out.rgb)

    def bare_step():
        b = src._batch
        eng.train_step(b["origins"], b["directions"], b["rgb"], b["rel_camera_indices"])

    for _ in range(2):                             # alternate the variants: the host and the card are shared
        for name, fn in (("step_ms ErrorPixelSampler path", torch_step), ("step_ms FocalBatchSource path", source_step),
                         ("step_ms train_step alone (pre-made batch)", bare_step)):
            res.setdefault(name, []).append(round(per_step_ms(fn, args.steps), 3))
            if fn is torch_step:
                src.rebuild()
    src.check()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
