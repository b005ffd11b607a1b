"""Times focal-stage training of K blocks in one step (`start_block_stage(blocks=...)`) against K single-block steps,
and the routed residual hash scatter against the single-table one.

The engine is bench.py's focal workload: rig20 octree, march fineness 1, a log2T-21 global encoder and log2T-21
residual tables, H 64, 8192 rays per block.  For each K in --blocks, one K-block step (K * 8192 rays) is timed
against K steps of a single-block engine on the same K segments, the two alternated --reps times.  The scatter is
timed on the samples of one 8192-ray batch with fp16 x128 gradients, as the engine calls it: `gf_hash_backward_levels`
into one table, `gf_hash_backward_routed` with every ray routed to one table, and routed to 8 tables in 8 contiguous
segments.

    python tools/block_train_bench.py [--blocks 1 2 4 8] [--steps 20] [--reps 3]

Prints one JSON line: the card and its power limit, and ms per step / per scatter call for each variant."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RAYS_PER_BLOCK = 8192


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return torch.cuda.get_device_name()


def per_call_ms(fn, steps, warmup=3):
    """host clock around `steps` calls that ends in a device synchronise"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps


def event_ms(fn, calls, warmup=5):
    """CUDA events around `calls` launches"""
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--log2t", type=int, default=21)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "block_train_bench needs a CUDA device"
    from gfnerf_b200.engine import GFNeRFEngine
    from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore
    from gfnerf_b200.persoctree import rig_rays
    from tests.helpers import load_rig, make_sampler

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    rig = load_rig("rig20")
    n_cam = rig["c2w"].shape[0]
    Rb = RAYS_PER_BLOCK

    def engine(blocks):
        smp = make_sampler(rig, mode=0, device=dev)
        smp.generator = torch.Generator(device=dev).manual_seed(1234)
        smp.ray_march_fineness_decay_end_iter_ = 0.0
        smp.ray_march_fineness_ = 1.0
        eng = GFNeRFEngine(smp, log2_table_size=args.log2t, num_images=n_cam, seed=0)
        eng.start_block_stage(seed=100, blocks=blocks)
        return eng

    def batch(n, seed):
        o, d, cam = rig_rays(rig["c2w"], rig["intri"], n, seed=seed)
        t = torch.rand((n, 3), generator=torch.Generator().manual_seed(seed))
        return (torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev), t.to(dev), torch.from_numpy(cam).to(dev))

    res = {"card (name, power limit)": card(), "log2T": args.log2t, "hidden": 64, "rays_per_block": Rb,
           "steps": args.steps}
    single = engine(None)
    for K in args.blocks:
        multi = engine(list(range(K)))
        batches = [batch(K * Rb, 50 + s) for s in range(2)]
        segs = [[tuple(x[k * Rb:(k + 1) * Rb] for x in b) for k in range(K)] for b in batches]
        it = {"m": 0, "s": 0}

        def multi_step():
            multi.train_step(*batches[it["m"] % 2])
            it["m"] += 1

        def single_steps():
            for s in segs[it["s"] % 2]:
                single.train_step(*s)
            it["s"] += 1

        for _ in range(args.reps):                # alternated: the host and the card are shared
            res.setdefault(f"K={K} ms per K-block step", []).append(round(per_call_ms(multi_step, args.steps), 3))
            res.setdefault(f"K={K} ms per K single-block steps", []).append(round(per_call_ms(single_steps, args.steps), 3))
        del multi
        torch.cuda.empty_cache()

    # the scatter alone, on one batch's samples
    eng = engine(list(range(8)))
    o, d, _, _ = batch(Rb, 77)
    cs = eng.sampler.sample_compact(o, d)
    V = int(cs.total.item())
    cap = cs.pts01.shape[0]
    d_feat = (torch.randn((cap, 32), device=dev) * 1e-3 * 128).half()
    ray_id = cs.ray_id
    one = torch.zeros(Rb, dtype=torch.int32, device=dev)
    eight = torch.arange(8, dtype=torch.int32, device=dev).repeat_interleave(Rb // 8)
    cores, grads = eng.res_blocks, [o_.grad for o_ in eng.opt_res_blocks]
    refs1 = Hash3DAnchoredCore.grad_refs(cores[:1], grads[:1], dev)
    refs8 = Hash3DAnchoredCore.grad_refs(cores, grads, dev)
    g0 = grads[0].view(-1, 2)
    calls = 50
    res["scatter samples"] = V
    for _ in range(args.reps):
        for name, fn in (
                ("scatter ms gf_hash_backward_levels", lambda: cores[0].launch_backward(
                    cs.pts01, cs.anchor, d_feat, True, g0, d_n_ptr=cs.total, keep_x128=True)),
                ("scatter ms routed, K=1 route", lambda: Hash3DAnchoredCore.launch_backward_routed(
                    cores[:1], cs.pts01, cs.anchor, d_feat, True, ray_id, one, refs=refs1, d_n_ptr=cs.total,
                    keep_x128=True)),
                ("scatter ms routed, K=8 contiguous segments", lambda: Hash3DAnchoredCore.launch_backward_routed(
                    cores, cs.pts01, cs.anchor, d_feat, True, ray_id, eight, refs=refs8, d_n_ptr=cs.total,
                    keep_x128=True))):
            res.setdefault(name, []).append(round(event_ms(fn, calls), 4))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
