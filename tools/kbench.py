"""Scratch per-kernel timing on one GPU (CUDA events, L2-sized inputs). Not the bench contract."""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gfnerf_b200 import _lib  # noqa: E402
from gfnerf_b200.hash_3d_anchored import Hash3DAnchoredCore  # noqa: E402


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def ray_run_points(n, run=256, step=1.0 / 768, n_vol=512, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n_runs = n // run
    start = torch.rand(n_runs, 1, 3, device="cuda", generator=g) * 0.4 + 0.3
    d = torch.randn(n_runs, 1, 3, device="cuda", generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    k = torch.arange(run, device="cuda").view(1, run, 1)
    pts = (start + d * k * step).reshape(-1, 3).clamp(0.0, 1.0).contiguous()
    anc = torch.randint(0, n_vol, (n_runs, 1), device="cuda", generator=g).repeat(1, run).reshape(-1).to(torch.int32)
    return pts, anc.contiguous()


def main():
    log2T = int(os.environ.get("LOG2T", 19))
    n = int(os.environ.get("N", 1 << 23))
    n_vol = 512
    core = Hash3DAnchoredCore(log2T, n_vol)
    core.Reset()
    core.shadow(force=True)
    for label, step in (("ray-runs step 1/768", 1.0 / 768), ("ray-runs step 16/768", 16.0 / 768), ("random", None)):
        if step is None:
            pts = (torch.rand(n, 3, device="cuda") * 0.66 + 0.17).contiguous()
            anc = torch.randint(0, n_vol, (n,), device="cuda", dtype=torch.int32)
        else:
            pts, anc = ray_run_points(n, step=step, n_vol=n_vol)
        out16 = torch.empty((n, 32), dtype=torch.float16, device="cuda")
        t = timeit(lambda: core.launch_forward(pts, anc, out_f16=out16, recast=False))
        print(f"hash fwd  [{label}] n={n} log2T={log2T}: {t:.3f} ms  {n/t/1e6:.2f} Gpts/s  "
              f"{660*n/t/1e6:.0f} GB/s algorithmic")
        g16 = (torch.randn((n, 32), device="cuda") * 1e-2).half()
        gt = torch.zeros_like(core.feat_pool_)
        t = timeit(lambda: core.launch_backward(pts, anc, g16, True, gt))
        print(f"hash bwd  [{label}]: {t:.3f} ms  {n/t/1e6:.2f} Gpts/s  "
              f"{660*n/t/1e6:.0f} GB/s algorithmic")
    t = timeit(lambda: core.shadow(force=True))
    print(f"cast table: {t:.3f} ms")


if __name__ == "__main__":
    main()
