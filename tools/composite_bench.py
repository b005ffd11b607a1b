"""Times gf_composite_forward and gf_composite_backward (csrc/composite.cu) alone, with CUDA events, on the sample set
of one bench.py training batch: the global workload's 8192 rays sampled on the rig20 octree at march fineness 1, as
bench.py sets it up (6.59 M samples).  Densities and colours are seeded (the kernels' run time does not depend on
their values).  The bytes each call moves (264 MB forward, 290 MB backward) exceed the 126 MB L2 of a B200, so most of
them stream from HBM; calls are timed back to back, as in a training step, without flushing L2 in between.

    python tools/composite_bench.py [--iters 200]

Prints one JSON line: the card and its power limit, the sample count, ms per call and the algorithmic bytes over that
time for each kernel."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBPS = 7.7            # HGX B200 data sheet, one GPU


def time_ms(fn, iters):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / iters


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return torch.cuda.get_device_name() + ", power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("composite_bench: needs a CUDA device")
    from bench import RAYS_PER_GPU, load_rig, make_batches
    from gfnerf_b200 import _lib
    from tests.helpers import make_sampler
    rig = load_rig()
    sampler = make_sampler(rig, mode=0, device="cuda")
    sampler.generator = torch.Generator(device="cuda").manual_seed(1234)
    sampler.ray_march_fineness_decay_end_iter_ = 0.0
    sampler.ray_march_fineness_ = 1.0
    o, d, _, _ = make_batches(rig, RAYS_PER_GPU, 1, seed=1234)[0]
    cs = sampler.sample_compact(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda())
    R, V = cs.n_rays, int(cs.total.item())
    gen = torch.Generator(device="cuda").manual_seed(0)
    sigma = torch.exp(2 * torch.randn(V, generator=gen, device="cuda"))
    rgb = torch.rand((V, 3), generator=gen, device="cuda")
    offsets, delta, t = cs.offsets, cs.delta[:V].contiguous(), cs.t[:V].contiguous()
    weights, alphas, trans = (torch.empty(V, device="cuda") for _ in range(3))
    out_rgb, depth, acc, tmax = (torch.empty((R, 3), device="cuda"), torch.empty(R, device="cuda"),
                                 torch.empty(R, device="cuda"), torch.zeros(1, device="cuda"))
    g_rgb = torch.randn((R, 3), generator=gen, device="cuda")
    d_sigma, d_rgb = torch.empty(V, device="cuda"), torch.empty((V, 3), device="cuda")
    L, st, P = _lib.lib(), _lib.cur_stream(), _lib.ptr

    def fwd():
        _lib.check(L.gf_composite_forward(R, P(offsets), P(sigma), P(delta), P(rgb), P(t), P(weights), P(alphas),
                                          P(trans), P(out_rgb), P(depth), P(acc), P(tmax), st))

    def bwd():
        _lib.check(L.gf_composite_backward(R, P(offsets), P(sigma), P(delta), P(rgb), P(trans), P(g_rgb), None, None,
                                           P(d_sigma), P(d_rgb), st))

    for _ in range(5):
        fwd()
        bwd()
    torch.cuda.synchronize()
    ms_fwd, ms_bwd = time_ms(fwd, a.iters), time_ms(bwd, a.iters)
    # the bytes bench.py's roofline table counts: per sample 28 B read + 12 B written forward, 44 B backward
    b_fwd, b_bwd = 40.0 * V + 20.0 * R, 44.0 * V + 20.0 * R
    print(json.dumps({
        "card": card(), "rays": R, "samples": V, "iters": a.iters,
        "composite_fwd_ms": round(ms_fwd, 4), "composite_bwd_ms": round(ms_bwd, 4),
        "composite_fwd_TBps": round(b_fwd / ms_fwd / 1e9, 2), "composite_bwd_TBps": round(b_bwd / ms_bwd / 1e9, 2),
        "share_of_hbm_7p7": [round(b_fwd / ms_fwd / 1e9 / HBM_TBPS, 3), round(b_bwd / ms_bwd / 1e9 / HBM_TBPS, 3)],
    }))


if __name__ == "__main__":
    main()
