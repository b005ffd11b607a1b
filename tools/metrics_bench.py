"""Times gf_image_metrics (csrc/metrics.cu) on a batch of 8 seeded 1920 x 1080 image pairs -- 398 MB of input, more
than the 126 MB L2 of a B200, so every pass reads HBM -- against a torch fp32 restatement of the torchmetrics steps
(reflect pad, grouped conv2d with the 11 x 11 Gaussian, crop, mean; MSE and PSNR), which also checks the values.

    python tools/metrics_bench.py [--batch 8] [--height 1080] [--width 1920] [--iters 20]

Prints the card and its power limit, ms per image for both, the kernel sequence's input bytes over its time, and the
per-kernel split from a separate torch.profiler pass."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_TBPS = 7.7            # HGX B200 data sheet, one GPU


def torch_metrics(p, g):
    """torchmetrics' steps in fp32 on [B,H,W,3]: PeakSignalNoiseRatio(data_range=1) and functional SSIM defaults"""
    B = p.shape[0]
    p, g = p.permute(0, 3, 1, 2), g.permute(0, 3, 1, 2)                # [B,3,H,W] views
    mse = ((p - g) ** 2).flatten(1).mean(1)
    psnr = 10 * torch.log10(1 / mse)
    d = torch.arange(11, dtype=torch.float32, device=p.device) - 5
    k1 = torch.exp(-(d / 1.5) ** 2 / 2)
    k1 = k1 / k1.sum()
    kern = (k1[:, None] @ k1[None, :]).expand(3, 1, 11, 11)
    flat = lambda t: t.flatten(1)
    L = torch.maximum(flat(p).amax(1) - flat(p).amin(1), flat(g).amax(1) - flat(g).amin(1)).view(B, 1, 1, 1)
    c1, c2 = (0.01 * L) ** 2, (0.03 * L) ** 2
    pp, gp = F.pad(p, (5, 5, 5, 5), mode="reflect"), F.pad(g, (5, 5, 5, 5), mode="reflect")
    out = F.conv2d(torch.cat([pp, gp, pp * pp, gp * gp, pp * gp]), kern, groups=3).split(B)
    mu_p, mu_g = out[0], out[1]
    s_pp, s_gg, s_pg = out[2] - mu_p ** 2, out[3] - mu_g ** 2, out[4] - mu_p * mu_g
    full = ((2 * mu_p * mu_g + c1) * (2 * s_pg + c2)) / ((mu_p ** 2 + mu_g ** 2 + c1) * (s_pp + s_gg + c2))
    ssim = full[..., 5:-5, 5:-5].flatten(1).mean(1)
    return {"psnr": psnr, "ssim": ssim, "mse": mse}


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
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("metrics_bench: needs a CUDA device")
    from gfnerf_b200 import image_metrics
    B, H, W = a.batch, a.height, a.width
    gen = torch.Generator(device="cuda").manual_seed(0)
    gt = torch.rand((B, H, W, 3), generator=gen, device="cuda")
    # a smooth rendering error plus noise: realistic SSIM values, not those of two independent noise images
    yy = torch.linspace(0, 1, H, device="cuda").view(1, H, 1, 1)
    pred = (gt + 0.05 * torch.sin(20 * yy) + 0.02 * torch.randn((B, H, W, 3), generator=gen, device="cuda"))
    pred = pred.clamp_(0, 1)
    in_bytes = 2 * B * H * W * 3 * 4

    for _ in range(3):                                                  # module load, smem opt-in, cuDNN algorithms
        ours, ref = image_metrics(pred, gt), torch_metrics(pred, gt)
    torch.cuda.synchronize()
    ms_ours = time_ms(lambda: image_metrics(pred, gt), a.iters)
    ms_torch = time_ms(lambda: torch_metrics(pred, gt), max(3, a.iters // 4))
    dev = {k: float((ours[k].double() - ref[k].double()).abs().max()) for k in ours}
    rel = {k: float(((ours[k].double() - ref[k].double()).abs() / ref[k].double().abs()).max()) for k in ("psnr", "mse")}

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            image_metrics(pred, gt)
        torch.cuda.synchronize()
    per_kernel = {}
    for e in prof.key_averages():
        if "metrics_" in e.key:
            name = e.key.split("metrics_")[1].split("(")[0]
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
            per_kernel["metrics_" + name] = round(t / 1e3 / 5, 4)      # ms per call

    res = {
        "card": card(), "batch": B, "height": H, "width": W,
        "gf_image_metrics_ms": round(ms_ours, 4), "gf_image_metrics_ms_per_image": round(ms_ours / B, 4),
        "torch_fp32_ms": round(ms_torch, 4), "torch_fp32_ms_per_image": round(ms_torch / B, 4),
        "speedup": round(ms_torch / ms_ours, 2),
        "input_bytes": in_bytes, "input_bytes_per_s_TB": round(in_bytes / ms_ours / 1e9, 3),
        "share_of_hbm_7p7": round(in_bytes / ms_ours / 1e9 / HBM_TBPS, 3),
        "per_kernel_ms": per_kernel,
        "max_abs_dev_vs_torch": dev, "max_rel_dev_vs_torch": rel,
        "ssim": [round(float(x), 6) for x in ours["ssim"]], "psnr": [round(float(x), 4) for x in ours["psnr"]],
    }
    print(f"card: {res['card']}")
    print(f"gf_image_metrics: {ms_ours:.4f} ms for {B} x {W}x{H} = {ms_ours / B:.4f} ms/image; "
          f"torch fp32 restatement: {ms_torch / B:.4f} ms/image ({res['speedup']}x)")
    print(f"input {in_bytes / 1e6:.0f} MB / kernel time = {res['input_bytes_per_s_TB']} TB/s = "
          f"{res['share_of_hbm_7p7']} of 7.7 TB/s; per kernel (ms): {per_kernel}")
    print(f"max |ours - torch|: {dev}; relative psnr/mse: {rel}")
    print(json.dumps(res))
    if dev["ssim"] > 1e-5 or rel["mse"] > 1e-5:
        sys.exit("metrics_bench: the kernel and the torch restatement disagree")


if __name__ == "__main__":
    main()
