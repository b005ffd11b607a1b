#!/usr/bin/env python
"""bench.py -- training rays/sec of the GF-NeRF global stage (BASELINE.json config 2/3) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
  python bench.py --impl reference [--steps K] [--warmup W]      # the reference's own kernels on the host cores
  python bench.py ... --dump-outputs DIR                         # + what the last timed step computed, DIR/<name>.npy

A step = one full training iteration of the per-ray hot path on one batch of 8192 synthetic rays per GPU:
sample (octree traversal + march) -> hash encode -> MLP -> composite -> Charbonnier -> backward of all of it
-> [NCCL all-reduce of table / MLP / embedding gradients] -> Adam (16.8 M-entry table + MLP + embedding)
-> octree occupancy vote.  Workload: synthetic aerial rig of SURVEY.md 8(d) (400 cameras, prebuilt octree
fixture tests/golden/rig20.npz), Hash3DAnchored 16 levels log2T=19, 64-wide MLPs, training-mode march noise.

Prints ONE JSON line (rank 0).  Timing: CUDA events around exactly K steps after W warm-ups, barrier +
synchronize on both sides, max over ranks.  The per-step working set (table + Adam state 0.3 GB, sample
buffers ~1 GB) is several times the 126 MB L2, and a pool of distinct ray batches is cycled, so no L2 flush
is needed between iterations ("inputs larger than L2").
"""
import argparse
import glob
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RAYS_PER_GPU = 8192
LOG2T = 19
N_BATCHES = 8            # distinct ray batches cycled through
METRIC = "training rays/sec (fwd+bwd+optimizer), GF-NeRF global stage"


def load_rig():
    d = np.load(os.path.join(ROOT, "tests", "golden", "rig20.npz"))
    return {k: d[k] for k in d.files}


def make_batches(rig, n_rays, n_batches, seed):
    """(origins, directions, camera index, target rgb) per batch -- host arrays."""
    from gfnerf_b200.persoctree import rig_rays
    out = []
    for b in range(n_batches):
        o, d, cam = rig_rays(rig["c2w"], rig["intri"], n_rays, seed=seed * 1000 + b)
        hit = o + d * (o[:, 2:3] / np.maximum(-d[:, 2:3], 1e-3))
        target = (0.5 + 0.5 * np.sin(hit * np.array([1.3, 0.9, 0.0]) + np.array([0.0, 1.0, 2.0]))).astype(np.float32)
        out.append((o, d, cam, target))
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                r = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.rows.append([c.strip() for c in r.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle chain (a CPU restatement of the reference's kernels; the reference's own native code
# cannot be built here, SURVEY.md 8c), all host threads.
# --------------------------------------------------------------------------------------------
def oracle_step(orc, rig, state, batch):
    o, d, cam, target = batch
    R = o.shape[0]
    rng = state["rng"]
    noise = rng.uniform(0.5, 1.5, 1024 + R + 10).astype(np.float32) * np.float32(state["fineness"])
    smp = orc.sampler_get_samples(o, d, noise, rig["tree_nodes"], rig["pers_trans"])
    counts = smp["counts"]
    m = counts[:, None] > np.arange(1024)[None]
    pts01 = ((smp["warp_pts"][m] + np.float32(1.5)) * (np.float32(1.0) / np.float32(3.0))).astype(np.float32)
    anchors = smp["anchors"][m][:, 0]
    ray_id = np.repeat(np.arange(R), counts).astype(np.int32)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    feat = orc.hash_forward(state["table"], state["prim"], state["bias"], pts01, anchors, state["scales"])
    ray_emb = state["emb"][cam]
    sigma, rgb = orc.mlp_forward(state["mlp"], feat, ray_id, d, ray_emb, state["hidden"])
    delta, t = smp["dists"][m], smp["ts"][m]
    comp = orc.composite_forward(offsets, sigma, delta, rgb, t)
    loss, g_rgb = orc.charbonnier(comp["rgb"], target)
    d_sigma, d_rgb = orc.composite_backward(offsets, sigma, delta, rgb, g_rgb)
    d_feat, d_params, d_emb = orc.mlp_backward(state["mlp"], feat, ray_id, d, ray_emb, d_sigma, d_rgb, state["hidden"])
    g_table = orc.hash_backward(state["table"].shape[0] // 16, state["prim"], state["bias"], pts01, anchors, d_feat,
                                state["scales"])
    state["t"] += 1
    orc.adam_step(state["table"].reshape(-1), g_table.astype(np.float32).reshape(-1), state["m"], state["v"],
                  1e-2, 0.9, 0.999, 1e-15, state["t"])
    return loss, int(counts.sum())


def oracle_state(rig, log2T, hidden=64):
    from oracle import oracle as orc
    from tests.helpers import fast_primes
    rng = np.random.RandomState(0)
    n_vol = rig["pers_trans"].size // 576
    n = 16 * (1 << log2T) * 2
    H = hidden      # torch nn.Linear default init bounds, in the blob order of include/gfnerf_b200.h
    bound = 1 / np.sqrt(np.array([32] * (H * 33) + [H] * (16 * (H + 1)) + [63] * (H * 64) + [H] * (H * (H + 1)) + [H] * (3 * (H + 1))))
    return dict(rng=rng, fineness=1.0, table=rng.uniform(-1e-2, 1e-2, size=(n // 2, 2)).astype(np.float32),
                prim=fast_primes(16 * n_vol * 3, 7).reshape(16, n_vol, 3), bias=np.zeros((16 * n_vol, 3), np.float32),
                scales=orc.hash_level_scales(), mlp=(rng.uniform(-1, 1, size=bound.size) * bound).astype(np.float32), hidden=H,
                emb=rng.normal(size=(rig["c2w"].shape[0], 32)).astype(np.float32),
                m=np.zeros(n, np.float32), v=np.zeros(n, np.float32), t=0)


def time_oracle(rays, steps, warmup, log2T=LOG2T, hidden=64):
    from oracle import oracle as orc
    rig = load_rig()
    state = oracle_state(rig, log2T, hidden)
    batches = make_batches(rig, rays, max(2, min(4, steps)), seed=99)
    orc.set_num_threads(os.cpu_count() or 1)
    for w in range(warmup):
        oracle_step(orc, rig, state, batches[w % len(batches)])
    t0 = time.perf_counter()
    n_samples = 0
    for k in range(steps):
        _, v = oracle_step(orc, rig, state, batches[k % len(batches)])
        n_samples += v
    dt = time.perf_counter() - t0
    return rays * steps / dt, dt / steps * 1e3, orc.num_threads(), n_samples / steps


# --------------------------------------------------------------------------------------------
# CPU arm, kind "reference": the reference's OWN kernels on the host cores where the build container could compile them
# (oracle/_ref: the __global__ / __device__ bodies of Hash3DAnchored_cuda.cu and PersSampler_cuda.cu extracted at build
# time, every launch spread over all host threads), and torch on the CPU for the part of the path the reference itself
# runs as torch ops: MLPNetwork (nn.Linear stacks), trunc_exp, get_weights_f2nerf, the renderer's weighted sum,
# CharbonnierLoss, torch.optim.Adam over the whole table.  Dense like the reference: all R x 1024 slots go through the
# hash encoding and both MLPs (gfnerf/nerfacto_field.py:437-455; padding has delta = 0, hence weight 0).
# tcnn's SH-4 (un-vendored) is the oracle's restatement, evaluated per ray.
# --------------------------------------------------------------------------------------------
class ReferenceNativeCPU:
    FLAVOUR = "fma"      # g++ contracting mul+add pairs: the analogue of the nvcc -fmad=true build the reference ships

    def __init__(self, rig, log2T, hidden=64, seed=0):
        import torch
        from oracle import oracle as orc
        from oracle import ref_host as rh
        from tests.helpers import fast_primes
        self.torch, self.orc, self.rh = torch, orc, rh
        self.threads = os.cpu_count() or 1
        torch.set_num_threads(self.threads)
        rh.set_threads(self.threads, self.FLAVOUR)
        torch.manual_seed(seed)
        nn = torch.nn
        n_vol = rig["pers_trans"].size // 576
        self.local = 1 << log2T
        self.table = nn.Parameter(torch.empty(16 * self.local, 2).uniform_(-1e-2, 1e-2))     # nerfacto_field.py:200
        self.prim = fast_primes(16 * n_vol * 3, 7).reshape(16, n_vol, 3)
        self.bias = np.zeros((16 * n_vol, 3), np.float32)
        H = hidden
        self.base = nn.Sequential(nn.Linear(32, H), nn.ReLU(), nn.Linear(H, 16))               # gfnerf/mlp.py:25-57
        self.head = nn.Sequential(nn.Linear(63, H), nn.ReLU(), nn.Linear(H, H), nn.ReLU(), nn.Linear(H, 3), nn.Sigmoid())
        self.emb = nn.Embedding(rig["c2w"].shape[0], 32)
        params = [self.table] + list(self.base.parameters()) + list(self.head.parameters()) + list(self.emb.parameters())
        self.opt = torch.optim.Adam(params, lr=1e-2, eps=1e-15)                                # gfnerf/config.py:132-135
        self.nodes = np.ascontiguousarray(rig["tree_nodes"], np.uint8).copy()
        self.trans = np.ascontiguousarray(rig["pers_trans"], np.uint8)
        n_nodes = self.nodes.size // 128
        self.w_stats, self.a_stats = np.full(n_nodes, 1000, np.int64), np.full(n_nodes, 1000, np.int64)
        self.visit = np.zeros(n_nodes, np.int64)
        self.search_order = orc.search_order()
        self.rng = np.random.RandomState(seed)

        class TruncExp(torch.autograd.Function):          # nerfstudio/field_components/activations.py:23-38
            @staticmethod
            def forward(ctx, x):
                ctx.save_for_backward(x)
                return torch.exp(x)

            @staticmethod
            def backward(ctx, g):
                return g * torch.exp(ctx.saved_tensors[0].clamp(-15, 15))
        self.trunc_exp = TruncExp.apply

    # Hash3DAnchoredFunction::forward / backward (Hash3DAnchored_cuda.cu:160-239): the reference's kernels between the
    # reference's casts, done by torch as the reference does them (table -> fp16 every forward, :185; output -> fp32,
    # :195; grad * 128 -> fp16, :219; zero-filled fp16 gradient table, :221; -> fp32 / 128, :238)
    def _hash_args(self, pts01, anchors):
        import ctypes as C
        vp = lambda a: C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())
        if not hasattr(self, "_fidx"):
            self._fidx = (np.arange(16) * self.local).astype(np.int32)
            self._fsize = np.full(16, self.local, np.int32)
            self._prim32 = np.ascontiguousarray(self.prim, np.int32)
        return vp, C.c_int(pts01.shape[0]), C.c_int(self._prim32.shape[1])

    def _hash_forward(self, pts01, anchors):
        torch = self.torch
        vp, n, n_vol = self._hash_args(pts01, anchors)
        table = self.table.detach().to(torch.float16)
        out = torch.zeros((pts01.shape[0], 32), dtype=torch.float16)
        self.rh.lib(self.FLAVOUR).ref_hash_forward(n, n_vol, vp(table), vp(self._prim32), vp(self._fidx), vp(self._fsize),
                                                   vp(self.bias), vp(pts01), vp(anchors), vp(out))
        return out.float()

    def _hash_backward(self, pts01, anchors, grad):
        torch = self.torch
        vp, n, n_vol = self._hash_args(pts01, anchors)
        gin = (grad * 128.0).to(torch.float16).contiguous()
        gout = torch.zeros((16 * self.local, 2), dtype=torch.float16)
        self.rh.lib(self.FLAVOUR).ref_hash_backward(n, n_vol, vp(self._prim32), vp(self._fidx), vp(self._fsize),
                                                    vp(self.bias), vp(pts01), vp(anchors), vp(gin), vp(gout))
        return gout.float() / 128.0

    def step(self, batch):
        torch, rh = self.torch, self.rh
        o, d, cam, target = batch
        R, S = o.shape[0], 1024
        unit = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)               # PersSampler_cuda.cu:323
        noise = self.rng.uniform(0.5, 1.5, S + R + 10).astype(np.float32)                      # :380-389, fineness 1
        smp = rh.get_samples(o, unit, noise, self.nodes, self.trans, self.search_order, flavour=self.FLAVOUR)
        pts01 = ((smp["warp_pts"].reshape(-1, 3) + np.float32(1.5)) / np.float32(3.0)).astype(np.float32)
        anchors = np.ascontiguousarray(smp["anchors"].reshape(-1, 3)[:, 0])
        feat = self._hash_forward(pts01, anchors).requires_grad_(True)
        h = self.base(feat)
        sigma = self.trunc_exp(h[:, :1] + 1.0).view(R, S, 1)                                    # nerfacto_field.py:499
        sh = torch.from_numpy(self.orc.sh4(d)).view(R, 1, 16).expand(R, S, 16)
        emb = self.emb(torch.from_numpy(cam).long()).view(R, 1, 32).expand(R, S, 32)
        rgb = self.head(torch.cat([sh, h[:, 1:].view(R, S, 15), emb], -1).reshape(R * S, 63)).view(R, S, 3)
        tau = torch.from_numpy(smp["dists"]).view(R, S, 1) * sigma                               # rays.py:188-200
        alphas = 1.0 - torch.exp(-tau)
        trans = torch.exp(-torch.cat([torch.zeros(R, 1, 1), torch.cumsum(tau[:, :-1], 1)], 1))
        weights = torch.nan_to_num(alphas * trans)
        pred = (weights * rgb).sum(1)                                                            # renderers.py:97-110
        diff = pred - torch.from_numpy(target)
        loss = torch.sqrt(diff * diff + 1e-12).sum() / R                                         # losses.py:73-84
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self.table.grad = self._hash_backward(pts01, anchors, feat.grad)
        self.opt.step()
        rh.update_oct_nodes(smp["pts_idx_start_end"], np.ascontiguousarray(smp["anchors"][..., 1].reshape(-1)),
                            weights.detach().numpy().reshape(-1), alphas.detach().numpy().reshape(-1), self.nodes,
                            self.w_stats, self.a_stats, self.visit, flavour=self.FLAVOUR)
        return float(loss.detach()), int(smp["counts"].sum())


def time_reference_native(rays, steps, warmup, log2T=LOG2T, hidden=64):
    """-> (rays/s, ms/step, threads, mean valid samples per step) of ReferenceNativeCPU"""
    rig = load_rig()
    ref = ReferenceNativeCPU(rig, log2T, hidden)
    batches = make_batches(rig, rays, max(2, min(4, steps)), seed=99)
    for w in range(warmup):
        ref.step(batches[w % len(batches)])
    t0 = time.perf_counter()
    n_samples = 0
    for k in range(steps):
        loss, v = ref.step(batches[k % len(batches)])
        assert np.isfinite(loss)
        n_samples += v
    dt = time.perf_counter() - t0
    return rays * steps / dt, dt / steps * 1e3, ref.threads, n_samples / steps


def time_cpu_arm(rays, steps, warmup, hidden=64):
    """The CPU arm both legs report: the reference's own kernels (kind "reference") where oracle/_ref was built,
    otherwise -- or if anything about it fails on this box -- the oracle port (kind "port").
    -> (rays/s, ms/step, threads, samples/step, kind, note)"""
    note = None
    try:
        from oracle import ref_host as rh
        if rh.available(ReferenceNativeCPU.FLAVOUR):
            return time_reference_native(rays, steps, warmup, hidden=hidden) + ("reference", None)
        note = "oracle/_ref/libgf_ref_host_fma.so is not there (built where /root/reference exists)"
    except Exception as e:   # the baseline must never take the bench line down with it
        note = f"reference kernels failed here ({type(e).__name__}: {e})"
    return time_oracle(rays, steps, warmup, hidden=hidden) + ("port", note)


def time_reference_cpu_path():
    """BASELINE.json configs[0] -- the reference's own CPU-runnable path (nerfstudio torch hash encoding + MLPs +
    renderer, 4096 rays x 48 samples, fwd+bwd), the number the north star asks to be reported next to the GPU one:
    oracle/nerfacto_cpu.py (pinned to the reference's classes by tests/test_nerfacto_cpu.py), all host threads.
    A different workload from the GPU arm's (48 uniform samples per ray, no octree), hence its own key."""
    try:
        from oracle import nerfacto_cpu as nc
        rays_s, ms, threads = nc.time_cfg1(steps=5, warmup=2)
        return {"value": rays_s, "unit": "rays/s", "ms_per_step": ms, "cores": threads, "kind": "port",
                "workload": "BASELINE.json configs[0]: nerfstudio nerfacto, torch hash-encoding backend, "
                            "4096 rays x 48 samples, log2T=19, fwd+bwd (no optimizer), torch CPU",
                "sample": "median of 5 steps after 2 warm-ups"}
    except Exception as e:  # a reported side number must never take the bench line down with it
        return {"unavailable": f"{type(e).__name__}: {e}"}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rays = 256
    # K and W as asked, bounded so that the run ends within a few minutes (a 256-ray step of the reference's kernels
    # takes 1-2.5 s on 8-16 cores, of the oracle port ~0.7 s)
    steps, warmup = max(1, min(args.steps, 20)), max(1, min(args.warmup, 5))
    value, ms, cores, v, kind, note = time_cpu_arm(rays, steps, warmup, hidden=args.hidden)
    cpu = {"value": value, "unit": "rays/s", "cores": cores, "kind": kind, "sample": cpu_sample_text(kind, rays, v, steps, warmup)}
    if note:
        cpu["note"] = note
    if kind == "reference":      # the oracle port beside it (the round-1 / early round-2 comparator), a few steps
        pv, pms, pcores, pvs = time_oracle(rays, min(steps, 5), 1, hidden=args.hidden)
        cpu["port"] = {"value": pv, "unit": "rays/s", "cores": pcores, "ms_per_step": pms,
                       "sample": cpu_sample_text("port", rays, pvs, min(steps, 5), 1)}
    world = int(os.environ.get("WORLD_SIZE", "1"))
    emit(({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (f16 table gather / gradient atomics, like the reference)" if kind == "reference" else "f32",
        "data": "synthetic",
        "config": static_config("global", args.hidden, world, LOG2T),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cpu_reference_path": time_reference_cpu_path(),
    }))


def cpu_sample_text(kind, rays, samples, steps, warmup):
    what = ("the reference's own kernels (oracle/_ref: GetSamples, Hash3DAnchored forward / backward, UpdateOctNodes; "
            "all %d slots evaluated like the reference) + torch CPU for its torch part (MLPs, compositing, loss, dense Adam)"
            % (rays * 1024) if kind == "reference" else "the oracle port (valid samples only)")
    return (f"{rays} rays/step ({samples:.0f} valid samples) of the same workload (same rig / octree / table / MLP "
            f"shapes), {steps} steps after {warmup} warm-up(s), all host threads; {what}")


def static_config(workload, hidden, world, log2t):
    """The workload both arms are measured on -- identical in the CUDA arm's and the reference arm's JSON line, so the
    driver's config comparison sees one configuration; what a RUN did (sample counts, exchange path, ...) goes under
    `run`, the bounded sample of the CPU arm under `cpu_baseline.sample`."""
    return {"workload": workload_name(hidden) if workload == "global" else
            "GF-NeRF focal stage: frozen global Hash3DAnchored + MLPs, one zero-initialised residual "
            f"sub-encoder per GPU (log2T={log2t}), {RAYS_PER_GPU} rays/GPU/step, no gradient exchange",
            "rays_per_gpu": RAYS_PER_GPU, "log2T": log2t, "hidden": hidden,
            "slots_per_step_per_gpu": RAYS_PER_GPU * 1024,
            "l2_policy": "inputs larger than L2 (0.3 GB table+optimizer state, ~1 GB sample buffers, "
                         f"{N_BATCHES} ray batches cycled)",
            "level_addressing": "reference (level l = table rows [l*T/2, l*T/2 + T): windows overlap by half, "
                                "8.5*T of the 16*T rows reachable; DESIGN.md section 5)",
            "march_fineness": "1.0 (the steady state of the schedule: PersSampler.cpp:958-967 decays 16 -> 1 "
                              "over the first 10 k of 130 k iterations; the bench pins the other 120 k)",
            "parallelism": f"dp{world}" if world > 1 else "single GPU"}


def workload_name(hidden=64):
    return ("GF-NeRF global stage: Hash3DAnchored 16 levels log2T=19 + PersSampler (400-camera synthetic aerial rig), "
            f"{RAYS_PER_GPU} rays/GPU/step, up to 1024 samples/ray, H={hidden} MLPs, fwd+bwd+Adam")


def render_arm(args):
    """BASELINE config 5: forward-only render of 1920x1080 frames along a synthetic fly-over, log2T = 23 tables."""
    import torch
    from gfnerf_b200 import _lib
    from gfnerf_b200.engine import GFNeRFEngine
    from gfnerf_b200.persoctree import frame_rays
    from tests.helpers import make_sampler
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rig = load_rig()
    sampler = make_sampler(rig, mode=1, device=dev)
    eng = GFNeRFEngine(sampler, log2_table_size=23, num_images=rig["c2w"].shape[0], seed=0)
    eng.enc.feat_pool_.data.uniform_(-0.5, 0.5)      # post-training feature scale: opaque surfaces, realistic ray lengths
    eng.enc.shadow(force=True)
    W, H = 1920, 1080
    n_frames = 4
    frames = []
    for k in range(n_frames):                         # straight fly-over between two rig cameras
        c2w = rig["c2w"][10 + k].copy()
        o, d = frame_rays(c2w, rig["intri"][0], W, H)
        frames.append((torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)))
    steps, warmup = max(1, min(args.steps, 8)), 3
    for i in range(warmup):
        eng.render_image(*frames[i % n_frames])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _lib.launch_count()
    e0.record()
    for i in range(steps):
        rgb, depth, acc = eng.render_image(*frames[i % n_frames])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"rgb": rgb, "depth": depth, "accumulation": acc})
    emit(({
        "metric": "render rays/sec (forward only), 1920x1080 frames, log2T=23", "value": W * H / (ms * 1e-3),
        "unit": "rays/s", "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f16 tables + f16 tensor-core MLP, f32 geometry", "data": "synthetic",
        "config": {"workload": "forward-only render of 1920x1080 synthetic frames, Hash3DAnchored log2T=23, eval sampling, "
                               "32768-ray chunks", "frame_ms": ms, "fps": 1e3 / ms},
        "gpu_launches": int(_lib.launch_count() - l0),
        "check": {"rgb_mean": float(rgb.mean()), "acc_mean": float(acc.mean()), "finite": bool(torch.isfinite(rgb).all())},
    }))


def operator_api_arm(rig, dev, steps, warmup, hidden, log2t):
    """The same training iteration through the REFERENCE's operator boundary instead of the fused engine: the call
    sequence of gfnerf/nerfacto.py:522-619 (PersSampler.generate_ray_samples -> GFNeRFField -> get_weights_f2nerf ->
    RGB / depth / accumulation renderers -> octree feedback) on its dense [R, 1024] tensors, torch autograd for the
    backward, the caller's own torch.optim.Adam(lr 1e-2, eps 1e-15) (gfnerf/config.py:132-135) for the update --
    what a gf_pipeline.py user gets by swapping the reference's modules for gfnerf_b200's.  Host buffers in (pinned
    ray bundle + target, H2D inside the timed region), the loss read back every step."""
    import torch
    import gfnerf_b200 as gf
    from tests.helpers import rig_octree
    R = RAYS_PER_GPU
    ps = gf.PersSampler(rig["c2w"], rig["intri"], rig["bounds"], bbox_levels=10, mode=0, octree=rig_octree(rig),
                        ray_march_fineness_decay_end_iter=0, device=dev, seed=1234)
    field = gf.GFNeRFField(torch.zeros(2, 3), rig["c2w"].shape[0], log2_hashmap_size=log2t, hidden_dim=hidden,
                           hidden_dim_color=hidden, use_appearance_embedding=True, n_volumes=ps.get_n_volumes(),
                           generator=torch.Generator().manual_seed(0)).to(dev)
    model = gf.GFNeRFModel(ps, field).to(dev)
    model.train()
    params = list(field.base_encoding_init.get_params()) + list(field.base_network.parameters()) + \
        list(field.mlp_head.parameters()) + list(field.embedding_appearance.parameters())
    opt = torch.optim.Adam(params, lr=1e-2, eps=1e-15)
    host = make_batches(rig, R, N_BATCHES, seed=4321)
    pinned = [tuple(torch.from_numpy(a).pin_memory() for a in b) for b in host]
    ones = torch.ones(R, 1, device=dev)
    h2d = int(sum(a.numel() * a.element_size() for a in pinned[0]))

    def step(i):
        o, d, cam, tgt = (a.to(dev, non_blocking=True) for a in pinned[i % N_BATCHES])
        # steps: past the fineness decay and never on a ProcOctree milestone (every 1000), like the engine arm
        rb = gf.RayBundle(origins=o, directions=d, lookat_directions=d, pixel_area=ones, camera_indices=cam.view(-1, 1),
                          rel_camera_indices=cam.view(-1, 1), steps=torch.full((R, 1), 20001 + i % 900, device=dev))
        out = model.get_outputs(rb)
        diff = out["rgb"] - tgt
        loss = torch.sqrt(diff * diff + 1e-12).sum() / R          # CharbonnierLoss, losses.py:73-84
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return float(loss.item())                                 # D2H of the step's result

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    losses = [step(warmup + i) for i in range(steps)]
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    assert all(np.isfinite(losses)), losses
    return {"value": R / (ms * 1e-3), "unit": "rays/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
            "path": "gfnerf_b200.GFNeRFModel.get_outputs (PersSampler -> GFNeRFField -> get_weights_f2nerf -> renderers "
                    "-> UpdateOctNodes; dense [R,1024] tensors, all slots evaluated like the reference) + torch autograd "
                    "+ torch.optim.Adam: the drop-in for gfnerf/nerfacto.py:522-619 under nerfstudio's trainer"}


DUMP_TABLE_SAMPLE = 1 << 20     # hash-table entries in the dump (a fixed, seeded sample of the 16.8 M)


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy, float32 (float64 for integers), so that two builds of the project can be
    compared output for output on the same inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        a = a.astype(np.float64 if a.dtype.kind in "iub" else np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def step_arrays(out, eng):
    """What a caller of the training step receives (GFNeRFEngine.train_step's StepOutputs) and the model's parameters
    after it: MLPs, appearance embedding and a seeded sample of the hash table (the whole table is 64 MB of fp32)."""
    import torch
    table = eng.enc.feat_pool_.detach().reshape(-1)
    pick = torch.from_numpy(np.sort(np.random.RandomState(0).choice(table.numel(), min(DUMP_TABLE_SAMPLE, table.numel()),
                                                                    replace=False))).to(table.device)
    arrays = {"rgb": out.rgb, "depth": out.depth, "accumulation": out.accumulation, "loss": out.loss,
              "n_samples": out.n_samples, "mlp_params": eng.mlp, "hash_table_sample": table[pick]}
    if eng.emb is not None:
        arrays["appearance_embedding"] = eng.emb
    return arrays


# --------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def _quiet_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries (NCCL prints its version banner there) must not add to
    it: route file descriptor 1 to stderr for the whole run and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-operator-api", action="store_true",
                    help="skip the e2e_operator_api leg (the same step through GFNeRFModel.get_outputs + autograd)")
    ap.add_argument("--no-sample-ahead", action="store_true",
                    help="sample each batch at the start of its own step instead of under the previous backward")
    ap.add_argument("--workload", default="global", choices=["global", "focal", "render"],
                    help="global: BASELINE config 2/3 (the bench line).  focal: config 4 -- frozen global encoder + "
                         "one private residual sub-encoder per GPU (log2T 21), no gradient exchange.  render: config 5 "
                         "-- forward-only 1920x1080 frames, log2T 23, eval sampling; a step = one frame")
    ap.add_argument("--breakdown", action="store_true", help="print the per-kernel table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, "
                         "seeded inputs: the same arguments give the same inputs on every run)")
    ap.add_argument("--hidden", type=int, default=64, choices=[64, 128],
                    help="MLP width: 64 = the north star's / nerfstudio's default (the bench line); 128 = the "
                         "reference's shipped gf-nerf config (gfnerf/config.py:124-125)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        reference_arm(args)
        return
    args.warmup = max(args.warmup, 3)
    if args.workload == "render":
        render_arm(args)
        return

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (the hot path has no CPU fallback); "
                           "use --impl reference for the CPU restatement")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD

    from gfnerf_b200 import _lib
    from gfnerf_b200.engine import GFNeRFEngine
    from tests.helpers import make_sampler
    rig = load_rig()
    sampler = make_sampler(rig, mode=0, device=dev)
    sampler.generator = torch.Generator(device=dev).manual_seed(1234 + rank)
    # steady state of the schedule: the march fineness decays 16 -> 1 over the first 10 k of 130 k iterations
    # (PersSampler.cpp:958-967); the bench measures the fineness-1 regime the other 120 k iterations run in
    sampler.ray_march_fineness_decay_end_iter_ = 0.0
    sampler.ray_march_fineness_ = 1.0
    log2t = 21 if args.workload == "focal" else LOG2T
    # (the engine broadcasts rank 0's initial parameters when it is given a group)
    eng = GFNeRFEngine(sampler, log2_table_size=log2t, num_images=rig["c2w"].shape[0], seed=0, dist_group=group,
                       hidden=args.hidden)
    if args.workload == "focal":
        eng.start_block_stage(seed=100 + rank)

    host = make_batches(rig, RAYS_PER_GPU, N_BATCHES, seed=1234 + rank)
    pinned = [tuple(torch.from_numpy(a).pin_memory() for a in b) for b in host]
    resident = [tuple(a.to(dev, non_blocking=True) for a in b) for b in pinned]
    torch.cuda.synchronize()

    # the data loader knows the next batch: its rays are handed over one step early, so their sampling (which only
    # depends on the octree) runs underneath this step's backward pass
    ahead = not args.no_sample_ahead
    if os.environ.get("GF_PRESAMPLE_EARLY"):      # A/B: issue the next batch's sampling right after the octree vote
        eng.presample_after_mlp = False

    def step_resident(i, ahead=ahead):
        o, d, cam, tgt = resident[i % N_BATCHES]
        return eng.train_step(o, d, tgt, cam, next_rays=resident[(i + 1) % N_BATCHES][:2] if ahead else None)

    def step_e2e(i):
        # the public host-buffer entry point: pinned host batch in (H2D inside the step), the step's loss out (D2H)
        o, d, cam, tgt = pinned[i % N_BATCHES]
        return eng.train_step_host(o, d, tgt, cam, next_rays=pinned[(i + 1) % N_BATCHES][:2] if ahead else None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = []   # per timed() call: host milliseconds per step spent enqueueing (>= the device time => host-bound)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        eng.flush()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        t_host = time.perf_counter()
        for i in range(steps):
            out = fn(warmup + i)
        host_ms.append((time.perf_counter() - t_host) * 1e3 / steps)   # host time to ENQUEUE a step (no sync inside)
        eng.flush()            # the last step's (deferred, N > 1) optimizer step belongs to the timed region
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = _lib.launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, launches, out

    clocks = ClockSampler(local)
    if not os.environ.get("GF_NO_CLOCKS"):      # (A/B: does polling nvidia-smi perturb the timed region?)
        clocks.start()
    if os.environ.get("GF_MAIN_PRIO"):      # A/B: run the step on a non-default stream of the given priority
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=int(os.environ["GF_MAIN_PRIO"])))
    ms_total, launches, last = timed(step_resident, args.steps, args.warmup)
    clocks.stop_flag = True
    if args.dump_outputs and rank == 0:   # before the next leg's steps reuse the output buffers and move the parameters
        dump_outputs(args.dump_outputs, step_arrays(last, eng))
    ms_step = ms_total / args.steps
    value = RAYS_PER_GPU * world * args.steps / (ms_total * 1e-3)
    ms_e2e, _, _ = timed(step_e2e, args.steps, 3)       # the loss copies are stream-ordered: inside the timed region
    e2e_losses = eng.read_losses()
    assert len(e2e_losses) == args.steps + 3 and all(np.isfinite(e2e_losses)), e2e_losses
    e2e_value = RAYS_PER_GPU * world * args.steps / (ms_e2e * 1e-3)

    # per-kernel device times (same steps, events around every launch), for the roofline of the dominant kernel
    eng.enable_timers(True)
    n_prof = min(args.steps, 10)
    samples = 0
    for i in range(n_prof):   # one kernel at a time (no sampling ahead): the stage events need serial execution
        out = step_resident(args.warmup + args.steps + i, ahead=False)
        samples += int(out.n_samples.item())
    stages = eng.stage_times()
    eng.enable_timers(False)
    v_mean = samples / n_prof
    stage_ms = {k: t / c for k, (t, c) in stages.items()}
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "src": "fallback"}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        with open(pk) as f:
            j = json.load(f)
        peaks = {"hbm_gbs": j["hbm_gbs"], "bf16_tflops": j.get("bf16_tflops_sustained", j["bf16_tflops"]), "src": "measured"}
    # algorithmic bytes / flops per launch (DESIGN.md "roofline accounting")
    mlp_macs = float(114 * args.hidden + args.hidden * args.hidden)
    algo = {
        "hash_fwd": ("hbm", 660.0 * v_mean), "hash_bwd": ("hbm", 660.0 * v_mean),
        "sample_rays": ("hbm", 32.0 * v_mean + 24.0 * RAYS_PER_GPU), "compact": ("hbm", (32.0 + 36.0) * v_mean),
        "composite_fwd": ("hbm", (28.0 + 12.0) * v_mean + 20.0 * RAYS_PER_GPU),
        "composite_bwd": ("hbm", 44.0 * v_mean + 20.0 * RAYS_PER_GPU),
        # multiply-adds per sample of the two stacks: 32 H + 16 H + 63 H + H^2 + 3 H (11 392 at H = 64)
        "mlp_fwd": ("tensor", 2.0 * mlp_macs * v_mean), "mlp_bwd": ("tensor", 2.0 * 2.0 * mlp_macs * v_mean),
        # the 8.5 * T rows the levels can reach (the rest never gets a gradient: dense Adam leaves it untouched)
        "adam_table": ("hbm", 30.0 * 17 * (1 << log2t)),
    }
    kernels = []
    for name, ms in sorted(stage_ms.items(), key=lambda kv: -kv[1]):
        ent = {"kernel": name, "ms": round(ms, 4), "share": round(ms / sum(stage_ms.values()), 4)}
        if name in algo:
            bound, work = algo[name]
            if bound == "hbm":
                a = work / (ms * 1e-3) / 1e9
                ent.update({"bound": "hbm", "achieved": round(a, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": round(a / peaks["hbm_gbs"], 4)})
            else:
                a = work / (ms * 1e-3) / 1e12
                ent.update({"bound": "tensor", "achieved": round(a, 2), "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                            "frac": round(a / peaks["bf16_tflops"], 4)})
        kernels.append(ent)
    # DRAM traffic per launch of each kernel from the committed `ncu --set full` capture of this same command
    traffic = {}
    # the latest capture: profiles/traffic_latest.json (a copy of the newest rNN_traffic.json; tags do not sort by age)
    tp = os.path.join(ROOT, "profiles", "traffic_latest.json")
    if not os.path.exists(tp):
        tps = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
        tp = tps[-1] if tps else ""
    if tp:
        with open(tp) as f:
            cap = json.load(f)
            # kernels whose memory behaviour changed after the capture are listed as stale there: null, not a stale number
            traffic = {k: v["dram_bytes_per_launch"] for k, v in cap["kernels"].items() if k not in cap.get("stale", [])}
    for k in kernels:
        if k["kernel"] in traffic:
            k["traffic"] = traffic[k["kernel"]]
    top = next(k for k in kernels if "bound" in k)          # the dominant kernel of the step
    roofline = {k: top[k] for k in ("bound", "achieved", "peak", "unit", "frac")}
    roofline.update({"kernel": top["kernel"], "traffic": top.get("traffic"), "peak_source": peaks["src"],
                     "ms": top["ms"]})
    if top["kernel"] == "sample_rays":
        # the schema knows "hbm" and "tensor"; this kernel is neither (DESIGN.md 3.1): a serial recurrence per ray,
        # bound by instruction issue / latency, and in the step it runs a batch ahead underneath the backward pass
        roofline["note"] = ("latency-bound serial march (a recurrence in t per ray: ncu r02al ~60 % issue-active, ~265 "
                            "warp instructions per step of eight rays, 0.16 GB DRAM per launch), not HBM-bound; in the "
                            "step it runs a batch ahead on a side stream. Largest memory-bound kernels: see kernels[] "
                            "(hash_bwd: LSU data pipe / L2 atomics; hash_fwd: L1->L2 request path)")
    if top["kernel"] == "hash_bwd":
        roofline["note"] = ("effective bandwidth on ALGORITHMIC bytes (660 B per sample); the 17.8 MB of reachable table "
                            "rows are L2-resident at log2T = 19, so DRAM moves `traffic` bytes per launch (the gradient "
                            "rows in, the touched table lines once) and what bounds the kernel is the LSU data pipe and "
                            "the L2 atomic unit (ncu, steady state: l1tex data-pipe wavefronts 88.7 %, 262 M red sector "
                            "requests per launch, L2 79 %; DESIGN.md section 3)")
    if rank == 0 and args.breakdown:
        for k in kernels:
            print(k, file=sys.stderr)

    e2e_operator = None
    if rank == 0 and world == 1 and args.workload == "global" and not args.no_operator_api:
        try:
            e2e_operator = operator_api_arm(rig, dev, max(3, min(args.steps, 10)), 3, args.hidden, log2t)
        except Exception as e:   # a reported side number must never take the bench line down with it
            e2e_operator = {"unavailable": f"{type(e).__name__}: {e}"}
    cpu_baseline = cpu_reference_path = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_reference_path = time_reference_cpu_path()
        cv, cms, cores, cvs, kind, note = time_cpu_arm(256, 3, 1, hidden=args.hidden)
        cpu_baseline = {"value": cv, "unit": "rays/s", "cores": cores, "kind": kind,
                        "sample": cpu_sample_text(kind, 256, cvs, 3, 1)}
        if note:
            cpu_baseline["note"] = note
        if kind == "reference":
            pv, pms, pcores, pvs = time_oracle(256, 3, 1, hidden=args.hidden)
            cpu_baseline["port"] = {"value": pv, "unit": "rays/s", "cores": pcores,
                                    "sample": cpu_sample_text("port", 256, pvs, 3, 1)}

    if rank == 0:
        emit(({
            "metric": METRIC if args.workload == "global" else METRIC.replace("global stage", "focal stage"),
            "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16 tables + f16 tensor-core MLP, f32 accumulate / geometry / optimizer",
            "data": "synthetic",
            "config": static_config(args.workload, args.hidden, world, log2t),
            "run": {"samples_per_step_per_gpu": round(v_mean), "sample_ahead": bool(ahead),
                    # host milliseconds per step spent enqueueing the timed loops (resident, e2e).  Short runs show the
                    # host's real cost (~0.9 ms per step); in long runs the launch queue fills and the host is held
                    # back to just under the device time -- host-bound would be a value ABOVE the device time
                    "host_enqueue_ms_per_step": [round(x, 3) for x in host_ms[:2]],
                    "exchange": ("none (single GPU)" if world == 1 else "none (focal stage: private sub-encoders)"
                                 if args.workload == "focal" else
                                 "peer memory over NVLink: one kernel per rank = reduce-scatter (fp32 gradient rows, "
                                 "P2P loads) + Adam on the owned 1/N of the rows + all-gather (fp16 gather table, P2P "
                                 "stores), between two one-CTA cross-GPU barriers; octree votes: barrier + MAX over peer "
                                 "loads" if eng.peer is not None else
                                 "NCCL all-reduce of the fp32 table gradient + replicated Adam; octree votes: NCCL MAX")},
            "e2e": {"value": e2e_value, "unit": "rays/s",
                    "h2d_bytes_per_step": int(sum(a.numel() * a.element_size() for a in pinned[0])) * world,
                    "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps,
                    # the two legs of one run are different stretches of the same training run, and the hash scatter
                    # slows down over the first ~50 steps of training (fewer fp16-underflowed products to skip,
                    # DESIGN.md section 3): in a short run the later leg is slower for that reason, not because of
                    # its copies (200-step runs: e2e = resident + 0.02 ms, profiles/r02at_bench_n1.json)
                    "window": "training steps %d..%d of this run (the resident leg: %d..%d)" % (
                        args.warmup + args.steps + 3, args.warmup + 2 * args.steps + 3, args.warmup,
                        args.warmup + args.steps)},
            "e2e_operator_api": e2e_operator,
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "roofline": roofline,
            "kernels": kernels,
            "cpu_baseline": cpu_baseline,
            "cpu_reference_path": cpu_reference_path,
        }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
