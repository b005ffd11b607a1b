"""Every code path of the sampler and of the hash scatter / gather, against the CPU oracle.

The kernels run once per module on inputs built with numpy; the tests compare their outputs with the oracle's.

Sampler: adversarial rays (axis-aligned, -0.0 components, components either side of the 1e-6 slab threshold, origins
on faces, through a corner of eight leaves, inside leaves, rays that miss), noise windows that send some quads of a warp
through the guarded-intrinsic fallback and stall rays at the 1024-sample cap, small leaf caps and ray counts that leave
idle quads.  Counts / ids exact and floats within 1e-5 of the oracle.

Hash scatter: gradients small enough that every fp32 sum is exact (contributions are fp16 values / 128, multiples of
2^-31; below 2^-7 every partial sum fits the 24-bit significand), so the table must equal the oracle's fp64 sum bit for
bit whatever the summation order.  The point fixture gives every run length that selects one of the scatter's three
reductions.  At the usual 1e-3 gradient scale every row is bounded by (k-1) 2^-24 sum|c|.
"""
import re

import numpy as np
import pytest

from oracle import oracle as orc
from tests.helpers import hash_inputs, load_rig

S = 1024                                     # samples per ray (GF_MAX_SAMPLE_PER_RAY)
GLOBAL_NEAR, SAMPLE_L = np.float32(0.01), np.float32(1.0 / 256)   # tests/helpers.make_sampler
EXACT_LIMIT = 2.0 ** -7                      # largest sum|c| of a row for which every fp32 partial sum is exact


# ================================================================ sampler inputs (numpy only)
def node_table(rig):
    """centre xyz + side (byte 0), children (24), leaf flag (88), trans_idx (96) of every node"""
    nodes = rig["tree_nodes"].view(np.uint8).reshape(-1, 128)
    cs = nodes[:, :16].copy().view(np.float32)
    ch = nodes[:, 24:88].copy().view(np.int64)
    leaf = nodes[:, 88] == 1
    tr = nodes[:, 96:104].copy().view(np.int64)[:, 0]
    return cs, ch, leaf, tr


def _unit(v):
    v = np.asarray(v, np.float64)
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)


def _rig_rays(rig, n, seed):
    from gfnerf_b200.persoctree import rig_rays
    o, d, _ = rig_rays(rig["c2w"], rig["intri"], n, seed=seed)
    return o, d


def _pick_leaves(rig, count, seed):
    """leaves with a transform, one of every side length first, then random ones"""
    cs, _, leaf, tr = node_table(rig)
    ids = np.nonzero(leaf & (tr >= 0))[0]
    first = [ids[cs[ids, 3] == s][0] for s in np.unique(cs[ids, 3])]
    rest = np.random.RandomState(seed).choice(ids, size=max(0, count - len(first)), replace=False)
    return np.concatenate([first, rest])[:count]


def axis_rays(rig):
    cs, _, _, _ = node_table(rig)
    o, d = [], []
    for k, u in enumerate(_pick_leaves(rig, 9, 1)):
        c, side = cs[u, :3], cs[u, 3]
        for a in range(3):
            for s in (1.0, -1.0):
                e = np.zeros(3, np.float32)
                e[a] = s
                if k % 2:                                   # the other two components as -0.0
                    e[[b for b in range(3) if b != a]] = -0.0
                o.append(c - e * (2 * side + 3))
                d.append(e)
    # one small component just below / just above the |d| < 1e-6 slab threshold (unchanged by the normalisation)
    for u in _pick_leaves(rig, 4, 2):
        c, side = cs[u, :3], cs[u, 3]
        for a in range(3):
            b = (a + 1) % 3
            for tiny in (9.9e-7, 1.01e-6, -9.9e-7, -1.01e-6):
                e = np.zeros(3, np.float32)
                e[a] = 1.0 if tiny > 0 else -1.0
                e[b] = tiny
                p = c.copy()
                p[b] += np.float32(0.25) * side
                o.append(p - e * (2 * side + 3))
                d.append(e)
    return np.array(o, np.float32), np.array(d, np.float32)


def face_corner_rays(rig):
    cs, ch, leaf, tr = node_table(rig)
    o, d = [], []
    half = np.float32(0.5)
    for u in _pick_leaves(rig, 6, 3):
        c, side = cs[u, :3], cs[u, 3]
        for a in range(3):
            b, cc = (a + 1) % 3, (a + 2) % 3
            for s in (1.0, -1.0):
                p = c.copy()
                p[a] = c[a] + np.float32(s) * (side * half)      # exactly on the face, as get_intersection computes it
                tangent = np.zeros(3, np.float32)
                tangent[b] = 1.0
                inward = np.zeros(3, np.float32)
                inward[a] = -s
                oblique = inward.copy()
                oblique[b], oblique[cc] = 0.3, -0.2
                for e in (tangent, inward, _unit(oblique)):
                    o.append(p.copy())
                    d.append(e)
    # the corner shared by eight leaves: the centre of an interior node whose children are all leaves with a transform
    inner = [v for v in range(len(cs)) if not leaf[v] and (ch[v] >= 0).all()
             and all(leaf[w] and tr[w] >= 0 for w in ch[v])]
    assert inner, "fixture: no node with eight leaf children"
    for v in inner[:3]:
        c, side = cs[v, :3], cs[v, 3]
        for sx in (1, -1):
            for sy in (1, -1):
                for sz in (1, -1):
                    e = _unit([sx, sy, sz])
                    o.append(c - e * side)
                    d.append(e)
        for a in range(3):                                # along the edges between four of the leaves
            e = np.zeros(3, np.float32)
            e[a] = 1.0
            o.append(c - e * side)
            d.append(e)
    return np.array(o, np.float32), np.array(d, np.float32)


def other_origin_rays(rig):
    cs, _, _, _ = node_table(rig)
    rng = np.random.RandomState(4)
    o, d = [], []
    for u in _pick_leaves(rig, 12, 5):                    # inside a leaf: the march starts at global_near
        o.append(cs[u, :3].copy())
        d.append(_unit(rng.normal(size=3)))
    cams = rig["c2w"][:, :, 3]
    for k in rng.choice(cams.shape[0], size=12, replace=False):
        o.append(cams[k].copy())
        d.append(_unit(rng.normal(size=3) * [1, 1, 0.3] - [0, 0, 1]))
    # miss the root box, or start on / past it and point away
    for p, e in (([600, 600, 600], [1, 1, 1]), ([0, 0, 300], [0, 0, 1]), ([0, 0, -300], [0.1, 0, -1]),
                 ([300, 0, 0], [0, 1, 0]), ([256, 0, 0], [1, 0, 0]), ([0, -256, 5], [0.2, -1, 0]),
                 ([-400, 3, 3], [0, 0, 1]), ([0, 0, 300], [1, 0, 0])):
        o.append(np.array(p, np.float32))
        d.append(_unit(e))
    return np.array(o, np.float32), np.array(d, np.float32)


def _noise(R, runs=(), base=1.0):
    n = np.full(S + R + 10, base, np.float32)
    for lo, hi, v in runs:
        n[lo:hi] = v
    return n


def sampler_cases():
    """name -> dict(rig, o, d, noise, max_oct, scale_by_dis).  Ray r reads noise[r + k] at its k-th step."""
    r8, r20 = load_rig("rig8"), load_rig("rig20")
    cases = {}

    def add(name, o, d, rig="rig8", noise=None, max_oct=1024, sbd=1):
        R = o.shape[0]
        cases[name] = dict(rig=rig, o=np.ascontiguousarray(o, np.float32), d=np.ascontiguousarray(d, np.float32),
                           noise=_noise(R) if noise is None else noise.astype(np.float32),
                           max_oct=max_oct, sbd=sbd)

    add("axis", *axis_rays(r8))
    add("faces", *face_corner_rays(r8))
    add("origins", *other_origin_rays(r8))
    o, d = _rig_rays(r8, 40, 11)
    ax_o, ax_d = axis_rays(r8)
    o, d = np.concatenate([o, ax_o[:24]]), np.concatenate([d, ax_d[:24]])
    R = o.shape[0]
    # zeros and 1e-30 give a zero step (t stands still), 1e30 a step past every leaf: all three leave the range of the
    # fast division / square-root sequences, so those quads take the guarded intrinsics while their neighbours do not.
    # There the fast sequences happen to return the intrinsics' bits too.  They do not at FLT_MAX (finite): where the
    # step's |J d| is below 1/256 (far, large leaves, ~560 steps into these rays) step_warp / |J d| overflows, the
    # intrinsic division gives inf and ends the ray, the unguarded sequence gives NaN
    add("noise_zero_window", o, d, noise=_noise(R, [(12, 20, 0.0)]))
    add("noise_tiny_huge", o, d, noise=_noise(R, [(5, 9, 1e-30), (25, 29, 1e30), (50, 51, 0.0)]))
    add("noise_zero_tail", o, d, noise=_noise(R, [(60, S + R + 10, 0.0)]))          # stall at the cap
    add("noise_tiny_tail", o, d, noise=_noise(R, [(0, 4, 1e30), (80, S + R + 10, 1e-30)]))
    flt_max = np.finfo(np.float32).max
    add("noise_flt_max", o, d, noise=_noise(R, [(556, 566, flt_max)]))
    add("noise_flt_max_sbd0", o, d, noise=_noise(R, [(556, 566, flt_max)]), sbd=0)
    o, d = _rig_rays(r8, 48, 12)
    rng = np.random.RandomState(6)
    train_noise = rng.uniform(0.5, 1.5, S + 48 + 10).astype(np.float32)
    for mo in (1, 2, 7):
        for sbd in (1, 0):
            add(f"max_oct{mo}_sbd{sbd}", o, d, noise=train_noise, max_oct=mo, sbd=sbd)
    for R in (1, 7, 8, 9, 15, 16, 17, 55, 56, 57, 113):
        add(f"R{R}", *_rig_rays(r8, R, 100 + R))
    o, d = _rig_rays(r8, 64, 13)
    miss = rng.rand(64) < 0.5                     # long rays sharing warps with rays that miss the root box
    o[miss] = [600, 600, 600]
    d[miss] = _unit([1, 1, 1])
    add("mixed_miss", o, d)
    o, d = _rig_rays(r20, 96, 14)
    ax_o, ax_d = axis_rays(r20)
    add("rig20", np.concatenate([o, ax_o[::3]]), np.concatenate([d, ax_d[::3]]), rig="rig20",
        noise=np.random.RandomState(8).uniform(0.5, 1.5, S + 96 + ax_o[::3].shape[0] + 10))
    for c in cases.values():
        assert np.isfinite(c["o"]).all() and np.isfinite(c["d"]).all() and np.isfinite(c["noise"]).all()
    return cases


def oracle_samples(case, d_unit, rigs):
    rig = rigs[case["rig"]]
    return orc.sampler_get_samples(case["o"], d_unit, case["noise"], rig["tree_nodes"], rig["pers_trans"],
                                   global_near=GLOBAL_NEAR, sample_l=SAMPLE_L, scale_by_dis=bool(case["sbd"]),
                                   max_oct=int(case["max_oct"]))


# ================================================================ hash inputs (numpy only)
N_VOL = 3


def run_fixture(scales):
    """Points along rays, warp by warp (32 lanes), laid out so that the levels produce every run pattern the scatter
    distinguishes (see run_patterns).  An axis-aligned ray whose step is 1 / (m S_l) gives runs of exactly m lanes at
    level l; the rest are along-ray runs of random rays."""
    rng = np.random.RandomState(7)
    pts, vol = [], []

    def x_ray(level, m, lanes, shift=0.25, v=0):
        Sl = float(scales[level])
        c0 = np.floor(rng.uniform(0.2, 0.8, 3) * Sl)
        k = np.arange(lanes)
        p = np.empty((lanes, 3))
        p[:, 0] = (c0[0] + (k + shift) / m) / Sl
        p[:, 1] = (c0[1] + 0.5) / Sl
        p[:, 2] = (c0[2] + 0.5) / Sl
        return p, np.full(lanes, v)

    for level in (2, 9, 14):
        for m in (1, 2, 3, 4, 5, 8, 9, 16, 17, 32):
            p, v = x_ray(level, m, 32, v=rng.randint(N_VOL))
            pts.append(p)
            vol.append(v)
    # a run across a warp boundary: two warps of one ray, runs of 8 lanes shifted by 4
    p, v = x_ray(10, 8, 64, shift=4.25, v=1)
    pts.append(p)
    vol.append(v)
    # A-B-A in space (the ray doubles back), then the same cell under two volumes side by side and A again
    p, _ = x_ray(8, 10, 10)
    q, _ = x_ray(8, 10, 12)
    pts.append(np.concatenate([p, q[:10] + 1.0 / float(scales[8]), p[:10], p[:2]]))
    vol.append(np.zeros(32, np.int64))
    p, _ = x_ray(6, 32, 32)
    pts.append(p)
    vol.append(np.array([0] * 10 + [1] * 10 + [0] * 12))
    # along-ray samples of random rays, like the sampler emits them
    _, _, _, hp, ha = hash_inputs(640, N_VOL, 12, seed=3)
    pts.append(hp)
    vol.append(ha % N_VOL)
    pts, vol = np.concatenate(pts), np.concatenate(vol)
    n = pts.shape[0] - 11                       # n % 32 != 0: the last warp is partly idle
    return np.clip(pts[:n], 0, 1).astype(np.float32), vol[:n].astype(np.int64)


def level_keys(pts, vol, scale):
    """(cell, volume) of every point at one level, as the kernel computes it with a zero bias: floor(f32(x) f32(s))"""
    cell = np.floor(pts.astype(np.float32) * np.float32(scale)).astype(np.int64)
    return np.stack([cell[:, 0], cell[:, 1], cell[:, 2], vol], 1)


def run_patterns(pts, vol, scales):
    """The run structures the scatter sees, over all levels: runs are maximal spans of consecutive lanes of one warp
    with the same (cell, volume)."""
    n = pts.shape[0]
    lane = np.arange(n) % 32
    found = {"longest": set(), "cross_quarter": set(), "cross_warp": False, "aba": False, "two_volumes": False}
    for s in scales:
        key = level_keys(pts, vol, s)
        same_prev = np.zeros(n, bool)
        same_prev[1:] = (key[1:] == key[:-1]).all(1)
        found["cross_warp"] |= bool((same_prev & (lane == 0)).any())
        cell_same = np.zeros(n, bool)
        cell_same[1:] = (key[1:, :3] == key[:-1, :3]).all(1) & (key[1:, 3] != key[:-1, 3]) & (lane[1:] != 0)
        found["two_volumes"] |= bool(cell_same.any())
        head = ~same_prev | (lane == 0)
        for w0 in range(0, n, 32):
            h = head[w0:w0 + 32]
            starts = np.nonzero(h)[0]
            lengths = np.diff(np.append(starts, h.size))
            found["longest"].add(int(lengths.max()))
            if lengths.max() > 4:                 # the shared-memory path (runs longer than 4 lanes)
                for b in (8, 16, 24):
                    if b < h.size and not h[b]:
                        found["cross_quarter"].add(b)
            run_keys = [tuple(key[w0 + i]) for i in starts]
            found["aba"] |= len(set(run_keys)) < len(run_keys)
    return found


def cut_in_run(pts, vol, scales):
    """a device count that ends the batch in the middle of a run of the level with the longest runs"""
    key = level_keys(pts, vol, scales[0])
    for i in range(40, pts.shape[0] - 1):
        if i % 32 not in (0, 31) and (key[i - 1] == key[i]).all() and (key[i] == key[i + 1]).all():
            return i
    raise AssertionError("fixture: no run to cut")


def hash_grads(n, sigma, seed):
    rng = np.random.RandomState(seed)
    g = (rng.normal(size=(n, 32)) * sigma).astype(np.float32)
    g[rng.rand(n, 32) < 0.1] = 0.0                 # exact zeros and -0.0 inside runs
    g[rng.rand(n, 32) < 0.05] = -0.0
    return g


SIGMAS = {"e5": 1e-5, "e6": 1e-6, "e3": 1e-3}
TABLES = {"pow2": 1 << 12, "npow2": 3 << 10}         # local sizes (rows per level window)
GATHERS = {"g12": (4096, 5, 12), "g19": (16384, 37, 19)}


def hash_fixture(scales):
    pts, vol = run_fixture(scales)
    n = pts.shape[0]
    prim = hash_inputs(32, N_VOL, 4, seed=1)[1]
    rng = np.random.RandomState(9)
    bias_nz = rng.uniform(0, 1, size=(16 * N_VOL, 3)).astype(np.float32)
    inp = dict(h_pts=pts, h_vol=vol, h_prim=prim, h_bias_nz=bias_nz, h_ncut=np.int64(cut_in_run(pts, vol, scales)))
    for k, (name, sigma) in enumerate(SIGMAS.items()):
        inp["h_g_" + name] = hash_grads(n, sigma, 20 + k)
    for name, (gn, gv, l2) in GATHERS.items():
        feat, gprim, gbias, gpts, ganc = hash_inputs(gn, gv, l2, seed=gn + l2)
        gbias = np.random.RandomState(l2).uniform(0, 1, size=gbias.shape).astype(np.float32) if l2 == 12 else gbias
        inp.update({f"{name}_feat": feat, f"{name}_prim": gprim, f"{name}_bias": gbias, f"{name}_pts": gpts,
                    f"{name}_anc": ganc})
    return inp


def hash_calls():
    """(key, table, sigma, call, bias) of every backward launch; call in
    f32_i64 | f16_i32 | x128_i64 | groups_i32 | cut_i32"""
    out = []
    for tab in TABLES:
        for sg in SIGMAS:
            for call in ("f32_i64", "f16_i32", "x128_i64", "groups_i32", "cut_i32"):
                out.append((f"bw.{tab}.{sg}.{call}", tab, sg, call, False))
    for sg in ("e5", "e3"):
        out.append((f"bw.pow2.{sg}.bias", "pow2", sg, "f32_i64", True))
    return out


# ================================================================ the kernels, once
def _run_kernels(cases, inp):
    """every sampler case in both dense modes and compact, every scatter call of hash_calls() and every gather; returns
    the outputs as numpy arrays and the names of the kernels that ran"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from gfnerf_b200 import _lib
    from gfnerf_b200.perssampler import PersSamplerCore
    from tests.helpers import make_sampler

    res = {}
    dev = torch.device("cuda")
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    ar = torch.arange(S, device=dev)

    def put(key, t):
        res[key] = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)

    def dense(key, s, o, d, noise, mode):
        s.mode_ = mode
        world, warp, dirs, dists, ts, anchors, se, first = s.GetSamples(o, d, None, noise=noise)
        counts = s.last_counts_
        m = counts[:, None].long() > ar[None]
        put(key + ".counts", counts)
        put(key + ".start_end", se)
        put(key + ".first", first.reshape(-1))
        pad = {}
        for name, t in (("world", world), ("warp", warp), ("dirs", dirs), ("dists", dists), ("ts", ts),
                        ("anchors", anchors)):
            put(f"{key}.{name}", t[m])
            bits = t.view(torch.int64 if t.dtype == torch.int64 else torch.int32)
            pad[name] = int((bits[~m] != 0).sum())
        put(key + ".pad", np.array([pad[k] for k in sorted(pad)], np.int64))
        if mode == 0:
            put(key + ".n_oct", s._pending_n_oct[0])
            s._pending_n_oct = None

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        samplers = {}
        for rig in ("rig8", "rig20"):
            samplers[rig] = make_sampler(load_rig(rig), mode=1)
        for name in sorted(cases):
            c = cases[name]
            s = samplers[c["rig"]]
            s.max_oct_intersect_per_ray_ = int(c["max_oct"])
            s.scale_by_dis_ = bool(c["sbd"])
            o, d, noise = T(c["o"]), T(c["d"]), T(c["noise"])
            put(f"s.{name}.d_unit", PersSamplerCore._normalise(o, d)[1])
            for mode in (0, 1):
                dense(f"s.{name}.d{mode}", s, o, d, noise, mode)
            cs = s.sample_compact(o, d, noise=noise, want_n_oct=True)
            V = int(cs.total.item())
            key = f"s.{name}.c"
            for f in ("counts", "offsets", "total", "first_oct_dis"):
                put(f"{key}.{f}", getattr(cs, f))
            put(key + ".n_oct", s._pending_n_oct[0])
            s._pending_n_oct = None
            for f in ("pts01", "t", "delta", "anchor", "node", "ray_id"):
                put(f"{key}.{f}", getattr(cs, f)[:V])
        torch.cuda.synchronize()

        # ---- hash
        L, st, P = _lib.lib(), _lib.cur_stream(), _lib.ptr
        scales_d = torch.empty(16, device=dev)
        scales_h = np.zeros(16, np.float32)
        _lib.check(L.gf_hash_level_scales(P(scales_d), scales_h.ctypes.data, st))
        put("h.scales", scales_h)
        pts, vol = T(inp["h_pts"]), T(inp["h_vol"])
        vol32 = vol.to(torch.int32)
        prim = T(inp["h_prim"].astype(np.int32))
        bias_nz = T(inp["h_bias_nz"])
        n = pts.shape[0]
        n_dev = torch.tensor([int(inp["h_ncut"])], dtype=torch.int32, device=dev)
        for key, tab, sg, call, has_bias in hash_calls():
            local = TABLES[tab]
            g = T(inp["h_g_" + sg])
            g16 = (g * 128).half().contiguous()
            table = torch.zeros((16 * local, 2), dtype=torch.float32, device=dev)
            kind, anc_t = call.split("_")
            anc = vol if anc_t == "i64" else vol32
            grad, flags = (g, 0) if kind in ("f32", "cut") else (g16, 1)
            if kind == "x128":
                flags |= 2
            groups = ((0, 1), (1, 7), (7, 16)) if kind == "groups" else ((0, 16),)
            for l0, l1 in groups:
                _lib.check(L.gf_hash_backward_levels(
                    n, P(n_dev if kind == "cut" else None), N_VOL, local, P(prim), P(bias_nz if has_bias else None),
                    P(scales_d), P(pts), P(anc), int(anc.dtype == torch.int64), P(grad), flags, P(table), l0, l1, st))
            put(key, table)
        for name in GATHERS:
            feat16 = T(inp[name + "_feat"]).half().contiguous()
            gpts, ganc = T(inp[name + "_pts"]), T(inp[name + "_anc"])
            gprim, gbias = T(inp[name + "_prim"].astype(np.int32)), T(inp[name + "_bias"])
            out = torch.empty((gpts.shape[0], 32), device=dev)
            _lib.check(L.gf_hash_forward(gpts.shape[0], None, gprim.shape[1], feat16.shape[0] // 16, P(feat16), P(gprim),
                                         P(gbias if bool(gbias.any()) else None), P(scales_d), P(gpts), P(ganc), 1,
                                         None, P(out), st))
            put("fw." + name, out)
        torch.cuda.synchronize()
    kernels = sorted({e.key for e in prof.key_averages() if "_kernel" in e.key})
    return res, kernels


@pytest.fixture(scope="module")
def outputs():
    """inputs, kernel outputs, the kernels that ran and the oracle's sampler results"""
    cases = sampler_cases()
    inp = hash_fixture(orc.hash_level_scales())
    res, kernels = _run_kernels(cases, inp)
    rigs = {"rig8": load_rig("rig8"), "rig20": load_rig("rig20")}
    refs = {name: oracle_samples(c, res[f"s.{name}.d_unit"], rigs) for name, c in cases.items()}
    return dict(cases=cases, inp=inp, res=res, kernels=kernels, refs=refs)


def _template_args(kernels, name):
    return [m.group(1) for k in kernels for m in re.finditer(name + r"<([^>]*)>", k)]


@pytest.mark.gpu
def test_launched_instantiations(outputs, capsys):
    """the two sampler instantiations ran, and the gathers at log2T 12 and 19 (tables that fit the L2) took the
    prefetching variant.  The kernel list is printed (uncaptured) for the log."""
    kernels = outputs["kernels"]
    with capsys.disabled():
        print()
        for kern in kernels:
            print("    ", kern[:110])
    seen = {f"sample_rays_quad_kernel<{a}>" for a in _template_args(kernels, "sample_rays_quad_kernel")}
    assert seen == {"sample_rays_quad_kernel<true>", "sample_rays_quad_kernel<false>"}, seen
    prefetch = {a.split(",")[-1].strip() for a in _template_args(kernels, "hash_fwd_kernel")}
    assert prefetch == {"true"}, prefetch
    assert _template_args(kernels, "hash_bwd_kernel")


def _sample_mask(counts):
    return counts[:, None] > np.arange(S)[None]


@pytest.mark.gpu
def test_sampler_matches_oracle(outputs):
    cases, refs, res = outputs["cases"], outputs["refs"], outputs["res"]
    for name in cases:
        ref = refs[name]
        m = _sample_mask(ref["counts"])
        excl = np.concatenate([[0], np.cumsum(ref["counts"])[:-1]])
        tag = f"case {name}"
        for mode in (0, 1):
            p = f"s.{name}.d{mode}"
            assert np.array_equal(res[p + ".counts"], ref["counts"]), tag
            assert np.array_equal(res[p + ".start_end"][:, 0], excl), tag
            assert np.array_equal(res[p + ".start_end"][:, 1], excl + ref["counts"]), tag
            assert np.array_equal(res[p + ".first"].view(np.uint32), ref["first_oct_dis"].view(np.uint32)), tag
            if mode == 0:
                assert np.array_equal(res[p + ".n_oct"], ref["n_oct"]), tag
            assert np.array_equal(res[p + ".anchors"], ref["anchors"][m]), tag
            assert not res[p + ".pad"].any(), f"{tag}: padding must stay zero"
            for f, rf in (("world", "world_pts"), ("warp", "warp_pts"), ("dirs", "dirs"), ("dists", "dists"),
                          ("ts", "ts")):
                np.testing.assert_allclose(res[f"{p}.{f}"], ref[rf][m], rtol=1e-5, atol=1e-6, err_msg=f"{tag} {f}")
                if mode == 1 and res[f"{p}.{f}"].size:
                    print(f"{name} {f}: bit-equal fraction {np.mean(res[f'{p}.{f}'] == ref[rf][m]):.6f}")
        # compact == dense, bit for bit
        c, dn = f"s.{name}.c", f"s.{name}.d0"
        V = int(ref["counts"].sum())
        assert np.array_equal(res[c + ".counts"], ref["counts"]) and int(res[c + ".total"][0]) == V, tag
        assert np.array_equal(res[c + ".offsets"], np.append(excl, V)), tag
        assert np.array_equal(res[c + ".n_oct"], ref["n_oct"]), tag
        assert np.array_equal(res[c + ".first_oct_dis"].view(np.uint32), res[dn + ".first"].view(np.uint32)), tag
        pts01 = (res[dn + ".warp"] + np.float32(1.5)) * np.float32(1.0 / 3.0)
        assert np.array_equal(res[c + ".pts01"].view(np.uint32), pts01.view(np.uint32)), tag
        assert np.array_equal(res[c + ".t"].view(np.uint32), res[dn + ".ts"].view(np.uint32)), tag
        assert np.array_equal(res[c + ".delta"].view(np.uint32), res[dn + ".dists"].view(np.uint32)), tag
        assert np.array_equal(res[c + ".anchor"], res[dn + ".anchors"][:, 0]), tag
        assert np.array_equal(res[c + ".node"], res[dn + ".anchors"][:, 1]), tag
        assert np.array_equal(res[c + ".ray_id"], np.nonzero(m)[0]), tag
    # the noise windows did what they are for
    for name in ("noise_zero_tail", "noise_tiny_tail"):
        assert (refs[name]["counts"] == S).any(), name
    assert ((refs["noise_tiny_tail"]["counts"] == 0) & (refs["noise_tiny_tail"]["n_oct"] > 0)).any()
    assert np.isinf(refs["noise_flt_max_sbd0"]["dists"]).any()


def _scatter_ref(inp, scales, tab, sg, call, bias):
    local = TABLES[tab]
    n = int(inp["h_ncut"]) if call.startswith("cut") else inp["h_pts"].shape[0]
    b = inp["h_bias_nz"] if bias else np.zeros_like(inp["h_bias_nz"])
    args = (inp["h_prim"], b, inp["h_pts"][:n], inp["h_vol"][:n])
    g = inp["h_g_" + sg][:n]
    ref = orc.hash_backward(local, *args, g, scales)
    sum_abs = orc.hash_backward(local, *args, np.abs(g), scales)
    return ref, sum_abs, args, local


@pytest.mark.gpu
def test_hash_scatter_exact_sums(outputs):
    inp, res = outputs["inp"], outputs["res"]
    scales = res["h.scales"]
    for key, tab, sg, call, bias in hash_calls():
        if sg == "e3":
            continue
        ref, sum_abs, _, _ = _scatter_ref(inp, scales, tab, sg, call, bias)
        assert sum_abs.max() < EXACT_LIMIT, key
        want = ref.astype(np.float32) * np.float32(128 if call.startswith("x128") else 1)
        assert (want != 0).sum() > 1000, key
        got = res[key]
        bad = np.nonzero((got != want).any(1))[0]
        assert bad.size == 0, f"{key}: {bad.size} rows differ, first {bad[:5]}: {got[bad[:3]]} != {want[bad[:3]]}"


@pytest.mark.gpu
def test_hash_scatter_row_bound(outputs):
    """g ~ 1e-3: a sum of k terms in fp32, in any order, is within (k - 1) 2^-24 sum|c| of the exact sum"""
    inp, res = outputs["inp"], outputs["res"]
    scales = res["h.scales"]
    for key, tab, sg, call, bias in hash_calls():
        if sg != "e3":
            continue
        ref, sum_abs, args, local = _scatter_ref(inp, scales, tab, sg, call, bias)
        assert sum_abs.max() > EXACT_LIMIT, key     # outside the exact regime: the bound is what is tested
        _, idx = orc.hash_forward(np.zeros((16 * local, 2), np.float32), *args, scales, want_idx=True)
        k_row = np.bincount(idx.reshape(-1), minlength=16 * local)[:, None].astype(np.float64)
        bound = np.maximum(k_row - 1, 0) * 2.0 ** -24 * sum_abs
        unit = 128.0 if call.startswith("x128") else 1.0
        err = np.abs(res[key].astype(np.float64) / unit - ref)
        assert np.all(err <= bound), f"{key}: worst excess {(err - bound).max()}"
        assert not res[key][k_row[:, 0] == 0].any(), f"{key}: a row no sample reaches was written"


@pytest.mark.gpu
def test_hash_gather_bit_exact(outputs):
    inp, res = outputs["inp"], outputs["res"]
    scales = res["h.scales"]
    for name in GATHERS:
        ref = orc.hash_forward(inp[name + "_feat"], inp[name + "_prim"], inp[name + "_bias"], inp[name + "_pts"],
                               inp[name + "_anc"], scales)
        assert np.array_equal(res["fw." + name], ref), f"gather {name}"


# ================================================================ CPU checks of the fixtures
def test_run_fixture_covers_every_pattern():
    scales = orc.hash_level_scales()
    pts, vol = run_fixture(scales)
    f = run_patterns(pts, vol, scales)
    assert {1, 2, 3, 4, 5, 8, 9, 16, 17, 32} <= f["longest"], sorted(f["longest"])
    assert f["cross_quarter"] == {8, 16, 24}
    assert f["cross_warp"] and f["aba"] and f["two_volumes"], f
    assert pts.shape[0] % 32 != 0
    i = cut_in_run(pts, vol, scales)
    key = level_keys(pts, vol, scales[0])
    assert (key[i - 1] == key[i]).all() and i // 32 == (i - 1) // 32


def test_exact_regime_precondition():
    """the small gradient sets keep every row's sum|c| below 2^-7 (so the fp32 table sums are exact); 1e-3 does not"""
    scales = orc.hash_level_scales()
    inp = hash_fixture(scales)
    for key, tab, sg, call, bias in hash_calls():
        _, sum_abs, _, _ = _scatter_ref(inp, scales, tab, sg, call, bias)
        if sg == "e3":
            assert sum_abs.max() > EXACT_LIMIT, key
        else:
            assert sum_abs.max() < EXACT_LIMIT, (key, sum_abs.max())
    g6 = inp["h_g_e6"]
    assert (np.abs(g6 * 128) < 2.0 ** -14).any()                  # fp16 subnormals before the weights
    assert (np.signbit(g6) & (g6 == 0)).any() and ((g6 == 0) & ~np.signbit(g6)).any()


def test_adversarial_rays_reach_the_cap_and_zero():
    """on the oracle (directions normalised on the host): the noise windows stall rays at the 1024-sample cap at a
    constant t, end rays that do meet a leaf with no sample, and the other fixtures reach their branches"""
    cases = sampler_cases()
    rigs = {"rig8": load_rig("rig8"), "rig20": load_rig("rig20")}
    refs = {name: oracle_samples(c, _unit(c["d"]), rigs) for name, c in cases.items()}
    stalled = 0
    for name in ("noise_zero_tail", "noise_tiny_tail"):
        r = refs[name]
        cap = np.nonzero(r["counts"] == S)[0]
        assert cap.size > 0, name
        stalled += cap.size
        assert (r["ts"][cap, -1] == r["ts"][cap, -2]).all(), name
    zero = refs["noise_tiny_tail"]
    # FLT_MAX noise: without the distance scale an infinite step is an overflowing division step_warp / |J d|, where
    # the unguarded division sequence returns NaN; with it, some rays still end there
    for name in ("noise_flt_max_sbd0", "noise_flt_max"):
        inf_rays = np.isinf(refs[name]["dists"]).any(1)
        assert inf_rays.any() and (~inf_rays & (refs[name]["counts"] > 0)).any(), name
    assert ((zero["counts"] == 0) & (zero["n_oct"] > 0)).sum() >= 1
    ax = cases["axis"]["d"]
    assert (np.signbit(ax) & (ax == 0)).any() and ((np.abs(ax) > 0) & (np.abs(ax) < 1e-6)).any()
    assert ((np.abs(ax) > 1e-6) & (np.abs(ax) < 1.1e-6)).any()
    assert (refs["axis"]["counts"] > 0).all()
    for name in ("faces", "origins", "mixed_miss"):
        c = refs[name]["counts"]
        assert (c > 0).any() and (c == 0).any(), name
    for mo in (1, 2, 7):
        assert refs[f"max_oct{mo}_sbd1"]["n_oct"].max() == mo
    assert refs["rig20"]["counts"].max() > 0
    print("rays stalled at the cap:", stalled)

