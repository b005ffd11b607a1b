"""FocalBatchSource (gfnerf_b200/pixel_samplers.py, csrc/focal_batch.cu): focal-stage batches drawn on the device
from ErrorPixelSampler's distribution, with a sum tree of the error map kept current by the error feedback.

The distribution is checked against exact successive-sampling probabilities by chi-square, with ErrorPixelSampler
through the same test as a control; the chunk rule above 2^24 pixels by exact per-chunk counts; the tree, the map
and the batch contents bit for bit against a rebuild, update_error_map, Cameras.generate_rays and the collate gather;
and a 20-step focal loop against the same loop fed through the ErrorPixelSampler path."""
import numpy as np
import pytest
import torch
from scipy import stats

from gfnerf_b200 import pixel_samplers as ps
from gfnerf_b200.cameras import Cameras
from tests.helpers import load_rig, make_sampler

C24 = 2 ** 24


def _cams(n, dev="cuda"):
    g = torch.Generator().manual_seed(3)
    c2w = torch.eye(4)[:3].repeat(n, 1, 1) + 0.1 * torch.rand(n, 3, 4, generator=g)
    return Cameras(c2w.to(dev), fx=500.0, fy=510.0, cx=16.0, cy=12.0)


def _source(err, R, seed=0, ratio=0.2, n_cams=None, **kw):
    """A source over images of the error map's shape; image_idx = 2 * slot + 1 so that slot and camera differ."""
    n_img, h, w = err.shape[:3]
    g = torch.Generator().manual_seed(11)
    images = torch.rand(n_img, h, w, 3, generator=g).to(err.device)
    image_idx = torch.arange(n_img, device=err.device) * 2 + 1
    rel = torch.arange(n_img, device=err.device) + 100
    return ps.FocalBatchSource(images, err, _cams(n_cams or 2 * n_img + 1), image_idx, rel, num_rays_per_batch=R,
                               weighted_choice_ratio=ratio, seed=seed, **kw)


def _flat(rows, shape):
    n_img, h, w = shape
    return (rows[:, 0] * h + rows[:, 1]) * w + rows[:, 2]


def _chi2_pvalue(counts, p):
    """chi-square goodness of fit; cells with an expectation below 5 are pooled into one"""
    counts, p = np.asarray(counts, np.float64).ravel(), np.asarray(p, np.float64).ravel()
    exp = p * counts.sum()
    big = exp >= 5
    obs = np.append(counts[big], counts[~big].sum())
    e = np.append(exp[big], exp[~big].sum())
    keep = e > 0
    assert obs[~keep].sum() == 0, "a cell of probability 0 was drawn"
    return stats.chisquare(obs[keep], e[keep]).pvalue


def _pl_probabilities(w):
    """exact successive sampling: first pick w_a / S, ordered pair w_a / S * w_b / (S - w_a)"""
    w = np.asarray(w, np.float64)
    S = w.sum()
    first = w / S
    pair = first[:, None] * w[None, :] / (S - w[:, None])
    np.fill_diagonal(pair, 0.0)
    return first, pair


WEIGHTS = [0.0, 1.0, 2.0, 3.0, 0.5, 0.0, 4.0, 1.5, 0.25, 2.5, 0.0, 1.0, 3.5, 0.75, 2.0, 5.0]


@pytest.mark.gpu
def test_weighted_pairs_follow_successive_sampling():
    """n_w = 2 of a 16-pixel map: first picks and ordered pairs of >= 1e5 draws against the exact probabilities."""
    dev = torch.device("cuda:0")
    err = torch.tensor(WEIGHTS, device=dev).view(1, 4, 4, 1)
    src = _source(err, R=10, seed=5)                      # n_w = int(10 * 0.2) = 2, 8 uniform of 16
    assert src.n_weighted == 2
    K, reps = 100, 1000
    buf = torch.empty(K, 10, dtype=torch.int64, device=dev)
    src.next_batch()                                       # (not captured: the graph records the launches only)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for k in range(K):
            buf[k].copy_(_flat(src.next_batch()["slot_indices"], src.shape))
    pairs = torch.zeros(16 * 16, dtype=torch.int64, device=dev)
    uni = torch.zeros(16, dtype=torch.int64, device=dev)
    dup = torch.zeros((), dtype=torch.int64, device=dev)
    for _ in range(reps):
        g.replay()
        pairs += torch.bincount(buf[:, 0] * 16 + buf[:, 1], minlength=256)
        uni += torch.bincount(buf[:, 2:].reshape(-1), minlength=16)
        s = buf[:, 2:].sort(1).values
        dup += (s[:, 1:] == s[:, :-1]).sum() + (buf[:, 0] == buf[:, 1]).sum()
    src.check()
    assert int(dup) == 0                                   # each part is duplicate-free
    pairs = pairs.view(16, 16).cpu().numpy()
    first, pair = _pl_probabilities(WEIGHTS)
    zero = np.array(WEIGHTS) == 0
    assert pairs[zero].sum() == 0 and pairs[:, zero].sum() == 0   # zero-weight pixels never in the weighted part
    p1 = _chi2_pvalue(pairs.sum(1), first)
    p2 = _chi2_pvalue(pairs, pair)
    pu = _chi2_pvalue(uni.cpu().numpy(), np.full(16, 1 / 16))
    print("p-values: first pick", p1, "ordered pair", p2, "uniform part", pu)
    assert p1 > 1e-3 and p2 > 1e-3 and pu > 1e-3


def test_error_pixel_sampler_passes_the_same_test():
    """The control: the existing ErrorPixelSampler, through the same chi-square test (CPU generator)."""
    s = ps.ErrorPixelSampler(10, generator=torch.Generator().manual_seed(6))
    em = torch.tensor(WEIGHTS).view(1, 4, 4, 1)
    pairs = np.zeros((16, 16), np.int64)
    N = 100000
    rows = torch.stack([s.weighted_choice_multinomial(em.view(-1), 2, "cpu") for _ in range(N)]).numpy()
    np.add.at(pairs, (rows[:, 0], rows[:, 1]), 1)
    first, pair = _pl_probabilities(WEIGHTS)
    p1, p2 = _chi2_pvalue(pairs.sum(1), first), _chi2_pvalue(pairs, pair)
    print("p-values: first pick", p1, "ordered pair", p2)
    assert p1 > 1e-3 and p2 > 1e-3


@pytest.mark.gpu
def test_first_pick_marginals_on_a_larger_map():
    """A 3 x 40 x 50 map (several tiles, a partial last tile) with a hot region: first-pick marginals of 2e4 draws,
    and both parts duplicate-free."""
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(2)
    err = torch.rand(3, 40, 50, 1, generator=g) ** 4
    err[1, 10:14, 20:30] = 50.0
    err[2, :5] = 0.0
    err = err.to(dev)
    w = err.view(-1).double().cpu().numpy()
    src = _source(err, R=100, seed=9)                     # 20 weighted, 80 uniform
    firsts = torch.zeros(w.size, dtype=torch.int64, device=dev)
    for it in range(20000):
        f = _flat(src.next_batch()["slot_indices"], src.shape)
        firsts[f[0]] += 1
        if it % 500 == 0:
            wf, uf = f[:20].sort().values, f[20:].sort().values
            assert bool((wf[1:] != wf[:-1]).all()) and bool((uf[1:] != uf[:-1]).all())
            assert float(err.view(-1)[f[:20]].min()) > 0
    src.check()
    fc = firsts.cpu().numpy()
    assert fc[w == 0].sum() == 0
    p = _chi2_pvalue(fc, w / w.sum())
    print("first-pick p-value", p)
    assert p > 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("n,n_w,tail", [(C24 + 4096, 300, None),          # 1 chunk; n % 1 == 0
                                         (2 * C24, 201, "uniform"),        # exact multiple: remainder uniform
                                         (3 * C24, 200, "uniform"),
                                         (3 * C24 + 1000, 200, "tail")])   # n % 3 != 0: remainder from the tail
def test_chunk_rule(n, n_w, tail):
    dev = torch.device("cuda:0")
    err = torch.rand(1, 1, n, 1, device=dev, generator=torch.Generator(device=dev).manual_seed(1)) + 0.01
    src = _source(err, R=n_w, ratio=1.0, seed=3)
    assert src.n_weighted == n_w
    n_chunks = n // C24
    per, rest = n_w // n_chunks, n_w % n_chunks
    for _ in range(3):
        f = _flat(src.next_batch()["slot_indices"], src.shape)
        for c in range(n_chunks):
            part = f[c * per:(c + 1) * per]
            assert bool(((part >= c * C24) & (part < (c + 1) * C24)).all())
            assert part.unique().numel() == per
        r = f[n_chunks * per:]
        assert r.numel() == rest
        if tail == "tail":
            assert bool((r >= n_chunks * C24).all()) and r.unique().numel() == rest
        elif rest:
            assert bool((r >= 0).all() & (r < n).all()) and r.unique().numel() == rest
    src.check()


@pytest.mark.gpu
def test_too_few_nonzero_pixels_in_a_chunk_raises_in_check():
    dev = torch.device("cuda:0")
    err = torch.ones(1, 1, 3 * C24 + 1000, 1, device=dev)
    err[..., 3 * C24 + 1:, :] = 0.0                          # the tail chunk draws 2 but has one non-zero pixel
    src = _source(err, R=200, ratio=1.0)
    b = src.next_batch()
    assert bool((b["slot_indices"][:, 2] < err.shape[2]).all())     # flagged rows still index the map
    with pytest.raises(RuntimeError, match="fewer non-zero pixels"):
        src.check()
    src.check()                                               # the flag was cleared
    err2 = torch.zeros(2, 4, 4, 1, device=dev)
    err2[0, 0, 0] = 1.0
    src = _source(err2, R=10)                                 # 2 weighted, one non-zero pixel
    src.next_batch()
    with pytest.raises(RuntimeError, match="fewer non-zero pixels"):
        src.check()


@pytest.mark.gpu
def test_bad_maps_and_host_tensors_are_rejected():
    dev = torch.device("cuda:0")
    for bad in (-1.0, float("nan"), float("inf")):
        err = torch.rand(2, 8, 8, 1, device=dev)
        err[1, 3, 4] = bad
        with pytest.raises(ValueError):
            _source(err, R=16)
    err = torch.rand(2, 8, 8, 1)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ps.FocalBatchSource(torch.rand(2, 8, 8, 3), err, _cams(3), torch.arange(2), torch.arange(2))
    with pytest.raises(RuntimeError, match="no CPU path"):
        ps.FocalBatchSource(torch.rand(2, 8, 8, 3, device=dev), err, _cams(3), torch.arange(2, device=dev),
                            torch.arange(2, device=dev))
    src = _source(torch.rand(2, 8, 8, 1, device=dev), R=16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        src.update(torch.zeros(16, 3, dtype=torch.int64), torch.zeros(16, 3))
    with pytest.raises(ValueError):
        _source(torch.rand(1, 4, 4, 1, device=dev), R=40)    # 32 uniform of 16 pixels: random.sample's error
    # a NaN written by the feedback reaches the draw as torch.multinomial's invalid-distribution error
    b = src.next_batch()
    pred = b["rgb"].clone()
    pred[0, 0] = float("nan")
    src.update(b["slot_indices"], pred)
    src.next_batch()
    with pytest.raises(RuntimeError, match="non-finite"):
        src.check()


@pytest.mark.gpu
def test_batch_contents():
    dev = torch.device("cuda:0")
    err = torch.rand(4, 24, 32, 1, device=dev, generator=torch.Generator(device=dev).manual_seed(4))
    src = _source(err, R=512, seed=1)
    cams = src.cameras
    for _ in range(3):
        b = src.next_batch()
        sl = b["slot_indices"]
        c, y, x = sl[:, 0], sl[:, 1], sl[:, 2]
        assert torch.equal(b["rgb"], src.images[c, y, x])
        assert torch.equal(b["indices"][:, 0], src.image_idx[c]) and torch.equal(b["indices"][:, 1:], sl[:, 1:])
        assert torch.equal(b["rel_camera_indices"], src.rel_camera_idx[c])
        coords = torch.stack((y, x), -1).float() + 0.5
        ref = cams.generate_rays(b["indices"][:, 0], coords)
        assert torch.equal(b["origins"], ref.origins) and torch.equal(b["directions"], ref.directions)
    src.check()


@pytest.mark.gpu
def test_tree_and_map_after_updates():
    """Many updates, batches with repeated pixels included: the tree is bit-equal to a rebuild, the map to
    update_error_map wherever a batch names a pixel once, and a pixel named twice holds one of its rows' errors."""
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(8)
    err = torch.rand(3, 64, 100, 1, device=dev, generator=gen)
    ref = err.clone()
    src = _source(err, R=700, seed=2, ratio=0.5)            # 350 weighted + 350 uniform: the parts overlap
    n_twice = 0
    for it in range(40):
        b = src.next_batch()
        rows = b["slot_indices"].clone()
        if it % 4 == 3:                                      # a batch of the caller's own with repeated rows
            rows[100:200] = rows[:100]
        pred = torch.rand(rows.shape[0], 3, device=dev, generator=gen)
        gt = src.images[rows[:, 0], rows[:, 1], rows[:, 2]]
        src.update(rows, pred, gt_rgb=gt)
        e = ps.update_error_map(ref, rows, pred, gt, return_error=True)
        f = _flat(rows, src.shape)
        uniq, inv, cnt = f.unique(return_inverse=True, return_counts=True)
        once = cnt[inv] == 1
        got, want = err.view(-1), ref.view(-1)
        assert torch.equal(got[f[once]], want[f[once]])
        for p in uniq[cnt > 1].tolist():
            n_twice += 1
            assert float(got[p]) in e[f == p].tolist()
        want.copy_(got)                                      # both maps agree from here on
    assert n_twice > 0
    sums, counts = src.sums.clone(), src.counts.clone()
    src.rebuild()
    assert torch.equal(sums, src.sums) and torch.equal(counts, src.counts)
    src.check()


@pytest.mark.gpu
def test_no_sync_graph_replay_and_seed():
    dev = torch.device("cuda:0")
    err0 = torch.rand(2, 40, 60, 1, device=dev, generator=torch.Generator(device=dev).manual_seed(3))

    def eager(steps):
        err = err0.clone()
        src = _source(err, R=256, seed=21)
        out = []
        for _ in range(steps):
            b = src.next_batch()
            src.update(b["slot_indices"], b["rgb"] * 0.5)
            out.append((b["slot_indices"].clone(), b["origins"].clone(), err.clone()))
        return out

    a, b = eager(4), eager(4)
    for x, y in zip(a, b):                                   # the same seed gives the same batches
        assert all(torch.equal(p, q) for p, q in zip(x, y))
    assert not torch.equal(a[0][0], a[1][0])

    err = err0.clone()
    src = _source(err, R=256, seed=21)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        bt = src.next_batch()
        src.update(bt["slot_indices"], bt["rgb"] * 0.5)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.equal(bt["slot_indices"], a[0][0]) and torch.equal(err, a[0][2])

    err = err0.clone()
    src = _source(err, R=256, seed=21)
    pred = torch.empty(256, 3, device=dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        bt = src.next_batch()
        torch.mul(bt["rgb"], 0.5, out=pred)
        src.update(bt["slot_indices"], pred)
    for k in range(4):
        g.replay()
        assert torch.equal(bt["slot_indices"], a[k][0]) and torch.equal(bt["origins"], a[k][1])
        assert torch.equal(err, a[k][2])
    src.check()


@pytest.mark.gpu
def test_focal_loop_matches_the_error_pixel_sampler_path():
    """20 focal steps fed by the source, and the same 20 steps fed with the same rows through ErrorPixelSampler's
    collate gather, Cameras.generate_rays and update_error_map: bit-equal batches and maps, parameters within the
    gates of the engine tests (the hash scatter's fp32 atomics make training itself non-bit-reproducible)."""
    from gfnerf_b200.engine import GFNeRFEngine
    dev = torch.device("cuda:0")
    rig = load_rig("rig8")
    n_cam = rig["c2w"].shape[0]
    intri = torch.from_numpy(rig["intri"])
    cams = Cameras(torch.from_numpy(rig["c2w"]).to(dev), intri[:, 0, 0], intri[:, 1, 1], intri[:, 0, 2],
                   intri[:, 1, 2], width=1920, height=1080)
    slots = torch.arange(0, n_cam, 8, device=dev)                       # 8 images of the 64 cameras
    n_img = slots.numel()
    g = torch.Generator(device=dev).manual_seed(0)
    images = torch.rand(n_img, 1080, 1920, 3, device=dev, generator=g)
    err_a = torch.rand(n_img, 1080, 1920, 1, device=dev, generator=g)
    err_b = err_a.clone()
    rel = torch.arange(n_img, device=dev)
    R = 2048
    src = ps.FocalBatchSource(images, err_a, cams, slots, rel, num_rays_per_batch=R, seed=4)
    sampler = ps.ErrorPixelSampler(R)

    def engine():
        eng = GFNeRFEngine(make_sampler(rig, mode=1), log2_table_size=14, num_images=n_cam, seed=3)
        init = torch.rand(eng.enc.feat_pool_.shape, generator=torch.Generator().manual_seed(11)) * 0.02 - 0.01
        eng.enc.feat_pool_.data.copy_(init)
        eng.enc.shadow(force=True)
        eng.start_block_stage(log2_table_size=14, seed=5)
        return eng

    ea, eb = engine(), engine()
    la, lb = [], []
    for step in range(20):
        b = src.next_batch()
        rows = b["slot_indices"].clone()
        sampler.sample_method = lambda *a, **k: rows                     # the same rows, the reference's gather
        cb = sampler.collate_image_dataset_batch({"image": images, "error_map": err_b, "image_idx": slots,
                                                  "rel_camera_idx": rel}, R)
        ray = cams.generate_rays(cb["indices"][:, 0], cb["indices"][:, 1:].float() + 0.5)
        assert torch.equal(b["rgb"], cb["image"]) and torch.equal(b["indices"], cb["indices"])
        assert torch.equal(b["rel_camera_indices"], cb["rel_camera_indices"])
        assert torch.equal(b["origins"], ray.origins) and torch.equal(b["directions"], ray.directions)
        oa = ea.train_step(b["origins"], b["directions"], b["rgb"], b["rel_camera_indices"])
        ob = eb.train_step(ray.origins, ray.directions, cb["image"], cb["rel_camera_indices"])
        la.append(oa.loss.clone())
        lb.append(ob.loss.clone())
        src.update(b["slot_indices"], oa.rgb)
        ps.update_error_map(err_b, cb["slot_indices"], oa.rgb, cb["image"])      # the same out.rgb
        f = _flat(rows, src.shape)
        uniq, inv, cnt = f.unique(return_inverse=True, return_counts=True)
        once = cnt[inv] == 1
        assert torch.equal(err_a.view(-1)[f[once]], err_b.view(-1)[f[once]])
        err_b.view(-1)[f[~once]] = err_a.view(-1)[f[~once]]               # (which duplicate lands is unspecified)
        assert torch.equal(err_a, err_b)
    src.check()
    ea.flush()
    eb.flush()
    assert torch.allclose(torch.cat(la), torch.cat(lb), rtol=1e-3, atol=0)
    ra, rb = ea.res.feat_pool_.detach(), eb.res.feat_pool_.detach()
    assert float((ra - rb).abs().mean()) <= 1e-3 * float(ra.abs().mean())
