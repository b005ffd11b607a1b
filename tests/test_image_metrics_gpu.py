"""GPU: `image_metrics` (gf_image_metrics, csrc/metrics.cu) against the float64 oracle (oracle/image_metrics.py, the
torchmetrics steps), its edge cases, batching, determinism, CUDA-graph capture, a held-out view that training
improves, and `GFNeRFModel.get_image_metrics_and_images`."""
import numpy as np
import pytest
import torch

from oracle import image_metrics as orc_im
from tests.helpers import load_rig, make_sampler

pytestmark = pytest.mark.gpu

# SSIM is a mean of per-pixel ratios whose variances E[x^2] - mu^2 come from fp32 sums of 121 products.  The kernel
# takes the moments of x - x0, x0 the centre pixel of its 32 x 32 tile, so a moment of magnitude m = (x - x0)^2 is
# off by a few fp32 ulps of m (~2.4e-7 m), and the ratio by about that over C2 = 9e-4 L^2.  The worst case is a large
# flat region whose tile shift lies across an edge of height d: sigma = 0 there but m ~ d^2, up to ~2.6e-4 d^2 / L^2
# per pixel; averaged over the image this stays below 1e-5 in every case here.  MSE and PSNR are summed in double.
SSIM_ATOL = 1e-5
MSE_RTOL = 1e-6


def _content(kind, B, H, W, seed):
    rng = np.random.RandomState(seed)
    y = np.linspace(0, 1, H)[None, :, None, None]
    x = np.linspace(0, 1, W)[None, None, :, None]
    ch = np.arange(3)[None, None, None, :]
    if kind == "noise":
        g = rng.rand(B, H, W, 3)
        p = rng.rand(B, H, W, 3)
    elif kind == "ramps":
        ph = rng.rand(B, 1, 1, 3) * 6
        g = 0.5 + 0.4 * np.sin(3 * x + 2 * y + ph + ch)
        p = np.clip(g + 0.03 * np.sin(17 * x - 11 * y + ch) + 0.01 * rng.randn(B, H, W, 3), 0, 1)
    elif kind == "flat":
        # large constant regions (the cancellation E[x^2] - mu^2 at its worst), a few edges, noise in one corner
        g = np.broadcast_to(np.where((x < 0.6) & (y < 0.5), 0.83, 0.27), (B, H, W, 3)).copy()
        g[:, : H // 3, : W // 4] += 0.1 * rng.rand(B, H // 3, W // 4, 3)
        p = g.copy()
        p[:, H // 2:, W // 2:] = 0.61
    elif kind == "wide":
        # values outside [0, 1]: the data range L is larger than 1
        g = rng.rand(B, H, W, 3) * 2.5 - 0.7
        p = g + 0.2 * np.sin(5 * x + ch) + 0.05 * rng.randn(B, H, W, 3)
    else:
        raise ValueError(kind)
    return p.astype(np.float32), g.astype(np.float32)


def _check_against_oracle(p, g, what):
    from gfnerf_b200 import image_metrics
    got = image_metrics(torch.from_numpy(p).cuda(), torch.from_numpy(g).cuda())
    ref = orc_im.image_metrics(p, g)
    got = {k: v.cpu().numpy().astype(np.float64) for k, v in got.items()}
    d_ssim = np.abs(got["ssim"] - ref["ssim"]).max()
    d_mse = (np.abs(got["mse"] - ref["mse"]) / ref["mse"]).max()
    d_psnr = (np.abs(got["psnr"] - ref["psnr"]) / np.abs(ref["psnr"])).max()
    print(f"{what}: ssim |d| {d_ssim:.2e}  mse rel {d_mse:.2e}  psnr rel {d_psnr:.2e}  ssim {got['ssim']}")
    assert d_ssim <= SSIM_ATOL, (what, got["ssim"], ref["ssim"])
    assert d_mse <= MSE_RTOL and d_psnr <= MSE_RTOL, (what, got, ref)
    return got, ref


@pytest.mark.parametrize("kind", ["noise", "ramps", "flat", "wide"])
@pytest.mark.parametrize("H,W", [(11, 11), (12, 300), (37, 1001), (1080, 1920)])
@pytest.mark.parametrize("B", [1, 3])
def test_matches_oracle(B, H, W, kind):
    """Worst deviations measured on one B200 (printed per case): SSIM 7.4e-6 absolute (flat regions, 37 x 1001;
    every other content <= 1.9e-7), MSE 5.3e-8 and PSNR 5.1e-8 relative."""
    p, g = _content(kind, B, H, W, seed=H * 7 + W + B)
    _check_against_oracle(p, g, f"B={B} {H}x{W} {kind}")


def test_identical_images_and_constant_images():
    from gfnerf_b200 import image_metrics
    p, _ = _content("noise", 2, 40, 53, seed=9)
    t = torch.from_numpy(p).cuda()
    m = image_metrics(t, t.clone())
    assert torch.isinf(m["psnr"]).all() and (m["psnr"] > 0).all() and (m["mse"] == 0).all()
    assert float((m["ssim"] - 1).abs().max()) <= 1e-6
    a = torch.full((1, 20, 30, 3), 0.3, device="cuda")
    b = torch.full((1, 20, 30, 3), 0.8, device="cuda")
    m = image_metrics(a, b)
    assert torch.isnan(m["ssim"]).all()                    # L = 0: C1 = C2 = 0 and 0 / 0
    assert abs(float(m["mse"][0]) - 0.25) < 1e-7


def test_rejects_bad_input():
    from gfnerf_b200 import image_metrics
    good = torch.rand(16, 16, 3, device="cuda")
    for bad_p, bad_g in [(torch.rand(10, 16, 3, device="cuda"), torch.rand(10, 16, 3, device="cuda")),
                         (torch.rand(16, 10, 3, device="cuda"), torch.rand(16, 10, 3, device="cuda")),
                         (good.double(), good.double()),
                         (good.half(), good),
                         (good.cpu(), good.cpu()),
                         (good, good.cpu()),
                         (good, torch.rand(16, 17, 3, device="cuda")),
                         (good, good[None]),
                         (torch.rand(16, 16, 4, device="cuda"), torch.rand(16, 16, 4, device="cuda")),
                         (torch.rand(16, 16, device="cuda"), torch.rand(16, 16, device="cuda"))]:
        with pytest.raises(RuntimeError):
            image_metrics(bad_p, bad_g)


def test_batch_equals_single_images_and_repeats_bit_for_bit():
    from gfnerf_b200 import image_metrics
    ps, gs = [], []
    for i, kind in enumerate(["noise", "ramps", "flat", "wide", "noise"]):
        p, g = _content(kind, 1, 45, 77, seed=i)
        ps.append(p), gs.append(g)
    P, G = torch.from_numpy(np.concatenate(ps)).cuda(), torch.from_numpy(np.concatenate(gs)).cuda()
    m1, m2 = image_metrics(P, G), image_metrics(P, G)
    for k in m1:
        assert torch.equal(m1[k], m2[k]), k
    for i in range(P.shape[0]):
        # image i alone: a fresh 16-byte-aligned copy, and a view at an offset that is not (3 * 45 * 77 floats)
        for pi, gi in [(P[i].clone(), G[i].clone()), (P[i], G[i])]:
            mi = image_metrics(pi, gi)
            for k in m1:
                assert torch.equal(mi[k][0], m1[k][i]), (i, k)


def test_cuda_graph_capture_and_replay():
    from gfnerf_b200 import image_metrics
    p0, g0 = _content("ramps", 2, 70, 130, seed=3)
    p1, g1 = _content("noise", 2, 70, 130, seed=4)
    sp, sg = torch.from_numpy(p0).cuda(), torch.from_numpy(g0).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        image_metrics(sp, sg)                                # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = image_metrics(sp, sg)
    sp.copy_(torch.from_numpy(p1)), sg.copy_(torch.from_numpy(g1))
    graph.replay()
    torch.cuda.synchronize()
    eager = image_metrics(torch.from_numpy(p1).cuda(), torch.from_numpy(g1).cuda())
    for k in eager:
        assert torch.equal(out[k], eager[k]), k


def _scene_colour(o, d):
    """the synthetic scene of tests/test_engine_gpu.py::test_training_reduces_loss_and_prunes: colour is a smooth
    function of the ray's ground hit point"""
    hit = o + d * (o[:, 2:3] / np.maximum(-d[:, 2:3], 1e-3))
    return (0.5 + 0.5 * np.sin(hit * np.array([1.3, 0.9, 0.0]) + np.array([0.0, 1.0, 2.0]))).astype(np.float32)


HELD_OUT = 3
N_STEPS = 150
MIN_GAIN_DB = 8.0


def test_training_improves_a_held_out_view():
    """Train on rays of every rig8 camera except one, render the held-out camera at 1/10 resolution (192 x 108,
    intrinsics scaled) and measure it with image_metrics against the analytic scene colour: the metrics equal the
    oracle's on the rendered image, and PSNR rises by at least MIN_GAIN_DB over N_STEPS steps.  Measured on one B200:
    PSNR 8.42 -> 20.27 dB (+11.8 dB), SSIM 0.732 -> 0.845 after 150 steps; the bound of 8 dB leaves a third of the gain
    as margin."""
    from gfnerf_b200 import image_metrics
    from gfnerf_b200.engine import GFNeRFEngine
    from gfnerf_b200.persoctree import frame_rays, rig_rays
    rig = load_rig("rig8")
    eng = GFNeRFEngine(make_sampler(rig, mode=0), log2_table_size=16, num_images=rig["c2w"].shape[0], seed=1)
    s = 10
    intri = rig["intri"][HELD_OUT].copy()
    intri[:2] /= s
    W, H = int(round(2 * intri[0, 2])), int(round(2 * intri[1, 2]))
    o_v, d_v = frame_rays(rig["c2w"][HELD_OUT], intri, W, H)
    gt = torch.from_numpy(_scene_colour(o_v, d_v).reshape(H, W, 3)).cuda()
    to_v, td_v = torch.from_numpy(o_v).cuda(), torch.from_numpy(d_v).cuda()

    def view_metrics():
        rgb, _, _ = eng.render_image(to_v, td_v, rel_camera_index=HELD_OUT)
        rgb = rgb.view(H, W, 3)
        m = image_metrics(rgb, gt)
        ref = orc_im.image_metrics(rgb.cpu().numpy(), gt.cpu().numpy())
        assert abs(float(m["ssim"][0]) - ref["ssim"][0]) <= SSIM_ATOL
        assert abs(float(m["mse"][0]) - ref["mse"][0]) <= MSE_RTOL * ref["mse"][0]
        assert abs(float(m["psnr"][0]) - ref["psnr"][0]) <= MSE_RTOL * abs(ref["psnr"][0])
        return float(m["psnr"][0]), float(m["ssim"][0])

    psnr0, ssim0 = view_metrics()
    R = 2048
    for it in range(N_STEPS):
        o, d, cam = rig_rays(rig["c2w"], rig["intri"], 2 * R, seed=100 + it)
        keep = np.nonzero(cam != HELD_OUT)[0][:R]
        o, d, cam = o[keep], d[keep], cam[keep]
        eng.train_step(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(),
                       torch.from_numpy(_scene_colour(o, d)).cuda(), torch.from_numpy(cam).cuda())
    psnr1, ssim1 = view_metrics()
    print(f"held-out view {W}x{H}: PSNR {psnr0:.3f} -> {psnr1:.3f} dB, SSIM {ssim0:.4f} -> {ssim1:.4f}")
    assert psnr1 - psnr0 >= MIN_GAIN_DB


def test_rendered_frame_against_perturbed_copy():
    """A 1920 x 1080 frame of render_image on rig8 (random table) against a copy with noise and a shifted block.
    Measured on one B200: SSIM 1.0e-8 absolute, MSE 8.3e-9 relative from the oracle."""
    from gfnerf_b200.engine import GFNeRFEngine
    from gfnerf_b200.persoctree import frame_rays
    rig = load_rig("rig8")
    eng = GFNeRFEngine(make_sampler(rig, mode=1), log2_table_size=15, num_images=rig["c2w"].shape[0], seed=0)
    torch.manual_seed(7)
    eng.enc.feat_pool_.data.uniform_(-0.5, 0.5)
    eng.enc.shadow(force=True)
    W, H = 1920, 1080
    o, d = frame_rays(rig["c2w"][3], rig["intri"][3], W, H)
    rgb, _, _ = eng.render_image(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), rel_camera_index=3)
    p = rgb.view(1, H, W, 3).cpu().numpy()
    rng = np.random.RandomState(0)
    g = np.clip(p + 0.02 * rng.randn(*p.shape), 0, 1)
    g[:, 200:500, 300:900] = p[:, 205:505, 300:900]
    _check_against_oracle(p, g.astype(np.float32), "render_image 1920x1080")


def test_model_get_image_metrics_and_images():
    from gfnerf_b200 import image_metrics
    from gfnerf_b200.persoctree import frame_rays
    from tests.test_operator_api_gpu import build
    rig = load_rig("rig8")
    eng, model = build(rig)
    W, H = 96, 54
    intri = rig["intri"][5].copy()
    intri[:2] /= 20
    o, d = frame_rays(rig["c2w"][5], intri, W, H)
    rgb, _, _ = eng.render_image(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), rel_camera_index=5)
    rgb = rgb.view(H, W, 3)
    gt = torch.from_numpy(_scene_colour(o, d).reshape(H, W, 3))          # on the host, as a dataloader hands it over
    metrics_dict, images_dict = model.get_image_metrics_and_images({"rgb": rgb}, {"image": gt})
    m = image_metrics(rgb, gt.cuda())
    assert set(metrics_dict) == {"psnr", "ssim"}
    assert metrics_dict["psnr"] == float(m["psnr"][0]) and metrics_dict["ssim"] == float(m["ssim"][0])
    assert set(images_dict) == {"img"} and images_dict["img"].shape == (H, 2 * W, 3)
    assert torch.equal(images_dict["img"][:, :W].cpu(), gt) and torch.equal(images_dict["img"][:, W:], rgb)
