"""The float64 image-metrics oracle (oracle/image_metrics.py) against the definition and hand-computable cases, on the
CPU.  The GPU kernel is held to this oracle in tests/test_image_metrics_gpu.py."""
import numpy as np
import pytest

from oracle import image_metrics as im


@pytest.mark.parametrize("H,W,seed", [(11, 11, 0), (12, 17, 1), (23, 11, 2), (40, 57, 3)])
def test_pad_and_crop_form_equals_direct_windows(H, W, seed):
    rng = np.random.RandomState(seed)
    p, g = rng.rand(H, W, 3), rng.rand(H, W, 3) * 1.5 - 0.2
    a, b = im.ssim_map(p, g), im.ssim_direct(p, g)
    assert a.shape == b.shape == (3, H - 10, W - 10)
    assert np.abs(a - b).max() < 1e-12


def test_window_is_torchmetrics_gaussian():
    k = im.gaussian_window()
    assert k.shape == (11, 11) and abs(k.sum() - 1) < 1e-15
    assert np.allclose(k, k.T) and np.argmax(k) == 5 * 11 + 5
    g = np.exp(-((np.arange(11) - 5) / 1.5) ** 2 / 2)
    assert np.allclose(k[5] / k[5, 5], g)


def test_identical_images():
    rng = np.random.RandomState(4)
    p = rng.rand(20, 31, 3)
    m = im.image_metrics(p, p)
    assert m["psnr"][0] == np.inf and m["mse"][0] == 0
    assert abs(m["ssim"][0] - 1) < 1e-12


@pytest.mark.parametrize("a,b", [(0.2, 0.7), (0.9, 0.1), (0.5, 0.55)])
def test_constant_images_with_unit_range(a, b):
    """sigma terms vanish, so the C2 factors cancel: SSIM = (2ab + C1) / (a^2 + b^2 + C1), C1 = 0.01^2"""
    p, g = np.full((15, 14, 3), a), np.full((15, 14, 3), b)
    c1 = 0.01 ** 2
    m = im.image_metrics(p, g, L=1.0)
    assert abs(m["ssim"][0] - (2 * a * b + c1) / (a * a + b * b + c1)) < 1e-12
    assert abs(m["mse"][0] - (a - b) ** 2) < 1e-15
    assert abs(m["psnr"][0] - 10 * np.log10(1 / (a - b) ** 2)) < 1e-9


@pytest.mark.parametrize("d", [0.25, -0.1, 3.0])
def test_uniform_offset_gives_mse_d_squared(d):
    rng = np.random.RandomState(5)
    p = rng.rand(2, 13, 16, 3)
    m = im.image_metrics(p + d, p)
    np.testing.assert_allclose(m["mse"], d * d, rtol=1e-12)
    np.testing.assert_allclose(m["psnr"], -20 * np.log10(abs(d)), rtol=1e-12)
