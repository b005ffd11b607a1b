"""Float64 restatement of the image metrics of nerfstudio's nerfacto evaluation (test infrastructure only): torchmetrics'
`PeakSignalNoiseRatio(data_range=1.0)` and functional `structural_similarity_index_measure` with its defaults, one
image at a time, following torchmetrics' steps: Gaussian window (size 11, sigma 1.5, normalised, outer product),
reflect pad by 5, 2-D correlation of p, g, p^2, g^2, p g with the window, the SSIM map, crop of 5 on every side, mean.

Images are [H, W, 3] (or [B, H, W, 3]) arrays in any float dtype; everything is computed in float64.  The 2-D
correlation is evaluated by FFT (scipy.signal.fftconvolve; rounding ~1e-15 of the values), `ssim_direct` evaluates the
same definition window by window and is what the FFT form is checked against."""
import numpy as np
from scipy.signal import fftconvolve

KSIZE, SIGMA, PAD = 11, 1.5, 5


def gaussian_window(ksize=KSIZE, sigma=SIGMA):
    d = np.arange(ksize, dtype=np.float64) - (ksize - 1) / 2
    g = np.exp(-(d / sigma) ** 2 / 2)
    g /= g.sum()
    return np.outer(g, g)


def data_range(p, g):
    return max(p.max() - p.min(), g.max() - g.min())


def _ssim_terms(mu_p, mu_g, e_pp, e_gg, e_pg, L):
    c1, c2 = (0.01 * L) ** 2, (0.03 * L) ** 2
    s_pp, s_gg, s_pg = e_pp - mu_p ** 2, e_gg - mu_g ** 2, e_pg - mu_p * mu_g
    return ((2 * mu_p * mu_g + c1) * (2 * s_pg + c2)) / ((mu_p ** 2 + mu_g ** 2 + c1) * (s_pp + s_gg + c2))


def ssim_map(pred, gt, L=None):
    """SSIM per (channel, y, x) of the valid-window region, [3, H - 10, W - 10], by torchmetrics' pad-and-crop form.
    L: the data range; by default max(max p - min p, max g - min g), torchmetrics' default."""
    p = np.moveaxis(np.asarray(pred, np.float64), -1, 0)           # [3, H, W]
    g = np.moveaxis(np.asarray(gt, np.float64), -1, 0)
    if L is None:
        L = data_range(p, g)
    maps = np.stack([p, g, p * p, g * g, p * g])                    # [5, 3, H, W]
    padded = np.pad(maps, ((0, 0), (0, 0), (PAD, PAD), (PAD, PAD)), mode="reflect")
    k = gaussian_window()
    out = fftconvolve(padded, k[None, None, ::-1, ::-1], mode="valid", axes=(-2, -1))   # correlation, [5, 3, H, W]
    full = _ssim_terms(*out, L)
    return full[:, PAD:-PAD, PAD:-PAD]


def ssim_direct(pred, gt, L=None):
    """The same map evaluated window by window from the definition (no padding): slow, for small images."""
    p = np.moveaxis(np.asarray(pred, np.float64), -1, 0)
    g = np.moveaxis(np.asarray(gt, np.float64), -1, 0)
    if L is None:
        L = data_range(p, g)
    k = gaussian_window()
    C, H, W = p.shape
    out = np.empty((C, H - 2 * PAD, W - 2 * PAD))
    for c in range(C):
        for y in range(H - 2 * PAD):
            for x in range(W - 2 * PAD):
                wp, wg = p[c, y:y + KSIZE, x:x + KSIZE], g[c, y:y + KSIZE, x:x + KSIZE]
                out[c, y, x] = _ssim_terms((k * wp).sum(), (k * wg).sum(), (k * wp * wp).sum(), (k * wg * wg).sum(),
                                           (k * wp * wg).sum(), L)
    return out


def image_metrics(pred, gt, L=None):
    """{"psnr", "ssim", "mse"} as float64 arrays [B] for [B, H, W, 3] inputs (scalars' arrays of length 1 for
    [H, W, 3]).  L fixes the SSIM data range (the kernel always derives it per image)."""
    pred, gt = np.asarray(pred, np.float64), np.asarray(gt, np.float64)
    if pred.ndim == 3:
        pred, gt = pred[None], gt[None]
    out = {"psnr": [], "ssim": [], "mse": []}
    for p, g in zip(pred, gt):
        mse = np.mean((p - g) ** 2)
        with np.errstate(divide="ignore"):
            out["psnr"].append(10.0 * np.log10(1.0 / mse) if mse > 0 else np.inf)
        out["mse"].append(mse)
        out["ssim"].append(ssim_map(p, g, L).mean())
    return {k: np.array(v) for k, v in out.items()}
