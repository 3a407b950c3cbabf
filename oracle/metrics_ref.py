"""TEST INFRASTRUCTURE ONLY (imported by tests/, never by the product path).

float64 numpy restatement of the image-quality metrics of csrc/metrics.cu (snrf_image_metrics, metrics.image_metrics):
  SSIM as pytorch-ssim computes it: an 11 x 11 Gaussian window w = outer(g, g), g[i] ~ exp(-(i - 5)^2 / 4.5) normalised
  (sigma 1.5); per channel, zero-padded correlation with padding 5 -- F.conv2d(img, window, padding=5, groups=3) --
  gives mu_x, mu_y, s_xx = E[x^2] - mu_x^2, s_yy, s_xy = E[xy] - mu_x mu_y; the map is
  ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)), C1 = 0.01^2, C2 = 0.03^2.
  The mask only selects which map values and squared errors are averaged (over the masked pixels and the 3 channels).
  uint8 ground truth is read as float32(v) / float32(255).
The window is applied as two 1-D passes (the same sums as the 2-D window up to rounding); tests/test_metrics_cpu.py
pins this against a direct loop over window positions and against torch's F.conv2d.
"""
import numpy as np

C1, C2 = 0.01 ** 2, 0.03 ** 2


def gaussian_window():
    i = np.arange(11, dtype=np.float64)
    g = np.exp(-((i - 5.0) ** 2) / 4.5)
    return g / g.sum()


def local_mean(img, g=None):
    """[H, W] float64 -> the zero-padded (padding 5) correlation with outer(g, g), [H, W]."""
    g = gaussian_window() if g is None else g
    H, W = img.shape
    p = np.zeros((H + 10, W + 10))
    p[5:5 + H, 5:5 + W] = img
    h = sum(g[k] * p[:, k:k + W] for k in range(11))
    return sum(g[k] * h[k:k + H, :] for k in range(11))


def ssim_map(x, y):
    """x, y [H, W, 3] float64 -> the SSIM map [H, W, 3]."""
    out = np.empty(x.shape)
    for c in range(x.shape[-1]):
        a, b = x[..., c], y[..., c]
        mx, my = local_mean(a), local_mean(b)
        sxx, syy, sxy = local_mean(a * a) - mx * mx, local_mean(b * b) - my * my, local_mean(a * b) - mx * my
        out[..., c] = ((2 * mx * my + C1) * (2 * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2))
    return out


def to_unit(img):
    """uint8 -> float32(v) / float32(255); float -> as is; both as float64."""
    img = np.asarray(img)
    if img.dtype == np.uint8:
        return (img.astype(np.float32) / np.float32(255.0)).astype(np.float64)
    return img.astype(np.float64)


def image_metrics(pred, gt, mask=None):
    """pred, gt [N, H, W, 3] (or [H, W, 3]); mask [N, H, W] / [N, H, W, 1] bool or None.
    -> {"mse", "psnr", "ssim", "count"}: float64 arrays [N] (NaN MSE / SSIM where the mask is empty)."""
    x, y = to_unit(pred), to_unit(gt)
    if x.ndim == 3:
        x, y = x[None], y[None]
        mask = None if mask is None else np.asarray(mask)[None]
    N, H, W, _ = x.shape
    m = np.ones((N, H, W), dtype=bool) if mask is None else np.asarray(mask).reshape(N, H, W).astype(bool)
    out = {k: np.empty(N) for k in ("mse", "psnr", "ssim", "count")}
    for n in range(N):
        cnt = int(m[n].sum())
        out["count"][n] = cnt
        if cnt == 0:
            out["mse"][n] = out["ssim"][n] = out["psnr"][n] = np.nan
            continue
        out["ssim"][n] = ssim_map(x[n], y[n])[m[n]].sum() / (3.0 * cnt)
        out["mse"][n] = ((x[n] - y[n]) ** 2)[m[n]].sum() / (3.0 * cnt)
        with np.errstate(divide="ignore"):
            out["psnr"][n] = -10.0 * np.log10(out["mse"][n])
    return out
