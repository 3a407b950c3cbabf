"""CPU: the float64 restatement of the image metrics (oracle/metrics_ref.py) against the SSIM definition itself -- a
direct loop over window positions, torch's F.conv2d(..., padding=5, groups=3) in float64 -- and closed-form cases."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import metrics_ref as mr


def _direct_ssim_map(x, y):
    """The definition term by term: every pixel, every window position, zero outside the image."""
    i = np.arange(11.0)
    g = np.exp(-((i - 5) ** 2) / 4.5)
    w = np.outer(g / g.sum(), g / g.sum())
    H, W, C = x.shape
    out = np.empty(x.shape)
    for c in range(C):
        for py in range(H):
            for px in range(W):
                m = np.zeros(5)
                for a in range(11):
                    for b in range(11):
                        yy, xx = py + a - 5, px + b - 5
                        if 0 <= yy < H and 0 <= xx < W:
                            u, v = x[yy, xx, c], y[yy, xx, c]
                            m += w[a, b] * np.array([u, v, u * u, v * v, u * v])
                sxx, syy, sxy = m[2] - m[0] ** 2, m[3] - m[1] ** 2, m[4] - m[0] * m[1]
                out[py, px, c] = ((2 * m[0] * m[1] + mr.C1) * (2 * sxy + mr.C2)) / \
                    ((m[0] ** 2 + m[1] ** 2 + mr.C1) * (sxx + syy + mr.C2))
    return out


def _conv_ssim_map(x, y):
    """pytorch-ssim's _ssim in float64: F.conv2d with the 2-D window, padding 5, one group per channel."""
    g = torch.tensor(mr.gaussian_window(), dtype=torch.float64)
    win = (g[:, None] @ g[None, :]).expand(3, 1, 11, 11).contiguous()
    a = torch.tensor(x).permute(2, 0, 1)[None]
    b = torch.tensor(y).permute(2, 0, 1)[None]
    mu1, mu2 = F.conv2d(a, win, padding=5, groups=3), F.conv2d(b, win, padding=5, groups=3)
    s11 = F.conv2d(a * a, win, padding=5, groups=3) - mu1 * mu1
    s22 = F.conv2d(b * b, win, padding=5, groups=3) - mu2 * mu2
    s12 = F.conv2d(a * b, win, padding=5, groups=3) - mu1 * mu2
    m = ((2 * mu1 * mu2 + mr.C1) * (2 * s12 + mr.C2)) / ((mu1 * mu1 + mu2 * mu2 + mr.C1) * (s11 + s22 + mr.C2))
    return m[0].permute(1, 2, 0).numpy()


def _pair(H, W, seed):
    rng = np.random.default_rng(seed)
    x = rng.random((H, W, 3))
    return x, np.clip(x + 0.1 * rng.standard_normal((H, W, 3)), 0, 1)


def test_window_is_the_normalised_gaussian():
    g = mr.gaussian_window()
    assert g.shape == (11,) and abs(g.sum() - 1.0) < 1e-15
    assert np.array_equal(g, g[::-1])
    assert abs(g[4] / g[5] - math.exp(-1.0 / 4.5)) < 1e-14


@pytest.mark.parametrize("H,W", [(1, 1), (3, 4), (7, 5), (13, 9)])
def test_map_matches_direct_window_loop(H, W):
    x, y = _pair(H, W, H * 100 + W)
    assert np.abs(mr.ssim_map(x, y) - _direct_ssim_map(x, y)).max() < 1e-12


@pytest.mark.parametrize("H,W", [(1, 1), (7, 5), (37, 53), (64, 96)])
def test_map_matches_torch_conv2d(H, W):
    x, y = _pair(H, W, H + W)
    assert np.abs(mr.ssim_map(x, y) - _conv_ssim_map(x, y)).max() < 1e-12


def test_identical_images_give_one():
    x, _ = _pair(37, 53, 1)
    m = mr.image_metrics(x[None], x[None])
    assert abs(m["ssim"][0] - 1.0) < 1e-12 and m["mse"][0] == 0.0 and m["psnr"][0] == np.inf and m["count"][0] == 37 * 53


def test_constant_images():
    # interior pixels (window fully inside): sigma = 0, so SSIM = (2ab + C1) / (a^2 + b^2 + C1)
    a, b = 0.3, 0.7
    x, y = np.full((31, 31, 3), a), np.full((31, 31, 3), b)
    m = mr.ssim_map(x, y)
    assert abs(m[15, 15, 0] - (2 * a * b + mr.C1) / (a * a + b * b + mr.C1)) < 1e-12
    r = mr.image_metrics(x, y)
    assert abs(r["mse"][0] - (a - b) ** 2) < 1e-15
    assert abs(r["psnr"][0] + 10 * math.log10((a - b) ** 2)) < 1e-9


def test_symmetric_in_its_arguments():
    x, y = _pair(20, 30, 2)
    assert np.abs(mr.ssim_map(x, y) - mr.ssim_map(y, x)).max() < 1e-15


def test_mask_selects_but_does_not_change_statistics():
    x, y = _pair(20, 30, 3)
    mask = np.random.default_rng(4).random((20, 30)) < 0.3
    r = mr.image_metrics(x, y, mask[..., None])
    full = mr.ssim_map(x, y)
    assert r["count"][0] == mask.sum()
    assert abs(r["ssim"][0] - full[mask].mean()) < 1e-14
    assert abs(r["mse"][0] - ((x - y) ** 2)[mask].mean()) < 1e-15
    empty = mr.image_metrics(x, y, np.zeros((20, 30), dtype=bool))
    assert empty["count"][0] == 0 and np.isnan(empty["mse"][0]) and np.isnan(empty["ssim"][0])


def test_uint8_ground_truth_is_float32_division():
    v = np.arange(256, dtype=np.uint8).reshape(16, 16, 1).repeat(3, -1)
    assert np.array_equal(mr.to_unit(v), (torch.tensor(v).float() / torch.tensor(255.0)).double().numpy())
