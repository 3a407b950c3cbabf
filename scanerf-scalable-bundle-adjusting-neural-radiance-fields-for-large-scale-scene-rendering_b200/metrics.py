"""Image-quality metrics of rendered views on the device: per-image MSE, PSNR and SSIM (csrc/metrics.cu).

The reference scores held-out views on the host every 1000 training steps (tile.py:810-864) and in
rendering.py's `val` mode, with tools/ssim.py.  Here one call scores a batch of images without leaving
the device and without a host synchronisation, so a training loop or a frame renderer can evaluate as it goes.

SSIM is the formulation of pytorch-ssim, which NeRF code of this lineage ships:
  - window: 11 x 11 Gaussian, sigma 1.5, the outer product of the normalised g[i] ~ exp(-(i - 5)^2 / 4.5);
  - local statistics per channel by zero-padded correlation (padding 5), i.e. F.conv2d(img, window, padding=5, groups=3):
    mu_x, mu_y, s_xx = E[x^2] - mu_x^2, s_yy = E[y^2] - mu_y^2, s_xy = E[xy] - mu_x mu_y;
  - map ((2 mu_x mu_y + C1)(2 s_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(s_xx + s_yy + C2)), C1 = 0.01^2, C2 = 0.03^2;
  - the mask does not change the local statistics, it selects which map values and squared errors are averaged.
MSE and SSIM are means over the masked pixels and the 3 channels; an image whose mask is empty gets NaN and count 0.
"""
import ctypes

import torch

import scanerf_b200_capi as capi

_TILE_H, _TILE_W = 16, 32          # output tile of one CTA of csrc/metrics.cu: the scratch holds 3 doubles per tile


def _check(t, name, dtypes):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t)}")
    capi._require_cuda(t, name)
    if t.dtype not in dtypes:
        raise RuntimeError(f"{name} must have dtype {' or '.join(str(d) for d in dtypes)}, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")


def image_metrics(pred, gt, mask=None):
    """pred [N,H,W,3] (or [H,W,3], taken as N = 1) float32; gt of the same shape, uint8 (divided by 255) or float32
    in [0, 1]; mask None or bool [N,H,W] / [N,H,W,1] (True = score the pixel).
    -> {"mse", "psnr", "ssim", "count"}: float32 device tensors [N]; psnr = -10 log10(mse)."""
    _check(pred, "pred", (torch.float32,))
    _check(gt, "gt", (torch.uint8, torch.float32))
    if pred.dim() not in (3, 4) or pred.shape[-1] != 3:
        raise RuntimeError(f"pred must be [N,H,W,3] or [H,W,3], got {tuple(pred.shape)}")
    if gt.shape != pred.shape:
        raise RuntimeError(f"gt has shape {tuple(gt.shape)}, pred {tuple(pred.shape)}")
    if gt.device != pred.device:
        raise RuntimeError(f"gt lives on {gt.device}, pred on {pred.device}")
    N, H, W = (1,) + tuple(pred.shape[:2]) if pred.dim() == 3 else tuple(pred.shape[:3])
    if mask is not None:
        _check(mask, "mask", (torch.bool,))
        lead = tuple(pred.shape[:-1])
        if tuple(mask.shape) not in (lead, lead + (1,)):
            raise RuntimeError(f"mask must have shape {lead} or {lead + (1,)}, got {tuple(mask.shape)}")
        if mask.device != pred.device:
            raise RuntimeError(f"mask lives on {mask.device}, pred on {pred.device}")
    out = torch.empty(3, N, dtype=torch.float32, device=pred.device)
    tiles = -(-H // _TILE_H) * -(-W // _TILE_W)
    scratch = torch.empty(max(N * tiles * 3, 1), dtype=torch.float64, device=pred.device)
    capi.check(capi.lib().snrf_image_metrics(
        capi.ptr(pred), capi.ptr(gt), capi.c_int(int(gt.dtype == torch.uint8)), capi.ptr(mask),
        capi.c_int(N), capi.c_int(H), capi.c_int(W), capi.ptr(out[0]), capi.ptr(out[1]), capi.ptr(out[2]),
        capi.ptr(scratch), ctypes.c_size_t(scratch.numel() * 8), capi.stream()), "snrf_image_metrics")
    mse, ssim, count = out.unbind(0)
    return {"mse": mse, "psnr": -10.0 * torch.log10(mse), "ssim": ssim, "count": count}


def with_means(m):
    """Per-view metrics -> the same dict plus "mean_mse", "mean_psnr", "mean_ssim" (means over the views with a non-empty
    mask), as device scalars."""
    m = dict(m)
    for k in ("mse", "psnr", "ssim"):
        m["mean_" + k] = torch.nanmean(m[k])
    return m

