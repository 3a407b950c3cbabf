"""GPU: the image metrics kernel (csrc/metrics.cu via metrics.image_metrics) against the float64 restatement
(oracle/metrics_ref.py) from 1x1 to 1080p, its determinism and input checks; TileStep.render_image against the
hand-written chunk loop, TileStep.evaluate on a trained tile, render_frame.evaluate_frames against image_metrics of
render_frame's output, and neither of the two synchronising with the host.
Bars: mean SSIM within 1e-5 absolute, MSE within 1e-6 relative, PSNR within 1e-4 dB."""
import os
import tempfile

import numpy as np
import pytest
import torch

import scenes
from conftest import load_pkg
from oracle import metrics_ref as mr
from test_psnr_gpu import _target
from test_sync_free_gpu import _sync_warnings
from test_tile_step_gpu import _tile

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
SSIM_TOL, MSE_RTOL, PSNR_TOL = 1e-5, 1e-6, 1e-4


def _images(N, H, W, seed):
    gen = torch.Generator().manual_seed(seed)
    pred = torch.rand(N, H, W, 3, generator=gen)
    gt = (pred + 0.08 * torch.randn(N, H, W, 3, generator=gen)).clamp(0, 1)
    return pred, gt


def _compare(got, ref, label):
    ref_cnt = ref["count"]
    assert np.array_equal(got["count"].cpu().numpy(), ref_cnt), label
    live = ref_cnt > 0
    g = {k: got[k].double().cpu().numpy() for k in ("mse", "psnr", "ssim")}
    for k in ("mse", "psnr", "ssim"):
        assert np.all(np.isnan(g[k][~live])), (label, k, g[k])
    if not live.any():
        return
    e_ssim = float(np.abs(g["ssim"][live] - ref["ssim"][live]).max())
    e_mse = float((np.abs(g["mse"][live] - ref["mse"][live]) / ref["mse"][live]).max())
    e_psnr = float(np.abs(g["psnr"][live] - ref["psnr"][live]).max())
    print(f"{label}: max |dSSIM| {e_ssim:.2e}, max rel dMSE {e_mse:.2e}, max |dPSNR| {e_psnr:.2e} dB "
          f"(SSIM {ref['ssim'][live].min():.4f}..{ref['ssim'][live].max():.4f})")
    assert e_ssim <= SSIM_TOL and e_mse <= MSE_RTOL and e_psnr <= PSNR_TOL, label


@pytest.mark.parametrize("N,H,W", [(3, 1, 1), (3, 7, 5), (3, 37, 53), (2, 540, 960), (2, 1080, 1920)])
@pytest.mark.parametrize("gt_dtype", ["uint8", "float32"])
def test_kernel_matches_restatement(N, H, W, gt_dtype):
    load_pkg()
    from metrics import image_metrics
    pred, gt = _images(N, H, W, N * H * W)
    if gt_dtype == "uint8":
        gt = (gt * 255).round().to(torch.uint8)
    pred_np, gt_np = pred.numpy(), gt.numpy()
    pd, gd = pred.to(DEV), gt.to(DEV)
    _compare(image_metrics(pd, gd), mr.image_metrics(pred_np, gt_np), f"{N}x{H}x{W} {gt_dtype}")
    # a random mask on image 0, all-false on image 1, all-true on the rest; [N,H,W] and [N,H,W,1] alike
    mask = torch.rand(N, H, W, generator=torch.Generator().manual_seed(7)) < 0.4
    mask[1] = False
    mask[2:] = True
    ref = mr.image_metrics(pred_np, gt_np, mask.numpy())
    _compare(image_metrics(pd, gd, mask.to(DEV)), ref, f"{N}x{H}x{W} {gt_dtype} masked")
    _compare(image_metrics(pd, gd, mask[..., None].to(DEV)), ref, f"{N}x{H}x{W} {gt_dtype} masked [N,H,W,1]")
    # one image as [H,W,3]
    one = image_metrics(pd[0], gd[0])
    assert one["ssim"].shape == (1,)
    _compare(one, mr.image_metrics(pred_np[:1], gt_np[:1]), f"{H}x{W} {gt_dtype} single")


def test_all_false_mask_gives_nan_and_zero_count():
    load_pkg()
    from metrics import image_metrics
    pred, gt = _images(2, 40, 70, 1)
    m = image_metrics(pred.to(DEV), gt.to(DEV), torch.zeros(2, 40, 70, dtype=torch.bool, device=DEV))
    assert torch.equal(m["count"].cpu(), torch.zeros(2))
    for k in ("mse", "psnr", "ssim"):
        assert torch.isnan(m[k]).all(), k


def test_identical_images():
    load_pkg()
    from metrics import image_metrics
    pred, _ = _images(2, 45, 77, 2)
    m = image_metrics(pred.to(DEV), pred.to(DEV))
    assert torch.equal(m["mse"].cpu(), torch.zeros(2)) and torch.isinf(m["psnr"]).all()
    assert (m["ssim"] - 1).abs().max().item() < 1e-6


def test_two_calls_are_bit_identical():
    load_pkg()
    from metrics import image_metrics
    pred, gt = _images(2, 540, 960, 3)
    mask = (torch.rand(2, 540, 960, generator=torch.Generator().manual_seed(5)) < 0.5).to(DEV)
    a = image_metrics(pred.to(DEV), gt.to(DEV), mask)
    b = image_metrics(pred.to(DEV), gt.to(DEV), mask)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_bad_inputs_are_refused():
    load_pkg()
    from metrics import image_metrics
    pred, gt = _images(2, 16, 24, 4)
    pd, gd = pred.to(DEV), gt.to(DEV)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        image_metrics(pred, gd)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        image_metrics(pd, gt)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        image_metrics(pd, gd, torch.ones(2, 16, 24, dtype=torch.bool))
    with pytest.raises(RuntimeError, match="contiguous"):
        image_metrics(pd.transpose(1, 2).contiguous().transpose(1, 2), gd)
    with pytest.raises(RuntimeError, match="contiguous"):
        image_metrics(pd, gd.transpose(1, 2).contiguous().transpose(1, 2))
    with pytest.raises(RuntimeError, match="contiguous"):
        image_metrics(pd, gd, torch.ones(2, 24, 16, dtype=torch.bool, device=DEV).transpose(1, 2))
    with pytest.raises(RuntimeError, match="shape"):
        image_metrics(pd, gd[:, :15].contiguous())
    with pytest.raises(RuntimeError, match=r"\[N,H,W,3\]"):
        image_metrics(pd[..., :2].contiguous(), gd[..., :2].contiguous())
    with pytest.raises(RuntimeError, match="shape"):
        image_metrics(pd, gd, torch.ones(2, 16, 23, dtype=torch.bool, device=DEV))
    with pytest.raises(RuntimeError, match="dtype"):
        image_metrics(pd.double(), gd)
    with pytest.raises(RuntimeError, match="dtype"):
        image_metrics(pd, gd.half())
    with pytest.raises(RuntimeError, match="dtype"):
        image_metrics(pd, gd, torch.ones(2, 16, 24, dtype=torch.uint8, device=DEV))


@pytest.mark.parametrize("stride,chunk", [(1, 1 << 16), (1, 1000), (2, 700)])
def test_render_image_matches_chunked_render_rays(stride, chunk):
    load_pkg()
    from hashgrid import INFERENCE
    step, _, _ = _tile(DEV)
    H, W = 48, 64
    for view in (0, 3):
        color, depth = step.render_image(view, H, W, stride=stride, chunk=chunk)
        rays_o, rays_d = step.full_image_rays(view, H, W, stride)
        n = rays_o.shape[0]
        assert n == color.shape[0] * color.shape[1]
        ref_c, ref_d = torch.zeros(n, 3, device=DEV), torch.zeros(n, 1, device=DEV)
        with torch.no_grad():
            for b in range(0, n, chunk):
                out, ok = step.render_rays(rays_o[b:b + chunk].contiguous(), rays_d[b:b + chunk].contiguous(), None, INFERENCE)
                if ok:
                    ref_c[b:b + chunk], ref_d[b:b + chunk] = out["pred_color"], out["pred_depth"]
        h, w = -(-H // stride), -(-W // stride)
        assert color.shape == (h, w, 3) and depth.shape == (h, w, 1)
        assert torch.equal(color, ref_c.reshape(h, w, 3)) and torch.equal(depth, ref_d.reshape(h, w, 1))
        assert color.abs().sum().item() > 0


def test_render_shared_depth_is_unchanged_on_render_image():
    """render_shared_depth renders through render_image: the maps equal the chunk loop it used to run itself."""
    import types
    load_pkg()
    from hashgrid import INFERENCE
    step, _, _ = _tile(DEV)
    H, W, batch = 47, 63, 1000
    step.consensus = types.SimpleNamespace(overlap_flags=torch.tensor([True, False, True, True], device=DEV))
    step.camera_ids = torch.tensor([10, 11, 12, 13], device=DEV)
    ids, maps = step.render_shared_depth(H, W, batch=batch)
    center, half = step.featureGrid.bbox_center, step.featureGrid.bbox_size / 2.0
    ref_ids, ref_maps = [], []
    with torch.no_grad():
        for i in (0, 2, 3):
            rays_o, rays_d = step.full_image_rays(i, H, W, stride=2)
            if not bool(torch.all(torch.abs(rays_o[0] - center) < half / 2.0)):
                continue
            depth = torch.zeros(rays_o.shape[0], 1, device=DEV)
            for b in range(0, rays_o.shape[0], batch):
                out, ok = step.render_rays(rays_o[b:b + batch].contiguous(), rays_d[b:b + batch].contiguous(), None, INFERENCE)
                if ok:
                    depth[b:b + batch] = out["pred_depth"]
            ref_ids.append(10 + i)
            ref_maps.append(depth.reshape((H + 1) // 2, (W + 1) // 2))
    assert ref_ids, "no camera inside the tile: the comparison would be empty"
    assert ids.tolist() == ref_ids
    assert torch.equal(maps, torch.stack(ref_maps))


def _trainable_tile():
    from tile_step import TileStep
    H, W, n_cam = 48, 64, 8
    gen = torch.Generator().manual_seed(0)
    Ks, c2w = scenes.camera_rig(n_cam, H, W, gen, center=(10.37, 3.21, 15.53), radius=4.83, fx=60.0)
    ply = os.path.join(tempfile.mkdtemp(), "mesh.ply")
    scenes.write_proxy_mesh_ply(ply, (0, 0, 0), (20, 13, 30), seed=0, ground_res=16, n_boxes=6)
    torch.manual_seed(0)
    step = TileStep(DEV, (0.0, 0.0, 0.0), (20.0, 13.0, 30.0), Ks, c2w, log2_hashmap_size=15, grid_resolution=(16, 512),
                    num_sample=32, num_bg_sample=32, mesh_path=ply, global_step=6000)
    ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    images = torch.stack([_target(torch.stack([torch.full_like(xs, v), xs, ys], -1).reshape(-1, 3), H, W).reshape(H, W, 3)
                          for v in range(n_cam)])
    return step, images, gen, H, W, n_cam


def test_evaluate_psnr_rises_with_training():
    load_pkg()
    step, images, gen, H, W, n_cam = _trainable_tile()
    img = images.to(DEV)
    views = list(range(n_cam))
    m0 = step.evaluate(views, img)
    for _ in range(200):
        locs = torch.stack([torch.randint(0, n_cam, (512,), generator=gen), torch.randint(0, W, (512,), generator=gen),
                            torch.randint(0, H, (512,), generator=gen)], -1).int()
        step.step_device(locs.to(DEV), _target(locs, H, W).to(DEV))
    m1 = step.evaluate(views, img)
    # the MSE of the kernel is torch's mean of the rendered images' squared error
    for v in views:
        color, _ = step.render_image(v, H, W)
        ref = torch.mean((color - img[v]) ** 2).item()
        assert abs(m1["mse"][v].item() - ref) <= MSE_RTOL * ref, (v, m1["mse"][v].item(), ref)
    assert torch.equal(m1["count"].cpu(), torch.full((n_cam,), float(H * W)))
    p0, p1 = m0["mean_psnr"].item(), m1["mean_psnr"].item()
    s0, s1 = m0["mean_ssim"].item(), m1["mean_ssim"].item()
    print(f"evaluate: mean PSNR {p0:.2f} -> {p1:.2f} dB, mean SSIM {s0:.4f} -> {s1:.4f} after 200 steps")
    assert p1 > p0 + 1.0, (p0, p1)
    assert abs(p1 - m1["psnr"].mean().item()) < 1e-4
    # masks: only the masked pixels are scored
    mask = torch.zeros(n_cam, H, W, 1, dtype=torch.bool, device=DEV)
    mask[:, 10:30, 5:50] = True
    mm = step.evaluate(views, img, mask)
    assert torch.equal(mm["count"].cpu(), torch.full((n_cam,), 20.0 * 45.0))


def test_evaluate_frames_matches_image_metrics_of_render_frame():
    load_pkg()
    import render_frame as rf
    from metrics import image_metrics
    step, _, _ = _tile(DEV)
    ts = rf.TileSet.from_hashgrid(step.featureGrid, step.decoder, DEV).finalize()
    H, W = 40, 56
    with torch.no_grad():
        c2ws = step.poses.c2w()[:3].detach()
    Ks = step.poses.ks[:3]
    gen = torch.Generator().manual_seed(9)
    images = (torch.rand(3, H, W, 3, generator=gen) * 255).to(torch.uint8).to(DEV)
    mask = (torch.rand(3, H, W, generator=gen) < 0.7).to(DEV)
    got = rf.evaluate_frames(ts, Ks, c2ws, images, H, W, masks=mask, adaptive=False)
    frames = []
    for k in range(3):
        d, s, _, _ = rf.render_frame(ts, H, W, Ks[k], c2ws[k], adaptive=False)
        frames.append(torch.clamp(d + s, 0, 1))
    ref = image_metrics(torch.stack(frames), images, mask)
    for k in ("mse", "psnr", "ssim", "count"):
        assert torch.equal(got[k], ref[k]), k
    torch.testing.assert_close(got["mean_psnr"], ref["psnr"].mean())


def test_evaluate_and_evaluate_frames_do_not_synchronise():
    load_pkg()
    import render_frame as rf
    step, images, _, H, W, n_cam = _trainable_tile()
    img = images.to(DEV)
    views = list(range(n_cam))
    step.evaluate(views, img)                              # first call: allocator warm-up
    assert _sync_warnings(lambda: step.evaluate(views, img)) == []
    ts = rf.TileSet.from_hashgrid(step.featureGrid, step.decoder, DEV).finalize()
    with torch.no_grad():
        c2ws = step.poses.c2w().detach()
    Ks = step.poses.ks
    rf.evaluate_frames(ts, Ks, c2ws, img, H, W, adaptive=False)
    assert _sync_warnings(lambda: rf.evaluate_frames(ts, Ks, c2ws, img, H, W, adaptive=False)) == []
    # the detector does see a synchronisation when there is one
    assert len(_sync_warnings(lambda: step.evaluate(views, img)["mean_psnr"].item())) >= 1
