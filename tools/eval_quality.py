"""Image quality of a trained tile, and the cost of measuring it.

Trains bench.py's default tile (config/default.yaml shape: 64 cameras at 960x540, 2^24-entry table, 128 + 128 samples)
for --steps steps on a smooth per-camera target image, once with the default step and once with early ray termination
(TileStep(ert_eps=1e-4)), on the same batches.  Each is scored with TileStep.evaluate on --views full-resolution views,
masked to the pixels that no training batch contained (held-out pixels).  Then times, with CUDA events,
TileStep.evaluate of one 960x540 view and metrics.image_metrics over a batch of 1080p frames (f32 prediction, uint8
ground truth, 8 frames = 250 MB of inputs: twice the L2, so they stream from HBM).  Prints one JSON line with the
device name and its power limit, queried in the same run.

    python tools/eval_quality.py [--steps 1000] [--views 4] [--frames 8]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402

DEV = torch.device("cuda:0")


def device_info():
    info = {"device": torch.cuda.get_device_name(DEV)}
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                       "-i", str(DEV.index or 0)], text=True, timeout=30)
        name, power, clock = [f.strip() for f in out.strip().splitlines()[0].split(",")]
        info.update({"smi_name": name, "power_limit": power, "sm_max_clock": clock})
    except Exception as e:   # the numbers below are still device-event times; say that the limit is unknown
        info["power_limit"] = f"not available ({type(e).__name__})"
    return info


def event_ms(fn, iters, warmup=2):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--views", type=int, default=4, help="cameras scored (evenly spaced)")
    ap.add_argument("--frames", type=int, default=8, help="1080p frames per image_metrics call in the timing")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_quality.py measures on a CUDA device; none is available")
    importlib.import_module(bench.PKG).install()
    from metrics import image_metrics
    from test_psnr_gpu import _target

    cfg = bench.WORKLOADS["default.yaml-single-tile"]
    H, W, n_cam = cfg["H"], cfg["W"], cfg["n_cam"]
    views = [round(i * n_cam / args.views) for i in range(args.views)]
    ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    images = torch.stack([_target(torch.stack([torch.full_like(xs, v), xs, ys], -1).reshape(-1, 3), H, W).reshape(H, W, 3)
                          for v in views]).to(DEV)
    slot = torch.full((n_cam,), -1, dtype=torch.long)
    slot[views] = torch.arange(len(views))
    slot = slot.to(DEV)

    gen = torch.Generator().manual_seed(0)
    batches = [(locs.to(DEV), _target(locs, H, W).to(DEV)) for locs, _ in bench.make_batches(cfg, args.steps, gen)]
    held_out = torch.ones(len(views), H, W, dtype=torch.bool, device=DEV)
    for locs, _ in batches:                                       # pixels of the scored views that training saw
        s = slot[locs[:, 0].long()]
        keep = s >= 0
        held_out[s[keep], locs[keep, 2].long(), locs[keep, 1].long()] = False

    quality = {}
    for name, kw in (("default", {}), ("ert_eps=1e-4", {"ert_eps": 1e-4})):
        step, _ = bench.build_tile(cfg, DEV, seed=0)
        step.featureGrid.ert_eps = float(kw.get("ert_eps", 0.0))
        before = step.evaluate(views, images, held_out)
        for locs, gt in batches:
            step.step_device(locs, gt)
        after = step.evaluate(views, images, held_out)
        quality[name] = {"psnr_db_step0": round(before["mean_psnr"].item(), 3), "psnr_db": round(after["mean_psnr"].item(), 3),
                         "ssim_step0": round(before["mean_ssim"].item(), 5), "ssim": round(after["mean_ssim"].item(), 5),
                         "psnr_db_per_view": [round(v, 3) for v in after["psnr"].tolist()]}
    held_px = int(held_out.sum().item())

    eval_ms = event_ms(lambda: step.evaluate(views[:1], images[:1], held_out[:1]), iters=10)
    gen = torch.Generator().manual_seed(1)
    pred = torch.rand(args.frames, 1080, 1920, 3, generator=gen).to(DEV)
    gt = (torch.rand(args.frames, 1080, 1920, 3, generator=gen) * 255).to(torch.uint8).to(DEV)
    metrics_ms = event_ms(lambda: image_metrics(pred, gt), iters=20)

    print(json.dumps({
        "workload": "default.yaml-single-tile", "train_steps": args.steps, "views": views, "held_out_pixels": held_px,
        "quality": quality,
        "evaluate_ms_per_960x540_view": round(eval_ms, 3),
        "image_metrics_ms_per_call": round(metrics_ms, 3), "image_metrics_frames_per_call": args.frames,
        "image_metrics_ms_per_1080p_frame": round(metrics_ms / args.frames, 4),
        **device_info()}))


if __name__ == "__main__":
    main()
