#!/usr/bin/env python
"""Cost of HashGrid.render_batch_rays(out_normal=True) at the C2 size of one render chain (2^14 rays x 128 samples, 16 x 2^24
x 2 table, foreground contraction), five variants timed alternately with CUDA events after a warm-up:
  * fused:       out_normal=True on the fused path (field encode with Jacobians, snrf_field_normal, tensor-core decoder);
  * torch:       out_normal=True on the torch branch (fused_decoder = False: reference-shaped encode operator, fp32 torch
                 decoder, torch.autograd.grad of sigma w.r.t. the samples with create_graph);
  * no_normal:   the fused call without normals.
Each in INFERENCE (forward) and in TRAIN (forward + backward of rgb, depth, the specular regulariser and a normal term).  The
torch branch needs the rays in an autograd graph, so these three get rays that require grad, as pose-refined rays do; the
fused encode then writes its Jacobians with or without normals.  Rays outside any graph (a plain render) pay that write only
for the normal, so fused_plain / no_normal_plain repeat the fused pair with such rays.
Evidence for profiles/, not a bench arm.   python tools/normal_bench.py [--out profiles/normal_bench.json]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

PKG = "scanerf-scalable-bundle-adjusting-neural-radiance-fields-for-large-scale-scene-rendering_b200"


def card():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, limit = [s.strip() for s in q.splitlines()[0].split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError):
        name, limit = torch.cuda.get_device_name(0), "unknown"
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("normal_bench: needs a CUDA device")
    importlib.import_module(PKG).install()
    from hashgrid import HashGrid, INFERENCE, TRAIN
    from hashgrid._decoder import ShallowMLP
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    hg = HashGrid(dev, torch.tensor([0.0, 0.0, 0.0], device=dev), torch.tensor([20.0, 13.0, 30.0], device=dev), 24, [16, 2048], 4,
                  False, "")
    g = torch.Generator(device=dev).manual_seed(0)
    with torch.no_grad():
        hg.HE.features.copy_(torch.randn(hg.HE.features.shape, device=dev, generator=g) * 0.3)
    dec = ShallowMLP(32).to(dev)
    R, S = 2 ** 14, 128
    o = torch.tensor([10.0, 6.5, 15.0], device=dev) + torch.randn(R, 3, device=dev, generator=g)
    d = torch.nn.functional.normalize(torch.randn(R, 3, device=dev, generator=g), dim=-1)
    z = (torch.rand(R, S, device=dev, generator=g) * 6).sort(-1)[0]
    dist = torch.cat([z[:, 1:] - z[:, :-1], torch.full((R, 1), 1e-3, device=dev)], -1)
    c = torch.randn(R, 3, device=dev, generator=g)

    def run(variant, train):
        hg.fused_decoder = variant != "torch"
        plain = variant.endswith("_plain")
        oo, dd = (o, d) if plain else (o.clone().requires_grad_(True), d.clone().requires_grad_(True))
        out, _ = hg.render_batch_rays(oo, dd, z, dist, dec, TRAIN if train else INFERENCE, hg.contract_fore,
                                      out_normal=not variant.startswith("no_normal"), global_step=9000)
        if train:
            loss = out["rgb"].sum() + out["depth"].sum() * 0.01 + out["l2_reg_specular"]
            if "normal" in out:
                loss = loss + (out["normal"] * c).sum()
            hg.HE.features.grad = None
            dec.zero_grad(set_to_none=True)
            loss.backward()
        hg.fused_decoder = True

    variants = ["fused", "torch", "no_normal", "fused_plain", "no_normal_plain"]
    res = {}
    for train in (False, True):
        phase = "train_fwd_bwd" if train else "inference"
        for _ in range(args.warmup):
            for v in variants:
                run(v, train)
        times = {v: [] for v in variants}
        for _ in range(args.reps):
            for v in variants:
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                run(v, train)
                b.record()
                torch.cuda.synchronize()
                times[v].append(a.elapsed_time(b))
        res[phase] = {v: {"ms_median": sorted(t)[len(t) // 2], "ms": t} for v, t in times.items()}
    # the normal kernel by itself (CUDA events around its C-ABI call, fused INFERENCE calls)
    import scanerf_b200_capi as capi
    capi.time_calls("snrf_field_normal")
    for _ in range(args.reps):
        run("fused_plain", False)
    ms = capi.timed_by_name().get("snrf_field_normal", [])
    capi.time_calls(None)
    name, limit = card()
    result = {"card": name, "power_limit": limit, "rays": R, "samples": S, "table_log2": 24, "reps": args.reps,
              "warmup": args.warmup, "snrf_field_normal_ms": sorted(ms)[len(ms) // 2] if ms else None, **res}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
