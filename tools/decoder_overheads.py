#!/usr/bin/env python
"""Fixed cost of the decoder kernels (weight staging incl. the composed matrices, TMEM allocation, gradient flush) against their
per-tile cost: forward / backward on N = 148 x 128 x k samples for k = 1, 4, 16, 64, 221 tiles per CTA (evidence for DESIGN 4.3).
  python tools/decoder_overheads.py [--out profiles/r4_decoder_overheads.json]"""
import argparse
import importlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_decoder_overheads.json"))
    args = ap.parse_args()
    pkg = importlib.import_module(bench.PKG)
    pkg.install()
    from hashgrid import _decoder, _field
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    dec = _decoder.ShallowMLP(32).to(dev)
    params = [p.detach().requires_grad_(True) for p in _decoder.decoder_params(dec)]
    S = 128
    rows = []
    for k in (1, 4, 16, 64, 221):
        N = 148 * 128 * k
        feats = (torch.randn(16, N, 2, device=dev) * 0.3).requires_grad_(True)
        rays_d = torch.randn(N // S, 3, device=dev)
        mask = torch.ones(32, device=dev)
        cot = torch.randn(N, 10, device=dev)

        def run():
            for q in params:                       # (as the training step: gradients start from None, autograd steals the kernel's buffers)
                q.grad = None
            feats.grad = None
            heads = _field.decoder_apply(feats, rays_d, mask, S, params)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            torch.cuda._sleep(30_000_000)          # the device idles ~15 ms while the host queues the launches: GPU time, not launch latency
            e[0].record()
            heads.backward(cot)
            e[1].record()
            return e
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fw, bw = [], []
        for _ in range(10):
            torch.cuda._sleep(10_000_000)
            f0.record()
            with torch.no_grad():
                _field.decoder_forward(feats.detach(), mask, rays_d, S, params)
            f1.record()
            e = run()
            torch.cuda.synchronize()
            fw.append(f0.elapsed_time(f1)); bw.append(e[0].elapsed_time(e[1]))
        row = {"tiles_per_cta": k, "samples": N, "fwd_ms": sorted(fw)[len(fw) // 2], "bwd_ms_incl_absmax": sorted(bw)[len(bw) // 2]}
        rows.append(row)
        print(json.dumps(row), flush=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rows) + "\n")


if __name__ == "__main__":
    main()
