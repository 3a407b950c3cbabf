#!/usr/bin/env python
"""A/B of decoder-backward scheduling knobs on the bench workload (evidence for DESIGN 4.3; not a bench arm).
  python tools/sweep_decoder.py [--out profiles/r3_decoder_sweep.json]"""
import argparse
import ctypes
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_decoder_sweep.json"))
    args = ap.parse_args()
    pkg = importlib.import_module(bench.PKG)
    pkg.install()
    import scanerf_b200_capi as capi
    cfg = bench.WORKLOADS["default.yaml-single-tile"]
    dev = torch.device("cuda:0")
    step, gen = bench.build_tile(cfg, dev, 0)
    batches = [(l.to(dev), g.to(dev)) for l, g in bench.make_batches(cfg, 14, gen)]
    lib = capi.lib()
    rows = []
    names = ("snrf_decoder_fwd", "snrf_decoder_bwd", "snrf_field_encode_fwd", "snrf_field_encode_bwd_adam")
    for merged, fold in ((2, 1), (2, 0), (1, 0), (2, 1), (2, 0), (0, 0), (2, 1)):
        lib.snrf_decoder_set_bwd_merged(ctypes.c_int(merged))
        lib.snrf_decoder_set_fwd_fold(ctypes.c_int(fold))
        ms, loss = bench._time_steps(step, batches, 4)
        capi.time_calls(names)
        for b in batches[:8]:
            step.step_device(*b)
        t = capi.timed_by_name()
        capi.time_calls(None)
        row = {"bwd_merged": merged, "fwd_fold": fold, "ms_per_step": ms, "loss": loss}
        for k in names:
            row[k + "_ms"] = sum(t.get(k, [])) / max(len(t.get(k, [])), 1)
        if merged == 2 and fold == 1:               # the render's decode pass always folds layer 2
            r = bench.bench_render(step, cfg, dev, frames=3, warm=1)
            row["render_ms_per_frame"] = r["ms_per_frame"]
        rows.append(row)
        print(json.dumps(row), flush=True)
    lib.snrf_decoder_set_bwd_merged(ctypes.c_int(2))
    lib.snrf_decoder_set_fwd_fold(ctypes.c_int(1))
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rows) + "\n")


if __name__ == "__main__":
    main()
