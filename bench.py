#!/usr/bin/env python
"""Headline benchmark: single-tile training rays/s (fwd + bwd + optimiser) of the ScaNeRF
per-tile hot path at config/default.yaml shape, on N B200s (one tile per GPU, weak scaling).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the hot path over one batch of 2^14 synthetic rays:
  pose chain -> ray generation -> occupancy / inverse-z sample placement (128 + 128 per ray)
  -> contraction -> 16-level hash encode -> decoder MLP -> compositing -> MSE
  -> backward through all of it (incl. the analytic pose gradient) -> sparse Adam + Adam.
`value`   : rays/s with the batches already resident in HBM (CUDA-event timed).
`e2e`     : rays/s through TileStep.step(): pinned host batch in, python float loss out (the loss of that step, copied to
            pinned memory right after the forward and read back inside the call; the backward is queued behind it).
`roofline`: the dominant kernel (hash-encode backward) timed live with CUDA events on its stream.
`cpu_baseline` / --impl reference: the reference's math restated on the CPU (oracle/), timed on
            this box's host cores on a bounded sample of the same workload.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = "scanerf-scalable-bundle-adjusting-neural-radiance-fields-for-large-scale-scene-rendering_b200"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# ----------------------------------------------------------------------------- workload
WORKLOADS = {
    # BASELINE.json configs[1]: config/default.yaml single-tile training with pose refinement
    "default.yaml-single-tile": dict(tile_corner=(0.0, 0.0, 0.0), tile_size=(20.0, 13.0, 30.0), log2T=24,
                                     grid_resolution=(32, 8192), n_cam=64, H=540, W=960, fx=600.0,
                                     batch_log2=14, S=128, S_bg=128, sampler_log2dim=4),
    # BASELINE.json configs[0] shape (used by the CPU legs' bounded sample and by quick checks)
    "c1-small": dict(tile_corner=(0.0, 0.0, 0.0), tile_size=(20.0, 13.0, 30.0), log2T=19,
                     grid_resolution=(16, 512), n_cam=16, H=270, W=480, fx=300.0,
                     batch_log2=12, S=64, S_bg=64, sampler_log2dim=4),
}
# BASELINE.json configs[4] shape (8-GPU run: 64 tiles x 2^22-entry tables, 8 resident tiles per rank)
WORKLOADS["city-64-tiles"] = dict(WORKLOADS["default.yaml-single-tile"], log2T=22, tiles_total=64, n_cam=32, shared_cams=8)
ENC_FWD_BYTES, ENC_BWD_BYTES = 1164, 2200      # algorithmic bytes per sample point, SURVEY.md section 8(d)


def make_batches(cfg, n, gen):
    """`n` batches of (locs [B,3] i32 = (view, px, py), gt [B,3] f32): the same 2x2-patch pixel
    set for every camera, as TILE.train_one_step draws it (tile.py:902-915)."""
    import torch
    B = 2 ** cfg["batch_log2"]
    per_cam = B // cfg["n_cam"]
    n_patch = per_cam // 4
    out = []
    for _ in range(n):
        px = torch.randperm(cfg["W"] - 2, generator=gen)[:n_patch]
        py = torch.randperm(cfg["H"] - 2, generator=gen)[:n_patch]
        x = torch.stack([px, px + 1, px, px + 1], -1).reshape(-1)
        y = torch.stack([py, py, py + 1, py + 1], -1).reshape(-1)
        view = torch.arange(cfg["n_cam"]).repeat_interleave(x.numel())
        locs = torch.stack([view, x.repeat(cfg["n_cam"]), y.repeat(cfg["n_cam"])], -1).int()
        gt = torch.rand(locs.shape[0], 3, generator=gen)
        out.append((locs.contiguous(), gt.contiguous()))
    return out


def build_tile(cfg, dev, seed):
    import torch
    import scenes
    from tile_step import TileStep
    gen = torch.Generator().manual_seed(seed)
    c = [cfg["tile_corner"][i] + cfg["tile_size"][i] * f for i, f in enumerate((0.5, 0.25, 0.5))]
    Ks, c2w = scenes.camera_rig(cfg["n_cam"], cfg["H"], cfg["W"], gen, center=tuple(c),
                                radius=0.3 * min(cfg["tile_size"][0], cfg["tile_size"][2]), fx=cfg["fx"])
    tmp = tempfile.mkdtemp(prefix="snrf_bench_")
    ply = os.path.join(tmp, "mesh.ply")
    scenes.write_proxy_mesh_ply(ply, cfg["tile_corner"], cfg["tile_size"], seed=seed)
    torch.manual_seed(seed)
    step = TileStep(dev, cfg["tile_corner"], cfg["tile_size"], Ks, c2w, log2_hashmap_size=cfg["log2T"],
                    grid_resolution=cfg["grid_resolution"], num_sample=cfg["S"], num_bg_sample=cfg["S_bg"],
                    mesh_path=ply, sampler_log2dim=cfg["sampler_log2dim"], global_step=10000)
    return step, gen



def build_tile_row(cfg, dev, n_tiles, mine, overlap=0.2):
    """BASELINE configs[3] shape (config/community.yaml:5-12: TILE_SIZE [20,13,30], OVERLAP_RATIO 0.2): `n_tiles` tiles in a
    row along x, neighbours overlapping by 20 %.  Every tile has its own ring of cfg['n_cam'] cameras; the `shared` ring
    cameras of tile t nearest to tile t+1 are ALSO training views of tile t+1, where they replace that tile's `shared`
    cameras nearest to tile t -- so only the boundary cameras are seen by two tiles (the overlap set of the ADMM consensus).
    Builds the tiles listed in `mine`; returns ([TileStep], [generator], global camera count)."""
    import torch
    import scenes
    from tile_step import TileStep
    n_cam, shared = cfg["n_cam"], cfg.get("shared_cams", 16)
    size = cfg["tile_size"]
    rigs = []
    for t in range(n_tiles):                      # every rank derives the same global rig
        gen = torch.Generator().manual_seed(1000 + t)
        corner = (cfg["tile_corner"][0] + t * (1.0 - overlap) * size[0], cfg["tile_corner"][1], cfg["tile_corner"][2])
        c = [corner[i] + size[i] * f for i, f in enumerate((0.5, 0.25, 0.5))]
        Ks, c2w = scenes.camera_rig(n_cam, cfg["H"], cfg["W"], gen, center=tuple(c), radius=0.3 * min(size[0], size[2]), fx=cfg["fx"])
        order = torch.argsort(c2w[:, 0, 3])        # by camera x position
        rigs.append(dict(corner=corner, Ks=Ks, c2w=c2w, low=order[:shared], high=order[-shared:], ids=torch.arange(n_cam) + t * n_cam))
    steps, gens = [], []
    for t in mine:
        r = rigs[t]
        keep = torch.ones(n_cam, dtype=torch.bool)
        Ks, c2w, ids = r["Ks"], r["c2w"], r["ids"]
        if t > 0:                                  # swap my cameras nearest to the left neighbour for its cameras nearest to me
            keep[r["low"]] = False
            left = rigs[t - 1]
            Ks = torch.cat([Ks[keep], left["Ks"][left["high"]]])
            c2w = torch.cat([c2w[keep], left["c2w"][left["high"]]])
            ids = torch.cat([ids[keep], left["ids"][left["high"]]])
        tmp = tempfile.mkdtemp(prefix="snrf_bench_")
        ply = os.path.join(tmp, "mesh.ply")
        scenes.write_proxy_mesh_ply(ply, r["corner"], size, seed=t)
        torch.manual_seed(t)
        st = TileStep(dev, r["corner"], size, Ks, c2w, log2_hashmap_size=cfg["log2T"], grid_resolution=cfg["grid_resolution"],
                      num_sample=cfg["S"], num_bg_sample=cfg["S_bg"], mesh_path=ply, sampler_log2dim=cfg["sampler_log2dim"],
                      global_step=10000)
        st.enable_consensus(ids.tolist(), n_tiles * n_cam, rho=100.0)
        steps.append(st)
        gens.append(torch.Generator().manual_seed(2000 + t))
    return steps, gens, n_tiles * n_cam

# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first(self, timeout=8.0):
        """nvidia-smi needs a moment before its first line: the timed region (a fraction of a second) starts after it."""
        t_end = time.time() + timeout
        while self.proc is not None and not self.rows and time.time() < t_end:
            time.sleep(0.05)

    def summary(self, t0, t1):
        if self.proc is not None:
            time.sleep(0.15)                       # one more sampling interval, so that the end of the region is covered
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = max(mx, int(float(f[1])))
                if t0 <= t <= t1:
                    sm.append(int(float(f[0])))
                    reasons |= {n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")}
            except ValueError:
                continue
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU legs
class CpuPort:
    """The reference's math on the CPU (oracle/: C hash encode + torch MLP / compositing,
    fwd + bwd incl. grad_features and grad_points) on `rays` rays of the workload."""

    def __init__(self, cfg, rays, threads):
        import torch
        from oracle import torch_ref as tr
        self.tr, self.cfg, self.rays = tr, cfg, rays
        os.environ["ORACLE_THREADS"] = str(threads)
        torch.set_num_threads(threads)
        gen = torch.Generator().manual_seed(0)
        L, T = 16, 2 ** cfg["log2T"]
        size = torch.tensor(cfg["tile_size"]) * 2.0
        aspect = size / size.min()
        self.res = tr.resolution_ladder((aspect * cfg["grid_resolution"][0]).int(), (aspect * cfg["grid_resolution"][1]).int())
        self.table = (torch.randn(L, T, 2, generator=gen) * 1e-2).requires_grad_(True)
        self.mlp = {k: v.requires_grad_(True) for k, v in tr.init_mlp(gen).items()}
        center = torch.tensor(cfg["tile_corner"]) + torch.tensor(cfg["tile_size"]) / 2
        self.size, self.min_bbox = size, center - size / 2
        self.o = center + (torch.rand(rays, 3, generator=gen) - 0.5) * torch.tensor(cfg["tile_size"]) * 0.5
        self.d = torch.nn.functional.normalize(torch.randn(rays, 3, generator=gen), dim=-1)
        S, Sb = cfg["S"], cfg["S_bg"]
        self.z_f = torch.linspace(0.05, 0.45, S)[None] * float(min(cfg["tile_size"])) * torch.ones(rays, 1)
        self.d_f = torch.full_like(self.z_f, float(self.z_f[0, 1] - self.z_f[0, 0]))
        self.z_b, self.d_b, _ = tr.inverse_z_sampling(self.o, self.d, center, size, Sb, False)
        self.target = torch.rand(rays, 3, generator=gen)

    def step(self):
        """One fwd+bwd pass; returns seconds."""
        import torch
        tr = self.tr
        t0 = time.perf_counter()
        o_ = self.o.clone().requires_grad_(True)
        fg, _ = tr.render_batch_rays(self.table, self.res, self.mlp, o_, self.d, self.z_f, self.d_f, self.min_bbox,
                                     self.size, 10000, False, False)
        bg, _ = tr.render_batch_rays(self.table, self.res, self.mlp, o_, self.d, self.z_b, self.d_b, self.min_bbox,
                                     self.size, 10000, True, True)
        rgb = fg["rgb"] + fg["T_left"][:, None] * bg["rgb"]
        loss = torch.mean((rgb - self.target) ** 2) + 0.01 * (fg["l2_reg_specular"] + bg["l2_reg_specular"])
        loss.backward()
        dt = time.perf_counter() - t0
        self.table.grad = None
        return dt


def run_reference(args, cfg, name):
    """--impl reference: the reference's CUDA extensions have no CPU build, so its CPU arm is the
    restatement under oracle/ (kind "port"), all host threads, a bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # per step: large enough that the threaded C encode and torch's MLP run at their best rate (~1.5 s / step);
    # SNRF_REF_RAYS shrinks it for the contract test of this arm
    rays = int(os.environ.get("SNRF_REF_RAYS", "2048"))
    from oracle import native as on
    on.build()
    port = CpuPort(cfg, rays, cores)
    ts = []
    for i in range(args.warmup + args.steps):
        t = port.step()
        if i >= args.warmup:
            ts.append(t)
    sec = sum(ts) / len(ts)
    v = rays / sec
    print(json.dumps({
        "impl": "reference", "metric": "train rays/s (fwd+bwd)", "value": v, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": name, "sample": f"{rays} rays x {cfg['S']}+{cfg['S_bg']} samples per step, T=2^{cfg['log2T']}"},
        "cpu_baseline": {"value": v, "unit": "rays/s", "cores": cores, "kind": "port",
                         "sample": f"{rays} rays x {cfg['S'] + cfg['S_bg']} samples, fwd+bwd, C hash encode + torch MLP/composite"},
        "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def measured_peak_gbs():
    """(HBM GB/s, source): the driver-written measured copy bandwidth, else the profiling recipe's fallback."""
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        if "hbm_gbs" in peaks:
            return peaks["hbm_gbs"], "measured"
    except Exception:
        pass
    return 6650.0, "fallback"


# ----------------------------------------------------------------------------- render leg
def bench_render(step, cfg, dev, H=1080, W=1920, frames=5, warm=2):
    """BASELINE.json configs[2]: full-frame 1920x1080 inference of the trained-from-random tile through the
    multi-tile render operators (ray/tile intersection -> sample -> fused fp16 encode + tensor-core decoder ->
    accumulate, foreground + background), Mrays/s.  Device-timed, no host synchronisation inside a frame."""
    import torch
    import render_frame as rf
    ts = rf.TileSet.from_hashgrid(step.featureGrid, step.decoder, dev).finalize()
    K = step.poses.ks[0].clone()
    K[0, 0] *= W / cfg["W"]; K[1, 1] *= H / cfg["H"]; K[0, 2] = W / 2.0; K[1, 2] = H / 2.0
    with torch.no_grad():
        c2w = step.poses.c2w()[0].detach()
    for _ in range(warm):
        rf.render_frame(ts, H, W, K, c2w)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(frames):
        out = rf.render_frame(ts, H, W, K, c2w)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / frames
    # roofline of the field evaluation (the encode + decode passes behind pts_inference / bg_pts_inference_v2), timed
    # live on one more frame: algorithmic bytes per sample = 16 levels x 8 corners x 4 B of fp16 table + 28 B of
    # outputs + the sample's inputs (z 4 B; foreground also dist 4 B + slots 8 B)
    import scanerf_b200_capi as capi
    capi.time_calls(("snrf_pts_inference", "snrf_bg_pts_inference_v2"))
    rf.render_frame(ts, H, W, K, c2w)
    k_ms, _ = capi.timed_results()
    capi.time_calls(None)
    S, Sb = 128, 128
    alg = H * W * (S * (512 + 28 + 16) + Sb * (512 + 28 + 4))
    peak, src = measured_peak_gbs()
    achieved = alg / (sum(k_ms) * 1e-3) / 1e9 if k_ms else None
    return {"metric": "render Mrays/s", "value": H * W / ms / 1e3, "unit": "Mrays/s", "ms_per_frame": ms,
            "config": {"workload": "render 1920x1080, 1 tile, 128 + 128 samples per ray, fp16 table 16 x 2^%d x 2" % cfg["log2T"],
                       "frames": frames, "finite": bool(torch.isfinite(out[0]).all())},
            "roofline": {"kernel": "field evaluation (snrf_pts_inference + snrf_bg_pts_inference_v2: level-major fp16 encode pass + tcgen05 decode pass)",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "peak_source": src, "unit": "GB/s",
                         "frac": achieved / peak if achieved else None, "alg_bytes_per_frame": alg, "ms_per_frame": sum(k_ms),
                         "calls_timed": len(k_ms), "share_of_frame": sum(k_ms) / ms if k_ms else None}}



# ----------------------------------------------------------------------------- further legs (outside the headline's timed region)
def _time_steps(step, batches, warm):
    import torch
    for b in batches[:warm]:
        step.step_device(*b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for b in batches[warm:]:
        loss = step.step_device(*b)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (len(batches) - warm), float(loss)


def bench_variants(step, cfg, dev, gen, devb, plain_ms):
    """BASELINE.md section 3: (a) the default.yaml step WITH its multi-view warp loss (config/default.yaml:32-45 has
    WEIGHT_WARP_LOSS 1.0: view selection, projection into 10 neighbour views, colour fetch, masked re-render of the
    neighbour rays), (b) BASELINE.json configs[0] (C1: 2^19 table, 4096 rays x 64 + 64 samples) on the GPU path."""
    import torch
    out = {}
    # (b) first: its tile is small and is freed again
    c1 = WORKLOADS["c1-small"]
    s1, g1 = build_tile(c1, dev, seed=1)
    b1 = [(l.to(dev), t.to(dev)) for l, t in make_batches(c1, 25, g1)]
    ms, _ = _time_steps(s1, b1, 5)
    B1 = b1[0][0].shape[0]
    out["c1"] = {"workload": "c1-small: 16 x 2^19 x 2 table, %d rays x %d samples" % (B1, c1["S"] + c1["S_bg"]),
                 "ms_per_step": ms, "value": B1 / (ms * 1e-3), "unit": "rays/s", "steps": 20}
    del s1, b1
    # (a) the warp loss on the headline tile
    N, H, W = cfg["n_cam"], cfg["H"], cfg["W"]
    images = torch.randint(0, 256, (N, H, W, 3), generator=gen, dtype=torch.uint8)
    occl = torch.ones(N, H, W, 1, dtype=torch.bool)
    step.enable_warp_loss(images, alpha=0.5, gamma=2.0, weight=1.0, occlusions=occl)
    ms, loss = _time_steps(step, devb[:14], 4)
    step.warp = None
    B = devb[0][0].shape[0]
    out["warp_loss"] = {"workload": "default.yaml single tile + warp loss (10 neighbour views per ray re-rendered)",
                        "ms_per_step": ms, "value": B / (ms * 1e-3), "unit": "rays/s", "steps": 10, "loss_finite": loss == loss,
                        "ms_per_step_without": plain_ms,
                        "table_update": "scatter + sparse Adam fused per slice (the neighbour re-render carries no graph: one encode in the backward)"}
    # (c) early ray termination in training (opt-in, TileStep(ert_eps)): the random-initialised field of the headline is
    # nearly transparent, nothing terminates there; an OPAQUE field (density head bias + 5: rays saturate within a few samples,
    # as in a converged tile) shows what the backward kernels skip.  Same tile, same batches, with and without.
    with torch.no_grad():
        step.decoder.sigma_layer.mlp[0].bias += 5.0
    ert = {}
    for eps in (0.0, 1e-4, 0.0, 1e-4):
        step.featureGrid.ert_eps = eps
        ms, loss = _time_steps(step, devb[:14], 4)
        ert.setdefault(eps, []).append(ms)
    step.featureGrid.ert_eps = 0.0
    with torch.no_grad():
        step.decoder.sigma_layer.mlp[0].bias -= 5.0
    m0, m1 = sum(ert[0.0]) / len(ert[0.0]), sum(ert[1e-4]) / len(ert[1e-4])
    out["ert_opaque_field"] = {"workload": "default.yaml single tile, density bias + 5 (opaque field), ert_eps 1e-4 vs 0",
                               "ms_per_step": m1, "ms_per_step_without": m0, "value": B / (m1 * 1e-3), "unit": "rays/s",
                               "steps": 20, "note": "opt-in approximation (the reference back-propagates every sample); off in the headline"}
    return out


def bench_reference_cuda(cfg, dev, steps=10, warm=3):
    """The north star's real denominator: the REFERENCE's own CUDA extensions (unmodified sources rebuilt for sm_100a into
    oracle/_ref by oracle/build_ref.py) in the reference's own op-by-op torch graph with its dense table Adam
    (tools/ref_cuda_step.py), same workload, same box, outside the headline's timed region.  None when oracle/_ref is
    not there."""
    import torch
    import oracle
    if oracle.ref_module("CUDA_EXT") is None or oracle.ref_module("HASHGRID_EMBED") is None:
        return None
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ref_cuda_step
    import scenes
    gen = torch.Generator().manual_seed(0)
    c = [cfg["tile_corner"][i] + cfg["tile_size"][i] * f for i, f in enumerate((0.5, 0.25, 0.5))]
    Ks, c2w = scenes.camera_rig(cfg["n_cam"], cfg["H"], cfg["W"], gen, center=tuple(c),
                                radius=0.3 * min(cfg["tile_size"][0], cfg["tile_size"][2]), fx=cfg["fx"])
    ply = os.path.join(tempfile.mkdtemp(prefix="snrf_ref_"), "mesh.ply")
    scenes.write_proxy_mesh_ply(ply, cfg["tile_corner"], cfg["tile_size"], seed=0)
    torch.manual_seed(0)
    ref = ref_cuda_step.build_reference_step(dev, cfg["tile_corner"], cfg["tile_size"], Ks, c2w, cfg["log2T"], cfg["grid_resolution"],
                                             cfg["sampler_log2dim"], cfg["S"], cfg["S_bg"], ply)
    batches = [(l.to(dev), g.to(dev)) for l, g in make_batches(cfg, warm + steps, gen)]
    ms, loss = _time_steps(ref, batches, warm)
    B = batches[0][0].shape[0]
    return {"what": "reference CUDA extensions (hashgrid_bg_kernel.cu, helper_kernel.cu ... rebuilt unmodified for sm_100a) in the "
                    "reference's torch graph (torch MLP / compositing / pose chain, dense torch Adam over the table), same workload",
            "ms_per_step": ms, "value": B / (ms * 1e-3), "unit": "rays/s", "steps": steps, "warmup": warm, "loss": loss}

def bench_reference_drivers(cfg, steps=12):
    """What a user of the reference gets without touching their code: the reference's UNCHANGED tile.py (TILE.train_one_step,
    tile.py:880-1015, from oracle/_ref/ref_drivers.zip) at the headline's size, once on this repo's drop-in packages and once on
    the reference's own extensions (oracle/_ref/*.so), each in its own process (tests/ref_driver_harness.py).  Its step keeps
    the driver's own torch code -- dense torch.optim.Adam over the whole table (tile.py:301), the torch pose chain and loss --
    so it is slower than TileStep on either arm.  None when oracle/_ref is not there."""
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_drivers.zip")):
        return None
    out = {"what": "reference tile.py unchanged, TILE.train_one_step, 2^%d table, 2^14 rays x %d + %d samples, %d cameras; wall clock "
                   "per step over %d steps after one warm-up step" % (cfg["log2T"], cfg["S"], cfg["S_bg"], cfg["n_cam"], steps - 1)}
    tmp = tempfile.mkdtemp(prefix="snrf_drv_bench_")
    for arm in ("dropin", "reference"):
        res = os.path.join(tmp, arm + ".json")
        cmd = [sys.executable, os.path.join(ROOT, "tests", "ref_driver_harness.py"), "--arm", arm, "--steps", str(steps),
               "--log2T", str(cfg["log2T"]), "--bs-log2", "14", "--samples", str(cfg["S"]), "--cams", str(cfg["n_cam"]), "--out", res]
        try:
            subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=240, check=True)
            r = json.load(open(res))
            out[arm] = {"ms_per_step": r["ms_per_step"], "value": 2 ** 14 / (r["ms_per_step"] * 1e-3), "unit": "rays/s",
                        "last_loss": r["losses"][-1], "hashgrid_module": r["modules"]["hashgrid"].replace(ROOT, ".")}
        except Exception as e:                                  # evidence leg: never takes the headline down with it
            out[arm] = {"error": repr(e)[:200]}
    if "ms_per_step" in out.get("dropin", {}) and "ms_per_step" in out.get("reference", {}):
        out["ratio"] = out["reference"]["ms_per_step"] / out["dropin"]["ms_per_step"]
    return out


def dump_outputs(out_dir, timed_loss, cfg, dev, seed, batch, rows=1 << 20):
    """--dump-outputs: writes <name>.npy (float32; row indices float64) so that two builds can be compared output for output.
      loss.npy       the loss the last timed TileStep.step_device returned: what a caller of the timed path receives.
      seeded_step.*  one more step_device on the last timed batch, by a tile built afresh from the benchmark's seed: its loss,
                     the pose offsets, the decoder and a fixed, seeded sample of `rows` rows of the hash table and its Adam
                     moments (GiBs in full at the headline size).
    The timed tile's own parameters are not written: its backward accumulates with float atomics, whose order varies from run
    to run, and the table's Adam (eps 1e-15) turns near-cancelling sums into updates of +-lr, so its state drifts apart between
    two runs of one build within a few steps (B200, headline size, 2^20 sampled rows: after 1 step the table agrees within
    1e-7, after 2 steps 2427 rows differ by up to 1e-4, after 30 steps most rows and every pose offset differ; the loss after
    30 steps agrees within 1e-5 relative).  A step from the seeded state has the same inputs in every run."""
    import numpy as np
    import torch
    step, _ = build_tile(cfg, dev, seed)
    seeded_loss = step.step_device(*batch)
    table = step.featureGrid.HE.features.detach()
    flat = lambda t: t.reshape(-1, table.shape[-1])
    n = flat(table).shape[0]
    idx = np.sort(np.random.default_rng(0).choice(n, min(rows, n), replace=False))
    idx_dev = torch.from_numpy(idx).to(table.device)
    sel = lambda t: flat(t)[idx_dev]
    arrays = {"loss": timed_loss, "seeded_step.loss": seeded_loss, "seeded_step.table_rows": idx.astype(np.float64),
              "seeded_step.table": sel(table)}
    opt = step.featureGrid_optimizer
    if hasattr(opt, "params"):                                   # vdbAdam: [param, exp_avg, exp_avg_sq] per parameter
        arrays["seeded_step.table_exp_avg"], arrays["seeded_step.table_exp_avg_sq"] = sel(opt.params[0][1]), sel(opt.params[0][2])
    arrays["seeded_step.se3_refine"] = step.poses.se3_refine
    for k, p in step.decoder.named_parameters():
        arrays["seeded_step.decoder." + k] = p
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        if not isinstance(a, np.ndarray):
            a = a.detach().float().cpu().numpy()
        np.save(os.path.join(out_dir, k + ".npy"), a)

# ----------------------------------------------------------------------------- main arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="default.yaml-single-tile", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-render", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the warp-loss / C1 / reference-CUDA legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's loss, and what one step from the seeded tile computes "
                         "on the last timed batch, to DIR/<name>.npy")
    args = ap.parse_args()
    cfg, name = WORKLOADS[args.workload], args.workload
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs: the GPU path only (--impl ours)")
        return run_reference(args, cfg, name)

    import torch
    import torch.distributed as dist
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs: one GPU only (the tiles of a multi-GPU run train in an ADMM consensus)")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pkg = importlib.import_module(PKG)
    pkg.install()
    import scanerf_b200_capi as capi

    K, Wm = args.steps, args.warmup
    if world == 1:
        # BASELINE configs[1]: one tile, no exchange
        step, gen = build_tile(cfg, dev, seed=rank)
        steps, gens, n_cam_global, tiles_total = [step], [gen], cfg["n_cam"], 1
        SYN = 0
    else:
        # BASELINE configs[3] / [4]: a row of tiles with 20 % overlap sharded round-robin over the ranks
        # (admm_trainer.py:74-83), several resident tiles per rank trained in turn (:241-250), only the boundary cameras
        # shared between neighbouring tiles, ADMM pose consensus = one NCCL all-reduce for all resident tiles
        tiles_total = world * cfg.get("tiles_per_rank", 2) if "tiles_total" not in cfg else cfg["tiles_total"]
        mine = list(range(rank, tiles_total, world))
        steps, gens, n_cam_global = build_tile_row(cfg, dev, tiles_total, mine)
        step, gen = steps[0], gens[0]
        # config/default.yaml:5 has SYN_ITERS 100 over 40 000 steps; the driver times 20 steps, so the bench exchanges every
        # 10 (two exchanges inside the timed region) and reports the share of the step time they take
        SYN = cfg.get("syn_iters_bench", 10)
        from admm import PoseConsensus, synchronize_tiles
        exchange = PoseConsensus(n_cam_global, dev)
        synchronize_tiles(exchange, steps)        # first synchronisation before training (admm_trainer.py:218-231)
    counter = {"i": 0}
    sync_events = []

    def maybe_sync():
        if SYN and counter["i"] % SYN == 0:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            synchronize_tiles(exchange, steps)
            e1.record()
            sync_events.append((e0, e1))
        counter["i"] += 1

    last_losses = []

    def run_device(batch):
        maybe_sync()
        last_losses[:] = [st.step_device(*b) for st, b in zip(steps, batch)]

    def run_e2e(batch):
        maybe_sync()
        return [st.step(*b) for st, b in zip(steps, batch)]
    per_tile = [make_batches(cfg, Wm + K, g) for g in gens]
    host = [[(l.pin_memory(), g.pin_memory()) for l, g in pt] for pt in per_tile]
    host = [[h[i] for h in host] for i in range(Wm + K)]                      # [step][tile]
    devb_all = [[(l.to(dev), g.to(dev)) for l, g in batch] for batch in host]
    devb = [batch[0] for batch in devb_all]                                    # the first resident tile's batches
    B = host[0][0][0].shape[0]
    T_res = len(steps)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, batches):
        for b in batches[:Wm]:
            fn(b)
        counter["i"] = 0                  # the timed region starts with a consensus exchange (world > 1)
        sync_events.clear()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for b in batches[Wm:]:
            fn(b)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        sync_ms = sum(a.elapsed_time(b_) for a, b_ in sync_events)
        if world > 1:
            t = torch.tensor([ms, sync_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, sync_ms = float(t[0].item()), float(t[1].item())
        return ms, t0, time.time(), sync_ms, len(sync_events)

    # setup, before any measurement: a few steps on throw-away batches so that CUDA context, kernel attributes and the
    # caching allocator reach steady state
    for st, g in zip(steps, gens):
        for l, t in make_batches(cfg, 6, g):
            st.step_device(l.to(dev), t.to(dev))
    torch.cuda.synchronize()
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.wait_first()
    # (1) device-resident inputs
    capi.launch_count = 0
    ms_dev, t0, t1, sync_ms, n_sync = timed(run_device, devb_all)
    launches = capi.launch_count
    # (2) end to end: pinned host in, loss float out
    ms_e2e, _, t2, _, _ = timed(run_e2e, host)
    clk = clocks.summary(t0, t2) if clocks else None
    # (3) the dominant kernels, timed live on their stream over the same steps: the encode forward through CUDA events
    #     around its C-ABI call; the encode backward -- now a sequence of launches (geometry + ray gradient, then per
    #     L2-resident table slice: scatter, sparse Adam) -- through the library's own per-class event timing
    #     (snrf_field_set_profile: events between the launches on the launching stream, one synchronise at the end).
    import ctypes
    opt = step.featureGrid_optimizer
    fused = bool(getattr(step, "fused_table_update", False)) and hasattr(opt, "begin_fused")
    TIMED = ("snrf_field_encode_fwd", "snrf_field_encode_bwd", "snrf_decoder_fwd", "snrf_decoder_bwd", "snrf_composite_fwd",
             "snrf_composite_bwd", "snrf_field_encode_bwd_adam", "snrf_adam_step", "snrf_sample_grid", "snrf_bg_inverse_z",
             "snrf_compute_ray_fwd", "snrf_compute_ray_bwd", "snrf_pose_fwd", "snrf_pose_bwd")
    capi.time_calls(TIMED)
    prof = []
    if fused:
        capi.lib().snrf_field_set_profile(ctypes.c_int(1))
    for b in devb[Wm:]:
        step.step_device(*b)
        if fused:
            out4 = (ctypes.c_float * 4)()
            capi.lib().snrf_field_last_profile(out4)
            prof.append(tuple(out4))
    if fused:
        capi.lib().snrf_field_set_profile(ctypes.c_int(0))
    torch.cuda.synchronize()
    by_name = capi.timed_by_name()
    capi.time_calls(None)
    N_pts = B * (cfg["S"] + cfg["S_bg"])
    fwd_ms = by_name.get("snrf_field_encode_fwd", [])
    k_ms = by_name.get("snrf_field_encode_bwd", [])
    # mean CUDA-event time of every C-ABI entry point of the step (one call each per step; the fused backward + update is
    # timed with its profiling synchronisation on, so its figure here is an upper bound -- roofline has the exact split)
    kernel_ms = {k: sum(v) / len(v) for k, v in sorted(by_name.items()) if v}
    # touched table floats of one step (what the sparse update moves): entries whose second moment changed
    touched = None
    if hasattr(opt, "params"):
        m_before, v_before = opt.params[0][1].clone(), opt.params[0][2].clone()
        step.step_device(*devb[-1])
        touched = int(((opt.params[0][1] != m_before) | (opt.params[0][2] != v_before)).sum().item())
        del m_before, v_before

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peak_gbs()
    try:
        traffic_file = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        traffic_file = {}

    def roof(kernel, ms_list, alg_bytes, traffic_key, extra=None):
        n = max(len(ms_list), 1)
        avg = sum(ms_list) / n if ms_list else float("nan")
        ach = alg_bytes / (avg * 1e-3) / 1e9 if ms_list else float("nan")
        t = traffic_file.get(traffic_key) if cfg["log2T"] == 24 else None      # the ncu capture is of the 2^24-entry workload
        r = {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
             "frac": ach / peak, "traffic": t.get("bytes") if isinstance(t, dict) else t,
             "traffic_source": (t.get("source") if isinstance(t, dict) else None),
             "avg_launch_ms": avg, "launches_timed": len(ms_list), "alg_bytes_per_launch": alg_bytes,
             "share_of_step": avg / (ms_dev / K / T_res) if ms_list else None}
        if extra:
            r.update(extra)
        return r
    if fused:
        # per kernel class, from the library's own events between the launches on the launching stream.  When classes run
        # concurrently (the sparse coarse levels on the side stream) only geometry [0] and the whole scatter + Adam phase
        # [3] are separable: the per-class split then comes from a few more steps with the side stream off.
        import statistics as st
        mean = lambda xs: sum(xs) / max(len(xs), 1)
        phase_ms = [p[0] + p[3] for p in prof]
        capi.lib().snrf_field_set_coarse_concurrent(ctypes.c_int(0))
        capi.lib().snrf_field_set_profile(ctypes.c_int(1))
        serial = []
        for b_ in devb[Wm:Wm + 8]:
            step.step_device(*b_)
            out4 = (ctypes.c_float * 4)()
            capi.lib().snrf_field_last_profile(out4)
            serial.append(tuple(out4))
        capi.lib().snrf_field_set_profile(ctypes.c_int(0))
        capi.lib().snrf_field_set_coarse_concurrent(ctypes.c_int(1))
        # time the concurrent run saves, attributed to the two classes in proportion to their serial times
        gain = mean(phase_ms) / max(mean([p[0] + p[1] + p[2] for p in serial]), 1e-9)
        bwd_ms = [(p[0] + p[1]) * gain for p in serial]
        adam_ms = [p[2] * gain for p in serial]
        roofline = roof("encode backward = field_geom_raygrad_kernel + field_scatter_slice_kernel x table slices (inside snrf_field_encode_bwd_adam)",
                        bwd_ms, ENC_BWD_BYTES * N_pts, "encode_bwd",
                        {"geom_raygrad_ms": mean([p[0] for p in serial]), "scatter_ms_serial": mean([p[1] for p in serial]),
                         "adam_ms_serial": mean([p[2] for p in serial]), "whole_phase_ms_as_run": mean(phase_ms), "concurrency_gain": gain,
                         "note": "CUDA events between the launches on the launching stream inside the C call (snrf_field_set_profile); "
                                 "per-class times measured with the coarse-level side stream off and scaled by whole_phase_as_run / serial_sum"})
        roofline_update = roof("adam_slice_kernel x table slices (sparse Adam over touched entries, gradient read from the L2-resident scratch)",
                               adam_ms, 28 * (touched or 0), "adam_slices",
                               {"touched_floats_per_step": touched, "alg_bytes_per_touched_float": 28})
        roofline_both = roof("encode backward + table update, the whole snrf_field_encode_bwd_adam sequence as run", phase_ms,
                             ENC_BWD_BYTES * N_pts + 28 * (touched or 0), "encode_bwd_adam")
    else:
        bwd_only = k_ms
        roofline = roof("field_bwd_kernel (snrf_field_encode_bwd: hash-encode backward)", bwd_only, ENC_BWD_BYTES * N_pts, "snrf_field_encode_bwd")
        roofline_update = roofline_both = None
    roofline_fwd = roof("field_fwd_kernel (snrf_field_encode_fwd: position + contraction + 16-level encode + Jacobian store)",
                        fwd_ms, ENC_FWD_BYTES * N_pts, "encode_fwd")
    rays_per_step = world * T_res * B                   # one step = one training step of every resident tile of every rank
    line = {
        "metric": "train rays/s (fwd+bwd)", "value": K * rays_per_step / (ms_dev * 1e-3), "unit": "rays/s", "n_gpus": world,
        "steps": K, "warmup": Wm, "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": name if world == 1 else (("community.yaml-tile-row" if name == "default.yaml-single-tile" else name) + ": row of %d tiles of default.yaml size with 20 %% overlap, %d boundary cameras shared per neighbour pair" % (tiles_total, cfg.get("shared_cams", 16))),
                   "tiles_per_gpu": T_res, "tiles_total": tiles_total, "rays_per_step": rays_per_step, "rays_per_tile_step": B,
                   "samples_per_ray": cfg["S"] + cfg["S_bg"],
                   "hash_table": f"16 x 2^{cfg['log2T']} x 2 f32 per tile", "cameras_per_tile": cfg["n_cam"], "cameras_global": n_cam_global,
                   "pose_refinement": True,
                   "table_update": "scatter + sparse Adam fused per L2-resident slice" if fused else "gradient table + sparse Adam",
                   "parallelism": f"tile-parallel x{world}" + (f", {T_res} resident tiles per rank trained in turn, NCCL pose consensus (one all-reduce of [{n_cam_global}, 8] f32 for all resident tiles) every {SYN} steps" if world > 1 else ""),
                   "l2_policy": "inputs larger than L2 (%.1f GiB table + %.1f GiB Adam moments per tile, random gathers)" % (2.0 ** (cfg["log2T"] - 23), 2.0 ** (cfg["log2T"] - 22))},
        "e2e": {"value": K * rays_per_step / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": T_res * B * 3 * 4 * 2,
                "d2h_bytes_per_step": 4 * T_res},
        "gpu_launches": launches,
        "clocks": clk,
        "roofline": roofline,
        "roofline_fwd": roofline_fwd,
        "kernel_ms": kernel_ms,
    }
    try:
        tf_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained", 1397.7)
    except Exception:
        tf_peak = 1397.7
    if "snrf_decoder_fwd" in kernel_ms and "snrf_decoder_bwd" in kernel_ms:
        dec_ms = kernel_ms["snrf_decoder_fwd"] + kernel_ms["snrf_decoder_bwd"]
        ach = 82368.0 * N_pts / (dec_ms * 1e-3) / 1e12
        line["roofline_decoder"] = {"kernel": "decoder_fwd4_kernel + grad_absmax_kernel + decoder_bwd_kernel (tcgen05 / TMEM)", "bound": "tensor",
                                    "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak,
                                    "useful_flop_per_sample": 82368, "fwd_ms": kernel_ms["snrf_decoder_fwd"], "bwd_ms": kernel_ms["snrf_decoder_bwd"],
                                    "share_of_step": dec_ms / (ms_dev / K / T_res),
                                    "note": "useful fp32-equivalent FLOPs (SURVEY 8d); the kernels issue 3 fp16 MMAs per product (hi/lo split) "
                                            "and the backward recomputes the forward, so the tensor pipe does ~4x this"}
    if roofline_update is not None:
        line["roofline_update"] = roofline_update
        line["roofline_bwd_and_update"] = roofline_both
    if world > 1:
        line["consensus"] = {"exchanges_in_timed_region": n_sync, "ms_total": sync_ms, "consensus_ms_share": sync_ms / ms_dev,
                             "every_steps": SYN, "payload_bytes": n_cam_global * 8 * 4,
                             "share_at_reference_SYN_ITERS_100": (sync_ms / max(n_sync, 1)) / (100 * ms_dev / K),
                             "what": "commit + consensus + synchronize of every resident tile (tile.py:477-508, admm_trainer.py:124-179) "
                                     "as one NCCL all-reduce + the per-tile dual update, CUDA-event timed, max over ranks"}
    if world == 1 and not args.no_render:
        line["render"] = bench_render(step, cfg, dev)
    if world == 1 and not args.no_variants:
        line["variants"] = bench_variants(step, cfg, dev, gen, devb, ms_dev / K)
        ref = bench_reference_cuda(cfg, dev)
        if ref is not None:
            ref["ratio_value"] = line["value"] / ref["value"]
            ref["ratio_e2e"] = line["e2e"]["value"] / ref["value"]
        line["reference_cuda"] = ref
        line["reference_drivers"] = bench_reference_drivers(cfg)
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        from oracle import native as on
        on.build()
        rays, passes = 2048, 8
        port = CpuPort(cfg, rays, cores)
        port.step()                                           # untimed: thread pools, allocator
        sec = sum(port.step() for _ in range(passes)) / passes
        line["cpu_baseline"] = {"value": rays / sec, "unit": "rays/s", "cores": cores, "kind": "port",
                                "sample": f"{rays} rays x {cfg['S'] + cfg['S_bg']} samples of the same workload, fwd+bwd, "
                                          f"mean of {passes} passes ({passes * sec:.1f} s of CPU work)"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_losses[0], cfg, dev, rank, devb[-1])
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
