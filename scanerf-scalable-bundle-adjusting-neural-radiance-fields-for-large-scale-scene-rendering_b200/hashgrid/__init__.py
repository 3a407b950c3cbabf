"""Drop-in for the reference's `hashgrid` package: the per-tile radiance field.

`HashGrid` keeps the reference class's constructor, attributes and method names
(hashgrid/__init__.py:33-596 of the reference) so `tile.py` / `rendering.py` run
unchanged, but the work behind `render_*_rays` goes through the sm_100a kernels of
libscanerf_b200.so: occupancy sampler, hash encode fwd/bwd, fused compositing
(and, when the decoder is the stock ShallowMLP, the fused tensor-core field kernel).
"""
import os

import numpy as np
import torch
import torch.nn as nn

from .PyHashGrid import PyHashGrid
from .PyHashGridBG import PyHashGridBG
from .lib.HASHGRID import *  # noqa: F401,F403  (operator surface, incl. Sampler)
from .lib import HASHGRID as _ops
from . import _decoder, _field, _render

from cuda import bg_inverse_z_sampling, ray_aabb_intersection, sample_points_grid, voxelize_mesh

try:                      # the reference does `from cfg import *` (TRAIN = 0, INFERENCE = 1)
    from cfg import TRAIN, INFERENCE
except Exception:         # cfg.py:1
    TRAIN, INFERENCE = 0, 1

N_LEVELS = 16


def _pow2_shape(log2dim):
    return tuple(int(2 ** int(v)) for v in log2dim)


class HashGrid(nn.Module):
    """One tile's field: a 16-level hash grid over the contracted space of the doubled
    tile box, a boolean occupancy grid over the tile itself and the render helpers."""

    # route ShallowMLP-shaped decoders through the tcgen05 decoder kernels (bf16 operands,
    # f32 accumulation); False keeps the decoder module's own torch forward (fp32)
    fused_decoder = True
    # with fused_decoder: also fuse sample position + contraction + hash encode (csrc/field_encode.cu);
    # False keeps torch contraction + the reference-shaped encode operator
    fused_encode = True
    # early ray termination in TRAINING (opt-in; 0 = off = the reference's semantics: every sample evaluated and
    # back-propagated, hashgrid/__init__.py:512-596).  > 0: samples behind transmittance < ert_eps are composited with weight 0
    # and skipped by the backward of the compositing, the decoder and the encode scatter (fused path only).
    ert_eps = 0.0

    def __init__(self, device, bbox_corner, bbox_size, log2_hashmap_size=24, grid_resolution=[32, 2048],
                 sampler_log2dim=4, init_outside=False, model_path="", near=None, far=None):
        super().__init__()
        self.device = device
        self.bbox_center = bbox_corner + bbox_size / 2.0
        self.bbox_size = bbox_size * 2                      # doubled: the outer half is background
        self.min_bbox = self.bbox_center - self.bbox_size / 2.0
        self.max_bbox = self.bbox_center + self.bbox_size / 2.0
        self.log2_hashmap_size = log2_hashmap_size
        aspect = self.bbox_size / self.bbox_size.min()
        self.finest_resolution = (aspect * grid_resolution[1]).int().cpu()
        self.base_resolution = (aspect * grid_resolution[0]).int().cpu()
        self.HE = PyHashGridBG(self.device, self.min_bbox, self.bbox_size, n_levels=N_LEVELS,
                               n_features_per_level=2, log2_hashmap_size=log2_hashmap_size,
                               base_resolution=self.base_resolution, finest_resolution=self.finest_resolution,
                               init_mode="xavier").to(device)
        self.sampler = _ops.Sampler()
        self.last_sampler_log2dim = sampler_log2dim
        self.sampler_log2dim = sampler_log2dim - torch.log2(self.bbox_size.max() / self.bbox_size).int()
        grid = torch.zeros(_pow2_shape(self.sampler_log2dim), dtype=torch.bool)
        outside = torch.zeros_like(grid)
        # occupancy covers the tile proper = the inner half of the doubled box
        voxelize_mesh(self.sampler_log2dim.cpu(), (self.min_bbox + self.bbox_size / 4.0).cpu(),
                      (self.bbox_size / 2.0).cpu(), model_path, grid, init_outside, outside)
        if near is not None and far is not None:
            grid[:, -int(near / far * grid.shape[1]):, :] = False
        self.occupied_grid = grid.to(self.device)
        self.outside = outside.to(self.device)
        self._refresh_grid_resolution()

    def _refresh_grid_resolution(self):
        self.grid_resolution = torch.tensor(_pow2_shape(self.sampler_log2dim), dtype=torch.int32, device=self.device)

    # ------------------------------------------------------------------ state
    def export_check_point(self):
        return {"occupied_grid": self.occupied_grid.detach().cpu().numpy(),
                "sampler_log2dim": self.sampler_log2dim.detach().cpu().numpy(),
                "grid_resolution": self.grid_resolution.detach().cpu().numpy(),
                "features": self.HE.features.detach().cpu().numpy()}

    def load_check_point(self, ckp):
        up = lambda a: torch.from_numpy(a).to(self.device)
        self.occupied_grid = up(ckp["occupied_grid"])
        self.sampler_log2dim = up(ckp["sampler_log2dim"])
        self.grid_resolution = up(ckp["grid_resolution"])
        self.HE.features = nn.Parameter(up(ckp["features"]))

    def export(self, path):
        """feature.npz for the renderer: fp16 table + occupancy (hashgrid/__init__.py:248-257)."""
        np.savez(os.path.join(path, "feature.npz"),
                 features=self.HE.features.detach().cpu().numpy().astype(np.float16),
                 occupied_grid=self.occupied_grid.detach().cpu(),
                 block_corner=self.min_bbox.cpu().numpy(), block_size=self.bbox_size.cpu().numpy(),
                 grid_log2dim=self.sampler_log2dim.cpu().numpy(), resolution=self.HE.resolution.cpu().numpy())

    def load(self, path):
        f = np.load(os.path.join(path, "feature.npz"))
        up = lambda a: torch.from_numpy(a).to(self.device)
        self.HE.features = nn.Parameter(up(f["features"]).float())
        self.occupied_grid = up(f["occupied_grid"])
        self.block_corner = up(f["block_corner"])
        self.block_size = up(f["block_size"])
        self.sampler_log2dim = up(f["grid_log2dim"])
        self.HE.resolution = up(f["resolution"])

    def toCPU(self):
        self.HE.resolution = self.HE.resolution.cpu()

    def toGPU(self):
        self.HE.resolution = self.HE.resolution.to(self.device)

    def vis_gird(self, path, bg=False):
        """Debug dump of the occupied cells as an OBJ of boxes (reference: tools.draw_AABB);
        written only when the reference's `tools` package is importable."""
        if bg:
            return
        try:
            from tools import tools
        except Exception:
            return
        log2dim = self.sampler_log2dim.cpu()
        cell = (self.bbox_size / 2.0).cpu() / (2 ** log2dim)
        ijk = torch.nonzero(self.occupied_grid.cpu()).float()
        centers = ijk * cell + cell / 2.0 + (self.min_bbox + self.bbox_size / 4.0).cpu()
        v, f = tools.draw_AABB(centers.numpy(), (torch.ones_like(centers) * cell).numpy())
        tools.mesh2obj(os.path.join(path, "grid.obj"), v, f)

    # ------------------------------------------------------------------ pruning
    def generateMeshGrid(self, step, max_res, device="cpu", ox=0, oy=0, oz=0):
        ax = [torch.arange(0, max_res[i], step, device=device) for i in range(3)]
        X, Y, Z = torch.meshgrid(*ax, indexing="ij")
        return torch.stack([X + ox, Y + oy, Z + oz], -1).reshape(-1, 3)

    @torch.no_grad()
    def pruning_tile_grid(self, global_step, decoder, sub_split=False, pruning_th=0.4, batch_size=92 ** 3):
        """Re-evaluate max alpha inside every occupied cell (optionally split 2x) and keep
        cells above `pruning_th` (hashgrid/__init__.py:138-214)."""
        scale = 2 if sub_split else 1
        log2dim = self.sampler_log2dim + (1 if sub_split else 0)
        grid_res = (2 ** log2dim).to(self.device)
        total_res = self.finest_resolution / (4.0 if global_step < 10000 else 2.0)
        per_cell = ((total_res / 2.0).to(self.device) / grid_res).int()
        occ = self.occupied_grid
        for dim in range(3):
            occ = occ.repeat_interleave(scale, dim=dim)
        locs = torch.nonzero(occ).long()
        corner = locs / grid_res
        inner = self.generateMeshGrid(1, per_cell, device=self.device) / (per_cell * grid_res)
        cells_per_batch = max(int(batch_size / torch.prod(per_cell)), 1)
        peak = torch.zeros(locs.shape[0], device=self.device)
        mask32 = self.weight_feature(global_step)[None, :].repeat_interleave(2, dim=-1)
        params = self._fused_ready(decoder)          # stock ShallowMLP: the density head comes from the tensor-core decoder
        unit_d = torch.tensor([[0.0, 0.0, 1.0]], device=self.device)
        for i in range(0, locs.shape[0], cells_per_batch):
            pts = (corner[i:i + cells_per_batch, None, :] + inner[None]) * 2 - 1
            n = pts.shape[0]
            if params is not None:
                feats = self.HE(pts.reshape(-1, 3)).reshape(-1, 32)
                sigma = _field.decoder_forward(feats, mask32[0].contiguous(), unit_d, feats.shape[0], params)[:, :1]
            else:
                sigma = decoder.inference_sigma(self.HE(pts.reshape(-1, 3)) * mask32)
            alpha = 1 - torch.exp(-1.0 * sigma)
            peak[i:i + n] = alpha.reshape(n, -1).max(dim=-1)[0]
        keep = locs[peak > pruning_th]
        new_grid = torch.zeros(_pow2_shape(log2dim), dtype=torch.bool, device=self.device)
        new_grid[keep[:, 0], keep[:, 1], keep[:, 2]] = True
        self.sampler_log2dim = log2dim
        self.occupied_grid = new_grid
        self._refresh_grid_resolution()
        print(f"finished pruning resolution: {grid_res.tolist()} occupied: {int(new_grid.sum())}")

    @torch.no_grad()
    def pruning_grid(self, global_step, decoder, log2dim, pruning_th):
        assert log2dim >= self.last_sampler_log2dim, f"log2dim {log2dim} last_sampler_log2dim {self.last_sampler_log2dim}"
        split = log2dim != self.last_sampler_log2dim
        if split:
            self.last_sampler_log2dim = self.last_sampler_log2dim + 1
        self.pruning_tile_grid(global_step, decoder, sub_split=split, pruning_th=pruning_th)

    # ------------------------------------------------------------------ level masks
    def weight_feature(self, global_step):
        """Coarse-to-fine level weights [16] (hashgrid/__init__.py:228-235)."""
        alpha = max(min(global_step / 10000 * 8 + 8, 16), 0)
        cached = getattr(self, "_level_weights", None)
        if cached is not None and cached[0] == alpha:       # constant once the schedule has saturated: no launches
            return cached[1]
        k = torch.arange(N_LEVELS, dtype=torch.float32, device=self.device)
        w = (1 - torch.cos((alpha - k).clamp(min=0, max=1) * np.pi)) / 2
        self._level_weights = (alpha, w, w.repeat_interleave(2))
        return w

    def level_mask32(self, global_step):
        """weight_feature repeated per feature channel [32] (cached with it)."""
        self.weight_feature(global_step)
        return self._level_weights[2]

    def weight_bg_feature(self, ratio):
        alpha = torch.clamp(ratio * 8 + 8, 0, 16)
        k = torch.arange(N_LEVELS, dtype=torch.float32, device=self.device)
        w = (1 - torch.cos((alpha - k[None]).clamp(min=0, max=1) * np.pi)) / 2
        return w.repeat_interleave(2, dim=-1)

    # ------------------------------------------------------------------ sampling
    def _inner_box(self):
        """(corner, size, centre) of the foreground box = the inner half of the doubled tile box (cached constants)."""
        box = getattr(self, "_inner_box_cache", None)
        if box is None or box[3] is not self.min_bbox or box[4] is not self.bbox_size:
            box = ((self.min_bbox + self.bbox_size / 4.0).contiguous(), (self.bbox_size / 2.0).contiguous(), self.bbox_center.contiguous(),
                   self.min_bbox, self.bbox_size)
            self._inner_box_cache = box
        return box

    def samplePoints(self, rays_o, rays_d, num_sample, out=None):
        """Occupancy-proportional foreground samples; -1 rows = ray sees nothing.  out = (z_vals, dists) buffers to fill."""
        if out is None:
            shape = (rays_o.shape[0], num_sample)
            z_vals = torch.empty(shape, dtype=torch.float32, device=self.device)
            dists = torch.empty(shape, dtype=torch.float32, device=self.device)
        else:
            z_vals, dists = out
        z_vals.fill_(-1.0); dists.fill_(-1.0)
        corner, size, _, _, _ = self._inner_box()
        sample_points_grid(rays_o, rays_d, z_vals, dists, corner, size, self.occupied_grid, self.sampler_log2dim)
        return z_vals, dists

    def invalid_sampling_underground(self, rays_o, rays_d, bound):
        exit_pt = rays_o + bound[:, 1:] * rays_d
        floor = (self.bbox_center - self.bbox_size / 4.0)[1]
        return ~(torch.abs(exit_pt[:, 1] - floor) < 0.0001)

    @torch.no_grad()
    def background_sampling(self, fmesh, rays_o, rays_d, num_samples):
        z_vals, valid = fmesh.background_sampling(rays_o, rays_d, num_samples, float(self.bbox_size.cpu().max()) / 10)
        dists = torch.cat([z_vals[:, 1:] - z_vals[:, :-1], 1e-6 * torch.ones_like(z_vals[:, :1])], -1)
        return z_vals, dists, valid

    @torch.no_grad()
    def inverse_z_sampling(self, rays_o, rays_d, num_sample, invalid_underground=True, perturb=False, out=None):
        """Inverse-depth samples from the tile exit to 1e6 (hashgrid/__init__.py:305-337).  On the device the whole
        expression is one kernel (bit-identical to the torch ops below); out = (z_vals, dists) buffers to fill."""
        if rays_o.is_cuda and self.fused_encode:
            lin = getattr(self, "_linspace", None)
            if lin is None or lin.numel() != num_sample:
                lin = self._linspace = torch.linspace(0.0, 1.0, steps=num_sample, device=self.device)
            R = rays_o.shape[0]
            z_vals, dists = out if out is not None else (torch.empty(R, num_sample, dtype=torch.float32, device=self.device),
                                                         torch.empty(R, num_sample, dtype=torch.float32, device=self.device))
            valid = torch.empty(R, dtype=torch.bool, device=self.device)
            _, size, center, _, _ = self._inner_box()
            bg_inverse_z_sampling(rays_o, rays_d, center, size, lin, z_vals, dists, valid, invalid_underground)
            return z_vals, dists, valid
        bounds = torch.full((rays_o.shape[0], 2), -1, dtype=torch.float32, device=rays_o.device)
        ray_aabb_intersection(rays_o, rays_d, self.bbox_center, self.bbox_size / 2.0, bounds)
        if invalid_underground:
            valid = self.invalid_sampling_underground(rays_o, rays_d, bounds)
        else:
            valid = torch.ones_like(rays_d[..., 0]).bool()
        bounds[torch.any(bounds == -1, dim=-1), 1:] = 0.1
        t = torch.linspace(0.0, 1.0, steps=num_sample, device=self.device)[None, :]
        z_vals = 1.0 / (1.0 / (bounds[:, 1:] + 1e-6) * (1.0 - t) + 1.0 / 1e6 * t)
        z_vals = z_vals.expand([rays_o.shape[0], num_sample])
        dists = torch.cat([z_vals[:, 1:] - z_vals[:, :-1], 1e-6 * torch.ones_like(z_vals[:, :1])], -1)
        return z_vals, dists, valid

    # ------------------------------------------------------------------ rendering
    def cal_integrate_weight(self, sigma, z_vals, dists, rays_d, infinity=True):
        """weights [R,S,1], T_left [R] -- torch form kept for external callers (tile.py:710);
        the render path uses the fused compositing kernel instead."""
        dists = dists * torch.norm(rays_d[..., None, :], dim=-1)
        if infinity:
            dists[:, -1] = 1e10
        if (dists < 0).sum() > 0:
            raise AssertionError("negative sample spacing")
        alpha = 1.0 - torch.exp(-sigma * dists[..., None])
        ones = torch.ones((alpha.shape[0], 1, 1), device=rays_d.device)
        T = torch.cumprod(torch.cat([ones, 1.0 - alpha + 1e-6], 1), 1)[:, :-1]
        return alpha * T, T[:, -1, 0]

    def accumulate(self, weights, attr):
        return torch.sum(weights * attr, 1)

    def inference_sigma(self, samples, decoder):
        shape = samples.shape
        feats = self.HE(samples.reshape(-1, 3))
        return decoder.inference_sigma(feats.reshape(*shape[:-1], 32))

    def compute_normal(self, samples, decoder):
        samples = samples.requires_grad_(True)
        sigma = self.inference_sigma(samples, decoder)
        normal = torch.autograd.grad(outputs=sigma, inputs=samples, grad_outputs=torch.ones_like(sigma),
                                     create_graph=True, retain_graph=True, only_inputs=True)[0]
        return -1.0 * normal / (normal.norm(2, dim=-1, keepdim=True) + 1e-8), sigma

    def contract_fore(self, x):
        return (x - self.min_bbox) / self.bbox_size * 4.0 - 2.0, None

    def contract_bg(self, x):
        x = (x - self.min_bbox) / self.bbox_size * 4.0 - 2.0
        n, _ = torch.max(torch.abs(x), dim=-1, keepdim=True)
        return x * ((2 - 1.0 / n) / n), None

    def _scatter_back(self, valid, out, rays_o, rays_d, names):
        full = {"rgb": torch.zeros_like(rays_o), "depth": torch.zeros_like(rays_d[..., :1]),
                "T_left": torch.ones_like(rays_d[..., :1]), "specular": torch.zeros_like(rays_o),
                "diffuse": torch.zeros_like(rays_o)}
        full["rgb"][valid] = out["rgb"]
        full["depth"][valid] = out["depth"]
        full["T_left"][valid, 0] = out["T_left"]
        full["specular"][valid] = out["specular"]
        full["diffuse"][valid] = out["diffuse"]
        return {names[k]: v for k, v in full.items()}

    def _fused_ready(self, decoder, out_normal=False):
        """(decoder parameters | None): the sync-free fused path needs the stock ShallowMLP and a CUDA table."""
        if not (self.fused_decoder and self.fused_encode) or out_normal or not self.HE.features.is_cuda:
            return None
        return _decoder.decoder_params(decoder)

    def render_rays_masked(self, rays_o, rays_d, z_vals, dists, valid, params, mode, contract_mode, infinity, global_step):
        """The fused render chain over ALL rays with a validity mask instead of the reference's boolean
        compaction (hashgrid/__init__.py:419-451): masked-out rays are skipped inside every kernel and come
        back with the values the reference scatters for them (colour 0, depth 0, T_left 1).  Static shapes,
        no device->host synchronisation anywhere."""
        R, S = z_vals.shape
        mask32 = self.level_mask32(global_step)
        ert = _render.ErtState(self.ert_eps) if (self.ert_eps > 0 and mode is TRAIN) else None
        feats = _field.field_encode(rays_o, rays_d, z_vals, self.HE.features, self.HE.resolution, self.min_bbox,
                                    self.bbox_size, contract_mode, valid, 0, ert)
        heads = _field.decoder_apply(feats, rays_d, mask32, S, params, valid, ert)
        return _render.composite_packed(heads, z_vals, dists, rays_d, infinity, train=(mode is TRAIN), valid=valid, ert=ert)

    def _fore_bg_rows(self, rays_o, rays_d, num_sample, decoder, mode, occlusion_mask=None, global_step=0,
                      invalid_underground=True):
        """The joint 2R-ray batch up to the compositing rows: (row [2R,16], weights [2R,S], v_f, v_b) or None when the
        fused path is not available (non-stock decoder)."""
        params = self._fused_ready(decoder)
        if params is None:
            return None
        R = rays_o.shape[0]
        # both samplers write straight into the halves of the joint [2R, S] buffers
        z2 = torch.empty(2 * R, num_sample, dtype=torch.float32, device=self.device)
        dist2 = torch.empty(2 * R, num_sample, dtype=torch.float32, device=self.device)
        z_f, d_f = self.samplePoints(rays_o, rays_d, num_sample, out=(z2[:R], dist2[:R]))
        v_f = torch.all(z_f != -1, dim=-1)
        z_b, d_b, v_b = self.inverse_z_sampling(rays_o, rays_d, num_sample, invalid_underground, out=(z2[R:], dist2[R:]))
        if occlusion_mask is not None:
            v_f, v_b = v_f & occlusion_mask[..., 0], v_b & occlusion_mask[..., 0]
        o2, d2 = torch.cat([rays_o, rays_o], 0), torch.cat([rays_d, rays_d], 0)
        valid2 = torch.cat([v_f, v_b], 0)
        mask32 = self.level_mask32(global_step)
        ert = _render.ErtState(self.ert_eps) if (self.ert_eps > 0 and mode is TRAIN) else None
        feats = _field.field_encode(o2, d2, z2, self.HE.features, self.HE.resolution, self.min_bbox, self.bbox_size, 3, valid2, R, ert)
        heads = _field.decoder_apply(feats, d2, mask32, num_sample, params, valid2, ert)
        row, weights = _render.CompositePackedFn.apply(heads, z2, dist2, d2, R, valid2, ert)      # rays >= R end at infinity
        return row, weights, v_f, v_b

    def render_fore_bg_rays(self, rays_o, rays_d, num_sample, decoder, mode, occlusion_mask=None, global_step=0,
                            invalid_underground=True):
        """render_fore_rays + render_bg_rays ("IZ" background, same sample count) as ONE batch of 2R rays through
        every kernel: rays [0, R) are the foreground chain, rays [R, 2R) the background chain (the encode kernel
        switches the contraction, the compositing kernel the infinite last step, at ray R).  Halves the launches
        and -- the point -- streams the hash table through L2 once per step instead of once per chain.
        Returns (fore dict, background dict) with the keys of the two separate calls, or None when the fused path
        is not available (non-stock decoder)."""
        rows = self._fore_bg_rows(rays_o, rays_d, num_sample, decoder, mode, occlusion_mask, global_step, invalid_underground)
        if rows is None:
            return None
        row, weights, v_f, v_b = rows
        R = rays_o.shape[0]
        train = mode is TRAIN
        fg = _render._finish(row[:R], weights[:R], train, v_f)
        bg = _render._finish(row[R:], weights[R:], train, v_b)
        fg.update({"pred_color": fg["rgb"], "pred_depth": fg["depth"], "T_left": fg["T_left"][:, None], "fore_valid": v_f})
        bg.update({"T_left": bg["T_left"][:, None], "valid": v_b})
        return fg, bg

    def fore_bg_colour_loss(self, rays_o, rays_d, num_sample, decoder, gt_color, l2_weight=0.01, global_step=0,
                            invalid_underground=True):
        """The training step's colour loss straight from the joint batch's compositing rows: the merge of the two chains
        (tile.py:661-681), the clamp, the masked MSE (criterions.py:126-147) and `l2_weight` x the specular L2 regulariser
        (tile.py:999) with their gradient as ONE kernel (_render.JointLossFn) instead of ~60 small torch launches.  Same value and
        gradients as TileStep.loss computes from render_fore_bg_rays.  None when the fused path is not available."""
        rows = self._fore_bg_rows(rays_o, rays_d, num_sample, decoder, TRAIN, None, global_step, invalid_underground)
        if rows is None:
            return None
        row, _, v_f, v_b = rows
        return _render.JointLossFn.apply(row, v_f, v_b, gt_color, l2_weight)

    def render_fore_rays(self, rays_o, rays_d, num_sample, decoder, mode, occlusion_mask=None, infinity=False, **kwargs):
        z_vals, dists = self.samplePoints(rays_o, rays_d, num_sample)
        valid = torch.all(z_vals != -1, dim=-1)
        if occlusion_mask is not None:
            valid = valid & occlusion_mask[..., 0]
        params = self._fused_ready(decoder)
        if params is not None:
            # deviation from the reference: a batch without any valid ray still returns (dict, True) -- all
            # zeros / T_left = 1 -- instead of (None, False); deciding that on the host would cost a sync
            out = self.render_rays_masked(rays_o, rays_d, z_vals, dists, valid, params, mode, 1, infinity, kwargs["global_step"])
            res = dict(out)
            # pred_depth is its own tensor (not a view of the packed output row): TILE.render_rays accumulates the background
            # into it IN PLACE (tile.py:673), and a view would invalidate the row's other columns for autograd
            res.update({"pred_color": out["rgb"], "pred_depth": out["depth"].clone(), "T_left": out["T_left"][:, None],
                        "specular": out["specular"], "diffuse": out["diffuse"], "fore_valid": valid})
            return res, True
        out, ok = self.render_batch_rays(rays_o[valid], rays_d[valid], z_vals[valid], dists[valid], decoder, mode,
                                         self.contract_fore, out_normal=False, infinity=infinity,
                                         global_step=kwargs["global_step"])
        if ok is False:
            return None, False
        res = dict(out)
        res.update(self._scatter_back(valid, out, rays_o, rays_d,
                                      {"rgb": "pred_color", "depth": "pred_depth", "T_left": "T_left",
                                       "specular": "specular", "diffuse": "diffuse"}))
        res["fore_valid"] = valid
        return res, True

    def render_bg_rays(self, rays_o, rays_d, num_sample, decoder, mode, occlusion_mask=None, infinity=True, **kwargs):
        if kwargs["bg_mode"] == "IZ":
            z_vals, dists, valid = self.inverse_z_sampling(rays_o, rays_d, num_sample, kwargs["invalid_underground"])
        elif kwargs["bg_mode"] == "BS":
            z_vals, dists, valid = self.background_sampling(kwargs["fmesh"], rays_o, rays_d, num_sample)
        else:
            return None, False
        if occlusion_mask is not None:
            valid = valid & occlusion_mask[..., 0]
        params = self._fused_ready(decoder)
        if params is not None:
            out = self.render_rays_masked(rays_o, rays_d, z_vals, dists, valid, params, mode, 2, infinity, kwargs["global_step"])
            res = dict(out)
            res.update({"T_left": out["T_left"][:, None], "valid": valid})
            return res, True
        out, ok = self.render_batch_rays(rays_o[valid], rays_d[valid], z_vals[valid], dists[valid], decoder, mode,
                                         self.contract_bg, out_normal=False, infinity=infinity,
                                         global_step=kwargs["global_step"])
        if ok is False:
            return None, ok
        res = dict(out)
        res.update(self._scatter_back(valid, out, rays_o, rays_d,
                                      {"rgb": "rgb", "depth": "depth", "T_left": "T_left",
                                       "specular": "specular", "diffuse": "diffuse"}))
        res["valid"] = valid
        return res, ok

    def render_batch_rays(self, rays_o, rays_d, z_vals, dists, decoder, mode, contract_func, out_normal=False,
                          infinity=False, **kwargs):
        """samples -> contraction -> hash encode -> level mask -> decoder -> compositing
        (hashgrid/__init__.py:512-596).  Returns (dict, True) or (None, False) for an empty batch."""
        if z_vals.shape[0] == 0:
            return None, False
        R, S = z_vals.shape
        render_mode = mode
        mask16 = self.weight_feature(kwargs["global_step"])
        params = _decoder.decoder_params(decoder) if self.fused_decoder else None
        mode = 1 if contract_func == self.contract_fore else (2 if contract_func == self.contract_bg else 0)
        if params is not None and mode != 0 and self.fused_encode and self.HE.features.is_cuda:
            # fully fused path: sample position + contraction + hash encode in one kernel (level-major
            # features), the stock ShallowMLP on the tensor cores, packed head rows straight into compositing
            jac = [] if out_normal else None
            feats = _field.field_encode(rays_o, rays_d, z_vals, self.HE.features, self.HE.resolution, self.min_bbox,
                                        self.bbox_size, mode, jac_out=jac)
            mask32 = mask16.repeat_interleave(2)
            if out_normal:
                # the reference differentiates sigma w.r.t. the samples with torch.autograd.grad (hashgrid/__init__.py:547-556)
                # and accumulates the normal detached: one forward kernel on the encode's features and Jacobians gives the
                # same normal, and the Jacobians are released here unless the encode kept them for the ray gradient
                n = _field.field_normal(feats, jac.pop(), mask32, params, rays_o.contiguous(), rays_d.contiguous(),
                                        z_vals.contiguous(), self.min_bbox, self.bbox_size, mode)
            heads = _field.decoder_apply(feats, rays_d, mask32, S, params)
            out = _render.composite_packed(heads, z_vals, dists, rays_d, infinity, train=(render_mode is TRAIN))
            if out_normal:
                out["normal"] = self.accumulate(out["weights"], n.view(R, S, 3))
            return out, True
        samples = rays_o[:, None, :] + z_vals[..., None] * rays_d[:, None, :]
        if contract_func is not None:
            cx, extra_w = contract_func(samples.reshape(-1, 3))
        else:
            cx, extra_w = samples.reshape(-1, 3), None
        feats = self.HE(cx)
        if params is not None and extra_w is None and not out_normal:
            # stock ShallowMLP: the whole decoder runs on the tensor cores (csrc/decoder.cu) and
            # hands packed head rows straight to the compositing kernel; out_normal differentiates the torch decoder below
            heads = _field.decoder_apply(feats, rays_d, mask16.repeat_interleave(2), S, params)
            return _render.composite_packed(heads, z_vals, dists, rays_d, infinity, train=(render_mode is TRAIN)), True
        mask32 = mask16[None, None, :].repeat_interleave(2, dim=-1)
        if extra_w is not None:
            mask32 = mask32 * extra_w.reshape(R, S, 32)
        heads = decoder(torch.cat([feats.reshape(R, S, 32), rays_d[:, None, :].repeat(1, S, 1)], -1), weight_feature=mask32)
        out = _render.composite(heads, z_vals, dists, rays_d, infinity, train=(render_mode is TRAIN))
        if out_normal:
            ones = torch.ones_like(heads["sigma"], requires_grad=False)
            n = torch.autograd.grad(outputs=heads["sigma"], inputs=samples, grad_outputs=ones, create_graph=True,
                                    retain_graph=True, only_inputs=True)[0]
            n = -1.0 * n / (n.norm(2, dim=-1, keepdim=True) + 1e-8)
            out["normal"] = self.accumulate(out["weights"], n.detach())
        return out, True
