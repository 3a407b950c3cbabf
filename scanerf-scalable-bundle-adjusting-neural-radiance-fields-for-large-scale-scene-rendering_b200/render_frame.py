"""Host-side mirror of the reference's multi-tile inference driver, reduced to the hot path:
RenderingHashGrid.parse_blocks (rendering.py:93-174) and render_rays_base (rendering.py:286-544).

Everything numeric runs in the sm_100a render kernels behind the reference's HASHGRID operator
names (csrc/render.cu, csrc/infer.cu); this class only sequences them the way the reference does:
  ray/tile intersections -> near-to-far tile order -> [sample -> assign tiles -> fused encode + decoder
  -> accumulate] per traced tile -> exit tiles -> inverse-z background samples -> fused evaluation ->
  accumulate -> blend.
The reference synchronises with the host three times per frame (rendering.py:313, 346, 451) to size
its loops; here the loop bounds come from the tile count (a ray crosses at most `num_tiles` tiles, at
most 4 exit tiles), so a frame is issued without any device->host synchronisation.
`rendering.py` itself drives the same operators unchanged through `import hashgrid`.
"""
import numpy as np
import torch

from hashgrid.lib import HASHGRID as ops

MISS = 1e7


class TileSet:
    """The renderer's scene: per-tile fp16 tables, flat decoder parameters, occupancy grids (rendering.py:93-174)."""

    def __init__(self, device):
        self.device = device
        self.tables, self.params, self.res, self.occ, self.corner, self.size, self.log2dim = [], [], [], [], [], [], []

    def add_tile(self, features_f16, flat_params, resolution, occupied_grid, block_corner, block_size, grid_log2dim):
        """One exported tile: feature.npz contents (hashgrid/__init__.py:248-257) + the flat decoder vector
        (rendering.py:101-113).  block_corner / block_size are those of the DOUBLED tile box, as exported."""
        self.tables.append(torch.as_tensor(features_f16).to(torch.float16))
        self.params.append(torch.as_tensor(flat_params, dtype=torch.float32))
        self.res.append(torch.as_tensor(resolution, dtype=torch.int32))
        self.occ.append(torch.as_tensor(occupied_grid).reshape(-1).bool())
        self.corner.append(torch.as_tensor(block_corner, dtype=torch.float32))
        self.size.append(torch.as_tensor(block_size, dtype=torch.float32))
        self.log2dim.append(torch.as_tensor(grid_log2dim, dtype=torch.int32))

    @classmethod
    def from_hashgrid(cls, hashgrid, decoder, device):
        """A one-tile scene straight from a training-side HashGrid + decoder (what export_tile writes)."""
        from hashgrid._decoder import flatten_for_inference
        ts = cls(device)
        ts.add_tile(hashgrid.HE.features.detach().half(), flatten_for_inference(decoder), hashgrid.HE.resolution,
                    hashgrid.occupied_grid, hashgrid.min_bbox, hashgrid.bbox_size, hashgrid.sampler_log2dim)
        return ts

    @classmethod
    def from_exported(cls, tile_dirs, device):
        """Trained tiles as TILE.export_tile wrote them (tile.py:509-532), read the way the reference's renderer does
        (rendering.py:86-174): <dir>/feature.npz + <dir>/decoder.pth, whose Linear weights / biases are taken in
        state_dict key order (tools/utils.py:399-410) and flattened per layer as bias then W^T."""
        import os
        ts = cls(device)
        for d in tile_dirs:
            f = np.load(os.path.join(d, "feature.npz"))
            sd = torch.load(os.path.join(d, "decoder.pth"), map_location="cpu", weights_only=True)
            weights = [v for k, v in sd.items() if "weight" in k]
            bias = [v for k, v in sd.items() if "weight" not in k and "bias" in k]
            flat = torch.cat([t for w, b in zip(weights, bias) for t in (b.flatten(), w.t().contiguous().flatten())]).float()
            ts.add_tile(f["features"], flat, f["resolution"], f["occupied_grid"], f["block_corner"], f["block_size"], f["grid_log2dim"])
        return ts.finalize()

    def finalize(self):
        dev = self.device
        self.feature_tables = torch.stack(self.tables).to(dev).contiguous()
        self.flat_params = torch.stack(self.params).to(dev).contiguous()
        self.resolution = torch.stack(self.res).to(dev).contiguous()
        sizes = [int(o.numel()) for o in self.occ]
        self.grid_starts = torch.tensor(np.cumsum([0] + sizes)[:-1], dtype=torch.int64, device=dev)
        self.occupied_grid = torch.cat(self.occ).to(dev).contiguous()
        self.grid_log2dim = torch.stack(self.log2dim).to(dev).contiguous()
        corner, size = torch.stack(self.corner).to(dev), torch.stack(self.size).to(dev)
        # the foreground box is the inner half of the exported (doubled) box: rendering.py:164-165
        self.block_corner = (corner + size / 4.0).contiguous()
        self.block_size = (size / 2.0).contiguous()
        self.num_tiles = len(sizes)
        # occupancy dilated across tile overlaps, used for sample placement only (rendering.py:168-173)
        self.fake_occupied_grid = self.occupied_grid.clone()
        for i in range(self.num_tiles):
            ops.process_occupied_grid(i, sizes[i], self.block_corner, self.block_size, self.occupied_grid, self.grid_starts,
                                      self.grid_log2dim, self.fake_occupied_grid)
        return self


def pinhole_rays(H, W, K, c2w, device):
    """rendering.compute_rays (rendering.py:272-284): pixel centres (+0.5), camera-to-world rotation."""
    j, i = torch.meshgrid(torch.arange(H, dtype=torch.float32, device=device), torch.arange(W, dtype=torch.float32, device=device),
                          indexing="ij")
    dirs = torch.stack([(i + 0.5 - K[0, 2]) / K[0, 0], (j + 0.5 - K[1, 2]) / K[1, 1], torch.ones_like(i)], -1)
    rays_d = (dirs[..., None, :] * c2w[:3, :3]).sum(-1)
    rays_o = c2w[:3, 3].expand(rays_d.shape)
    return rays_o.reshape(-1, 3).contiguous(), rays_d.reshape(-1, 3).contiguous()


@torch.no_grad()
def render_rays(ts, rays_o, rays_d, num_sample=128, num_bg_sample=128, sample_range=1e6, max_tracing=None, adaptive=True):
    """render_rays_base (rendering.py:286-544) for a flat batch of rays.  Returns per-ray
    (diffuse [B,3], specular [B,3], depth [B,1], transparency [B,1]).
    adaptive (scenes of several tiles): read the number of tracing rounds (the most tiles any ray crosses) and of
    background slots in use back from the device, as the reference does (rendering.py:318-320, 470) -- two host
    synchronisations per call that save the empty rounds.  adaptive=False runs the worst-case counts and never
    synchronises (for callers that pipeline frames or capture the call in a CUDA graph); both give the same image.
    The slots in use are counted by tile id, not by positive weight as at rendering.py:470: an exit tile whose exit
    point lies on one of its x-z edges has weight 0 and can precede a weighted slot, which that count would drop."""
    dev, B, nb = rays_o.device, rays_o.shape[0], ts.num_tiles
    f32 = torch.float32
    intersections = torch.full((B, nb, 2), MISS, dtype=f32, device=dev)
    ops.ray_block_intersection(rays_o, rays_d, ts.block_corner, ts.block_size, intersections)
    tracing_blocks = torch.argsort(intersections[..., 0], dim=-1).int().contiguous()
    transparency = torch.ones(B, 1, dtype=f32, device=dev)
    diffuse, specular = torch.zeros(B, 3, dtype=f32, device=dev), torch.zeros(B, 3, dtype=f32, device=dev)
    depth = torch.zeros(B, 1, dtype=f32, device=dev)
    tracing_idx = torch.zeros(B, 1, dtype=torch.int32, device=dev)
    z_start = torch.zeros(B, 1, dtype=f32, device=dev)
    z_vals, dists = torch.empty(B, num_sample, dtype=f32, device=dev), torch.empty(B, num_sample, dtype=f32, device=dev)
    block_idxs = torch.empty(B, num_sample, 4, dtype=torch.int16, device=dev)
    pts_d, pts_s = torch.empty(B, num_sample, 3, dtype=f32, device=dev), torch.empty(B, num_sample, 3, dtype=f32, device=dev)
    pts_a = torch.empty(B, num_sample, 1, dtype=f32, device=dev)
    if max_tracing is None:
        # a ray meets each tile at most once: nb rounds always suffice
        max_tracing = int((intersections[..., 0] != MISS).sum(-1).max()) if (adaptive and nb > 1) else nb
    for _ in range(max_tracing):
        running = (tracing_idx < nb) & (transparency > 1e-5)
        z_vals.fill_(-1.0); dists.fill_(-1.0); block_idxs.fill_(-1)
        ops.sample_points(rays_o, rays_d, ts.block_corner, ts.block_size, ts.fake_occupied_grid, ts.grid_starts, ts.grid_log2dim,
                          tracing_blocks, intersections, tracing_idx, z_start, z_vals, dists)
        ops.prepare_points(z_vals, running, intersections, block_idxs)
        ops.pts_inference(rays_o, rays_d, z_vals, dists, block_idxs, ts.feature_tables, ts.flat_params, ts.resolution, ts.occupied_grid,
                          ts.grid_starts, ts.grid_log2dim, ts.block_corner, ts.block_size, pts_d, pts_s, pts_a)
        ops.accumulate_color(pts_d, pts_s, pts_a, transparency, z_vals, diffuse, specular, depth)
    # ---- background through the exit tile(s)
    bg_bidxs = torch.full((B, 4), -1, dtype=torch.int16, device=dev)
    bg_w = torch.zeros(B, 4, dtype=f32, device=dev)
    ops.update_outgoing_bidx(rays_o, rays_d, ts.block_corner, ts.block_size, tracing_blocks, intersections, bg_bidxs, bg_w, 0.12, False)
    bg_w = bg_w / torch.sum(bg_w, dim=-1, keepdim=True)
    bg_d, bg_s, bg_z = torch.zeros(B, 3, dtype=f32, device=dev), torch.zeros(B, 3, dtype=f32, device=dev), torch.zeros(B, 1, dtype=f32, device=dev)
    if num_bg_sample != num_sample:
        pts_d, pts_s = torch.empty(B, num_bg_sample, 3, dtype=f32, device=dev), torch.empty(B, num_bg_sample, 3, dtype=f32, device=dev)
        pts_a = torch.empty(B, num_bg_sample, 1, dtype=f32, device=dev)
    bg_zv = torch.empty(B, num_bg_sample, dtype=f32, device=dev)
    n_bg = min(4, nb)                     # at most min(4, tiles) exit tiles share the farthest face
    if adaptive and nb > 1:
        n_bg = int((bg_bidxs >= 0).sum(-1).max())      # the exit tiles fill the slots from 0
    for i in range(n_bg):
        bg_zv.fill_(-1.0); pts_d.zero_(); pts_s.zero_(); pts_a.zero_()
        ops.inverse_z_sampling(intersections, bg_bidxs[..., i].contiguous(), bg_zv, sample_range)
        ops.bg_pts_inference_v2(rays_o, rays_d, bg_zv, bg_bidxs, i, ts.block_corner, ts.block_size, ts.resolution, ts.feature_tables,
                                ts.flat_params, pts_d, pts_s, pts_a)
        t, td, tsp, tz = torch.ones(B, 1, dtype=f32, device=dev), torch.zeros(B, 3, dtype=f32, device=dev), \
            torch.zeros(B, 3, dtype=f32, device=dev), torch.zeros(B, 1, dtype=f32, device=dev)
        ops.accumulate_color(pts_d, pts_s, pts_a, t, bg_zv, td, tsp, tz)
        w = torch.nan_to_num(bg_w[:, i:i + 1], nan=0.0)       # rays that hit nothing have 0/0 weights (NaN in the reference)
        bg_d += td * w; bg_s += tsp * w; bg_z += tz * w
    diffuse = diffuse + transparency * bg_d
    specular = specular + transparency * bg_s
    depth = depth + transparency * bg_z
    return diffuse, specular, depth, transparency


@torch.no_grad()
def render_frame(ts, H, W, K, c2w, **kw):
    rays_o, rays_d = pinhole_rays(H, W, K, c2w, ts.device)
    d, s, z, t = render_rays(ts, rays_o, rays_d, **kw)
    return d.reshape(H, W, 3), s.reshape(H, W, 3), z.reshape(H, W, 1), t.reshape(H, W, 1)


@torch.no_grad()
def evaluate_frames(ts, Ks, c2ws, images, H, W, masks=None, **render_kw):
    """rendering.py's `val` mode over a TileSet: each camera (Ks [V,3,3], c2ws [V,3,4] on the device) rendered with
    render_frame(**render_kw), rgb = clamp(diffuse + specular, 0, 1) as the training path composes it, and scored against
    `images` [V,H,W,3] (uint8 or float32 in [0, 1]) within `masks` [V,H,W(,1)] bool or None.
    -> metrics.image_metrics' per-view {"mse", "psnr", "ssim", "count"} [V] plus "mean_mse", "mean_psnr", "mean_ssim", all
    device tensors.  With adaptive=False nothing synchronises with the host."""
    from metrics import image_metrics, with_means
    pred = torch.empty(len(c2ws), H, W, 3, dtype=torch.float32, device=ts.device)
    for k in range(len(c2ws)):
        d, s, _, _ = render_frame(ts, H, W, Ks[k], c2ws[k], **render_kw)
        torch.clamp(d + s, 0, 1, out=pred[k])
    return with_means(image_metrics(pred, images, masks))
