"""Host-side mirror of the reference's per-tile training step, reduced to the hot path:
TILE.render_rays (tile.py:639-692) and the RGB-loss part of TILE.train_one_step
(tile.py:880-1015), with the reference's optimiser settings (tile.py:299-343).

Everything numeric runs in the sm_100a kernels of libscanerf_b200.so:
  ray generation + analytic pose gradient   csrc/rays.cu       (compute_ray_forward/backward)
  occupancy-bounded sample placement        csrc/rays.cu       (sample_points_grid, ray_aabb)
  hash encode fwd/bwd, decoder, compositing HashGrid.render_*_rays (csrc/hash_encode.cu, field, composite)
  sparse Adam over touched table entries    csrc/adam.cu       (vdbAdam)
The se(3) chain on the [N_cam, 6] pose parameters stays in torch (a few hundred floats).
This class is what bench.py and smoke() drive; `tile.py` itself drives the same HashGrid
methods unchanged.
"""
import torch
import torch.nn as nn

import scanerf_b200_capi as capi  # noqa: F401  (fails loudly when the native library is missing)
from cuda import compute_ray_backward, compute_ray_forward
from hashgrid import HashGrid, TRAIN, INFERENCE
from hashgrid._decoder import ShallowMLP
from vdbAdam import vdbAdam


# ----------------------------------------------------------------------------- se(3)
def _taylor(x, kind, nth=10):
    """camera.py:118-141: Taylor series of sin(x)/x, (1-cos x)/x^2, (x-sin x)/x^3."""
    ans = torch.zeros_like(x)
    denom = 1.0
    for i in range(nth + 1):
        if kind == "A":
            if i > 0:
                denom *= (2 * i) * (2 * i + 1)
        elif kind == "B":
            denom *= (2 * i + 1) * (2 * i + 2)
        else:
            denom *= (2 * i + 2) * (2 * i + 3)
        ans = ans + (-1) ** i * x ** (2 * i) / denom
    return ans


def se3_to_SE3(wu):
    """camera.py:84-95: [N,6] (rotation, translation generators) -> [N,3,4]."""
    w, u = wu.split([3, 3], dim=-1)
    w0, w1, w2 = w.unbind(-1)
    O = torch.zeros_like(w0)
    wx = torch.stack([torch.stack([O, -w2, w1], -1), torch.stack([w2, O, -w0], -1), torch.stack([-w1, w0, O], -1)], -2)
    theta = w.norm(dim=-1)[..., None, None]
    eye = torch.eye(3, device=wu.device)
    A, B, C = _taylor(theta, "A"), _taylor(theta, "B"), _taylor(theta, "C")
    R = eye + A * wx + B * wx @ wx
    V = eye + B * wx + C * wx @ wx
    return torch.cat([R, V @ u[..., None]], -1)


def pose_invert(p):
    """camera.py:37-43"""
    R, t = p[..., :3], p[..., 3:]
    Ri = R.transpose(-1, -2)
    return torch.cat([Ri, -Ri @ t], -1)


def pose_compose(a, b):
    """camera.py:45-60 for two poses: x -> b(a(x))."""
    Ra, ta, Rb, tb = a[..., :3], a[..., 3:], b[..., :3], b[..., 3:]
    return torch.cat([Rb @ Ra, Rb @ ta + tb], -1)


class RayGenFn(torch.autograd.Function):
    """(c2w [N,3,4], Ks [N,3,3], locs [B,3] i32 = (view, px, py)) -> rays_o, rays_d [B,3];
    backward = the analytic bundle-adjustment gradient dL/dc2w (cuda/compute_ray_kernel.cu:45-92
    semantics with the ray-indexed gradients)."""

    @staticmethod
    def forward(ctx, c2w, Ks, locs):
        B = locs.shape[0]
        rays_o = torch.empty(B, 3, dtype=torch.float32, device=c2w.device)
        rays_d = torch.empty(B, 3, dtype=torch.float32, device=c2w.device)
        compute_ray_forward(rays_o, rays_d, Ks.reshape(-1, 9), c2w.reshape(-1, 12), locs)
        ctx.save_for_backward(Ks, locs)
        ctx.n = c2w.shape[0]
        return rays_o, rays_d

    @staticmethod
    def backward(ctx, g_o, g_d):
        Ks, locs = ctx.saved_tensors
        g = torch.zeros(ctx.n, 12, dtype=torch.float32, device=Ks.device)
        compute_ray_backward(g_o.contiguous(), g_d.contiguous(), Ks.reshape(-1, 9), g, locs)
        return g.reshape(ctx.n, 3, 4), None, None


class PoseChainFn(torch.autograd.Function):
    """(se3_refine [N,6], base_w2c [N,3,4]) -> c2w [N,3,4] = invert(compose([se3_to_SE3(se3_refine), base_w2c])):
    the whole se(3) chain of CAM.get_rts + Pose.invert in one kernel each way (csrc/pose.cu)."""

    @staticmethod
    def forward(ctx, se3, base):
        n = se3.shape[0]
        se3c, basec = se3.detach().contiguous(), base.contiguous()
        if not se3c.is_cuda:
            raise RuntimeError("pose chain: CUDA tensors required (no CPU fallback)")
        out = torch.empty(n, 3, 4, dtype=torch.float32, device=se3.device)
        capi.check(capi.lib().snrf_pose_fwd(capi.ptr(se3c), capi.ptr(basec), capi.ptr(out), capi.c_int(n), capi.stream()), "snrf_pose_fwd")
        ctx.save_for_backward(se3c, basec)
        return out

    @staticmethod
    def backward(ctx, g):
        se3c, basec = ctx.saved_tensors
        n = se3c.shape[0]
        g = g.contiguous()
        out = torch.empty(n, 6, dtype=torch.float32, device=g.device)
        capi.check(capi.lib().snrf_pose_bwd(capi.ptr(se3c), capi.ptr(basec), capi.ptr(g), capi.ptr(out), capi.c_int(n), capi.stream()), "snrf_pose_bwd")
        return out, None


class Poses(nn.Module):
    """camera_utils.CAM (camera_utils.py:40-89): w2c = se3_to_SE3(se3_refine) o (noise o ori_w2c)."""

    def __init__(self, Ks, c2ws, device, noise=None):
        super().__init__()
        self.device = device
        self.num_camera = c2ws.shape[0]
        self.ori_rts = pose_invert(c2ws.to(device))
        self.se3_refine = nn.Parameter(torch.zeros(self.num_camera, 6, dtype=torch.float32, device=device))
        self.rts = self.ori_rts.clone() if noise is None else pose_compose(se3_to_SE3(noise.to(device)), self.ori_rts)
        self.ks = Ks.to(device).contiguous()

    def get_rts(self):
        return pose_compose(se3_to_SE3(self.se3_refine), self.rts)

    def c2w(self):
        return PoseChainFn.apply(self.se3_refine, self.rts)

    def rays(self, locs):
        return RayGenFn.apply(self.c2w(), self.ks, locs)


class TileStep:
    """One tile: field + decoder + poses + optimisers, and the training step over one ray batch."""

    def __init__(self, device, tile_corner, tile_size, Ks, c2ws, log2_hashmap_size=24, grid_resolution=(32, 8192),
                 num_sample=128, num_bg_sample=128, mesh_path="", sampler_log2dim=4, pose_noise=None,
                 lr_table=1e-3, lr_decoder=1e-3, lr_cam=1e-4, global_step=10000, invalid_underground=False,
                 dense_table_adam=False, ert_eps=0.0):
        self.device = device
        f = lambda v: torch.as_tensor(v, dtype=torch.float32, device=device)
        self.featureGrid = HashGrid(device, f(tile_corner), f(tile_size), log2_hashmap_size, list(grid_resolution),
                                    sampler_log2dim, False, mesh_path)
        # early ray termination in training (opt-in, 0 = the reference's semantics; see HashGrid.ert_eps)
        self.featureGrid.ert_eps = float(ert_eps)
        self.decoder = ShallowMLP(32).to(device)
        self.poses = Poses(Ks, c2ws, device, pose_noise)
        self.num_sample, self.num_bg_sample = num_sample, num_bg_sample
        self.global_step = global_step
        self.invalid_underground = invalid_underground
        if dense_table_adam:     # what tile.py:301 does: dense torch Adam over the whole table
            self.featureGrid_optimizer = torch.optim.Adam(
                [{"params": self.featureGrid.parameters(), "lr": lr_table, "betas": (0.9, 0.99), "eps": 1e-15}])
        else:                    # sparse update of the touched entries only, gradient cleared in the same pass
            self.featureGrid_optimizer = vdbAdam(list(self.featureGrid.parameters()), lr=lr_table, betas=(0.9, 0.99),
                                                 eps=1e-15, bias_correction="standard", fused_zero_grad=True)
        # tile.py:317-326; fused=True: the 17 small tensors of the decoder and the pose offsets in one kernel per group
        # instead of ~15 foreach launches (same update rule)
        self.optimizer = torch.optim.Adam([
            {"params": self.decoder.parameters(), "lr": lr_decoder, "weight_decay": 1e-6},
            {"params": self.poses.se3_refine, "lr": lr_cam}], fused=torch.device(device).type == "cuda")
        # foreground / background chains on two CUDA streams (see render_rays): measured on B200 at default.yaml shape it
        # buys nothing at steady state (14.04 vs 14.10 ms / step) and costs allocator growth while the per-stream pools
        # settle, so it is off by default
        self.two_streams = False
        self.fused_table_update = True  # encode backward applies the sparse Adam slice by slice (see _table_backward)
        self.joint_chains = True        # foreground + background as one 2R-ray batch per kernel (render_fore_bg_rays)
        self._loss_host, self._loss_event, self._loss_wanted = None, None, False      # step(): early loss readback
        self.fused_loss = True          # step_device: merge + clamp + masked MSE + L2 regulariser and their gradient as one kernel
        self._side = None
        self.consensus = None           # ADMM state, see enable_consensus()
        self.camera_ids = None
        self.warp = None                # multi-view warp loss, see enable_warp_loss()

    def _side_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
            # parameter gradients are accumulated from both streams by design (autograd orders them with events)
            if hasattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch"):
                torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
        return self._side

    # ADMM pose consensus across tiles (admm_trainer.py:218-262, tile.py:477-508, consensus.py)
    def enable_consensus(self, camera_ids, num_camera_global, rho=100.0, group=None):
        """camera_ids: global ids [n_cam] of this tile's cameras.  Afterwards `synchronize()` exchanges poses with
        the other ranks (one NCCL all-reduce) and the loss carries the ADMM penalty (criterions.py:107-108)."""
        from admm import ConsensusManager, PoseConsensus
        self.camera_ids = torch.as_tensor(camera_ids, dtype=torch.long, device=self.device)
        self.consensus = ConsensusManager(self.poses.se3_refine, rho, self.device)
        self.exchange = PoseConsensus(num_camera_global, self.device, group)
        self.confidence = torch.ones(self.camera_ids.shape[0], dtype=torch.float32, device=self.device)

    def enable_warp_loss(self, images, alpha, gamma, weight=1.0, start_step=0, occlusions=None, topK=10):
        """criterions.py:92-97: adds the multi-view warp loss (warp_loss.WarpLoss) to the step.  images [N,H,W,3] uint8
        (or float in [0,1]) become device-resident; occlusions [N,H,W,1] bool or None."""
        from warp_loss_fused import WarpLoss
        self.warp = WarpLoss(self, images, alpha, gamma, topK=topK)
        self.warp_weight, self.warp_start = float(weight), int(start_step)
        self.warp_occlusions = occlusions.to(self.device).contiguous() if occlusions is not None else None

    def synchronize(self):
        """TILE.commit + master consensus + TILE.synchronize as one collective (every SYN_ITERS steps)."""
        out = self.exchange.exchange([(self.poses.se3_refine, self.camera_ids, self.confidence)])[0]
        self.consensus.update(out["shared_poses"], out["overlap_idxs"])

    # ---- shared depth / occlusion masks (tile.py:432-475, 366-430)
    def full_image_rays(self, view, H, W, stride=1):
        """All pixel rays of one camera (CAM.getRays(H, W, view_idx=[i]), camera_utils.py:91-141), every `stride`-th pixel."""
        ys, xs = torch.meshgrid(torch.arange(0, H, stride, device=self.device), torch.arange(0, W, stride, device=self.device), indexing="ij")
        locs = torch.stack([torch.full_like(xs, int(view)), xs, ys], -1).reshape(-1, 3).int().contiguous()
        with torch.no_grad():
            return self.poses.rays(locs)

    @torch.no_grad()
    def render_image(self, view, H, W, stride=1, chunk=1 << 16):
        """TILE.render_image_rays (tile.py:724-756): every `stride`-th pixel of camera `view` rendered in chunks of `chunk`
        rays with the inference path.  -> (color [h, w, 3], depth [h, w, 1]), h = ceil(H / stride), w = ceil(W / stride).
        No host synchronisation."""
        rays_o, rays_d = self.full_image_rays(view, H, W, stride)
        n = rays_o.shape[0]
        color = torch.zeros(n, 3, device=self.device)
        depth = torch.zeros(n, 1, device=self.device)
        for b in range(0, n, chunk):
            out, ok = self.render_rays(rays_o[b:b + chunk].contiguous(), rays_d[b:b + chunk].contiguous(), None, INFERENCE)
            if ok:
                color[b:b + chunk] = out["pred_color"]
                depth[b:b + chunk] = out["pred_depth"]
        h, w = (H + stride - 1) // stride, (W + stride - 1) // stride
        return color.reshape(h, w, 3), depth.reshape(h, w, 1)

    @torch.no_grad()
    def evaluate(self, views, images, masks=None, H=None, W=None):
        """Held-out view evaluation (tile.py:810-864): renders each camera of `views` (ints) at H x W (default: the images'
        size) and scores it against `images` [V,H,W,3] (uint8 or float32 in [0, 1], on the device) within `masks`
        [V,H,W(,1)] bool or None.  -> metrics.image_metrics' per-view {"mse", "psnr", "ssim", "count"} [V] plus their
        means "mean_mse", "mean_psnr", "mean_ssim", all device tensors; nothing synchronises until a value is read."""
        from metrics import image_metrics, with_means
        H = images.shape[-3] if H is None else H
        W = images.shape[-2] if W is None else W
        pred = torch.empty(len(views), H, W, 3, device=self.device)
        for k, v in enumerate(views):
            pred[k] = self.render_image(int(v), H, W)[0]
        return with_means(image_metrics(pred, images, masks))

    @torch.no_grad()
    def render_shared_depth(self, H, W, batch=1 << 16):
        """TILE.render_shared_depth: for every overlap camera of this tile whose centre lies INSIDE the tile's (doubled) box,
        the half-resolution depth map of the tile's current field.  -> (global camera ids [k], maps [k, H//2, W//2])."""
        if self.consensus is None:
            raise RuntimeError("render_shared_depth: enable_consensus() first (the overlap cameras come from the exchange)")
        center, half = self.featureGrid.bbox_center, self.featureGrid.bbox_size / 2.0
        cam_centres = self.poses.c2w()[:, :, 3]                                            # = the rays' origin
        ids, maps = [], []
        for i in torch.nonzero(self.consensus.overlap_flags)[:, 0].tolist():
            if not bool(torch.all(torch.abs(cam_centres[i] - center) < half / 2.0)):       # tile.py:445-448
                continue
            ids.append(int(self.camera_ids[i]))
            maps.append(self.render_image(i, H, W, stride=2, chunk=batch)[1][..., 0])      # TILE.render_depth_rays, tile.py:714-722
        if not ids:
            return torch.zeros(0, dtype=torch.long, device=self.device), torch.zeros(0, (H + 1) // 2, (W + 1) // 2, device=self.device)
        return torch.tensor(ids, dtype=torch.long, device=self.device), torch.stack(maps)

    @torch.no_grad()
    def update_occlusion_mask(self, have, maps, H, W, kernel_size=91):
        """TILE.update_occlusion_mask: have [n_cam] bool, maps [n_cam, H//2, W//2] = the exchanged depth of this tile's cameras
        (DepthExchange.exchange(..., want_ids=self.camera_ids)).  A pixel of a camera OUTSIDE the tile stays a training pixel
        only where the shared depth lies behind the ray's entry into the tile box; the kept region is eroded by a
        kernel_size box filter.  -> occlusions [n_cam, H, W, 1] bool (True = use the pixel)."""
        n = self.poses.num_camera
        occl = torch.ones(n, H, W, 1, dtype=torch.bool, device=self.device)
        center, half = self.featureGrid.bbox_center, self.featureGrid.bbox_size / 2.0
        kernel = torch.ones(1, 1, kernel_size, kernel_size, device=self.device)
        from cuda import ray_aabb_intersection
        for i in torch.nonzero(have)[:, 0].tolist():
            rays_o, rays_d = self.full_image_rays(i, H, W)
            if bool(torch.all(torch.abs(rays_o[0] - center) < half / 2.0)):               # camera inside the tile: nothing hides it
                continue
            depth = maps[i].repeat_interleave(2, 0).repeat_interleave(2, 1)[:H, :W].reshape(-1, 1)
            bounds = torch.full((rays_o.shape[0], 2), -1.0, device=self.device)
            ray_aabb_intersection(rays_o.contiguous(), rays_d.contiguous(), center, half, bounds)
            vis = ((depth > bounds[:, :1]) & (bounds[:, :1] != -1)).reshape(1, 1, H, W).float()
            vis = 1.0 - torch.nn.functional.conv2d(1.0 - vis, kernel, padding=kernel_size // 2).clamp(0, 1)
            occl[i] = vis.bool().reshape(H, W, 1)
        self.shared_occlusions = occl
        return occl

    # tile.py:639-692
    def render_rays(self, rays_o, rays_d, occlusion_mask=None, mode=TRAIN):
        # The foreground and the background chains (sample -> encode -> decoder -> composite) are independent until the
        # colours are merged; with two_streams they are issued on two CUDA streams (the backward follows: autograd runs on
        # the streams of the forward ops).
        joint = None
        if self.joint_chains and self.num_sample == self.num_bg_sample:
            # both chains as one batch of 2R rays through every kernel (HashGrid.render_fore_bg_rays)
            joint = self.featureGrid.render_fore_bg_rays(rays_o, rays_d, self.num_sample, self.decoder, mode,
                                                         occlusion_mask=occlusion_mask, global_step=self.global_step,
                                                         invalid_underground=self.invalid_underground)
        if joint is not None:
            (fg, bg), ret_fg, ret_bg = joint, True, True
            out = {"rays_o": rays_o, "rays_d": rays_d, "ret_fg": True}
            out.update(fg)
        else:
            side = self._side_stream() if self.two_streams else None
            if side is not None:
                main = torch.cuda.current_stream()
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    bg, ret_bg = self.featureGrid.render_bg_rays(rays_o, rays_d, self.num_bg_sample, self.decoder, mode,
                                                                 occlusion_mask=occlusion_mask, global_step=self.global_step,
                                                                 bg_mode="IZ", infinity=True, fmesh=None,
                                                                 invalid_underground=self.invalid_underground)
            fg, ret_fg = self.featureGrid.render_fore_rays(rays_o, rays_d, self.num_sample, self.decoder, mode,
                                                           occlusion_mask=occlusion_mask, global_step=self.global_step)
            out = {"rays_o": rays_o, "rays_d": rays_d, "ret_fg": ret_fg}
            if ret_fg:
                out.update(fg)
            else:
                out["fore_valid"] = torch.zeros(rays_d[..., 0].shape, dtype=torch.bool, device=self.device)
            if side is not None:
                torch.cuda.current_stream().wait_stream(side)
                if ret_bg:
                    for v in bg.values():             # produced on the side stream, consumed (and freed) on the main one
                        if torch.is_tensor(v):
                            v.record_stream(torch.cuda.current_stream())
            else:
                bg, ret_bg = self.featureGrid.render_bg_rays(rays_o, rays_d, self.num_bg_sample, self.decoder, mode,
                                                             occlusion_mask=occlusion_mask, global_step=self.global_step,
                                                             bg_mode="IZ", infinity=True, fmesh=None,
                                                             invalid_underground=self.invalid_underground)
        if ret_fg is False and ret_bg is False:
            return None, False
        out["ret_bg"] = ret_bg
        if ret_bg:
            out["bg_valid"] = bg["valid"]
            if ret_fg:
                T = fg["T_left"]
                out["pred_color"] = out["pred_color"] + T * bg["rgb"]
                out["pred_depth"] = out["pred_depth"] + T * bg["depth"]
                out["pred_specular"] = fg["specular"] + T * bg["specular"]
                out["pred_diffuse"] = fg["diffuse"] + T * bg["diffuse"]
                if mode == TRAIN:
                    out["l2_reg_specular"] = out["l2_reg_specular"] + bg["l2_reg_specular"]
            else:
                out["pred_color"], out["pred_depth"] = bg["rgb"], bg["depth"]
                out["pred_specular"], out["pred_diffuse"] = bg["specular"], bg["diffuse"]
                if mode == TRAIN:
                    out["l2_reg_specular"] = bg["l2_reg_specular"]
        else:
            out["pred_specular"], out["pred_diffuse"] = fg["specular"], fg["diffuse"]
        return out, True

    def loss(self, locs, gt_color):
        rays_o, rays_d = self.poses.rays(locs)
        out, ok = self.render_rays(rays_o, rays_d, None, TRAIN)
        if not ok:
            return None, None
        # criterions.py:126-147: MSE over the rays that were rendered at all (fore_valid | bg_valid) -- as a masked mean,
        # the reference's boolean indexing would synchronise with the host
        valid = out["fore_valid"] if out["ret_fg"] else None
        if out["ret_bg"]:
            valid = out["bg_valid"] if valid is None else valid | out["bg_valid"]
        sq = (out["pred_color"] - gt_color) ** 2
        mse = (sq * valid[:, None]).sum() / (3.0 * valid.sum().clamp_min(1))
        loss = mse + 0.01 * out["l2_reg_specular"]                         # tile.py:999
        if self.warp is not None and self.global_step >= self.warp_start and self.warp_weight > 0:
            # "Warp Loss" item (criterions.py:92-97, 148-163) with its warming schedule (:19-22)
            w = self.warp_weight * max(min(self.global_step / 10000.0, 1.0), 0.0)
            loss = loss + w * self.warp(self.global_step, out["rays_o"], out["rays_d"], out["pred_depth"], out["pred_diffuse"],
                                        out["pred_specular"], gt_color, valid, self.warp_occlusions)
        if self.consensus is not None and self.consensus.has_overlap:
            loss = loss + self.consensus.camera_loss()                     # "Admm Loss", weight 1 (criterions.py:107-108)
        return loss, out

    def _table_backward(self):
        """The explicit opt-in for where the table gradient goes (hashgrid/_gradmode.py).  vdbAdam: scatter + update fusion, the
        gradient table never exists -- it needs exactly one encode of the table in the BACKWARD, which also holds with the warp
        loss: its re-render of the neighbour rays (warp_loss.py:355-377, compute_visibility) runs without a graph, only the
        main chain is differentiated (vdbAdam raises if a second encode ever reaches the backward).  Otherwise: accumulate
        into `.grad` in place."""
        from hashgrid import _gradmode
        opt = self.featureGrid_optimizer
        if isinstance(opt, vdbAdam):
            return opt.table_backward(fused=self.fused_table_update)
        return _gradmode.table_backward("direct")

    def loss_fused(self, locs, gt_color):
        """The loss of `loss()` without its dictionary of intermediate images: the colour terms come from one kernel
        (HashGrid.fore_bg_colour_loss).  None when that path does not apply (warp loss, separate chains, non-stock decoder)."""
        if not (getattr(self, "fused_loss", False) and self.joint_chains and self.warp is None and self.num_sample == self.num_bg_sample):
            return None
        rays_o, rays_d = self.poses.rays(locs)
        loss = self.featureGrid.fore_bg_colour_loss(rays_o, rays_d, self.num_sample, self.decoder, gt_color, 0.01,
                                                    self.global_step, self.invalid_underground)
        if loss is not None and self.consensus is not None and self.consensus.has_overlap:
            loss = loss + self.consensus.camera_loss()                     # "Admm Loss", weight 1 (criterions.py:107-108)
        return loss

    def step_device(self, locs, gt_color):
        """Inputs already on the device.  Returns the loss as a device scalar (no host sync)."""
        loss = self.loss_fused(locs, gt_color)
        if loss is None:
            loss, _ = self.loss(locs, gt_color)
        if loss is None:
            self.global_step += 1
            loss = torch.zeros((), device=self.device)
            self._post_loss(loss)
            return loss
        self._post_loss(loss.detach())
        self.featureGrid_optimizer.zero_grad()
        self.optimizer.zero_grad()
        with self._table_backward():
            loss.backward()
        self.featureGrid_optimizer.step()
        self.optimizer.step()
        self.global_step += 1
        return loss.detach()

    # ------------------------------------------------------------------ on-disk formats (tile.py:509-572, 35-45, 67-68, 128-136, 302-338)
    def export_tile(self, output_dir, visible_poses=None):
        """tile-<idx>/ as the reference's renderer reads it (rendering.py:86-113): feature.npz (fp16 table, occupancy,
        doubled box, grid_log2dim, resolution), decoder.pth (ShallowMLP state_dict), cams.npz (c2ws, ks, idxs)."""
        import os
        import numpy as np
        os.makedirs(output_dir, exist_ok=True)
        self.featureGrid.export(output_dir)
        torch.save(self.decoder.state_dict(), os.path.join(output_dir, "decoder.pth"))
        with torch.no_grad():
            c2ws = self.poses.c2w().detach().cpu().numpy()
        if visible_poses is None:
            visible_poses = self.camera_ids.cpu().numpy() if self.camera_ids is not None else np.arange(c2ws.shape[0])
        np.savez(os.path.join(output_dir, "cams.npz"), c2ws=c2ws, ks=self.poses.ks.detach().cpu().numpy(), idxs=np.array(visible_poses))
        return output_dir

    def export_check_point(self, output_dir, tile_idx=0):
        """checkpoint-<step>-<tile>.pt with the reference's keys (tile.py:534-572).  `poses` (the refined se(3) offsets)
        is an extra key: the reference's resume restores the optimiser moments of se3_refine but not its value."""
        import os
        ck = {"global_step": self.global_step, "hashgrid": self.featureGrid.export_check_point(),
              "admm": self.consensus.export_check_point() if self.consensus is not None else None,
              "decoder": self.decoder.state_dict(), "featureGrid_optimizer": self.featureGrid_optimizer.state_dict(),
              "optimizer": self.optimizer.state_dict(), "poses": self.poses.se3_refine.detach().cpu()}
        os.makedirs(output_dir, exist_ok=True)
        path = os.path.join(output_dir, f"checkpoint-{self.global_step}-{tile_idx}.pt")
        torch.save(ck, path)
        return path

    def load_check_point(self, path_or_dict):
        """Resume from export_check_point() output -- or from a checkpoint the reference wrote (no `poses` key)."""
        ck = path_or_dict if isinstance(path_or_dict, dict) else torch.load(path_or_dict, map_location=self.device, weights_only=False)
        self.global_step = int(ck["global_step"])
        table = self.featureGrid.HE.features
        self.featureGrid.load_check_point(ck["hashgrid"])
        if self.featureGrid.HE.features is not table:            # keep the Parameter the optimiser holds
            with torch.no_grad():
                table.copy_(self.featureGrid.HE.features)
            self.featureGrid.HE.features = table
        self.decoder.load_state_dict(ck["decoder"])
        self.featureGrid_optimizer.load_state_dict(ck["featureGrid_optimizer"])
        self.optimizer.load_state_dict(ck["optimizer"])
        if ck.get("admm") is not None and self.consensus is not None:
            self.consensus.load_check_point(ck["admm"])
        if ck.get("poses") is not None:
            with torch.no_grad():
                self.poses.se3_refine.copy_(ck["poses"].to(self.device))

    def _post_loss(self, loss):
        """step(): the loss starts its way to the host as soon as the forward has produced it -- a copy into pinned memory and
        an event BEFORE the backward is issued -- so that reading it does not wait for the backward / the optimisers."""
        if getattr(self, "_loss_host", None) is not None and self._loss_wanted:
            self._loss_host.copy_(loss.reshape(1), non_blocking=True)
            self._loss_event.record()

    def step(self, locs_host, gt_host):
        """The end-to-end call: pinned host batch in, python float loss out.  The float is this step's loss, read back inside the
        call; the call returns once the FORWARD has run on the device (the backward and the updates are queued behind it), so
        a training loop that logs the loss every step keeps the device busy instead of draining it once per step."""
        if getattr(self, "_loss_host", None) is None:
            self._loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
            self._loss_event = torch.cuda.Event()
        self._loss_wanted = True
        try:
            locs = locs_host.to(self.device, non_blocking=True)
            gt = gt_host.to(self.device, non_blocking=True)
            self.step_device(locs, gt)
        finally:
            self._loss_wanted = False
        self._loss_event.synchronize()
        return float(self._loss_host[0])
