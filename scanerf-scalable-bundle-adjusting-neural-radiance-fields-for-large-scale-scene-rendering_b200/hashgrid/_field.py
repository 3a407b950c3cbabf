"""Bridge to the tensor-core decoder kernels (csrc/decoder.cu): the reference's
network.ShallowMLP.forward (network.py:151-190) evaluated by tcgen05 MMAs, as an
autograd.Function over (features, decoder parameters, ray directions)."""
import ctypes

import torch
from torch.utils.weak import WeakIdKeyDictionary

import scanerf_b200_capi as capi
from . import _gradmode
from scanerf_b200_capi import c_float, c_int, c_void_p, ptr

f32 = torch.float32


def set_precision(split=True):
    """True (default): error-compensated bf16x3 operands in the forward GEMMs (fp32-grade heads);
    False: plain bf16 operands (fastest, ~1 % error in the directional branch)."""
    capi.lib().snrf_decoder_set_precision(c_int(1 if split else 0))


def _param_array(params):
    ps = [p.detach().contiguous() for p in params]
    for p in ps:
        if not p.is_cuda or p.dtype != f32:
            raise RuntimeError("decoder parameters must be float32 CUDA tensors (no CPU fallback)")
    arr = (ctypes.c_void_p * 16)(*[p.data_ptr() for p in ps])
    return arr, ps


def _layout(feats):
    """[N,32] row-major -> (N, 0);  [16,N,2] level-major (snrf_field_encode_* layout) -> (N, 1)."""
    if feats.dim() == 3:
        if feats.shape[0] != 16 or feats.shape[2] != 2:
            raise RuntimeError(f"level-major features must be [16, N, 2], got {tuple(feats.shape)}")
        return int(feats.shape[1]), 1
    return int(feats.shape[0]), 0


def decoder_forward(feats, mask32, rays_d, S, params, valid=None):
    """feats [N,32] f32 (or level-major [16,N,2]), mask32 [32] f32 or None, rays_d [R,3] (sample n ->
    ray n // S), params = the 16 tensors of hashgrid._decoder.decoder_params().  Returns heads [N,10] =
    (sigma, tint3, diffuse3, specular3)."""
    N, lm = _layout(feats)
    feats = feats.contiguous()
    rays_d = rays_d.contiguous()
    if not feats.is_cuda:
        raise RuntimeError("decoder_forward: CUDA tensors required (no CPU fallback)")
    out = torch.empty(N, 10, dtype=f32, device=feats.device)
    arr, keep = _param_array(params)
    m = mask32.contiguous() if mask32 is not None else None
    rc = capi.lib().snrf_decoder_fwd(ptr(feats), ptr(m), ptr(rays_d), arr, ptr(out), c_int(N), c_int(int(S)), c_int(lm), ptr(valid), capi.stream())
    capi.check(rc, "snrf_decoder_fwd")
    return out


class DecoderFn(torch.autograd.Function):
    """(feats [N,32], rays_d [R,3], mask32 [32] | None, S, *16 params) -> heads [N,10].
    Backward recomputes the forward tile by tile on the tensor cores (nothing is saved but the
    inputs) and returns d/d feats, d/d rays_d (through the SH view encoding) and d/d params."""

    @staticmethod
    def forward(ctx, feats, rays_d, mask32, S, valid, ert, *params):
        feats = feats.contiguous()
        rays_d = rays_d.contiguous()
        heads = decoder_forward(feats, mask32, rays_d, S, params, valid)
        ctx.S = int(S)
        ctx.ert = ert           # _render.ErtState | None: its sample flags exist by the time the backward runs
        ctx.has_mask, ctx.has_valid = mask32 is not None, valid is not None
        ctx.save_for_backward(feats, rays_d, mask32 if mask32 is not None else feats.new_empty(0),
                              valid if valid is not None else feats.new_empty(0), heads, *params)
        return heads

    @staticmethod
    def backward(ctx, g_heads):
        feats, rays_d, mask32, valid, heads = ctx.saved_tensors[:5]
        params = ctx.saved_tensors[5:]
        N, lm = _layout(feats)
        g_heads = g_heads.contiguous()
        g_feats = torch.empty_like(feats)
        g_d = torch.zeros_like(rays_d) if ctx.needs_input_grad[1] else None
        sizes = [p.numel() for p in params]
        flat = torch.zeros(sum(sizes), dtype=f32, device=feats.device)
        g_params, o = [], 0
        for p, n in zip(params, sizes):
            g_params.append(flat[o:o + n].view_as(p))
            o += n
        arr, keep = _param_array(params)
        garr = (ctypes.c_void_p * 16)(*[g.data_ptr() for g in g_params])
        m = mask32.contiguous() if ctx.has_mask else None
        args = (ptr(feats), ptr(m), ptr(rays_d), arr, ptr(g_heads), ptr(g_feats), ptr(g_d), garr,
                c_int(N), c_int(ctx.S), c_int(lm), ptr(valid) if ctx.has_valid else c_void_p(0), ptr(heads))
        if ctx.ert is not None and ctx.ert.sample_live is not None:
            rc = capi.lib().snrf_decoder_bwd_ert(*args, ptr(ctx.ert.sample_live), capi.stream())
        else:
            rc = capi.lib().snrf_decoder_bwd(*args, capi.stream())
        capi.check(rc, "snrf_decoder_bwd")
        return (g_feats, g_d, None, None, None, None) + tuple(g_params)


def decoder_apply(feats, rays_d, mask32, S, params, valid=None, ert=None):
    """valid (bool [R] or None): samples of rays flagged False are skipped (rows left unwritten).
    ert (_render.ErtState | None): early ray termination -- the backward skips the samples the compositing flagged dead."""
    return DecoderFn.apply(feats, rays_d, mask32, S, valid, ert, *params)


# resolution tensor (by identity: the entry dies with the tensor) -> (its version counter when counted, count)
_small_levels_cache = WeakIdKeyDictionary()
SMALL_LEVEL_LOG2 = 22          # levels with at most this many grid vertices are reduced in one pass (tools/sweep_small_levels.py)


def small_levels(resolution):
    """Number of leading levels whose grid has at most 2^22 vertices ((rx+1)(ry+1)(rz+1)): however large the hash table,
    such a level touches few entries, and the fused backward reduces it in one pass (snrf_field_encode_bwd_adam).
    Read back from the device once per resolution tensor and in-place change of it."""
    cacheable = not resolution.is_inference()          # (inference tensors have no version counter)
    hit = _small_levels_cache.get(resolution) if cacheable else None
    if hit is not None and hit[0] == resolution._version:
        return hit[1]
    r = resolution.detach().cpu().long() + 1
    verts = r[:, 0] * r[:, 1] * r[:, 2]
    n = 0
    while n < verts.shape[0] and int(verts[n]) <= (1 << SMALL_LEVEL_LOG2):
        n += 1
    if cacheable:
        _small_levels_cache[resolution] = (resolution._version, n)
    return n


class FieldEncodeFn(torch.autograd.Function):
    """(rays_o [R,3], rays_d [R,3], z_vals [R,S], features [16,T,2], resolution, box_min, box_size, mode)
    -> level-major features [16, R*S, 2]: sample position, space contraction (mode 1 = fore, 2 =
    background) and hash encode in one kernel (csrc/field_encode.cu).  The forward stores the per-level
    Jacobians; the backward is a pure gradient scatter into `features.grad` (accumulated in place, no dense
    temporary) and returns d/d rays_o, d/d rays_d.  Where the table gradient goes is decided by
    `_gradmode`: returned densely (default, autograd-conformant), accumulated into `features.grad` ("direct"), or
    consumed on the spot by the sparse Adam update ("fused": snrf_field_encode_bwd_adam).
    `jac_out` (a list or None) receives the Jacobians [16, 3, R*S, 2], computed for it also when the rays need no gradient;
    they are kept for the backward only when the rays do."""

    @staticmethod
    def forward(ctx, rays_o, rays_d, z_vals, features, resolution, box_min, box_size, mode, valid, split=0, ert=None, jac_out=None):
        R, S = z_vals.shape
        ctx.ert = ert
        N, L, T = R * S, int(features.shape[0]), int(features.shape[1])
        rays_o, rays_d, z_vals = rays_o.contiguous(), rays_d.contiguous(), z_vals.contiguous()
        for t in (rays_o, rays_d, z_vals, features):
            if not t.is_cuda or t.dtype != f32:
                raise RuntimeError("field encode: float32 CUDA tensors required (no CPU fallback)")
        need_pos = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        out = torch.empty(L, N, 2, dtype=f32, device=z_vals.device)
        jac = torch.empty(L, 3, N, 2, dtype=f32, device=z_vals.device) if (need_pos or jac_out is not None) else None
        feats = features.detach().contiguous()
        box_min, box_size = box_min.contiguous(), box_size.contiguous()
        rc = capi.lib().snrf_field_encode_fwd(ptr(rays_o), ptr(rays_d), ptr(z_vals), c_void_p(0), ptr(box_min), ptr(box_size),
                                              c_int(int(mode)), ptr(feats), ptr(resolution), ptr(out), ptr(jac), ptr(valid), c_int(int(split)), c_int(N), c_int(S),
                                              c_int(L), c_int(T), capi.stream())
        capi.check(rc, "snrf_field_encode_fwd")
        ctx.mode, ctx.split, ctx.dims = int(mode), int(split), (N, S, L, T)
        ctx.small_levels = small_levels(resolution)
        ctx.features = features
        if jac_out is not None:
            jac_out.append(jac)
        ctx.save_for_backward(rays_o, rays_d, z_vals, resolution, box_min, box_size, jac if need_pos else out.new_empty(0),
                              valid if valid is not None else out.new_empty(0))
        ctx.has_jac, ctx.has_valid = need_pos, valid is not None
        return out

    @staticmethod
    def backward(ctx, g_out):
        rays_o, rays_d, z_vals, resolution, box_min, box_size, jac, valid = ctx.saved_tensors
        N, S, L, T = ctx.dims
        features = ctx.features
        g_out = g_out.contiguous()
        g_o = torch.zeros_like(rays_o) if ctx.needs_input_grad[0] else None
        g_d = torch.zeros_like(rays_d) if ctx.needs_input_grad[1] else None
        mode = _gradmode.mode() if (features.is_leaf and features.requires_grad) else None
        common = (ptr(rays_o), ptr(rays_d), ptr(z_vals), c_void_p(0), ptr(box_min), ptr(box_size), c_int(ctx.mode), ptr(resolution),
                  ptr(g_out), ptr(jac) if ctx.has_jac else c_void_p(0), ptr(g_o), ptr(g_d), c_void_p(0))
        live = ctx.ert.sample_live if (ctx.ert is not None and ctx.ert.sample_live is not None) else None
        sfx = "_ert" if live is not None else ""
        tail = (ptr(valid) if ctx.has_valid else c_void_p(0), c_int(ctx.split), c_int(N), c_int(S), c_int(L), c_int(T)) + \
               ((ptr(live),) if live is not None else ()) + (capi.stream(),)
        if mode == "fused" and _gradmode.optimizer().owns(features):
            # scatter + sparse Adam in one pass: the table gradient never exists in HBM
            opt = _gradmode.optimizer()
            m, v, hyper, step, scratch = opt.begin_fused(features, ctx.small_levels)
            cpts = torch.empty(3, N, dtype=f32, device=g_out.device)
            fn = getattr(capi.lib(), "snrf_field_encode_bwd_adam" + sfx)
            rc = fn(*common, ptr(features.data), ptr(m), ptr(v), c_float(hyper["lr"]), c_float(hyper["beta1"]),
                    c_float(hyper["beta2"]), c_float(hyper["eps"]), c_int(step), ptr(scratch),
                    ctypes.c_longlong(scratch.shape[0]), c_int(ctx.small_levels), ptr(cpts), *tail)
            capi.check(rc, "snrf_field_encode_bwd_adam")
            capi.launch_count += int(capi.lib().snrf_field_last_launch_count()) - 1     # one C call, many kernels
            return g_o, g_d, None, None, None, None, None, None, None, None, None, None
        direct = mode is not None
        if direct:
            # the training step's explicit opt-in (_gradmode.table_backward): accumulate in place, no dense temporary
            if features.grad is None:
                features.grad = torch.zeros_like(features)
            g_table, first = features.grad, False
        else:
            # autograd-conformant default: a dense grad_features, shared by the encodes of one backward pass (_gradmode)
            g_table, first = _gradmode.shared_table_grad(features)
        rc = getattr(capi.lib(), "snrf_field_encode_bwd" + sfx)(*common, ptr(g_table), *tail)
        capi.check(rc, "snrf_field_encode_bwd")
        return g_o, g_d, None, (g_table if first else None), None, None, None, None, None, None, None, None


def field_encode(rays_o, rays_d, z_vals, features, resolution, box_min, box_size, mode, valid=None, split=0, ert=None, jac_out=None):
    """valid (bool [R] or None): rays flagged False are skipped (their feature rows are left unwritten).
    mode 3: rays [0, split) are contracted with the fore map, rays [split, R) with the background map.
    ert (_render.ErtState | None): early ray termination -- the backward skips the samples the compositing flagged dead.
    jac_out (list | None): receives the forward's per-level Jacobians (see FieldEncodeFn), e.g. for field_normal."""
    return FieldEncodeFn.apply(rays_o, rays_d, z_vals, features, resolution, box_min, box_size, mode, valid, split, ert, jac_out)


def field_normal(feats, jac, mask32, params, rays_o, rays_d, z_vals, box_min, box_size, mode, valid=None, normal=None, grad=None):
    """Surface normal -d sigma/dx / (|d sigma/dx| + 1e-8) at every sample of a field_encode call (snrf_field_normal): feats
    [16, N, 2] and jac [16, 3, N, 2] from that call, mask32 [32] the level mask, params the 16 decoder tensors
    (hashgrid._decoder.decoder_params), mode 1 (fore) or 2 (background) as there.  Forward only: nothing is differentiated.
    Returns normal [N, 3]; `normal` / `grad` ([N, 3], optional) are buffers to write, grad receiving d sigma / dx itself.
    Rows of rays flagged False in `valid` are left as they are."""
    R, S = z_vals.shape
    N = R * S
    if tuple(feats.shape) != (16, N, 2) or tuple(jac.shape) != (16, 3, N, 2):
        raise RuntimeError(f"field_normal: features [16, {N}, 2] and Jacobians [16, 3, {N}, 2] required, "
                           f"got {tuple(feats.shape)} and {tuple(jac.shape)}")
    for t in (feats, jac, rays_o, rays_d, z_vals):
        if not t.is_cuda or t.dtype != f32 or not t.is_contiguous():
            raise RuntimeError("field_normal: contiguous float32 CUDA tensors required (no CPU fallback)")
    if normal is None:
        normal = torch.empty(N, 3, dtype=f32, device=feats.device)
    arr, keep = _param_array(params)
    m = mask32.contiguous() if mask32 is not None else None
    rc = capi.lib().snrf_field_normal(ptr(feats), ptr(jac), ptr(m), arr, c_int(int(mode)), ptr(box_min.contiguous()),
                                      ptr(box_size.contiguous()), ptr(rays_o), ptr(rays_d), ptr(z_vals), ptr(valid), ptr(normal),
                                      ptr(grad), c_int(N), c_int(S), capi.stream())
    capi.check(rc, "snrf_field_normal")
    return normal
