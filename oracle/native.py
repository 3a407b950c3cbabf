"""ctypes/numpy face of oracle/scanerf_oracle.c (TEST INFRASTRUCTURE ONLY).

Every function takes and returns numpy arrays; sizes are small enough for the
C oracle to finish in seconds.  See scanerf_oracle.c for the reference
file:line each function restates.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libscanerf_oracle.so")
_lib = None


def build(force=False):
    src = os.path.join(_HERE, "scanerf_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return _SO


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else ctypes.c_void_p(0)


def hash_encode_fwd(points, table, res, corner=None, size=None, want_idx=False):
    points, table, res = _f32(points), _f32(table), _i32(res)
    B, (L, T) = points.shape[0], table.shape[:2]
    out = np.zeros((B, L, 2), np.float32)
    idx = np.zeros((B, L, 8), np.uint32) if want_idx else None
    c = _f32(corner) if corner is not None else None
    s = _f32(size) if size is not None else None
    lib().oracle_hash_encode_fwd(_p(points), _p(table), _p(res), _p(c), _p(s), _p(out), _p(idx),
                                 ctypes.c_int(B), ctypes.c_int(L), ctypes.c_int(T))
    return (out, idx) if want_idx else out


def hash_encode_bwd(points, grad_in, table, res, corner=None, size=None):
    points, grad_in, table, res = _f32(points), _f32(grad_in), _f32(table), _i32(res)
    B, (L, T) = points.shape[0], table.shape[:2]
    gp = np.zeros((B, 3), np.float32)
    gt = np.zeros_like(table)
    c = _f32(corner) if corner is not None else None
    s = _f32(size) if size is not None else None
    lib().oracle_hash_encode_bwd(_p(points), _p(grad_in), _p(table), _p(res), _p(c), _p(s), _p(gp), _p(gt),
                                 ctypes.c_int(B), ctypes.c_int(L), ctypes.c_int(T))
    return gp, gt


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def compute_ray_fwd(Ks, C2Ws, locs):
    Ks, C2Ws, locs = _f32(Ks), _f32(C2Ws), _i32(locs)
    B = locs.shape[0]
    o, d = np.zeros((B, 3), np.float32), np.zeros((B, 3), np.float32)
    lib().oracle_compute_ray_fwd(_p(o), _p(d), _p(Ks), _p(C2Ws), _p(locs), ctypes.c_int(B))
    return o, d


def compute_ray_bwd(g_o, g_d, Ks, locs, n_cam, ref_index_bug=False):
    g_o, g_d, Ks, locs = _f32(g_o), _f32(g_d), _f32(Ks), _i32(locs)
    g = np.zeros((n_cam, 12), np.float32)
    lib().oracle_compute_ray_bwd(_p(g_o), _p(g_d), _p(Ks), _p(g), _p(locs), ctypes.c_int(locs.shape[0]),
                                 ctypes.c_int(int(ref_index_bug)))
    return g


def ray_aabb(rays_o, rays_d, centers, sizes):
    rays_o, rays_d = _f32(rays_o), _f32(rays_d)
    centers, sizes = _f32(centers).reshape(-1, 3), _f32(sizes).reshape(-1, 3)
    B, K = rays_o.shape[0], centers.shape[0]
    out = np.zeros((B, K, 2), np.float32)
    lib().oracle_ray_aabb(_p(rays_o), _p(rays_d), _p(centers), _p(sizes), _p(out), ctypes.c_int(B), ctypes.c_int(K))
    return out


def sample_points_grid(rays_o, rays_d, corner, size, occupied, log2dim, S, fill=-1.0):
    rays_o, rays_d, corner, size = _f32(rays_o), _f32(rays_d), _f32(corner), _f32(size)
    occ, log2dim = _u8(occupied), _i32(log2dim)
    B = rays_o.shape[0]
    z = np.full((B, S), fill, np.float32)
    d = np.full((B, S), fill, np.float32)
    counts = np.zeros(B, np.int32)
    lib().oracle_sample_points_grid(_p(rays_o), _p(rays_d), _p(z), _p(d), _p(corner), _p(size), _p(occ),
                                    _p(log2dim), _p(counts), ctypes.c_int(B), ctypes.c_int(S))
    return z, d, counts


def background_sampling(starts, bg_depth, S, sample_range):
    starts, bg_depth = _f32(starts), _f32(bg_depth)
    B = starts.shape[0]
    z = np.zeros((B, S), np.float32)
    lib().oracle_background_sampling(_p(starts), _p(bg_depth), _p(z), ctypes.c_int(B), ctypes.c_int(S),
                                     ctypes.c_float(sample_range))
    return z


def sample_insideout(rays_o, rays_d, S, Sbg, center, size, far):
    rays_o, rays_d, center, size = _f32(rays_o), _f32(rays_d), _f32(center), _f32(size)
    B = rays_o.shape[0]
    z, zb = np.zeros((B, S), np.float32), np.zeros((B, Sbg), np.float32)
    lib().oracle_sample_insideout.restype = ctypes.c_int
    miss = lib().oracle_sample_insideout(_p(rays_o), _p(rays_d), ctypes.c_int(S), ctypes.c_int(Sbg), _p(center),
                                         _p(size), ctypes.c_float(far), _p(z), _p(zb), ctypes.c_int(B))
    return z, zb, miss


def adam_step(params, grads, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, step, row_stride=None, half_state=False):
    """In-place on float32 copies; returns (params, exp_avg, exp_avg_sq).  params [K,D]."""
    p, g = _f32(params).copy(), _f32(grads)
    m, v = _f32(exp_avg).copy(), _f32(exp_avg_sq).copy()
    K, D = p.shape
    rs = D if row_stride is None else row_stride
    lib().oracle_adam_step(_p(p), _p(g), _p(m), _p(v), ctypes.c_longlong(K), ctypes.c_int(D), ctypes.c_int(rs),
                           ctypes.c_int(int(half_state)), ctypes.c_float(lr), ctypes.c_float(beta1),
                           ctypes.c_float(beta2), ctypes.c_float(eps), ctypes.c_int(step))
    return p, m, v


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _scene(corners, sizes, occupied, starts, log2dim):
    return _f32(corners), _f32(sizes), _u8(occupied), _i64(starts), _i32(log2dim)


def render_sample(rays_o, rays_d, corners, sizes, occupied, starts, log2dim, order, isect, tracing_idx, z_start, z_vals, dists):
    """One call of the multi-tile render sampler; tracing_idx [B], z_start [B], z_vals / dists [B,S] are updated in place
    (they must be contiguous int32 / float32 arrays)."""
    rays_o, rays_d, order, isect = _f32(rays_o), _f32(rays_d), _i32(order), _f32(isect)
    c, s, occ, st, l2 = _scene(corners, sizes, occupied, starts, log2dim)
    for a, t in ((tracing_idx, np.int32), (z_start, np.float32), (z_vals, np.float32), (dists, np.float32)):
        assert a.dtype == t and a.flags.c_contiguous
    B, nb, S = rays_o.shape[0], c.shape[0], z_vals.shape[1]
    lib().oracle_render_sample(_p(rays_o), _p(rays_d), _p(c), _p(s), _p(occ), _p(st), _p(l2), _p(order), _p(isect), _p(tracing_idx),
                               _p(z_start), _p(z_vals), _p(dists), ctypes.c_int(B), ctypes.c_int(nb), ctypes.c_int(S))


def firsthit_block(rays_o, rays_d, corners, sizes, occupied, starts, log2dim, order, isect, hit_init=-1):
    rays_o, rays_d, order, isect = _f32(rays_o), _f32(rays_d), _i32(order), _f32(isect)
    c, s, occ, st, l2 = _scene(corners, sizes, occupied, starts, log2dim)
    B, nb = rays_o.shape[0], c.shape[0]
    hit = np.full(B, hit_init, np.int16)
    lib().oracle_firsthit_block(_p(rays_o), _p(rays_d), _p(c), _p(s), _p(occ), _p(st), _p(l2), _p(order), _p(isect), _p(hit),
                                ctypes.c_int(B), ctypes.c_int(nb))
    return hit


def process_occupied(bidx, total_grid, corners, sizes, occupied, starts, log2dim, target):
    """Returns a copy of `target` (the concatenated grids) with tile bidx's occupied cells dilated into the other tiles."""
    c, s, occ, st, l2 = _scene(corners, sizes, occupied, starts, log2dim)
    tgt = _u8(target).copy()
    lib().oracle_process_occupied(ctypes.c_int(bidx), ctypes.c_int(total_grid), _p(c), _p(s), _p(occ), _p(st), _p(l2), _p(tgt),
                                  ctypes.c_int(c.shape[0]))
    return tgt


def outgoing_bidx(rays_o, rays_d, corners, sizes, order, isect, skip=False):
    rays_o, rays_d, corners, sizes, order, isect = _f32(rays_o), _f32(rays_d), _f32(corners), _f32(sizes), _i32(order), _f32(isect)
    B, nb = order.shape
    ids, w = np.full((B, 4), -1, np.int16), np.zeros((B, 4), np.float32)
    lib().oracle_outgoing_bidx(_p(rays_o), _p(rays_d), _p(corners), _p(sizes), _p(order), _p(isect), _p(ids), _p(w),
                               ctypes.c_int(int(skip)), ctypes.c_int(B), ctypes.c_int(nb))
    return ids, w
