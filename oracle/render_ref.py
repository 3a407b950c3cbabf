"""TEST INFRASTRUCTURE ONLY (imported by tests/, never by the product path).

numpy restatement of the reference's multi-tile render stages and of the fastMesh queries -- small,
loop-based (seconds for a few hundred rays), each function citing the reference it follows:
  ray_block_intersection   hashgrid/src/rendering_kernel.cu:126-153  (RayAABBIntersection: hashgrid/include/cuda_utils.h:564-613)
  prepare_points           :391-431
  accumulate_color         :623-674
  inverse_z_sampling       :815-851  (inverse_z_sample_bound: cuda_utils.h:61-75)
  update_outgoing_bidx     :1262-1373
  get_last_block           :1211-1241
  sample_points            :178-382   (cell walk: dda.h:206-268)
  ray_firsthit_block       :704-812
  process_occupied_grid    :1478-1565
  fastMesh build           fastMesh/include/tile_structure.h:13-106
  fastMesh fisrtHit        fastMesh/src/fastMesh_kernel.cu:230-329 (+ dda.h:7-131, cuda_utils.h:403-436)
The loop forms of the sampler, first hit, dilation and exit tiles check their C restatements (oracle/native.py), which
serve frame-sized batches; the simple stages also have vectorised forms for those (prepare_points_vec, inverse_z_vec,
get_last_block_vec, inside_bidx, accumulate64).
Parity: pinned on the GPU box against the rebuilt reference extensions (oracle/_ref/HASHGRID.so,
fastMesh.so) by tests/test_render_gpu.py / tests/test_mesh_gpu.py; the reference holds no golden
vectors for these ops.  The sampler / fused evaluation stages are covered by oracle/native.py
(occupancy walk, hash encode) and oracle/torch_ref.py (decoder).
"""
import numpy as np

f32 = np.float32
MISS = f32(1e7)


def _safe_div(a, b):
    return f32(a) / f32(b) if b != 0 else f32(1e8)


def ray_aabb(o, d, center, half):
    """cuda_utils.h:564-613 -> (near, far) or (-1, -1); near clamps at 0, far starts at 1e5."""
    lo_acc, hi_acc = f32(0), f32(100000.0)
    for a in range(3):
        inv = _safe_div(1.0, d[a])
        lo, hi = f32(f32(center[a] - half[a] - o[a]) * inv), f32(f32(center[a] + half[a] - o[a]) * inv)
        if hi < lo:
            lo, hi = hi, lo
        if hi < lo_acc or lo > hi_acc:
            return f32(-1), f32(-1)
        lo_acc, hi_acc = max(lo_acc, lo), min(hi_acc, hi)
        if lo_acc > hi_acc:
            return f32(-1), f32(-1)
    return lo_acc, hi_acc


def ray_block_intersection(rays_o, rays_d, corners, sizes):
    B, nb = rays_o.shape[0], corners.shape[0]
    out = np.full((B, nb, 2), MISS, f32)
    for b in range(nb):
        half = (sizes[b] * f32(0.5)).astype(f32)
        center = (corners[b] + half).astype(f32)
        for i in range(B):
            n, fr = ray_aabb(rays_o[i], rays_d[i], center, half)
            if n != -1:
                out[i, b] = (n, fr)
    return out


def prepare_points(z_vals, running, intersections):
    B, S = z_vals.shape
    nb = intersections.shape[1]
    out = np.full((B, S, 4), -1, np.int16)
    for i in range(B):
        if not running[i]:
            continue
        for k in range(S):
            z = z_vals[i, k]
            if z == -1:
                continue
            idx = 0
            for b in range(nb):
                if intersections[i, b, 0] <= z <= intersections[i, b, 1] and idx < 4:
                    out[i, k, idx] = b
                    idx += 1
    return out


def accumulate_color(pts_diffuse, pts_specular, pts_alpha, transparency, z_vals, diffuse, specular, depth):
    T, dif, spe, dep = transparency.copy(), diffuse.copy(), specular.copy(), depth.copy()
    B, S = z_vals.shape
    for i in range(B):
        t = f32(T[i, 0])
        if t < 1e-5:
            continue
        for k in range(S):
            a = f32(pts_alpha[i, k, 0])
            dif[i] += t * pts_diffuse[i, k]
            spe[i] += t * pts_specular[i, k]
            dep[i, 0] += t * a * z_vals[i, k]
            t = f32(t * (1 - a))
        T[i, 0] = t
    return T, dif, spe, dep


def inverse_z_sampling(intersections, related_bidx, S, sample_range, fill=-1.0):
    B = intersections.shape[0]
    z = np.full((B, S), fill, f32)
    for i in range(B):
        b = int(related_bidx[i])
        if b == -1 or intersections[i, b, 0] == MISS:
            continue
        near = f32(intersections[i, b, 1])
        far = f32(near + f32(sample_range))
        inv_near, inv_far = f32(1) / near, f32(1) / far
        inv_bound, step = f32(inv_far - inv_near), f32(1) / f32(S - 1)
        for k in range(S):
            z[i, k] = f32(1) / f32(f32(f32(step * f32(k)) * inv_bound) + inv_near)
    return z


def get_last_block(tracing_blocks, intersections):
    B, nb = tracing_blocks.shape
    out = np.full(B, -1, np.int32)
    for i in range(B):
        for s in range(nb):
            b = tracing_blocks[i, s]
            if intersections[i, b, 0] == MISS:
                break
            out[i] = b
    return out


def update_outgoing_bidx(rays_o, rays_d, corners, sizes, tracing_blocks, intersections, skip=False):
    B, nb = tracing_blocks.shape
    ids, w = np.full((B, 4), -1, np.int16), np.zeros((B, 4), f32)
    for i in range(B):
        far, cur = f32(-1), []
        for s in range(nb):
            b = int(tracing_blocks[i, s])
            n, fr = intersections[i, b]
            if n == MISS:
                break
            if not skip and (n > far and far != -1):
                break
            if fr > far:
                far, cur = fr, [b]
            elif fr == far and len(cur) < 4:
                cur.append(b)
        if far == -1:
            continue
        if len(cur) == 1:
            ids[i, 0], w[i, 0] = cur[0], 1.0
            continue
        p = (rays_o[i] + far * rays_d[i]).astype(f32)
        for k, b in enumerate(cur):
            q = np.clip((p - corners[b]) / sizes[b], 0, 1).astype(f32)
            dis = ((f32(0.5) - np.abs(q - f32(0.5))) * sizes[b]).astype(f32)
            if dis[0] != 0 and dis[2] != 0:
                w[i, k] = dis[0] * dis[2]
            elif dis[0] != 0:
                w[i, k] = dis[0]
            elif dis[2] != 0:
                w[i, k] = dis[2]
            ids[i, k] = b
    return ids, w


def _fma(a, b, c):
    """float32 a * b + c with one rounding (the product of two float32 is exact in float64)."""
    return f32(np.float64(a) * np.float64(b) + np.float64(c))


class _Walk:
    """dda.h:206-268 (DDASatateScene_v2) in the tile's local frame: start cell clamped into the grid, tie rule x if
    (tx < ty and tx <= tz), y if (ty < tz and ty <= tx), else z."""

    def __init__(self, o, d, t0, n, cell):
        p = [_fma(t0, d[a], o[a]) for a in range(3)]
        self.n, self.c = n, [min(max(int(p[a] / cell[a]), 0), n[a] - 1) for a in range(3)]
        self.s = [1 if d[a] >= 0 else -1 for a in range(3)]
        self.tmax, self.tdel = [], []
        for a in range(3):
            nxt = f32(f32(self.c[a] + self.s[a]) * cell[a])
            if self.s[a] < 0:
                nxt = f32(nxt + cell[a])
            self.tmax.append(f32(max(_safe_div(f32(nxt - p[a]), d[a]), f32(0)) + t0))
            self.tdel.append(abs(_safe_div(cell[a], d[a])))
        self.t0 = f32(t0)

    def cells(self):
        """Yields (cell, t0, t1) until the walk leaves the grid."""
        while not (any(c < 0 or c >= n for c, n in zip(self.c, self.n)) or all(t <= 0 for t in self.tmax)):
            tm = self.tmax
            m = [tm[0] < tm[1] and tm[0] <= tm[2], tm[1] < tm[2] and tm[1] <= tm[0]]
            m.append(not (m[0] or m[1]))
            t1 = tm[m.index(True)]
            yield tuple(self.c), self.t0, t1
            self.t0 = t1
            for a in range(3):
                if m[a]:
                    self.tmax[a] = f32(self.tmax[a] + self.tdel[a])
                    self.c[a] += self.s[a]


def _tile(corners, sizes, occupied, starts, log2dim, b):
    n = [1 << int(v) for v in log2dim[b]]
    cell = [f32(sizes[b][a] / f32(n[a])) for a in range(3)]
    ly, lz = int(log2dim[b][1]), int(log2dim[b][2])
    occ = occupied[int(starts[b]):]
    return n, cell, lambda c: bool(occ[(c[0] << (ly + lz)) | (c[1] << lz) | c[2]])


def sample_points(rays_o, rays_d, corners, sizes, occupied, starts, log2dim, tracing_blocks, intersections, tracing_idx, z_start,
                  S, fill=-1.0):
    """rendering_kernel.cu:178-382, one call: each ray goes on through its tiles (near to far) from tracing_idx and
    samples the first with occupied segments beyond z_start, S samples over the segments, (int)(len / total * S) each
    and the rest on the last; the walk starts at near on the first tile and at z_start (previous far) after it.
    Returns (tracing_idx, z_start, z_vals, dists)."""
    B, nb = tracing_blocks.shape
    ti, zs = np.array(tracing_idx, np.int32).copy(), np.array(z_start, f32).copy()
    z, dist = np.full((B, S), fill, f32), np.full((B, S), fill, f32)
    for i in range(B):
        step, t = int(ti[i]), f32(zs[i])
        while step < nb:
            b = int(tracing_blocks[i, step])
            near, far = intersections[i, b]
            if near == MISS:
                break
            if t >= far:
                step += 1
                continue
            if step == 0:
                t = near
            n, cell, on = _tile(corners, sizes, occupied, starts, log2dim, b)
            o = (rays_o[i] - corners[b]).astype(f32)
            segs = [(t0, t1) for c, t0, t1 in _Walk(o, rays_d[i], t, n, cell).cells() if on(c) and f32(t1 - t0) > 0]
            if not segs:
                t, step = far, step + 1
                continue
            total = f32(0)
            for t0, t1 in segs:
                total = f32(total + f32(t1 - t0))
            num = 0
            for k, (t0, t1) in enumerate(segs):
                cnt = min(max(int(f32(f32(f32(t1 - t0) / total) * f32(S))), 1), S - num)
                if k == len(segs) - 1:
                    cnt = S - num
                if cnt > 0:
                    interval = f32(f32(t1 - t0) / f32(cnt))
                    for j in range(cnt):
                        z[i, num + j], dist[i, num + j] = _fma(j, interval, t0), interval
                num += cnt
            t, step = far, step + 1
            break
        ti[i], zs[i] = step, t
    return ti, zs, z, dist


def ray_firsthit_block(rays_o, rays_d, corners, sizes, occupied, starts, log2dim, tracing_blocks, intersections):
    """rendering_kernel.cu:704-812: of the tiles whose walk over [near, far] meets an occupied cell, the one with the
    nearest far; else the last tile the ray enters; -1 for a ray that enters none."""
    B, nb = tracing_blocks.shape
    hit = np.full(B, -1, np.int16)
    for i in range(B):
        dis, last = MISS, -1
        for s in range(nb):
            b = int(tracing_blocks[i, s])
            near, far = intersections[i, b]
            if near == MISS:
                break
            n, cell, on = _tile(corners, sizes, occupied, starts, log2dim, b)
            o = (rays_o[i] - corners[b]).astype(f32)
            if any(on(c) for c, _, _ in _Walk(o, rays_d[i], near, n, cell).cells()) and dis > far:
                hit[i], dis = b, far
            last = b
        if last != -1 and hit[i] == -1:
            hit[i] = last
    return hit


def process_occupied_grid(bidx, corners, sizes, occupied, starts, log2dim, target):
    """rendering_kernel.cu:1478-1565: every occupied cell of tile bidx sets, in each other tile, the cells that hold one
    of its eight corners (a corner at q in [0, 1)^3 of that tile).  Returns the updated copy of `target`."""
    tgt = np.array(target, np.uint8).copy()
    n, cell, on = _tile(corners, sizes, occupied, starts, log2dim, bidx)
    for x in range(n[0]):
        for y in range(n[1]):
            for z in range(n[2]):
                if not on((x, y, z)):
                    continue
                p0 = [_fma(v, cell[a], corners[bidx][a]) for a, v in enumerate((x, y, z))]
                for b in range(corners.shape[0]):
                    if b == bidx:
                        continue
                    l2 = [int(v) for v in log2dim[b]]
                    for j in range(8):
                        v = ((j >> 2) & 1, (j >> 1) & 1, j & 1)
                        q = [f32(f32(f32(p0[a] + f32(v[a] * cell[a])) - corners[b][a]) / sizes[b][a]) for a in range(3)]
                        if all(0 <= qa < 1 for qa in q):
                            c = [int(f32(q[a] * f32(1 << l2[a]))) for a in range(3)]
                            tgt[int(starts[b]) + ((c[0] << (l2[1] + l2[2])) | (c[1] << l2[2]) | c[2])] = 1
    return tgt


# ------------------------------------------------------------------------------------------------ vectorised, frame-sized
# The same stages over whole arrays, for batches of millions of rays (the loop forms above take seconds per few hundred).

def prepare_points_vec(z_vals, running, intersections):
    """prepare_points: the first four tiles (in index order) whose [near, far] holds each sample of a running ray."""
    B, S = z_vals.shape
    out = np.full((B, S, 4), -1, np.int16)
    rows = np.nonzero(np.asarray(running, bool).reshape(-1) & (z_vals != -1).any(-1))[0]
    z, it = z_vals[rows], intersections[rows]
    sub, cnt = out[rows], np.zeros(z.shape, np.int64)
    for b in range(intersections.shape[1]):
        m = (z != -1) & (z >= it[:, b, 0, None]) & (z <= it[:, b, 1, None]) & (cnt < 4)
        r, k = np.nonzero(m)
        sub[r, k, cnt[r, k]] = b
        cnt += m
    out[rows] = sub
    return out


def inverse_z_vec(intersections, related_bidx, S, sample_range, z_vals):
    """inverse_z_sampling into a copy of z_vals: S samples in inverse depth from the exit of tile related_bidx[i] to
    exit + sample_range, 1 / fma(step * k, 1/far - 1/near, 1/near); rows of -1 tiles or misses keep z_vals."""
    z = np.array(z_vals, f32).copy()
    b = np.asarray(related_bidx).astype(np.int64)
    rows = np.nonzero(b != -1)[0]
    bound = intersections[rows, b[rows]]
    rows, bound = rows[bound[:, 0] != MISS], bound[bound[:, 0] != MISS]
    near = bound[:, 1].astype(f32)
    sk = (f32(1) / f32(S - 1)) * np.arange(S, dtype=f32)
    with np.errstate(divide="ignore", invalid="ignore"):          # exits at depth 0 give inf / NaN, as in the kernel
        inv_near, inv_far = f32(1) / near, f32(1) / (near + f32(sample_range))
        inv_bound = (inv_far - inv_near).astype(f32)
        z[rows] = f32(1) / (sk[None, :].astype(np.float64) * inv_bound[:, None] + inv_near[:, None]).astype(f32)
    return z


def get_last_block_vec(tracing_blocks, intersections):
    """get_last_block: the last tile of the order before the first miss, -1 if the first is a miss."""
    B, nb = tracing_blocks.shape
    hit = np.take_along_axis(intersections[..., 0], tracing_blocks.astype(np.int64), 1) != MISS
    n = np.where(hit.all(-1), nb, np.argmin(hit, -1))
    return np.where(n > 0, tracing_blocks[np.arange(B), np.maximum(n - 1, 0)], -1).astype(np.int32)


def inside_bidx(rays_o, corners, sizes, ids, w):
    """update_outgoing_bidx_v2 (rendering_kernel.cu:1405-1472) into copies of ids / w: the first four tiles (in index
    order) that contain the ray origin, weight = product of the distances to the faces on all three axes."""
    ids, w = np.array(ids).copy(), np.array(w, f32).copy()
    cnt = np.zeros(rays_o.shape[0], np.int64)
    for b in range(corners.shape[0]):
        loc = ((rays_o - corners[b]) / sizes[b]).astype(f32)
        r = np.nonzero(((loc >= 0) & (loc <= 1)).all(-1) & (cnt < 4))[0]
        dis = ((f32(0.5) - np.abs(loc[r] - f32(0.5))) * sizes[b]).astype(f32)
        ids[r, cnt[r]] = b
        w[r, cnt[r]] = (dis[:, 0] * dis[:, 1]).astype(f32) * dis[:, 2]
        cnt[r] += 1
    return ids, w


def accumulate64(pts_diffuse, pts_specular, pts_alpha, transparency, z_vals, diffuse, specular, depth):
    """accumulate_color in float64: front to back, T carried across calls, rays entering with T < 1e-5 untouched.
    Returns (T [B], diffuse [B,3], specular [B,3], depth [B])."""
    T = np.array(transparency, np.float64).reshape(-1)
    dif, spe, dep = np.array(diffuse, np.float64), np.array(specular, np.float64), np.array(depth, np.float64).reshape(-1)
    go = T >= 1e-5
    t, a = T[go], np.asarray(pts_alpha, np.float64).reshape(T.shape[0], -1)[go]
    pd, ps, z = np.asarray(pts_diffuse, np.float64)[go], np.asarray(pts_specular, np.float64)[go], np.asarray(z_vals, np.float64)[go]
    d_, s_, z_ = dif[go], spe[go], dep[go]
    for k in range(a.shape[1]):
        d_ += t[:, None] * pd[:, k]
        s_ += t[:, None] * ps[:, k]
        z_ += t * a[:, k] * z[:, k]
        t = t * (1 - a[:, k])
    T[go], dif[go], spe[go], dep[go] = t, d_, s_, z_
    return T, dif, spe, dep


# ------------------------------------------------------------------------------------------------ fastMesh
def mesh_build(verts, faces, side=64):
    """tile_structure.h:13-106: cubic grid anchored at the vertex AABB minimum, cell = max extent / 64; a face is
    listed in every cell its AABB overlaps.  Returns (origin, cell, {cell index -> [face ids]})."""
    verts = np.asarray(verts, f32)
    mn, mx = verts.min(0), verts.max(0)
    cell = f32((mx - mn).max() / f32(side))
    inv = f32(1) / cell
    lists = {}
    smax = mn + f32(side) * cell
    for fi, f in enumerate(np.asarray(faces)):
        tri = verts[f]
        lo, hi = tri.min(0), tri.max(0)
        ctr, half = (lo + hi) * f32(0.5), (hi - lo) * f32(0.5)
        lo, hi = ctr - half, ctr + half
        if (hi <= mn).any() or (lo >= smax).any():
            continue
        i0 = np.clip(((lo - mn) * inv).astype(np.int64), 0, side - 1)
        i1 = np.clip(((hi - mn) * inv).astype(np.int64), 0, side - 1)
        for x in range(i0[0], i1[0] + 1):
            for y in range(i0[1], i1[1] + 1):
                for z in range(i0[2], i1[2] + 1):
                    lists.setdefault((x << 12) | (y << 6) | z, []).append(fi)
    return mn.astype(f32), cell, lists


def _ray_triangle(o, d, v0, v1, v2):
    """cuda_utils.h:403-436: Moeller-Trumbore with back-face rejection (det < 1e-8)."""
    e1, e2, s = v1 - v0, v2 - v0, o - v0
    p = np.cross(d, e2)
    det = f32(np.dot(e1, p))
    if det < 1e-8:
        return f32(-1e8)
    det = f32(1) / det
    u = f32(np.dot(s, p)) * det
    if u < 0 or u > 1:
        return f32(-1e8)
    q = np.cross(s, e1)
    v = f32(np.dot(d, q)) * det
    if v < 0 or v > 1 or u + v < 0 or u + v > 1:
        return f32(-1e8)
    return f32(np.dot(e2, q)) * det


def mesh_first_hit(mesh, verts, faces, o, d, side=64, max_steps=4096):
    """fastMesh_kernel.cu:230-295: walk the cells from the origin (index space, cell size 1); in each listed cell test
    all its faces two-sided; return the nearest t > 0 of the FIRST cell that has any hit, 0 if none."""
    origin, cell, lists = mesh
    verts = np.asarray(verts, f32)
    inv = f32(1) / cell
    p = ((np.asarray(o, f32) - origin) * inv).astype(f32)
    d = np.asarray(d, f32)
    c = np.clip(p.astype(np.int64), 0, side - 1)
    step = np.where(d >= 0, 1, -1)
    nxt = (c + step).astype(f32) + (step < 0)
    tmax = np.array([max(_safe_div(nxt[a] - p[a], d[a]), f32(0)) for a in range(3)], f32)
    tdel = np.array([abs(_safe_div(1.0, d[a])) for a in range(3)], f32)
    for _ in range(max_steps):
        if (c < 0).any() or (c >= side).any() or (tmax <= 0).all():
            break
        mx = tmax[0] < tmax[1] and tmax[0] <= tmax[2]
        my = tmax[1] < tmax[2] and tmax[1] <= tmax[0]
        mz = tmax[2] < tmax[0] and tmax[2] <= tmax[1]
        if not (mx or my or mz):
            mz = True
        key = (int(c[0]) << 12) | (int(c[1]) << 6) | int(c[2])
        if key in lists:
            best = f32(1e8)
            for fi in lists[key]:
                A, B_, C = verts[faces[fi][0]], verts[faces[fi][1]], verts[faces[fi][2]]
                n = np.cross(B_ - A, C - B_)
                t = _ray_triangle(o, d, A, C, B_) if np.dot(d, n) > 0 else _ray_triangle(o, d, A, B_, C)
                if 0 < t < best:
                    best = t
            if best != f32(1e8):
                return best
        a = 0 if mx else (1 if my else 2)
        tmax[a] += tdel[a]
        c[a] += step[a]
    return f32(0)
