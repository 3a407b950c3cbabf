"""Seeded synthetic inputs shared by the tests (and by bench.py)."""
import numpy as np
import torch


def camera_rig(n_cam, H, W, gen, center=(10.0, 3.0, 15.0), radius=6.0, fx=600.0):
    """Cameras on a ring looking at `center`.  Returns Ks [N,3,3], c2w [N,3,4] (float32)."""
    ang = torch.linspace(0, 2 * np.pi, n_cam + 1)[:-1] + 0.1 * torch.rand(n_cam, generator=gen)
    c = torch.tensor(center)
    pos = torch.stack([c[0] + radius * torch.cos(ang), c[1] + 0.5 * torch.rand(n_cam, generator=gen),
                       c[2] + radius * torch.sin(ang)], -1)
    fwd = torch.nn.functional.normalize(c[None] - pos + 0.3 * torch.randn(n_cam, 3, generator=gen), dim=-1)
    up = torch.tensor([0.0, 1.0, 0.0]).expand_as(fwd)
    right = torch.nn.functional.normalize(torch.cross(fwd, up, dim=-1), dim=-1)
    down = torch.cross(fwd, right, dim=-1)
    R = torch.stack([right, down, fwd], -1)          # columns = camera axes in world
    c2w = torch.cat([R, pos[..., None]], -1).float()
    K = torch.tensor([[fx, 0, W / 2.0], [0, fx, H / 2.0], [0, 0, 1.0]]).expand(n_cam, 3, 3).contiguous()
    return K.float(), c2w


def random_rays(B, gen, corner, size, inside=True):
    """Ray origins in/around the box and random directions (some axis-parallel, some zero components)."""
    corner, size = torch.as_tensor(corner, dtype=torch.float32), torch.as_tensor(size, dtype=torch.float32)
    u = torch.rand(B, 3, generator=gen)
    o = corner + size * (u if inside else (u * 2.0 - 0.5))
    d = torch.randn(B, 3, generator=gen)
    k = max(B // 16, 1)
    d[:k, 0] = 0.0                      # exercise safe_divide
    d[k:2 * k, 1] = 0.0
    d[2 * k:3 * k] = torch.tensor([0.0, 0.0, 1.0])
    d = d * (0.5 + torch.rand(B, 1, generator=gen))      # not normalised
    return o.contiguous(), d.contiguous()


def occupancy(log2dim, gen, p=0.3):
    shape = [2 ** int(v) for v in log2dim]
    return torch.rand(shape, generator=gen) < p


def tracing_layout(gen):
    """Four renderer tiles (foreground boxes, corner + size) along x with one grid resolution each, so that the grid
    offsets are uneven: 0 and 1 overlap on x in [6, 8], 1 and 2 share the face x = 14, and 3 lies beyond a gap
    (x in [22, 26]).  Occupancy: tile 1 all set, tile 2 all empty, tiles 0 and 3 about 45 % random.  Returns
    corners [4,3], sizes [4,3], log2dim [4,3] (int32), the concatenated grids (bool), their starts (int64)."""
    corners = torch.tensor([[0.0, 0.0, 0.0], [6.0, 0.0, 2.0], [14.0, 0.0, 2.0], [26.0, 0.0, -1.0]])
    sizes = torch.tensor([[8.0, 6.0, 8.0], [8.0, 6.0, 8.0], [8.0, 6.0, 8.0], [8.0, 6.0, 12.0]])
    log2dim = torch.tensor([[3, 2, 3], [4, 2, 3], [3, 3, 4], [2, 2, 2]], dtype=torch.int32)
    grids = [occupancy(l, gen, p=0.45).reshape(-1) for l in log2dim]
    grids[1][:] = True
    grids[2][:] = False
    n = [int(g.numel()) for g in grids]
    return corners, sizes, log2dim, torch.cat(grids), torch.tensor(np.cumsum([0] + n)[:-1], dtype=torch.int64)


def write_proxy_mesh_ply(path, corner, size, seed=0, n_boxes=20, ground_res=64):
    """Procedural proxy mesh for a tile: a gently rolling heightfield ground over the tile
    footprint (y is up, ground near the tile floor) plus `n_boxes` axis-aligned boxes standing
    on it.  Written as binary little-endian PLY: vertex float32 x,y,z; face uchar-counted int32
    vertex_indices -- the layout the reference's reader accepts (fastMesh/include/plyIO.h:215-278).
    Returns (verts [V,3] float32, faces [F,3] int32)."""
    rng = np.random.RandomState(seed)
    corner, size = np.asarray(corner, np.float32), np.asarray(size, np.float32)
    n = ground_res
    gx, gz = np.meshgrid(np.linspace(0, 1, n), np.linspace(0, 1, n), indexing="ij")
    gy = 0.05 + 0.03 * np.sin(6.0 * gx) * np.cos(5.0 * gz)
    verts = [np.stack([corner[0] + gx * size[0], corner[1] + gy * size[1], corner[2] + gz * size[2]], -1).reshape(-1, 3)]
    idx = np.arange(n * n).reshape(n, n)
    a, b, c, d = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[:-1, 1:].ravel(), idx[1:, 1:].ravel()
    faces = [np.stack([a, b, c], -1), np.stack([b, d, c], -1)]
    base = n * n
    cube_f = np.array([[0, 1, 2], [1, 3, 2], [4, 6, 5], [5, 6, 7], [0, 4, 1], [1, 4, 5],
                       [2, 3, 6], [3, 7, 6], [0, 2, 4], [2, 6, 4], [1, 5, 3], [3, 5, 7]])
    for _ in range(n_boxes):
        c0 = corner + size * np.array([rng.uniform(0.1, 0.8), 0.05, rng.uniform(0.1, 0.8)], np.float32)
        ext = size * np.array([rng.uniform(0.03, 0.12), rng.uniform(0.1, 0.6), rng.uniform(0.03, 0.12)], np.float32)
        cv = np.array([[i, j, k] for i in (0, 1) for j in (0, 1) for k in (0, 1)], np.float32) * ext + c0
        verts.append(cv)
        faces.append(cube_f + base)
        base += 8
    V = np.concatenate(verts).astype(np.float32)
    F = np.concatenate(faces).astype(np.int32)
    with open(path, "wb") as f:
        f.write((f"ply\nformat binary_little_endian 1.0\nelement vertex {len(V)}\nproperty float x\nproperty float y\n"
                 f"property float z\nelement face {len(F)}\nproperty list uchar int vertex_indices\nend_header\n").encode())
        f.write(V.tobytes())
        rec = np.zeros(len(F), dtype=[("n", "u1"), ("i", "<i4", 3)])
        rec["n"], rec["i"] = 3, F
        f.write(rec.tobytes())
    return V, F
