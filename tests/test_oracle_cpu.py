"""CPU: properties of the oracle itself (it is the checker, so it gets checked)."""
import numpy as np
import torch

from oracle import native as on
import scenes


def _ladder(base, fin, L=16):
    b = np.exp((np.log(fin) - np.log(base)) / (L - 1))
    return np.stack([(base * b ** i) for i in range(L)]).astype(np.int32)


def test_hash_encode_matches_numpy_restatement():
    """Independent numpy restatement of the hash + trilinear blend (different code
    path from the C oracle) agrees with it, indices bit-exact."""
    rng = np.random.default_rng(0)
    L, T, B = 16, 2 ** 14, 500
    table = rng.standard_normal((L, T, 2)).astype(np.float32)
    res = _ladder(np.array([16., 16., 16.]), np.array([512., 512., 512.]))
    pts = rng.uniform(-2, 2, (B, 3)).astype(np.float32)
    out, idx = on.hash_encode_fwd(pts, table, res, want_idx=True)
    u = (pts + np.float32(2.0)) * np.float32(0.25)
    for l in (0, 7, 15):
        v = u * (res[l] - 1).astype(np.float32)
        i = v.astype(np.int32)
        w = v - i.astype(np.float32)
        acc = np.zeros((B, 2), np.float64)
        for c in range(8):
            dx, dy, dz = (c >> 2) & 1, (c >> 1) & 1, c & 1
            h = ((i[:, 0] + dx).astype(np.uint32) * np.uint32(1)) ^ ((i[:, 1] + dy).astype(np.uint32) * np.uint32(2654435761)) \
                ^ ((i[:, 2] + dz).astype(np.uint32) * np.uint32(805459861))
            h &= np.uint32(T - 1)
            assert np.array_equal(h, idx[:, l, c])
            wc = (w[:, 0] if dx else 1 - w[:, 0]) * (w[:, 1] if dy else 1 - w[:, 1]) * (w[:, 2] if dz else 1 - w[:, 2])
            acc += wc[:, None].astype(np.float64) * table[l][h]
        assert np.abs(acc - out[:, l]).max() < 1e-5


def test_hash_backward_is_adjoint_of_forward():
    """<out(table), g> is linear in table: grad_table must reproduce it exactly (fp64 check),
    and grad_points matches a central finite difference."""
    rng = np.random.default_rng(1)
    L, T, B = 16, 2 ** 10, 300
    table = rng.standard_normal((L, T, 2)).astype(np.float32)
    res = _ladder(np.array([16., 16., 16.]), np.array([256., 256., 256.]))
    pts = rng.uniform(-1.9, 1.9, (B, 3)).astype(np.float32)
    g = rng.standard_normal((B, L, 2)).astype(np.float32)
    out = on.hash_encode_fwd(pts, table, res)
    gp, gt = on.hash_encode_bwd(pts, g, table, res)
    lhs = float((out.astype(np.float64) * g).sum())
    rhs = float((gt.astype(np.float64) * table).sum())
    assert abs(lhs - rhs) <= 1e-4 * abs(lhs)
    # bbox variant: same cell structure when the box is [-2,2]^3 scaled
    corner, size = np.array([-2, -2, -2], np.float32), np.array([4, 4, 4], np.float32)
    out_b = on.hash_encode_fwd(pts, table, res, corner, size)
    assert np.abs(out_b - out).max() < 5e-4      # same grid, different fp32 prologue


def test_sampler_properties():
    g = torch.Generator().manual_seed(0)
    corner, size = np.zeros(3, np.float32), np.array([20, 13, 30], np.float32)
    o, d = scenes.random_rays(2000, g, corner, size)
    log2dim = [4, 3, 4]
    occ = scenes.occupancy(log2dim, g, p=0.4).numpy()
    S = 64
    z, di, cnt = on.sample_points_grid(o.numpy(), d.numpy(), corner, size, occ, log2dim, S)
    hit = cnt > 0
    assert hit.any() and (~hit).any()
    assert np.all(z[~hit] == -1) and np.all(di[~hit] == -1)
    zz, dd = z[hit], di[hit]
    assert np.all(zz != -1), "a ray with any occupied segment receives all S samples"
    assert np.all(np.diff(zz, axis=1) >= -1e-4), "z sorted along the ray"
    assert np.all(dd > 0)
    # all-empty grid: nothing written; all-full grid: samples cover [near, far)
    z0, _, c0 = on.sample_points_grid(o.numpy(), d.numpy(), corner, size, np.zeros_like(occ), log2dim, S)
    assert np.all(z0 == -1) and np.all(c0 == 0)
    z1, d1, c1 = on.sample_points_grid(o.numpy(), d.numpy(), corner, size, np.ones_like(occ), log2dim, S)
    b = on.ray_aabb(o.numpy(), d.numpy(), corner + size / 2, size)[:, 0]
    ok = c1 > 0
    assert np.allclose((d1[ok]).sum(1), (b[ok, 1] - b[ok, 0]), rtol=2e-3, atol=1e-3)


def test_ray_backward_is_adjoint():
    rng = np.random.default_rng(2)
    N, B = 4, 64
    K = np.tile(np.array([600, 0, 480, 0, 600, 270, 0, 0, 1], np.float32), (N, 1))
    C = rng.standard_normal((N, 12)).astype(np.float32)
    locs = np.stack([rng.integers(0, N, B), rng.integers(0, 960, B), rng.integers(0, 540, B)], -1).astype(np.int32)
    go, gd = rng.standard_normal((B, 3)).astype(np.float32), rng.standard_normal((B, 3)).astype(np.float32)
    o, d = on.compute_ray_fwd(K, C, locs)
    g = on.compute_ray_bwd(go, gd, K, locs, N)
    lhs = float((o.astype(np.float64) * go).sum() + (d.astype(np.float64) * gd).sum())
    rhs = float((g.astype(np.float64) * C).sum())       # forward is linear in C2W
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), 1.0)


def test_render_oracle_invariants():
    """oracle/render_ref.py sanity on the CPU: inverse-z samples start at the tile exit, front-to-back accumulation
    conserves T + sum of alpha T, the cell walk finds a triangle placed in front of the ray."""
    from oracle import render_ref as rr
    isect = np.array([[[1.0, 4.0], [1e7, 1e7]]], np.float32)
    z = rr.inverse_z_sampling(isect, np.array([0], np.int16), 8, 1e6)
    assert abs(z[0, 0] - 4.0) < 1e-5 and np.all(np.diff(z[0]) > 0) and abs(z[0, -1] - (4.0 + 1e6)) / 1e6 < 1e-2      # fp32: 1 / (1e-6-sized reciprocal)
    assert np.all(rr.inverse_z_sampling(isect, np.array([-1], np.int16), 8, 1e6) == -1)
    rng = np.random.RandomState(0)
    a = rng.rand(3, 9, 1).astype(np.float32) * 0.5
    ones = np.ones((3, 9, 3), np.float32)
    T, dif, _, _ = rr.accumulate_color(a * ones, a * ones, a, np.ones((3, 1), np.float32), np.ones((3, 9), np.float32),
                                       np.zeros((3, 3), np.float32), np.zeros((3, 3), np.float32), np.zeros((3, 1), np.float32))
    assert np.allclose(dif[:, 0] + T[:, 0], 1.0, atol=1e-5)          # sum_k alpha_k T_k + T_end = 1
    V = np.array([[0, 0, 1], [4, 0, 1], [0, 4, 1], [4, 4, 1], [0, 0, 0], [4, 4, 4]], np.float32)
    F = np.array([[0, 1, 2], [1, 3, 2]], np.int32)                     # a quad in the z = 1 plane (faces ON the AABB minimum are skipped by the build, as in the reference)
    mesh = rr.mesh_build(V, F)
    t = rr.mesh_first_hit(mesh, V, F, np.array([1.0, 1.0, 3.0], np.float32), np.array([0.0, 0.0, -1.0], np.float32))
    assert abs(t - 2.0) < 1e-4
    assert rr.mesh_first_hit(mesh, V, F, np.array([1.0, 1.0, 3.0], np.float32), np.array([0.0, 0.0, 1.0], np.float32)) == 0
    ids, w = rr.update_outgoing_bidx(np.zeros((1, 3), np.float32), np.array([[1.0, 0, 0]], np.float32), np.zeros((2, 3), np.float32),
                                     np.ones((2, 3), np.float32), np.array([[0, 1]], np.int32), np.array([[[0, 2.0], [1.0, 3.0]]], np.float32))
    assert ids[0, 0] == 1 and w[0, 0] == 1.0


def test_tracing_restatements_agree():
    """The C restatements of the multi-tile render tracing stages (sampler, first hit, occupancy dilation, exit tiles)
    and the vectorised forms of the simple stages against the loop forms of oracle/render_ref.py, on the tiles of
    scenes.tracing_layout (overlap, shared face, gap, uneven grids) and a few hundred rays from inside, outside and
    beyond the tiles.  Tile ids and tracing state bit-exact; depths within 1e-6 relative."""
    from oracle import render_ref as rr
    g = torch.Generator().manual_seed(5)
    corners, sizes, l2d, occ, starts = (t.numpy() for t in scenes.tracing_layout(g))
    B, S, nb = 300, 16, 4
    o, d = scenes.random_rays(B, g, [-4.0, -1.0, -3.0], [40.0, 8.0, 16.0], inside=True)
    o, d = o.numpy(), d.numpy()
    isect = np.where(on.ray_aabb(o, d, corners + sizes / 2, sizes) == -1, np.float32(1e7), on.ray_aabb(o, d, corners + sizes / 2, sizes))
    assert np.array_equal(isect, rr.ray_block_intersection(o, d, corners, sizes))
    order = np.argsort(isect[..., 0], -1, kind="stable").astype(np.int32)
    assert (isect[..., 0] != 1e7).sum(-1).max() >= 3 and (isect[..., 0] == 1e7).all(-1).any()
    fake = occ.astype(np.uint8)
    for b in range(nb):
        got = on.process_occupied(b, int(2 ** l2d[b].sum()), corners, sizes, occ, starts, l2d, fake)
        want = rr.process_occupied_grid(b, corners, sizes, occ, starts, l2d, fake)
        assert np.array_equal(got, want), f"process_occupied tile {b}"
        fake = got
    assert fake[starts[2]:starts[3]].any() and (fake >= occ).all()
    ti, zs = np.zeros(B, np.int32), np.zeros(B, np.float32)
    for _ in range(nb):
        z, di = np.full((B, S), -1, np.float32), np.full((B, S), -1, np.float32)
        wti, wzs, wz, wdi = rr.sample_points(o, d, corners, sizes, fake, starts, l2d, order, isect, ti, zs, S)
        on.render_sample(o, d, corners, sizes, fake, starts, l2d, order, isect, ti, zs, z, di)
        assert np.array_equal(ti, wti) and np.array_equal(z == -1, wz == -1)
        for x, y in ((zs, wzs), (z, wz), (di, wdi)):
            assert np.allclose(x, y, rtol=1e-6, atol=0)
        running = ti < nb
        assert np.array_equal(rr.prepare_points_vec(z, running, isect), rr.prepare_points(z, running, isect))
    assert np.array_equal(ti, (isect[..., 0] != 1e7).sum(-1)), "after nb calls every ray stops at its first missed tile"
    assert np.array_equal(on.firsthit_block(o, d, corners, sizes, fake, starts, l2d, order, isect),
                          rr.ray_firsthit_block(o, d, corners, sizes, fake, starts, l2d, order, isect))
    assert np.array_equal(rr.get_last_block_vec(order, isect), rr.get_last_block(order, isect))
    ids, w = on.outgoing_bidx(o, d, corners, sizes, order, isect)
    wids, ww = rr.update_outgoing_bidx(o, d, corners, sizes, order, isect)
    assert np.array_equal(ids, wids) and np.allclose(w, ww, rtol=1e-4, atol=1e-5)      # the loop form rounds o + far d twice
    assert (ids[:, 1] >= 0).any()
    z = rr.inverse_z_vec(isect, ids[:, 0], 12, 1e6, np.full((B, 12), -1, np.float32))
    wz = rr.inverse_z_sampling(isect, ids[:, 0], 12, 1e6)
    assert np.array_equal(z == -1, wz == -1) and np.allclose(z, wz, rtol=1e-5)
    rng = np.random.default_rng(0)
    pd, ps, pa = rng.random((B, S, 3), np.float32), rng.random((B, S, 3), np.float32), rng.random((B, S, 1), np.float32) * 0.3
    init = [rng.random((B, 1), np.float32), rng.random((B, 3), np.float32), rng.random((B, 3), np.float32), rng.random((B, 1), np.float32)]
    init[0][::7] = 1e-6
    zz = np.repeat(z, 2, 1)[:, :S]
    for x, y in zip(rr.accumulate64(pd, ps, pa, init[0], zz, *init[1:]), rr.accumulate_color(pd, ps, pa, init[0], zz, *init[1:])):
        assert np.allclose(x.reshape(y.shape), y, rtol=1e-5, atol=1e-5)
