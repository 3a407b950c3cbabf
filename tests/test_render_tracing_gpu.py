"""GPU: the tracing stages of the multi-tile renderer (csrc/render.cu) and the frame driver render_frame.render_rays against
CPU restatements that share no code with them (oracle/scanerf_oracle.c, oracle/render_ref.py, the field restatement of
test_render_gpu), at the launch geometry of a 1920 x 1080 frame.

render.cu caps every grid at 32 blocks per SM, so a frame runs each grid-stride loop for several rounds (the sampler four on
148 SMs, the accumulation 28); every stage test first asserts the round count it claims from the SM count.  The scene
(scenes.tracing_layout) has four tiles with one grid resolution each: two overlap, two share a face, one lies beyond a gap;
one grid is all set, one all empty.  The rays come from a pinhole camera inside a tile and one outside (their centre column
and row have exactly zero direction components), from random origins around the tiles, and from beyond every tile.
Bars: tile ids, tracing state and occupancy grids bit-exact; depths and blend weights 1e-6 relative; accumulation 1e-5
against float64; the composited frame 1e-4 (colours, transparency) and 1e-4 relative (depth)."""
import numpy as np
import pytest
import torch

import scenes
from conftest import load_pkg
from oracle import native as on
from oracle import render_ref as rr
from test_render_gpu import field_restatement, make_scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MISS = np.float32(1e7)
W, H = 1920, 1080
B_FRAME, S = W * H, 32


def _ops():
    load_pkg()
    from hashgrid.lib import HASHGRID as ops
    import scanerf_b200_capi as capi
    return ops, int(capi.lib().snrf_device_sm_count())


def _rounds(n, threads, sms, per_block=None):
    """Grid-stride rounds of a render.cu launch over n items: grid1d caps the grid at sms * 32 blocks (the accumulation
    at sms * 64 blocks of 8 rays)."""
    per_round = sms * 64 * per_block if per_block else sms * 32 * threads
    return (n + per_round - 1) // per_round


def _tile_scene(tiles=(0, 1, 2, 3)):
    """scenes.tracing_layout with the tables, decoders and hash resolutions of make_scene, restricted to `tiles`."""
    corners, sizes, l2d, occ, starts = scenes.tracing_layout(torch.Generator().manual_seed(3))
    a, b = make_scene(3, seed=21), make_scene(3, seed=22)
    tables, params, res, mlps = torch.cat([a["tables"], b["tables"]]), torch.cat([a["params"], b["params"]]), torch.cat([a["res"], b["res"]]), a["mlps"] + b["mlps"]
    ix = list(tiles)
    n = [int(2 ** l2d[t].sum()) for t in ix]
    grids = [occ[int(starts[t]):int(starts[t]) + k] for t, k in zip(ix, n)]
    return dict(corners=corners[ix].contiguous(), sizes=sizes[ix].contiguous(), l2d=l2d[ix].contiguous(), occ=torch.cat(grids),
                starts=torch.tensor(np.cumsum([0] + n)[:-1], dtype=torch.int64), n=n, nb=len(ix), tables=tables[ix].contiguous(),
                params=params[ix].contiguous(), res=res[ix].contiguous(), mlps=[mlps[t] for t in ix], T=a["T"])


def _cameras(w, h):
    """Two axis-aligned pinhole cameras; the principal point is a pixel centre, so column w/2 and row h/2 have exactly zero
    x / y camera components.  One sits inside tile 0 looking along +x (through every tile), one outside looking along +z."""
    load_pkg()
    import render_frame as rf
    K = torch.tensor([[0.5 * w, 0.0, w / 2 + 0.5], [0.0, 0.5 * w, h / 2 + 0.5], [0.0, 0.0, 1.0]])
    inside = torch.tensor([[0.0, 0.0, 1.0, 3.3], [0.0, -1.0, 0.0, 2.7], [1.0, 0.0, 0.0, 4.1]])
    outside = torch.tensor([[1.0, 0.0, 0.0, 11.3], [0.0, -1.0, 0.0, 2.9], [0.0, 0.0, 1.0, -9.0]])
    return [rf.pinhole_rays(h, w, K, c2w, "cpu") for c2w in (inside, outside)]


def _rays(w, h, n_random, n_miss, seed):
    """Both cameras at w x h, n_random rays from around the tiles, n_miss rays beyond every tile pointing away."""
    g = torch.Generator().manual_seed(seed)
    cams = _cameras(w, h)
    o_r, d_r = scenes.random_rays(n_random, g, [-4.0, -1.0, -3.0], [40.0, 8.0, 16.0])
    o_m = torch.tensor([40.0, 3.0, 4.0]) + torch.rand(n_miss, 3, generator=g) * 5
    d_m = torch.nn.functional.normalize(torch.rand(n_miss, 3, generator=g) + torch.tensor([0.2, -0.5, -0.5]), dim=-1)
    o = torch.cat([cams[0][0], cams[1][0], o_r, o_m]).contiguous()
    d = torch.cat([cams[0][1], cams[1][1], d_r, d_m]).contiguous()
    return o, d


def _rel(x, y):
    """Largest |x - y| / |y| over the finite entries."""
    m = np.isfinite(y) & (y != 0)
    return float((np.abs(x[m].astype(np.float64) - y[m]) / np.abs(y[m])).max()) if m.any() else 0.0


def _isect(o, d, sc):
    c, s = sc["corners"].numpy(), sc["sizes"].numpy()
    t = on.ray_aabb(o, d, c + s / 2, s)
    return np.where(t == -1, MISS, t).astype(np.float32)


def _grid(ops, sc):
    """(GPU scene tensors, the dilated occupancy on the GPU, the C restatement's)."""
    g = {k: sc[k].to(DEV) for k in ("corners", "sizes", "l2d", "occ", "starts")}
    fake = g["occ"].clone()
    want = sc["occ"].numpy().astype(np.uint8)
    for b in range(sc["nb"]):
        ops.process_occupied_grid(b, sc["n"][b], g["corners"], g["sizes"], g["occ"], g["starts"], g["l2d"], fake)
        want = on.process_occupied(b, sc["n"][b], sc["corners"].numpy(), sc["sizes"].numpy(), sc["occ"].numpy(), sc["starts"].numpy(),
                                   sc["l2d"].numpy(), want)
    return g, fake, want


@pytest.fixture(scope="module")
def frame():
    """The scene, a frame of rays, their intersections and tracing order (both from the GPU), the dilated grid."""
    ops, sms = _ops()
    sc = _tile_scene()
    o, d = _rays(W // 2, H // 2, 3 * B_FRAME // 8, B_FRAME // 8, seed=1)
    assert o.shape[0] == B_FRAME
    od, dd = o.to(DEV), d.to(DEV)
    g, fake, fake_want = _grid(ops, sc)
    isect = torch.full((B_FRAME, sc["nb"], 2), float(MISS), device=DEV)
    ops.ray_block_intersection(od, dd, g["corners"], g["sizes"], isect)
    order = torch.argsort(isect[..., 0], dim=-1).int().contiguous()
    torch.cuda.synchronize()
    return dict(ops=ops, sms=sms, sc=sc, o=o.numpy(), d=d.numpy(), od=od, dd=dd, g=g, fake=fake, fake_want=fake_want, isect=isect,
                isect_h=isect.cpu().numpy(), order=order, order_h=order.cpu().numpy())


def test_intersections_dilation_and_sampler_at_frame_geometry(frame):
    """ray_block_intersection, process_occupied_grid for every tile, then nb rounds of sample_points -> prepare_points as
    render_rays issues them, until every ray has finished its tiles."""
    f, sc = frame, frame["sc"]
    ops, nb = f["ops"], sc["nb"]
    assert _rounds(B_FRAME, 256, f["sms"]) >= 2 and _rounds(B_FRAME, 128, f["sms"]) >= 4, "sampler / intersection rounds"
    assert _rounds(B_FRAME * S, 256, f["sms"]) >= 50, "prepare_points rounds"
    want = _isect(f["o"], f["d"], sc)
    got = f["isect_h"]
    assert np.array_equal(got == MISS, want == MISS) and np.allclose(got, want, rtol=1e-6, atol=0)
    hits = (got[..., 0] != MISS).sum(-1)
    assert (hits == nb).any() and (hits == 0).any() and (hits >= 2).mean() > 0.2
    assert np.array_equal(f["fake"].cpu().numpy().astype(np.uint8), f["fake_want"]), "dilated occupancy grids must be bit-exact"
    assert f["fake_want"][int(sc["starts"][2]):int(sc["starts"][3])].any(), "the empty tile receives cells from its neighbour"
    ti, zs = torch.zeros(B_FRAME, 1, dtype=torch.int32, device=DEV), torch.zeros(B_FRAME, 1, device=DEV)
    ti_h, zs_h = np.zeros(B_FRAME, np.int32), np.zeros(B_FRAME, np.float32)
    z, di = torch.empty(B_FRAME, S, device=DEV), torch.empty(B_FRAME, S, device=DEV)
    bi = torch.empty(B_FRAME, S, 4, dtype=torch.int16, device=DEV)
    sampled, err = np.zeros(B_FRAME, np.int64), 0.0
    for rnd in range(nb):
        running = (ti < nb).contiguous()
        z.fill_(-1.0); di.fill_(-1.0); bi.fill_(-1)
        ops.sample_points(f["od"], f["dd"], f["g"]["corners"], f["g"]["sizes"], f["fake"], f["g"]["starts"], f["g"]["l2d"], f["order"],
                          f["isect"], ti, zs, z, di)
        ops.prepare_points(z, running, f["isect"], bi)
        torch.cuda.synchronize()
        run_h = ti_h < nb
        z_h, di_h = np.full((B_FRAME, S), -1, np.float32), np.full((B_FRAME, S), -1, np.float32)
        on.render_sample(f["o"], f["d"], sc["corners"].numpy(), sc["sizes"].numpy(), f["fake_want"], sc["starts"].numpy(), sc["l2d"].numpy(),
                         f["order_h"], got, ti_h, zs_h, z_h, di_h)
        zg, dg = z.cpu().numpy(), di.cpu().numpy()
        assert np.array_equal(ti.cpu().numpy()[:, 0], ti_h), f"round {rnd}: tracing_idx"
        assert np.array_equal(zs.cpu().numpy()[:, 0], zs_h), f"round {rnd}: z_start"
        assert np.array_equal(zg == -1, z_h == -1), f"round {rnd}: sampled rays / the -1 pattern"
        assert np.allclose(zg, z_h, rtol=1e-6, atol=0) and np.allclose(dg, di_h, rtol=1e-6, atol=0), f"round {rnd}: z_vals / dists"
        err = max(err, _rel(zg, z_h), _rel(dg, di_h))
        assert np.array_equal(bi.cpu().numpy(), rr.prepare_points_vec(zg, run_h, got)), f"round {rnd}: block_idxs"
        sampled += (z_h[:, 0] != -1)
    assert np.array_equal(ti_h, (got[..., 0] != MISS).sum(-1)), "after nb rounds every ray stops at its first missed tile"
    assert sampled.max() >= 3 and (sampled == 0).any() and (ti_h == nb).any()
    print(f"sampler: worst relative error of z_vals / dists {err:.2e}")


def test_exit_tiles_first_hit_and_inverse_z_at_frame_geometry(frame):
    """ray_firsthit_block, get_last_block, update_outgoing_bidx (as render_rays calls it), update_outgoing_bidx_v2 and
    inverse_z_sampling of the first two exit slots."""
    f, sc = frame, frame["sc"]
    ops, B = f["ops"], B_FRAME
    assert _rounds(B, 128, f["sms"]) >= 4 and _rounds(B, 256, f["sms"]) >= 2
    c, s, args = sc["corners"].numpy(), sc["sizes"].numpy(), (f["od"], f["dd"], f["g"]["corners"], f["g"]["sizes"])
    hit = torch.full((B, 1), -1, dtype=torch.int16, device=DEV)
    ops.ray_firsthit_block(*args, f["fake"], f["g"]["starts"], f["g"]["l2d"], f["order"], f["isect"], hit)
    last = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    ops.get_last_block(f["order"], last, f["isect"])
    ids, w = torch.full((B, 4), -1, dtype=torch.int16, device=DEV), torch.zeros(B, 4, device=DEV)
    ops.update_outgoing_bidx(*args, f["order"], f["isect"], ids, w, 0.12, False)
    ids2, w2 = torch.full((B, 4), -1, dtype=torch.int16, device=DEV), torch.full((B, 4), 0.25, device=DEV)
    ops.update_outgoing_bidx_v2(*args, f["order"], f["isect"], ids2, w2)
    torch.cuda.synchronize()
    want_hit = on.firsthit_block(f["o"], f["d"], c, s, f["fake_want"], sc["starts"].numpy(), sc["l2d"].numpy(), f["order_h"], f["isect_h"])
    assert np.array_equal(hit.cpu().numpy()[:, 0], want_hit)
    assert len(np.unique(want_hit)) == sc["nb"] + 1
    assert np.array_equal(last.cpu().numpy(), rr.get_last_block_vec(f["order_h"], f["isect_h"]))
    want_ids, want_w = on.outgoing_bidx(f["o"], f["d"], c, s, f["order_h"], f["isect_h"])
    got_ids, got_w = ids.cpu().numpy(), w.cpu().numpy()
    assert np.array_equal(got_ids, want_ids) and (want_ids[:, 1] >= 0).any()
    assert np.allclose(got_w, want_w, rtol=1e-6, atol=0)
    errs = {"outgoing weights": _rel(got_w, want_w)}
    want_ids2, want_w2 = rr.inside_bidx(f["o"], c, s, np.full((B, 4), -1, np.int16), np.full((B, 4), 0.25, np.float32))
    assert np.array_equal(ids2.cpu().numpy(), want_ids2) and (want_ids2[:, 1] >= 0).any()
    assert np.allclose(w2.cpu().numpy(), want_w2, rtol=1e-6, atol=0)
    errs["inside weights"] = _rel(w2.cpu().numpy(), want_w2)
    for slot in range(2):
        z = torch.full((B, S), 7.5, device=DEV)
        ops.inverse_z_sampling(f["isect"], ids[:, slot].contiguous(), z, 1e6)
        want = rr.inverse_z_vec(f["isect_h"], want_ids[:, slot], S, 1e6, np.full((B, S), 7.5, np.float32))
        zg = z.cpu().numpy()
        assert np.array_equal(zg == 7.5, want == 7.5), "rows without that exit tile keep the caller's fill"
        assert np.allclose(zg, want, rtol=1e-6, atol=0, equal_nan=True)
        errs[f"inverse z slot {slot}"] = _rel(zg, want)
    print("worst relative errors:", {k: f"{v:.2e}" for k, v in errs.items()})


def test_accumulate_at_frame_geometry():
    """accumulate_color over a frame of 32-sample rays (28 grid-stride rounds of 8-ray blocks on 148 SMs) against float64:
    transparency, diffuse, specular and depth within 1e-5 (relative above 1); rays entering with T < 1e-5 are untouched."""
    ops, sms = _ops()
    B = B_FRAME
    assert _rounds(B, 256, sms, per_block=8) >= 20
    g = torch.Generator(device=DEV).manual_seed(4)
    pa = torch.rand(B, S, 1, device=DEV, generator=g) * 0.2
    pd, ps = torch.rand(B, S, 3, device=DEV, generator=g) * pa, torch.rand(B, S, 3, device=DEV, generator=g) * pa
    z = torch.rand(B, S, device=DEV, generator=g).cumsum(-1)
    T0 = torch.rand(B, 1, device=DEV, generator=g)
    T0[::7] = 5e-6
    init = [T0, torch.rand(B, 3, device=DEV, generator=g), torch.rand(B, 3, device=DEV, generator=g), torch.rand(B, 1, device=DEV, generator=g)]
    out = [t.clone() for t in init]
    ops.accumulate_color(pd, ps, pa, out[0], z, out[1], out[2], out[3])
    torch.cuda.synchronize()
    step, worst = 1 << 18, {}
    for i0 in range(0, B, step):
        sl = slice(i0, i0 + step)
        h = lambda t: t[sl].cpu().numpy()
        want = rr.accumulate64(h(pd), h(ps), h(pa), h(init[0]), h(z), h(init[1]), h(init[2]), h(init[3]))
        for name, x, y, x0 in zip(("T", "diffuse", "specular", "depth"), out, want, init):
            x = h(x).reshape(y.shape).astype(np.float64)
            e = np.abs(x - y) / np.maximum(1.0, np.abs(y))
            assert np.all(e <= 1e-5), f"{name}: {e.max()}"
            worst[name] = max(worst.get(name, 0.0), float(e.max()))
            skip = h(init[0])[:, 0] < 1e-5
            assert np.array_equal(h(x0).reshape(y.shape)[skip], x[skip].astype(np.float32))
    print("accumulate: worst errors against float64", {k: f"{v:.2e}" for k, v in worst.items()})


# ------------------------------------------------------------------------------------------------------------ frame driver
def frame_restatement(sc, o, d, S, Sb, sample_range=1e6):
    """render_frame.render_rays on the CPU: the C restatements of the tracing stages, the numpy forms of the simple ones,
    field_restatement for the field ("fore" per round, "slot" per exit slot with the normalised weights) and float64
    accumulation.  The tracing order is the device argsort of the restated intersections (ties keep the driver's order).
    Returns diffuse, specular [B,3], depth, T [B] (NaN background where it is not defined), the rays with a foreground
    sample near a cell face [B], and the exit tiles [B,4] with their normalised weights [B,4]."""
    B, nb = o.shape[0], sc["nb"]
    c, s, l2d, starts = sc["corners"].numpy(), sc["sizes"].numpy(), sc["l2d"].numpy(), sc["starts"].numpy()
    isect = _isect(o.numpy(), d.numpy(), sc)
    order = torch.argsort(torch.from_numpy(isect).to(DEV)[..., 0], dim=-1).int().cpu().numpy()
    fake = sc["occ"].numpy().astype(np.uint8)
    for b in range(nb):
        fake = on.process_occupied(b, sc["n"][b], c, s, sc["occ"].numpy(), starts, l2d, fake)
    T, dif, spe, dep = np.ones(B), np.zeros((B, 3)), np.zeros((B, 3)), np.zeros(B)
    ti, zs = np.zeros(B, np.int32), np.zeros(B, np.float32)
    near_rays = np.zeros(B, bool)
    for _ in range(nb):
        running = (ti < nb) & (T > 1e-5)
        z, di = np.full((B, S), -1, np.float32), np.full((B, S), -1, np.float32)
        on.render_sample(o.numpy(), d.numpy(), c, s, fake, starts, l2d, order, isect, ti, zs, z, di)
        bi = rr.prepare_points_vec(z, running, isect)
        pd, ps, pa, _, near = field_restatement("fore", sc, o, d, torch.from_numpy(z), torch.from_numpy(di), torch.from_numpy(bi))
        near_rays |= near.any(-1)
        T, dif, spe, dep = rr.accumulate64(pd, ps, pa, T, z, dif, spe, dep)
    ids, w = on.outgoing_bidx(o.numpy(), d.numpy(), c, s, order, isect)
    with np.errstate(invalid="ignore"):
        w = np.nan_to_num(w / w.sum(-1, keepdims=True), nan=0.0)
    bg = np.zeros((B, 7))
    undefined = np.zeros(B, bool)
    for i in range(4):
        if not (ids[:, i] >= 0).any():
            break
        bz = rr.inverse_z_vec(isect, ids[:, i], Sb, sample_range, np.full((B, Sb), -1, np.float32))
        # a ray that leaves its tile within a few hundredths of its origin gets a last inverse-z sample at infinity or behind
        # the origin (1 / (1/far - 1/near + 1/near) in float32), in the reference as well: its background is not defined
        with np.errstate(invalid="ignore"):
            bad = (ids[:, i] >= 0) & ~(np.isfinite(bz) & (bz > 0)).all(-1)
        undefined |= bad
        r = np.nonzero(~bad)[0]
        pd, ps, pa, _, _ = field_restatement("slot", sc, o[r], d[r], torch.from_numpy(bz[r]), None, torch.from_numpy(ids[r]), step=i)
        _, td, tsp, tz = rr.accumulate64(pd, ps, pa, np.ones(len(r)), bz[r], np.zeros((len(r), 3)), np.zeros((len(r), 3)), np.zeros(len(r)))
        bg[r] += np.concatenate([td, tsp, tz[:, None]], 1) * w[r, i:i + 1]
    bg[undefined] = np.nan
    return dif + T[:, None] * bg[:, :3], spe + T[:, None] * bg[:, 3:6], dep + T * bg[:, 6], T, near_rays, ids, w


def _tileset(sc):
    """TileSet from the exported (doubled) boxes: corner - size / 2, 2 size."""
    import render_frame as rf
    ts = rf.TileSet(DEV)
    for i in range(sc["nb"]):
        k = int(sc["starts"][i])
        ts.add_tile(sc["tables"][i], sc["params"][i], sc["res"][i], sc["occ"][k:k + sc["n"][i]], sc["corners"][i] - sc["sizes"][i] / 2,
                    sc["sizes"][i] * 2, sc["l2d"][i])
    ts.finalize()
    assert torch.equal(ts.block_corner.cpu(), sc["corners"]) and torch.equal(ts.block_size.cpu(), sc["sizes"])
    return ts


def _check_frame(got, want, ok):
    """Colours and transparency within 1e-4, depth within 1e-4 relative, on the rays `ok`."""
    d, s, z, T = (t.cpu().double().numpy() for t in got)
    wd, ws, wz, wT = want
    errs = {"diffuse": np.abs(d[ok] - wd[ok]).max(), "specular": np.abs(s[ok] - ws[ok]).max(), "T": np.abs(T[ok, 0] - wT[ok]).max(),
            "depth (rel)": (np.abs(z[ok, 0] - wz[ok]) / np.maximum(np.abs(wz[ok]), 1.0)).max()}
    for name, e in errs.items():
        assert e < 1e-4, f"{name}: {e}"
    return errs


@pytest.mark.parametrize("tiles", [(0,), (0, 1, 2), (0, 1, 2, 3)])
def test_render_rays_against_frame_restatement(tiles):
    """render_frame.render_rays, adaptive and worst-case, each against frame_restatement and bit for bit against each other,
    on 4096 rays (both cameras, random and missing rays), S = 32, Sb = 24.  The sampler starts every occupied segment on a cell face, so most sampled rays have a
    sample that field_restatement flags as near one; the restatement forms the sample positions in the kernels' float32
    order, so those rays are compared too.  Left out are only the rays (< 1 %) whose background is not defined."""
    _ops()
    import render_frame as rf
    sc = _tile_scene(tiles)
    o, d = _rays(32, 16, 2048, 1024, seed=7 + len(tiles))
    Sb = 24
    ts = _tileset(sc)
    want_d, want_s, want_z, want_T, near, ids, _ = frame_restatement(sc, o, d, S, Sb)
    ok = np.isfinite(want_d).all(-1)
    assert ok.mean() > 0.99, f"{1 - ok.mean():.3%} of the rays have an undefined background"
    assert (want_T < 0.5).mean() > 0.1 and near.mean() > 0.1
    if len(tiles) > 1:
        assert (ids[:, 1] >= 0).any()
    images = []
    for adaptive in (True, False):
        got = rf.render_rays(ts, o.to(DEV), d.to(DEV), num_sample=S, num_bg_sample=Sb, adaptive=adaptive)
        assert bool(torch.isfinite(got[0][torch.from_numpy(ok).to(DEV)]).all())
        errs = _check_frame(got, (want_d, want_s, want_z, want_T), ok)
        print(f"tiles {tiles}, adaptive={adaptive}: worst errors {errs}, rays with a sample near a cell face {near.mean():.1%}, "
              f"left out {1 - ok.mean():.2%}")
        images.append(got)
    same = lambda a, b: torch.equal(torch.nan_to_num(a, nan=-7.0), torch.nan_to_num(b, nan=-7.0))
    assert all(same(a, b) for a, b in zip(*images)), "adaptive and worst-case round counts give the same image"


def test_render_rays_evaluates_a_background_slot_behind_a_zero_weight():
    """A ray that leaves two tiles at one depth, through an x-z edge of the first (exit weights [0, 5], normalised [0, 1]),
    alone in its batch: adaptive=True must still evaluate slot 1 and equal adaptive=False bit for bit."""
    _ops()
    import render_frame as rf
    raw = make_scene(2, seed=5)
    n = raw["n_cells"]
    sc = dict(raw, corners=torch.tensor([[0.0, 0.0, 0.0], [0.0, 0.0, 5.0]]), sizes=torch.tensor([[10.0, 6.0, 10.0], [10.0, 6.0, 10.0]]),
              occ=torch.zeros(2 * n, dtype=torch.bool), n=[n, n])
    o, d = torch.tensor([[4.0, 3.0, 4.0]]), torch.tensor([[1.0, 0.0, 1.0]])
    want_d, want_s, want_z, want_T, near, ids, w = frame_restatement(sc, o, d, S, 24)
    assert ids[0].tolist() == [0, 1, -1, -1] and w[0].tolist() == [0.0, 1.0, 0.0, 0.0]
    assert want_d[0].max() > 1e-3, "the background through slot 1 is visible"
    ts = _tileset(sc)
    got = rf.render_rays(ts, o.to(DEV), d.to(DEV), num_sample=S, num_bg_sample=24)
    worst = rf.render_rays(ts, o.to(DEV), d.to(DEV), num_sample=S, num_bg_sample=24, adaptive=False)
    for a, b in zip(got, worst):
        assert torch.equal(a, b), "adaptive=True drops the weighted slot behind the zero-weight one"
    _check_frame(got, (want_d, want_s, want_z, want_T), np.ones(1, bool))
