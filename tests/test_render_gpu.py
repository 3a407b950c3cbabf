"""GPU: the multi-tile inference renderer ops (csrc/render.cu, csrc/infer.cu behind the reference's
HASHGRID operator names) against the UNMODIFIED reference extension rebuilt into
oracle/_ref/HASHGRID.so, stage by stage on the same inputs, plus CPU restatements of the simple
stages and of the field evaluation in its three modes (C hash-encode oracle + torch decoder restatement).
Bars: tile ids / tracing state / sample-to-tile assignment bit-exact; depths 1e-6; per-sample
colours and alpha 1e-4 (the north star's composited-RGB tolerance)."""
import numpy as np
import pytest
import torch

from conftest import load_pkg, ref_module
from oracle import native as on
from oracle import torch_ref as tr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MISS = 1e7


def make_scene(nb=2, T=2 ** 14, seed=0, log2dim=(3, 2, 3)):
    g = torch.Generator().manual_seed(seed)
    corners = torch.tensor([[0.0, 0.0, 0.0], [8.0, 0.0, 1.0], [3.0, 0.0, 9.0]])[:nb].contiguous()
    sizes = torch.tensor([[10.0, 6.0, 12.0], [10.0, 6.0, 12.0], [12.0, 6.0, 8.0]])[:nb].contiguous()
    tables = (torch.randn(nb, 16, T, 2, generator=g) * 0.3).half()
    res = torch.stack([torch.stack([(torch.tensor([16.0, 12.0, 20.0]) * (1.38 ** l)).int() for l in range(16)]) for _ in range(nb)]).int()
    mlps = [tr.init_mlp(g) for _ in range(nb)]
    for m in mlps:
        for k in m:
            if k.endswith("bias"):
                m[k] = 0.05 * torch.randn(m[k].shape, generator=g)
    params = torch.stack([torch.cat([torch.cat([m[k + ".bias"], m[k + ".weight"].t().flatten()]) for k in tr.MLP_KEYS]) for m in mlps])
    assert params.shape == (nb, 13994)
    n_cells = int(np.prod([2 ** v for v in log2dim]))
    occ = torch.rand(nb * n_cells, generator=g) < 0.45
    starts = (torch.arange(nb) * n_cells).long()
    l2d = torch.tensor([list(log2dim)] * nb, dtype=torch.int32)
    return dict(corners=corners, sizes=sizes, tables=tables, res=res.contiguous(), params=params.contiguous(), occ=occ, starts=starts,
                l2d=l2d, mlps=mlps, nb=nb, T=T, n_cells=n_cells)


def make_rays(B, seed):
    g = torch.Generator().manual_seed(seed)
    o = torch.tensor([9.0, 3.0, 6.0]) + torch.randn(B, 3, generator=g) * torch.tensor([6.0, 1.0, 5.0])
    d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g) * torch.tensor([1.0, 0.25, 1.0]), dim=-1)
    d = d * (0.6 + torch.rand(B, 1, generator=g))
    return o.contiguous(), d.contiguous()


def dev(sc):
    return {k: (v.to(DEV) if isinstance(v, torch.Tensor) else v) for k, v in sc.items()}


def both(fn_name, ours, ref, make_args):
    """Run op `fn_name` of both modules on fresh copies of the same arguments; returns the two lists."""
    a, b = make_args(), make_args()
    getattr(ours, fn_name)(*a)
    if ref is not None:
        getattr(ref, fn_name)(*b)
    torch.cuda.synchronize()
    return a, (b if ref is not None else None)


def _ops():
    load_pkg()
    from hashgrid.lib import HASHGRID as ours
    return ours, ref_module("HASHGRID")


@pytest.mark.parametrize("nb,B", [(1, 500), (3, 6000)])
def test_render_pipeline_stage_by_stage(nb, B):
    ours, ref = _ops()
    sc = dev(make_scene(nb))
    o, d = (t.to(DEV) for t in make_rays(B, nb * B))
    S = 32
    # ---- ray / tile intersections
    (a, r) = both("ray_block_intersection", ours, ref, lambda: [o, d, sc["corners"], sc["sizes"], torch.full((B, nb, 2), MISS, device=DEV)])
    isect = a[-1]
    half = sc["sizes"] / 2
    want = on.ray_aabb(o.cpu().numpy(), d.cpu().numpy(), (sc["corners"] + half).cpu().numpy(), sc["sizes"].cpu().numpy())
    want = np.where(want == -1, MISS, want).reshape(B, nb, 2)
    assert np.allclose(isect.cpu().numpy(), want, rtol=1e-6, atol=1e-6)
    if r is not None:
        assert torch.equal(isect, r[-1])
    tracing_blocks = torch.argsort(isect[..., 0], dim=-1).int().contiguous()
    # ---- occupancy dilation across overlapping tiles
    fake = sc["occ"].clone()
    fake_r = sc["occ"].clone()
    for i in range(nb):
        ours.process_occupied_grid(i, sc["n_cells"], sc["corners"], sc["sizes"], sc["occ"], sc["starts"], sc["l2d"], fake)
        if ref is not None:
            ref.process_occupied_grid(i, sc["n_cells"], sc["corners"], sc["sizes"], sc["occ"], sc["starts"], sc["l2d"], fake_r)
    torch.cuda.synchronize()
    assert bool((fake | ~sc["occ"]).all()), "dilation never clears a cell"
    if ref is not None:
        assert torch.equal(fake, fake_r)
    if nb > 1:
        assert int(fake.sum()) > int(sc["occ"].sum())
    # ---- tracing loop: sample -> assign -> evaluate -> accumulate (two rounds exercise the resumable state)
    tracing_idx = torch.zeros(B, 1, dtype=torch.int32, device=DEV)
    z_start = torch.zeros(B, 1, device=DEV)
    T_, dif, spe, dep = torch.ones(B, 1, device=DEV), torch.zeros(B, 3, device=DEV), torch.zeros(B, 3, device=DEV), torch.zeros(B, 1, device=DEV)
    for rnd in range(2):
        running = ((tracing_idx < nb) & (T_ > 1e-5)).contiguous()
        mk = lambda: [o, d, sc["corners"], sc["sizes"], fake, sc["starts"], sc["l2d"], tracing_blocks, isect, tracing_idx.clone(),
                      z_start.clone(), torch.full((B, S), -1.0, device=DEV), torch.full((B, S), -1.0, device=DEV)]
        a, r = both("sample_points", ours, ref, mk)
        ti, zs, z, di = a[-4:]
        assert ((z == -1).all(-1) | (z != -1).all(-1)).all(), "a ray is sampled completely or not at all"
        if r is not None:
            assert torch.equal(ti, r[-4]), "tracing_idx must be bit-exact"
            assert torch.equal(z == -1, r[-2] == -1)
            for x, y in zip((zs, z, di), r[-3:]):
                assert torch.allclose(x, y, rtol=1e-6, atol=1e-6)
        a, r = both("prepare_points", ours, ref, lambda: [z, running, isect, torch.full((B, S, 4), -1, dtype=torch.int16, device=DEV)])
        bi = a[-1]
        zc, ic = z.cpu().numpy(), isect.cpu().numpy()
        inside = (zc[:, :, None] >= ic[:, None, :, 0]) & (zc[:, :, None] <= ic[:, None, :, 1]) & (zc[:, :, None] != -1) & running.cpu().numpy()[:, :, None]
        assert np.array_equal((bi.cpu().numpy() >= 0).sum(-1), inside.sum(-1)), "sample-to-tile assignment count"
        if r is not None:
            assert torch.equal(bi, r[-1]), "block_idxs must be bit-exact"
        mk = lambda: [o, d, z, di, bi, sc["tables"], sc["params"], sc["res"], sc["occ"], sc["starts"], sc["l2d"], sc["corners"], sc["sizes"],
                      torch.zeros(B, S, 3, device=DEV), torch.zeros(B, S, 3, device=DEV), torch.zeros(B, S, 1, device=DEV)]
        a, r = both("pts_inference", ours, ref, mk)
        pd, ps, pa = a[-3:]
        assert (rnd > 0 or float(pa.max()) > 0.01) and float(pa.min()) > -1e-3      # a sample a rounding error outside its tile has a (tiny) negative face weight, as in the reference
        if r is not None:
            for name, x, y in zip(("diffuse", "specular", "alpha"), (pd, ps, pa), r[-3:]):
                err = float((x - y).abs().max())
                assert err < 1e-4, f"pts_inference {name}: max abs err {err}"
        mk = lambda: [pd, ps, pa, T_.clone(), z, dif.clone(), spe.clone(), dep.clone()]
        a, r = both("accumulate_color", ours, ref, mk)
        if r is not None:
            for x, y in zip((a[3], a[5], a[6], a[7]), (r[3], r[5], r[6], r[7])):
                assert torch.allclose(x, y, rtol=1e-5, atol=1e-6)
        # numpy restatement of the front-to-back accumulation (rendering_kernel.cu:623-674)
        Tn, dn = T_.cpu().numpy()[:, 0].copy(), dif.cpu().numpy().copy()
        pdn, pan = pd.cpu().numpy(), pa.cpu().numpy()[..., 0]
        go = Tn >= 1e-5
        for k in range(S):
            dn[go] += Tn[go, None] * pdn[go, k]
            Tn[go] *= 1 - pan[go, k]
        assert np.allclose(a[5].cpu().numpy(), dn, rtol=1e-4, atol=1e-5) and np.allclose(a[3].cpu().numpy()[:, 0], Tn, rtol=1e-4, atol=1e-6)
        T_, dif, spe, dep = a[3], a[5], a[6], a[7]
        tracing_idx, z_start = ti, zs
    # ---- background: exit tiles, inverse-z samples, contracted evaluation
    mk = lambda: [o, d, sc["corners"], sc["sizes"], tracing_blocks, isect, torch.full((B, 4), -1, dtype=torch.int16, device=DEV),
                  torch.zeros(B, 4, device=DEV), 0.12, False]
    a, r = both("update_outgoing_bidx", ours, ref, mk)
    bgb, bgw = a[6], a[7]
    hit_any = (isect[..., 0] != MISS).any(-1)
    assert torch.equal(bgb[:, 0] != -1, hit_any)
    if r is not None:
        assert torch.equal(bgb, r[6]) and torch.allclose(bgw, r[7], rtol=1e-6, atol=1e-6)
    Sb = 24
    slot0 = bgb[..., 0].contiguous()
    a, r = both("inverse_z_sampling", ours, ref, lambda: [isect, slot0, torch.full((B, Sb), -1.0, device=DEV), 1e6])
    bz = a[2]
    far = torch.gather(isect[..., 1], 1, slot0.long().clamp_min(0)[:, None])[:, 0]
    assert torch.allclose(bz[hit_any, 0], far[hit_any], rtol=1e-5) and bool((bz[~hit_any] == -1).all())
    if r is not None:
        assert torch.allclose(bz, r[2], rtol=1e-6, atol=1e-6)
    mk = lambda: [o, d, bz, bgb, 0, sc["corners"], sc["sizes"], sc["res"], sc["tables"], sc["params"],
                  torch.full((B, Sb, 3), 0.5, device=DEV), torch.full((B, Sb, 3), 0.5, device=DEV), torch.full((B, Sb, 1), 0.5, device=DEV)]
    a, r = both("bg_pts_inference_v2", ours, ref, mk)
    assert bool((a[-1][~hit_any] == 0.5).all()), "rays without an exit tile keep the caller's rows"
    if r is not None:
        for name, x, y in zip(("diffuse", "specular", "alpha"), a[-3:], r[-3:]):
            # a ray that leaves its tile at depth ~0 gets an infinite last sample and NaN there -- in the reference too
            assert torch.equal(torch.isfinite(x), torch.isfinite(y)), f"bg_pts_inference_v2 {name}: non-finite pattern differs"
            x, y = torch.nan_to_num(x, nan=0.0, posinf=0.0, neginf=0.0), torch.nan_to_num(y, nan=0.0, posinf=0.0, neginf=0.0)
            err = float((x - y).abs().max())
            assert err < 1e-4, f"bg_pts_inference_v2 {name}: max abs err {err}"
    mk = lambda: [o, d, bz, bgb, torch.where(bgb >= 0, torch.ones_like(bgw), torch.zeros_like(bgw)) * 0.7, sc["corners"], sc["sizes"], sc["res"],
                  sc["tables"], sc["params"], torch.zeros(B, Sb, 3, device=DEV), torch.zeros(B, Sb, 3, device=DEV), torch.zeros(B, Sb, 1, device=DEV)]
    a, r = both("bg_pts_inference", ours, ref, mk)
    if r is not None:
        for name, x, y in zip(("diffuse", "specular", "alpha"), a[-3:], r[-3:]):
            assert torch.equal(torch.isfinite(x), torch.isfinite(y)), f"bg_pts_inference {name}: non-finite pattern differs"
            x, y = torch.nan_to_num(x, nan=0.0, posinf=0.0, neginf=0.0), torch.nan_to_num(y, nan=0.0, posinf=0.0, neginf=0.0)
            err = float((x[hit_any] - y[hit_any]).abs().max())
            assert err < 1e-4, f"bg_pts_inference {name}: max abs err {err}"
    # ---- the small helpers
    a, r = both("get_last_block", ours, ref, lambda: [tracing_blocks, torch.full((B,), -7, dtype=torch.int32, device=DEV), isect])
    if r is not None:
        assert torch.equal(a[1], r[1])
    a, r = both("ray_firsthit_block", ours, ref, lambda: [o, d, sc["corners"], sc["sizes"], fake, sc["starts"], sc["l2d"], tracing_blocks, isect,
                                                           torch.full((B, 1), -1, dtype=torch.int16, device=DEV)])
    if r is not None:
        assert torch.equal(a[-1], r[-1])
    a, r = both("update_outgoing_bidx_v2", ours, ref, lambda: [o, d, sc["corners"], sc["sizes"], tracing_blocks, isect,
                                                                torch.full((B, 4), -1, dtype=torch.int16, device=DEV), torch.zeros(B, 4, device=DEV)])
    if r is not None:
        assert torch.equal(a[6], r[6]) and torch.allclose(a[7], r[7], rtol=1e-6, atol=1e-6)


def _fma(a, b, c):
    """float32 a * b + c with one rounding, as the kernels' contracted expressions (the product is exact in float64)."""
    return (np.asarray(a, np.float64) * b + c).astype(np.float32)


def _encode(u, table, res):
    """The C oracle's hash encode (hash_encode_fwd) of table coordinates u [N,3] float32 -> [N,32], one level at a time
    in the box [0, res - 1]: the oracle then locates the cell at v = u * (res - 1) as the kernels form it.  (Its
    background mapping (x + 2) / 4 cannot hold every float32 u, and with these tables one ulp of u moves the
    specular head by up to 1e-3.)"""
    feats = np.empty((u.shape[0], 16, 2), np.float32)
    for l in range(16):
        r = res[l].astype(np.float32) - 1
        feats[:, l:l + 1] = on.hash_encode_fwd(u * r, table[l:l + 1], res[l:l + 1], corner=np.zeros(3, np.float32), size=r)
    return feats.reshape(-1, 32)


def field_restatement(mode, sc, o, d, z, dist, slots, blend=None, step=0):
    """CPU restatement of the field evaluation of pts_inference ("fore", rendering_kernel.cu:467-621),
    bg_pts_inference ("blend", :871-1008) and bg_pts_inference_v2 ("slot", :1011-1171) on host tensors.

    A sample visits its tile slots in order up to the first -1, each distinct tile once.  Foreground:
    q = (p - corner) / size, face weight w from dis = (0.5 - |q - 0.5|) * size (dis.x * dis.z, else dis.x,
    else dis.z, whichever are non-zero), added to the weight sum even where the occupancy cell is empty; the
    field is evaluated only where it is set, at u = q / 2 + 0.25, and alpha = 1 - exp(-sigma * dist * |d|).
    Background: contraction of the 2x-normalised position, w = the blend weight ("slot": the one slot `step`,
    w = 1), alpha = 1 - exp(-sigma * step length), the last step 1e7, no |d|.  The sums are normalised by the
    weight sum where it is positive, except for "slot".  The geometry is float32 in the kernel's order (with its
    fused multiply-adds), the encode is the C oracle on the fp16 table (_encode), the decoder torch_ref.shallow_mlp
    in float64.

    Returns diffuse [B,S,3], specular [B,S,3], alpha [B,S,1] (float64), `keep` [B,S] (rows the op leaves
    alone: "slot" rays without a tile in that slot) and `near` [B,S] (foreground samples within 1e-4 of a face of an
    occupancy cell or of one of their tiles, where the kernel's FMA contraction may decide differently)."""
    B, S = z.shape
    N = B * S
    f32 = lambda t: t.numpy().astype(np.float32)
    o, d, z = f32(o), f32(d), f32(z)
    corners, sizes = f32(sc["corners"]), f32(sc["sizes"])
    ray, k = np.repeat(np.arange(B), S), np.tile(np.arange(S), B)
    p = _fma(z.reshape(N, 1), d[ray], o[ray])
    if mode == "fore":
        ids = slots.numpy().reshape(N, 4).astype(np.int64)
        scale = f32(dist).reshape(N) * np.sqrt((d[ray] * d[ray]).sum(-1))
    else:
        ids = slots.numpy().astype(np.int64)[ray]
        if mode == "slot":
            ids = np.concatenate([ids[:, step:step + 1], np.full((N, 3), -1)], 1)
        znext = np.concatenate([z[:, 1:], z[:, -1:]], 1).reshape(N)
        scale = np.where(k == S - 1, np.float32(1e7), znext - z.reshape(N))
    wsum, acc, near = np.zeros(N), np.zeros((N, 7)), np.zeros(N, bool)
    open_ = np.ones(N, bool)
    for s in range(4):
        open_ &= ids[:, s] >= 0
        first = open_.copy()
        for j in range(s):
            first &= ids[:, j] != ids[:, s]
        for b in np.unique(ids[first, s]):
            n = np.nonzero(first & (ids[:, s] == b))[0]
            bc, bs = corners[b], sizes[b]
            if mode == "fore":
                q = (p[n] - bc) / bs
                dis = (np.float32(0.5) - np.abs(q - np.float32(0.5))) * bs
                w = np.where((dis[:, 0] != 0) & (dis[:, 2] != 0), dis[:, 0] * dis[:, 2], np.where(dis[:, 0] != 0, dis[:, 0], dis[:, 2]))
                l2 = sc["l2d"][b].numpy().astype(np.int64)
                cell = q * (1 << l2).astype(np.float32)
                g = np.clip(cell.astype(np.int64), 0, (1 << l2) - 1)
                active = sc["occ"].numpy()[int(sc["starts"][b]) + ((g[:, 0] << (l2[1] + l2[2])) | (g[:, 1] << l2[2]) | g[:, 2])]
                near[n] |= (np.abs(cell - np.round(cell)) * (bs / (1 << l2)) < 1e-4).any(-1)
                u = _fma(q, 0.5, 0.25)
            else:
                q = np.float32(2) * (p[n] - bc) / bs - np.float32(1)
                nrm = np.abs(q).max(-1, keepdims=True)
                assert (nrm > 1).all(), "background samples lie outside the tile (u in [0, 1])"
                u = _fma(q, (np.float32(2) - np.float32(1) / nrm) / nrm, 2) * np.float32(0.25)
                w = blend.numpy()[ray[n], s] if mode == "blend" else np.ones(len(n), np.float32)
                active = np.ones(len(n), bool)
            wsum[n] += w
            if not active.any():
                continue
            na = n[active]
            feats = _encode(u[active], sc["tables"][b].float().numpy(), sc["res"][b].numpy())
            mlp = {key: v.double() for key, v in sc["mlps"][b].items()}
            h = tr.shallow_mlp(mlp, torch.from_numpy(feats).double(), torch.from_numpy(d[ray[na]]).double(),
                               torch.ones(32, dtype=torch.float64))
            wa = torch.from_numpy(w[active]).double() * (1 - torch.exp(-h["sigma"][:, 0] * torch.from_numpy(scale[na]).double()))
            acc[na] += torch.cat([wa[:, None] * h["diffuse"], wa[:, None] * h["tint"] * h["specular"], wa[:, None]], 1).numpy()
    if mode != "slot":
        pos = wsum > 0
        acc[pos] /= wsum[pos, None]
    keep = ids[:, 0] < 0 if mode == "slot" else np.zeros(N, bool)
    return acc[:, :3].reshape(B, S, 3), acc[:, 3:6].reshape(B, S, 3), acc[:, 6:].reshape(B, S, 1), keep.reshape(B, S), near.reshape(B, S)


@pytest.mark.parametrize("nb,B,S", [(1, 64, 16), (1, 300, 7), (1, 37, 19), (3, 211, 7), (3, 1, 1), (2, 130, 128)])
@pytest.mark.parametrize("mode", ["fore", "blend", "slot"])
def test_pts_inference_against_cpu_restatement(mode, nb, B, S):
    """pts_inference / bg_pts_inference / bg_pts_inference_v2 against field_restatement, per sample within 1e-4.
    One scene tile takes the single-tile passes (decode with four tiles in flight for S >= 16, two below; blended
    background excepted), several take the grouped path; B * S is not a multiple of the 128-row decode tile or the
    256-row block.  Every sample row is written (over a sentinel) except those the op leaves alone, and
    unassigned foreground samples give exact zeros."""
    ours, _ = _ops()
    seed = 11 + nb + S
    sc = make_scene(nb, seed=seed)
    scd = dev(sc)
    o, d = make_rays(B, seed)
    g = torch.Generator().manual_seed(seed)
    dist = blend = None
    step = 1
    if mode == "fore":
        z = (torch.rand(B, S, generator=g) * 6.0).sort(-1)[0].contiguous()
        dist = torch.rand(B, S, generator=g) * 0.1 + 0.01
        isect = torch.full((B, nb, 2), MISS, device=DEV)
        ours.ray_block_intersection(o.to(DEV), d.to(DEV), scd["corners"], scd["sizes"], isect)
        bi = torch.full((B, S, 4), -1, dtype=torch.int16, device=DEV)
        ours.prepare_points(z.to(DEV), torch.ones(B, 1, dtype=torch.bool, device=DEV), isect, bi)
        slots = bi.cpu()
        if nb > 1:                       # a tile behind a -1 slot is ignored
            extra = (torch.rand(B, S, generator=g) < 0.1) & (slots[..., 0] >= 0) & (slots[..., 1] == -1)
            slots[..., 2] = torch.where(extra, (slots[..., 0] + 1) % nb, slots[..., 2])
    else:
        z = (40 + torch.rand(B, S, generator=g).cumsum(-1)).contiguous()     # beyond every tile
        slots = torch.randint(-1, nb, (B, 4), generator=g).to(torch.int16)      # with -1 gaps and repeated tiles
        blend = torch.rand(B, 4, generator=g) + 0.05
    outs = [torch.full((B, S, 3), 7.0, device=DEV), torch.full((B, S, 3), 7.0, device=DEV), torch.full((B, S, 1), 7.0, device=DEV)]
    args = (o.to(DEV), d.to(DEV), z.to(DEV))
    field = (scd["corners"], scd["sizes"], scd["res"], scd["tables"], scd["params"])
    if mode == "fore":
        ours.pts_inference(*args, dist.to(DEV), slots.to(DEV), scd["tables"], scd["params"], scd["res"], scd["occ"], scd["starts"],
                           scd["l2d"], scd["corners"], scd["sizes"], *outs)
    elif mode == "blend":
        ours.bg_pts_inference(*args, slots.to(DEV), blend.to(DEV), *field, *outs)
    else:
        ours.bg_pts_inference_v2(*args, slots.to(DEV), step, *field, *outs)
    torch.cuda.synchronize()
    got = [t.cpu() for t in outs]
    want_d, want_s, want_a, keep, near = field_restatement(mode, sc, o, d, z, dist, slots, blend, step)
    keep = torch.from_numpy(keep)
    for t in got:
        assert bool((t[keep] == 7.0).all()), "rows of rays without a tile in this slot keep the caller's values"
        assert bool((t[~keep] != 7.0).all()), "every other sample row is written"
    if mode == "fore":
        none = slots[..., 0] == -1
        assert all(bool((t[none] == 0).all()) for t in got), "unassigned samples give zeros"
    assert near.mean() < 0.01, f"{near.mean():.3%} of the samples lie within 1e-4 of a cell face"
    m = torch.from_numpy(~near) & ~keep
    if B * S > 1:
        assert int((want_a[m.numpy()] != 0).sum()) > 0.05 * B * S, "too few samples evaluated to test anything"
    for name, x, y in zip(("diffuse", "specular", "alpha"), got, (want_d, want_s, want_a)):
        err = float((x.double()[m] - torch.from_numpy(y)[m]).abs().max()) if bool(m.any()) else 0.0
        assert err < 1e-4, f"{mode} {name}: max abs err {err}"


def _render_with(mod, sc, o, d, S, Sb):
    """rendering.RenderingHashGrid.render_rays_base (rendering.py:286-544) sequenced over module `mod`."""
    B, nb = o.shape[0], sc["nb"]
    isect = torch.full((B, nb, 2), MISS, device=DEV)
    mod.ray_block_intersection(o, d, sc["corners"], sc["sizes"], isect)
    order = torch.argsort(isect[..., 0], dim=-1).int().contiguous()
    fake = sc["occ"].clone()
    for i in range(nb):
        mod.process_occupied_grid(i, sc["n_cells"], sc["corners"], sc["sizes"], sc["occ"], sc["starts"], sc["l2d"], fake)
    T_, dif, spe, dep = torch.ones(B, 1, device=DEV), torch.zeros(B, 3, device=DEV), torch.zeros(B, 3, device=DEV), torch.zeros(B, 1, device=DEV)
    ti, zs = torch.zeros(B, 1, dtype=torch.int32, device=DEV), torch.zeros(B, 1, device=DEV)
    max_tracing = int(torch.mean((isect != MISS).float(), dim=-1).sum(dim=-1).max().cpu())
    for _ in range(max_tracing):
        running = (ti < max_tracing) & (T_ > 1e-5)
        if running.sum() == 0:
            break
        z, di = torch.full((B, S), -1.0, device=DEV), torch.full((B, S), -1.0, device=DEV)
        mod.sample_points(o, d, sc["corners"], sc["sizes"], fake, sc["starts"], sc["l2d"], order, isect, ti, zs, z, di)
        bi = torch.full((B, S, 4), -1, dtype=torch.int16, device=DEV)
        mod.prepare_points(z, running, isect, bi)
        pd, ps, pa = torch.zeros(B, S, 3, device=DEV), torch.zeros(B, S, 3, device=DEV), torch.zeros(B, S, 1, device=DEV)
        mod.pts_inference(o, d, z, di, bi, sc["tables"], sc["params"], sc["res"], sc["occ"], sc["starts"], sc["l2d"], sc["corners"], sc["sizes"], pd, ps, pa)
        mod.accumulate_color(pd, ps, pa, T_, z, dif, spe, dep)
    bgb, bgw = torch.full((B, 4), -1, dtype=torch.int16, device=DEV), torch.zeros(B, 4, device=DEV)
    mod.update_outgoing_bidx(o, d, sc["corners"], sc["sizes"], order, isect, bgb, bgw, 0.12, False)
    bgw = bgw / torch.sum(bgw, dim=-1, keepdim=True)
    bd, bs = torch.zeros(B, 3, device=DEV), torch.zeros(B, 3, device=DEV)
    for i in range(int((bgw > 0).sum(dim=-1).max().cpu())):
        bz = torch.full((B, Sb), -1.0, device=DEV)
        mod.inverse_z_sampling(isect, bgb[..., i].contiguous(), bz, 1e6)
        pd, ps, pa = torch.zeros(B, Sb, 3, device=DEV), torch.zeros(B, Sb, 3, device=DEV), torch.zeros(B, Sb, 1, device=DEV)
        mod.bg_pts_inference_v2(o, d, bz, bgb, i, sc["corners"], sc["sizes"], sc["res"], sc["tables"], sc["params"], pd, ps, pa)
        t, td, tsp, tz = torch.ones(B, 1, device=DEV), torch.zeros(B, 3, device=DEV), torch.zeros(B, 3, device=DEV), torch.zeros(B, 1, device=DEV)
        mod.accumulate_color(pd, ps, pa, t, bz, td, tsp, tz)
        bd += td * bgw[:, i:i + 1]
        bs += tsp * bgw[:, i:i + 1]
    return dif + T_ * bd, spe + T_ * bs, T_


@pytest.mark.parametrize("nb", [1, 3])
def test_render_rays_driver_matches_reference_sequence(nb):
    """render_frame.render_rays (our sync-free mirror of render_rays_base) against the reference's own
    operator sequence run on the rebuilt reference extension; composited colours within 1e-4."""
    ours, ref = _ops()
    if ref is None:
        pytest.skip("oracle/_ref/HASHGRID.so not built")
    import render_frame as rf
    raw = make_scene(nb)
    sc = dev(raw)
    B, S, Sb = 3000, 32, 24
    o, d = (t.to(DEV) for t in make_rays(B, 77 + nb))
    want_d, want_s, want_T = _render_with(ref, sc, o, d, S, Sb)
    ts = rf.TileSet(DEV)
    for i in range(nb):       # TileSet takes the exported (doubled) boxes: corner - size/2, 2 size
        n = raw["n_cells"]
        ts.add_tile(raw["tables"][i], raw["params"][i], raw["res"][i], raw["occ"][i * n:(i + 1) * n], raw["corners"][i] - raw["sizes"][i] / 2,
                    raw["sizes"][i] * 2, raw["l2d"][i])
    ts.finalize()
    assert torch.allclose(ts.block_corner, sc["corners"]) and torch.allclose(ts.block_size, sc["sizes"])
    got_d, got_s, _, got_T = rf.render_rays(ts, o, d, num_sample=S, num_bg_sample=Sb)
    ok = torch.isfinite(want_d).all(-1) & torch.isfinite(want_s).all(-1)    # the reference yields NaN for rays that hit no tile
    assert int(ok.sum()) > B // 2
    assert float((got_d[ok] - want_d[ok]).abs().max()) < 1e-4
    assert float((got_s[ok] - want_s[ok]).abs().max()) < 1e-4
    assert float((got_T - want_T).abs().max()) < 1e-4
    assert bool(torch.isfinite(got_d[ok]).all())
    # the worst-case round counts (no host synchronisation) give the same image as the counts read back from the device
    d2, s2, _, T2 = rf.render_rays(ts, o, d, num_sample=S, num_bg_sample=Sb, adaptive=False)
    same = lambda a, b: torch.equal(torch.nan_to_num(a, nan=-7.0), torch.nan_to_num(b, nan=-7.0))     # (non-finite where the reference is)
    assert same(d2, got_d) and same(s2, got_s) and same(T2, got_T)


def test_simple_stages_against_numpy_oracle():
    """csrc/render.cu stages against the loop-form numpy restatement oracle/render_ref.py (small case)."""
    from oracle import render_ref as rr
    ours, _ = _ops()
    nb, B, S = 3, 300, 16
    raw = make_scene(nb)
    sc = dev(raw)
    o, d = make_rays(B, 123)
    od, dd = o.to(DEV), d.to(DEV)
    isect = torch.full((B, nb, 2), MISS, device=DEV)
    ours.ray_block_intersection(od, dd, sc["corners"], sc["sizes"], isect)
    want = rr.ray_block_intersection(o.numpy(), d.numpy(), raw["corners"].numpy(), raw["sizes"].numpy())
    assert np.array_equal(isect.cpu().numpy() == MISS, want == MISS)
    assert np.allclose(isect.cpu().numpy(), want, rtol=1e-6, atol=1e-6)
    order = torch.argsort(isect[..., 0], dim=-1).int().contiguous()
    g = torch.Generator().manual_seed(9)
    z = (torch.rand(B, S, generator=g) * 25).sort(-1)[0]
    z[::5] = -1.0
    running = torch.rand(B, 1, generator=g) < 0.8
    bi = torch.full((B, S, 4), -1, dtype=torch.int16, device=DEV)
    ours.prepare_points(z.to(DEV), running.to(DEV), isect, bi)
    assert np.array_equal(bi.cpu().numpy(), rr.prepare_points(z.numpy(), running.numpy()[:, 0], isect.cpu().numpy()))
    pd, ps, pa = torch.rand(B, S, 3, generator=g), torch.rand(B, S, 3, generator=g), torch.rand(B, S, 1, generator=g) * 0.3
    T0 = torch.rand(B, 1, generator=g)
    T0[::7] = 1e-6
    acc = [T0.clone().to(DEV), torch.rand(B, 3, generator=g).to(DEV), torch.rand(B, 3, generator=g).to(DEV), torch.rand(B, 1, generator=g).to(DEV)]
    init = [t.cpu().numpy().copy() for t in acc]
    ours.accumulate_color(pd.to(DEV), ps.to(DEV), pa.to(DEV), acc[0], z.to(DEV), acc[1], acc[2], acc[3])
    for got, w in zip(acc, rr.accumulate_color(pd.numpy(), ps.numpy(), pa.numpy(), init[0], z.numpy(), init[1], init[2], init[3])):
        assert np.allclose(got.cpu().numpy(), w, rtol=1e-5, atol=1e-5)
    last = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    ours.get_last_block(order, last, isect)
    assert np.array_equal(last.cpu().numpy(), rr.get_last_block(order.cpu().numpy(), isect.cpu().numpy()))
    ob, ow = torch.full((B, 4), -1, dtype=torch.int16, device=DEV), torch.zeros(B, 4, device=DEV)
    ours.update_outgoing_bidx(od, dd, sc["corners"], sc["sizes"], order, isect, ob, ow, 0.12, False)
    wb, ww = rr.update_outgoing_bidx(o.numpy(), d.numpy(), raw["corners"].numpy(), raw["sizes"].numpy(), order.cpu().numpy(), isect.cpu().numpy())
    assert np.array_equal(ob.cpu().numpy(), wb) and np.allclose(ow.cpu().numpy(), ww, rtol=1e-4, atol=1e-5)
    bz = torch.full((B, 12), -1.0, device=DEV)
    ours.inverse_z_sampling(isect, ob[:, 0].contiguous(), bz, 1e6)
    wz = rr.inverse_z_sampling(isect.cpu().numpy(), wb[:, 0], 12, 1e6)
    fin = np.isfinite(wz)
    assert np.array_equal(np.isfinite(bz.cpu().numpy()), fin) and np.allclose(bz.cpu().numpy()[fin], wz[fin], rtol=1e-5)
