"""GPU: the training kernels at the launch geometry of the C2 workload (BASELINE.json: 2^14 rays x 128 samples per chain, joint
fore + background batch of 2^15 rays = 2^22 samples, 16 x 2^24 x 2 table) against float64 references.

The parity tests of the other files run every persistent / grid-stride kernel for exactly one round; the state that is only
carried from the second round on (TMEM accumulators and mbarrier phases of the decoder backward across a CTA's tiles, the
grid-stride loops of the scatter, the Adam slices and the compositing, the side stream + programmatic-dependent-launch chain of
the fused scatter + Adam) is checked here against references that share no code with the kernels.  Every test first asserts
the geometry it claims (rounds per CTA / warp / thread, launch counts), computed from the SM count and the sizes, so that a
changed default that falls back to one round fails instead of passing silently."""
import ctypes

import pytest
import torch

from conftest import load_pkg
from oracle import native as on
from oracle import torch_ref as tr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
L, T, R, S = 16, 2 ** 24, 2 ** 14, 128          # C2: one chain; the joint batch has 2R rays
N_C2 = 2 * R * S                                  # 2^22 samples
N_RAGGED, S_RAGGED = 148 * 128 * 3 + 77, 64       # about three backward tiles per CTA, ragged last tile
ROWS = 128                                        # decoder tile (decoder_core.cuh kRows)


@pytest.fixture(autouse=True)
def _pkg():
    load_pkg()


def _capi():
    import scanerf_b200_capi as capi
    return capi


def _sms():
    return int(_capi().lib().snrf_device_sm_count())


def _rel_l2(a, b):
    return float((a.double() - b).norm() / b.norm().clamp_min(1e-30))


# ------------------------------------------------------------------------------------------------------------------------
# A. decoder
# ------------------------------------------------------------------------------------------------------------------------

def _decoder_case(N, S, seed):
    """Decoder parameters with non-zero biases, level-major features [16,N,2] as the field encode writes them, a partial
    level mask, ray directions [ceil(N/S),3] -- all float32 on the GPU."""
    from hashgrid._decoder import ShallowMLP, decoder_params
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    dec = ShallowMLP(32)
    for p in dec.parameters():
        if p.dim() == 1:
            p.data = torch.randn(p.shape, generator=g) * 0.05
    params = [p.detach().to(DEV) for p in decoder_params(dec)]
    gd = torch.Generator(device=DEV).manual_seed(seed)
    feats = torch.randn(16, N, 2, device=DEV, generator=gd) * 0.3
    mask32 = tr.level_mask(5500).repeat_interleave(2).to(DEV)          # levels 0..11 on, 12 at 0.35, 13..15 off
    assert 0.0 < float(mask32[24]) < 1.0 and float(mask32[-1]) == 0.0
    rays_d = torch.randn((N + S - 1) // S, 3, device=DEV, generator=gd) * 1.7
    return params, feats, mask32, rays_d


def _ref_params(params):
    return {k + s: p.double().clone().requires_grad_(True)
            for i, k in enumerate(tr.MLP_KEYS) for s, p in ((".weight", params[2 * i]), (".bias", params[2 * i + 1]))}


def _ref_heads(P, feats_rm, dirs, mask32):
    o = tr.shallow_mlp(P, feats_rm, dirs, mask32)
    return torch.cat([o["sigma"], o["tint"], o["diffuse"], o["specular"]], -1)


def _reference_decoder(params, feats, mask32, rays_d, S, cot=None, chunk=2 ** 20):
    """float64 oracle.torch_ref.shallow_mlp over [16,N,2] features, in chunks of samples.  Returns the heads [N,10], or with
    a cotangent [N,10] the gradients (features [N,32] row-major, rays_d, the 16 parameters in decoder_params order)."""
    N = feats.shape[1]
    P = _ref_params(params)
    m = mask32.double()
    d64 = rays_d.double().clone().requires_grad_(True)
    out = torch.empty(N, 32 if cot is not None else 10, dtype=torch.float64, device=DEV)
    for c0 in range(0, N, chunk):
        c1 = min(N, c0 + chunk)
        f = feats[:, c0:c1].permute(1, 0, 2).reshape(c1 - c0, 32).double()
        dirs = d64[torch.arange(c0, c1, device=DEV) // S]
        if cot is None:
            with torch.no_grad():
                out[c0:c1] = _ref_heads(P, f, dirs, m)
            continue
        f.requires_grad_(True)
        (_ref_heads(P, f, dirs, m) * cot[c0:c1].double()).sum().backward()
        out[c0:c1] = f.grad
    if cot is None:
        return out
    return out, d64.grad, [P[k + s].grad for k in tr.MLP_KEYS for s in (".weight", ".bias")]


def _bwd_geometry(N):
    tiles = (N + ROWS - 1) // ROWS
    grid = min(_sms(), tiles)                 # snrf_decoder_bwd: one CTA per SM, each loops over its tiles
    return tiles, grid


def _dead_tile_between_live_ones(tile_live, grid):
    """A CTA whose tile sequence (tile b, b + grid, ...) skips a dead tile after a live one and processes a live one after it."""
    for b in range(grid):
        seq = tile_live[b::grid].tolist()
        for i in range(1, len(seq) - 1):
            if not seq[i] and any(seq[:i]) and any(seq[i + 1:]):
                return True
    return False


def _check_grads(tag, g_feats_rm, g_d, g_params, want, live_rows):
    want_f, want_d, want_p = want
    errs = {"feats": _rel_l2(g_feats_rm[live_rows], want_f[live_rows]), "rays_d": _rel_l2(g_d, want_d)}
    for i, (a, b) in enumerate(zip(g_params, want_p)):
        errs[f"param{i}{tuple(b.shape)}"] = _rel_l2(a, b)
    print(f"{tag}: rel L2 errs", {k: f"{v:.2e}" for k, v in errs.items()})
    for k, v in errs.items():
        assert v < 2e-3, f"{tag} {k}: {v}"


@pytest.mark.parametrize("N,S", [(N_C2, S), (N_RAGGED, S_RAGGED)])
def test_decoder_forward_against_float64(N, S):
    """The default forward (four tiles in flight, layer 2 folded) over many rounds of four tiles per CTA."""
    from hashgrid import _field
    tiles = (N + ROWS - 1) // ROWS
    grid = min(_sms(), (tiles + 3) // 4)
    rounds = (tiles + 4 * grid - 1) // (4 * grid)
    assert rounds >= (50 if N == N_C2 else 1) and (N % ROWS != 0) == (N == N_RAGGED), (tiles, grid, rounds)
    params, feats, mask32, rays_d = _decoder_case(N, S, 1)
    heads = _field.decoder_forward(feats, mask32, rays_d, S, params)
    want = _reference_decoder(params, feats, mask32, rays_d, S)
    err = (heads.double() - want).abs()
    print(f"decoder fwd N={N}: max abs err per head", [f"{float(err[:, a:b].max()):.2e}" for a, b in ((0, 1), (1, 4), (4, 7), (7, 10))])
    assert bool(torch.isfinite(heads).all())
    assert float(err.max()) < 1e-4


@pytest.mark.parametrize("N,S,masked", [(N_C2, S, False), (N_C2, S, True), (N_RAGGED, S_RAGGED, True)])
def test_decoder_backward_against_float64(N, S, masked):
    """The default backward (layer 2 folded, forward heads reused) through _field.decoder_apply: about 221 tiles per CTA at
    C2 (TMEM weight-gradient accumulators and the mbarrier phase carried across tiles, the per-CTA composition of dW2 / dW3a /
    dW_heads / db2 after the last one).  masked: every 7th tile and 10 % of the other rays masked out, so that CTAs skip dead
    tiles in the middle of their sequence; the masked rows of the cotangent are NaN (never read)."""
    from hashgrid import _field
    tiles, grid = _bwd_geometry(N)
    assert tiles / grid >= (200 if N == N_C2 else 3), (tiles, grid)
    params, feats, mask32, rays_d = _decoder_case(N, S, 2)
    nr = rays_d.shape[0]
    gd = torch.Generator(device=DEV).manual_seed(3)
    cot = torch.randn(N, 10, device=DEV, generator=gd)
    valid, live = None, torch.ones(N, dtype=torch.bool, device=DEV)
    if masked:
        ray_tile = torch.arange(nr, device=DEV) * S // ROWS
        valid = (ray_tile % 7 != 3) & (torch.rand(nr, device=DEV, generator=gd) > 0.1)
        live = valid.repeat_interleave(S)[:N]
        tile_live = torch.zeros(tiles * ROWS, dtype=torch.bool, device=DEV)
        tile_live[:N] = live
        tile_live = tile_live.reshape(tiles, ROWS).any(1)
        assert _dead_tile_between_live_ones(tile_live.cpu(), grid)
        cot[~live] = float("nan")
    f = feats.clone().requires_grad_(True)
    d = rays_d.clone().requires_grad_(True)
    p = [q.clone().requires_grad_(True) for q in params]
    heads = _field.decoder_apply(f, d, mask32, S, p, valid)
    heads.backward(cot)
    torch.cuda.synchronize()
    want = _reference_decoder(params, feats, mask32, rays_d, S, torch.where(live[:, None], cot, torch.zeros_like(cot)))
    _check_grads(f"decoder bwd N={N} masked={masked}", f.grad.permute(1, 0, 2).reshape(N, 32), d.grad, [q.grad for q in p], want, live)


def test_decoder_backward_ert_dead_tiles():
    """snrf_decoder_bwd_ert at C2 with hand-set early-ray-termination flags: every 5th ray (= tile) terminated before its
    first sample, the others after a random number of samples.  Dead samples contribute nothing, and their grad_feats rows
    are left unwritten (a NaN sentinel survives)."""
    capi = _capi()
    N, S_ = N_C2, S
    tiles, grid = _bwd_geometry(N)
    assert tiles / grid >= 200
    params, feats, mask32, rays_d = _decoder_case(N, S_, 4)
    nr = rays_d.shape[0]
    gd = torch.Generator(device=DEV).manual_seed(5)
    cut = torch.randint(1, S_ + 1, (nr,), device=DEV, generator=gd)
    cut[torch.arange(nr, device=DEV) % 5 == 2] = 0
    live = (torch.arange(S_, device=DEV)[None, :] < cut[:, None]).reshape(-1)[:N]
    tile_live = live.reshape(tiles, ROWS).any(1)
    assert _dead_tile_between_live_ones(tile_live.cpu(), grid) and bool((~live[tile_live.repeat_interleave(ROWS)]).any())
    sample_live = live.to(torch.uint8)
    cot = torch.randn(N, 10, device=DEV, generator=gd)          # dead rows carry values the backward must ignore
    from hashgrid import _field
    heads = _field.decoder_forward(feats, mask32, rays_d, S_, params)
    g_feats = torch.full_like(feats, float("nan"))
    g_d = torch.zeros_like(rays_d)
    g_params = [torch.zeros_like(q) for q in params]
    arr = (ctypes.c_void_p * 16)(*[q.data_ptr() for q in params])
    garr = (ctypes.c_void_p * 16)(*[q.data_ptr() for q in g_params])
    from scanerf_b200_capi import c_int, c_void_p, ptr
    rc = capi.lib().snrf_decoder_bwd_ert(ptr(feats), ptr(mask32), ptr(rays_d), arr, ptr(cot), ptr(g_feats), ptr(g_d), garr,
                                         c_int(N), c_int(S_), c_int(1), c_void_p(0), ptr(heads), ptr(sample_live), capi.stream())
    capi.check(rc, "snrf_decoder_bwd_ert")
    torch.cuda.synchronize()
    g_rm = g_feats.permute(1, 0, 2).reshape(N, 32)
    assert bool(torch.isnan(g_rm[~live]).all()), "rows of dead samples are left unwritten"
    want = _reference_decoder(params, feats, mask32, rays_d, S_, cot * live[:, None])
    _check_grads("decoder bwd ert", g_rm, g_d, g_params, want, live)


# ------------------------------------------------------------------------------------------------------------------------
# B. scatter + Adam at T = 2^24
# ------------------------------------------------------------------------------------------------------------------------
LR, B1, B2, EPS = 1e-2, 0.9, 0.99, 1e-15
KTHREADS = 256                                    # field_encode.cu kThreads


def _grid_x(n):
    """field_encode.cu grid_x: at most four waves of eight CTAs per SM."""
    want, wave = (n + KTHREADS - 1) // KTHREADS, _sms() * 8
    return max(want, 1) if want <= wave else wave * min(4, (want + wave - 1) // wave)


def _joint_batch():
    from test_fullsize_gpu import _inputs
    res, bmin, bsize, o1, d1, z1 = _inputs(21)
    _, _, _, o2, d2, z2 = _inputs(22)
    o, d = torch.cat([o1, o2]), torch.cat([d1, d2])
    z = torch.cat([z1, z2 * 40.0 + 12.0]).contiguous()           # background-range depths for the second half
    return res, bmin, bsize, o, d, z


def _contracted(o, d, z, bmin, bsize, split):
    """The points the fused kernel encodes, built in torch: fore map for rays [0, split), background map for the rest."""
    x = (o[:, None, :] + z[..., None] * d[:, None, :])
    fore = (torch.arange(o.shape[0], device=o.device) < split)[:, None, None]
    return torch.where(fore, tr.contract_fore(x, bmin, bsize), tr.contract_bg(x, bmin, bsize)).reshape(-1, 3)


@pytest.fixture(scope="module")
def scatter_adam_case():
    """Inputs of two fused steps and their oracle gradients (C oracle, CPU): table gradients of both steps, ray gradients
    of the first (the table values enter only there, and both steps start the same rays from the same table)."""
    load_pkg()
    res, bmin, bsize, o, d, z = _joint_batch()
    nr = o.shape[0]
    gen = torch.Generator(device=DEV).manual_seed(23)
    table = torch.randn(L, T, 2, device=DEV, generator=gen) * 0.1
    valid = torch.rand(nr, device=DEV, generator=gen) < 0.8
    cots = [torch.randn(L, nr * S, 2, device=DEV, generator=gen) for _ in range(2)]
    vmask = valid.repeat_interleave(S)[None, :, None]
    pts = _contracted(o, d, z, bmin, bsize, R).cpu().numpy()
    tab, rs = table.cpu().numpy(), res.cpu().numpy()
    gts, gp = [], None
    for k, cot in enumerate(cots):
        gpk, gt = on.hash_encode_bwd(pts, (cot * vmask).permute(1, 0, 2).contiguous().cpu().numpy(), tab, rs)
        gts.append(torch.from_numpy(gt))
        gp = gpk if k == 0 else gp
    del tab
    # ray gradients of step 1: the oracle's d/d points through the contraction, float64 autograd
    o64, d64 = o.double().requires_grad_(True), d.double().requires_grad_(True)
    x = _contracted(o64, d64, z.double(), bmin.double(), bsize.double(), R)
    (x * torch.from_numpy(gp).to(DEV).double()).sum().backward()
    return dict(res=res, bmin=bmin, bsize=bsize, o=o, d=d, z=z, table=table, valid=valid, cots=cots, gts=gts,
                g_o=o64.grad, g_d=d64.grad)


def _adam_ref(p, m, v, g, step):
    nz = g != 0
    m1 = torch.where(nz, B1 * m + (1 - B1) * g, m)
    v1 = torch.where(nz, B2 * v + (1 - B2) * g * g, v)
    upd = (LR / (1 - B1 ** step)) * m1 / ((v1 / (1 - B2 ** step)).sqrt() + EPS)
    return torch.where(nz, p - upd, p), m1, v1


@pytest.mark.parametrize("plain", [False, True])
def test_scatter_adam_fusion_against_oracle_and_float64_adam(scatter_adam_case, plain):
    """snrf_field_encode_bwd_adam under the default plan at T = 2^24 (4 coarse levels in one pass each on the side stream,
    12 fine levels in 2 index ranges, 56 scatter / Adam launches chained by programmatic dependent launch), 2^22 samples
    (the scatter's grid-stride loop runs several rounds, and so does every Adam slice's), two steps.  plain: the same plan
    as plain launches on one stream -- if only the default arm fails, the fault is in the ordering, not in the slicing."""
    capi = _capi()
    from hashgrid import _field
    from vdbAdam import vdbAdam
    c = scatter_adam_case
    res, o, d, z, valid = c["res"], c["o"], c["d"], c["z"], c["valid"]
    nr = o.shape[0]
    N = nr * S
    sms = _sms()
    # ---- geometry of the default plan
    assert N == N_C2 and _field.small_levels(res) == 4
    assert N > 4 * 8 * sms * KTHREADS and (N + _grid_x(N) * KTHREADS - 1) // (_grid_x(N) * KTHREADS) >= 2, "scatter rounds"
    for n4 in (T // 2, 2 ** 23 // 2):                        # float4 groups of a coarse level / of a fine slice
        gx = min((n4 + 2 * KTHREADS - 1) // (2 * KTHREADS), 16 * sms)
        assert (n4 + gx * 2 * KTHREADS - 1) // (gx * 2 * KTHREADS) >= 2, "Adam slice rounds"
    lib = capi.lib()
    t = torch.nn.Parameter(c["table"].clone())
    opt = vdbAdam([t], lr=LR, betas=(B1, B2), eps=EPS, bias_correction="standard", fused_zero_grad=True)
    p_ref = c["table"].double()
    m_ref, v_ref = torch.zeros_like(p_ref), torch.zeros_like(p_ref)
    if plain:
        lib.snrf_field_set_pdl(ctypes.c_int(0))
        lib.snrf_field_set_coarse_concurrent(ctypes.c_int(0))
    try:
        for step, (cot, gt) in enumerate(zip(c["cots"], c["gts"]), start=1):
            before = (t.detach().clone(), opt.params[0][1].clone(), opt.params[0][2].clone())
            oo, dd = o.clone().requires_grad_(True), d.clone().requires_grad_(True)
            enc = _field.field_encode(oo, dd, z, t, res, c["bmin"], c["bsize"], 3, valid, R)
            opt.zero_grad()
            with opt.table_backward(fused=True):
                enc.backward(cot)
            opt.step()
            torch.cuda.synchronize()
            assert int(lib.snrf_field_last_launch_count()) == 1 + 2 * (4 + 12 * 2)
            assert t.grad is None, "the fused path must not materialise a gradient table"
            assert float(opt._scratch.abs().max()) == 0.0, "scratch must be left all-zero"
            g = gt.to(DEV).double()
            p_ref, m_ref, v_ref = _adam_ref(p_ref, m_ref, v_ref, g, step)
            p, m, v = t.detach(), opt.params[0][1], opt.params[0][2]
            zero = g == 0
            for name, a, b in (("p", p, before[0]), ("m", m, before[1]), ("v", v, before[2])):
                assert torch.equal(a[zero], b[zero]), f"step {step}: {name} changed where the gradient is zero"
            touched = (p != before[0]) | (m != before[1]) | (v != before[2])      # (m, v can round back to their old values)
            residue = g.abs() <= 1e-5 * float(g.abs().max())
            off = touched != ~zero
            assert not bool((off & ~residue).any()), f"step {step}: touched sets differ at {int((off & ~residue).sum())} entries"
            em = float((m.double() - m_ref).abs().max()) / float(m_ref.abs().max())
            ev = float((v.double() - v_ref).abs().max()) / float(v_ref.abs().max())
            fp = float(((p.double() - p_ref).abs() > 1e-5).double().mean())
            eo = float((oo.grad.double() - c["g_o"]).abs().max()) / float(c["g_o"].abs().max())
            ed = float((dd.grad.double() - c["g_d"]).abs().max()) / float(c["g_d"].abs().max())
            print(f"plain={plain} step {step}: touched {int(touched.sum())}, set differences {int(off.sum())} (residues), m {em:.2e}, "
                  f"v {ev:.2e}, p off > 1e-5: {fp:.2e}" + (f", rays_o {eo:.2e}, rays_d {ed:.2e}" if step == 1 else ""))
            assert em < 1e-5 and ev < 1e-5, (em, ev)
            assert fp < 1e-4, fp
            if step == 1:
                assert eo < 2e-5 and ed < 2e-5, (eo, ed)
            del before, touched, residue, off, zero, g
    finally:
        lib.snrf_field_set_pdl(ctypes.c_int(1))
        lib.snrf_field_set_coarse_concurrent(ctypes.c_int(1))
    assert opt.t == 2


# ------------------------------------------------------------------------------------------------------------------------
# C. compositing of the joint batch and the joint loss
# ------------------------------------------------------------------------------------------------------------------------

def test_composite_joint_batch_against_float64():
    """composite_packed over the 2^15-ray joint batch in one launch (rays >= 2^14 end at infinity): each warp composites
    several rays.  Against oracle.torch_ref.composite in float64, per chain, over the valid rays."""
    from hashgrid import _render
    Rj = 2 * R
    nwarps = min((Rj + 7) // 8, _sms() * 8) * 8               # composite.cu grid_rays: blocks of 8 warps, at most 8 per SM
    assert Rj >= 2 * nwarps + 1, (Rj, nwarps)
    g = torch.Generator().manual_seed(31)
    heads = torch.rand(Rj * S, 10, generator=g)
    heads[:, 0] *= 3.0
    z = torch.cumsum(torch.rand(Rj, S, generator=g) * 0.1 + 0.01, -1)
    dists = torch.cat([z[:, 1:] - z[:, :-1], torch.full((Rj, 1), 1e-6)], -1)
    d = torch.randn(Rj, 3, generator=g) * 1.3
    valid = torch.rand(Rj, generator=g) < 0.9
    keys = ("rgb", "depth", "T_left", "tint", "diffuse", "specular")
    cot = {k: torch.randn(Rj, 3 if k not in ("depth", "T_left") else 1, generator=g) for k in keys}
    cot["T_left"] = cot["T_left"][:, 0]
    cot["weights"] = torch.randn(Rj, S, 1, generator=g)
    hp, dg = heads.to(DEV).requires_grad_(True), d.to(DEV).requires_grad_(True)
    out = _render.composite_packed(hp, z.to(DEV), dists.to(DEV), dg, R, True, valid.to(DEV))
    loss = sum((out[k] * cot[k].to(DEV)).sum() for k in cot) + 0.3 * out["l2_reg_specular"]
    loss.backward()
    torch.cuda.synchronize()
    # reference: each chain on its valid rays
    h64, d64 = heads.double().requires_grad_(True), d.double().requires_grad_(True)
    nv = int(valid.sum())
    loss_ref, refs = 0.0, {}
    for r0, inf in ((0, False), (R, True)):
        idx = r0 + torch.nonzero(valid[r0:r0 + R])[:, 0]
        hv = h64.view(Rj, S, 10)[idx]
        hd = {"sigma": hv[..., 0:1], "tint": hv[..., 1:4], "diffuse": hv[..., 4:7], "specular": hv[..., 7:10]}
        ref = tr.composite(hd, z[idx].double(), dists[idx].double(), d64[idx], inf, train=True)
        loss_ref = loss_ref + sum((ref[k] * cot[k][idx].double()).sum() for k in cot) + 0.3 * ref["l2_reg_specular"] * len(idx) / nv
        refs[inf] = (idx, ref)
    loss_ref.backward()
    for inf, (idx, ref) in refs.items():
        for k in keys + ("weights",):
            err = float((out[k].detach().cpu()[idx].double() - ref[k]).abs().max())
            assert err < 1e-4, f"chain infinity={inf} {k}: {err}"
    dead = ~valid.to(DEV)
    assert float(out["weights"][dead].abs().max()) == 0.0 and bool((out["T_left"][dead] == 1).all())
    assert float(dg.grad[dead].abs().max()) == 0.0
    live_rows = valid.repeat_interleave(S)
    for name, (a, b) in {"sigma": (0, 1), "tint": (1, 4), "diffuse": (4, 7), "specular": (7, 10)}.items():
        got, want = hp.grad.cpu()[live_rows, a:b].double(), h64.grad[live_rows, a:b]
        scale = max(float(want.abs().max()), 1e-6)
        err = float((got - want).abs().max())
        assert err < 2e-4 * scale + 3e-7, f"grad {name}: {err} vs scale {scale}"
    scale = max(float(d64.grad.abs().max()), 1e-6)
    assert float((dg.grad.cpu().double() - d64.grad).abs().max()) < 2e-4 * scale + 3e-7


@pytest.mark.parametrize("Rl,rounds", [(R, 1), (2 ** 18, 2)])
def test_joint_loss_against_float64(Rl, rounds):
    """snrf_joint_loss (merge of the two chains, clamp, masked MSE, specular L2 term) at the C2 batch and at a batch where
    its grid-stride loop runs twice, colours clamped on both sides, against a float64 torch restatement."""
    from hashgrid import _render
    gx = min((Rl + 255) // 256, _sms() * 4)
    assert (Rl + gx * 256 - 1) // (gx * 256) == rounds
    g = torch.Generator().manual_seed(41)
    row = torch.rand(2 * Rl, 16, generator=g)
    row[:, 4:10] = row[:, 4:10] * 1.2 - 0.3                  # diffuse + specular in [-0.6, 1.8): clamped at 0 and at 1
    vf, vb = torch.rand(Rl, generator=g) < 0.7, torch.rand(Rl, generator=g) < 0.6
    gt = torch.rand(Rl, 3, generator=g)
    w = 0.25
    rg = row.to(DEV).requires_grad_(True)
    loss = _render.JointLossFn.apply(rg, vf.to(DEV), vb.to(DEV), gt.to(DEV), w)
    loss.backward()
    r64 = row.double().requires_grad_(True)
    f, b = r64[:Rl], r64[Rl:]
    rgb_f, rgb_b = (f[:, 4:7] + f[:, 7:10]).clamp(0, 1), (b[:, 4:7] + b[:, 7:10]).clamp(0, 1)
    clamped = float(((f[:, 4:7] + f[:, 7:10] > 1) | (f[:, 4:7] + f[:, 7:10] < 0)).double().mean())
    assert 0.1 < clamped < 0.9
    pred = rgb_f + f[:, 13:14] * rgb_b
    valid = (vf | vb).double()[:, None]
    n = lambda m: max(int(m.sum()), 1)
    ref = ((pred - gt.double()) ** 2 * valid).sum() / (3 * n(vf | vb)) \
        + w * (f[:, 10:13].sum() / (3 * n(vf)) + b[:, 10:13].sum() / (3 * n(vb)))
    ref.backward()
    assert abs(float(loss) - float(ref)) <= 1e-6 * abs(float(ref)), (float(loss), float(ref))
    scale = float(r64.grad.abs().max())
    assert float((rg.grad.cpu().double() - r64.grad).abs().max()) <= 1e-6 * scale
