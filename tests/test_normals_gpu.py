"""GPU: surface normals of HashGrid.render_batch_rays(out_normal=True) on the fused field path (snrf_field_normal).

The reference differentiates sigma w.r.t. the samples with torch.autograd.grad (hashgrid/__init__.py:547-556) and accumulates
the normal detached.  The fused path evaluates g = d sigma / dx forward only, from the field encode's features and per-level
Jacobians.  Checked here: the kernel against a float64 restatement of the chain, the render call against the CPU oracle and
against the torch branch it replaces (also at the C2 launch geometry), the other outputs and the training gradients against the
calls without normals, and degenerate inputs."""
import math

import pytest
import torch

from conftest import load_pkg
from oracle import torch_ref as tr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BOX_MIN = torch.tensor([-10.0, -6.5, -15.0])        # the doubled box of a (20, 13, 30) tile at the origin
BOX_SIZE = torch.tensor([40.0, 26.0, 60.0])


@pytest.fixture(autouse=True)
def _pkg():
    load_pkg()


def _rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def _params(seed, b_sigma):
    """Decoder parameters in decoder_params order: xavier weights (oracle.torch_ref.init_mlp), non-zero biases, the sigma bias
    set to `b_sigma` (it places sigma_pre relative to the softplus threshold of 20)."""
    g = torch.Generator().manual_seed(seed)
    p = tr.init_mlp(g)
    for k in tr.MLP_KEYS:
        p[k + ".bias"] = torch.randn(p[k + ".bias"].shape, generator=g) * 0.1
    p["sigma_layer.mlp.0.bias"] = torch.tensor([float(b_sigma)])
    return [p[k + s] for k in tr.MLP_KEYS for s in (".weight", ".bias")]


def _reference_grad(params, feats, jac, mask32, x, mode):
    """float64 restatement: g = d sigma / dx from level-major features [16,N,2], Jacobians [16,3,N,2] (w.r.t. the contracted
    point) and the world-space samples x [N,3] (float32, as the kernel forms them).  Also returns sigma_pre."""
    P = [p.double() for p in params]
    W1, b1, W2, b2, ws, bs = P[0], P[1], P[2], P[3], P[4][0], P[5][0]
    m = mask32.double()
    f = feats.double().permute(1, 0, 2).reshape(-1, 32)                    # channel 2 l + c
    z1 = (f * m) @ W1.t() + b1
    a1 = torch.exp(-50.0 * z1 * z1)
    u = W2[:32].t() @ ws
    c = ws @ b2[:32] + bs
    pre = a1 @ u + c
    dsp = torch.where(pre > 20.0, torch.ones_like(pre), torch.sigmoid(pre))
    gz = dsp[:, None] * (-100.0 * z1 * a1) * u
    gf = m * (gz @ W1)                                                      # [N,32]
    gc = torch.einsum("nlc,lanc->na", gf.reshape(-1, 16, 2), jac.double())
    x64 = x.double().clone().requires_grad_(True)
    bmin, bsize = BOX_MIN.double(), BOX_SIZE.double()
    cx = tr.contract_fore(x64, bmin, bsize) if mode == 1 else tr.contract_bg(x64, bmin, bsize)
    gx = torch.autograd.grad(cx, x64, grad_outputs=gc)[0]
    return gx, pre


def _kernel_case(mode, seed, R=512, S=8):
    g = torch.Generator().manual_seed(seed)
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
    z = torch.rand(R, S, generator=g).sort(-1)[0] * (8.0 if mode == 1 else 400.0)
    z[:, 0] = 0.0                                                           # sample 0 of every ray sits at o
    if mode == 1:
        o = BOX_MIN + torch.rand(R, 3, generator=g) * BOX_SIZE
        # samples on and next to the faces of the doubled box (contracted coordinate +-2)
        face = torch.randint(0, 3, (R // 4,), generator=g)
        side = torch.randint(0, 2, (R // 4,), generator=g).float()
        o[torch.arange(R // 4), face] = (BOX_MIN + side[:, None] * BOX_SIZE)[torch.arange(R // 4), face] + \
            (torch.rand(R // 4, generator=g) - 0.5) * 1e-3
    else:
        # affine-normalised point u with |u|_inf in (1, 3]; the first quarter sits next to a face of the inner box (|u|_inf
        # just above 1), the second quarter next to an edge between two cube faces (|u_i| = |u_j| +- 1e-3)
        uu = (torch.rand(R, 3, generator=g) * 2 - 1)
        k = torch.randint(0, 3, (R,), generator=g)
        sgn = torch.where(torch.rand(R, generator=g) < 0.5, -1.0, 1.0)
        nrm = 1.0 + torch.rand(R, generator=g) * 2.0
        nrm[: R // 4] = 1.0 + torch.rand(R // 4, generator=g) * 1e-3
        uu = uu * nrm[:, None] * 0.999
        uu[torch.arange(R), k] = sgn * nrm
        j = (k[R // 4: R // 2] + 1) % 3
        q = torch.arange(R // 4, R // 2)
        off = (0.2 + 0.8 * torch.rand(R // 4, generator=g)) * 1e-3 * torch.where(torch.rand(R // 4, generator=g) < 0.5, -1.0, 1.0)
        uu[q, j] = torch.where(uu[q, j] < 0, -1.0, 1.0) * (nrm[q] + off)   # clear of a tie in float32 and float64 alike
        o = BOX_MIN + (uu + 2.0) / 4.0 * BOX_SIZE
    feats = torch.randn(16, R * S, 2, generator=g) * 0.4
    jac = torch.randn(16, 3, R * S, 2, generator=g) * 5.0
    mask32 = tr.level_mask(5500).repeat_interleave(2)                       # levels 0..11 on, 12 partial, 13..15 off
    valid = torch.rand(R, generator=g) < 0.85
    return o, d, z, feats, jac, mask32, valid


def _run_kernel(params, o, d, z, feats, jac, mask32, valid, mode, sentinel=7.0):
    from hashgrid import _field
    R, S = z.shape
    normal = torch.full((R * S, 3), sentinel, device=DEV)
    grad = torch.full((R * S, 3), sentinel, device=DEV)
    _field.field_normal(feats.to(DEV), jac.to(DEV), mask32.to(DEV), [p.to(DEV) for p in params], o.to(DEV), d.to(DEV), z.to(DEV),
                        BOX_MIN.to(DEV), BOX_SIZE.to(DEV), mode, valid=valid.to(DEV) if valid is not None else None,
                        normal=normal, grad=grad)
    torch.cuda.synchronize()
    return normal.cpu(), grad.cpu()


def _sample_pos(o, d, z):
    """o + z d with separately rounded multiply and add (torch's order, and the kernel's)."""
    return (o[:, None, :] + z[..., None] * d[:, None, :]).reshape(-1, 3)


# ------------------------------------------------------------------------------------------------------------------------
# 1. the kernel against float64
# ------------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("side", ["below", "straddle", "above"])
def test_kernel_matches_float64_restatement(mode, side):
    """g = d sigma / dx within 1e-5 relative L2 of a float64 restatement; normals within 1e-4 rad where |g| is above 1e-3 of
    its median (below that floor the direction of g is set by rounding); rows of masked-out rays untouched.  The sigma bias
    puts sigma_pre below, across or above torch's softplus threshold of 20."""
    o, d, z, feats, jac, mask32, valid = _kernel_case(mode, 5 + mode)
    x = _sample_pos(o, d, z)
    pre0 = _reference_grad(_params(11 + mode, 0.0), feats, jac, mask32, x, mode)[1]
    bias = {"below": 19.5 - float(pre0.max()), "straddle": 20.0 - float(pre0.median()), "above": 20.5 - float(pre0.min())}[side]
    params = _params(11 + mode, bias)
    normal, grad = _run_kernel(params, o, d, z, feats, jac, mask32, valid, mode)
    S = z.shape[1]
    live = valid.repeat_interleave(S)
    assert bool((normal[~live] == 7.0).all()) and bool((grad[~live] == 7.0).all()), "rows of masked-out rays were written"
    g_ref, pre = _reference_grad(params, feats, jac, mask32, x, mode)
    g_ref, pre = g_ref[live], pre[live]
    above = float((pre > 20.0).double().mean())
    assert {"below": above == 0.0, "straddle": 0.3 < above < 0.7, "above": above == 1.0}[side], above
    err = _rel_l2(grad[live], g_ref)
    assert err < 1e-5, f"d sigma / dx: relative L2 {err:.3e}"
    mag = g_ref.norm(dim=-1)
    big = mag > 1e-3 * mag.median()
    assert float(big.double().mean()) > 0.95
    a, b = normal[live][big].double(), -g_ref[big]
    ang = torch.atan2(torch.linalg.cross(a, b).norm(dim=-1), (a * b).sum(-1))
    assert float(ang.max()) < 1e-4, f"normal angle error {float(ang.max()):.3e} rad"


# ------------------------------------------------------------------------------------------------------------------------
# render_batch_rays helpers
# ------------------------------------------------------------------------------------------------------------------------

def _grid(log2T=15, seed=0, scale=0.3):
    from hashgrid import HashGrid
    from hashgrid._decoder import ShallowMLP
    dev = torch.device(DEV)
    torch.manual_seed(seed)
    hg = HashGrid(dev, torch.tensor([0.0, 0.0, 0.0], device=dev), torch.tensor([20.0, 13.0, 30.0], device=dev), log2T, [16, 256], 4,
                  False, "")
    g = torch.Generator(device=DEV).manual_seed(seed)
    with torch.no_grad():
        hg.HE.features.copy_(torch.randn(hg.HE.features.shape, device=DEV, generator=g) * scale)
    dec = ShallowMLP(32).to(dev)
    with torch.no_grad():
        for p in dec.parameters():
            if p.dim() == 1:
                p.copy_(torch.randn(p.shape, device=DEV, generator=g) * 0.1)
    return hg, dec


def _rays(R, S, bg, seed):
    g = torch.Generator().manual_seed(seed)
    o = torch.tensor([10.0, 6.5, 15.0]) + torch.randn(R, 3, generator=g)
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
    z = (torch.rand(R, S, generator=g) * 6).sort(-1)[0]
    if bg:
        z = 20.0 + z * 30.0
    dist = torch.cat([z[:, 1:] - z[:, :-1], torch.full((R, 1), 1e-3)], -1)
    return o.to(DEV), d.to(DEV), z.to(DEV), dist.to(DEV)


def _render(hg, dec, o, d, z, dist, bg, mode, out_normal=True, step=9000):
    contract = hg.contract_bg if bg else hg.contract_fore
    out, ok = hg.render_batch_rays(o, d, z, dist, dec, mode, contract, out_normal=out_normal, infinity=bg, global_step=step)
    assert ok
    return out


# ------------------------------------------------------------------------------------------------------------------------
# 2. end to end against the CPU oracle
# ------------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("bg", [False, True])
def test_render_normal_matches_cpu_oracle(bg):
    """render_batch_rays(out_normal=True) in INFERENCE against oracle.torch_ref: samples and contraction in float32 as the
    reference forms them, the C oracle's encode with its point gradients (HashEncodeCPU), the decoder in float64, g by
    torch.autograd.grad, weights by torch_ref.integrate_weights in float64.  The per-ray bar of 2e-4 covers the bf16x3
    decoder's weights (about 1e-5 against float64, test_production_geometry_gpu) and the float32 g (about 1e-6 relative)."""
    from hashgrid import INFERENCE
    from hashgrid._decoder import decoder_params
    hg, dec = _grid()
    R, S = 256, 64
    o, d, z, dist = _rays(R, S, bg, 21 + bg)
    out = _render(hg, dec, o, d, z, dist, bg, INFERENCE)
    got = out["normal"].cpu().double()
    # CPU oracle
    params = [p.detach().cpu() for p in decoder_params(dec)]
    P = {k + s: params[2 * i + j].double() for i, k in enumerate(tr.MLP_KEYS) for j, s in enumerate((".weight", ".bias"))}
    oc, dc, zc = o.cpu(), d.cpu(), z.cpu()
    x = _sample_pos(oc, dc, zc).clone().requires_grad_(True)
    bmin, bsize = hg.min_bbox.cpu(), hg.bbox_size.cpu()
    cx = tr.contract_bg(x, bmin, bsize) if bg else tr.contract_fore(x, bmin, bsize)
    feats = tr.HashEncodeCPU.apply(cx, hg.HE.features.detach().cpu(), hg.HE.resolution.cpu()).reshape(-1, 32).double()
    mask32 = tr.level_mask(9000).repeat_interleave(2).double()
    heads = tr.shallow_mlp(P, feats, dc.double().repeat_interleave(S, 0), mask32)
    sigma = heads["sigma"]
    gx = torch.autograd.grad(sigma.sum(), x)[0].double()
    n_ref = -gx / (gx.norm(dim=-1, keepdim=True) + 1e-8)
    w, _ = tr.integrate_weights(sigma.detach().reshape(R, S, 1), dist.cpu().double(), dc.double(), bg)
    ref = (w * n_ref.reshape(R, S, 3)).sum(1)
    err = float((got - ref).abs().max())
    print(f"normal vs CPU oracle (bg={bg}): max abs {err:.3e}, |ref| mean {float(ref.norm(dim=-1).mean()):.3f}")
    assert float(ref.norm(dim=-1).mean()) > 0.05, "the case must have rays with visible surfaces"
    assert err < 2e-4, f"per-ray normal differs from the CPU oracle by {err:.3e}"


# ------------------------------------------------------------------------------------------------------------------------
# 3. against the torch branch at production geometry
# ------------------------------------------------------------------------------------------------------------------------

def test_fused_normal_matches_torch_branch_at_c2_geometry():
    """2^14 rays x 128 samples with a 2^24 table (one chain of the C2 workload).  The normal kernel's grid-stride loop runs
    many rounds at this size.  Per-ray normals of the fused path against the torch branch (fused_decoder = False: torch
    encode operator, fp32 torch decoder, autograd.grad)."""
    import scanerf_b200_capi as capi
    from hashgrid import INFERENCE
    R, S = 2 ** 14, 128
    N = R * S
    sms = int(capi.lib().snrf_device_sm_count())
    ctas = min(math.ceil(N / 256), 2 * sms)                 # snrf_field_normal's launch (include/scanerf_b200.h)
    rounds = N / (ctas * 256)
    assert ctas == 2 * sms and rounds >= 8, f"{rounds:.1f} grid-stride rounds per thread"
    hg, dec = _grid(log2T=24, seed=3, scale=0.3)
    for bg in (False, True):
        o, d, z, dist = _rays(R, S, bg, 31 + bg)
        fused = _render(hg, dec, o, d, z, dist, bg, INFERENCE)
        hg.fused_decoder = False
        try:
            ref = _render(hg, dec, o.clone().requires_grad_(True), d, z, dist, bg, INFERENCE)
        finally:
            hg.fused_decoder = True
        err = (fused["normal"] - ref["normal"].detach()).abs().max(dim=-1)[0]
        print(f"C2 fused vs torch branch (bg={bg}): max {float(err.max()):.3e}, p99.9 {float(err.quantile(0.999)):.3e}")
        assert float(ref["normal"].norm(dim=-1).mean()) > 0.05
        assert float(err.max()) < 1e-3, f"per-ray normal differs from the torch branch by {float(err.max()):.3e}"
        del fused, ref
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------------
# 4. no side effects on the other outputs
# ------------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("rays_grad", [False, True])
@pytest.mark.parametrize("bg", [False, True])
def test_other_outputs_are_bitwise_unchanged(bg, rays_grad):
    from hashgrid import TRAIN
    hg, dec = _grid(seed=4)
    o, d, z, dist = _rays(300, 32, bg, 41 + bg)
    if rays_grad:
        o, d = o.requires_grad_(True), d.requires_grad_(True)
    a = _render(hg, dec, o, d, z, dist, bg, TRAIN, out_normal=True)
    b = _render(hg, dec, o, d, z, dist, bg, TRAIN, out_normal=False)
    for k in ("rgb", "depth", "T_left", "diffuse", "specular", "weights", "l2_reg_specular"):
        assert torch.equal(a[k], b[k]), k
    assert "normal" in a and "normal" not in b


# ------------------------------------------------------------------------------------------------------------------------
# 5. TRAIN mode
# ------------------------------------------------------------------------------------------------------------------------

def _train_grads(hg, dec, o, d, z, dist, bg, c):
    from hashgrid import TRAIN
    hg.HE.features.grad = None
    dec.zero_grad(set_to_none=True)
    oo, dd = o.clone().requires_grad_(True), d.clone().requires_grad_(True)
    out = _render(hg, dec, oo, dd, z, dist, bg, TRAIN)
    (out["rgb"].sum() + out["depth"].sum() * 0.01 + out["l2_reg_specular"] + (out["normal"] * c).sum()).backward()
    return [hg.HE.features.grad.clone(), oo.grad.clone(), dd.grad.clone()] + [p.grad.clone() for p in dec.parameters()], out


@pytest.mark.parametrize("bg", [False, True])
def test_train_gradients_match_torch_branch(bg):
    """The normal is detached: its loss term reaches the field through the compositing weights only.  Gradients of the
    table, decoder parameters, rays_o and rays_d against the torch branch (fused_decoder = False).  The two branches run
    different decoders: the tensor-core one computes its backward from bf16 operands (at most 4.6e-4 relative L2 against
    float64 in test_production_geometry_gpu), the torch one in fp32, so the bar is that test's 2e-3 rather than the 1e-4
    of fused against unfused encode with one decoder.  Against the fused call without normals whose loss adds the same
    term through `weights`, the gradients agree to 1e-6."""
    from hashgrid import TRAIN
    hg, dec = _grid(seed=5)
    o, d, z, dist = _rays(200, 32, bg, 51 + bg)
    c = torch.randn(200, 3, generator=torch.Generator().manual_seed(52)).to(DEV)
    fused, out = _train_grads(hg, dec, o, d, z, dist, bg, c)
    # the same loss through the call without normals: (normal * c).sum() = sum_rs w_rs (n_rs . c_r) with n detached
    from hashgrid import _field
    from hashgrid._decoder import decoder_params
    nrm = out["normal"].detach()
    jac = []
    feats = _field.field_encode(o, d, z, hg.HE.features.detach(), hg.HE.resolution, hg.min_bbox, hg.bbox_size, 2 if bg else 1,
                                jac_out=jac)
    n = _field.field_normal(feats, jac.pop(), hg.level_mask32(9000), decoder_params(dec), o, d, z, hg.min_bbox, hg.bbox_size,
                            2 if bg else 1).view(200, 32, 3)
    k = (n * c[:, None, :]).sum(-1)
    hg.HE.features.grad = None
    dec.zero_grad(set_to_none=True)
    oo, dd = o.clone().requires_grad_(True), d.clone().requires_grad_(True)
    plain = _render(hg, dec, oo, dd, z, dist, bg, TRAIN, out_normal=False)
    (plain["rgb"].sum() + plain["depth"].sum() * 0.01 + plain["l2_reg_specular"] + (plain["weights"][..., 0] * k).sum()).backward()
    alt = [hg.HE.features.grad.clone(), oo.grad.clone(), dd.grad.clone()] + [p.grad.clone() for p in dec.parameters()]
    assert torch.allclose(nrm, (plain["weights"] * n).sum(1), atol=1e-6)
    for a, b in zip(fused, alt):
        assert _rel_l2(a, b) < 1e-6
    hg.fused_decoder = False
    try:
        ref, _ = _train_grads(hg, dec, o, d, z, dist, bg, c)
    finally:
        hg.fused_decoder = True
    names = ["table", "rays_o", "rays_d"] + [n for n, _ in dec.named_parameters()]
    errs = {name: _rel_l2(a, b) for name, a, b in zip(names, fused, ref)}
    print(f"TRAIN gradients fused vs torch branch (bg={bg}): " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < 2e-3}
    assert not bad, f"gradients differ from the torch branch: {bad}"


# ------------------------------------------------------------------------------------------------------------------------
# 6. degenerate inputs
# ------------------------------------------------------------------------------------------------------------------------

def test_degenerate_inputs():
    from hashgrid import INFERENCE
    hg, dec = _grid(seed=6)
    o, d, z, dist = _rays(64, 16, False, 61)
    assert not o.requires_grad and not d.requires_grad        # rays outside any autograd graph take the fused path
    out = _render(hg, dec, o, d, z, dist, False, INFERENCE)
    assert out["normal"].shape == (64, 3) and bool(torch.isfinite(out["normal"]).all())
    assert float(out["normal"].norm(dim=-1).max()) > 0.1
    # all weights 0 (zero sample spacing, finite last step): normal 0
    flat = _render(hg, dec, o, d, z, torch.zeros_like(dist), False, INFERENCE)
    assert float(flat["weights"].abs().max()) == 0.0
    assert float(flat["normal"].abs().max()) == 0.0
    # zero table: g = 0 everywhere, normal 0 and no NaN
    with torch.no_grad():
        hg.HE.features.zero_()
    zero = _render(hg, dec, o, d, z, dist, False, INFERENCE)
    assert bool(torch.isfinite(zero["normal"]).all()) and float(zero["normal"].abs().max()) == 0.0
    assert float(zero["weights"].max()) > 0.0
