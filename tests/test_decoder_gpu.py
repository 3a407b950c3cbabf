"""GPU: decoder MLP on the tensor cores (tcgen05 / TMEM) -- conventions self-test and parity of
the fused decoder forward/backward against the torch restatement of network.ShallowMLP
(oracle/torch_ref.py, pinned by tests/golden/py_golden_mlp.npz)."""
import numpy as np
import pytest
import torch

from conftest import load_pkg

pytestmark = pytest.mark.gpu


def _bf16(x):
    return x.to(torch.bfloat16).to(torch.float32)


def test_umma_selftest_three_gemm_shapes():
    load_pkg()
    import scanerf_b200_capi as capi
    from scanerf_b200_capi import ptr
    g = torch.Generator().manual_seed(0)
    X, W, G = torch.randn(128, 64, generator=g), torch.randn(64, 64, generator=g), torch.randn(128, 64, generator=g)
    dev = "cuda:0"
    Xd, Wd, Gd = X.to(dev), W.to(dev), G.to(dev)
    Y, DX, DW = torch.zeros(128, 64, device=dev), torch.zeros(128, 64, device=dev), torch.zeros(64, 64, device=dev)
    DWo, YS = torch.zeros(64, 16, device=dev), torch.zeros(128, 16, device=dev)
    capi.check(capi.lib().snrf_umma_selftest(ptr(Xd), ptr(Wd), ptr(Gd), ptr(Y), ptr(DX), ptr(DW), ptr(DWo), ptr(YS),
                                             capi.stream()), "snrf_umma_selftest")
    torch.cuda.synchronize()
    Xb, Wb, Gb = _bf16(X).double(), _bf16(W).double(), _bf16(G).double()
    for name, got, want in (("Y", Y, Xb @ Wb.T), ("DX", DX, Gb @ Wb), ("DW", DW, 2 * Gb.T @ Xb),
                            ("DWo", DWo, Gb.T @ Xb[:, 32:48]), ("YS", YS, Xb[:, 32:64] @ Wb[0:16, 0:32].T)):
        err = float((got.cpu().double() - want).abs().max())
        assert err < 1e-3, f"{name}: max abs err {err}"


def _decoder_and_inputs(N, S, seed):
    from hashgrid._decoder import ShallowMLP, decoder_params
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    dec = ShallowMLP(32)
    for p in dec.parameters():                      # non-zero biases so that every term is exercised
        if p.dim() == 1:
            p.data = torch.randn(p.shape, generator=g) * 0.05
    feats = torch.randn(N, 32, generator=g) * 0.3
    mask = torch.rand(32, generator=g)
    rays_d = torch.randn((N + S - 1) // S, 3, generator=g) * 1.7
    return dec, decoder_params(dec), feats, mask, rays_d


@pytest.mark.parametrize("N,S,masked", [(128, 128, False), (128 * 37 + 5, 64, True), (4096 * 5 + 77, 16, True), (128 * 9, 100, False),
                                        (128 * 700 + 3, 128, False)])
def test_four_tiles_in_flight_forward_equals_one_sample_per_ray_forward(N, S, masked):
    """The forward with four tiles in flight (in-place operand tiles, layer 2 folded into its consumers, the SH term of layer 3
    added per ray in fp32) against the same samples restated one per ray (S = 1 < kMinS4: each sample gets its ray's direction
    and flag), which snrf_decoder_fwd runs on the two-tile kernel.  Both kernels normalise the direction per sample, so the
    heads agree (the SH term is exact instead of split-compensated, everything else is the same arithmetic): level-major and
    row-major inputs, ragged last tile, rays masked out, tiles that straddle many rays."""
    load_pkg()
    from hashgrid import _field
    dec, params, feats, mask, rays_d = _decoder_and_inputs(N, S, N + 3)
    dev = "cuda:0"
    valid = (torch.rand(rays_d.shape[0], generator=torch.Generator().manual_seed(1)) < 0.7).to(dev) if masked else None
    pd = [p.to(dev) for p in params]
    d, m = rays_d.to(dev), mask.to(dev)
    d1 = d.repeat_interleave(S, 0)[:N]
    valid1 = valid.repeat_interleave(S)[:N] if masked else None
    for lm in (False, True):
        f = feats.to(dev)
        if lm:
            f = f.reshape(N, 16, 2).permute(1, 0, 2).contiguous()
        a = _field.decoder_forward(f, m, d1, 1, pd, valid1)
        b = _field.decoder_forward(f, m, d, S, pd, valid)
        torch.cuda.synchronize()
        if valid is not None:
            a, b = a[valid1], b[valid1]
        assert bool(torch.isfinite(b).all())
        assert float((a - b).abs().max()) < 2e-5, (lm, float((a - b).abs().max()))


@pytest.mark.parametrize("split", [True, False])
@pytest.mark.parametrize("N,S", [(128, 128), (1000, 8), (128 * 37 + 5, 64)])
def test_decoder_forward_matches_torch(N, S, split):
    load_pkg()
    from hashgrid import _field
    dec, params, feats, mask, rays_d = _decoder_and_inputs(N, S, N)
    dirs = rays_d.repeat_interleave(S, 0)[:N]
    with torch.no_grad():
        ref = dec(torch.cat([feats, dirs], -1), weight_feature=mask)
    dev = "cuda:0"
    _field.set_precision(split)
    try:
        out = _field.decoder_forward(feats.to(dev), mask.to(dev), rays_d.to(dev), S, [p.to(dev) for p in params]).cpu()
    finally:
        _field.set_precision(True)
    got = {"sigma": out[:, 0:1], "tint": out[:, 1:4], "diffuse": out[:, 4:7], "specular": out[:, 7:10]}
    # split (hi + lo, three products) operands: fp32-grade, bar 1e-4 absolute on every head (so composited RGB stays within 1e-4);
    # plain (hi only) operands: the Gaussian activations amplify the operand rounding to ~1 %
    max_tol, rel_tol = (1e-4, 5e-5) if split else (4e-2, 2e-2)
    for k in got:
        err = float((got[k] - ref[k]).abs().max())
        mean_rel = float((got[k] - ref[k]).abs().mean() / ref[k].abs().mean())
        print(f"decoder fwd split={split} {k}: max abs err {err:.2e}, mean rel err {mean_rel:.2e}")
        assert err < max_tol, f"{k}: max abs err {err}"
        assert mean_rel < rel_tol, f"{k}: mean relative err {mean_rel}"


@pytest.mark.parametrize("inputs", ["row_major", "level_major", "masked"])
@pytest.mark.parametrize("split", [True, False])
@pytest.mark.parametrize("N,S", [(128, 128), (128 * 5 + 17, 32), (4096 * 3, 128)])
def test_decoder_backward_matches_torch(N, S, split, inputs):
    """The backward (layer 2 folded into its consumers: six dependent stages per tile, dW2 / dW3a / dW_heads / db2 composed
    per CTA) against fp32 torch autograd.  inputs: row-major features [N,32]; level-major features [16,N,2] (the layout of the
    field encode); row-major with every third ray masked out (its samples get no gradient, their grad_feats rows are not
    compared; at S = 128 such a tile has no live sample)."""
    load_pkg()
    from hashgrid import _field
    dec, params, feats, mask, rays_d = _decoder_and_inputs(N, S, N + 1)
    g = torch.Generator().manual_seed(3)
    cot = torch.randn(N, 10, generator=g)
    valid = live = None
    if inputs == "masked":
        valid = torch.arange(rays_d.shape[0]) % 3 != 1
        live = valid.repeat_interleave(S)[:N]
    # torch reference (fp32, CPU)
    f_ref = feats.clone().requires_grad_(True)
    d_ref = rays_d.clone().requires_grad_(True)
    o = dec(torch.cat([f_ref, d_ref.repeat_interleave(S, 0)[:N]], -1), weight_feature=mask)
    ref_heads = torch.cat([o["sigma"], o["tint"], o["diffuse"], o["specular"]], -1)
    (ref_heads * (cot if live is None else cot * live[:, None])).sum().backward()
    # tensor-core path
    dev = "cuda:0"
    f_in = feats.reshape(N, 16, 2).permute(1, 0, 2).contiguous() if inputs == "level_major" else feats
    f_gpu = f_in.to(dev).requires_grad_(True)
    d_gpu = rays_d.to(dev).requires_grad_(True)
    p_gpu = [p.detach().to(dev).requires_grad_(True) for p in params]
    _field.set_precision(split)
    try:
        heads = _field.decoder_apply(f_gpu, d_gpu, mask.to(dev), S, p_gpu, None if valid is None else valid.to(dev))
        (heads * cot.to(dev)).sum().backward()
        torch.cuda.synchronize()
    finally:
        _field.set_precision(True)

    def rel(a, b):      # relative error in the L2 sense
        return float((a.cpu() - b).norm() / b.norm().clamp_min(1e-20))
    g_feats = f_gpu.grad.permute(1, 0, 2).reshape(N, 32) if inputs == "level_major" else f_gpu.grad
    if live is None:
        errs = {"feats": rel(g_feats, f_ref.grad)}
    else:
        errs = {"feats": rel(g_feats[live.to(dev)], f_ref.grad[live])}
    errs["rays_d"] = rel(d_gpu.grad, d_ref.grad)
    for q, p in zip(p_gpu, params):
        errs[f"param{tuple(p.shape)}"] = rel(q.grad, p.grad)
    print(f"decoder bwd split={split} rel L2 errs:", {k: f"{v:.2e}" for k, v in errs.items()})
    # split: every gradient within 2e-3 (the north star's tolerance for the 16-bit operand path): the input-gradient
    # chain is error-compensated (hi + lo operands), the weight-gradient GEMMs read the fp16 hi parts of dz and of the
    # activations (2^-12 operand rounding each; round 1's bf16 activations needed a 5e-3 bar here).
    # plain (hi only) operands: the Gaussian activations amplify operand rounding.
    for k, v in errs.items():
        tol = 2e-3 if split else 2e-1
        assert v < tol, f"{k}: {v}"


@pytest.mark.parametrize("scale", [1e-9, 1.0, 3e4])
def test_decoder_backward_is_scale_invariant(scale):
    """The fp16 gradient operands are range-managed by a power-of-two scale taken from max |grad_heads|: the backward of
    `scale * cot` must be `scale` times the backward of `cot` (to rounding) from 1e-9 to 3e4, and a cotangent whose rows
    span twelve orders of magnitude keeps the 2e-3 bar against fp32 torch."""
    load_pkg()
    from hashgrid import _field
    N, S = 128 * 6 + 5, 32
    dec, params, feats, mask, rays_d = _decoder_and_inputs(N, S, 77)
    g = torch.Generator().manual_seed(5)
    cot = torch.randn(N, 10, generator=g) * (10.0 ** (-12.0 * torch.rand(N, 1, generator=g)))      # per-sample magnitudes 1 .. 1e-12
    f_ref = feats.clone().requires_grad_(True)
    d_ref = rays_d.clone().requires_grad_(True)
    o = dec(torch.cat([f_ref, d_ref.repeat_interleave(S, 0)[:N]], -1), weight_feature=mask)
    (torch.cat([o["sigma"], o["tint"], o["diffuse"], o["specular"]], -1) * cot).sum().backward()
    dev = "cuda:0"
    f_gpu = feats.to(dev).requires_grad_(True)
    d_gpu = rays_d.to(dev).requires_grad_(True)
    p_gpu = [p.detach().to(dev).requires_grad_(True) for p in params]
    heads = _field.decoder_apply(f_gpu, d_gpu, mask.to(dev), S, p_gpu)
    (heads * (cot * scale).to(dev)).sum().backward()
    torch.cuda.synchronize()

    def rel(a, b):
        return float((a.cpu() / scale - b).norm() / b.norm().clamp_min(1e-30))
    errs = {"feats": rel(f_gpu.grad, f_ref.grad), "rays_d": rel(d_gpu.grad, d_ref.grad)}
    for q, p in zip(p_gpu, params):
        errs[f"param{tuple(p.shape)}"] = rel(q.grad, p.grad)
    assert all(torch.isfinite(q.grad).all() for q in p_gpu) and torch.isfinite(f_gpu.grad).all()
    for k, v in errs.items():
        assert v < 2e-3, f"{k}: {v} at scale {scale}"
