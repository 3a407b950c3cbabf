"""GPU: edge cases of the operator surface -- empty batches (every op is a no-op and raises nothing),
ragged sizes (sample counts that are not multiples of a warp; the field evaluation's ragged batches are
cases of test_render_gpu.py::test_pts_inference_against_cpu_restatement), argument validation
(dtype / device / shape errors are raised on the host, before any launch)."""
import numpy as np
import pytest
import torch

from conftest import load_pkg
from test_render_gpu import dev, make_rays, make_scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def z(*shape, dtype=torch.float32):
    return torch.zeros(*shape, dtype=dtype, device=DEV)


def test_empty_batches_are_noops():
    load_pkg()
    import cuda as C
    from hashgrid.lib import HASHGRID as H
    sc = dev(make_scene(2))
    nb = 2
    Ks, C2Ws = z(3, 9), z(3, 12)
    C.compute_ray_forward(z(0, 3), z(0, 3), Ks, C2Ws, z(0, 3, dtype=torch.int32))
    g = z(3, 12)
    C.compute_ray_backward(z(0, 3), z(0, 3), Ks, g, z(0, 3, dtype=torch.int32))
    assert float(g.abs().max()) == 0.0
    C.ray_aabb_intersection(z(0, 3), z(0, 3), z(3), torch.ones(3, device=DEV), z(0, 2))
    occ = torch.ones(8, 4, 8, dtype=torch.bool, device=DEV)
    C.sample_points_grid(z(0, 3), z(0, 3), z(0, 16), z(0, 16), z(3), torch.ones(3, device=DEV), occ,
                         torch.tensor([3, 2, 3], dtype=torch.int32, device=DEV))
    p = z(0, 8)
    C.adam_step_sparse(p, z(0, 8), z(0, 8), z(0, 8), 1e-3, 0.9, 0.99, 1e-15, 1)
    # render stages
    H.ray_block_intersection(z(0, 3), z(0, 3), sc["corners"], sc["sizes"], z(0, nb, 2))
    H.prepare_points(z(0, 8), z(0, 1, dtype=torch.bool), z(0, nb, 2), z(0, 8, 4, dtype=torch.int16))
    H.pts_inference(z(0, 3), z(0, 3), z(0, 8), z(0, 8), z(0, 8, 4, dtype=torch.int16), sc["tables"], sc["params"], sc["res"], sc["occ"],
                    sc["starts"], sc["l2d"], sc["corners"], sc["sizes"], z(0, 8, 3), z(0, 8, 3), z(0, 8, 1))
    H.bg_pts_inference_v2(z(0, 3), z(0, 3), z(0, 8), z(0, 4, dtype=torch.int16), 0, sc["corners"], sc["sizes"], sc["res"], sc["tables"],
                          sc["params"], z(0, 8, 3), z(0, 8, 3), z(0, 8, 1))
    H.bg_pts_inference(z(0, 3), z(0, 3), z(0, 8), z(0, 4, dtype=torch.int16), z(0, 4), sc["corners"], sc["sizes"], sc["res"], sc["tables"],
                       sc["params"], z(0, 8, 3), z(0, 8, 3), z(0, 8, 1))
    H.accumulate_color(z(0, 8, 3), z(0, 8, 3), z(0, 8, 1), z(0, 1), z(0, 8), z(0, 3), z(0, 3), z(0, 1))
    H.inverse_z_sampling(z(0, nb, 2), z(0, dtype=torch.int16), z(0, 8), 1e6)
    H.get_last_block(z(0, nb, dtype=torch.int32), z(0, dtype=torch.int32), z(0, nb, 2))
    H.update_outgoing_bidx(z(0, 3), z(0, 3), sc["corners"], sc["sizes"], z(0, nb, dtype=torch.int32), z(0, nb, 2),
                           z(0, 4, dtype=torch.int16), z(0, 4), 0.12, False)
    # hash encode
    out = z(0, 16, 2)
    H.embedding_bg_forward_cuda(z(0, 3), out, sc["tables"][0].float().contiguous(), sc["res"][0].contiguous())
    torch.cuda.synchronize()


def test_background_slot_leaves_rows_of_rays_without_a_tile():
    load_pkg()
    from hashgrid.lib import HASHGRID as H
    nb, B, S = 3, 77, 13
    sc = dev(make_scene(nb, seed=5))
    o, d = (t.to(DEV) for t in make_rays(B, 9))
    zv = (torch.rand(B, S, generator=torch.Generator().manual_seed(1)) * 30 + 1).sort(-1)[0].to(DEV).contiguous()
    ids = torch.randint(-1, nb, (B, 4), generator=torch.Generator().manual_seed(2)).to(torch.int16).to(DEV)
    outs = [torch.full((B, S, 3), 7.0, device=DEV), torch.full((B, S, 3), 7.0, device=DEV), torch.full((B, S, 1), 7.0, device=DEV)]
    H.bg_pts_inference_v2(o, d, zv, ids, 2, sc["corners"], sc["sizes"], sc["res"], sc["tables"], sc["params"], *outs)
    torch.cuda.synchronize()
    skip = ids[:, 2] == -1
    assert skip.any() and (~skip).any()
    assert bool((outs[2][skip] == 7.0).all()) and bool((outs[0][skip] == 7.0).all())
    assert bool((outs[2][~skip] != 7.0).all())
    assert bool(((outs[2][~skip] >= 0) & (outs[2][~skip] <= 1)).all())


def test_accumulate_ragged_sample_counts():
    """accumulate_color with S = 1, 33, 100 (not multiples of the 32-sample stage) against the sequential definition."""
    load_pkg()
    from hashgrid.lib import HASHGRID as H
    from oracle import render_ref as rr
    for S in (1, 33, 100):
        g = torch.Generator().manual_seed(S)
        B = 50
        pd, ps = torch.rand(B, S, 3, generator=g), torch.rand(B, S, 3, generator=g)
        pa = torch.rand(B, S, 1, generator=g) * 0.3
        zv = torch.rand(B, S, generator=g).sort(-1)[0]
        T = torch.rand(B, 1, generator=g)
        T[::7] = 1e-6                                          # finished rays are skipped
        dif, spe, dep = torch.rand(B, 3, generator=g), torch.rand(B, 3, generator=g), torch.rand(B, 1, generator=g)
        wT, wd, ws, wz = rr.accumulate_color(pd.numpy(), ps.numpy(), pa.numpy(), T.numpy(), zv.numpy(), dif.numpy(), spe.numpy(), dep.numpy())
        a = [t.to(DEV).contiguous() for t in (pd, ps, pa, T, zv, dif, spe, dep)]
        H.accumulate_color(*a)
        torch.cuda.synchronize()
        assert np.allclose(a[3].cpu().numpy(), wT, rtol=1e-5, atol=1e-7)
        assert np.allclose(a[5].cpu().numpy(), wd, rtol=1e-5, atol=1e-6) and np.allclose(a[6].cpu().numpy(), ws, rtol=1e-5, atol=1e-6)
        assert np.allclose(a[7].cpu().numpy(), wz, rtol=1e-5, atol=1e-6)


def test_argument_validation():
    load_pkg()
    import cuda as C
    from hashgrid.lib import HASHGRID as H
    sc = dev(make_scene(1))
    with pytest.raises((TypeError, RuntimeError, ValueError)):       # wrong dtype
        C.compute_ray_forward(z(4, 3), z(4, 3), z(3, 9), z(3, 12), z(4, 3))          # locs must be int32
    with pytest.raises((TypeError, RuntimeError, ValueError)):       # host tensor
        C.ray_aabb_intersection(torch.zeros(4, 3), z(4, 3), z(3), z(3), z(4, 2))
    with pytest.raises(RuntimeError):                                # params of the wrong width
        H.pts_inference(z(1, 3), z(1, 3), z(1, 8), z(1, 8), z(1, 8, 4, dtype=torch.int16), sc["tables"], z(1, 100), sc["res"], sc["occ"],
                        sc["starts"], sc["l2d"], sc["corners"], sc["sizes"], z(1, 8, 3), z(1, 8, 3), z(1, 8, 1))
    with pytest.raises(RuntimeError):                                # table size not a power of two
        H.pts_inference(z(1, 3), z(1, 3), z(1, 8), z(1, 8), z(1, 8, 4, dtype=torch.int16), z(1, 16, 1000, 2, dtype=torch.float16), sc["params"],
                        sc["res"], sc["occ"], sc["starts"], sc["l2d"], sc["corners"], sc["sizes"], z(1, 8, 3), z(1, 8, 3), z(1, 8, 1))
    with pytest.raises(RuntimeError):                                # slot out of range
        H.bg_pts_inference_v2(z(1, 3), z(1, 3), z(1, 8), z(1, 4, dtype=torch.int16), 4, sc["corners"], sc["sizes"], sc["res"], sc["tables"],
                              sc["params"], z(1, 8, 3), z(1, 8, 3), z(1, 8, 1))
    # the decoder backward takes the head activations from the forward's output: heads_fwd = NULL is rejected
    import ctypes
    import scanerf_b200_capi as capi
    from hashgrid._decoder import ShallowMLP, decoder_params
    from scanerf_b200_capi import c_int, c_void_p, ptr
    params = [p.detach().to(DEV) for p in decoder_params(ShallowMLP(32))]
    grads = [torch.zeros_like(p) for p in params]
    arr = (ctypes.c_void_p * 16)(*[p.data_ptr() for p in params])
    garr = (ctypes.c_void_p * 16)(*[g.data_ptr() for g in grads])
    N, S = 256, 128
    feats, rays_d, g_heads, g_feats = z(N, 32), z(N // S, 3), torch.ones(N, 10, device=DEV), z(N, 32)
    rc = capi.lib().snrf_decoder_bwd(ptr(feats), c_void_p(0), ptr(rays_d), arr, ptr(g_heads), ptr(g_feats), c_void_p(0), garr,
                                     c_int(N), c_int(S), c_int(0), c_void_p(0), c_void_p(0), capi.stream())
    torch.cuda.synchronize()
    assert rc != 0 and b"heads_fwd" in capi.lib().snrf_last_error()
    assert all(float(g.abs().max()) == 0.0 for g in grads)
