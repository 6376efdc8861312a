"""CPU tests of the soft depth reference (tests/soft_depth_ref.py soft_depth_blend, PyTorch3D's SoftDepthShader verbatim) against
the closed form the CUDA kernels evaluate (mvr_mesh_soft.cu mesh_soft_depth_kernel / mesh_soft_depth_backward_kernel):

  over the valid entries k of a pixel's K-list, nearest first: p_k = sigmoid(-dists_k / sigma), c_k = sum_{j <= k} p_j,
  m_k = min(c_k, 1);  depth = sum_k (m_k - m_prev) z_k + (1 - m_last) bg;
  d/d z_k = g (m_k - m_prev);  k_end = the last entry with c_k <= 1, Z_stop = z of the next valid entry or bg;
  d/d p_j = g (z_j - Z_stop) for j <= k_end, 0 past it;  d/d dists_j = -(1 / sigma) p_j (1 - p_j) d/d p_j.

Forward and autograd gradients in fp64, with -1 holes mid-list, cumsums of exactly 1, K = 1, empty pixels, background 0."""
import numpy as np
import pytest
import torch

import soft_depth_ref

D = torch.float64


def closed_form(p2f, zbuf, dists, sigma, bg, g):
    """The kernels' per-pixel loops in fp64 -> depth (N,H,W,1), d/d zbuf, d/d dists."""
    N, H, W, K = p2f.shape
    depth = torch.zeros((N, H, W, 1), dtype=D)
    gz, gd = torch.zeros_like(zbuf), torch.zeros_like(dists)
    for n, y, x in np.ndindex(N, H, W):
        valid = [k for k in range(K) if p2f[n, y, x, k] >= 0]
        prob = {k: float(torch.sigmoid(-dists[n, y, x, k] / sigma)) for k in valid}
        c, zstop, cum = 0.0, bg, {}
        for k in valid:
            c += prob[k]
            cum[k] = c
        for k in valid:
            if cum[k] > 1.0:
                zstop = float(zbuf[n, y, x, k])
                break
        d, mprev, gg = 0.0, 0.0, float(g[n, y, x, 0])
        for k in valid:
            mk = min(cum[k], 1.0)
            d += (mk - mprev) * float(zbuf[n, y, x, k])
            gz[n, y, x, k] = gg * (mk - mprev)
            mprev = mk
            if cum[k] <= 1.0:
                gd[n, y, x, k] = -(1.0 / sigma) * prob[k] * (1.0 - prob[k]) * gg * (float(zbuf[n, y, x, k]) - zstop)
        depth[n, y, x, 0] = d + (1.0 - mprev) * bg
    return depth, gz, gd


def fragments(seed, N=2, H=5, W=6, K=4, sigma=1e-4):
    """Random K-lists with -1 holes (anywhere in the list, as clipped faces leave them) and signed distances around the
    sigmoid's active range."""
    gen = torch.Generator().manual_seed(seed)
    p2f = torch.randint(-1, 5, (N, H, W, K), generator=gen)
    zbuf = torch.where(p2f >= 0, 1 + 3 * torch.rand(N, H, W, K, dtype=D, generator=gen), torch.full((N, H, W, K), -1.0, dtype=D))
    dists = torch.where(p2f >= 0, 2 * sigma * torch.randn(N, H, W, K, dtype=D, generator=gen), torch.full((N, H, W, K), -1.0, dtype=D))
    return p2f, zbuf, dists


def check(p2f, zbuf, dists, sigma, bg, seed=0):
    zbuf, dists = zbuf.clone().requires_grad_(), dists.clone().requires_grad_()
    out = soft_depth_ref.soft_depth_blend(p2f, zbuf, dists, sigma, bg)
    g = torch.randn(out.shape, dtype=D, generator=torch.Generator().manual_seed(seed + 100))
    out.backward(g)
    ref, gz, gd = closed_form(p2f, zbuf.detach(), dists.detach(), sigma, bg, g)
    assert torch.allclose(out.detach(), ref, rtol=1e-12, atol=1e-12 * max(abs(bg), 1.0)), float((out.detach() - ref).abs().max())
    assert torch.allclose(zbuf.grad, gz, rtol=1e-12, atol=1e-14)
    scale = max(float(gd.abs().max()), 1.0)
    assert float((dists.grad - gd).abs().max()) <= 1e-12 * scale, float((dists.grad - gd).abs().max())
    return out.detach(), zbuf.grad, dists.grad


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_lists_with_holes(seed):
    p2f, zbuf, dists = fragments(seed)
    assert ((p2f[..., :-1] < 0) & (p2f[..., 1:] >= 0)).any(), "no hole in front of a valid entry"
    check(p2f, zbuf, dists, 1e-4, 100.0, seed)


def test_cumsum_of_exactly_one():
    """Probabilities of exactly 0.5 (dists 0) reach c = 1 exactly; torch's clamp passes the gradient at c = 1, so the entry
    that reaches 1 is still <= k_end.  Pixel 0: Z_stop is the entry after it; pixel 1: the list ends there (hole in between),
    so Z_stop is the background."""
    sigma = 1e-3
    p2f = torch.tensor([[[[3, -1, 5, 7, 2], [1, -1, 3, -1, -1]]]])
    zbuf = torch.tensor([[[[1.5, -1.0, 2.0, 2.5, 3.0], [1.0, -1.0, 1.4, -1.0, -1.0]]]], dtype=D)
    dists = torch.tensor([[[[0.0, -1.0, 0.0, 1e-4, -1e-4], [0.0, -1.0, 0.0, -1.0, -1.0]]]], dtype=D)
    prob = torch.sigmoid(-dists / sigma)
    assert float(prob[0, 0, 0, 0] + prob[0, 0, 0, 2]) == 1.0 and float(prob[0, 0, 1, 0] + prob[0, 0, 1, 2]) == 1.0
    out, gz, gd = check(p2f, zbuf, dists, sigma, 100.0)
    # the entries after the one reaching 1 get neither weight nor a probability gradient
    assert float(gz[0, 0, 0, 3]) == 0.0 and float(gd[0, 0, 0, 3]) == 0.0 and float(gd[0, 0, 0, 4]) == 0.0
    assert float(gd[0, 0, 0, 2]) != 0.0 and float(gd[0, 0, 1, 2]) != 0.0
    assert float(out[0, 0, 1, 0]) == 0.5 * 1.0 + 0.5 * 1.4


def test_k1():
    p2f, zbuf, dists = fragments(3, K=1)
    check(p2f, zbuf, dists, 1e-4, 100.0)


def test_empty_pixels_hold_the_background_with_zero_gradient():
    N, H, W, K = 1, 3, 4, 3
    p2f = torch.full((N, H, W, K), -1)
    zbuf, dists = torch.full((N, H, W, K), -1.0, dtype=D), torch.full((N, H, W, K), -1.0, dtype=D)
    out, gz, gd = check(p2f, zbuf, dists, 1e-4, 7.5)
    assert torch.equal(out, torch.full_like(out, 7.5))
    assert float(gz.abs().max()) == 0.0 and float(gd.abs().max()) == 0.0


def test_background_zero():
    p2f, zbuf, dists = fragments(4)
    p2f[0, 0] = -1      # a row of empty pixels
    out, _, _ = check(p2f, zbuf, dists, 1e-4, 0.0)
    empty = (p2f < 0).all(-1)
    assert empty.any() and bool((out[..., 0][empty] == 0).all())


def test_pytorch3d_soft_depth_shader_on_the_same_fragments():
    """PyTorch3D's own SoftDepthShader, where it is installed."""
    pytest.importorskip("pytorch3d")
    from pytorch3d.renderer import BlendParams, FoVPerspectiveCameras
    from pytorch3d.renderer.mesh.rasterizer import Fragments
    from pytorch3d.renderer.mesh.shader import SoftDepthShader
    p2f, zbuf, dists = fragments(5)
    bary = torch.zeros(p2f.shape + (3,), dtype=D)
    frag = Fragments(pix_to_face=p2f, zbuf=zbuf, bary_coords=bary, dists=dists)
    shader = SoftDepthShader(cameras=FoVPerspectiveCameras(), blend_params=BlendParams(sigma=1e-4))
    got = shader(frag, None, zfar=100.0)
    want = soft_depth_ref.soft_depth_blend(p2f, zbuf, dists, 1e-4, 100.0)
    assert torch.allclose(got.to(D), want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("near", [False, True])
def test_restatement_on_given_projection_is_render_mesh_view_soft(near):
    """render_mesh_view_soft_depth(ndc=project_perspective(verts)) recomputes the fragments the way torch_ref.render_mesh_view_soft
    does: the same depth and the same gradients w.r.t. vertices and camera, near-plane clipping included."""
    from mvtn_b200 import ops, synth
    from oracle import torch_ref as tr
    k00, k11 = ops.fov_projection_scale()
    v, f = synth.make_mesh(300, 281 if near else 24)
    dist = 1.12 if near else 2.2
    R, T, _ = tr.look_at_view_transform(torch.tensor([dist]), torch.tensor([10.0]), torch.tensor([15.0]))
    z_clip = 0.5 if near else None
    out = []
    for given in (False, True):
        vd = v.to(D).requires_grad_()
        Rr, Tr = R[0].to(D).requires_grad_(), T[0].to(D).requires_grad_()
        ndc = tr.project_perspective(vd, Rr, Tr, k00, k11) if given else None
        dep, frag = soft_depth_ref.render_mesh_view_soft_depth(vd, f, Rr, Tr, k00, k11, 32, 32, 6, 3e-3, sigma=1e-3, background=4.0,
                                                          z_clip=z_clip, ndc=ndc)
        (dep * torch.linspace(-1, 1, 32 * 32, dtype=D).view(32, 32)).sum().backward()
        out.append((dep.detach(), frag["pix_to_face"], vd.grad, Rr.grad, Tr.grad))
    assert int((out[0][1] >= 0).sum()) > 50
    for a, b in zip(*out):
        assert torch.equal(a, b)
