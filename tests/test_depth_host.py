"""CPU tests of the hard depth shader (no GPU needed).

The GPU tests of shader="hard_depth" compare with fp64 autograd of the depth restatements of tests/depth_ref.py; here those
restatements are pinned to the C oracle: their forward to its zbuf[..., 0] (clipped case included), their gradient to its
rasterizer backwards (rasterize_meshes_backward / rasterize_points_backward with grad_zbuf = the depth cotangent) chained through
the projection.  Also: the new C entry points reject bad arguments with a status, and the options the depth cannot honour raise.
"""
import numpy as np
import pytest
import torch

import depth_ref
from mvtn_b200 import _lib, ops, synth

K00, K11 = ops.fov_projection_scale()
BGD = 100.0
D = torch.float64


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-12))


# (faces, seed, views (azim, elev, dist), perspective_correct, cull, z_clip)
MESH_CASES = {
    "persp": (600, 3, None, True, False, None),
    "no_persp_cull": (600, 4, None, False, True, None),
    "near_plane": (260, 5, ([15.0, 140.0, -80.0], [10.0, -35.0, 50.0], [1.15, 1.22, 1.3]), True, False, 0.5),
}


def _mesh_scene(oracle, name):
    nf, seed, views, persp, cull, z_clip = MESH_CASES[name]
    v, f = synth.make_mesh(nf, seed)
    if views is None:
        az, el, di = (t.numpy().ravel() for t in synth.learned_spherical_views(1, 3, seed + 1))
    else:
        az, el, di = (np.array(x, np.float32) for x in views)
    R, T, C = oracle.look_at(az, el, di)
    flags = (oracle.PERSPECTIVE_CORRECT if persp else 0) | (oracle.CULL_BACKFACES if cull else 0)
    return v, f, R, T, C, flags, persp, cull, z_clip


@pytest.mark.parametrize("name", list(MESH_CASES))
def test_mesh_depth_restatement_matches_oracle_zbuf(oracle, name):
    v, f, R, T, C, flags, persp, cull, z_clip = _mesh_scene(oracle, name)
    H, W = 40, 48
    voff, foff = np.array([0, v.shape[0]], np.int32), np.array([0, f.shape[0]], np.int32)
    nrm = oracle.vertex_normals(v.numpy(), f.numpy())
    rgb = np.full((v.shape[0], 3), 0.5, np.float32)
    o = oracle.mesh_forward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, 3, R, T, C, np.ones((1, 3), np.float32),
                            np.zeros(3, np.float32), K00, K11, -1.0 if z_clip is None else z_clip, H, W, 1, flags)
    if z_clip is not None:
        assert o["straddle"] > 0
    mism = 0
    for n in range(3):
        # the restatement in fp32 on the oracle's IEEE projection: the same fragments and the same depth
        depth, p2f = depth_ref.render_mesh_view_depth(v, f, torch.from_numpy(R[n]), torch.from_numpy(T[n]), K00, K11, H, W, persp, cull,
                                               z_clip=z_clip, background=BGD)
        op2f = o["pix_to_face"][n, ..., 0]
        bad = p2f.numpy() != op2f
        mism += int(bad.sum())
        ok = ~bad
        want = np.where(op2f >= 0, o["zbuf"][n, ..., 0], BGD)
        assert (op2f >= 0).sum() > 50
        assert np.abs(depth.numpy()[ok] - want[ok]).max() <= 1e-5 * np.abs(want[ok & (op2f >= 0)]).max()
        assert (depth.numpy()[ok & (op2f < 0)] == BGD).all()
    assert mism <= 4      # fp32 torch vs the C oracle's written operation order: pixels a rounding error away from an edge


@pytest.mark.parametrize("name", [n for n, c in MESH_CASES.items() if c[5] is None])      # (the oracle's backward takes unclipped faces)
def test_mesh_depth_restatement_gradient_matches_oracle_rasterizer_backward(oracle, name):
    from oracle import torch_ref as tr
    v, f, R, T, C, flags, persp, cull, z_clip = _mesh_scene(oracle, name)
    H, W = 40, 48
    rng = np.random.default_rng(7)
    Rd, Td = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T))
    vd = v.to(D).requires_grad_()
    loss_ref, chain = 0, 0
    for n in range(3):
        fv32 = oracle.project_perspective(v.numpy(), R[n], T[n], K00, K11)[f.numpy()]
        p2f, _, _, _ = oracle.rasterize_meshes(fv32, np.array([0], np.int32), np.array([f.shape[0]], np.int32), H, W, 1, flags)
        g = (rng.standard_normal((H, W)) * (p2f[0, ..., 0] >= 0)).astype(np.float32)
        gfv = oracle.rasterize_meshes_backward(fv32, p2f, g[None, ..., None], np.zeros((1, H, W, 1, 3), np.float32), flags)
        fv = tr.project_perspective(vd, Rd[n], Td[n], K00, K11)[f]
        chain = chain + (fv * torch.from_numpy(gfv).to(D)).sum()
        depth, _ = depth_ref.render_mesh_view_depth(vd, f, Rd[n], Td[n], K00, K11, H, W, persp, cull,
                                             p2f=torch.from_numpy(p2f[0, ..., 0]).long(), background=BGD)
        loss_ref = loss_ref + (depth * torch.from_numpy(g).to(D)).sum()
    want = torch.autograd.grad(chain, (Rd, Td, vd))
    got = torch.autograd.grad(loss_ref, (Rd, Td, vd))
    for a, b in zip(got, want):
        assert rel(a, b) < 1e-4


def test_mesh_depth_restatement_gradient_with_clipping_matches_central_differences(oracle):
    """The near-plane clipped chain (clip_faces), which the oracle's rasterizer backward does not take: fp64 autograd of the
    restatement against its central differences, the fragments held fixed."""
    v, f, R, T, C, flags, persp, cull, z_clip = _mesh_scene(oracle, "near_plane")
    H = W = 32
    g = torch.from_numpy(np.random.default_rng(3).standard_normal((H, W)))
    Rd = torch.from_numpy(R[0]).to(D).requires_grad_()
    Td = torch.from_numpy(T[0]).to(D)
    vd = v.to(D)
    depth, p2f = depth_ref.render_mesh_view_depth(vd, f, Rd, Td, K00, K11, H, W, persp, cull, z_clip=z_clip, background=BGD)
    fg = p2f >= 0
    (gR,) = torch.autograd.grad((depth * g * fg).sum(), Rd)
    # central differences with the fragments held fixed (the depth is piecewise smooth: differentiate inside each piece)
    eps = 1e-6
    num = torch.zeros(3, 3, dtype=D)
    for i in range(3):
        for j in range(3):
            vals = []
            for s in (eps, -eps):
                Rp = Rd.detach().clone()
                Rp[i, j] += s
                dp, pp = depth_ref.render_mesh_view_depth(vd, f, Rp, Td, K00, K11, H, W, persp, cull, z_clip=z_clip, background=BGD)
                assert (pp == p2f).all()
                vals.append(float((dp * g * fg).sum()))
            num[i, j] = (vals[0] - vals[1]) / (2 * eps)
    assert rel(gR, num) < 1e-5


def _cloud_scene(oracle, seed, M=3):
    pts = synth.make_cloud(400, seed)
    az, el, di = (t.numpy().ravel() for t in synth.learned_spherical_views(1, M, seed + 1))
    R, T, _ = oracle.look_at(az, el, di)
    return pts, R, T, (1.0 / di.astype(np.float64)).astype(np.float32)


@pytest.mark.parametrize("K", [1, 4])
def test_points_depth_restatement_matches_oracle_zbuf(oracle, K):
    pts, R, T, s = _cloud_scene(oracle, 21)
    H, W, rad = 40, 40, 0.04
    o = oracle.points_forward(pts.numpy()[None], np.ones(3, np.float32), 3, R, T, s, rad, np.zeros(3, np.float32), H, W, K, 0)
    for n in range(3):
        depth, idx = depth_ref.render_points_view_depth(pts, torch.from_numpy(R[n]), torch.from_numpy(T[n]), float(s[n]), rad, H, W,
                                                 background=BGD)
        assert (idx[..., 0].numpy() == o["idx"][n, ..., 0]).all()
        want = np.where(o["idx"][n, ..., 0] >= 0, o["zbuf"][n, ..., 0], BGD)
        assert (o["idx"][n, ..., 0] >= 0).sum() > 50
        assert np.abs(depth.numpy() - want).max() <= 1e-6 * np.abs(want).max()


def test_points_depth_restatement_gradient_matches_oracle_rasterizer_backward(oracle):
    pts, R, T, s = _cloud_scene(oracle, 22)
    H, W, rad = 40, 40, 0.04
    rng = np.random.default_rng(9)
    Rd, Td = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T))
    pd = pts.to(D).requires_grad_()
    loss_ref, chain = 0, 0
    for n in range(3):
        pv = ((pts.to(D) * float(s[n])) @ Rd[n].detach() + Td[n].detach()).numpy().astype(np.float32)
        idx, _, _ = oracle.rasterize_points(pv, np.array([0], np.int32), np.array([pv.shape[0]], np.int32), rad, H, W, 1)
        g = (rng.standard_normal((H, W)) * (idx[0, ..., 0] >= 0)).astype(np.float32)
        gp = oracle.rasterize_points_backward(pv, idx, g[None, ..., None], np.zeros((1, H, W, 1), np.float32))
        p = (pd * float(s[n])) @ Rd[n] + Td[n]
        chain = chain + (p * torch.from_numpy(gp).to(D)).sum()
        depth, _ = depth_ref.render_points_view_depth(pd, Rd[n], Td[n], float(s[n]), rad, H, W, background=BGD,
                                               idx=torch.from_numpy(idx[0]).long())
        loss_ref = loss_ref + (depth * torch.from_numpy(g).to(D)).sum()
    want = torch.autograd.grad(chain, (Rd, Td, pd))
    got = torch.autograd.grad(loss_ref, (Rd, Td, pd))
    for a, b in zip(got, want):
        assert rel(a, b) < 1e-6


def test_depth_entry_points_reject_bad_arguments():
    lib = _lib.load()
    # null pointers / options the depth cannot honour: a status, before any CUDA call
    assert lib.mvr_mesh_depth_forward(None, None, None, 1, 1, 3, 1, 3, 1, None, None, 1.0, 1.0, -1.0, 100.0, 8, 8, 0, None, None,
                                      None, None, 0, None) == -5
    assert lib.mvr_mesh_depth_forward(None, None, None, 1, 1, 3, 1, 3, 1, None, None, 1.0, 1.0, -1.0, 100.0, 8, 8,
                                      _lib.IMAGES_BF16, None, None, None, None, 0, None) == -11
    assert lib.mvr_mesh_depth_backward(None, None, None, 1, 1, 3, 1, 3, None, None, 1.0, 1.0, -1.0, 8, 8, 0, None, None, None,
                                       None, None, None, 0, None) == -5
    assert lib.mvr_points_depth_forward(None, 1, 4, 1, None, None, None, 0.01, 100.0, 8, 8, 0, None, None, None, None, 0, None) == -6
    assert lib.mvr_points_depth_forward(None, 1, 4, 1, None, None, None, 0.0, 100.0, 8, 8, 0, None, None, None, None, 0, None) == -4
    assert lib.mvr_points_depth_backward(None, 1, 4, 1, None, None, None, 0.01, 8, 8, 0, None, None, None, None, None, None, None,
                                         None, 0, None) == -6


def test_depth_shader_rejects_options():
    from mvtn_b200 import MVRenderer
    for kw in (dict(normalize=((0.5,) * 3, (0.2,) * 3)), dict(out_dtype=torch.bfloat16), dict(blur_radius=1e-4)):
        with pytest.raises(ValueError):
            MVRenderer(4, shader="hard_depth", **kw)
    with pytest.raises(ValueError):
        ops._check_depth_options(None, torch.bfloat16)
