"""CPU tests of the colour gradients (no GPU needed).

The GPU tests of the colour gradients compare with fp64 autograd of oracle/torch_ref.py; here that reference is pinned to
central differences of a forward it does not share: the C oracle's mesh_forward (HardPhong) and render_mesh_view_soft's own
fp64 forward (SoftPhong; the C oracle has no soft forward).  Both images are linear in the colours -- the blend weights do not
depend on them -- so the differences are exact up to rounding.  Also: the new C entry points reject null pointers with a status.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import _lib, ops, synth

K00, K11 = ops.fov_projection_scale()
LIGHT = np.array([[0.3, 1.0, -0.5]], np.float32)
BG = np.array([0.2, 0.3, 0.4], np.float32)
OBJ = np.array([0.9, 0.7, 0.5], np.float32)


def _scene(oracle, faces, seed, M, per_vertex):
    v, f = synth.make_mesh(faces, seed)
    views = synth.learned_spherical_views(1, M, seed + 1)
    R, T, Cc = oracle.look_at(*(t.numpy().ravel() for t in views))
    nrm = oracle.vertex_normals(v.numpy(), f.numpy())
    rgb = np.random.default_rng(seed).random((v.shape[0], 3)).astype(np.float32) if per_vertex else OBJ.copy()
    return v, f, R, T, Cc, nrm, rgb


def _directions(rgb, seed):
    """The three unit directions of one colour, or three random directions over every per-vertex colour."""
    if rgb.size == 3:
        return [np.eye(3, dtype=np.float64)[i] for i in range(3)]
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(rgb.shape) for _ in range(3)]


@pytest.mark.parametrize("per_vertex", [False, True], ids=["object_rgb", "vertex_rgb"])
@pytest.mark.parametrize("seed", [11, 12])
def test_hard_phong_colour_gradient_of_the_restatement_matches_central_differences(oracle, seed, per_vertex):
    from oracle import torch_ref as tr
    H = W = 40
    M = 2
    v, f, R, T, Cc, nrm, rgb = _scene(oracle, 300, seed, M, per_vertex)
    voff, foff = np.array([0, v.shape[0]], np.int32), np.array([0, f.shape[0]], np.int32)
    g = np.random.default_rng(seed + 100).standard_normal((M, 3, H, W))

    def loss(c):
        o = oracle.mesh_forward(v.numpy(), f.numpy(), voff, foff, nrm, c.astype(np.float32), M, R, T, Cc, LIGHT, BG, K00, K11,
                                -1.0, H, W, 1, oracle.PERSPECTIVE_CORRECT)
        return float((o["images"].astype(np.float64) * g).sum()), o["pix_to_face"]

    _, p2f = loss(rgb)
    d = torch.float64
    leaf = torch.from_numpy(rgb).to(d).requires_grad_()
    vd = v.to(d)
    total = 0
    for m in range(M):
        col = leaf if per_vertex else leaf.expand(v.shape[0], 3)
        img, _ = tr.render_mesh_view(vd, f, torch.from_numpy(nrm).to(d), col, *(torch.from_numpy(x[m]).to(d) for x in (R, T, Cc)),
                                     torch.from_numpy(LIGHT[0]).to(d), torch.from_numpy(BG).to(d), K00, K11, H, W,
                                     p2f=torch.from_numpy(p2f[m, :, :, 0]).long())
        total = total + (img * torch.from_numpy(g[m])).sum()
    total.backward()
    grad = leaf.grad.numpy()
    assert np.abs(grad).max() > 0
    h = 0.25
    for k, e in enumerate(_directions(rgb, seed)):
        fd = (loss(rgb + h * e)[0] - loss(rgb - h * e)[0]) / (2 * h)
        an = float((grad * e).sum())
        assert abs(fd - an) <= 1e-4 * max(abs(an), 1.0), (k, fd, an)


@pytest.mark.parametrize("per_vertex", [False, True], ids=["object_rgb", "vertex_rgb"])
@pytest.mark.parametrize("seed", [21, 22])
def test_soft_phong_colour_gradient_of_the_restatement_matches_central_differences(oracle, seed, per_vertex):
    from oracle import torch_ref as tr
    H = W = 32
    K, blur, sigma, gamma = 4, 3e-3, 1e-3, 1e-2
    M = 2
    v, f, R, T, Cc, nrm, rgb = _scene(oracle, 200, seed, M, per_vertex)
    d = torch.float64
    vd, nd = v.to(d), torch.from_numpy(nrm).to(d)
    g = torch.from_numpy(np.random.default_rng(seed + 100).standard_normal((M, 4, H, W)))
    frags = []
    for m in range(M):
        fv32 = torch.from_numpy(oracle.project_perspective(v.numpy(), R[m], T[m], K00, K11))[f]
        frags.append(tr.rasterize_meshes_soft(fv32, H, W, K, blur)[0])

    def loss(c):
        out = 0
        for m in range(M):
            col = c if c.dim() == 2 else c.expand(v.shape[0], 3)
            img, _ = tr.render_mesh_view_soft(vd, f, nd, col, *(torch.from_numpy(x[m]).to(d) for x in (R, T, Cc)),
                                              torch.from_numpy(LIGHT[0]).to(d), torch.from_numpy(BG).to(d), K00, K11, H, W, K, blur,
                                              "soft_phong", sigma=sigma, gamma=gamma, p2f=frags[m])
            out = out + (img * g[m]).sum()
        return out

    leaf = torch.from_numpy(rgb).to(d).requires_grad_()
    loss(leaf).backward()
    grad = leaf.grad.numpy()
    assert np.abs(grad).max() > 0
    h = 0.25
    with torch.no_grad():
        for k, e in enumerate(_directions(rgb, seed)):
            et = torch.from_numpy(e)
            c0 = torch.from_numpy(rgb).to(d)
            fd = float(loss(c0 + h * et) - loss(c0 - h * et)) / (2 * h)
            an = float((grad * e).sum())
            assert abs(fd - an) <= 1e-8 * max(abs(an), 1.0), (k, fd, an)


def test_colour_gradient_entry_points_reject_null_pointers():
    lib = _lib.load()
    rc = lib.mvr_mesh_backward_rgb(None, None, None, 1, 1, 3, 1, 3, None, None, None, None, 0, None, 1.7, 1.7, 0.5, 64, 64, 1, 0,
                                   None, None, None, None, None, None, None, None, None, 0, None, None)
    assert rc < 0 and b"null pointer" in lib.mvr_last_error_string()
    rc = lib.mvr_mesh_soft_backward_rgb(None, None, None, 1, 1, 3, 1, 3, None, None, None, None, 0, None, None, 1.7, 1.7, 0.5, 3e-3,
                                        64, 64, 4, 0, 0, 1e-4, 1e-4, 1.0, 100.0, None, None, None, None, None, None, None, None, 0,
                                        None, None)
    assert rc < 0 and b"null pointer" in lib.mvr_last_error_string()
