"""CPU tests of the oracle (oracle/mvr_oracle.c): analytic known-answer vectors (G1-G4 of SURVEY 8c), an
exact-rational rasterizer written here, the independent torch restatement (oracle/torch_ref.py),
torch.autograd for every hand-derived backward, and the committed golden hashes (G5).

PARITY UNPINNED: the reference holds no tests or fixtures for this path and PyTorch3D is absent, so
these vectors are derived from the published algorithm, not from reference outputs.
"""
import hashlib
import math
import os
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import torch_ref as tr
from mvtn_b200 import synth
from mvtn_b200.ops import fov_projection_scale
from conftest import GOLDEN

K00, K11 = fov_projection_scale()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def rel(a, b, floor=1e-6):
    """max |a-b| relative to the largest reference magnitude (floored: NormWeighted K=1 has ~0 gradients)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), floor))


# ------------------------------------------------------------------------------------------- G1 cameras
def test_look_at_axis_aligned_kat(oracle):
    # azim=0, elev=0, dist=2.2 => C=(0,0,2.2), R=diag(-1,1,-1), T=(0,0,2.2)  (SURVEY 8c.2)
    R, T, C = oracle.look_at([0.0], [0.0], [2.2])
    assert np.allclose(C[0], [0, 0, 2.2], atol=1e-7)
    assert np.allclose(R[0], np.diag([-1.0, 1.0, -1.0]), atol=1e-7)
    assert np.allclose(T[0], [0, 0, 2.2], atol=1e-6)
    # azim=90 => camera on +X looking at the origin: world origin maps to view (0,0,d)
    R, T, C = oracle.look_at([90.0], [0.0], [3.0])
    assert np.allclose(C[0], [3, 0, 0], atol=1e-6)
    assert np.allclose(np.zeros(3) @ R[0] + T[0], [0, 0, 3], atol=1e-6)
    # a point between camera and origin is nearer (smaller view z); +Y stays up
    assert (np.array([1.0, 0, 0]) @ R[0] + T[0])[2] == pytest.approx(2.0, abs=1e-6)
    assert (np.array([0, 1.0, 0]) @ R[0] + T[0])[1] == pytest.approx(1.0, abs=1e-6)


@pytest.mark.parametrize("views", [synth.circular_views(1, 12), synth.circular_views(1, 12, 35.0),
                                   synth.spherical_views(1, 12), synth.spherical_views(1, 20)])
def test_look_at_view_grids_are_rotations(oracle, views):
    az, el, di = (t.numpy().ravel() for t in views)
    R, T, C = oracle.look_at(az, el, di)
    assert oracle.count_invalid_rotations(R) == 0
    for i in range(len(az)):
        assert np.allclose(R[i] @ R[i].T, np.eye(3), atol=1e-6)
        assert np.linalg.det(R[i]) == pytest.approx(1.0, abs=1e-5)
        assert np.allclose(np.linalg.norm(C[i]), di[i], rtol=1e-6)
        assert np.allclose(-C[i] @ R[i], T[i], atol=1e-6)        # T = -R^T C
        assert np.allclose(T[i], [0, 0, di[i]], atol=1e-5)          # look-at-origin: origin on the optical axis


def test_spherical_grid_matches_reference_layout():
    # SURVEY 8c G1: 12 views -> elev {-60 x3, 0 x6, 60 x3}; 20 views -> {-67.5 x3, -22.5 x7, 22.5 x7, 67.5 x3}
    _, e12 = synth.unit_spherical_grid(12)
    assert sorted(np.round(e12, 3).tolist()) == [-60.0] * 3 + [0.0] * 6 + [60.0] * 3
    _, e20 = synth.unit_spherical_grid(20)
    assert sorted(np.round(e20, 3).tolist()) == [-67.5] * 3 + [-22.5] * 7 + [22.5] * 7 + [67.5] * 3


def test_look_at_matches_torch_restatement(oracle):
    g = torch.Generator().manual_seed(0)
    az = torch.rand(200, generator=g) * 360 - 180
    el = torch.rand(200, generator=g) * 178 - 89
    di = torch.rand(200, generator=g) * 3 + 1
    R, T, C = oracle.look_at(az.numpy(), el.numpy(), di.numpy())
    R2, T2, C2 = tr.look_at_view_transform(di, el, az)
    assert np.abs(R - R2.numpy()).max() < 5e-6
    assert np.abs(T - T2.numpy()).max() < 5e-6
    assert np.abs(C - C2.numpy()).max() < 5e-6


def test_look_at_backward_matches_autograd(oracle):
    g = torch.Generator().manual_seed(1)
    az = (torch.rand(64, generator=g) * 360 - 180).double().requires_grad_()
    el = (torch.rand(64, generator=g) * 170 - 85).double().requires_grad_()
    di = (torch.rand(64, generator=g) * 3 + 1).double().requires_grad_()
    gR = torch.randn(64, 3, 3, generator=g).double(); gT = torch.randn(64, 3, generator=g).double()
    gC = torch.randn(64, 3, generator=g).double()
    R, T, C = tr.look_at_view_transform(di, el, az)
    # R, T and C are separate outputs of the oracle's look_at: reproduce that graph (C detached from R, T)
    ((R * gR).sum() + (T * gT).sum() + (C * gC).sum()).backward()
    ga, ge, gd = oracle.look_at_backward(az.detach().numpy(), el.detach().numpy(), di.detach().numpy(),
                                         gR.numpy(), gT.numpy(), gC.numpy())
    assert rel(ga, az.grad.numpy()) < 1e-5
    assert rel(ge, el.grad.numpy()) < 1e-5
    assert rel(gd, di.grad.numpy()) < 1e-5


POLE_COT_K = 64      # conditioning bar: |a - b| <= POLE_COT_K * eps_fp32 * (largest intermediate cotangent of the view)


def pole_views(n_az=9):
    """Elevations at and next to the poles, each at n_az azimuths: exactly +-90 and +-270 (the fp32 x axis is clamped and
    replaced), a few fp32 ulps either side of 90 (clamped, not replaced: the guard must flag them), 89.999 and 89.99 (ill
    conditioned, not clamped) and 89 / 0 as controls."""
    f = np.float32
    ulp = np.spacing(f(90))
    els = [90.0, -90.0, 270.0, -270.0, 89.999, -89.999, 89.99, -89.99, 89.0, 0.0] + \
          [float(f(90) + k * ulp) for k in (-3, -1, 1, 3)]
    az = np.linspace(-180, 180, n_az, endpoint=False).astype(f) + f(7.5)
    return (np.repeat(az[None], len(els), 0).ravel(), np.repeat(np.array(els, f), n_az), np.full(len(els) * n_az, 2.2, f))


def test_look_at_backward_at_the_poles_matches_fp32_autograd(oracle):
    """At elevation +-90 the fp32 forward and a double one take different branches (fp32 cos(fp32(pi/2)) = -4.4e-8, double
    6e-17: the y normalisation is clamped in double only), and the fp32 angle lies on the other side of the pole.  The
    oracle's double backward follows the fp32 forward's branches and there its rounded angles, so it differentiates what
    fp32 PyTorch3D computes.  The chain builds cotangents of 1e7 there that cancel to O(1): fp32 autograd is held to
    POLE_COT_K eps_fp32 times the view's largest intermediate cotangent (fp32 autograd lands within 31 of them on the pole
    views of these tests), which is tight for d azim and d dist (small cotangents reach them) and loose for d elev at the
    pole, where the fp32 result is rounding noise of that size."""
    az, el, di = pole_views()
    n = az.size
    g = torch.Generator().manual_seed(11)
    gR, gT, gC = torch.randn(n, 3, 3, generator=g), torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g)
    ta, te, td, cot = tr.look_at_backward_fp32(*(torch.from_numpy(t) for t in (di, el, az)), gR, gT, gC)
    ga, ge, gd = oracle.look_at_backward(az, el, di, gR.numpy(), gT.numpy(), gC.numpy())
    R, _, _ = oracle.look_at(az, el, di)
    valid = np.array([oracle.count_invalid_rotations(R[i:i + 1]) == 0 for i in range(n)])
    assert valid[np.isin(np.abs(el), [90.0, 270.0])].all()        # replaced x: a rotation, the guard lets it through
    assert not valid[np.abs(np.abs(el) - 90) < 1e-5].all() and np.isfinite(np.r_[ga, ge, gd]).all()
    bar = POLE_COT_K * np.finfo(np.float32).eps * cot.numpy().astype(np.float64)
    deg = math.pi / 180
    for mine, ref, scale in ((ta, ga, deg), (te, ge, deg), (td, gd, 1.0)):
        assert (np.abs(mine.numpy().astype(np.float64) - ref) <= bar * scale + 1e-5 * np.abs(ref).max()).all()
    # where the angles are well conditioned the plain 1e-5 bar holds
    calm = np.abs(el) <= 89.0
    for mine, ref in ((ta, ga), (te, ge), (td, gd)):
        assert rel(mine.numpy()[calm], ref[calm]) < 1e-5


def test_degenerate_elevation_is_flagged(oracle):
    # exactly-vertical view: up x z = 0 -> x axis collapses -> R is not a rotation (ops.py:156-165 guard)
    R = np.zeros((1, 3, 3), np.float32); R[0, :, 2] = [0, -1, 0]
    assert oracle.count_invalid_rotations(R) == 1
    assert oracle.count_invalid_rotations(np.eye(3, dtype=np.float32)[None]) == 0
    refl = np.diag([1.0, 1.0, -1.0]).astype(np.float32)[None]     # det = -1
    assert oracle.count_invalid_rotations(refl) == 1


# ------------------------------------------------------------------------- exact-rational mini rasterizer
def exact_cover(tri, S):
    """Strict-interior coverage of pixel centres computed with Fractions (no rounding anywhere)."""
    cov = np.zeros((S, S), bool)
    (x0, y0), (x1, y1), (x2, y2) = [(Fraction(a), Fraction(b)) for a, b in tri]
    area = (x2 - x0) * (y1 - y0) - (y2 - y0) * (x1 - x0)
    for yi in range(S):
        yf = Fraction(-1) + Fraction(2 * (S - 1 - yi) + 1, S)
        for xi in range(S):
            xf = Fraction(-1) + Fraction(2 * (S - 1 - xi) + 1, S)
            e0 = (xf - x1) * (y2 - y1) - (yf - y1) * (x2 - x1)
            e1 = (xf - x2) * (y0 - y2) - (yf - y2) * (x0 - x2)
            e2 = (xf - x0) * (y1 - y0) - (yf - y0) * (x1 - x0)
            cov[yi, xi] = all(e * area > 0 for e in (e0, e1, e2))
    return cov


@pytest.mark.parametrize("tri", [
    [(-0.5, -0.5), (0.5, -0.5), (0.0, 0.75)],          # CCW in NDC
    [(0.5, -0.5), (-0.5, -0.5), (0.0, 0.75)],          # CW (back-facing): still rendered without culling
    [(-0.875, -0.875), (0.875, -0.875), (-0.875, 0.875)],   # edges through pixel centres: strict inequality
    [(-1.5, -1.5), (1.5, -1.5), (0.0, 1.5)],           # partly off-screen
])
def test_single_triangle_coverage_kat(oracle, tri):
    S = 8
    fv = np.array([[tri[0] + (1.0,), tri[1] + (1.0,), tri[2] + (1.0,)]], np.float32)   # dyadic coords: exact in fp32
    p2f, zbuf, bary, dists = oracle.rasterize_meshes(fv, [0], [1], S, S, 1, oracle.PERSPECTIVE_CORRECT)
    want = exact_cover(tri, S)
    assert ((p2f[0, :, :, 0] == 0) == want).all()
    assert (p2f[0, :, :, 0][~want] == -1).all()
    assert np.allclose(zbuf[0, :, :, 0][want], 1.0)
    assert (zbuf[0, :, :, 0][~want] == -1).all() and (bary[0][~want] == -1).all()
    assert np.allclose(bary[0, :, :, 0][want].sum(-1), 1.0, atol=1e-6)
    assert (dists[0, :, :, 0][want] <= 0).all()          # inside => signed distance is negative


def test_pixel_grid_orientation(oracle):
    # a small triangle in the +X,+Y NDC quadrant must land top-LEFT (+X points left, +Y up: SURVEY 8c.1)
    tri = [(0.5, 0.5), (0.9, 0.5), (0.7, 0.9)]
    fv = np.array([[t + (2.0,) for t in tri]], np.float32)
    p2f, *_ = oracle.rasterize_meshes(fv, [0], [1], 16, 16, 1, 0)
    ys, xs = np.nonzero(p2f[0, :, :, 0] == 0)
    assert len(ys) > 0 and ys.max() < 8 and xs.max() < 8


def test_two_overlapping_triangles_depth_order_and_ties(oracle):
    S = 8
    big = [(-0.9, -0.9, 2.0), (0.9, -0.9, 2.0), (0.0, 0.9, 2.0)]
    near = [(-0.5, -0.5, 1.0), (0.5, -0.5, 1.0), (0.0, 0.5, 1.0)]
    fv = np.array([big, near, big], np.float32)          # face 2 duplicates face 0: exact depth tie
    p2f, zbuf, _, _ = oracle.rasterize_meshes(fv, [0], [3], S, S, 3, 0)
    cov_big = exact_cover([b[:2] for b in big], S); cov_near = exact_cover([b[:2] for b in near], S)
    both = cov_big & cov_near
    assert (p2f[0][both][:, 0] == 1).all() and (p2f[0][both][:, 1] == 0).all() and (p2f[0][both][:, 2] == 2).all()
    only = cov_big & ~cov_near
    assert (p2f[0][only][:, 0] == 0).all() and (p2f[0][only][:, 1] == 2).all() and (p2f[0][only][:, 2] == -1).all()
    assert (np.diff(zbuf[0][both], axis=-1) >= 0).all()  # ascending depth
    # K=1 keeps the SMALLER index on an exact tie (G4)
    p1, *_ = oracle.rasterize_meshes(fv[[0, 2]], [0], [2], S, S, 1, 0)
    assert set(np.unique(p1)) <= {-1, 0}


def test_backface_cull_and_degenerate_faces(oracle):
    S = 8
    ccw = [(-0.5, -0.5, 1.0), (0.5, -0.5, 1.0), (0.0, 0.75, 1.0)]
    cw = [ccw[1], ccw[0], ccw[2]]
    for tri in (ccw, cw):
        area = (tri[0][0] - tri[1][0]) * (tri[2][1] - tri[1][1]) - (tri[0][1] - tri[1][1]) * (tri[2][0] - tri[1][0])
        p, *_ = oracle.rasterize_meshes(np.array([tri], np.float32), [0], [1], S, S, 1, oracle.CULL_BACKFACES)
        assert ((p >= 0).any()) == (area > 0)            # [upstream] back_face = face_area < 0
    sliver = [(-0.5, 0.0, 1.0), (0.5, 0.0, 1.0), (0.0, 0.0, 1.0)]     # zero area
    behind = [(-0.5, -0.5, -1.0), (0.5, -0.5, 1.0), (0.0, 0.75, 1.0)]  # a vertex behind the camera: z_invalid
    for tri in (sliver, behind):
        p, *_ = oracle.rasterize_meshes(np.array([tri], np.float32), [0], [1], S, S, 1, 0)
        assert (p == -1).all()


# ------------------------------------------------------------------------------------------- G3 points
def test_single_point_radius_kat(oracle):
    S = 8   # pixel centres at +-0.125, +-0.375, ...: nearest four are at distance sqrt(2)/8 = 0.17678 from (0,0)
    pt = np.array([[0.0, 0.0, 1.0]], np.float32)
    for r, n_hit in ((0.17, 0), (0.18, 4), (0.39, 4), (0.40, 12)):   # next ring at sqrt(.125^2+.375^2) = 0.39528
        idx, zbuf, d2 = oracle.rasterize_points(pt, [0], [1], r, S, S, 1)
        assert (idx >= 0).sum() == n_hit, (r, (idx >= 0).sum())
    idx, zbuf, d2 = oracle.rasterize_points(pt, [0], [1], 0.18, S, S, 2)
    assert np.allclose(d2[idx >= 0], 2 * 0.125 ** 2) and (zbuf[idx >= 0] == 1.0).all()
    assert (idx[..., 1] == -1).all() and (d2[idx < 0] == -1).all()
    # strict inequality: radius^2 exactly equal to dist2 does not hit (dyadic values: exact in fp32)
    idx, *_ = oracle.rasterize_points(np.array([[0.125, 0.125, 1.0]], np.float32), [0], [1], 0.25, S, S, 1)
    assert (idx >= 0).sum() == 1 + 2 * 0   # only its own pixel: neighbours are at exactly 0.25
    # behind the camera
    idx, *_ = oracle.rasterize_points(np.array([[0.0, 0.0, -0.5]], np.float32), [0], [1], 0.5, S, S, 1)
    assert (idx == -1).all()


def test_duplicate_points_tie_goes_to_smaller_index(oracle):
    pts = np.array([[0.1, 0.1, 1.0], [0.1, 0.1, 1.0], [0.1, 0.1, 0.5]], np.float32)
    idx, zbuf, _ = oracle.rasterize_points(pts, [0], [3], 0.3, 8, 8, 3)
    hit = idx[0, :, :, 0] >= 0
    assert hit.any()
    assert (idx[0][hit] == [2, 0, 1]).all()


def test_compositors_kat(oracle):
    feats = np.array([[1.0, 0.0], [0.0, 1.0], [0.5, 0.5]], np.float32)     # (C=3, P=2)
    idx = np.array([0, 1], np.int32).reshape(1, 2, 1, 1)
    al = np.array([0.5, 0.25], np.float32).reshape(1, 2, 1, 1)
    norm = oracle.composite_forward(feats, al, idx, False)[0, :, 0, 0]
    assert np.allclose(norm, [0.5 / 0.75, 0.25 / 0.75, 0.5], atol=1e-6)
    alpha = oracle.composite_forward(feats, al, idx, True)[0, :, 0, 0]
    assert np.allclose(alpha, [0.5, 0.5 * 0.25, 0.5 * 0.5 + 0.5 * 0.25 * 0.5], atol=1e-6)
    # all-empty pixel -> zeros; norm clamp at 1e-4
    e = oracle.composite_forward(feats, al, -np.ones_like(idx), False)
    assert (e == 0).all()
    tiny = oracle.composite_forward(feats, al * 1e-6, idx, False)[0, :, 0, 0]
    assert np.allclose(tiny, [0.5e-6 / 1e-4, 0.25e-6 / 1e-4, 0.375e-6 / 1e-4], rtol=1e-5)


# --------------------------------------------------------------------- oracle vs independent torch restatement
@pytest.mark.parametrize("seed,faces,H,persp,cull", [(1, 300, 32, True, False), (2, 700, 40, True, True),
                                                     (3, 500, 24, False, False)])
def test_mesh_forward_matches_torch_restatement(oracle, seed, faces, H, persp, cull):
    v, f = synth.make_mesh(faces, seed)
    az, el, di = synth.learned_spherical_views(1, 4, seed)
    R, T, C = oracle.look_at(az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel())
    nrm = oracle.vertex_normals(v.numpy(), f.numpy())
    assert np.abs(nrm - tr.vertex_normals(v, f).numpy()).max() < 1e-6
    voff = np.array([0, v.shape[0]], np.int32); foff = np.array([0, f.shape[0]], np.int32)
    rgb = np.random.RandomState(seed).rand(v.shape[0], 3).astype(np.float32)
    light = np.array([[0.3, 1.0, -0.5]], np.float32); bg = np.array([0.2, 0.4, 0.6], np.float32)
    flags = (oracle.PERSPECTIVE_CORRECT if persp else 0) | (oracle.CULL_BACKFACES if cull else 0)
    o = oracle.mesh_forward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, 4, R, T, C, light, bg, K00, K11, 0.5, H, H, 2, flags)
    n_tie_free_mismatch = 0
    for n in range(4):
        Rn, Tn, Cn = (torch.from_numpy(x[n]).double() for x in (R, T, C))
        fv = tr.project_perspective(v.double(), Rn, Tn, K00, K11)[f]
        p2, zb, ba = tr.rasterize_meshes_naive(fv, H, H, 2, persp, cull)
        mism = p2.numpy() != o["pix_to_face"][n]
        n_tie_free_mismatch += int(mism.sum())
        ok = ~mism
        assert np.abs(zb.numpy()[ok] - o["zbuf"][n][ok]).max() < 1e-5
        img, _ = tr.render_mesh_view(v.double(), f, torch.from_numpy(nrm).double(), torch.from_numpy(rgb).double(), Rn, Tn, Cn,
                                     torch.from_numpy(light[0]).double(), torch.from_numpy(bg).double(), K00, K11, H, H,
                                     persp, cull, p2f=torch.from_numpy(o["pix_to_face"][n, ..., 0]).long())
        assert np.abs(img.numpy() - o["images"][n]).max() < 1e-5
    # fp64 restatement vs fp32 oracle: only pixels a rounding error away from an edge may differ
    assert n_tie_free_mismatch <= 4


def test_mesh_backward_matches_autograd(oracle):
    v, f = synth.make_mesh(300, 1)
    az = torch.tensor([10., 130., -95., 23.4]); el = torch.tensor([5., 30., 40., -60.]); di = torch.tensor([2.2, 2.0, 1.8, 3.0])
    R, T, C = oracle.look_at(az.numpy(), el.numpy(), di.numpy())
    H, M = 32, 4
    nrm = oracle.vertex_normals(v.numpy(), f.numpy())
    voff = np.array([0, v.shape[0]], np.int32); foff = np.array([0, f.shape[0]], np.int32)
    light = np.array([[0.3, 1.0, -0.5]], np.float32); bg = np.full(3, 0.99999, np.float32)
    rgb = np.random.RandomState(0).rand(v.shape[0], 3).astype(np.float32)
    o = oracle.mesh_forward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, M, R, T, C, light, bg, K00, K11, 0.5, H, H, 1,
                            oracle.PERSPECTIVE_CORRECT)
    gimg = np.random.RandomState(1).randn(M, 3, H, H).astype(np.float32)
    bw = oracle.mesh_backward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, M, R, T, C, light, K00, K11, H, H, 1,
                              oracle.PERSPECTIVE_CORRECT, o["pix_to_face"], gimg, want_verts=True)
    D = torch.float64
    Rd, Td, Cd = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T, C))
    vd = v.to(D).requires_grad_(); nd = torch.from_numpy(nrm).to(D).requires_grad_()
    loss = 0
    for n in range(M):
        img, _ = tr.render_mesh_view(vd, f, nd, torch.from_numpy(rgb).to(D), Rd[n], Td[n], Cd[n], torch.from_numpy(light[0]).to(D),
                                     torch.from_numpy(bg).to(D), K00, K11, H, H, p2f=torch.from_numpy(o["pix_to_face"][n, ..., 0]).long())
        loss = loss + (img * torch.from_numpy(gimg[n]).to(D)).sum()
    loss.backward()
    assert rel(bw["gR"], Rd.grad.numpy()) < 2e-5
    assert rel(bw["gT"], Td.grad.numpy()) < 2e-5
    assert rel(bw["gC"], Cd.grad.numpy()) < 2e-5
    assert rel(bw["grad_verts"], vd.grad.numpy()) < 5e-5
    assert rel(bw["grad_normals"], nd.grad.numpy()) < 2e-5


def test_mesh_backward_matches_finite_differences(oracle):
    """The whole hand-derived chain of the C oracle -- d image -> Phong -> barycentrics -> projection -> (dR, dT, dC) ->
    look_at backward -> d azim / elev / dist -- against central differences of its OWN forward: no torch_ref, no autograd.
    The image is one large triangle that fills every view (no silhouette, so the loss is smooth in the camera) with
    per-vertex colours and normals that are not the face normal (so interpolation, diffuse and specular terms all move)."""
    H, M = 24, 3
    v = np.array([[-9.0, -7.0, 0.3], [9.0, -7.0, -0.2], [0.0, 11.0, 0.1]], np.float32)
    f = np.array([[0, 1, 2]], np.int32)
    nrm = np.array([[0.3, 0.1, 1.0], [-0.2, 0.2, 1.0], [0.1, -0.3, 1.0]], np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    rgb = np.array([[0.9, 0.2, 0.3], [0.1, 0.8, 0.4], [0.3, 0.3, 0.9]], np.float32)
    light = np.array([[0.3, 0.2, 1.0]], np.float32); bg = np.zeros(3, np.float32)
    az0 = np.array([8.0, -12.0, 3.0]); el0 = np.array([5.0, 10.0, -7.0]); di0 = np.array([2.2, 2.6, 3.1])
    g = np.random.RandomState(3).randn(M, 3, H, H).astype(np.float32)

    def loss(az, el, di, want_grad=False):
        R, T, C = oracle.look_at(az, el, di)
        o = oracle.mesh_forward(v, f, [0, 3], [0, 1], nrm, rgb, M, R, T, C, light, bg, K00, K11, 0.5, H, H, 1, oracle.PERSPECTIVE_CORRECT)
        assert (o["pix_to_face"] == 0).all()                  # the triangle fills every view: coverage never changes
        val = float((o["images"].astype(np.float64) * g).sum())
        if not want_grad:
            return val
        b = oracle.mesh_backward(v, f, [0, 3], [0, 1], nrm, rgb, M, R, T, C, light, K00, K11, H, H, 1, oracle.PERSPECTIVE_CORRECT,
                                 o["pix_to_face"], g)
        return val, oracle.look_at_backward(az, el, di, b["gR"], b["gT"], b["gC"])

    _, (ga, ge, gd) = loss(az0, el0, di0, want_grad=True)
    for name, grad, h in (("azim", ga, 0.25), ("elev", ge, 0.25), ("dist", gd, 0.02)):
        for i in range(M):
            args = {"azim": az0.copy(), "elev": el0.copy(), "dist": di0.copy()}
            args[name][i] += h
            up = loss(args["azim"], args["elev"], args["dist"])
            args[name][i] -= 2 * h
            dn = loss(args["azim"], args["elev"], args["dist"])
            fd = (up - dn) / (2 * h)
            scale = max(abs(fd), float(np.abs(grad).max()), 1e-6)
            assert abs(grad[i] - fd) <= 2e-3 * scale, (name, i, float(grad[i]), fd)


def test_rasterize_meshes_backward_operator(oracle):
    # operator-level backward ([upstream] RasterizeMeshesBackwardCpu): grad_bary and grad_zbuf -> grad_face_verts
    g = torch.Generator().manual_seed(3)
    fv = torch.tensor([[[-0.6, -0.5, 1.0], [0.7, -0.4, 1.5], [0.1, 0.8, 2.0]],
                       [[-0.3, -0.7, 1.2], [0.5, 0.1, 0.9], [-0.6, 0.6, 1.1]]])
    H = 12
    for persp in (True, False):
        flags = oracle.PERSPECTIVE_CORRECT if persp else 0
        p2f, zbuf, bary, _ = oracle.rasterize_meshes(fv.numpy(), [0], [2], H, H, 2, flags)
        gz = torch.randn(1, H, H, 2, generator=g); gb = torch.randn(1, H, H, 2, 3, generator=g)
        got = oracle.rasterize_meshes_backward(fv.numpy(), p2f, gz.numpy(), gb.numpy(), flags)
        fvd = fv.double().requires_grad_()
        yf = tr.pix_centers(H, torch.float64)[:, None, None].expand(H, H, 2)
        xf = tr.pix_centers(H, torch.float64)[None, :, None].expand(H, H, 2)
        idx = torch.from_numpy(p2f[0]).long()
        b = tr.bary_coords(xf, yf, fvd[idx.clamp_min(0)], persp)
        z = (b * fvd[idx.clamp_min(0)][..., 2]).sum(-1)
        m = (idx >= 0).double()
        ((b * gb[0].double()).sum(-1) * m + z * gz[0].double() * m).sum().backward()
        assert rel(got, fvd.grad.numpy()) < 2e-5


@pytest.mark.parametrize("mode,K", [("norm", 1), ("norm", 4), ("alpha", 1), ("alpha", 4)])
def test_points_forward_backward_match_torch(oracle, mode, K):
    pts = synth.make_clouds(1, 200, 3)
    az = torch.tensor([10., 130., -95.]); el = torch.tensor([5., 30., -60.]); di = torch.tensor([2.2, 1.8, 3.0])
    R, T, _ = oracle.look_at(az.numpy(), el.numpy(), di.numpy())
    M, H, rad = 3, 24, 0.08
    inv = (1.0 / di).numpy()
    feat = np.random.RandomState(2).rand(200, 3).astype(np.float32)
    bg = np.array([0.1, 0.2, 0.3], np.float32)
    flag = oracle.COMPOSITE_ALPHA if mode == "alpha" else 0
    po = oracle.points_forward(pts.numpy(), feat[None], M, R, T, inv, rad, bg, H, H, K, flag)
    gimg = np.random.RandomState(4).randn(M, 3, H, H).astype(np.float32)
    pb = oracle.points_backward(pts.numpy(), feat[None], M, R, T, inv, rad, H, H, K, flag, po["idx"], gimg,
                                want_points=True, want_rgb=True)
    D = torch.float64
    pd = pts[0].to(D).requires_grad_(); fd = torch.from_numpy(feat).to(D).requires_grad_()
    Rq, Tq, sq = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T, inv))
    loss = 0
    for n in range(M):
        img, idx = tr.render_points_view(pd, fd.T, Rq[n], Tq[n], sq[n], rad, torch.from_numpy(bg).to(D), H, H, K, mode == "alpha")
        assert (idx.numpy() != po["idx"][n]).sum() <= 2          # fp64 vs fp32 boundary pixels only
        same = (idx.numpy() == po["idx"][n]).all(-1)
        assert np.abs(img.detach().numpy() - po["images"][n])[:, same].max() < 1e-5
        img2, _ = tr.render_points_view(pd, fd.T, Rq[n], Tq[n], sq[n], rad, torch.from_numpy(bg).to(D), H, H, K, mode == "alpha",
                                        idx=torch.from_numpy(po["idx"][n]).long())
        loss = loss + (img2 * torch.from_numpy(gimg[n]).to(D)).sum()
    loss.backward()
    assert rel(pb["gR"], Rq.grad.numpy()) < 2e-5
    assert rel(pb["gT"], Tq.grad.numpy()) < 2e-5
    assert rel(pb["g_inv_dist"], sq.grad.numpy()) < 2e-5
    assert rel(pb["grad_points"][0], pd.grad.numpy()) < 2e-5
    assert rel(pb["grad_rgb"][0], fd.grad.numpy()) < 2e-5


def test_points_backward_matches_finite_differences(oracle):
    """The point path's hand-derived chain -- d image -> alpha compositor -> dists2 -> projection (R, T, 1 / dist scale) ->
    look_at backward -> d azim / elev / dist -- against central differences of the oracle's OWN forward (no torch_ref).
    The scene is chosen so that the rendered loss is continuous in the camera: alpha compositing over a black background
    (a covered pixel whose weights vanish meets the background continuously), K >= the depth complexity (front / back
    pairs: no point is ever dropped from a pixel's K-list), well separated pairs.  Pixel centres entering or leaving a disc
    leave kinks, hence the loose tolerance; a wrong factor (degrees, -1 / dist^2, a sign) is off by far more."""
    rs = np.random.RandomState(5)
    gx, gy = np.meshgrid(np.linspace(-0.75, 0.75, 4), np.linspace(-0.5, 0.5, 3))
    front = np.stack([gx.ravel(), gy.ravel(), 0.15 + 0.1 * rs.rand(12)], 1)
    back = front.copy(); back[:, 2] -= 0.35; back[:, :2] += 0.03 * rs.randn(12, 2)
    pts = np.concatenate([front, back])[None].astype(np.float32)
    M, H, rad, K = 3, 48, 0.08, 2
    feat = rs.rand(1, pts.shape[1], 3).astype(np.float32)
    bg = np.zeros(3, np.float32)
    g = rs.randn(M, 3, H, H).astype(np.float32)
    az0 = np.array([4.0, -9.0, 12.0]); el0 = np.array([3.0, 8.0, -6.0]); di0 = np.array([2.2, 2.4, 2.0])

    def loss(az, el, di, want_grad=False):
        R, T, _ = oracle.look_at(az, el, di)
        inv = (1.0 / di).astype(np.float32)
        o = oracle.points_forward(pts, feat, M, R, T, inv, rad, bg, H, H, K, oracle.COMPOSITE_ALPHA)
        val = float((o["images"].astype(np.float64) * g).sum())
        if not want_grad:
            return val
        assert (o["idx"][..., 1] >= 0).mean() > 0.02            # second layers are populated
        b = oracle.points_backward(pts, feat, M, R, T, inv, rad, H, H, K, oracle.COMPOSITE_ALPHA, o["idx"], g)
        ga, ge, gd = oracle.look_at_backward(az, el, di, b["gR"], b["gT"], np.zeros_like(b["gT"]))
        return val, (ga, ge, gd + b["g_inv_dist"] * (-1.0 / di ** 2))      # dist also scales the cloud (renderer.py:142)

    _, (ga, ge, gd) = loss(az0, el0, di0, want_grad=True)
    for name, grad, h in (("azim", ga, 0.02), ("elev", ge, 0.02), ("dist", gd, 0.002)):
        for i in range(M):
            args = {"azim": az0.copy(), "elev": el0.copy(), "dist": di0.copy()}
            args[name][i] += h
            up = loss(args["azim"], args["elev"], args["dist"])
            args[name][i] -= 2 * h
            dn = loss(args["azim"], args["elev"], args["dist"])
            fd = (up - dn) / (2 * h)
            scale = max(abs(fd), float(np.abs(grad).max()), 1e-6)
            assert abs(grad[i] - fd) <= 0.1 * scale, (name, i, float(grad[i]), fd)


def test_point_projection_scales_by_inverse_distance(oracle):
    # renderer.py:141-143: the ONLY place dist enters an orthographic image is the 1/dist cloud scaling
    R, T, _ = oracle.look_at([0.0], [0.0], [2.0])
    p = oracle.project_orthographic(np.array([[0.5, 0.25, 0.0]], np.float32), R[0], T[0], 0.5)
    assert np.allclose(p[0], [-0.25, 0.125, 2.0], atol=1e-6)


def test_perspective_projection_kat(oracle):
    # x_ndc = x_v * K00 / z_v with K00 = 1/tan(30 deg)  (SURVEY 8c.3)
    assert K00 == pytest.approx(1.0 / math.tan(math.radians(30.0)), rel=1e-6) and K00 == K11
    R, T, _ = oracle.look_at([0.0], [0.0], [2.0])
    p = oracle.project_perspective(np.array([[0.5, 0.5, 0.0], [0.0, 0.0, 1.0]], np.float32), R[0], T[0], K00, K11)
    assert np.allclose(p[0], [-0.5 * K00 / 2.0, 0.5 * K00 / 2.0, 2.0], atol=1e-6)
    assert np.allclose(p[1], [0.0, 0.0, 1.0], atol=1e-6)


def test_phong_shading_closed_form_kat(oracle):
    """A large triangle in the world plane z = 0 facing the camera at (0, 0, 2.2), light direction (0.3, 0.2, 1): every
    covered pixel has a closed-form colour -- ambient 0.5 + diffuse 0.3 (n.l) + specular 0.2 (v.r)^64 with
    r = -l + 2 (n.l) n ([upstream] lighting.py / shading.py, constants of renderer.py:190-191), evaluated at the world
    point the pixel centre back-projects to (which is what perspective-correct interpolation must reproduce).  Pins the
    pixel grid (x left, y up), the FoV constants, the interpolation and the Phong constants independently of
    torch_ref.py; float64 here, 1e-5 against the fp32 oracle."""
    H = W = 32
    v = np.array([[-3.0, -2.0, 0.0], [3.0, -2.0, 0.0], [0.0, 4.0, 0.0]], np.float32)
    f = np.array([[0, 1, 2]], np.int32)
    nrm = oracle.vertex_normals(v, f)
    sign = float(np.sign(nrm[0, 2]))
    assert np.allclose(nrm, [[0, 0, sign]] * 3, atol=1e-7) and sign != 0
    if sign < 0:                                     # face the camera (+z): flip the winding
        f = f[:, ::-1].copy(); nrm = oracle.vertex_normals(v, f)
        assert np.allclose(nrm, [[0, 0, 1.0]] * 3, atol=1e-7)
    d = 2.2
    R, T, C = oracle.look_at([0.0], [0.0], [d])
    light = np.array([[0.3, 0.2, 1.0]], np.float32)
    rgb = np.array([0.9, 0.6, 0.3], np.float32); bg = np.array([0.1, 0.2, 0.7], np.float32)
    o = oracle.mesh_forward(v, f, [0, 3], [0, 1], nrm, rgb, 1, R, T, C, light, bg, K00, K11, 0.5, H, W, 1, oracle.PERSPECTIVE_CORRECT)
    img, p2f = o["images"][0], o["pix_to_face"][0, ..., 0]
    assert (p2f >= 0).mean() > 0.5
    l = light[0].astype(np.float64); l /= np.linalg.norm(l)
    n = np.array([0.0, 0.0, 1.0])
    k = float(K00)
    worst = 0.0
    for yi in range(H):
        for xi in range(W):
            xf = 1.0 - (2 * xi + 1) / W; yf = 1.0 - (2 * yi + 1) / H          # pixel centre in NDC: +x left, +y up
            xv, yv = xf * d / k, yf * d / k                                    # view-space point on the plane z_v = d
            P = np.array([-xv, yv, 0.0])                                       # R = diag(-1, 1, -1): world x = -view x
            inside = (P[1] > -2.0) and (P[1] < 4.0 - 2.0 * abs(P[0]))          # the triangle's three edges
            if not inside:
                if p2f[yi, xi] < 0:
                    assert np.allclose(img[:, yi, xi], bg, atol=1e-7)
                continue
            if p2f[yi, xi] < 0:
                continue                                                       # a centre within rounding of an edge
            cosang = float(n @ l)
            vdir = np.array([0.0, 0.0, d]) - P; vdir /= np.linalg.norm(vdir)
            r = -l + 2.0 * cosang * n
            spec = 0.2 * max(float(vdir @ r), 0.0) ** 64
            want = (0.5 + 0.3 * max(cosang, 0.0)) * rgb.astype(np.float64) + spec
            worst = max(worst, float(np.abs(img[:, yi, xi] - want).max()))
    assert worst <= 1e-5, worst
    assert abs(o["zbuf"][0][p2f >= 0] - d).max() <= 1e-5                        # the whole plane lies at view depth d


def test_near_plane_cull_counts_straddlers(oracle):
    v = np.array([[-0.3, -0.3, 1.9], [0.3, -0.3, 1.9], [0.0, 0.3, 1.9],     # fully behind z_clip after projection (z_v = 0.1)
                  [-0.3, -0.3, 1.7], [0.3, -0.3, 1.7], [0.0, 0.3, 0.0]], np.float32)   # straddles z_clip = 0.5
    f = np.array([[0, 1, 2], [3, 4, 5]], np.int32)
    R, T, C = oracle.look_at([0.0], [0.0], [2.0])
    nrm = oracle.vertex_normals(v, f)
    o = oracle.mesh_forward(v, f, [0, 6], [0, 2], nrm, np.ones(3, np.float32), 1, R, T, C, np.array([[0, 1.0, 0]], np.float32),
                            np.zeros(3, np.float32), K00, K11, 0.5, 16, 16, 1, oracle.PERSPECTIVE_CORRECT)
    assert o["straddle"] == 1
    assert not (o["pix_to_face"] == 0).any()        # culled face never rasterizes


# --------------------------------------------------------------------------------------------- G5 golden hashes
def test_golden_mesh_slice(oracle):
    g = np.load(os.path.join(GOLDEN, "mesh_c2_slice.npz"))
    vp, fp = g["verts"], g["faces"]
    nrm = oracle.vertex_normals(vp, fp)
    col = np.full(3, 0.99999, np.float32); light = np.array([[0, 1.0, 0]], np.float32)
    o = oracle.mesh_forward(vp, fp, [0, vp.shape[0]], [0, fp.shape[0]], nrm, col, 12, g["R"], g["T"], g["C"], light, col,
                            float(g["k00"]), float(g["k11"]), 0.5, 224, 224, 1, oracle.PERSPECTIVE_CORRECT)
    assert sha(o["pix_to_face"]) == str(g["p2f_sha256"])
    assert sha(o["zbuf"]) == str(g["zbuf_sha256"])
    assert sha(o["bary"]) == str(g["bary_sha256"])
    assert ((o["pix_to_face"][..., 0] >= 0).sum(axis=(1, 2)) == g["covered"]).all()
    assert np.abs(o["images"][:, :, ::16, ::16] - g["image_probe"]).max() < 1e-6


def test_golden_mesh_clip(oracle):
    g = np.load(os.path.join(GOLDEN, "mesh_clip.npz"))
    vp, fp = g["verts"], g["faces"]
    nrm = oracle.vertex_normals(vp, fp)
    col = np.full(3, 0.99999, np.float32); light = np.array([[0, 1.0, 0]], np.float32)
    o = oracle.mesh_forward(vp, fp, [0, vp.shape[0]], [0, fp.shape[0]], nrm, col, 3, g["R"], g["T"], g["C"], light, col,
                            float(g["k00"]), float(g["k11"]), 0.5, 96, 96, 2, oracle.PERSPECTIVE_CORRECT)
    assert o["straddle"] == int(g["straddle"]) > 0
    assert sha(o["pix_to_face"]) == str(g["p2f_sha256"]) and sha(o["zbuf"]) == str(g["zbuf_sha256"])
    assert sha(o["bary"]) == str(g["bary_sha256"]) and sha(o["dists"]) == str(g["dists_sha256"])
    assert np.abs(o["images"][:, :, ::8, ::8] - g["image_probe"]).max() < 1e-6


def test_golden_points(oracle):
    g = np.load(os.path.join(GOLDEN, "points_c1.npz"))
    col = np.full(3, 0.99999, np.float32)
    o = oracle.points_forward(g["points"], col, 12, g["R"], g["T"], g["inv_dist"], 0.006, np.zeros(3, np.float32), 224, 224, 1, 0)
    assert sha(o["idx"]) == str(g["idx_sha256"]) and sha(o["zbuf"]) == str(g["zbuf_sha256"]) and sha(o["dists2"]) == str(g["d2_sha256"])
    assert np.allclose(o["images"].astype(np.float64).sum(axis=(1, 2, 3)), g["image_sum"], rtol=1e-6)
    o4 = oracle.points_forward(g["points"], col, 12, g["R"], g["T"], g["inv_dist"], 0.02, np.zeros(3, np.float32), 224, 224, 4,
                               oracle.COMPOSITE_ALPHA)
    assert sha(o4["idx"]) == str(g["idx4_sha256"])


# --------------------------------------------------------------------- near-plane clipping ([upstream] clip.py)
def test_clip_faces_known_answers():
    """Hand-derived clipping of one triangle against z = 0.5 (no perspective correction: plain lerps)."""
    # case 3: vertex 0 in front (z = 1.5), vertices 1, 2 behind (z = 0.25) -> one triangle (p4, p5, p1), w = 1/1.25 = 0.8
    fv = torch.tensor([[[0.0, 0.0, 1.5], [1.0, 0.0, 0.25], [0.0, 1.0, 0.25]]], dtype=torch.float64)
    fvc, c2u, conv = tr.clip_faces(fv, 0.5, False)
    assert fvc.shape == (1, 3, 3) and c2u.tolist() == [0]
    assert torch.allclose(fvc[0], torch.tensor([[0.8, 0.0, 0.5], [0.0, 0.8, 0.5], [0.0, 0.0, 1.5]], dtype=torch.float64))
    # columns = barycentrics of (p4, p5, p1) in the original triangle
    assert torch.allclose(conv[0], torch.tensor([[0.2, 0.2, 1.0], [0.8, 0.0, 0.0], [0.0, 0.8, 0.0]], dtype=torch.float64))
    # case 4: vertex 1 behind -> quad split into (p4, p2, p5), (p5, p2, p3) with p1 = v1, p2 = v2, p3 = v0
    fv = torch.tensor([[[0.0, 0.0, 1.0], [1.0, 0.0, 0.0], [0.0, 1.0, 1.0]]], dtype=torch.float64)
    fvc, c2u, conv = tr.clip_faces(fv, 0.5, False)
    assert fvc.shape == (2, 3, 3) and c2u.tolist() == [0, 0]
    p4 = torch.tensor([0.5, 0.5, 0.5], dtype=torch.float64); p5 = torch.tensor([0.5, 0.0, 0.5], dtype=torch.float64)
    assert torch.allclose(fvc[0], torch.stack([p4, fv[0, 2], p5])) and torch.allclose(fvc[1], torch.stack([p5, fv[0, 2], fv[0, 0]]))
    # every clipped vertex is the conv-weighted combination of the original ones (z exactly, xy because persp is off)
    for c in range(2):
        assert torch.allclose(conv[c].T @ fv[0], fvc[c])
    # perspective-correct: xy are interpolated un-projected and re-projected at the plane
    fv = torch.tensor([[[0.2, -0.4, 2.0], [1.0, 0.6, 0.25], [-0.8, 1.0, 0.25]]], dtype=torch.float64)
    fvc, _, conv = tr.clip_faces(fv, 0.5, True)
    world = fv[0, :, :2] * fv[0, :, 2:3]
    assert torch.allclose(fvc[0, :, :2] * fvc[0, :, 2:3], conv[0].T @ world) and torch.allclose(fvc[0, :2, 2], torch.tensor([0.5, 0.5], dtype=torch.float64))
    # untouched and fully-behind faces
    fv = torch.tensor([[[0, 0, 1.0], [1, 0, 1.0], [0, 1, 1.0]], [[0, 0, 0.1], [1, 0, 0.2], [0, 1, 0.3]]], dtype=torch.float64)
    fvc, c2u, conv = tr.clip_faces(fv, 0.5, True)
    assert c2u.tolist() == [0] and torch.equal(conv[0], torch.eye(3, dtype=torch.float64))


def _close_up(seed, faces=260, M=3):
    """A camera 1.15 - 1.3 away from a unit-sphere object: faces straddle z = 0.5 (mvtn.py:33 transform_distance)."""
    v, f = synth.make_mesh(faces, seed)
    az = torch.tensor([15., 140., -80.])[:M]; el = torch.tensor([10., -35., 50.])[:M]; di = torch.tensor([1.15, 1.22, 1.3])[:M]
    return v, f, az, el, di


def test_mesh_forward_with_clipping_matches_torch_restatement(oracle):
    v, f, az, el, di = _close_up(5)
    M, H = 3, 48
    R, T, C = oracle.look_at(az.numpy(), el.numpy(), di.numpy())
    nrm = oracle.vertex_normals(v.numpy(), f.numpy())
    voff = np.array([0, v.shape[0]], np.int32); foff = np.array([0, f.shape[0]], np.int32)
    rgb = np.random.RandomState(5).rand(v.shape[0], 3).astype(np.float32)
    light = np.array([[0.3, 1.0, -0.5]], np.float32); bg = np.array([0.2, 0.4, 0.6], np.float32)
    o = oracle.mesh_forward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, M, R, T, C, light, bg, K00, K11, 0.5, H, H, 1,
                            oracle.PERSPECTIVE_CORRECT)
    assert o["straddle"] > 0
    unclipped = oracle.mesh_forward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, M, R, T, C, light, bg, K00, K11, -1.0, H, H, 1,
                                    oracle.PERSPECTIVE_CORRECT)
    assert (unclipped["pix_to_face"] != o["pix_to_face"]).sum() > 0      # the clip removes what is nearer than the plane
    assert float(o["zbuf"][o["pix_to_face"] >= 0].min()) >= 0.5 - 1e-5
    mism = 0
    for n in range(M):
        Rn, Tn, Cn = (torch.from_numpy(x[n]).double() for x in (R, T, C))
        img, p2f = tr.render_mesh_view(v.double(), f, torch.from_numpy(nrm).double(), torch.from_numpy(rgb).double(), Rn, Tn, Cn,
                                       torch.from_numpy(light[0]).double(), torch.from_numpy(bg).double(), K00, K11, H, H, z_clip=0.5)
        bad = p2f.numpy() != o["pix_to_face"][n, ..., 0]
        mism += int(bad.sum())
        assert np.abs(img.numpy() - o["images"][n])[:, ~bad].max() < 1e-5
    assert mism <= 4          # fp64 restatement vs fp32 oracle: pixels a rounding error away from an edge


def test_mesh_backward_with_clipping_matches_autograd(oracle):
    for persp in (True, False):
        v, f, az, el, di = _close_up(6)
        M, H = 3, 40
        R, T, C = oracle.look_at(az.numpy(), el.numpy(), di.numpy())
        nrm = oracle.vertex_normals(v.numpy(), f.numpy())
        voff = np.array([0, v.shape[0]], np.int32); foff = np.array([0, f.shape[0]], np.int32)
        rgb = np.random.RandomState(6).rand(v.shape[0], 3).astype(np.float32)
        light = np.array([[0.3, 1.0, -0.5]], np.float32); bg = np.full(3, 0.99999, np.float32)
        flags = oracle.PERSPECTIVE_CORRECT if persp else 0
        o = oracle.mesh_forward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, M, R, T, C, light, bg, K00, K11, 0.5, H, H, 1, flags)
        assert o["straddle"] > 0
        gimg = np.random.RandomState(7).randn(M, 3, H, H).astype(np.float32)
        bw = oracle.mesh_backward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, M, R, T, C, light, K00, K11, H, H, 1, flags,
                                  o["pix_to_face"], gimg, want_verts=True, z_clip=0.5)
        D = torch.float64
        Rd, Td, Cd = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T, C))
        vd = v.to(D).requires_grad_(); nd = torch.from_numpy(nrm).to(D).requires_grad_()
        loss = 0
        n_clipped_px = 0
        for n in range(M):
            img, p2f = tr.render_mesh_view(vd, f, nd, torch.from_numpy(rgb).to(D), Rd[n], Td[n], Cd[n], torch.from_numpy(light[0]).to(D),
                                           torch.from_numpy(bg).to(D), K00, K11, H, H, perspective_correct=persp, z_clip=0.5)
            same = torch.from_numpy(o["pix_to_face"][n, ..., 0]).long() == p2f       # drop the rare edge-rounding pixels from both sides
            gm = torch.from_numpy(gimg[n]).to(D) * same[None]
            gimg[n] *= same.numpy()[None]
            loss = loss + (img * gm).sum()
            fv = tr.project_perspective(v.double(), Rd[n].detach(), Td[n].detach(), K00, K11)[f]
            strad = ((fv[:, :, 2] < 0.5).sum(1) % 3 != 0)
            n_clipped_px += int(strad[p2f.clamp_min(0)][p2f >= 0].sum())
        assert n_clipped_px > 20      # the test exercises the clipped-triangle chain, not just the ordinary one
        bw = oracle.mesh_backward(v.numpy(), f.numpy(), voff, foff, nrm, rgb, M, R, T, C, light, K00, K11, H, H, 1, flags,
                                  o["pix_to_face"], gimg, want_verts=True, z_clip=0.5)
        loss.backward()
        assert rel(bw["gR"], Rd.grad.numpy()) < 5e-5
        assert rel(bw["gT"], Td.grad.numpy()) < 5e-5
        assert rel(bw["gC"], Cd.grad.numpy()) < 5e-5
        assert rel(bw["grad_verts"], vd.grad.numpy()) < 1e-4
        assert rel(bw["grad_normals"], nd.grad.numpy()) < 5e-5


# ------------------------------------------------------------------------------------------------ soft rasterization (8f N3)
def _soft_setup(seed=3, faces=260, M=2):
    v, f = synth.make_mesh(faces, seed)
    az, el, di = synth.learned_spherical_views(1, M, seed + 2)
    return v, f, az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel()


def test_soft_rasterizer_reduces_to_the_hard_one_at_zero_blur(oracle):
    """blur_radius = 0, no barycentric clipping: the torch restatement of the blurred rasterizer is the C oracle's rasterizer
    (indices, depths, barycentrics and -- now signed -- distances, all inside => negative)."""
    v, f, az, el, di = _soft_setup()
    R, T, C = oracle.look_at(az, el, di)
    fv = torch.from_numpy(oracle.project_perspective(v.numpy(), R[0], T[0], K00, K11))[f]
    p2f, zb, ba, ds = tr.rasterize_meshes_soft(fv, 40, 40, 3, 0.0)
    o = oracle.rasterize_meshes(fv.numpy(), [0], [f.shape[0]], 40, 40, 3, oracle.PERSPECTIVE_CORRECT)
    assert (p2f.numpy() == o[0][0]).all() and (zb.numpy() == o[1][0]).all()
    assert np.abs(ba.numpy() - o[2][0]).max() < 1e-6 and np.abs(ds.numpy() - o[3][0]).max() < 1e-7
    assert (ds[p2f >= 0] <= 0).all()


def test_soft_silhouette_closed_form_kat():
    """One right triangle on a 16 x 16 image, blur radius 0.3 NDC: alpha of a pixel = sigmoid(-signed squared edge distance /
    sigma) ([upstream] sigmoid_alpha_blend with one fragment); pixels farther than the radius from the triangle have no fragment."""
    fv = torch.tensor([[[-0.5, -0.5, 2.0], [0.5, -0.5, 2.0], [-0.5, 0.5, 2.0]]])
    S, blur, sigma = 16, 0.09, 0.02
    p2f, zb, ba, ds = tr.rasterize_meshes_soft(fv, S, S, 2, blur, perspective_correct=False)
    img = tr.sigmoid_alpha_blend(torch.ones_like(ba), p2f, ds, sigma)
    xs = tr.pix_centers(S)
    import math as _m
    for yi in range(S):
        for xi in range(S):
            x, y = float(xs[xi]), float(xs[yi])
            inside = x > -0.5 and y > -0.5 and x + y < 0.0
            # distance to the three segments
            def seg(ax, ay, bx, by):
                dx, dy = bx - ax, by - ay
                t = min(max(((x - ax) * dx + (y - ay) * dy) / (dx * dx + dy * dy), 0.0), 1.0)
                return (x - ax - t * dx) ** 2 + (y - ay - t * dy) ** 2
            d2 = min(seg(-0.5, -0.5, 0.5, -0.5), seg(-0.5, -0.5, -0.5, 0.5), seg(0.5, -0.5, -0.5, 0.5))
            in_box = (-0.5 - 0.3 <= x <= 0.5 + 0.3) and (-0.5 - 0.3 <= y <= 0.5 + 0.3)
            frag = in_box and (inside or d2 < blur)
            if abs(d2 - blur) < 1e-4 or min(abs(x + 0.5), abs(y + 0.5), abs(x + y)) < 1e-4:
                continue      # on a boundary: either answer is a rounding matter
            assert (int(p2f[yi, xi, 0]) == 0) == frag, (yi, xi)
            want = 1.0 / (1.0 + _m.exp((-d2 if inside else d2) / sigma)) if frag else 0.0
            assert abs(float(img[yi, xi, 3]) - want) < 1e-5
            assert int(p2f[yi, xi, 1]) == -1


def test_softmax_blend_closed_form_and_clipped_barycentrics():
    """softmax_rgb_blend with one fragment: rgb = (w c + delta bg) / (w + delta), w = sigmoid(-d / sigma) (its z_inv IS the max),
    delta = exp((eps - z_inv) / gamma) clamped at eps; BarycentricClipForward clamps and renormalises."""
    b = torch.tensor([[-0.2, 0.6, 0.6], [0.3, 0.3, 0.4], [-1.0, -1.0, 3.0]])
    bc = tr.bary_clip(b)
    assert torch.allclose(bc, torch.tensor([[0.0, 0.5, 0.5], [0.3, 0.3, 0.4], [0.0, 0.0, 1.0]]))
    col = torch.tensor([[[[0.2, 0.4, 0.6], [0.0, 0.0, 0.0]]]]); p2f = torch.tensor([[[5, -1]]]); z = torch.tensor([[[3.0, -1.0]]])
    d = torch.tensor([[[-0.01, -1.0]]]); bg = torch.tensor([1.0, 0.0, 0.5])
    out = tr.softmax_rgb_blend(col, p2f, z, d, bg, sigma=0.01, gamma=0.5)
    w = 1 / (1 + math.exp(-1.0)); zi = (100 - 3.0) / 99; delta = max(math.exp((1e-10 - zi) / 0.5), 1e-10)
    want = [(w * c + delta * g) / (w + delta) for c, g in zip((0.2, 0.4, 0.6), (1.0, 0.0, 0.5))]
    assert torch.allclose(out[0, 0, :3], torch.tensor(want), atol=1e-6) and abs(float(out[0, 0, 3]) - w) < 1e-6


def test_soft_render_is_differentiable_and_matches_finite_differences(oracle):
    """render_mesh_view_soft (fp64): autograd of the silhouette w.r.t. the camera translation against central differences (the
    fragment assignment is frozen, as in PyTorch3D: the index is not differentiated)."""
    v, f, az, el, di = _soft_setup(seed=5, faces=120, M=1)
    R, T, C = oracle.look_at(az, el, di)
    D = torch.float64
    nrm = torch.from_numpy(oracle.vertex_normals(v.numpy(), f.numpy())).to(D)
    Rd, Cd = torch.from_numpy(R[0]).to(D), torch.from_numpy(C[0]).to(D)
    Td = torch.from_numpy(T[0]).to(D).requires_grad_()
    g = torch.randn(4, 24, 24, generator=torch.Generator().manual_seed(2), dtype=D)
    args = (v.to(D), f, nrm, torch.ones_like(v, dtype=D), Rd)

    def loss(Tt, shader, p2f=None):
        img, fr = tr.render_mesh_view_soft(*args, Tt, Cd, torch.tensor([0.3, 1.0, -0.5], dtype=D), torch.ones(3, dtype=D), K00, K11, 24, 24, 6,
                                           4e-3, shader, sigma=2e-3, gamma=5e-2, p2f=p2f)
        return (img * g).sum(), fr["pix_to_face"]
    for shader in ("soft_silhouette", "soft_phong"):
        val, p2f = loss(Td, shader)
        (gT,) = torch.autograd.grad(val, Td)
        for i in range(3):
            h = 1e-6
            e = torch.zeros(3, dtype=D); e[i] = h
            fd = (loss(Td.detach() + e, shader, p2f)[0] - loss(Td.detach() - e, shader, p2f)[0]) / (2 * h)
            # (2e-4, not 1e-6: where the perspective-correction denominator is clamped -- some blurred fragments outside their
            # face -- upstream's backward differentiates the unclamped sum, and the restatement follows upstream, not calculus)
            assert abs(float(gT[i]) - float(fd)) <= 2e-4 * max(1.0, abs(float(fd))), (shader, i, float(gT[i]), float(fd))


def test_regularizer_composed_gather_matches_reference_composition():
    """ops.py:138-178 (dropout2d on the 5-D tensor, batchwise flip, ReplicationPad2d, RandomCrop) restated with the reference's own
    torch / torchvision calls, against the ONE-gather form the CUDA kernel evaluates with the decisions drawn by
    mvtn_b200.augment.draw_regularizer: same seeds -> same tensor, bit for bit (so the draw order and the index algebra are right)."""
    import torch
    from oracle import torch_ref as tr
    from mvtn_b200.augment import draw_regularizer
    seen = set()
    for seed in range(48):
        x = torch.randn(2, 3, 3, 10, 10)
        p = [0, 0.3, 0.5][seed % 3]; aug = seed % 2 == 0; cr = [0.3, 0.0, 0.5, 0.15][seed % 4]
        torch.manual_seed(seed); ref = tr.regularize_rendered_views(x, p, aug, cr)
        torch.manual_seed(seed); sc, fl, sy, sx = draw_regularizer(x, p, aug, cr)
        assert torch.equal(ref, tr.regularize_gather(x, sc, fl, sy, sx)), (seed, p, aug, cr, fl, sy, sx)
        seen.add((fl, sy < 0, sy > 0, sx < 0, sx > 0, sc is not None))
    assert len(seen) >= 12      # flips, both shift signs on both axes, with and without dropped views all occurred
    x = torch.randn(1, 2, 3, 6, 6)
    sc, fl, sy, sx = draw_regularizer(x, 0, False)
    assert sc is None and not fl and sy == 0 and sx == 0
    torch.manual_seed(1); sc, _, _, _ = draw_regularizer(x, 1.0, False)
    assert torch.equal(sc, torch.zeros(2))
