"""shader="hard_depth" at the edges test_gpu_depth.py does not reach: odd image shapes, every binning branch in front of the
point depth kernel, unaligned outputs, empty and off-screen inputs, other background values, the 128-thread mesh scatter,
back-face culling at the near plane, per-vertex colours in the geometry, the mesh workspace's reuse hints across shaders,
and MVRenderer's redraw loop.

The references and bars are test_gpu_depth.py's: the depth bit for bit against the C oracle's zbuf[..., 0] (depth_background
where its pix_to_face / idx is -1) with 0 face or point id mismatches; R, T and dist gradients against fp64 autograd of
tests/depth_ref.py within GRAD_RTOL, point gradients within POINT_GRAD_RTOL, vertex gradients within VERT_GRAD_RTOL.  Every
case named after a branch asserts the launches of that branch (launches / expect_launches of test_gpu_branches.py).

One bar of its own: where two renders must give "the same" point or vertex gradients (another depth_background, per-vertex
colours in the geometry), the camera and dist gradients are compared bit for bit (fixed-order sums), the point and vertex
gradients within 1e-6 of their largest entry -- they are accumulated with float atomics, whose order changes run to run.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, _lib as L, ops, synth

import depth_ref
from test_gpu_branches import expect_launches, launches
from test_gpu_depth import (BGD, GRAD_RTOL, MESH, POINT_GRAD_RTOL, VERT_GRAD_RTOL, cams, check_depth, mesh_grads_ref, oracle_mesh,
                            oracle_points, rel)

pytestmark = pytest.mark.gpu

D = torch.float64
ATOMIC_RTOL = 1e-6         # point / vertex gradients of two renders that must agree (float atomics: order-dependent last bits)
TILE_DEPTH = "points_tile_kernel<1, 0, true>"
SHADE_DEPTH = "mesh_shade_kernel<false, 4, 4, false, true>"


def stream():
    return torch.cuda.current_stream().cuda_stream


def check_depth_small(depth, ids, oids, oz, bg, hits=True):
    """check_depth for images too small to hold its 100 covered pixels (or with nothing in view: hits=False): the same
    bit-exact comparison; some pixel covered unless hits is False."""
    depth, ids = depth.cpu(), ids.cpu()
    assert int((ids.numpy() != oids).sum()) == 0, f"{int((ids.numpy() != oids).sum())} id mismatches"
    want = torch.from_numpy(np.where(oids >= 0, oz, np.float32(bg)))
    assert torch.equal(depth, want), float((depth - want).abs().max())
    assert (oids >= 0).any() == hits


def check_parity(depth, ids, oids, oz, bg, hits=True):
    if hits and oids.size >= 2000:
        check_depth(depth, ids, oids, oz, bg)
    else:
        check_depth_small(depth, ids, oids, oz, bg, hits)


def expected_mask(idx, H, W):
    """The hit-mask words the forward must write: bit x % 32 of word x / 32 of each row, set iff idx[..., 0] >= 0."""
    N = idx.shape[0]
    words = (W + 31) // 32
    cov = torch.zeros(N, H, words * 32, dtype=torch.bool, device=idx.device)
    cov[:, :, :W] = idx[..., 0] >= 0
    weights = 2 ** torch.arange(32, device=idx.device, dtype=torch.int64)
    return (cov.view(N, H, words, 32).to(torch.int64) * weights).sum(-1)


def points_depth_raw(pts, M, R, T, dist, rad, bg, H, W, depth_ptr, idx, mask):
    """mvr_points_depth_forward straight through the C entry point (dist as the scale, as render_points(dist=...) passes it)."""
    lib = L.load()
    B, Np = pts.shape[:2]
    ws = ops.workspace(pts.device, lib.mvr_points_workspace_bytes(B, Np, M, H, W, 1, rad))
    L.check(lib.mvr_points_depth_forward(ops._ptr(pts), B, Np, M, R.data_ptr(), T.data_ptr(), dist.data_ptr(), rad, bg, H, W,
                                         L.SCALE_IS_DIST, depth_ptr, idx.data_ptr(), mask.data_ptr(), ws.data_ptr(), ws.numel(),
                                         stream()), "mvr_points_depth_forward")


def run_points(oracle, dev, pts, M, R, T, di, rad, H, W, fwd=None, bg=BGD, n_ref=None, g=None, hits=True, tag=""):
    """render_points(shader="hard_depth") with gradients to R, T, dist and the points -> dict.  fwd: prefix -> launches wanted in
    the forward; n_ref: clouds compared with the oracle and fp64 autograd (default all).  Checks the forward against the oracle,
    the hit mask against idx, the backward's kernels and the gradients against depth_ref (hits=False: nothing in view)."""
    B, Np = pts.shape[:2]
    N = B * M
    n_ref = B if n_ref is None else n_ref
    Rd, Td = torch.from_numpy(R).to(dev), torch.from_numpy(T).to(dev)
    pg = pts.to(dev).requires_grad_()
    Rg, Tg = Rd.clone().requires_grad_(), Td.clone().requires_grad_()
    dg = di.reshape(-1).to(dev).requires_grad_()

    def render():
        return ops.render_points(pg, torch.ones(3, device=dev), M, Rg, Tg, None, rad, torch.zeros(3, device=dev), (H, W), dist=dg,
                                 shader="hard_depth", depth_background=bg)

    want = {TILE_DEPTH: 1, "points_tile_kernel<1, 0>": 0, **(fwd or {})}
    counts, out = {}, None
    for p in want:
        o, counts[p] = launches(p, render)
        out = out or o
    expect_launches(counts, want, f"[{tag}] forward")
    depth, frag = out
    idx = frag["idx"]
    assert depth.shape == (N, 1, H, W) and idx.shape == (N, H, W, 1)
    # the hit mask (not part of the returned fragments): the same call through the C entry point
    lib = L.load()
    mask = torch.full((max(lib.mvr_points_hit_mask_words(B, M, H, W), 1),), -1, dtype=torch.int32, device=dev)
    d2, i2 = torch.empty_like(depth), torch.empty_like(idx)
    points_depth_raw(pg.detach(), M, Rd, Td, dg.detach(), rad, bg, H, W, d2.data_ptr(), i2, mask)
    assert torch.equal(d2, depth) and torch.equal(i2, idx)
    words = (W + 31) // 32
    assert torch.equal(mask[: N * H * words].view(N, H, words).to(torch.int64) & 0xFFFFFFFF, expected_mask(idx, H, W))
    nr = n_ref * M
    s = (1.0 / di.numpy().ravel().astype(np.float64)).astype(np.float32)
    if Np > 0:
        oidx, oz = oracle_points(oracle, pts[:n_ref], M, R[:nr], T[:nr], s[:nr], rad, H, W)
        check_parity(depth[:nr, 0], idx[:nr, ..., 0], oidx, oz, bg, hits)
    if g is None:
        g = torch.randn(N, 1, H, W, generator=torch.Generator().manual_seed(4))
    g = g.to(dev)
    _, nb = launches("points_depth_backward_kernel", lambda: depth.backward(g))
    assert nb == 1, nb
    res = dict(depth=depth.detach(), idx=idx, mask=mask, gR=Rg.grad, gT=Tg.grad, gd=dg.grad, gP=pg.grad, counts=counts)
    if Np == 0:
        return res
    Rr, Tr = (torch.from_numpy(x[:nr]).to(D).requires_grad_() for x in (R, T))
    pr = pts[:n_ref].to(D).requires_grad_()
    dr = di.reshape(-1)[:nr].to(D).requires_grad_()
    idc = idx.cpu()
    loss = 0
    for n in range(nr):
        dep, _ = depth_ref.render_points_view_depth(pr[n // M], Rr[n], Tr[n], 1.0 / dr[n], rad, H, W, background=bg, idx=idc[n].long())
        gn = torch.where(idc[n, ..., 0] >= 0, g[n, 0].cpu().to(D), 0.0)      # (a NaN cotangent on the background stays out)
        loss = loss + (dep * gn).sum()
    loss.backward()
    errs = dict(gR=rel(Rg.grad[:nr], Rr.grad), gT=rel(Tg.grad[:nr], Tr.grad), gd=rel(dg.grad[:nr], dr.grad))
    errs["gP"] = rel(pg.grad[:n_ref], pr.grad)
    print(f"[{tag}] launches {counts} grad errs " + " ".join(f"{k} {e:.1e}" for k, e in errs.items()))
    for k in ("gR", "gT", "gd"):
        assert errs[k] < GRAD_RTOL, (tag, k, errs[k])
    assert errs["gP"] < POINT_GRAD_RTOL, (tag, errs["gP"])
    assert (float(Rr.grad.abs().max()) > 0) == hits
    return res


def cloud_case(oracle, B, M, Np, seed):
    pts = synth.make_clouds(B, Np, seed)
    views = synth.learned_spherical_views(B, M, seed + 1)
    R, T, _, _ = cams(oracle, views, "cpu")
    return pts, R, T, views[2]


# ------------------------------------------------------------------------------------------------- points
@pytest.mark.parametrize("H,W", [(45, 70), (33, 31), (7, 5), (1, 1), (72, 64)])
def test_points_depth_odd_shapes(oracle, cuda_device, H, W):
    """W % 4 != 0 (the tile kernel's scalar background stores), W % 32 != 0 (tail lanes of the backward's hit-mask words),
    images smaller than one tile, and test_gpu_depth.py's shape as a control: forward, hit mask and gradients."""
    pts, R, T, di = cloud_case(oracle, 3, 4, 2048, 11)
    rad = 0.02 if H * W > 1000 else 0.15          # the small images: a radius that covers most of the (few) pixel centres
    res = run_points(oracle, cuda_device, pts, 4, R, T, di, rad, H, W, tag=f"{H}x{W}")
    assert bool((res["idx"][..., 0] < 0).any()) or H * W == 1      # background pixels too


def test_points_depth_unaligned_output(oracle, cuda_device):
    """W % 4 == 0 but the depth one float into a larger buffer (not 16-byte aligned): the background goes through the scalar
    stores.  Same depth, ids and hit mask bit for bit as the aligned call; the guard words on either side stay untouched."""
    dev = cuda_device
    B, M, Np, H, W, rad = 2, 2, 700, 48, 64, 0.03
    pts, R, T, di = cloud_case(oracle, B, M, Np, 21)
    pts, Rd, Td, dd = pts.to(dev), torch.from_numpy(R).to(dev), torch.from_numpy(T).to(dev), di.reshape(-1).to(dev)
    n = B * M * H * W
    lib = L.load()
    nw = lib.mvr_points_hit_mask_words(B, M, H, W)
    guard = -12345.5
    buf = torch.full((n + 2,), guard, device=dev)
    assert buf.data_ptr() % 16 == 0 and buf[1:].data_ptr() % 16 == 4
    outs = {}
    for name, ptr in (("aligned", None), ("offset", buf[1:].data_ptr())):
        dep = torch.full((n,), guard, device=dev)
        idx = torch.empty(B * M, H, W, 1, dtype=torch.int32, device=dev)
        mask = torch.full((nw,), -1, dtype=torch.int32, device=dev)
        _, k = launches(TILE_DEPTH, lambda: points_depth_raw(pts, M, Rd, Td, dd, rad, BGD, H, W, ptr or dep.data_ptr(), idx, mask))
        assert k == 1
        outs[name] = (buf[1:n + 1].clone() if ptr else dep, idx, mask)
    assert buf[0].item() == guard and buf[n + 1].item() == guard
    for a, b in zip(outs["aligned"], outs["offset"]):
        assert torch.equal(a, b)
    dep, idx, _ = outs["offset"]
    assert (dep == BGD).sum() > 1000
    oidx, oz = oracle_points(oracle, pts.cpu(), M, R, T, (1.0 / di.numpy().ravel().astype(np.float64)).astype(np.float32), rad, H, W)
    check_depth(dep.view(B * M, H, W), idx[..., 0], oidx, oz, BGD)


BINNING = {
    # name: (B, M, Np, H, W, radius, clouds compared with the oracle, launches)
    "fused_cs1_small_cloud": (1, 2, 400, 48, 48, 0.05, 1, {"points_bin_kernel_fused": 1, "points_bin_scan_kernel": 0}),
    "fused_cs1_148_views": (2, 74, 1024, 32, 32, 0.06, 1, {"points_bin_kernel_fused": 1, "points_bin_scan_kernel": 0}),
    "fused_cs4": (2, 2, 2048, 48, 48, 0.03, 2, {"points_bin_kernel_fused": 1, "points_bin_scan_kernel": 0}),
    "unfused_points": (2, 3, 20000, 64, 64, 0.01, 1, {"points_bin_kernel_fused": 0, "points_bin_kernel<": 2, "points_bin_scan_kernel": 1}),
    "unfused_tiles": (1, 1, 3000, 1056, 1056, 0.01, 1, {"points_bin_kernel_fused": 0, "points_bin_kernel<": 2, "points_bin_scan_kernel": 1}),
}


@pytest.mark.parametrize("name", list(BINNING))
def test_points_depth_binning_branches(oracle, cuda_device, name):
    """Each binning path in front of the depth tile kernel: the fused kernel as one CTA per view (Np < 512, or 148 views and
    more), as a cluster of 4 CTAs (fewer views than SMs), and the three-launch path for more than 16384 points or more than
    1024 tiles (1056^2 = 33 x 33 tiles).  The fused kernel launches under one name for both cluster sizes: the side is
    asserted from the host rule, the fused (or three-launch) path from the profiler."""
    B, M, Np, H, W, rad, n_ref, want = BINNING[name]
    N, ntiles = B * M, ((H + 31) // 32) * ((W + 31) // 32)
    fused = Np <= 16384 and ntiles <= 1024
    assert fused == (want["points_bin_kernel_fused"] == 1)
    if fused:
        cs = 4 if (Np > 4096 or (N < 148 and Np >= 512)) else 1
        assert cs == (4 if name == "fused_cs4" else 1)
    pts, R, T, di = cloud_case(oracle, B, M, Np, 100 + Np % 97)
    res = run_points(oracle, cuda_device, pts, M, R, T, di, rad, H, W, fwd=want, n_ref=n_ref, tag=name)
    assert (res["idx"][: n_ref * M, ..., 0] >= 0).sum() > 100


@pytest.mark.parametrize("where", ["empty", "behind", "outside"])
def test_points_depth_nothing_in_view(oracle, cuda_device, where):
    """An empty cloud (Np = 0: no binning at all), a cloud behind every camera and one outside every view's frustum: every
    pixel depth_background, idx -1, the hit mask 0, camera, dist and point gradients exactly 0, no error."""
    dev = cuda_device
    B, M, H, W = 2, 3, 40, 36
    pts, R, T, di = cloud_case(oracle, B, M, 1500, 31)
    if where == "empty":
        pts = pts[:, :0].contiguous()
    elif where == "behind":
        T = T.copy(); T[:, 2] = -3.0                  # view z in about (-4, -2)
    else:
        T = T.copy(); T[:, 0] = 9.0                   # NDC x about 9 +- 1, the image spans +-1
    want = {"points_bin_kernel": 0} if where == "empty" else {}
    res = run_points(oracle, dev, pts, M, R, T, di, 0.05, H, W, fwd=want, hits=False, tag=where)
    assert torch.equal(res["depth"], torch.full((B * M, 1, H, W), BGD, device=dev))
    assert (res["idx"] == -1).all() and (res["mask"] == 0).all()
    for k in ("gR", "gT", "gd", "gP"):
        assert torch.equal(res[k], torch.zeros_like(res[k])), k


@pytest.mark.parametrize("bg", [0.0, -3.0, float("inf")])
def test_points_depth_background_values(oracle, cuda_device, bg):
    """depth_background 0, -3 and +inf: held exactly by every uncovered pixel (the oracle's comparison); the gradients are finite
    and those of the default background, and a cotangent of NaN on the background pixels changes none of them."""
    dev = cuda_device
    B, M, H, W, rad = 2, 3, 40, 44, 0.03
    pts, R, T, di = cloud_case(oracle, B, M, 1200, 41)
    g = torch.randn(B * M, 1, H, W, generator=torch.Generator().manual_seed(8))
    res = run_points(oracle, dev, pts, M, R, T, di, rad, H, W, bg=bg, g=g, tag=f"bg={bg}")
    ref = run_points(oracle, dev, pts, M, R, T, di, rad, H, W, bg=100.0, g=g, tag="bg=100")
    bgpix = res["idx"][..., 0] < 0
    assert bgpix.sum() > 100 and torch.equal(res["idx"], ref["idx"])
    assert (res["depth"][:, 0][bgpix] == bg).all()
    g_nan = g.clone()
    g_nan[:, 0][bgpix.cpu()] = float("nan")
    nan = run_points(oracle, dev, pts, M, R, T, di, rad, H, W, bg=bg, g=g_nan, tag=f"bg={bg} NaN cotangent")
    for other in (ref, nan):
        for k in ("gR", "gT", "gd"):
            assert torch.isfinite(res[k]).all() and torch.equal(res[k], other[k]), k
        assert torch.isfinite(other["gP"]).all() and rel(other["gP"], res["gP"]) < ATOMIC_RTOL


# ------------------------------------------------------------------------------------------------- meshes
def run_mesh(oracle, dev, meshes, M, H, W, R, T, C, persp=True, cull=False, fwd=None, vert_rgb=None, n_ref=None, tag=""):
    """render_meshes(shader="hard_depth") with gradients to R, T and the vertices; forward against the oracle on the first
    n_ref meshes (default all), backward's kernels asserted.  -> dict."""
    B = len(meshes)
    N = B * M
    n_ref = B if n_ref is None else n_ref
    nr = n_ref * M
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev, vert_rgb=vert_rgb)
    vp = torch.cat([v for v, _ in meshes]).to(dev).requires_grad_()
    Rg, Tg = (torch.from_numpy(x).to(dev).requires_grad_() for x in (R, T))
    Cd = torch.from_numpy(C).to(dev)

    def render():
        return ops.render_meshes(geom, M, Rg, Tg, Cd, torch.ones(1, 3, device=dev), torch.ones(3, device=dev), torch.zeros(3, device=dev),
                                 (H, W), cull_backfaces=cull, perspective_correct=persp, verts=vp, shader="hard_depth",
                                 depth_background=BGD)

    want = {SHADE_DEPTH: 1, "mesh_shade_kernel<false, 4, 4, false>": 0, **(fwd or {})}
    counts, out = {}, None
    for p in want:
        o, counts[p] = launches(p, render)
        out = out or o
    expect_launches(counts, want, f"[{tag}] forward")
    depth, frag = out
    p2f = frag["pix_to_face"][..., 0].cpu()
    straddle = int(frag["counters"][L.CNT_STRADDLE]) > 0
    flags = (oracle.PERSPECTIVE_CORRECT if persp else 0) | (oracle.CULL_BACKFACES if cull else 0)
    op2f, ozbuf, _ = oracle_mesh(oracle, meshes[:n_ref], M, R[:nr], T[:nr], C[:nr], H, W, flags, 0.5 if persp else -1.0)
    check_parity(depth[:nr, 0], p2f[:nr], op2f, ozbuf, BGD)
    g = torch.randn(N, 1, H, W, generator=torch.Generator().manual_seed(5))
    back = {"mesh_depth_backward_kernel<true>": 1, "mesh_backward_finish_kernel": 1}
    nb = {}
    for p in back:
        for t in (Rg, Tg, vp):
            t.grad = None
        _, nb[p] = launches(p, lambda: depth.backward(g.to(dev), retain_graph=True))
    expect_launches(nb, back, f"[{tag}] backward")
    gRr, gTr, gVr = mesh_grads_ref(oracle, meshes[:n_ref], M, R[:nr], T[:nr], p2f[:nr], g[:nr], H, W, persp, cull,
                                   0.5 if straddle else None)
    nv = sum(v.shape[0] for v, _ in meshes[:n_ref])
    errs = dict(gR=rel(Rg.grad[:nr], gRr), gT=rel(Tg.grad[:nr], gTr), gV=rel(vp.grad[:nv], torch.cat(gVr)))
    print(f"[{tag}] launches {counts} straddle {straddle} grad errs " + " ".join(f"{k} {e:.1e}" for k, e in errs.items()))
    assert errs["gR"] < GRAD_RTOL and errs["gT"] < GRAD_RTOL, (tag, errs)
    assert errs["gV"] < VERT_GRAD_RTOL, (tag, errs)
    return dict(depth=depth.detach(), p2f=frag["pix_to_face"], straddle=straddle, gR=Rg.grad, gT=Tg.grad, gV=vp.grad,
                gVr=gVr, counts=counts)


def test_mesh_depth_128_thread_scatter(oracle, cuda_device):
    """max_faces > 32768 takes the 128-thread scatter (mesh_scatter_kernel<8, false, 128>) in front of the depth shade pass:
    one mesh of ~40 000 faces x 3 views."""
    mesh = synth.make_mesh(40000, 12)
    assert mesh[1].shape[0] > 32768
    R, T, C, _ = cams(oracle, synth.learned_spherical_views(1, 3, 13), "cpu")
    want = {"mesh_scatter_kernel<8, false, 128>": 1, "mesh_scatter_kernel<4, false>": 0}
    run_mesh(oracle, cuda_device, [mesh], 3, 96, 96, R, T, C, fwd=want, tag="40k faces")


RAGGED = [(600, 3), (1500, 4), (300, 5)]


@pytest.mark.parametrize("H,W", [(45, 70), (33, 31), (7, 5)])
def test_mesh_depth_odd_shapes_cull_no_persp(oracle, cuda_device, H, W):
    """A ragged batch at W % 4 != 0 / W % 32 != 0 / smaller than one tile, with cull_backfaces=True and
    perspective_correct=False (no near-plane clipping)."""
    meshes = [synth.make_mesh(nf, s) for nf, s in RAGGED]
    R, T, C, _ = cams(oracle, synth.learned_spherical_views(3, 4, 7), "cpu")
    res = run_mesh(oracle, cuda_device, meshes, 4, H, W, R, T, C, persp=False, cull=True,
                   fwd={"mesh_shade_clipped_kernel": 0}, tag=f"{H}x{W} cull nopersp")
    assert not res["straddle"]


def test_mesh_depth_near_plane_cull_odd_width(oracle, cuda_device):
    """MESH["near_plane"]'s views (faces cross z = 0.5) at W = 45 with back faces culled, on a ragged batch of two meshes: the
    clipped depth pass runs, and depth and gradients match."""
    c = MESH["near_plane"]
    meshes = [synth.make_mesh(nf, s) for nf, s in c["meshes"]] + [synth.make_mesh(600, 3)]
    views = tuple(t.expand(2, 3).contiguous() for t in c["views"])
    R, T, C, _ = cams(oracle, views, "cpu")
    res = run_mesh(oracle, cuda_device, meshes, 3, 48, 45, R, T, C, cull=True, fwd={"mesh_shade_clipped_kernel<false, true>": 1},
                   tag="near plane cull W=45")
    assert res["straddle"]


def test_mesh_depth_nothing_in_view(oracle, cuda_device):
    """A ragged batch where mesh 0's last view points away from it (the mesh behind the camera) and mesh 1 covers no pixel in
    any view (behind, beside, below): those views are all depth_background with pix_to_face -1, their R / T gradients are
    exactly 0, and so are mesh 1's vertex gradients; the rest matches the oracle and fp64 autograd."""
    dev = cuda_device
    M = 3
    meshes = [synth.make_mesh(nf, s) for nf, s in RAGGED]
    R, T, C, _ = cams(oracle, synth.learned_spherical_views(3, M, 17), "cpu")
    T = T.copy()
    T[2] = (0.0, 0.0, -2.2)                       # mesh 0, view 2: the camera looks away from the object
    T[3] = (0.0, 0.0, -2.2)
    T[4] = (40.0, 0.0, 2.2)
    T[5] = (0.0, -40.0, 2.2)
    off = [2, 3, 4, 5]
    res = run_mesh(oracle, dev, meshes, M, 48, 48, R, T, C, tag="nothing in view")
    for n in off:
        assert torch.equal(res["depth"][n], torch.full_like(res["depth"][n], BGD)) and (res["p2f"][n] == -1).all(), n
        assert torch.equal(res["gR"][n], torch.zeros(3, 3, device=dev)) and torch.equal(res["gT"][n], torch.zeros(3, device=dev)), n
    on = [n for n in range(3 * M) if n not in off]
    assert all(bool((res["p2f"][n] >= 0).any()) for n in on)
    nv0, nv1 = meshes[0][0].shape[0], meshes[1][0].shape[0]
    assert torch.equal(res["gV"][nv0: nv0 + nv1], torch.zeros(nv1, 3, device=dev))
    assert float(res["gVr"][1].abs().max()) == 0 and float(res["gV"][:nv0].abs().max()) > 0


def test_mesh_depth_with_per_vertex_colours(oracle, cuda_device):
    """MVRenderer's geometry when it is given per-vertex colours (PackedMeshes(vert_rgb=...)): the depth masks the colours off,
    so depth bits, pix_to_face and gradients are those of the geometry built without them."""
    meshes = [synth.make_mesh(nf, s) for nf, s in RAGGED]
    R, T, C, _ = cams(oracle, synth.learned_spherical_views(3, 2, 23), "cpu")
    nv = sum(v.shape[0] for v, _ in meshes)
    rgb = torch.rand(nv, 3, generator=torch.Generator().manual_seed(1))
    a = run_mesh(oracle, cuda_device, meshes, 2, 56, 60, R, T, C, vert_rgb=rgb, tag="vert_rgb")
    b = run_mesh(oracle, cuda_device, meshes, 2, 56, 60, R, T, C, tag="no vert_rgb")
    assert torch.equal(a["depth"], b["depth"]) and torch.equal(a["p2f"], b["p2f"])
    assert torch.equal(a["gR"], b["gR"]) and torch.equal(a["gT"], b["gT"])
    assert rel(a["gV"], b["gV"]) < ATOMIC_RTOL


# ------------------------------------------------------------------------------------------------- workspace reuse
def test_mesh_workspace_reuse_across_shaders(oracle, cuda_device):
    """ops._ws_mesh's hints are keyed by (B, M, H, W, K, total_verts), not by the shader: a hard Phong K = 1 forward, a depth
    forward and a K = 1 soft silhouette trust each other's re-armed key plane (on the depth path the clipped pass re-arms the
    pixels of faces crossing the near plane).  A fixed interleaving of Phong, depth, the soft shaders and a point render, far and
    near-plane views, gives every output and fragment of its cold-workspace reference bit for bit, and takes the armed hint for
    depth -> Phong and Phong -> depth.  The depth backward right after its forward (projection reused) equals the cold one, and
    so does one behind a Phong forward of other views (re-projected)."""
    dev = cuda_device
    key = (dev.index, ops._stream(dev))
    H, M = 64, 3
    m = synth.make_meshes(2, 1500, 61)
    geom = ops.PackedMeshes([v for v, _ in m], [f for _, f in m], dev)
    far = (torch.tensor([[15.0, 140.0, -80.0], [200.0, 33.0, 77.0]]), torch.tensor([[10.0, -35.0, 50.0], [0.0, 20.0, -15.0]]),
           torch.tensor([[2.2, 2.0, 2.5], [1.9, 2.25, 3.0]]))
    near = (far[0] + 30.0, far[1], torch.tensor([[1.12, 1.2, 1.3], [1.15, 1.25, 1.18]]))
    cam = {name: cams(oracle, v, dev)[3] for name, v in (("far", far), ("near", near))}
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0, 1.0, 0]], device=dev)
    pts = synth.make_clouds(2, 256, 62).to(dev)
    K_OF = {"phong": 1, "depth": 1, "soft_silhouette": 1, "soft_phong": 2}

    def render(shader, views, R=None, T=None):
        Rv, Tv, Cv = cam[views]
        R, T = (Rv if R is None else R), (Tv if T is None else T)
        if shader == "phong":
            img, fr = ops.render_meshes(geom, M, R, T, Cv, light, col, col, H, fragments=True)
        elif shader == "depth":
            img, fr = ops.render_meshes(geom, M, R, T, Cv, light, col, col, H, shader="hard_depth", depth_background=BGD)
        else:
            img, fr = ops.render_meshes(geom, M, R, T, Cv, light, col, col, H, faces_per_pixel=K_OF[shader], shader=shader, blur_radius=1e-4)
        return img, fr

    def snapshot(img, fr):
        return [img.detach().clone()] + [v.clone() for k, v in sorted(fr.items()) if k != "counters" and v is not None]

    ref = {}
    for shader in K_OF:
        for views in ("far", "near"):
            ops._ws_mesh.pop(key, None)
            img, fr = render(shader, views)
            ref[shader, views] = snapshot(img, fr)
            if views == "near":
                assert int(fr["counters"][L.CNT_STRADDLE]) > 0, shader
    ops._ws_mesh.pop(key, None)
    seq = [("depth", "near"), ("phong", "far"), ("depth", "far"), ("phong", "near"), ("soft_silhouette", "far"), ("depth", "near"),
           ("phong", "near"), ("points", "far"), ("depth", "far"), ("soft_phong", "near"), ("phong", "far"), ("depth", "near"),
           ("soft_silhouette", "near"), ("phong", "far"), ("depth", "far")]
    taken, prev = {}, None
    for i, (shader, views) in enumerate(seq):
        if shader == "points":
            Rv, Tv, _ = cam[views]
            ops.render_points(pts, col, M, Rv, Tv, None, 0.02, col * 0, H, dist=far[2].to(dev).reshape(-1))
            assert ops._ws_mesh.get(key) is None
            prev = shader
            continue
        st = ops._ws_mesh.get(key)
        ws = ops._workspaces.get(key)
        layout = (geom.B, M, H, H, K_OF[shader], geom.total_verts)
        hit = isinstance(st, dict) and ws is not None and st.get("armed") == (ws.data_ptr(), layout)
        taken[prev, shader] = taken.get((prev, shader), 0) + int(hit)
        out = snapshot(*render(shader, views))
        for j, (a, b) in enumerate(zip(out, ref[shader, views])):
            assert torch.equal(a, b), (i, shader, views, j)
        prev = shader
    print(f"armed hints taken: {taken}")
    assert taken.get(("depth", "phong"), 0) >= 1 and taken.get(("phong", "depth"), 0) >= 1
    # backwards: cold (re-projected), warm (projection reused), and out of order (another forward in between: re-projected)
    cot = torch.randn(2 * M, 1, H, H, device=dev, generator=torch.Generator(device=dev).manual_seed(5))

    def depth_grads(views, mode):
        Rg, Tg = (t.clone().requires_grad_() for t in cam[views][:2])
        if mode == "cold":
            ops._ws_mesh.pop(key, None)
        dep, _ = render("depth", views, Rg, Tg)
        if mode == "cold":
            ops._ws_mesh.pop(key, None)
        elif mode == "warm":
            assert ops._ws_mesh[key]["proj"] is not None
        else:
            render("phong", "far" if views == "near" else "near")
        _, n = launches("mesh_project_kernel", lambda: dep.backward(cot))
        assert n == (0 if mode == "warm" else 1), (views, mode, n)
        return Rg.grad, Tg.grad

    for views in ("near", "far"):
        cold = depth_grads(views, "cold")
        assert float(cold[0].abs().max()) > 0
        for mode in ("warm", "out_of_order"):
            got = depth_grads(views, mode)
            assert torch.equal(got[0], cold[0]) and torch.equal(got[1], cold[1]), (views, mode)


# ------------------------------------------------------------------------------------------------- renderer
def pole_angles(B, M):
    """(B, M) views at exactly +-90 degrees (accepted by the rotation guard) and 1e-4 degrees off the pole (rejected: the x axis
    is clamped but not replaced), mixed with ordinary ones."""
    e = torch.tensor([90.0, -90.0, 89.9999, 30.0, -89.9999, 0.0])
    el = e.repeat((B * M + 5) // 6)[: B * M].reshape(B, M)
    az = torch.linspace(-170, 170, B * M).reshape(B, M)
    return az, el, torch.full((B, M), 2.2)


@pytest.mark.parametrize("pc", [False, True])
def test_depth_mvrenderer_redraw_loop(cuda_device, pc):
    """MVRenderer(shader="hard_depth") with views at and next to the poles: the guard rejects the near-pole rotations, the redraw
    loop draws new angles and renders again (a second camera launch); the returned depth is the ops-level depth of the cameras
    the renderer returns, bit for bit, and the angle gradients are finite."""
    dev = cuda_device
    torch.manual_seed(0)
    B, M, H = 2, 6, 48
    az, el, di = (t.to(dev).requires_grad_() for t in pole_angles(B, M))
    r = MVRenderer(M, image_size=H, pc_rendering=pc, shader="hard_depth", depth_background=BGD, light_direction="fixed",
                   points_radius=0.03).eval()
    if pc:
        obj = synth.make_clouds(B, 2048, 71).to(dev)
        (img, cameras), k = launches("look_at_forward", lambda: r(None, obj, az, el, di))
    else:
        obj = [(v.to(dev), f.to(dev)) for v, f in synth.make_meshes(B, 800, 72)]
        (img, cameras), k = launches("look_at_forward", lambda: r(obj, None, az, el, di))
    assert k >= 2, "the redraw loop did not run"
    assert img.shape == (B, M, 1, H, H)
    Rk, Tk = cameras.R.detach(), cameras.T.detach()
    if pc:
        ref, _ = ops.render_points(obj, torch.ones(3, device=dev), M, Rk, Tk, None, 0.03, torch.zeros(3, device=dev), H,
                                   dist=di.detach().reshape(-1), shader="hard_depth", depth_background=BGD)
    else:
        geom = ops.PackedMeshes([v for v, _ in obj], [f for _, f in obj], dev)
        ref, _ = ops.render_meshes(geom, M, Rk, Tk, cameras.get_camera_center().detach(), torch.ones(1, 3, device=dev), None,
                                   torch.zeros(3, device=dev), H, shader="hard_depth", depth_background=BGD)
    assert torch.equal(img.detach().reshape(B * M, 1, H, H), ref)
    assert (ref < BGD).sum() > 100
    g = torch.randn(B, M, 1, H, H, generator=torch.Generator().manual_seed(3)).to(dev)
    (img * g).sum().backward()
    for t in (az, el, di):
        assert t.grad is not None and torch.isfinite(t.grad).all()
    assert float(el.grad.abs().max()) > 0
