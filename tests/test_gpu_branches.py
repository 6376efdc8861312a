"""GPU tests of the dispatch branches behind the public entry points (run on the B200 box with `-m gpu`).

mvr_points_forward / mvr_points_backward / mvr_mesh_backward choose among many kernels and template instances from the
sizes and pointers they are given: three-launch or fused binning (and the fused kernel's cluster size), tiled or generic K,
the backward's register-resident or generic layers, per-point / uniform / no colour gradient, the strip or the plain mesh
backward with vertex gradients.  Every case here compares the CUDA result with the CPU oracle (or the fp64 torch
restatement) at the bars of test_gpu_parity.py, and proves that it reached its branch: the library's launch profiler
(mvr_profile_enable / mvr_profile_collect) counts the launches of the kernel the case is about, so a later change of a
threshold cannot silently move a case off its branch.
"""
import ctypes as C
import time

import numpy as np
import pytest
import torch

from mvtn_b200 import _lib as L
from mvtn_b200 import ops, synth
from test_gpu_parity import GRAD_RTOL, IMG_ATOL, K00, K11, NORM, POINT_GRAD_RTOL, cams, pack_np, rel

pytestmark = pytest.mark.gpu

VERT_GRAD_RTOL = 5e-4          # test_mesh_vertex_gradients' bar (DESIGN.md section 2: the fp32 floor of the vertex chain)


def launches(prefix, fn):
    """fn() with the launch profiler armed for kernels whose name starts with `prefix` (a leading '(' and 'mvr::' are
    ignored; template arguments are spelled as at the launch site) -> (fn's result, number of such launches)."""
    lib = L.load()
    L.check(lib.mvr_profile_enable(prefix.encode()), "mvr_profile_enable")
    try:
        out = fn()
    finally:
        ms, n = C.c_double(0.0), C.c_int(0)
        L.check(lib.mvr_profile_collect(C.byref(ms), C.byref(n)), "mvr_profile_collect")
    return out, n.value


def expect_launches(counts, want, what):
    """want: prefix -> 0 (must not launch) or k >= 1 (at least k launches)."""
    for p, w in want.items():
        got = counts[p]
        assert (got == 0) if w == 0 else (got >= w), f"{what}: {p!r} launched {got} times, want {'0' if w == 0 else f'>= {w}'}"


def stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------------- points
def points_from_view(oracle, p_view, views):
    """World points whose orthographic projection in the first view of `views` is (about) p_view (P,3): x, y in NDC,
    z the view depth -- for clouds placed on purpose (image edges, one tile)."""
    R, T, _ = oracle.look_at(*(t.numpy().ravel() for t in views))
    s = 1.0 / float(views[2].reshape(-1)[0])
    X = (p_view.astype(np.float64) - T[0].astype(np.float64)) @ R[0].astype(np.float64).T / s
    return torch.from_numpy(X.astype(np.float32))[None].contiguous()


def centres_within(oracle, pts, views, n, radius, H, W, cols=None, rows=None):
    """Per point of cloud 0: how many pixel centres (of the given columns / rows, default all) lie strictly inside the
    radius in view n -- the kernels' test, dx*dx + dy*dy < r*r in fp32, on the oracle's projection."""
    R, T, _ = oracle.look_at(*(t.numpy().ravel() for t in views))
    inv = np.float32(1.0) / np.float32(views[2].reshape(-1)[n])            # torch's fp32 1.0 / dist
    p = oracle.project_orthographic(pts[0].numpy(), R[n], T[n], inv)
    cols = np.arange(W) if cols is None else np.asarray(cols)
    rows = np.arange(H) if rows is None else np.asarray(rows)
    xf = np.array([pix_to_ndc(W - 1 - i, W, H) for i in cols], np.float32)
    yf = np.array([pix_to_ndc(H - 1 - j, H, W) for j in rows], np.float32)
    dx = p[:, 0:1] - xf[None]
    dy = p[:, 1:2] - yf[None]
    d2 = (dx * dx)[:, None, :] + (dy * dy)[:, :, None]                     # (P, rows, cols), fp32
    r2 = np.float32(radius) * np.float32(radius)
    return ((d2 < r2) & (p[:, 2:3, None] >= 0)).sum(axis=(1, 2))


def pix_to_ndc(i, S1, S2):
    """mvr_common.cuh pix_to_ndc in fp32: NDC coordinate of the centre of flipped pixel index i."""
    rng = np.float32(2.0)
    if S1 > S2:
        rng = np.float32(S1 // S2) * rng
    off = rng / np.float32(2.0)
    return np.float32(-off + (rng * np.float32(i) + off) / np.float32(S1))


def run_points_case(oracle, dev, pts, views, H, W, K, radius, mode, per_point=False, want_points=True, want_rgb=True,
                    fwd=None, bwd=None, backward=True, tag=""):
    """render_points (fragments on) -> idx / zbuf / dists2 bit-exact, images <= 1e-5; backward with the point / colour
    gradients requested per case -> gR, gT, g_inv_dist (and what was requested) <= 1e-5 of each tensor's largest entry.
    fwd: prefix -> launches wanted in the forward (one forward per prefix, all identical); bwd: (prefix, k) of the backward."""
    B, Np = pts.shape[:2]
    M = views[0].shape[1]
    N = B * M
    R, T, Cc, (Rd, Td, Cd) = cams(oracle, views, dev)
    inv = (1.0 / views[2].reshape(-1)).contiguous()
    if per_point:
        rgb = torch.rand(B, Np, 3, generator=torch.Generator().manual_seed(3))
    else:
        rgb = torch.tensor([0.9, 0.6, 0.3])                  # distinct channels: a swapped colour gradient shows
    bg = torch.tensor([0.1, 0.2, 0.3])
    Rg, Tg, sg = Rd.clone().requires_grad_(), Td.clone().requires_grad_(), inv.to(dev).requires_grad_()
    pg, fg = pts.to(dev).requires_grad_(want_points), rgb.to(dev).requires_grad_(want_rgb)

    def render():
        return ops.render_points(pg, fg, M, Rg, Tg, sg, radius, bg.to(dev), (H, W), points_per_pixel=K, compositor=mode, fragments=True)

    counts = {}
    out = None
    for p in (fwd or {}):
        o, counts[p] = launches(p, render)
        out = out or o
    img, frag = out if out is not None else render()
    expect_launches(counts, fwd or {}, f"[{tag}] forward")
    flags = oracle.COMPOSITE_ALPHA if mode == "alpha" else 0
    t0 = time.perf_counter()
    o = oracle.points_forward(pts.numpy(), rgb.numpy(), M, R, T, inv.numpy(), radius, bg.numpy(), H, W, K, flags)
    t_orc = time.perf_counter() - t0
    idx = frag["idx"].cpu().numpy()
    assert (idx == o["idx"]).all(), f"[{tag}] {int((idx != o['idx']).sum())} point index mismatches"
    assert (frag["zbuf"].cpu().numpy() == o["zbuf"]).all(), f"[{tag}] zbuf"
    assert (frag["dists"].cpu().numpy() == o["dists2"]).all(), f"[{tag}] dists2"
    img_err = float(np.abs(img.detach().cpu().numpy() - o["images"]).max())
    assert img_err <= IMG_ATOL, (tag, img_err)
    errs = {}
    if backward:
        g = torch.randn(N, 3, H, W, generator=torch.Generator().manual_seed(6))
        _, nb = launches(bwd[0], lambda: img.backward(g.to(dev)))
        expect_launches({bwd[0]: nb}, {bwd[0]: bwd[1]}, f"[{tag}] backward")
        counts[bwd[0]] = nb
        t0 = time.perf_counter()
        ob = oracle.points_backward(pts.numpy(), rgb.numpy(), M, R, T, inv.numpy(), radius, H, W, K, flags, idx, g.numpy(),
                                    want_points=want_points, want_rgb=want_rgb)
        t_orc += time.perf_counter() - t0
        assert np.abs(ob["gR"]).max() > 1e-3, f"[{tag}] degenerate case: the reference camera gradient is ~0"
        mine = {"gR": Rg.grad, "gT": Tg.grad, "g_inv_dist": sg.grad}
        if want_points:
            mine["grad_points"] = pg.grad
        else:
            assert pg.grad is None
        if want_rgb:
            mine["grad_rgb"] = fg.grad
        for k, v in mine.items():
            errs[k] = rel(v, ob[k])
        for k, e in errs.items():
            assert e < POINT_GRAD_RTOL, (tag, k, e)
    print(f"[{tag}] launches {counts}  image err {img_err:.1e}  grad errs " + " ".join(f"{k} {e:.1e}" for k, e in errs.items()) +
          f"  oracle {t_orc:.2f}s")
    return dict(idx=idx, o=o, counts=counts)


def bwd_prefix(kt, vrgb, gu):
    return f"points_backward_kernel<{kt}, {str(vrgb).lower()}, {str(gu).lower()}>"


# ---- 1. binning thresholds
@pytest.mark.parametrize("K", [1, 4])
@pytest.mark.parametrize("Np", [16384, 16385, 40000])
def test_points_binning_paths_at_the_point_threshold(oracle, cuda_device, Np, K):
    """Up to BIN_FUSED_MAX_POINTS = 16384 points one fused kernel bins a view; one point more takes the three-launch path
    (pixel table, count, scan, fill)."""
    fused = Np <= 16384
    want = {"points_bin_kernel_fused": 1, "points_bin_scan_kernel": 0} if fused else \
        {"points_bin_kernel_fused": 0, "points_bin_kernel<": 2, "points_bin_scan_kernel": 1}
    mode = "alpha"
    res = run_points_case(oracle, cuda_device, synth.make_clouds(1, Np, 40 + K), synth.learned_spherical_views(1, 2, 41), 96, 96, K,
                          0.02, mode, fwd=want, bwd=(bwd_prefix(K, False, True), 1), tag=f"bin Np={Np} K={K}")
    assert (res["idx"][..., K - 1] >= 0).sum() > 100


@pytest.mark.parametrize("B,M,Np,cs", [(2, 74, 4096, 1), (2, 74, 4097, 4), (1, 147, 4096, 4), (1, 2, 511, 1), (1, 2, 512, 4)])
def test_points_fused_binning_cluster_size_thresholds(oracle, cuda_device, B, M, Np, cs):
    """The fused binning kernel runs as a cluster of 4 CTAs per view when Np > 4096 or (fewer views than SMs and
    Np >= 512), else as one CTA: both sides of both thresholds.  The two launch under the same name, so the side is asserted
    from the host rule and the launch of the fused kernel (and not the three-launch path) from the profiler."""
    N = B * M
    assert cs == (4 if (Np > 4096 or (N < 148 and Np >= 512)) else 1)
    res = run_points_case(oracle, cuda_device, synth.make_clouds(B, Np, 50 + Np), synth.learned_spherical_views(B, M, 51), 32, 32, 4,
                          0.06, "alpha", fwd={"points_bin_kernel_fused": 1, "points_bin_scan_kernel": 0},
                          bwd=(bwd_prefix(4, False, True), 1), tag=f"cluster N={N} Np={Np} cs={cs}")
    assert (res["idx"][..., 3] >= 0).sum() > 10


def wide_view_cloud(oracle):
    """One view at 264 x 4096 (9 x 128 = 1152 tiles): ~1300 points spread over the whole NDC range (x in +-15, y in +-1) and a
    cluster of 200 on the last pixel column x = 4095 (NDC x = -14.996), where the layers go deep."""
    g = np.random.default_rng(7)
    n_field, n_edge = 1300, 200
    field = np.stack([g.uniform(-14.9, 14.9, n_field), g.uniform(-0.95, 0.95, n_field), g.uniform(0.5, 3.0, n_field)], 1)
    edge = np.stack([g.uniform(-15.02, -14.94, n_edge), g.uniform(-0.3, 0.3, n_edge), g.uniform(0.5, 3.0, n_edge)], 1)
    views = (torch.tensor([[0.0]]), torch.tensor([[0.0]]), torch.tensor([[2.0]]))
    return points_from_view(oracle, np.concatenate([field, edge]), views), views


@pytest.mark.parametrize("K,mode", [(4, "alpha"), (5, "norm")])
def test_points_wide_view_more_than_1024_tiles(oracle, cuda_device, K, mode):
    """More than BIN_FUSED_MAX_TILES = 1024 tiles sends a small cloud down the three-launch binning (K = 4); with K = 5 the
    generic path (global key plane, scatter + resolve) writes pixel column 4095, the largest x its 12-bit queue field holds."""
    H, W = 264, 4096
    assert ((H + 31) // 32) * ((W + 31) // 32) == 1152
    pts, views = wide_view_cloud(oracle)
    if K == 4:
        fwd = {"points_bin_kernel<": 2, "points_bin_scan_kernel": 1, "points_tile_kernel<4,": 1}
    else:
        fwd = {"points_scatter_kernel": 1, "points_resolve_kernel<0>": 1}
    res = run_points_case(oracle, cuda_device, pts, views, H, W, K, 0.03, mode, per_point=(mode == "norm"), fwd=fwd,
                          bwd=(bwd_prefix(K if K == 4 else 0, mode == "norm", mode != "norm"), 1), tag=f"wide K={K}")
    idx = res["idx"]
    assert (idx[0, :, W - 1, 0] >= 0).sum() > 10 and (idx[0, :, W - 1, K - 1] >= 0).any()      # the edge column is covered, deeply
    assert (idx[0, :, : W // 2, 0] >= 0).sum() > 1000                                           # and so is the rest of the view


# ---- 2. K sweep
K_SWEEP = [2, 5, 6, 7, 9, 16, 64]


@pytest.mark.parametrize("mode", ["alpha", "norm"])
@pytest.mark.parametrize("K", K_SWEEP)
def test_points_k_sweep(oracle, cuda_device, K, mode):
    """Every K up to 64, forward and backward: K = 2 is tiled and register-resident in the backward, every other K here takes
    the generic forward (scatter + points_resolve_kernel<0>) and the generic backward (KT = 0).  The cloud is dense enough
    that every layer is filled somewhere (K = 64: at least 50 pixels hold 64 points).  Norm-weighted cases use per-point
    colours (with one colour the normalised image is that colour and the camera gradients vanish)."""
    per_point = mode == "norm"
    if K == 2:
        fwd, kt = {"points_tile_kernel<2,": 1, "points_scatter_kernel": 0}, 2
    else:
        fwd, kt = {"points_scatter_kernel": 1, "points_resolve_kernel<0>": 1}, 0
    res = run_points_case(oracle, cuda_device, synth.make_clouds(1, 1200, 60 + K), synth.learned_spherical_views(1, 2, 61), 40, 40, K,
                          0.12, mode, per_point=per_point, fwd=fwd, bwd=(bwd_prefix(kt, per_point, not per_point), 1),
                          tag=f"K={K} {mode}")
    idx = res["idx"]
    assert (idx[..., K - 1] >= 0).sum() >= (50 if K == 64 else 1)
    assert ((idx[..., 1:] != idx[..., :-1]) | (idx[..., 1:] < 0)).all()      # no point twice in a pixel's layers


# ---- 3. queue overflow by construction
@pytest.mark.parametrize("K", [1, 4, 8])
def test_points_tile_queue_overflow(oracle, cuda_device, K):
    """Tile kernel: 600 points inside one 32 x 32 tile, radius larger than the tile's diagonal -- every point covers all 1024
    pixel centres of the tile, so every full round of 256 points has 256 x 1024 candidates for the 2048-entry queue and the
    rest are inserted in place."""
    H = W = 64
    radius = 1.5                                            # tile = 32 px = 1.0 NDC; diagonal 1.414
    g = np.random.default_rng(K)
    # tile (0, 0) = pixels x, y in [0, 32) = NDC x, y in (0, 1] (pixel 0 is the left/top edge: +X left, +Y up)
    p_view = np.stack([g.uniform(0.02, 0.98, 600), g.uniform(0.02, 0.98, 600), g.uniform(0.5, 3.0, 600)], 1)
    views = (torch.tensor([[0.0]]), torch.tensor([[0.0]]), torch.tensor([[2.0]]))
    pts = points_from_view(oracle, p_view, views)
    cnt = centres_within(oracle, pts, views, 0, radius, H, W, cols=range(32), rows=range(32))
    assert cnt.size >= 512 and (cnt == 1024).all(), "every point must cover the whole tile"
    mode = "alpha" if K == 1 else "norm"
    per_point = mode == "norm"
    kt = K if K in (1, 4) else 0
    res = run_points_case(oracle, cuda_device, pts, views, H, W, K, radius, mode, per_point=per_point,
                          fwd={f"points_tile_kernel<{K},": 1}, bwd=(bwd_prefix(kt, per_point, not per_point), 1), tag=f"tile overflow K={K}")
    assert (res["idx"][0, :32, :32, K - 1] >= 0).all()


@pytest.mark.parametrize("K", [3, 5])
def test_points_scatter_queue_overflow(oracle, cuda_device, K):
    """Generic scatter: the 256 point ids of the first CTA each cover more than 16 pixel centres, so together more than
    PS_CAP = 4096 (point, pixel) candidates: the CTA's queue fills and the rest are inserted in place."""
    H = W = 64
    radius = 0.1                                            # pitch 2 / 64: ~32 pixel centres per point
    views = synth.learned_spherical_views(1, 2, 71)
    pts = synth.make_clouds(1, 700, 70)
    for n in range(2):
        cnt = centres_within(oracle, pts, views, n, radius, H, W)
        assert (cnt[:256] > 16).all() and int(cnt[:256].sum()) > 4096, (n, int(cnt[:256].min()), int(cnt[:256].sum()))
    res = run_points_case(oracle, cuda_device, pts, views, H, W, K, radius, "alpha",
                          fwd={"points_scatter_kernel": 1, "points_resolve_kernel<0>": 1}, bwd=(bwd_prefix(0, False, True), 1),
                          tag=f"scatter overflow K={K}")
    assert (res["idx"][..., K - 1] >= 0).sum() > 100


# ---- 4. backward instances
BWD_VARIANTS = {
    # name: (per-point colours, colour requires grad, points require grad)
    "point_rgb": (True, True, True),
    "uniform_rgb_grad": (False, True, True),
    "uniform_rgb_grad_no_points": (False, True, False),
    "cameras_only": (False, False, False),               # MVRenderer's training step: no point or colour gradients
}


@pytest.mark.parametrize("variant", list(BWD_VARIANTS))
@pytest.mark.parametrize("K", [1, 2, 4, 3])
def test_points_backward_instances(oracle, cuda_device, K, variant):
    """points_backward_kernel<KT, VRGB, GU> for KT in {1, 2, 4, 0 (K = 3)} x {per-point colour, one colour with its gradient
    (with and without point gradients), cameras only}: camera gradients always, point / colour gradients where requested."""
    per_point, want_rgb, want_points = BWD_VARIANTS[variant]
    kt = K if K in (1, 2, 4) else 0
    mode = "norm" if (per_point and K in (2, 3)) else "alpha"
    run_points_case(oracle, cuda_device, synth.make_clouds(2, 400, 80 + K), synth.learned_spherical_views(2, 2, 81), 48, 48, K, 0.05, mode,
                    per_point=per_point, want_points=want_points, want_rgb=want_rgb,
                    bwd=(bwd_prefix(kt, per_point, want_rgb and not per_point), 1), tag=f"bwd K={K} {variant} {mode}")


# ---- 5. alignment
def _points_inputs(oracle, dev, K, B=2, M=2, Np=500, H=48, W=70):
    pts = synth.make_clouds(B, Np, 90 + K).to(dev)
    R, T, Cc, (Rd, Td, Cd) = cams(oracle, synth.learned_spherical_views(B, M, 91), dev)
    inv = torch.full((B * M,), 1 / 2.2, device=dev)
    col = torch.tensor([0.9, 0.6, 0.3], device=dev)
    return pts, R, T, Rd, Td, inv, col


@pytest.mark.parametrize("K", [1, 2, 4])
def test_points_backward_takes_a_misaligned_idx(oracle, cuda_device, K):
    """The backward reads a pixel's K ids as one int2 / int4 only when idx is aligned to 4 K bytes; an idx one int32 off (a slice
    of a larger buffer) takes the generic KT = 0 kernel.  K = 1 has no such requirement (any int32 pointer is aligned): the
    offset call still runs the K = 1 kernel.  Both calls agree with the oracle and with each other."""
    dev = cuda_device
    B, M, Np, H, W = 2, 2, 500, 48, 70
    pts, R, T, Rd, Td, inv, col = _points_inputs(oracle, dev, K)
    img, frag = ops.render_points(pts, col, M, Rd, Td, inv, 0.05, torch.zeros(3, device=dev), (H, W), points_per_pixel=K,
                                  compositor="alpha", fragments=True)
    idx = frag["idx"]
    buf = torch.empty(idx.numel() + 1, dtype=torch.int32, device=dev)
    buf[1:].copy_(idx.reshape(-1))
    idx_off = buf[1:]
    assert idx.data_ptr() % (4 * K) == 0 and idx_off.data_ptr() % 4 == 0
    assert (idx_off.data_ptr() % (4 * K) != 0) == (K > 1)
    g = torch.randn(B * M, 3, H, W, device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    lib = L.load()
    ws = ops.workspace(dev, lib.mvr_points_workspace_bytes(B, Np, M, H, W, K, 0.05))
    outs = {}
    for name, ix, kt in (("aligned", idx, K), ("offset", idx_off, K if K == 1 else 0)):
        gR = torch.empty(B * M, 3, 3, device=dev); gT = torch.empty(B * M, 3, device=dev); gs = torch.empty(B * M, device=dev)
        gP = torch.zeros_like(pts); gF = torch.zeros(3, device=dev)

        def call():
            L.check(lib.mvr_points_backward(pts.data_ptr(), col.data_ptr(), B, Np, M, Rd.data_ptr(), Td.data_ptr(), inv.data_ptr(), 0.05,
                                            H, W, K, L.COMPOSITE_ALPHA, None, ix.data_ptr(), None, g.data_ptr(), gR.data_ptr(), gT.data_ptr(),
                                            gs.data_ptr(), gP.data_ptr(), gF.data_ptr(), ws.data_ptr(), ws.numel(), stream()), "bwd")
        _, n = launches(f"points_backward_kernel<{kt},", call)
        assert n == 1, (name, kt, n)
        outs[name] = dict(gR=gR, gT=gT, g_inv_dist=gs, grad_points=gP, grad_rgb=gF)
    ob = oracle.points_backward(pts.cpu().numpy(), col.cpu().numpy(), M, R, T, inv.cpu().numpy(), 0.05, H, W, K, oracle.COMPOSITE_ALPHA,
                                idx.cpu().numpy(), g.cpu().numpy(), want_points=True, want_rgb=True)
    bitwise = {}
    for k in ob:
        for name in outs:
            assert rel(outs[name][k], ob[k]) < POINT_GRAD_RTOL, (name, k)
        assert rel(outs["offset"][k], outs["aligned"][k].cpu().numpy()) < POINT_GRAD_RTOL, k
        bitwise[k] = bool(torch.equal(outs["offset"][k], outs["aligned"][k]))
    assert float(outs["aligned"]["gR"].abs().max()) > 0
    print(f"[misaligned idx K={K}] offset kernel KT={K if K == 1 else 0}; bit-identical to the aligned call: {bitwise}")


@pytest.mark.parametrize("K", [2, 4])
def test_points_forward_rejects_a_misaligned_idx(oracle, cuda_device, K):
    """The forward stores a pixel's K ids as one int2 / int4 for K = 2 / 4: an idx not aligned to 4 K bytes is rejected on the
    host with status -10 before anything is launched; an aligned slice of the same buffer renders normally."""
    dev = cuda_device
    B, M, Np, H, W = 2, 2, 500, 48, 70
    pts, R, T, Rd, Td, inv, col = _points_inputs(oracle, dev, K)
    lib = L.load()
    bg = torch.zeros(3, device=dev)
    ref_img, ref = ops.render_points(pts, col, M, Rd, Td, inv, 0.05, bg, (H, W), points_per_pixel=K, compositor="alpha", fragments=True)
    n_idx = B * M * H * W * K
    buf = torch.full((n_idx + 8,), 7, dtype=torch.int32, device=dev)
    img = torch.empty(B * M, 3, H, W, device=dev)
    ws = ops.workspace(dev, lib.mvr_points_workspace_bytes(B, Np, M, H, W, K, 0.05))

    def fwd(ptr):
        return lib.mvr_points_forward(pts.data_ptr(), col.data_ptr(), B, Np, M, Rd.data_ptr(), Td.data_ptr(), inv.data_ptr(), 0.05,
                                      bg.data_ptr(), H, W, K, L.COMPOSITE_ALPHA, None, img.data_ptr(), ptr, None, None, None,
                                      ws.data_ptr(), ws.numel(), stream())
    assert buf.data_ptr() % 16 == 0
    for off in range(1, K):                                  # every misaligned int32 offset
        n0 = lib.mvr_launch_count()
        rc = fwd(buf.data_ptr() + 4 * off)
        assert rc == -10 and b"aligned" in lib.mvr_last_error_string(), (off, rc)
        assert lib.mvr_launch_count() == n0
    torch.cuda.synchronize()
    assert (buf == 7).all()                                  # nothing was written
    off = K                                                  # the next aligned slice (4 K bytes in)
    L.check(fwd(buf.data_ptr() + 4 * off), "mvr_points_forward")
    assert torch.equal(buf[off:off + n_idx].view_as(ref["idx"]), ref["idx"]) and torch.equal(img, ref_img)


# ------------------------------------------------------------------------------------------------- meshes
def ragged_meshes():
    """Three meshes of ~60, ~1200 and ~200 faces: every vertex offset but the first is non-zero."""
    return [synth.make_mesh(60, 101), synth.make_mesh(1200, 102), synth.make_mesh(200, 103)]


MESH_LIGHT = [[0.3, 1.0, -0.5]]
MESH_COL = [0.9, 0.7, 0.5]
GV_CASES = {
    # name: (H, W, K, per-vertex colour, bf16 normalised cotangent, kernel)
    "strip_uniform_rgb": (64, 64, 1, False, False, "mesh_backward_kernel_strip<2, false, true>"),
    "strip_vertex_rgb": (64, 64, 1, True, False, "mesh_backward_kernel_strip<2, true, true>"),
    "plain_uniform_rgb_w97_k2": (97, 97, 2, False, False, "mesh_backward_kernel<2, false, true>"),
    "plain_vertex_rgb_w97": (97, 97, 1, True, False, "mesh_backward_kernel<2, true, true>"),
    "plain_bf16_normalised": (64, 64, 1, False, True, "mesh_backward_kernel<2, false, true>"),
}


def _mesh_setup(oracle, dev, meshes, M, vrgb, seed=5):
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev, vert_rgb=vrgb)
    views = synth.learned_spherical_views(len(meshes), M, seed)
    R, T, Cc, (Rd, Td, Cd) = cams(oracle, views, dev)
    return geom, views, R, T, Cc, Rd, Td, Cd


@pytest.mark.parametrize("name", list(GV_CASES))
def test_mesh_vertex_gradient_kernels_match_the_oracle(oracle, cuda_device, name):
    """mvr_mesh_backward with grad_verts / grad_normals on a ragged batch, against the oracle's raw outputs (before the normals
    chain): the strip and the plain kernel, one colour and per-vertex colours, and a bf16 normalised cotangent (plain kernel
    only).  The per-mesh vertex offsets enter the atomics' addresses: a wrong offset moves a mesh's gradients to another's rows."""
    dev = cuda_device
    H, W, K, per_vertex, bf16, kernel = GV_CASES[name]
    meshes = ragged_meshes()
    B, M = len(meshes), 2
    vp, fp, voff, foff = pack_np(meshes)
    assert (np.diff(voff) > 0).all() and voff[1] > 0
    vrgb = torch.rand(voff[-1], 3, generator=torch.Generator().manual_seed(9)) if per_vertex else None
    geom, views, R, T, Cc, Rd, Td, Cd = _mesh_setup(oracle, dev, meshes, M, vrgb)
    light = torch.tensor(MESH_LIGHT, device=dev); col = torch.tensor(MESH_COL, device=dev)
    img, frag = ops.render_meshes(geom, M, Rd, Td, Cd, light, None if per_vertex else col, col * 0.5, (H, W), faces_per_pixel=K,
                                  normalize=NORM if bf16 else None, out_dtype=torch.bfloat16 if bf16 else None)
    p2f = frag["pix_to_face"]
    g = torch.randn(B * M, 3, H, W, generator=torch.Generator().manual_seed(4))
    gd = g.to(dev).to(torch.bfloat16 if bf16 else torch.float32).contiguous()
    lib = L.load()
    N, Vt, Ft = B * M, geom.total_verts, geom.total_faces
    gR = torch.empty(N, 3, 3, device=dev); gT = torch.empty(N, 3, device=dev); gC = torch.empty(N, 3, device=dev)
    gV = torch.zeros(Vt, 3, device=dev); gN = torch.zeros(Vt, 3, device=dev)
    ws = ops.workspace(dev, lib.mvr_mesh_workspace_bytes(B, M, H, W, K, Vt, Ft))
    flags = L.PERSPECTIVE_CORRECT | (L.RGB_PER_ELEMENT if per_vertex else 0) | (L.IMAGES_BF16 if bf16 else 0)

    def call():
        L.check(lib.mvr_mesh_backward(geom.geometry.data_ptr(), geom.vert_off.data_ptr(), geom.face_off.data_ptr(), B, M, Vt, Ft,
                                      geom.max_verts, Rd.data_ptr(), Td.data_ptr(), Cd.data_ptr(), light.data_ptr(), 0,
                                      None if per_vertex else col.data_ptr(), K00, K11, 0.5, H, W, K, flags,
                                      ops._out_norm(NORM) if bf16 else None, p2f.data_ptr(), gd.data_ptr(), gR.data_ptr(), gT.data_ptr(),
                                      gC.data_ptr(), gV.data_ptr(), gN.data_ptr(), ws.data_ptr(), ws.numel(), stream()), "mvr_mesh_backward")
    _, n = launches(kernel, call)
    assert n == 1, (kernel, n)
    std = torch.tensor(NORM[1]).view(1, 3, 1, 1)
    g_raw = (gd.float().cpu() / std).numpy() if bf16 else g.numpy()
    nrm = oracle.packed_vertex_normals(vp, fp, voff, foff)
    rgb = vrgb.numpy() if per_vertex else np.array(MESH_COL, np.float32)
    t0 = time.perf_counter()
    ob = oracle.mesh_backward(vp, fp, voff, foff, nrm, rgb, M, R, T, Cc, np.array(MESH_LIGHT, np.float32), K00, K11, H, W, K,
                              oracle.PERSPECTIVE_CORRECT, p2f.cpu().numpy(), g_raw, want_verts=True)
    t_orc = time.perf_counter() - t0
    for b in range(B):      # every mesh of the batch receives vertex gradients
        assert np.abs(ob["grad_verts"][voff[b]:voff[b + 1]]).max() > 0 and np.abs(ob["grad_normals"][voff[b]:voff[b + 1]]).max() > 0
    errs = {k: rel(v, ob[k]) for k, v in (("gR", gR), ("gT", gT), ("gC", gC))}
    errs.update(grad_verts=rel(gV, ob["grad_verts"]), grad_normals=rel(gN, ob["grad_normals"]))
    print(f"[{name}] {kernel} x{n}  errs " + " ".join(f"{k} {e:.1e}" for k, e in errs.items()) + f"  oracle {t_orc:.2f}s")
    for k in ("gR", "gT", "gC"):
        assert errs[k] < GRAD_RTOL, (k, errs[k])
    for k in ("grad_verts", "grad_normals"):
        assert errs[k] < VERT_GRAD_RTOL, (k, errs[k])


def test_mesh_normals_backward_ragged_batch(cuda_device):
    """mvr_mesh_normals_backward (d/d unit normals -> d/d vertices through [upstream] Meshes._compute_vertex_normals) on the
    ragged batch, against torch.autograd of torch_ref.vertex_normals in fp64, mesh by mesh."""
    from oracle import torch_ref as tr
    dev = cuda_device
    meshes = ragged_meshes()
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    vp, fp, voff, foff = pack_np(meshes)
    gn = torch.randn(geom.total_verts, 3, generator=torch.Generator().manual_seed(8))
    gN = gn.to(dev).contiguous(); gV = torch.zeros(geom.total_verts, 3, device=dev)
    lib = L.load()

    def call():
        L.check(lib.mvr_mesh_normals_backward(geom.geometry.data_ptr(), geom.vert_off.data_ptr(), geom.face_off.data_ptr(), geom.B,
                                              geom.total_verts, geom.total_faces, geom.max_faces, gN.data_ptr(), gV.data_ptr(), stream()),
                "mvr_mesh_normals_backward")
    _, n = launches("geom_normals_bwd_face_kernel", call)
    assert n == 1
    vd = torch.from_numpy(vp).double().requires_grad_()
    loss = 0
    for b, (_, f) in enumerate(meshes):
        s = slice(int(voff[b]), int(voff[b + 1]))
        loss = loss + (tr.vertex_normals(vd[s], f) * gn[s].double()).sum()
    loss.backward()
    for b in range(len(meshes)):
        s = slice(int(voff[b]), int(voff[b + 1]))
        assert float(vd.grad[s].abs().max()) > 0
    err = rel(gV, vd.grad.numpy())
    print(f"[normals backward] geom_normals_bwd_face_kernel x{n}  err {err:.1e}")
    assert err < VERT_GRAD_RTOL


def test_mesh_vertex_gradients_ragged_end_to_end(oracle, cuda_device):
    """render_meshes(..., verts=vg) on the ragged batch against torch.autograd of the fp64 restatement (as
    test_mesh_vertex_gradients does for one mesh); then the fused entry mvr_mesh_backward_angles, followed by
    mvr_mesh_normals_backward, gives the vertex gradient of the two-node chain (_LookAt + render_meshes) -- to the order of
    the atomics -- and its angle gradients."""
    from oracle import torch_ref as tr
    dev = cuda_device
    meshes = ragged_meshes()
    B, M, H = len(meshes), 2, 64
    vp, fp, voff, foff = pack_np(meshes)
    views = synth.learned_spherical_views(B, M, 6)
    R, T, Cc, (Rd, Td, Cd) = cams(oracle, views, dev)
    f_packed = torch.cat([f for _, f in meshes]).to(dev)
    nv, nf = [v.shape[0] for v, _ in meshes], [f.shape[0] for _, f in meshes]
    vg = torch.from_numpy(vp).to(dev).requires_grad_()
    geom = ops.PackedMeshes.from_packed(vg.detach(), f_packed, nv, nf)
    col = torch.tensor(MESH_COL, device=dev); light = torch.tensor(MESH_LIGHT, device=dev)
    img, frag = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col, H, verts=vg)
    g = torch.randn(B * M, 3, H, H, generator=torch.Generator().manual_seed(4))
    _, n = launches("mesh_backward_kernel_strip<2, false, true>", lambda: img.backward(g.to(dev)))
    assert n == 1
    p2f = frag["pix_to_face"].cpu().numpy()
    D = torch.float64
    vd = torch.from_numpy(vp).to(D).requires_grad_()
    loss = 0
    for b, (_, f) in enumerate(meshes):
        s = slice(int(voff[b]), int(voff[b + 1]))
        nd = tr.vertex_normals(vd[s], f)
        for m in range(M):
            k = b * M + m
            im, _ = tr.render_mesh_view(vd[s], f, nd, torch.tensor(MESH_COL, dtype=D).expand(nv[b], 3), torch.from_numpy(R[k]).to(D),
                                        torch.from_numpy(T[k]).to(D), torch.from_numpy(Cc[k]).to(D), torch.tensor(MESH_LIGHT[0], dtype=D),
                                        torch.tensor(MESH_COL, dtype=D), K00, K11, H, H, p2f=torch.from_numpy(p2f[k, ..., 0]).long())
            loss = loss + (im * g[k].to(D)).sum()
    loss.backward()
    err = rel(vg.grad, vd.grad.numpy())
    assert err < VERT_GRAD_RTOL, err
    # the fused angles entry against the two-node chain
    a, e, d = (t.to(dev).reshape(-1).clone().requires_grad_() for t in views)
    R2, T2, C2, _ = ops._LookAt.apply(a, e, d)
    vg2 = torch.from_numpy(vp).to(dev).requires_grad_()
    img2, frag2 = ops.render_meshes(geom, M, R2, T2, C2, light, col, col, H, verts=vg2)
    cot = g.to(dev)
    img2.backward(cot)
    lib = L.load()
    Vt, Ft = geom.total_verts, geom.total_faces
    gV = torch.zeros(Vt, 3, device=dev); gN = torch.zeros(Vt, 3, device=dev)
    ga, ge, gd = (torch.empty(B * M, device=dev) for _ in range(3))
    ws = ops.workspace(dev, lib.mvr_mesh_workspace_bytes(B, M, H, H, 1, Vt, Ft))
    Rc, Tc, Cc2 = (t.detach().contiguous() for t in (R2, T2, C2))

    def fused():
        L.check(lib.mvr_mesh_backward_angles(geom.geometry.data_ptr(), geom.vert_off.data_ptr(), geom.face_off.data_ptr(), B, M, Vt, Ft,
                                             geom.max_verts, Rc.data_ptr(), Tc.data_ptr(), Cc2.data_ptr(), light.data_ptr(), 0, col.data_ptr(),
                                             K00, K11, 0.5, H, H, 1, L.PERSPECTIVE_CORRECT, None, frag2["pix_to_face"].data_ptr(), cot.data_ptr(),
                                             a.detach().data_ptr(), e.detach().data_ptr(), d.detach().data_ptr(), ga.data_ptr(), ge.data_ptr(),
                                             gd.data_ptr(), None, None, None, gV.data_ptr(), gN.data_ptr(), ws.data_ptr(), ws.numel(), stream()),
                "mvr_mesh_backward_angles")
        L.check(lib.mvr_mesh_normals_backward(geom.geometry.data_ptr(), geom.vert_off.data_ptr(), geom.face_off.data_ptr(), B, Vt, Ft,
                                              geom.max_faces, gN.data_ptr(), gV.data_ptr(), stream()), "mvr_mesh_normals_backward")
    _, n = launches("mesh_backward_kernel_strip<2, false, true>", fused)
    assert n == 1
    err_fused = rel(gV, vg2.grad.cpu().numpy())
    err_angles = max(rel(x, y.grad.cpu().numpy()) for x, y in ((ga, a), (ge, e), (gd, d)))
    print(f"[ragged end to end] vertex grad err {err:.1e} vs fp64; fused angles entry vs two-node chain: verts {err_fused:.1e} "
          f"angles {err_angles:.1e}")
    assert err_fused < POINT_GRAD_RTOL and err_angles < POINT_GRAD_RTOL
    assert float(vg2.grad.abs().max()) > 0 and float(a.grad.abs().max()) > 0
