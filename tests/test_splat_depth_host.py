"""CPU tests of the splat depth reference (tests/splat_depth_ref.py) against the per-pixel loop the CUDA kernels evaluate
(mvr_points.cu composite_hit_pixel<..., SPLAT> / points_splat_backward_kernel):

  over the valid entries k of a pixel's K-list, nearest first: alpha_k = 1 - d2_k / r^2, c_k = sum_{j <= k} alpha_j,
  m_k = min(c_k, 1), stopping after the first entry with c_k > 1;  depth = sum_k (m_k - m_prev) z_k + (1 - m_last) bg;
  d/d z_k = g (m_k - m_prev);  Z_stop = z of the first entry with c > 1, else bg;  d/d alpha_j = g (z_j - Z_stop) while c_j <= 1.

Forward and autograd gradients in fp64: sums of exactly 1, alpha = 1, K = 1, empty pixels, background 0, a slightly negative
alpha, lists that saturate before their end.  Then the restatement's fragments against the C oracle, and the argument checks
of the C entry points."""
import numpy as np
import pytest
import torch

import splat_depth_ref
from mvtn_b200 import _lib as L

D = torch.float64


def loop(idx, zbuf, alpha, bg, g):
    """The kernels' per-pixel loops in fp64 -> depth (N,H,W,1), d/d zbuf, d/d alpha."""
    N, H, W, K = idx.shape
    depth = torch.zeros((N, H, W, 1), dtype=D)
    gz, ga = torch.zeros_like(zbuf), torch.zeros_like(alpha)
    for n, y, x in np.ndindex(N, H, W):
        ks = [k for k in range(K) if idx[n, y, x, k] >= 0]
        c, zstop = 0.0, bg
        for k in ks:
            c += float(alpha[n, y, x, k])
            if c > 1.0:
                zstop = float(zbuf[n, y, x, k])
                break
        c, mprev, d, gg = 0.0, 0.0, 0.0, float(g[n, y, x, 0])
        for k in ks:
            c += float(alpha[n, y, x, k])
            mk = min(c, 1.0)
            d += (mk - mprev) * float(zbuf[n, y, x, k])
            gz[n, y, x, k] = gg * (mk - mprev)
            mprev = mk
            if c <= 1.0:
                ga[n, y, x, k] = gg * (float(zbuf[n, y, x, k]) - zstop)
            if c > 1.0:
                break
        depth[n, y, x, 0] = d + (1.0 - mprev) * bg
    return depth, gz, ga


def lists(seed, N=2, H=5, W=6, K=4, amax=0.9):
    """Random K-lists (filled slots a prefix, as the rasterizer leaves them), ascending z, alpha in (0, amax]."""
    gen = torch.Generator().manual_seed(seed)
    n = torch.randint(0, K + 1, (N, H, W, 1), generator=gen)
    idx = torch.where(torch.arange(K) < n, torch.randint(0, 50, (N, H, W, K), generator=gen), torch.full((N, H, W, K), -1))
    z = (1 + 3 * torch.rand(N, H, W, K, dtype=D, generator=gen)).sort(-1).values
    zbuf = torch.where(idx >= 0, z, torch.full_like(z, -1.0))
    alpha = torch.where(idx >= 0, amax * torch.rand(N, H, W, K, dtype=D, generator=gen) + 1e-3, torch.zeros_like(z))
    return idx, zbuf, alpha


def check(idx, zbuf, alpha, bg, seed=0):
    zbuf, alpha = zbuf.clone().requires_grad_(), alpha.clone().requires_grad_()
    out = splat_depth_ref.splat_depth_blend(idx, zbuf, alpha, bg)
    g = torch.randn(out.shape, dtype=D, generator=torch.Generator().manual_seed(seed + 100))
    out.backward(g)
    ref, gz, ga = loop(idx, zbuf.detach(), alpha.detach(), bg, g)
    assert torch.allclose(out.detach(), ref, rtol=1e-12, atol=1e-12 * max(abs(bg), 1.0)), float((out.detach() - ref).abs().max())
    assert torch.allclose(zbuf.grad, gz, rtol=1e-12, atol=1e-14)
    assert torch.allclose(alpha.grad, ga, rtol=1e-12, atol=1e-12 * max(abs(bg), 1.0)), float((alpha.grad - ga).abs().max())
    return out.detach(), zbuf.grad, alpha.grad


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_lists(seed):
    idx, zbuf, alpha = lists(seed)
    c = alpha.cumsum(-1)
    assert ((c > 1) & (idx >= 0)).any() and ((c[..., -1] <= 1) & (idx[..., 0] >= 0)).any(), "both saturated and open pixels"
    check(idx, zbuf, alpha, 100.0, seed)


def test_list_saturating_before_its_end():
    """c passes 1 at the second of four entries: the later two get no weight and no gradient; the second's z is Z_stop."""
    idx = torch.tensor([[[[4, 9, 2, 7]]]])
    zbuf = torch.tensor([[[[1.0, 1.5, 2.0, 2.5]]]], dtype=D)
    alpha = torch.tensor([[[[0.7, 0.6, 0.9, 0.2]]]], dtype=D)
    out, gz, ga = check(idx, zbuf, alpha, 100.0)
    assert abs(float(out) - (0.7 * 1.0 + 0.3 * 1.5)) < 1e-15
    assert float(gz[0, 0, 0, 2]) == 0 and float(gz[0, 0, 0, 3]) == 0 and float(ga[0, 0, 0, 1:].abs().max()) == 0
    assert float(ga[0, 0, 0, 0]) != 0


def test_sum_of_exactly_one():
    """alpha 0.5 + 0.5 reaches c = 1 exactly: the clamp passes the gradient there (c <= 1), the loop goes on, and Z_stop is the
    next entry (pixel 0) or the background (pixel 1, where the list ends)."""
    idx = torch.tensor([[[[3, 5, 7], [1, 2, -1]]]])
    zbuf = torch.tensor([[[[1.5, 2.0, 2.5], [1.0, 1.4, -1.0]]]], dtype=D)
    alpha = torch.tensor([[[[0.5, 0.5, 0.25], [0.5, 0.5, 0.0]]]], dtype=D)
    out, gz, ga = check(idx, zbuf, alpha, 100.0)
    assert float(gz[0, 0, 0, 2]) == 0.0 and float(ga[0, 0, 0, 2]) == 0.0
    assert float(ga[0, 0, 0, 1]) != 0.0 and float(ga[0, 0, 1, 1]) != 0.0
    assert float(out[0, 0, 1, 0]) == 0.5 * 1.0 + 0.5 * 1.4


def test_alpha_one_point_on_a_pixel_centre():
    """alpha = 1 (d2 = 0): the first entry takes all the weight; c = 1 exactly, so its alpha keeps a gradient toward Z_stop."""
    idx = torch.tensor([[[[3, 5], [8, -1]]]])
    zbuf = torch.tensor([[[[1.2, 2.0], [1.7, -1.0]]]], dtype=D)
    alpha = torch.tensor([[[[1.0, 0.3], [1.0, 0.0]]]], dtype=D)
    out, _, ga = check(idx, zbuf, alpha, 100.0)
    assert float(out[0, 0, 0, 0]) == 1.2 and float(out[0, 0, 1, 0]) == 1.7
    assert float(ga[0, 0, 0, 0]) != 0 and float(ga[0, 0, 1, 0]) != 0


def test_k1():
    idx, zbuf, alpha = lists(3, K=1, amax=1.0)
    check(idx, zbuf, alpha, 100.0)


def test_empty_pixels_hold_the_background_with_zero_gradient():
    idx = torch.full((1, 3, 4, 3), -1)
    zbuf, alpha = torch.full((1, 3, 4, 3), -1.0, dtype=D), torch.zeros((1, 3, 4, 3), dtype=D)
    out, gz, ga = check(idx, zbuf, alpha, 7.5)
    assert torch.equal(out, torch.full_like(out, 7.5))
    assert float(gz.abs().max()) == 0.0 and float(ga.abs().max()) == 0.0


def test_background_zero():
    idx, zbuf, alpha = lists(4)
    idx[0, 0] = -1      # a row of empty pixels
    out, _, _ = check(idx, zbuf, alpha, 0.0)
    empty = (idx < 0).all(-1)
    assert empty.any() and bool((out[..., 0][empty] == 0).all())


def test_slightly_negative_alpha():
    """A point one ulp outside the weight radius (the raster radius is r * r in fp32, the weight radius the double r * r rounded):
    alpha is kept negative, not clamped -- it lowers c and weighs its z negatively."""
    idx = torch.tensor([[[[2, 6, 4], [2, 6, -1]]]])
    zbuf = torch.tensor([[[[1.0, 1.3, 1.6], [1.0, 1.3, -1.0]]]], dtype=D)
    alpha = torch.tensor([[[[0.6, -1e-7, 0.5], [-1e-7, 0.3, 0.0]]]], dtype=D)
    out, _, ga = check(idx, zbuf, alpha, 100.0)
    assert float(out[0, 0, 1, 0]) == pytest.approx(-1e-7 * 1.0 + 0.3 * 1.3 + (1 - 0.3 + 1e-7) * 100.0, rel=1e-14)
    assert float(ga[0, 0, 0, 1]) != 0


def test_given_stop_decision():
    """stopped= replaces the decision c > 1 taken from alpha: a pixel whose c is 1 + 1e-12 in fp64 but which the kernels saw
    saturate one entry later is blended as they did."""
    idx = torch.tensor([[[[1, 2, 3]]]])
    zbuf = torch.tensor([[[[1.0, 2.0, 3.0]]]], dtype=D)
    alpha = torch.tensor([[[[0.5, 0.5 + 1e-12, 0.5]]]], dtype=D)
    own = splat_depth_ref.splat_depth_blend(idx, zbuf, alpha, 100.0)
    given = splat_depth_ref.splat_depth_blend(idx, zbuf, alpha, 100.0, stopped=torch.tensor([[[[False, False, True]]]]))
    assert float(own) == pytest.approx(0.5 + 0.5 * 2.0, abs=1e-11)
    assert float(given) == pytest.approx(0.5 + (0.5 + 1e-12) * 2.0 + (1 - 1.0 - 1e-12) * 3.0, abs=1e-11)


@pytest.mark.parametrize("K,H,W", [(1, 24, 24), (4, 20, 27), (8, 31, 18)])
def test_restatement_fragments_are_the_oracle_s(oracle, K, H, W):
    """render_points_view_splat_depth's idx and zbuf equal the C oracle's points_forward(..., K) fragments (square and
    non-square images), and its alpha is 1 - dists2 / r^2."""
    from mvtn_b200 import synth
    B, Np, M, rad = 2, 300, 2, 0.06
    pts = synth.make_clouds(B, Np, 21)
    az, el, di = synth.learned_spherical_views(B, M, 22)
    R, T, _ = oracle.look_at(*(t.numpy().ravel().astype(np.float32) for t in (az, el, di)))
    s = (1.0 / di.numpy().ravel().astype(np.float64)).astype(np.float32)
    o = oracle.points_forward(pts.numpy(), np.ones(3, np.float32), M, R, T, s, rad, np.zeros(3, np.float32), H, W, K, 0)
    for n in range(B * M):
        # the oracle's fp32 projection, through an identity view: the fragments are decided in fp32, as by the oracle
        p32 = torch.from_numpy(oracle.project_orthographic(pts[n // M].numpy(), R[n], T[n], s[n]))
        _, frag = splat_depth_ref.render_points_view_splat_depth(p32, torch.eye(3), torch.zeros(3), 1.0, rad, H, W, K)
        assert torch.equal(frag["idx"].int(), torch.from_numpy(o["idx"][n])), n
        assert int((frag["idx"] >= 0).sum()) > 20
        valid = frag["idx"] >= 0
        assert torch.equal(frag["zbuf"][valid], torch.from_numpy(o["zbuf"][n])[valid])
        want = 1 - torch.from_numpy(o["dists2"][n]).to(D) / (rad * rad)
        assert float((frag["alpha"][valid].to(D) - want[valid]).abs().max()) < 1e-6


# ------------------------------------------------------------------------------------------------- argument checks
FAKE = 1 << 20      # never dereferenced: every call below is refused before any CUDA call


def _args(lib, entry, **kw):
    a = dict(points=FAKE, B=1, Np=100, M=2, R=FAKE, T=FAKE, s=FAKE, radius=0.02, bg=100.0, H=16, W=16, K=4, flags=0)
    if entry == "forward":
        a.update(depth=FAKE, idx=FAKE, mask=FAKE)
    else:
        a.update(idx=FAKE, mask=FAKE, grad_depth=FAKE, gR=FAKE, gT=FAKE, gs=FAKE, gP=None)
    a.update(ws=FAKE, ws_bytes=None, stream=None)
    a.update(kw)
    if a["ws_bytes"] is None:
        a["ws_bytes"] = lib.mvr_points_workspace_bytes(a["B"], a["Np"], a["M"], a["H"], a["W"], a["K"], a["radius"])
    return list(a.values())


NAN, INF = float("nan"), float("inf")
CASES = [(dict(K=0), -3, b"points_per_pixel"), (dict(K=65), -3, b"points_per_pixel"), (dict(bg=INF), -7, b"depth_background"),
         (dict(bg=-INF), -7, b"depth_background"), (dict(bg=NAN), -7, b"depth_background"), (dict(ws_bytes=1), -8, b"workspace too small"),
         (dict(flags=L.IMAGES_BF16), -11, b"MVR_SCALE_IS_DIST only"), (dict(flags=L.IDX_SPARSE), -11, b"MVR_SCALE_IS_DIST only"),
         (dict(flags=L.COMPOSITE_ALPHA), -11, b"MVR_SCALE_IS_DIST only"),
         (dict(flags=L.RGB_PER_ELEMENT | L.SCALE_IS_DIST), -11, b"MVR_SCALE_IS_DIST only"), (dict(R=None), -6, b"null pointer"),
         (dict(mask=None), -6, b"null pointer"), (dict(radius=0.0), -4, b"radius"), (dict(H=0), -2, b"image size")]


@pytest.mark.skipif(torch.cuda.is_available(), reason="the pointers are fake: they must never reach a device")
@pytest.mark.parametrize("entry", ["forward", "backward"])
def test_splat_depth_argument_checks(entry):
    """Each bad argument alone: the status, a message naming it and the entry point, no launch.  B * M = 0 returns 0 at once."""
    try:
        lib = L.load()
    except Exception as e:      # noqa: BLE001 -- the library needs the CUDA runtime to load
        pytest.skip(f"libmvr_b200.so does not load here: {e}")
    fn = getattr(lib, f"mvr_points_splat_depth_{entry}")
    for kw, code, what in CASES:
        n0 = lib.mvr_launch_count()
        rc = fn(*_args(lib, entry, **kw))
        msg = lib.mvr_last_error_string()
        assert rc == code, (entry, kw, rc, msg)
        assert what in msg and f"mvr_points_splat_depth_{entry}".encode() in msg, (entry, kw, msg)
        assert lib.mvr_launch_count() == n0
    for B, M in ((0, 2), (1, 0)):
        n0 = lib.mvr_launch_count()
        assert fn(*_args(lib, entry, B=B, M=M, points=None, R=None, T=None, s=None, ws=None, ws_bytes=0)) == 0
        assert lib.mvr_launch_count() == n0
