"""shader="splat_depth" on the GPU: the K nearest points of each pixel blended into one depth plane by the cumulative sum of their
splat weights alpha = 1 - d2 / r^2 clamped at 1, depth_background taking what is left; differentiable w.r.t. the cameras, the
scale and the points across splat edges.

1. Parity, tiled K (1, 2, 4, 8) and generic K (3, 5, 16, 64), square and non-square images (W % 4 != 0 included): idx equal to
   mvr_points_forward's and the C oracle's at the same K; depth within 1e-5, R / T / dist and point gradients within 1e-4 of fp64
   autograd of tests/splat_depth_ref.py on the kernels' fp32 projection (straight through).  The decision "c > 1" of a pixel whose
   sum lies within rounding of 1 is taken from the kernels' fp32 sum (mirrored on the host); the test counts the pixels where it
   differs from the fp64 one.  Bit-identical output for both compositors.
2. The kernels that run, and those that must not.
3. Determinism: camera and dist gradients bit-identical over two runs and with / without point gradients.
4. What hard depth cannot do: an in-plane offset of a cloud gets no gradient from hard_depth and the fp64 one from splat_depth.
5. Empty inputs: no points, and a view whose points are all behind the camera.
6. MVRenderer(pc_rendering=True, shader="splat_depth").
7. A seeded fit of a cloud offset to target depth maps with an unmasked loss.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, ops, synth

import splat_depth_ref
from test_gpu_branches import expect_launches, launches

pytestmark = pytest.mark.gpu

GRAD_RTOL = 1e-4           # R / T / dist gradients: max |error| over the tensor's largest entry (test_gpu_depth.py)
POINT_GRAD_RTOL = 1e-4     # point gradients (float atomics)
DEPTH_RTOL = 1e-5
BGD = 4.0                  # a background just behind the clouds (views at distance 2.2, clouds scaled by 1 / dist)
D = torch.float64


def rel(a, b):
    a, b = torch.as_tensor(a).detach().double().cpu(), torch.as_tensor(b).detach().double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-12))


def stopped_f32(idx, dists2, radius):
    """'this entry or an earlier one took c past 1' as the kernels decide it: alpha = 1 - d2 / r^2 and the running sum in fp32,
    r^2 the double radius * radius rounded to fp32."""
    r2 = np.float32(radius * radius)
    a = np.where(idx >= 0, (np.float32(1.0) - dists2.astype(np.float32) / r2).astype(np.float32), np.float32(0.0))
    c = np.zeros(a.shape[:-1], np.float32)
    stop = np.zeros(a.shape, bool)
    for k in range(a.shape[-1]):
        c = (c + a[..., k]).astype(np.float32)
        stop[..., k] = (stop[..., k - 1] if k else False) | ((c > np.float32(1.0)) & (idx[..., k] >= 0))
    return torch.from_numpy(stop)


class Scene:
    def __init__(self, oracle, B=3, Np=2048, M=4, H=64, W=64, K=4, radius=0.03, bg=BGD, seed=11):
        self.B, self.Np, self.M, self.H, self.W, self.K, self.rad, self.bg = B, Np, M, H, W, K, radius, bg
        self.pts = synth.make_clouds(B, Np, seed)
        self.views = synth.learned_spherical_views(B, M, seed + 1)
        az, el, di = (t.numpy().ravel().astype(np.float32) for t in self.views)
        self.R, self.T, _ = oracle.look_at(az, el, di)
        self.di = di
        self.s = (1.0 / di.astype(np.float64)).astype(np.float32)
        self.g = torch.randn(B * M, 1, H, W, generator=torch.Generator().manual_seed(seed + 2))

    def tensors(self, dev, point_grad=True):
        pg = self.pts.to(dev).requires_grad_(point_grad)
        Rg, Tg = (torch.from_numpy(x).to(dev).requires_grad_() for x in (self.R, self.T))
        dg = torch.from_numpy(self.di).to(dev).requires_grad_()
        return pg, Rg, Tg, dg

    def render(self, dev, t, compositor="norm", shader="splat_depth", fragments=False):
        pg, Rg, Tg, dg = t
        return ops.render_points(pg, torch.ones(3, device=dev), self.M, Rg, Tg, None, self.rad, torch.zeros(3, device=dev),
                                 (self.H, self.W), points_per_pixel=self.K, compositor=compositor, dist=dg, shader=shader,
                                 depth_background=self.bg, fragments=fragments)

    def reference(self, oracle, idx, dists2):
        """fp64 autograd of render_points_view_splat_depth on the given fragments, on the kernels' fp32 projection (the oracle's,
        straight through), the saturation decision from the fp32 sum -> depth (n,1,H,W), gR, gT, g dist, g points, (pixels whose
        decision was substituted, the largest |c - 1| of the fp64 sum there)."""
        Rr, Tr = (torch.from_numpy(x).to(D).requires_grad_() for x in (self.R, self.T))
        pr = self.pts.to(D).requires_grad_()
        dr = torch.from_numpy(self.di).to(D).requires_grad_()
        stop32 = stopped_f32(idx.numpy(), dists2, self.rad)
        loss, deps, subst, off1 = 0, [], 0, 0.0
        for n in range(self.B * self.M):
            b = n // self.M
            p64 = (pr[b] * (1.0 / dr[n])) @ Rr[n] + Tr[n]
            p32 = torch.from_numpy(oracle.project_orthographic(self.pts[b].numpy(), self.R[n], self.T[n], self.s[n])).to(D)
            ndc = p64 + (p32 - p64).detach()
            dep, frag = splat_depth_ref.render_points_view_splat_depth(None, None, None, None, self.rad, self.H, self.W, self.K,
                                                                      self.bg, idx=idx[n].long(), stopped=stop32[n], ndc=ndc)
            with torch.no_grad():
                valid = frag["idx"] >= 0
                c64 = frag["alpha"].cumsum(-1)
                stop64 = ((c64 > 1) & valid).cumsum(-1) > 0
                differ = (stop64 != stop32[n]) & valid
                if differ.any():
                    subst += int(differ.any(-1).sum())
                    off1 = max(off1, float((c64[differ] - 1).abs().max()))
            deps.append(dep.detach())
            loss = loss + (dep * self.g[n, 0].to(D)).sum()
        loss.backward()
        return torch.stack(deps)[:, None], Rr.grad, Tr.grad, dr.grad, pr.grad, (subst, off1)


# K, (H, W), radius, compositor: tiled K in {1, 2, 4, 8}, generic K otherwise
CASES = {
    "k1": (1, (64, 64), 0.03, "norm"),
    "k2_nonsquare": (2, (48, 80), 0.04, "alpha"),
    "k4_w66": (4, (72, 66), 0.02, "norm"),
    "k8": (8, (64, 64), 0.05, "alpha"),
    "k3": (3, (56, 56), 0.03, "norm"),
    "k5_w70": (5, (40, 70), 0.025, "alpha"),
    "k16": (16, (64, 64), 0.05, "norm"),
    "k64": (64, (32, 36), 0.05, "norm"),
}


# ------------------------------------------------------------------------------------------------- 1. parity, 2. launches, 3. determinism
@pytest.mark.parametrize("case", list(CASES))
def test_splat_depth_matches_the_torch_restatement(oracle, cuda_device, case):
    K, (H, W), rad, compositor = CASES[case]
    dev = cuda_device
    tiled = K in (1, 2, 4, 8)
    sc = Scene(oracle, H=H, W=W, K=K, radius=rad)
    t = sc.tensors(dev)
    fwd = {"points_splat_tile_kernel": 1 if tiled else 0, "points_splat_resolve_kernel": 0 if tiled else 1,
           "points_tile_kernel": 0, "points_resolve_kernel": 0}
    counts, out = {}, None
    for pfx in fwd:
        o, counts[pfx] = launches(pfx, lambda: sc.render(dev, t, compositor))
        out = out or o
    expect_launches(counts, fwd, f"[{case}] forward")
    depth, frag = out
    assert depth.shape == (sc.B * sc.M, 1, H, W) and depth.dtype == torch.float32
    idx = frag["idx"]
    assert idx.shape == (sc.B * sc.M, H, W, K)
    # the same bits whatever the compositor; idx is the colour path's and the oracle's at the same K
    other, ofrag = sc.render(dev, t, "alpha" if compositor == "norm" else "norm")
    assert torch.equal(other, depth) and torch.equal(ofrag["idx"], idx)
    _, cfrag = sc.render(dev, t, compositor, shader="composite", fragments=True)
    assert torch.equal(cfrag["idx"], idx)
    o = oracle.points_forward(sc.pts.numpy(), np.ones(3, np.float32), sc.M, sc.R, sc.T, sc.s, rad, np.zeros(3, np.float32), H, W, K, 0)
    assert int((idx.cpu().numpy() != o["idx"]).sum()) == 0
    covered = int((o["idx"][..., 0] >= 0).sum())
    assert covered > 500
    empty = torch.from_numpy(o["idx"][..., 0] < 0)
    assert bool((depth[:, 0].cpu()[empty] == sc.bg).all())
    g = sc.g.to(dev)
    back = {"points_splat_backward_kernel": 1, "points_backward_reduce_kernel": 1, "points_backward_kernel": 0,
            "points_depth_backward_kernel": 0}
    nb = {}
    for pfx in back:
        for x in t:
            x.grad = None
        _, nb[pfx] = launches(pfx, lambda: depth.backward(g, retain_graph=True))
    expect_launches(nb, back, f"[{case}] backward")
    gP, gR, gT, gd = (x.grad.clone() for x in t)
    # determinism: again, and without point gradients
    for point_grad in (True, False):
        t2 = sc.tensors(dev, point_grad)
        d2, _ = sc.render(dev, t2, compositor)
        d2.backward(g)
        assert torch.equal(t2[1].grad, gR) and torch.equal(t2[2].grad, gT) and torch.equal(t2[3].grad, gd), point_grad
    ref, gRr, gTr, gdr, gPr, subst = sc.reference(oracle, idx.cpu(), o["dists2"])
    e_d, e_R, e_T, e_s, e_P = rel(depth, ref), rel(gR, gRr), rel(gT, gTr), rel(gd, gdr), rel(gP, gPr)
    print(f"[{case}] depth {e_d:.1e}  R {e_R:.1e}  T {e_T:.1e}  dist {e_s:.1e}  points {e_P:.1e}  saturation decisions taken from "
          f"fp32: {subst[0]} of {covered} covered pixels (fp64 sum within {subst[1]:.1e} of 1 there)")
    assert e_d < DEPTH_RTOL, e_d
    assert e_R < GRAD_RTOL and e_T < GRAD_RTOL and e_s < GRAD_RTOL, (e_R, e_T, e_s)
    assert e_P < POINT_GRAD_RTOL, e_P
    assert subst[1] < 1e-5, subst
    # the in-plane columns of dR carry a gradient (hard depth leaves them 0)
    assert float(gR[:, :, :2].abs().max()) > 0.1 * float(gR.abs().max())


# ------------------------------------------------------------------------------------------------- 4. what hard depth cannot do
def test_splat_depth_moves_a_cloud_sideways_where_hard_depth_cannot(oracle, cuda_device):
    """One cloud, one view; the loss is the squared difference to the depth of the cloud 0.03 to the side along the view's x
    axis.  d loss / d t for an offset t along that axis: under hard_depth only fp32 rounding (its point gradient lies along the
    view's z axis), below 1e-5 of splat_depth's; splat_depth's equals fp64 autograd of the restatement."""
    dev = cuda_device
    sc = Scene(oracle, B=1, M=1, H=64, W=64, K=8, radius=0.03, seed=41)
    u = torch.from_numpy(sc.R[0][:, 0].copy())      # world direction of the view's x axis (X_view = X R + T)
    Rd, Td = (torch.from_numpy(x).to(dev) for x in (sc.R, sc.T))
    dd = torch.from_numpy(sc.di).to(dev)
    grads = {}
    for shader in ("hard_depth", "splat_depth"):
        def depth(shift):
            pts = sc.pts.to(dev) + shift * u.to(dev)
            return ops.render_points(pts, torch.ones(3, device=dev), 1, Rd, Td, None, sc.rad, torch.zeros(3, device=dev), 64,
                                     points_per_pixel=8, dist=dd, shader=shader, depth_background=sc.bg)
        with torch.no_grad():
            target, _ = depth(torch.tensor(0.0, device=dev))
        tt = torch.tensor(0.03, device=dev, requires_grad=True)
        dep, frag = depth(tt)
        loss = ((dep - target) ** 2).sum()
        loss.backward()
        grads[shader] = float(tt.grad)
        print(f"[{shader}] loss {float(loss.detach()):.4e}  d loss / d t {grads[shader]:.4e}")
        assert float(loss.detach()) > 0
    # fp64: the same cotangent through the restatement, on the splat render's fragments and the kernels' fp32 projection
    pts32 = (sc.pts.to(dev) + torch.tensor(0.03, device=dev) * u.to(dev)).cpu()      # the shifted cloud the kernels saw
    tr64 = torch.zeros((), dtype=D, requires_grad=True)
    g = (2 * (dep - target)).detach().cpu().to(D)
    idx = frag["idx"][0].cpu().long()
    o = oracle.points_forward(pts32.numpy(), np.ones(3, np.float32), 1, sc.R, sc.T, sc.s, sc.rad, np.zeros(3, np.float32), 64, 64, 8, 0)
    assert torch.equal(torch.from_numpy(o["idx"][0]).long(), idx)
    p32 = torch.from_numpy(oracle.project_orthographic(pts32[0].numpy(), sc.R[0], sc.T[0], sc.s[0])).to(D)
    p64 = ((pts32[0].to(D) + tr64 * u.to(D)) * (1.0 / float(sc.di[0]))) @ torch.from_numpy(sc.R[0]).to(D) + torch.from_numpy(sc.T[0]).to(D)
    ndc = p64 + (p32 - p64).detach()
    stop = stopped_f32(o["idx"][0], o["dists2"][0], sc.rad)
    dep64, _ = splat_depth_ref.render_points_view_splat_depth(None, None, None, None, sc.rad, 64, 64, 8, sc.bg, idx=idx, stopped=stop, ndc=ndc)
    (dep64 * g[0, 0]).sum().backward()
    want = float(tr64.grad)
    print(f"splat_depth d loss / d t {grads['splat_depth']:.6e}, fp64 {want:.6e}")
    assert abs(grads["splat_depth"] - want) < 1e-4 * abs(want)
    assert abs(grads["hard_depth"]) < 1e-5 * abs(grads["splat_depth"])


# ------------------------------------------------------------------------------------------------- 5. empty inputs
@pytest.mark.parametrize("K", [4, 5])
def test_splat_depth_empty_inputs(cuda_device, K):
    """No points at all, and views whose points are all behind the camera: exactly the background, idx all -1, zero gradients."""
    dev = cuda_device
    B, M, H, W = 2, 2, 40, 44
    for Np in (0, 512):
        pts = (synth.make_clouds(B, Np, 3) if Np else torch.zeros(B, 0, 3)).to(dev).requires_grad_()
        R = torch.eye(3, device=dev).repeat(B * M, 1, 1).requires_grad_()
        T = torch.tensor([[0.0, 0.0, -10.0]] * (B * M), device=dev, requires_grad=True)      # z = X_z / dist - 10 < 0: behind
        dd = torch.full((B * M,), 2.2, device=dev, requires_grad=True)
        dep, frag = ops.render_points(pts, torch.ones(3, device=dev), M, R, T, None, 0.05, torch.zeros(3, device=dev), (H, W),
                                      points_per_pixel=K, dist=dd, shader="splat_depth", depth_background=-3.5)
        assert torch.equal(dep, torch.full_like(dep, -3.5)), Np
        assert bool((frag["idx"] == -1).all())
        dep.backward(torch.randn_like(dep))
        for x in (pts, R, T, dd):
            assert torch.equal(x.grad, torch.zeros_like(x)), Np


# ------------------------------------------------------------------------------------------------- 6. MVRenderer
def test_mvrenderer_splat_depth(cuda_device):
    dev = cuda_device
    B, M, H, K, rad = 1, 12, 64, 4, 0.03
    pts = synth.make_clouds(B, 1024, 31).to(dev)
    views = tuple(t.to(dev) for t in synth.learned_spherical_views(B, M, 32))
    kw = dict(image_size=H, pc_rendering=True, shader="splat_depth", points_per_pixel=K, points_radius=rad, depth_background=BGD,
              object_color="custom")
    for cg in (None, True):      # a 12-view batch: cuda_graph=None would replay a colour step from a graph
        r = MVRenderer(M, cuda_graph=cg, **kw).eval()
        a, e, d = (t.clone().requires_grad_() for t in views)
        col = torch.tensor([0.3, 0.6, 0.9], device=dev, requires_grad=True)
        img, cams = r(None, pts, a, e, d, color=col)
        assert img.shape == (B, M, 1, H, H) and img.dtype == torch.float32 and not r._point_graphs
        assert type(cams).__name__ == "FoVOrthographicCameras"
        g = torch.randn(B, M, 1, H, H, generator=torch.Generator().manual_seed(33)).to(dev)
        (img * g).sum().backward()
        assert col.grad is None
        # the ops-level chain: look_at, render_points(dist=...), look_at backward plus the scale term of d dist
        Rk, Tk, _ = ops.look_at_view_transform(d.detach(), e.detach(), a.detach(), return_centers=True)
        Rk, Tk = Rk.detach().requires_grad_(), Tk.detach().requires_grad_()
        dk = d.detach().reshape(-1).clone().requires_grad_()
        dep, frag = ops.render_points(pts, torch.ones(3, device=dev), M, Rk, Tk, None, rad, torch.zeros(3, device=dev), H,
                                      points_per_pixel=K, dist=dk, shader="splat_depth", depth_background=BGD)
        assert torch.equal(dep.view(B, M, 1, H, H), img.detach())
        assert torch.equal(frag["idx"], r.last_fragments["idx"])
        dep.backward(g.reshape(B * M, 1, H, H))
        ga, ge, gd = ops._look_at_backward_launch(*(t.detach().reshape(-1).float() for t in (a, e, d)), Rk.grad, Tk.grad, None)
        gd = gd + dk.grad
        for got, want in ((a.grad, ga), (e.grad, ge), (d.grad, gd)):
            assert float(want.abs().max()) > 0
            assert torch.allclose(got.reshape(-1), want, rtol=1e-6, atol=1e-6 * float(want.abs().max())), rel(got.reshape(-1), want)
    # rejected options
    for bad in (dict(normalize=((0.5,) * 3, (0.2,) * 3)), dict(out_dtype=torch.bfloat16), dict(keep_alpha=True)):
        with pytest.raises(ValueError):
            MVRenderer(M, **kw, **bad)
    for bad in (dict(normalize=((0.5,) * 3, (0.2,) * 3)), dict(out_dtype=torch.bfloat16)):
        with pytest.raises(ValueError):
            ops.render_points(pts, torch.ones(3, device=dev), M, cams.R, cams.T, None, rad, torch.zeros(3, device=dev), H,
                              dist=views[2].reshape(-1), shader="splat_depth", **bad)
    rm = MVRenderer(M, image_size=H, pc_rendering=False, shader="splat_depth")
    with pytest.raises(ValueError):
        rm([synth.make_mesh(300, 1)], None, *views)
    with pytest.raises(ValueError, match="splat_depth"):
        ops.render_points(pts, torch.ones(3, device=dev), M, cams.R, cams.T, None, rad, torch.zeros(3, device=dev), H,
                          dist=views[2].reshape(-1), shader="soft_depth")


# ------------------------------------------------------------------------------------------------- 7. seeded fit
def test_splat_depth_fit_of_a_cloud_offset_unmasked(cuda_device):
    """Adam on one offset added to every point of a cloud, through MVRenderer(shader="splat_depth") with point gradients, against
    the depth maps of the cloud at the origin (4 views, r = 0.03, K = 8: most covered pixels saturate).  The start is offset by
    (0.25, -0.2, 0.15), where the silhouettes only partly overlap; the loss is the mean squared depth difference over EVERY pixel
    (no mask).  Loss below 20 % of its start, offset error below half of its start (DESIGN.md section 8 records the run)."""
    dev = cuda_device
    torch.manual_seed(0)
    M, H = 4, 64
    pts = synth.make_clouds(1, 2048, 17).to(dev)
    az = torch.tensor([[20.0, 110.0, 200.0, 290.0]], device=dev)
    el = torch.tensor([[15.0, -20.0, 30.0, 5.0]], device=dev)
    di = torch.full((1, M), 2.2, device=dev)
    r = MVRenderer(M, image_size=H, pc_rendering=True, shader="splat_depth", points_per_pixel=8, points_radius=0.03,
                   depth_background=BGD).eval()
    with torch.no_grad():
        target, _ = r(None, pts, az, el, di)
        idx = r.last_fragments["idx"]
    off = torch.tensor([0.25, -0.2, 0.15], device=dev, requires_grad=True)
    with torch.no_grad():
        start, _ = r(None, pts + off, az, el, di)
        a, b = start < BGD - 1e-3, target < BGD - 1e-3
        iou = float((a & b).sum() / (a | b).sum())
        covered = idx[..., 0] >= 0
    opt = torch.optim.Adam([off], lr=0.02)
    err0 = float(off.detach().norm())
    losses = []
    for _ in range(80):
        opt.zero_grad()
        dep, _ = r(None, pts + off, az, el, di)
        loss = ((dep - target) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    err = float(off.detach().norm())
    print(f"splat depth fit: coverage IoU at the start {iou:.2f} ({int(covered.sum())} covered target pixels); loss "
          f"{losses[0]:.3e} -> {losses[-1]:.3e}, offset error {err0:.3f} -> {err:.4f}")
    assert iou < 0.9
    assert all(np.isfinite(losses))
    assert losses[-1] < 0.2 * losses[0]
    assert err < 0.5 * err0
