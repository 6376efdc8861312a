"""shader="hard_depth" on the GPU: the depth of the nearest fragment (meshes and point clouds) and its gradients.

Forward: the depth is compared bit for bit with the C oracle's zbuf[..., 0] (pix_to_face / idx with 0 mismatches), background
pixels hold depth_background.  Backward: camera, vertex and point gradients against fp64 autograd of tests/depth_ref.py's
render_mesh_view_depth / render_points_view_depth (pinned to the oracle's rasterizer backwards by tests/test_depth_host.py).
Also: determinism of the camera gradients, the kernels that run (and those that must not), the rejected options, the eager path
of small point batches, and a seeded fit of the view angles to target depth maps.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, _lib as L, ops, synth

import depth_ref
from test_gpu_branches import expect_launches, launches

pytestmark = pytest.mark.gpu

K00, K11 = ops.fov_projection_scale()
GRAD_RTOL = 1e-4           # R / T / dist gradients: max |error| over the tensor's largest entry
VERT_GRAD_RTOL = 5e-4      # vertex gradients (float atomics)
POINT_GRAD_RTOL = 1e-4     # point gradients (float atomics)
BGD = 77.0                 # a depth_background other than the default
D = torch.float64
PHONG_SHADE = ("mesh_shade_kernel<false, 4, 4, false>", "mesh_shade_kernel<false, 4, 4, true>", "mesh_shade_kernel<true")


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-12))


def cams(oracle, views, dev):
    az, el, di = (t.numpy().ravel().astype(np.float32) for t in views)
    R, T, C = oracle.look_at(az, el, di)
    return R, T, C, tuple(torch.from_numpy(x).to(dev) for x in (R, T, C))


# name -> meshes [(faces, seed)], M, (H, W), perspective_correct, cull, views (None: learned spherical), near-plane clipping
MESH = {
    "ragged": dict(meshes=[(600, 3), (1500, 4), (300, 5)], M=4, HW=(64, 64)),
    "nopersp_cull": dict(meshes=[(900, 6), (400, 7)], M=3, HW=(56, 56), persp=False, cull=True),
    "nonsquare": dict(meshes=[(800, 8)], M=3, HW=(48, 80)),
    # test_gpu_mesh_branches.SOFT["near_plane"]: a camera 1.12 - 1.3 from the object, faces cross z = 0.5
    "near_plane": dict(meshes=[(900, 281)], M=3, HW=(48, 48), near=True,
                       views=(torch.tensor([[15.0, 140.0, -80.0]]), torch.tensor([[10.0, -35.0, 50.0]]), torch.tensor([[1.12, 1.2, 1.3]]))),
}


def oracle_mesh(oracle, meshes, M, R, T, C, H, W, flags, z_clip):
    """The C oracle's K = 1 hard rasterizer over the packed batch -> pix_to_face (N,H,W), zbuf (N,H,W)."""
    vs, fs = [v.numpy() for v, _ in meshes], [f.numpy() for _, f in meshes]
    voff = np.cumsum([0] + [v.shape[0] for v in vs]).astype(np.int32)
    foff = np.cumsum([0] + [f.shape[0] for f in fs]).astype(np.int32)
    V, F = np.concatenate(vs), np.concatenate(fs)
    nrm = oracle.packed_vertex_normals(V, F, voff, foff)
    o = oracle.mesh_forward(V, F, voff, foff, nrm, np.full((V.shape[0], 3), 0.5, np.float32), M, R, T, C,
                            np.ones((1, 3), np.float32), np.zeros(3, np.float32), K00, K11, z_clip, H, W, 1, flags)
    return o["pix_to_face"][..., 0], o["zbuf"][..., 0], o


def check_depth(depth, p2f, op2f, ozbuf, bg):
    """Bit-exact depth and 0 face-id mismatches against the oracle."""
    depth, p2f = depth.cpu(), p2f.cpu()
    assert int((p2f.numpy() != op2f).sum()) == 0, f"{int((p2f.numpy() != op2f).sum())} pix_to_face mismatches"
    want = torch.from_numpy(np.where(op2f >= 0, ozbuf, np.float32(bg)))
    assert torch.equal(depth, want), float((depth - want).abs().max())
    assert (op2f >= 0).sum() > 100


def mesh_grads_ref(oracle, meshes, M, R, T, p2f, g, H, W, persp, cull, z_clip):
    """fp64 autograd of render_mesh_view_depth over every (mesh, view) with the GPU's fragments -> gR, gT, per-mesh gV.  The
    projected vertices take the values of the fp32 IEEE projection the kernels use (the oracle's, straight through): the
    comparison measures the depth chain, not how a 1-ulp change of a small face's corner moves its 1/area-conditioned gradient."""
    from oracle import torch_ref as tr
    Rr, Tr = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T))
    vds = [v.to(D).requires_grad_() for v, _ in meshes]
    loss = 0
    for b, (v, f) in enumerate(meshes):
        for m in range(M):
            n = b * M + m
            ndc = tr.project_perspective(vds[b], Rr[n], Tr[n], K00, K11)
            ndc = ndc + (torch.from_numpy(oracle.project_perspective(v.numpy(), R[n], T[n], K00, K11)).to(D) - ndc).detach()
            if z_clip is None:
                dep, _ = depth_ref.render_mesh_view_depth(None, f, None, None, K00, K11, H, W, persp, cull, p2f=p2f[n].long(), background=BGD,
                                                   ndc=ndc)
            else:
                dep, rp2f = depth_ref.render_mesh_view_depth(None, f, None, None, K00, K11, H, W, persp, cull, z_clip=z_clip, background=BGD,
                                                      ndc=ndc)
                assert (rp2f == p2f[n].long()).all()
            loss = loss + (dep * g[n, 0].to(D) * (p2f[n] >= 0)).sum()
    loss.backward()
    return Rr.grad, Tr.grad, [v.grad for v in vds]


@pytest.mark.parametrize("name", list(MESH))
def test_mesh_depth_forward_and_gradients(oracle, cuda_device, name):
    c = MESH[name]
    dev = cuda_device
    meshes = [synth.make_mesh(nf, seed) for nf, seed in c["meshes"]]
    B, M, (H, W) = len(meshes), c["M"], c["HW"]
    persp, cull, near = c.get("persp", True), c.get("cull", False), c.get("near", False)
    views = c.get("views") or synth.learned_spherical_views(B, M, c["meshes"][0][1] + 1)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    vp = torch.cat([v for v, _ in meshes]).to(dev).requires_grad_()
    Rg, Tg, Cg = (t.clone().requires_grad_() for t in (Rd, Td, Cd))
    light, obj, bg = torch.ones(1, 3, device=dev), torch.ones(3, device=dev), torch.zeros(3, device=dev)

    def render(verts=vp, K=1):
        return ops.render_meshes(geom, M, Rg, Tg, Cg, light, obj, bg, (H, W), faces_per_pixel=K, cull_backfaces=cull,
                                 perspective_correct=persp, verts=verts, shader="hard_depth", depth_background=BGD)

    want = {"mesh_shade_kernel<false, 4, 4, false, true>": 1, "mesh_scatter_kernel": 1}
    for p in PHONG_SHADE:
        want[p] = 0
    if near:
        want["mesh_shade_clipped_kernel<false, true>"] = 1
    counts, out = {}, None
    for p in want:
        o, counts[p] = launches(p, render)
        out = out or o
    expect_launches(counts, want, f"[{name}] forward")
    depth, frag = out
    assert depth.shape == (B * M, 1, H, W) and depth.dtype == torch.float32
    p2f = frag["pix_to_face"][..., 0].cpu()
    assert (int(frag["counters"][L.CNT_STRADDLE]) > 0) == near
    z_clip = 0.5 if near else None
    flags = (oracle.PERSPECTIVE_CORRECT if persp else 0) | (oracle.CULL_BACKFACES if cull else 0)
    op2f, ozbuf, _ = oracle_mesh(oracle, meshes, M, R, T, C, H, W, flags, 0.5 if persp else -1.0)
    check_depth(depth[:, 0], p2f, op2f, ozbuf, BGD)
    # faces_per_pixel does not change the depth (it always rasterizes with K = 1)
    d4, _ = render(None, K=4)
    assert torch.equal(d4, depth)

    g = torch.randn(B * M, 1, H, W, generator=torch.Generator().manual_seed(5))
    back = {"mesh_depth_backward_kernel<true>": 1, "mesh_backward_finish_kernel": 1, "mesh_backward_kernel": 0}
    nb = {}
    for p in back:
        for t in (Rg, Tg, Cg, vp):
            t.grad = None
        d, _ = render()
        _, nb[p] = launches(p, lambda: d.backward(g.to(dev)))
    expect_launches(nb, back, f"[{name}] backward")
    gR1, gT1 = Rg.grad.clone(), Tg.grad.clone()
    assert torch.equal(Cg.grad, torch.zeros_like(Cg))
    # determinism: the camera gradients are fixed-order sums -- the same bits on every call and without vertex gradients
    for t in (Rg, Tg, Cg):
        t.grad = None
    d, _ = render(None)
    _, n0 = launches("mesh_depth_backward_kernel<false>", lambda: d.backward(g.to(dev)))
    assert n0 == 1
    assert torch.equal(Rg.grad, gR1) and torch.equal(Tg.grad, gT1)
    gRr, gTr, gVr = mesh_grads_ref(oracle, meshes, M, R, T, p2f, g, H, W, persp, cull, z_clip)
    assert rel(gR1, gRr) < GRAD_RTOL, rel(gR1, gRr)
    assert rel(gT1, gTr) < GRAD_RTOL, rel(gT1, gTr)
    gv = vp.grad.cpu()
    off = 0
    for b, (v, _) in enumerate(meshes):
        e = rel(gv[off: off + v.shape[0]], gVr[b])
        assert e < VERT_GRAD_RTOL, (b, e)
        assert float(gVr[b].abs().max()) > 0
        off += v.shape[0]


def test_mesh_depth_configs1_shape(oracle, cuda_device):
    """BASELINE configs[1] (32 meshes of ~10 k faces x 12 views, 224^2): the full batch on the GPU, the first two meshes' 24 views
    against the oracle (depth bit-exact, 0 face mismatches) and their gradients against fp64 autograd -- small faces (a few pixels
    each), where forming g z_i before differencing would show as the sliver error of mvr_mesh_bwd.cu."""
    dev = cuda_device
    B, M, H = 32, 12, 224
    meshes = synth.make_meshes(B, 10000, 0)
    views = synth.learned_spherical_views(B, M, 1)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    vp = torch.cat([v for v, _ in meshes]).to(dev).requires_grad_()
    Rg, Tg = Rd.clone().requires_grad_(), Td.clone().requires_grad_()
    depth, frag = ops.render_meshes(geom, M, Rg, Tg, Cd, torch.ones(1, 3, device=dev), torch.ones(3, device=dev),
                                    torch.zeros(3, device=dev), H, verts=vp, shader="hard_depth", depth_background=BGD)
    g = torch.randn(B * M, 1, H, H, generator=torch.Generator().manual_seed(3))
    depth.backward(g.to(dev))
    sub = meshes[:2]
    p2f = frag["pix_to_face"][: 2 * M, ..., 0].cpu()
    op2f, ozbuf, _ = oracle_mesh(oracle, sub, M, R[: 2 * M], T[: 2 * M], C[: 2 * M], H, H, oracle.PERSPECTIVE_CORRECT, 0.5)
    check_depth(depth[: 2 * M, 0], p2f, op2f, ozbuf, BGD)
    gRr, gTr, gVr = mesh_grads_ref(oracle, sub, M, R[: 2 * M], T[: 2 * M], p2f, g[: 2 * M], H, H, True, False, None)
    eR, eT = rel(Rg.grad[: 2 * M], gRr), rel(Tg.grad[: 2 * M], gTr)
    nv = sub[0][0].shape[0] + sub[1][0].shape[0]
    eV = rel(vp.grad[:nv], torch.cat(gVr))
    print(f"configs[1] depth gradients: R {eR:.2e} T {eT:.2e} verts {eV:.2e}")
    assert eR < GRAD_RTOL and eT < GRAD_RTOL and eV < VERT_GRAD_RTOL


def test_mesh_depth_mvrenderer_collated_and_angle_gradients(oracle, cuda_device):
    """uint16 collated batches and lists through MVRenderer(shader="hard_depth"): the oracle's depth; the angle gradients are
    look_at backward of the ops-level camera gradients; vertex tensors that require grad get theirs; colour gets none."""
    dev = cuda_device
    B, M, H = 3, 4, 64
    meshes = [synth.make_mesh(700 + 200 * b, 40 + b) for b in range(B)]
    az, el, di = synth.learned_spherical_views(B, M, 9)
    hp = ops.collate_meshes(meshes)
    assert hp.faces.dtype == torch.int16
    r = MVRenderer(M, image_size=H, pc_rendering=False, shader="hard_depth", depth_background=BGD, object_color="white",
                   light_direction="fixed", faces_per_pixel=3).eval()
    img, cameras = r(hp, None, az.to(dev), el.to(dev), di.to(dev))
    assert img.shape == (B, M, 1, H, H)
    R, T, C = (t.detach().cpu().numpy() for t in (cameras.R, cameras.T, cameras.get_camera_center()))      # the renderer's cameras
    op2f, ozbuf, _ = oracle_mesh(oracle, meshes, M, R, T, C, H, H, oracle.PERSPECTIVE_CORRECT, 0.5)
    check_depth(img.reshape(B * M, H, H), r.last_fragments["pix_to_face"][..., 0], op2f, ozbuf, BGD)
    # list input with vertex gradients and angles that require grad: the general path
    verts = [v.clone().to(dev).requires_grad_() for v, _ in meshes]
    faces = [f.to(dev) for _, f in meshes]
    a, e, d = (t.clone().to(dev).requires_grad_() for t in (az, el, di))
    col = torch.tensor([0.3, 0.6, 0.9], device=dev, requires_grad=True)
    r2 = MVRenderer(M, image_size=H, pc_rendering=False, shader="hard_depth", depth_background=BGD, object_color="custom",
                    light_direction="fixed").eval()
    img2, _ = r2(list(zip(verts, faces)), None, a, e, d, color=col)
    g = torch.randn(B, M, 1, H, H, generator=torch.Generator().manual_seed(2)).to(dev)
    (img2 * g).sum().backward()
    assert col.grad is None
    assert all(v.grad is not None and float(v.grad.abs().max()) > 0 for v in verts)
    # ops level with the same cameras
    Rk, Tk, Ck = ops.look_at_view_transform(d.detach(), e.detach(), a.detach(), return_centers=True)
    Rk, Tk = Rk.detach().requires_grad_(), Tk.detach().requires_grad_()
    geom = ops.PackedMeshes([v.detach() for v in verts], faces, dev)
    dep, _ = ops.render_meshes(geom, M, Rk, Tk, Ck, torch.ones(1, 3, device=dev), None, torch.zeros(3, device=dev), H,
                               shader="hard_depth", depth_background=BGD)
    assert torch.equal(dep.view(B, M, 1, H, H), img2.detach())
    dep.backward(g.reshape(B * M, 1, H, H))
    ga, ge, gd = ops._look_at_backward_launch(*(t.detach().reshape(-1).float() for t in (a, e, d)), Rk.grad, Tk.grad, None)
    for got, want in ((a.grad, ga), (e.grad, ge), (d.grad, gd)):
        assert torch.allclose(got.reshape(-1), want, rtol=1e-6, atol=1e-6 * float(want.abs().max())), rel(got.reshape(-1), want)


# ------------------------------------------------------------------------------------------------- points
def oracle_points(oracle, pts, M, R, T, s, rad, H, W):
    o = oracle.points_forward(pts.numpy(), np.ones(3, np.float32), M, R, T, s, rad, np.zeros(3, np.float32), H, W, 1, 0)
    return o["idx"][..., 0], o["zbuf"][..., 0]


@pytest.mark.parametrize("K,compositor", [(1, "norm"), (4, "alpha"), (5, "norm"), (5, "alpha")])
def test_points_depth_forward_and_gradients(oracle, cuda_device, K, compositor):
    dev = cuda_device
    B, Np, M, H, W, rad = 3, 2048, 4, 72, 64, 0.02
    pts = synth.make_clouds(B, Np, 11)
    az, el, di = synth.learned_spherical_views(B, M, 12)
    R, T, _, (Rd, Td, _) = cams(oracle, (az, el, di), dev)
    s = (1.0 / di.numpy().ravel().astype(np.float64)).astype(np.float32)
    pg = pts.to(dev).requires_grad_()
    Rg, Tg = Rd.clone().requires_grad_(), Td.clone().requires_grad_()
    dg = di.reshape(-1).to(dev).requires_grad_()

    def render():
        return ops.render_points(pg, torch.ones(3, device=dev), M, Rg, Tg, None, rad, torch.zeros(3, device=dev), (H, W),
                                 points_per_pixel=K, compositor=compositor, dist=dg, shader="hard_depth", depth_background=BGD)

    want = {"points_tile_kernel<1, 0, true>": 1, "points_tile_kernel<1, 0>": 0, "points_resolve_kernel": 0}
    counts, out = {}, None
    for p in want:
        o, counts[p] = launches(p, render)
        out = out or o
    expect_launches(counts, want, f"[K={K} {compositor}] forward")
    depth, frag = out
    assert depth.shape == (B * M, 1, H, W)
    oidx, oz = oracle_points(oracle, pts, M, R, T, s, rad, H, W)
    check_depth(depth[:, 0], frag["idx"][..., 0], oidx, oz, BGD)
    g = torch.randn(B * M, 1, H, W, generator=torch.Generator().manual_seed(4)).to(dev)
    back = {"points_depth_backward_kernel": 1, "points_backward_reduce_kernel": 1, "points_backward_kernel": 0}
    nb = {}
    for p in back:
        for t in (pg, Rg, Tg, dg):
            t.grad = None
        d, _ = render()
        _, nb[p] = launches(p, lambda: d.backward(g))
    expect_launches(nb, back, f"[K={K}] backward")
    gR1, gT1, gd1 = Rg.grad.clone(), Tg.grad.clone(), dg.grad.clone()
    for t in (Rg, Tg, dg):
        t.grad = None
    pg.requires_grad_(False)
    d, _ = render()
    d.backward(g)
    pg.requires_grad_(True)
    assert torch.equal(Rg.grad, gR1) and torch.equal(Tg.grad, gT1) and torch.equal(dg.grad, gd1)
    Rr, Tr = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T))
    pr = pts.to(D).requires_grad_()
    dr = di.reshape(-1).to(D).requires_grad_()
    idx = frag["idx"].cpu()
    loss = 0
    for n in range(B * M):
        dep, _ = depth_ref.render_points_view_depth(pr[n // M], Rr[n], Tr[n], 1.0 / dr[n], rad, H, W, background=BGD, idx=idx[n].long())
        loss = loss + (dep * g[n, 0].cpu().to(D)).sum()
    loss.backward()
    assert rel(gR1, Rr.grad) < GRAD_RTOL and rel(gT1, Tr.grad) < GRAD_RTOL and rel(gd1, dr.grad) < GRAD_RTOL
    assert rel(pg.grad, pr.grad) < POINT_GRAD_RTOL, rel(pg.grad, pr.grad)


def test_points_depth_mvrenderer_eager_and_options(oracle, cuda_device):
    """A small point batch (which cuda_graph=None would replay from a graph) runs eagerly with shader="hard_depth" and gives the
    ops-level depth; the options the depth cannot honour raise."""
    dev = cuda_device
    M, H = 12, 64
    pts = synth.make_clouds(1, 1024, 31).to(dev)
    az, el, di = (t.to(dev) for t in synth.circular_views(1, M))
    r = MVRenderer(M, image_size=H, pc_rendering=True, shader="hard_depth", depth_background=BGD, points_per_pixel=4,
                   cuda_graph=None).eval()
    img, cams_ = r(None, pts, az, el, di)
    assert img.shape == (1, M, 1, H, H) and not r._point_graphs
    ref, _ = ops.render_points(pts, torch.ones(3, device=dev), M, cams_.R, cams_.T, None, r.points_radius,
                               torch.zeros(3, device=dev), H, dist=di.reshape(-1), shader="hard_depth", depth_background=BGD)
    assert torch.equal(img.reshape(M, 1, H, H), ref)
    for kw in (dict(normalize=((0.5,) * 3, (0.2,) * 3)), dict(out_dtype=torch.bfloat16)):
        with pytest.raises(ValueError):
            ops.render_points(pts, torch.ones(3, device=dev), M, cams_.R, cams_.T, None, 0.02, torch.zeros(3, device=dev), H,
                              dist=di.reshape(-1), shader="hard_depth", **kw)
    geom = ops.PackedMeshes([synth.make_mesh(300, 1)[0]], [synth.make_mesh(300, 1)[1]], dev)
    for kw in (dict(normalize=((0.5,) * 3, (0.2,) * 3)), dict(out_dtype=torch.bfloat16), dict(blur_radius=1e-4)):
        with pytest.raises(ValueError):
            ops.render_meshes(geom, M, cams_.R, cams_.T, cams_.R[:, 0], torch.ones(1, 3, device=dev), torch.ones(3, device=dev),
                              torch.zeros(3, device=dev), H, shader="hard_depth", **kw)


def test_depth_fit_of_view_angles(cuda_device):
    """Seeded fit: Adam on (azim, elev) through MVRenderer(shader="hard_depth") against target depth maps of an asymmetric mesh,
    from angles perturbed by up to 15 degrees.  The loss (mean squared depth difference over the pixels covered in both maps)
    must fall below 20 % of its start and the angle error below half of its start (DESIGN.md section 8 records the run)."""
    dev = cuda_device
    torch.manual_seed(0)
    M, H = 4, 96
    v, f = synth.make_mesh(2000, 17, amplitude=0.35)
    mesh = [(v.to(dev), f.to(dev))]
    az_t = torch.tensor([[20.0, 110.0, 200.0, 290.0]], device=dev)
    el_t = torch.tensor([[15.0, -20.0, 30.0, 5.0]], device=dev)
    di = torch.full((1, M), 2.2, device=dev)
    r = MVRenderer(M, image_size=H, pc_rendering=False, shader="hard_depth", light_direction="fixed").eval()
    with torch.no_grad():
        target, _ = r(mesh, None, az_t, el_t, di)
    pert = torch.tensor([[12.0, -15.0, 9.0, -10.0]], device=dev), torch.tensor([[-8.0, 10.0, -12.0, 7.0]], device=dev)
    az = (az_t + pert[0]).requires_grad_()
    el = (el_t + pert[1]).requires_grad_()
    opt = torch.optim.Adam([az, el], lr=0.5)
    err0 = float(torch.cat([(az - az_t).abs(), (el - el_t).abs()]).mean().detach())
    losses = []
    for _ in range(80):
        opt.zero_grad()
        dep, _ = r(mesh, None, az, el, di)
        both = (dep < 50) & (target < 50)
        loss = ((dep - target) ** 2 * both).sum() / both.sum()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    err = float(torch.cat([(az - az_t).abs(), (el - el_t).abs()]).mean().detach())
    print(f"depth fit: loss {losses[0]:.3e} -> {losses[-1]:.3e}, mean angle error {err0:.2f} -> {err:.2f} deg")
    assert losses[-1] < 0.2 * losses[0]
    assert err < 0.5 * err0
