"""GPU tests of mesh backwards that return vertex and colour gradients together (run on the B200 box with `-m gpu`).

Fitting a textured mesh asks for d loss / d positions and d loss / d colours in one backward.  That runs instances of their own:
mesh_backward_kernel(_strip)<2, *, true, true> (two warp-aggregated scatters per pixel with per-vertex colours, the running
colour sum next to the vertex scatter with one object colour, interleaved atomics in the clipped-pixel pass) and
mesh_soft_backward_kernel<true, true>.  Each case proves with `launches` which instance ran.

1. Hard path, every case of test_gpu_color_grads.HARD x {object colour, per-vertex colours}: vertex and colour gradients against
   ONE fp64 autograd pass of oracle/torch_ref.py (normals from vertex_normals, so the normals chain is included) at the bars each
   feature meets alone; camera gradients bit-identical to the colour-free instance <2, *, true>.
2. SoftPhong, every case of test_gpu_color_grads.SOFT_PHONG: the same against render_mesh_view_soft; camera gradients
   bit-identical over the four (vertex, colour) gradient combinations.
3. With vertex gradients on, the object colour's gradient is still bit-reproducible.
4. render_meshes_from_angles with an object colour that requires grad (the two-call route of _MeshRenderFromAngles.backward).
5. MVRenderer with vertex tensors and a colour that require grad, and a seeded joint fit of shape and per-vertex colours.
6. The C ABI: mvr_mesh_soft_backward_rgb in SoftSilhouette mode returns a zero colour gradient and leaves the rest unchanged.
7. MVRenderer(cache_geometry=True) does not reuse the geometry of vertices that require grad.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import _lib as L
from mvtn_b200 import MVRenderer, Meshes, ops, synth
from test_gpu_branches import MESH_COL, VERT_GRAD_RTOL, launches, stream
from test_gpu_color_grads import HARD, RGB_GRAD_RTOL, SOFT_PHONG, WHITE, HardScene, _soft_render
from test_gpu_mesh_branches import SOFT
from test_gpu_parity import K00, K11, NORM, rel
from test_gpu_soft_vertex_grads import CASES, Scene

pytestmark = pytest.mark.gpu

# (HARD case's kernel, per-vertex colours) -> the instance that returns vertex and colour gradients
HARD_JOINT = {
    ("strip", False): "mesh_backward_kernel_strip<2, false, true, true>",
    ("strip", True): "mesh_backward_kernel_strip<2, true, true, true>",
    ("plain", False): "mesh_backward_kernel<2, false, true, true>",
    ("plain", True): "mesh_backward_kernel<2, true, true, true>",
}
SOFT_JOINT = "mesh_soft_backward_kernel<true, true>"
NORMALS_BWD = "geom_normals_bwd_face_kernel"
RGB_SUM = "mesh_rgb_grad_sum_kernel"


def _vertex_only(joint):
    """The instance with vertex gradients and no colour gradient: <2, *, true, true> -> <2, *, true>."""
    assert joint.endswith(", true>")
    return joint[: -len(", true>")] + ">"


def _count(prefixes, backward, reset):
    """One backward per prefix (the launch profiler counts one prefix at a time), each after `reset` has cleared the leaves'
    gradients -> {prefix: launches}.  The leaves keep the gradients of the last backward."""
    counts = {}
    for pfx in prefixes:
        reset()
        _, counts[pfx] = launches(pfx, backward)
    return counts


def _clear(*tensors):
    for t in tensors:
        t.grad = None


def _per_mesh_max(grad, voff):
    return [float(grad[int(voff[b]):int(voff[b + 1])].abs().max()) for b in range(len(voff) - 1)]


# ------------------------------------------------------------------------------------------------- 1. hard path
def _hard_reference(sc, p2f, per_vertex, g_img):
    """ONE fp64 autograd pass of torch_ref.render_mesh_view with positions and colours as leaves, on the CUDA fragments (near the
    plane: on the restatement's own clipping rasterizer, compared bit for bit) -> (d/d positions, d/d colour, clipped pixels)."""
    from oracle import torch_ref as tr
    d = torch.float64
    g_raw = g_img.float().cpu()
    if sc.bf16:
        g_raw = g_raw / torch.tensor(NORM[1]).view(1, 3, 1, 1)
    vd = sc.vp.to(d, copy=True).requires_grad_()
    leaf = (sc.vrgb if per_vertex else torch.tensor(MESH_COL)).to(d, copy=True).requires_grad_()
    bg = torch.tensor(MESH_COL, dtype=d) * 0.5
    loss, nclip = 0, 0
    for b, (_, f) in enumerate(sc.meshes):
        s = slice(int(sc.voff[b]), int(sc.voff[b + 1]))
        nrm = tr.vertex_normals(vd[s], f)
        rgb = leaf[s] if per_vertex else leaf.expand(sc.nv[b], 3)
        for m in range(sc.M):
            n = b * sc.M + m
            Rn, Tn, Cn = (torch.from_numpy(x[n]).to(d) for x in (sc.R, sc.T, sc.Cc))
            light = sc.light[n if sc.light.shape[0] > 1 else 0].to(d)
            args = (vd[s], f, nrm, rgb, Rn, Tn, Cn, light, bg, K00, K11, sc.H, sc.W)
            if sc.near:
                img, rp2f = tr.render_mesh_view(*args, perspective_correct=sc.persp, cull_backfaces=sc.cull, z_clip=0.5)
                assert torch.equal(rp2f.long(), p2f[n, :, :, 0].cpu().long()), "fragments differ from the reference rasterizer"
                with torch.no_grad():
                    fv = tr.project_perspective(vd[s], Rn, Tn, K00, K11)[f]
                strad = ((fv[:, :, 2] < 0.5).sum(1) % 3) != 0
                nclip += int((strad[rp2f.clamp_min(0)] & (rp2f >= 0)).sum())
            else:
                img, _ = tr.render_mesh_view(*args, perspective_correct=sc.persp, cull_backfaces=sc.cull,
                                             p2f=p2f[n, :, :, 0].cpu().long())
            loss = loss + (img * g_raw[n].to(d)).sum()
    loss.backward()
    return vd.grad, leaf.grad, nclip


def _hard_leaves(sc, dev, per_vertex, with_rgb):
    cam = tuple(t.detach().clone().requires_grad_() for t in (sc.Rd, sc.Td, sc.Cd))
    v = sc.vp.to(dev).requires_grad_()
    leaf = (sc.vrgb.to(dev) if per_vertex else torch.tensor(MESH_COL, device=dev)).requires_grad_(with_rgb)
    return cam, v, leaf


def _hard_render(sc, per_vertex, cam, v, leaf):
    return sc.render(per_vertex, obj=None if per_vertex else leaf, rgb=leaf if per_vertex else None, cameras=cam, verts=v)


@pytest.mark.parametrize("per_vertex", [False, True], ids=["object_rgb", "vertex_rgb"])
@pytest.mark.parametrize("case", list(HARD))
def test_hard_vertex_and_colour_gradients_together(oracle, cuda_device, case, per_vertex):
    """Vertices, colour and R / T / C all require grad: the <2, *, true, true> instance runs once, the normals backward once (and
    for one object colour the fixed-order colour sum once); d/d positions within VERT_GRAD_RTOL and d/d colour within
    RGB_GRAD_RTOL of fp64 autograd; camera gradients bit-identical to the same render whose colour does not require grad (the
    <2, *, true> instance); every mesh of the batch gets vertex (and per-vertex colour) gradients."""
    dev = cuda_device
    c = HARD[case]
    sc = HardScene(oracle, c, dev)
    joint = HARD_JOINT[(c["kernel"], per_vertex)]
    # the colour does not require grad: the vertex-only instance
    cam0, v0, _ = leaves0 = _hard_leaves(sc, dev, per_vertex, False)
    img0, _ = _hard_render(sc, per_vertex, *leaves0)
    g = sc.cotangent(img0)
    counts0 = _count([_vertex_only(joint), joint], lambda: img0.backward(g, retain_graph=True), lambda: _clear(*cam0, v0))
    assert counts0 == {_vertex_only(joint): 1, joint: 0}, counts0
    # everything requires grad
    cam, v, leaf = leaves = _hard_leaves(sc, dev, per_vertex, True)
    img, frag = _hard_render(sc, per_vertex, *leaves)
    assert torch.equal(img.detach(), img0.detach())
    want = {joint: 1, NORMALS_BWD: 1, **({} if per_vertex else {RGB_SUM: 1})}
    counts = _count(want, lambda: img.backward(g, retain_graph=True), lambda: _clear(*cam, v, leaf))
    assert counts == want, counts
    ref_v, ref_c, nclip = _hard_reference(sc, frag["pix_to_face"], per_vertex, g)
    err_v, err_c = rel(v.grad, ref_v.numpy()), rel(leaf.grad, ref_c.numpy())
    print(f"[{case} {'vertex' if per_vertex else 'object'}] {joint}  launches {counts}  vertex grad err {err_v:.1e} "
          f"(bar {VERT_GRAD_RTOL:.0e})  colour grad err {err_c:.1e} (bar {RGB_GRAD_RTOL:.0e})  clipped pixels {nclip}")
    assert torch.isfinite(v.grad).all() and torch.isfinite(leaf.grad).all()
    assert err_v < VERT_GRAD_RTOL, err_v
    assert err_c < RGB_GRAD_RTOL, err_c
    for name, a, b in zip(("gR", "gT", "gC"), (t.grad for t in cam0), (t.grad for t in cam)):
        assert torch.equal(a, b), (name, float((a - b).abs().max()))
    assert all(x > 0 for x in _per_mesh_max(v.grad, sc.voff)), _per_mesh_max(v.grad, sc.voff)
    if per_vertex:
        assert all(x > 0 for x in _per_mesh_max(leaf.grad, sc.voff)), _per_mesh_max(leaf.grad, sc.voff)
    if sc.near:
        assert nclip > 0


# ------------------------------------------------------------------------------------------------- 2. SoftPhong
def _soft_reference(oracle, sc):
    """ONE fp64 autograd pass of torch_ref.render_mesh_view_soft with positions and the case's colours as leaves, on the reference
    rasterizer's fragments -> (d/d positions, d/d colour, fragment indices (n,H,W,K))."""
    from oracle import torch_ref as tr
    c, H, W, K = sc.c, sc.H, sc.W, sc.K
    d = torch.float64
    per_vertex = sc.vrgb is not None
    vd = sc.vp.to(d, copy=True).requires_grad_()
    leaf = (sc.vrgb if per_vertex else sc.obj).to(d, copy=True).requires_grad_()
    loss, p2fs = 0, []
    for b, (_, f) in enumerate(sc.meshes):
        s = slice(int(sc.voff[b]), int(sc.voff[b + 1]))
        nrm = tr.vertex_normals(vd[s], f)
        rgb = leaf[s] if per_vertex else leaf.expand(sc.nv[b], 3)
        for m in range(sc.M):
            n = b * sc.M + m
            fv32 = torch.from_numpy(oracle.project_perspective(sc.vp[s].numpy(), sc.R[n], sc.T[n], K00, K11))[f]
            rp2f, _, _, _, rp2c = tr.rasterize_meshes_soft(fv32, H, W, K, c["blur"], sc.persp, sc.clip, sc.cull,
                                                           z_clip=sc.z_clip, return_sub=True)
            p2fs.append(rp2f)
            light = sc.light[n if sc.light.shape[0] > 1 else 0]
            ref, _ = tr.render_mesh_view_soft(vd[s], f, nrm, rgb, *(torch.from_numpy(x[n]).to(d) for x in (sc.R, sc.T, sc.Cc)),
                                              light.to(d), sc.bg.to(d), K00, K11, H, W, K, c["blur"], "soft_phong",
                                              sigma=c["sigma"], gamma=c["gamma"], perspective_correct=sc.persp, clip_bary=sc.clip,
                                              cull_backfaces=sc.cull, p2f=None if sc.near else rp2f, z_clip=sc.z_clip,
                                              p2c=rp2c if sc.near else None)
            loss = loss + (ref * sc.g[n].to(d)).sum()
    loss.backward()
    return vd.grad, leaf.grad, torch.stack(p2fs)


def _soft_leaves(sc, dev, gv, gc):
    cam = tuple(torch.from_numpy(x).to(dev).requires_grad_() for x in (sc.R, sc.T, sc.Cc))
    v = sc.vp.to(dev).requires_grad_() if gv else None
    leaf = (sc.vrgb if sc.vrgb is not None else sc.obj).to(dev).requires_grad_(gc)
    return cam, v, leaf


def _soft_render_leaves(sc, dev, cam, v, leaf):
    return _soft_render(sc, dev, obj=leaf, rgb=leaf if sc.vrgb is not None else None, cameras=cam, verts=v)


@pytest.mark.parametrize("case", SOFT_PHONG)
def test_soft_phong_vertex_and_colour_gradients_together(oracle, cuda_device, case):
    """SoftPhong with positions, the case's colours (object or per-vertex) and R / T / C requiring grad: <true, true> runs once
    and the normals backward once; d/d positions within VERT_GRAD_RTOL, d/d colour within max(1e-5, 5e-9 / gamma) of fp64
    autograd; the camera gradients are bit-identical over the four (vertex, colour) gradient combinations."""
    c, shader = CASES[case]
    assert shader == "soft_phong"
    dev = cuda_device
    sc = Scene(oracle, c, shader)
    g = sc.g.to(dev)
    cams = {}
    for gv in (False, True):
        for gc in (False, True):
            cam, v, leaf = _soft_leaves(sc, dev, gv, gc)
            img, frag = _soft_render_leaves(sc, dev, cam, v, leaf)
            if gv and gc:
                want = {SOFT_JOINT: 1, NORMALS_BWD: 1}
                counts = _count(want, lambda: img.backward(g, retain_graph=True), lambda: _clear(*cam, v, leaf))
                assert counts == want, counts
                got_v, got_c, p2f = v.grad, leaf.grad, frag["pix_to_face"]
            else:
                img.backward(g)
            cams[(gv, gc)] = [t.grad for t in cam]
    ref_v, ref_c, rp2f = _soft_reference(oracle, sc)
    assert torch.equal(p2f.cpu().long(), rp2f), "fragments differ from the reference rasterizer"
    bar_c = max(1e-5, 5e-9 / c["gamma"])
    err_v, err_c = rel(got_v, ref_v.numpy()), rel(got_c, ref_c.numpy())
    print(f"[{case} {'vertex' if sc.vrgb is not None else 'object'}] {SOFT_JOINT}  launches {counts}  vertex grad err {err_v:.1e} "
          f"(bar {VERT_GRAD_RTOL:.0e})  colour grad err {err_c:.1e} (bar {bar_c:.0e})")
    assert torch.isfinite(got_v).all() and torch.isfinite(got_c).all()
    assert float(got_c.abs().max()) > 0
    assert all(x > 0 for x in _per_mesh_max(got_v, sc.voff)), _per_mesh_max(got_v, sc.voff)
    assert err_v < VERT_GRAD_RTOL, err_v
    assert err_c < bar_c, err_c
    for key, grads in cams.items():
        for name, a, b in zip(("gR", "gT", "gC"), cams[(False, False)], grads):
            assert torch.equal(a, b), (key, name, float((a - b).abs().max()))


# ------------------------------------------------------------------------------------------------- 3. determinism
@pytest.mark.parametrize("case", ["hard-c1_mesh_224_strip", "hard-k2_w97_plain", "hard-near_plane_clipped", "soft-ragged-soft_phong"])
def test_object_colour_gradient_is_bit_reproducible_with_vertex_gradients(oracle, cuda_device, case):
    """Only the object colour goes through the fixed-order partial sums: with vertex gradients on, its gradient is the same in
    every bit over two backwards."""
    dev = cuda_device
    kind, name = case.split("-", 1)
    if kind == "hard":
        sc = HardScene(oracle, HARD[name], dev)
        _, v, leaf = leaves = _hard_leaves(sc, dev, False, True)
        img, _ = _hard_render(sc, False, *leaves)
        g, joint = sc.cotangent(img), HARD_JOINT[(HARD[name]["kernel"], False)]
    else:
        sc = Scene(oracle, *CASES[name])
        assert sc.vrgb is None
        _, v, leaf = leaves = _soft_leaves(sc, dev, True, True)
        img, _ = _soft_render_leaves(sc, dev, *leaves)
        g, joint = sc.g.to(dev), SOFT_JOINT
    grads = []
    for i in range(2):
        _clear(v, leaf)
        _, n = launches(joint, lambda: img.backward(g, retain_graph=True))
        assert n == 1, (joint, n)
        grads.append(leaf.grad.clone())
    assert float(grads[0].abs().max()) > 0
    assert torch.equal(grads[0], grads[1]), (grads[0], grads[1])


# ------------------------------------------------------------------------------------------------- 4. the angles node
@pytest.mark.parametrize("K,light", [(1, "relative"), (2, "fixed")])
def test_mesh_from_angles_object_colour_gradient(cuda_device, K, light):
    """render_meshes_from_angles with an object colour that requires grad takes the two-call route (mvr_mesh_backward_rgb, then
    the camera backward): its angle gradients are bit-identical to the fused route without a colour gradient, its colour gradient
    equals that of _LookAt + render_meshes, and a loss that also reads T and C leaves the colour gradient unchanged and gives the
    angle gradients of the two-node chain."""
    dev = cuda_device
    B, M, S = 3, 4, 64
    ms = synth.make_meshes(B, 700, 41)
    geom = ops.PackedMeshes([m[0] for m in ms], [m[1] for m in ms], dev)
    col = torch.tensor([0.9, 0.5, 0.3], device=dev); bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    lt = None if light == "relative" else torch.tensor([[0.0, 1.0, 0.2]], device=dev)
    views = [t.to(dev) for t in synth.learned_spherical_views(B, M, 13)]
    cot = torch.randn(B * M, 3, S, S, device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    gc_kernel = "mesh_backward_kernel_strip<3, false, false, true>" if K == 1 else "mesh_backward_kernel<3, false, false, true>"

    def angles():
        return tuple(t.clone().requires_grad_() for t in views)

    def from_angles(a, e, d, c):
        return ops.render_meshes_from_angles(geom, M, a, e, d, lt, c, bg, S, faces_per_pixel=K)

    def chain(a, e, d, c):
        R, T, C, _ = ops._LookAt.apply(a, e, d)
        img, _ = ops.render_meshes(geom, M, R, T, C, C.detach() if lt is None else lt, c, bg, S, faces_per_pixel=K)
        return img, T, C

    # fused route, no colour gradient
    a1 = angles()
    img1, _, _ = from_angles(*a1, col)
    img1.backward(cot)
    # two-call route: the colour requires grad
    a2, c2 = angles(), col.clone().requires_grad_()
    img2, _, _ = from_angles(*a2, c2)
    assert torch.equal(img1, img2)
    _, n = launches(gc_kernel, lambda: img2.backward(cot))
    assert n == 1, (gc_kernel, n)
    for name, x, y in zip("aed", a1, a2):
        assert torch.equal(x.grad, y.grad), name
    assert all(float(t.grad.abs().sum()) > 0 for t in a2) and float(c2.grad.abs().max()) > 0
    # the colour gradient of the two-node chain
    a3, c3 = angles(), col.clone().requires_grad_()
    img3, _, _ = chain(*a3, c3)
    img3.backward(cot)
    err = rel(c2.grad, c3.grad.cpu().numpy())
    assert err < 1e-5, err
    # a loss that also reads the cameras
    a4, c4 = angles(), col.clone().requires_grad_()
    img4, (_, T4, C4, _), _ = from_angles(*a4, c4)
    ((img4 * cot).sum() + T4.sum() + C4.sum()).backward()
    a5, c5 = angles(), col.clone().requires_grad_()
    img5, T5, C5 = chain(*a5, c5)
    ((img5 * cot).sum() + T5.sum() + C5.sum()).backward()
    assert torch.equal(c4.grad, c2.grad)
    for name, x, y in zip("aed", a4, a5):
        assert torch.allclose(x.grad, y.grad, rtol=1e-5, atol=1e-6), name
    print(f"[angles node K={K} {light} light] colour grad vs two-node chain {err:.1e}")


# ------------------------------------------------------------------------------------------------- 5. MVRenderer
def _ops_joint_grads(vals, faces, colour, shape, views, M, S, w, shader, K):
    """The same render through ops (_LookAt + render_meshes(verts=, rgb= / obj_rgb=)) -> gradients of the packed positions, of
    the colour in the caller's layout and of azim / elev / dist."""
    dev = w.device
    B, nv, nf = len(vals), [v.shape[0] for v in vals], [f.shape[0] for f in faces]
    a, e, d = (t.detach().clone().requires_grad_() for t in views)
    R, T, C, _ = ops._LookAt.apply(a, e, d)
    vg = torch.cat(vals).to(dev).requires_grad_()
    cl = colour.detach().clone().requires_grad_()
    obj = rgb = None
    if shape == "obj":
        obj = cl
    else:
        rgb = torch.cat([torch.broadcast_to(cl, (B, max(nv), 3))[b, :n] for b, n in enumerate(nv)])
    geom = ops.PackedMeshes.from_packed(vg.detach(), torch.cat(faces).to(dev), nv, nf, vert_rgb=None if rgb is None else rgb.detach())
    kw = dict(shader=shader, blur_radius=2e-3, sigma=1e-3, gamma=1e-2, faces_per_pixel=K) if shader != "hard_phong" else {}
    img, _ = ops.render_meshes(geom, M, R, T, C, torch.tensor([[0.0, 1.0, 0.0]], device=dev), obj, WHITE.to(dev), S, verts=vg,
                               rgb=rgb, **kw)
    (img.view(B, M, -1, S, S)[:, :, :3] * w).sum().backward()
    return vg.grad, cl.grad, (a.grad, e.grad, d.grad)


@pytest.mark.parametrize("shape", ["obj", "per_object", "per_vertex"])
@pytest.mark.parametrize("shader", ["hard_phong", "soft_phong"])
def test_mvrenderer_vertex_and_colour_gradients(cuda_device, shader, shape):
    """A list of Meshes whose vertex tensors require grad and a colour (3,), (B,1,3) or (B,maxV,3) that requires grad, two steps
    with an in-place update in between: vertex and colour gradients equal the ops-level ones (to the order of the atomics), the
    angle gradients equal those of the ops-level _LookAt + render_meshes chain in every bit."""
    dev = cuda_device
    M, S = 3, 48
    meshes = synth.make_meshes(2, 300, 111)
    B, nv = len(meshes), [v.shape[0] for v, _ in meshes]
    base = torch.tensor([0.3, 0.6, 0.9])
    if shape == "obj":
        color = base.clone()
    elif shape == "per_object":
        color = torch.stack([base, base.flip(0)])[:, None, :].clone()
    else:
        color = torch.rand(B, max(nv), 3, generator=torch.Generator().manual_seed(112))
    color = color.to(dev).requires_grad_()
    K = 1 if shader == "hard_phong" else 4
    r = MVRenderer(M, image_size=S, pc_rendering=False, object_color="custom", light_direction="fixed", shader=shader,
                   faces_per_pixel=K, blur_radius=0.0 if shader == "hard_phong" else 2e-3, blend_sigma=1e-3, blend_gamma=1e-2).to(dev)
    views = synth.learned_spherical_views(B, M, 113)
    w = torch.rand(B, M, 3, S, S, generator=torch.Generator().manual_seed(114)).to(dev)
    vs = [v.clone().requires_grad_() for v, _ in meshes]      # host tensors, as a data loader hands them over
    faces = [f for _, f in meshes]
    mesh_in = [Meshes([v], [f]) for v, f in zip(vs, faces)]
    gen = torch.Generator().manual_seed(115)
    for step in range(2):
        _clear(color, *vs)
        az, el, di = (t.to(dev).requires_grad_() for t in views)
        img, _ = r(mesh_in, None, az, el, di, color=color)
        (img[:, :, :3] * w).sum().backward()
        gv_ops, gc_ops, ga_ops = _ops_joint_grads([v.detach() for v in vs], faces, color, shape, (az, el, di), M, S, w, shader, K)
        gv = torch.cat([v.grad for v in vs])
        err_v, err_c = rel(gv, gv_ops.cpu().numpy()), rel(color.grad, gc_ops.cpu().numpy())
        print(f"[MVRenderer {shader} {shape} step {step}] vs ops level: vertex grads {err_v:.1e}  colour grad {err_c:.1e}")
        assert all(float(v.grad.abs().max()) > 0 for v in vs) and float(color.grad.abs().max()) > 0
        assert err_v < 1e-5, err_v
        assert err_c < 1e-5, err_c
        for name, x, y in zip("aed", (az, el, di), ga_ops):
            assert torch.equal(x.grad, y), name
        with torch.no_grad():      # an optimiser step: the same tensors, updated in place
            for v in vs:
                v.add_(0.02 * torch.randn(v.shape, generator=gen))
            color.mul_(0.9)


TARGET_SCALE = (1.08, 0.94, 1.0)


def textured_mesh_fit(dev, steps=80, sigma=1e-4, gamma=1e-4, K=8, lr_scale=1e-2, lr_rgb=0.05):
    """Adam on the three axis scales s of a unit sphere (the vertex offsets v0 (s - 1), whose gradient is the renderer's vertex
    gradient) and on its per-vertex colours, started at s = 1 and grey, against four SoftPhong views (64x64) of the sphere
    scaled by TARGET_SCALE with known random colours, rendered by MVRenderer -> (losses, fitted scales)."""
    v0, f = synth.uv_sphere(16, 32)
    v0, f = v0.to(dev), f.to(dev)
    r = MVRenderer(4, image_size=64, pc_rendering=False, object_color="custom", light_direction="fixed", shader="soft_phong",
                   faces_per_pixel=K, blur_radius=float(np.log(1.0 / 1e-4 - 1.0)) * sigma, blend_sigma=sigma, blend_gamma=gamma).to(dev)
    az = torch.tensor([[0.0, 90.0, 180.0, 270.0]], device=dev); el = torch.tensor([[20.0, -30.0, 40.0, -10.0]], device=dev)
    di = torch.full((1, 4), 2.5, device=dev)
    target_rgb = torch.rand(v0.shape[0], 3, generator=torch.Generator().manual_seed(121)).to(dev)
    with torch.no_grad():
        target, _ = r([Meshes([v0 * torch.tensor(TARGET_SCALE, device=dev)], [f])], None, az, el, di, color=target_rgb[None])
    scale = torch.ones(3, device=dev, requires_grad=True)
    rgb = torch.full_like(target_rgb, 0.5).requires_grad_()
    opt = torch.optim.Adam([{"params": [scale], "lr": lr_scale}, {"params": [rgb], "lr": lr_rgb}])
    losses = []
    for _ in range(steps):
        opt.zero_grad()
        img, _ = r([Meshes([v0 * scale], [f])], None, az, el, di, color=rgb[None])
        loss = ((img - target) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    return losses, scale.detach().cpu()


def test_textured_mesh_fit(cuda_device):
    """Shape and texture fitted together at a small size (textured_mesh_fit: 80 steps, K = 8, sigma = gamma = 1e-4): the loss
    falls at least tenfold and stays finite, and the fitted scales move towards the target's."""
    losses, scale = textured_mesh_fit(cuda_device)
    target = torch.tensor(TARGET_SCALE)
    err0, err1 = float((1.0 - target).abs().max()), float((scale - target).abs().max())
    print(f"[textured mesh fit] loss {losses[0]:.3e} -> {losses[-1]:.3e}  scales {scale.tolist()}  max |s - target| {err0:.3f} -> {err1:.3f}")
    assert all(np.isfinite(losses))
    assert losses[-1] <= 0.1 * losses[0], losses
    assert err1 < 0.5 * err0, (scale, TARGET_SCALE)


# ------------------------------------------------------------------------------------------------- 6. C ABI, silhouette
@pytest.mark.parametrize("layout", ["object_rgb", "vertex_rgb"])
def test_soft_silhouette_through_the_colour_entry_point(oracle, cuda_device, layout):
    """mvr_mesh_soft_backward_rgb with mode 1 (SoftSilhouette), with and without vertex gradients: the colour gradient is exactly
    zero (one object colour: written over a NaN-filled buffer; per-vertex colours: nothing accumulated), the camera gradients are
    bit-identical to mvr_mesh_soft_backward's and the vertex gradients equal them to the order of the float atomics."""
    dev = cuda_device
    c = SOFT["ragged" if layout == "object_rgb" else "vertex_rgb"]
    sc = Scene(oracle, c, "soft_silhouette")
    per_vertex = sc.vrgb is not None
    assert per_vertex == (layout == "vertex_rgb")
    geom = ops.PackedMeshes.from_packed(sc.vp.to(dev), torch.cat([f for _, f in sc.meshes]).to(dev), sc.nv, sc.nf,
                                        vert_rgb=sc.vrgb.to(dev) if per_vertex else None)
    Rd, Td, Cd = (torch.from_numpy(x).to(dev) for x in (sc.R, sc.T, sc.Cc))
    light, obj, bg = sc.light.to(dev), sc.obj.to(dev), sc.bg.to(dev)
    _, frag = ops.render_meshes(geom, sc.M, Rd, Td, Cd, light, None if per_vertex else obj, bg, (sc.H, sc.W), faces_per_pixel=sc.K,
                                shader="soft_silhouette", blur_radius=c["blur"], sigma=c["sigma"], gamma=c["gamma"])
    p2f, g = frag["pix_to_face"], sc.g.to(dev).contiguous()
    lib = L.load()
    B, M, N, Vt, Ft = sc.B, sc.M, sc.B * sc.M, geom.total_verts, geom.total_faces
    ws = ops.workspace(dev, lib.mvr_mesh_workspace_bytes(B, M, sc.H, sc.W, sc.K, Vt, Ft))
    flags = L.PERSPECTIVE_CORRECT | L.CLIP_BARYCENTRIC | (L.RGB_PER_ELEMENT if per_vertex else 0)
    light_stride = 0 if light.shape[0] == 1 else 3

    def call(with_rgb, want_verts):
        gR, gT, gC = torch.empty(N, 3, 3, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, 3, device=dev)
        gV = torch.zeros(Vt, 3, device=dev) if want_verts else None
        gRGB = torch.zeros(Vt, 3, device=dev) if per_vertex else torch.full((3,), float("nan"), device=dev)
        args = (geom.geometry.data_ptr(), geom.vert_off.data_ptr(), geom.face_off.data_ptr(), B, M, Vt, Ft, geom.max_verts,
                Rd.data_ptr(), Td.data_ptr(), Cd.data_ptr(), light.data_ptr(), light_stride, (bg if per_vertex else obj).data_ptr(),
                bg.data_ptr(), K00, K11, 0.5, c["blur"], sc.H, sc.W, sc.K, flags, 1, c["sigma"], c["gamma"], 1.0, 100.0,
                p2f.data_ptr(), g.data_ptr(), gR.data_ptr(), gT.data_ptr(), gC.data_ptr(), None if gV is None else gV.data_ptr(), None,
                ws.data_ptr(), ws.numel(), stream())
        if with_rgb:
            L.check(lib.mvr_mesh_soft_backward_rgb(*args, gRGB.data_ptr()), "mvr_mesh_soft_backward_rgb")
        else:
            L.check(lib.mvr_mesh_soft_backward(*args), "mvr_mesh_soft_backward")
        return (gR, gT, gC), gV, gRGB

    for want_verts in (False, True):
        cams0, gV0, _ = call(False, want_verts)
        kernel = "mesh_soft_backward_kernel<true, true>" if want_verts else "mesh_soft_backward_kernel<false, true>"
        (cams1, gV1, gRGB), n = launches(kernel, lambda: call(True, want_verts))
        assert n == 1, (kernel, n)
        assert torch.equal(gRGB, torch.zeros_like(gRGB)), gRGB
        for name, a, b in zip(("gR", "gT", "gC"), cams0, cams1):
            assert torch.equal(a, b), (name, want_verts, float((a - b).abs().max()))
        assert float(cams0[0].abs().max()) > 0
        if want_verts:
            err = rel(gV1, gV0.cpu().numpy())
            print(f"[silhouette through the colour entry, {layout}] vertex grads vs mvr_mesh_soft_backward {err:.1e}")
            assert float(gV0.abs().max()) > 0
            assert err < 1e-5, err


# ------------------------------------------------------------------------------------------------- 7. cache_geometry
def test_cache_geometry_is_not_used_for_vertices_that_require_grad(cuda_device):
    """MVRenderer(cache_geometry=True) in a fitting loop: the same list of Meshes, whose vertex leaves are updated in place
    between steps, renders the second step at the updated positions -- images and vertex gradients as cache_geometry=False on
    the updated vertices.  Re-rendering a list with nothing requiring grad still reuses the cached geometry (no packing kernel)."""
    dev = cuda_device
    M, S = 3, 48
    meshes = synth.make_meshes(2, 300, 131)
    faces = [f for _, f in meshes]
    az, el, di = (t.to(dev) for t in synth.learned_spherical_views(2, M, 132))
    w = torch.rand(2, M, 3, S, S, generator=torch.Generator().manual_seed(133)).to(dev)

    def renderer(cache):
        return MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed", cache_geometry=cache).to(dev)

    def step(r, mesh_in, vs):
        _clear(*vs)
        img, _ = r(mesh_in, None, az, el, di)
        (img * w).sum().backward()
        return img.detach(), torch.cat([v.grad for v in vs])

    r = renderer(True)
    vs = [v.clone().requires_grad_() for v, _ in meshes]
    mesh_in = [Meshes([v], [f]) for v, f in zip(vs, faces)]
    step(r, mesh_in, vs)
    with torch.no_grad():
        gen = torch.Generator().manual_seed(134)
        for v in vs:
            v.add_(0.05 * torch.randn(v.shape, generator=gen))
    img_c, gv_c = step(r, mesh_in, vs)
    fresh = [v.detach().clone().requires_grad_() for v in vs]
    img_u, gv_u = step(renderer(False), [Meshes([v], [f]) for v, f in zip(fresh, faces)], fresh)
    err = rel(gv_c, gv_u.cpu().numpy())
    print(f"[cache_geometry, vertices that require grad] second step: images equal {torch.equal(img_c, img_u)}  vertex grads {err:.1e}")
    assert torch.equal(img_c, img_u)
    assert err < 1e-5, err
    # nothing requires grad: the second render of the same list packs nothing
    plain = [Meshes([v], [f]) for (v, _), f in zip(meshes, faces)]
    with torch.no_grad():
        r(plain, None, az, el, di)
        _, n_hit = launches("geom_pack_verts_kernel", lambda: r(plain, None, az, el, di))
        _, n_new = launches("geom_pack_verts_kernel", lambda: r(list(plain), None, az, el, di))
    assert n_hit == 0, n_hit
    assert n_new >= 1, n_new
