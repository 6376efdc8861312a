"""GPU tests of the colour gradients of the mesh path (run on the B200 box with `-m gpu`).

render_meshes(obj_rgb=c) with c requiring grad, render_meshes(rgb=vertex_colours) and MVRenderer(color=...) with a colour that
requires grad: mesh_backward_kernel(_strip)<..., GC = true> / mesh_soft_backward_kernel<GV, true> return d loss / d colour --
per vertex with warp-aggregated (hard) or plain (soft) atomics, for one object colour through per-warp partials and a fixed-order
sum (bit-reproducible).

1. Hard path against fp64 autograd of oracle/torch_ref.py (render_mesh_view on the CUDA fragments, bit-exact first), one object
   colour and per-vertex colours, at 1e-5 of the tensor's largest entry: the gradient is linear in the cotangent with
   coefficients bb kd in [0, 0.8] and no 1/area term.  Every case proves with `launches` which instance it ran.
2. SoftPhong over every case of test_gpu_mesh_branches.SOFT and test_gpu_parity.SOFT_CASES that uses it, at the soft RGBA bar.
3. Camera gradients are bit-identical with and without colour gradients; vertex gradients agree within VERT_GRAD_RTOL; without a
   colour gradient only the existing instances run.
4. The object colour's gradient is bit-reproducible.
5. MVRenderer: colours (3,), (B,1,3), (B,maxV,3) that require grad, list and collated input, hard / soft_phong, cuda_graph and
   cache_geometry; soft_silhouette gives no colour gradient; the point path's (3,) colour at <= 48 and > 48 views.
6. A seeded texture fit: Adam on per-vertex colours against four views rendered with known colours.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, Meshes, ops, synth
from mvtn_b200.util import torch_color
from test_gpu_branches import MESH_COL, MESH_LIGHT, VERT_GRAD_RTOL, launches, ragged_meshes
from test_gpu_mesh_branches import SOFT_PARAMS
from test_gpu_parity import K00, K11, NORM, cams, rel
from test_gpu_soft_vertex_grads import CASES as SOFT_VERT_CASES, Scene

pytestmark = pytest.mark.gpu

RGB_GRAD_RTOL = 1e-5
WHITE = torch_color("white", max_lightness=True).detach().clone().float()      # MVRenderer's default background


# ------------------------------------------------------------------------------------------------- 1. hard path
HARD = {
    # name: meshes (faces, seed), M, (H, W), K, options, kernel suffix (strip / plain)
    "c1_mesh_224_strip": dict(meshes=[(10000, 301)], M=2, HW=(224, 224), K=1, kernel="strip"),
    "ragged_strip": dict(meshes="ragged", M=2, HW=(64, 64), K=1, kernel="strip"),
    "k2_w97_plain": dict(meshes=[(1200, 302)], M=2, HW=(97, 97), K=2, kernel="plain"),
    "bf16_normalised_plain": dict(meshes=[(800, 303), (300, 304)], M=2, HW=(64, 64), K=1, bf16=True, kernel="plain"),
    "noperspective_cull": dict(meshes=[(800, 305)], M=2, HW=(64, 64), K=1, persp=False, cull=True, kernel="strip"),
    "light_per_view": dict(meshes=[(600, 306), (900, 307)], M=2, HW=(64, 64), K=1, light="camera", kernel="strip"),
    "near_plane_clipped": dict(meshes=[(900, 308)], M=3, HW=(48, 48), K=1, near=True, kernel="strip",
                               views=(torch.tensor([[15.0, 140.0, -80.0]]), torch.tensor([[10.0, -35.0, 50.0]]),
                                      torch.tensor([[1.12, 1.2, 1.3]]))),
}


def _kernel(c, per_vertex):
    if c["kernel"] == "strip":
        return f"mesh_backward_kernel_strip<{2 if per_vertex else 3}, {str(per_vertex).lower()}, false, true>"
    return f"mesh_backward_kernel<{2 if per_vertex else 3}, {str(per_vertex).lower()}, false, true>"


class HardScene:
    def __init__(self, oracle, c, dev):
        self.c, self.dev = c, dev
        self.meshes = ragged_meshes() if c["meshes"] == "ragged" else [synth.make_mesh(nf, s) for nf, s in c["meshes"]]
        self.B, self.M, (self.H, self.W), self.K = len(self.meshes), c["M"], c["HW"], c["K"]
        self.persp, self.cull, self.bf16, self.near = c.get("persp", True), c.get("cull", False), c.get("bf16", False), c.get("near", False)
        self.views = c.get("views") or synth.learned_spherical_views(self.B, self.M, 5)
        self.R, self.T, self.Cc, (self.Rd, self.Td, self.Cd) = cams(oracle, self.views, dev)
        self.nv = [v.shape[0] for v, _ in self.meshes]
        self.voff = np.cumsum([0] + self.nv)
        self.vp = torch.cat([v for v, _ in self.meshes])
        self.vrgb = torch.rand(int(self.voff[-1]), 3, generator=torch.Generator().manual_seed(9))
        self.light = torch.from_numpy(self.Cc.copy()) if c.get("light") == "camera" else torch.tensor(MESH_LIGHT)
        self.g = torch.randn(self.B * self.M, 3, self.H, self.W, generator=torch.Generator().manual_seed(4))

    def geom(self, per_vertex):
        return ops.PackedMeshes([v for v, _ in self.meshes], [f for _, f in self.meshes], self.dev,
                                vert_rgb=self.vrgb if per_vertex else None)

    def render(self, per_vertex, obj=None, rgb=None, cameras=None, verts=None, geom=None):
        dev = self.dev
        R, T, C = cameras or (self.Rd, self.Td, self.Cd)
        obj = obj if obj is not None else (None if per_vertex else torch.tensor(MESH_COL, device=dev))
        return ops.render_meshes(geom or self.geom(per_vertex), self.M, R, T, C, self.light.to(dev), obj,
                                 torch.tensor(MESH_COL, device=dev) * 0.5, (self.H, self.W), faces_per_pixel=self.K,
                                 perspective_correct=self.persp, cull_backfaces=self.cull, normalize=NORM if self.bf16 else None,
                                 out_dtype=torch.bfloat16 if self.bf16 else None, rgb=rgb, verts=verts)

    def cotangent(self, img):
        return self.g.to(self.dev).to(img.dtype)

    def reference(self, p2f, per_vertex, g_img):
        """fp64 autograd of torch_ref.render_mesh_view on the CUDA fragments (or, near the plane, on the restatement's own
        clipping rasterizer, compared bit for bit) -> (d loss / d colour, clipped pixel count)."""
        from oracle import torch_ref as tr
        d = torch.float64
        g_raw = g_img.float().cpu()
        if self.bf16:
            g_raw = g_raw / torch.tensor(NORM[1]).view(1, 3, 1, 1)
        leaf = (self.vrgb if per_vertex else torch.tensor(MESH_COL)).to(d).requires_grad_()
        loss, nclip = 0, 0
        for b, (_, f) in enumerate(self.meshes):
            s = slice(int(self.voff[b]), int(self.voff[b + 1]))
            vd = self.vp[s].to(d)
            nrm = tr.vertex_normals(vd, f)
            rgb = leaf[s] if per_vertex else leaf.expand(self.nv[b], 3)
            for m in range(self.M):
                n = b * self.M + m
                light = self.light[n if self.light.shape[0] > 1 else 0].to(d)
                args = (vd, f, nrm, rgb, *(torch.from_numpy(x[n]).to(d) for x in (self.R, self.T, self.Cc)), light,
                        torch.tensor(MESH_COL, dtype=d) * 0.5, K00, K11, self.H, self.W)
                if self.near:
                    img, rp2f = tr.render_mesh_view(*args, perspective_correct=self.persp, cull_backfaces=self.cull, z_clip=0.5)
                    assert torch.equal(rp2f.long(), p2f[n, :, :, 0].cpu().long()), "fragments differ from the reference rasterizer"
                    fv = tr.project_perspective(vd, *(torch.from_numpy(x[n]).to(d) for x in (self.R, self.T)), K00, K11)[f]
                    strad = ((fv[:, :, 2] < 0.5).sum(1) % 3) != 0
                    nclip += int((strad[rp2f.clamp_min(0)] & (rp2f >= 0)).sum())
                else:
                    img, _ = tr.render_mesh_view(*args, perspective_correct=self.persp, cull_backfaces=self.cull,
                                                 p2f=p2f[n, :, :, 0].cpu().long())
                loss = loss + (img * g_raw[n].to(d)).sum()
        loss.backward()
        return leaf.grad, nclip


@pytest.mark.parametrize("per_vertex", [False, True], ids=["object_rgb", "vertex_rgb"])
@pytest.mark.parametrize("case", list(HARD))
def test_hard_colour_gradients_match_the_torch_restatement(oracle, cuda_device, case, per_vertex):
    """d loss / d colour of the hard Phong path against fp64 autograd of the restatement, within 1e-5 of the largest entry;
    the intended GC instance runs once; the near-plane case has clipped pixels (backward_clipped_view's share)."""
    dev = cuda_device
    c = HARD[case]
    sc = HardScene(oracle, c, dev)
    if per_vertex:
        leaf = sc.vrgb.to(dev).requires_grad_()
        img, frag = sc.render(True, rgb=leaf)
    else:
        leaf = torch.tensor(MESH_COL, device=dev, requires_grad=True)
        img, frag = sc.render(False, obj=leaf)
    g = sc.cotangent(img)
    kernel = _kernel(c, per_vertex)
    _, n = launches(kernel, lambda: img.backward(g))
    assert n == 1, (kernel, n)
    ref, nclip = sc.reference(frag["pix_to_face"], per_vertex, g)
    err = rel(leaf.grad, ref.numpy())
    print(f"[{case} {'vertex' if per_vertex else 'object'}] colour grad err {err:.1e} (bar {RGB_GRAD_RTOL:.0e})  {kernel}  "
          f"max {float(leaf.grad.abs().max()):.3e}  clipped pixels {nclip}")
    assert torch.isfinite(leaf.grad).all()
    assert err < RGB_GRAD_RTOL, err
    if per_vertex:      # every mesh of the batch receives colour gradients
        assert all(float(leaf.grad[int(sc.voff[b]):int(sc.voff[b + 1])].abs().max()) > 0 for b in range(sc.B))
    if sc.near:
        assert nclip > 0


# ------------------------------------------------------------------------------------------------- 2. SoftPhong
SOFT_PHONG = [k for k, (c, s) in SOFT_VERT_CASES.items() if s == "soft_phong"]


def _soft_reference(oracle, sc, leaf_cpu, per_vertex):
    from oracle import torch_ref as tr
    c, H, W, K = sc.c, sc.H, sc.W, sc.K
    d = torch.float64
    loss, p2fs = 0, []
    for b, (_, f) in enumerate(sc.meshes):
        s = slice(int(sc.voff[b]), int(sc.voff[b + 1]))
        vd = sc.vp[s].to(d)
        nrm = tr.vertex_normals(vd, f)
        rgb = leaf_cpu[s] if per_vertex else leaf_cpu.expand(sc.nv[b], 3)
        for m in range(sc.M):
            n = b * sc.M + m
            fv32 = torch.from_numpy(oracle.project_perspective(sc.vp[s].numpy(), sc.R[n], sc.T[n], K00, K11))[f]
            rp2f, _, _, _, rp2c = tr.rasterize_meshes_soft(fv32, H, W, K, c["blur"], sc.persp, sc.clip, sc.cull,
                                                           z_clip=sc.z_clip, return_sub=True)
            p2fs.append(rp2f)
            light = sc.light[n if sc.light.shape[0] > 1 else 0]
            ref, _ = tr.render_mesh_view_soft(vd, f, nrm, rgb, *(torch.from_numpy(x[n]).to(d) for x in (sc.R, sc.T, sc.Cc)),
                                              light.to(d), sc.bg.to(d), K00, K11, H, W, K, c["blur"], "soft_phong",
                                              sigma=c["sigma"], gamma=c["gamma"], perspective_correct=sc.persp, clip_bary=sc.clip,
                                              cull_backfaces=sc.cull, p2f=None if sc.near else rp2f, z_clip=sc.z_clip,
                                              p2c=rp2c if sc.near else None)
            loss = loss + (ref * sc.g[n].to(d)).sum()
    loss.backward()
    return torch.stack(p2fs)


def _soft_render(sc, dev, obj=None, rgb=None, cameras=None, verts=None):
    c = sc.c
    geom = ops.PackedMeshes.from_packed(sc.vp.to(dev), torch.cat([f for _, f in sc.meshes]).to(dev), sc.nv, sc.nf,
                                        vert_rgb=None if sc.vrgb is None else sc.vrgb.to(dev))
    Rd, Td, Cd = cameras or (torch.from_numpy(x).to(dev) for x in (sc.R, sc.T, sc.Cc))
    return ops.render_meshes(geom, sc.M, Rd, Td, Cd, sc.light.to(dev), obj if sc.vrgb is None else None, sc.bg.to(dev),
                             (sc.H, sc.W), faces_per_pixel=sc.K, shader=sc.shader, blur_radius=c["blur"], sigma=c["sigma"],
                             gamma=c["gamma"], perspective_correct=sc.persp, cull_backfaces=sc.cull,
                             clip_barycentric_coords=sc.clip, rgb=rgb, verts=verts)


@pytest.mark.parametrize("case", SOFT_PHONG)
def test_soft_phong_colour_gradients_match_the_torch_restatement(oracle, cuda_device, case):
    """SoftPhong's colour gradient (object colour, or per-vertex colours where the case has them) against fp64 autograd of
    render_mesh_view_soft, within max(1e-5, 5e-9 / gamma) of the largest entry; mesh_soft_backward_kernel<false, true> runs."""
    c, shader = SOFT_VERT_CASES[case]
    dev = cuda_device
    sc = Scene(oracle, c, shader)
    per_vertex = sc.vrgb is not None
    if per_vertex:
        leaf = sc.vrgb.to(dev).requires_grad_()
        img, frag = _soft_render(sc, dev, rgb=leaf)
    else:
        leaf = sc.obj.to(dev).requires_grad_()
        img, frag = _soft_render(sc, dev, obj=leaf)
    _, n = launches("mesh_soft_backward_kernel<false, true>", lambda: img.backward(sc.g.to(dev)))
    assert n == 1, n
    leaf_cpu = (sc.vrgb if per_vertex else sc.obj).to(torch.float64).requires_grad_()
    rp2f = _soft_reference(oracle, sc, leaf_cpu, per_vertex)
    assert torch.equal(frag["pix_to_face"].cpu().long(), rp2f), "fragments differ from the reference rasterizer"
    bar = max(1e-5, 5e-9 / c["gamma"])
    err = rel(leaf.grad, leaf_cpu.grad.numpy())
    print(f"[{case}] soft colour grad err {err:.1e} (bar {bar:.0e})  max {float(leaf.grad.abs().max()):.3e}")
    assert torch.isfinite(leaf.grad).all()
    assert float(leaf.grad.abs().max()) > 0
    assert err < bar, err


# ------------------------------------------------------------------------------------------------- 3. independence
@pytest.mark.parametrize("per_vertex", [False, True], ids=["object_rgb", "vertex_rgb"])
@pytest.mark.parametrize("case", ["ragged_strip", "k2_w97_plain", "near_plane_clipped"])
def test_camera_and_vertex_gradients_do_not_depend_on_colour_gradients(oracle, cuda_device, case, per_vertex):
    """(gR, gT, gC) are bit-identical with and without a colour gradient, the vertex gradients agree within VERT_GRAD_RTOL
    when both are requested, and without a colour gradient no GC instance runs."""
    dev = cuda_device
    c = HARD[case]
    sc = HardScene(oracle, c, dev)
    out = {}
    for with_rgb in (False, True):
        cam = tuple(t.detach().clone().requires_grad_() for t in (sc.Rd, sc.Td, sc.Cd))
        leaf = (sc.vrgb.to(dev) if per_vertex else torch.tensor(MESH_COL, device=dev)).requires_grad_(with_rgb)
        img, _ = sc.render(per_vertex, obj=None if per_vertex else leaf, rgb=leaf if per_vertex else None, cameras=cam)
        g = sc.cotangent(img)
        if not with_rgb:
            gc = _kernel(c, per_vertex)
            existing = f"{gc.split('<')[0]}<3, {str(per_vertex).lower()}, false>"      # the camera-only instance
            counts = {}
            for pfx in (existing, gc):
                for t in cam:
                    t.grad = None
                _, counts[pfx] = launches(pfx, lambda: img.backward(g, retain_graph=True))
            assert counts == {existing: 1, gc: 0}, counts
        else:
            img.backward(g)
            assert leaf.grad is not None
        out[with_rgb] = [t.grad for t in cam]
    for name, a, b in zip(("gR", "gT", "gC"), out[False], out[True]):
        assert torch.equal(a, b), (name, float((a - b).abs().max()))
    # vertex gradients with and without the colour gradient
    gv = {}
    for with_rgb in (False, True):
        v = sc.vp.to(dev).requires_grad_()
        leaf = (sc.vrgb.to(dev) if per_vertex else torch.tensor(MESH_COL, device=dev)).requires_grad_(with_rgb)
        geom = ops.PackedMeshes.from_packed(v.detach(), torch.cat([f for _, f in sc.meshes]).to(dev), sc.nv,
                                            [f.shape[0] for _, f in sc.meshes], vert_rgb=sc.vrgb.to(dev) if per_vertex else None)
        img, _ = sc.render(per_vertex, obj=None if per_vertex else leaf, rgb=leaf if per_vertex else None, verts=v, geom=geom)
        img.backward(sc.cotangent(img))
        gv[with_rgb] = v.grad
    err = rel(gv[True], gv[False].cpu().numpy())
    print(f"[{case}] vertex grads with / without colour gradient: {err:.1e}")
    assert err < VERT_GRAD_RTOL, err


@pytest.mark.parametrize("case", ["phong_default_blend", "vertex_rgb-soft_phong"])
def test_soft_camera_gradients_do_not_depend_on_colour_gradients(oracle, cuda_device, case):
    c, shader = SOFT_VERT_CASES[case if case in SOFT_VERT_CASES else f"parity_{case}"]
    dev = cuda_device
    sc = Scene(oracle, c, shader)
    out = {}
    for with_rgb in (False, True):
        cam = tuple(torch.from_numpy(x).to(dev).requires_grad_() for x in (sc.R, sc.T, sc.Cc))
        leaf = (sc.vrgb if sc.vrgb is not None else sc.obj).to(dev).requires_grad_(with_rgb)
        img, _ = _soft_render(sc, dev, obj=leaf, rgb=leaf if sc.vrgb is not None else None, cameras=cam)
        img.backward(sc.g.to(dev))
        out[with_rgb] = [t.grad for t in cam]
    for name, a, b in zip(("gR", "gT", "gC"), out[False], out[True]):
        assert torch.equal(a, b), (name, float((a - b).abs().max()))


# ------------------------------------------------------------------------------------------------- 4. determinism
@pytest.mark.parametrize("case", ["c1_mesh_224_strip", "k2_w97_plain", "near_plane_clipped"])
def test_object_colour_gradient_is_bit_reproducible(oracle, cuda_device, case):
    dev = cuda_device
    sc = HardScene(oracle, HARD[case], dev)
    leaf = torch.tensor(MESH_COL, device=dev, requires_grad=True)
    img, _ = sc.render(False, obj=leaf)
    g = sc.cotangent(img)
    grads = []
    for _ in range(2):
        leaf.grad = None
        img.backward(g, retain_graph=True)
        grads.append(leaf.grad.clone())
    assert torch.equal(grads[0], grads[1]), (grads[0], grads[1])


# ------------------------------------------------------------------------------------------------- 5. MVRenderer
def _ops_colour_grads(meshes, az, el, di, M, S, w, shader, per_vertex_rgb, K=1):
    """The same render through ops (look_at + render_meshes) -> d loss / d per-vertex colours (Vtot,3)."""
    dev = az.device
    R, T, C, _ = ops._LookAt.apply(*(t.detach() for t in (az, el, di)))
    vs = [v for v, _ in meshes]
    leaf = per_vertex_rgb.detach().to(dev).requires_grad_()
    geom = ops.PackedMeshes.from_packed(torch.cat(vs).to(dev), torch.cat([f for _, f in meshes]).to(dev), [v.shape[0] for v in vs],
                                        [f.shape[0] for _, f in meshes], vert_rgb=leaf.detach())
    kw = dict(shader=shader, blur_radius=2e-3, sigma=1e-3, gamma=1e-2, faces_per_pixel=K) if shader != "hard_phong" else {}
    img, _ = ops.render_meshes(geom, M, R, T, C, torch.tensor([[0.0, 1.0, 0.0]], device=dev), None, WHITE.to(dev), S, rgb=leaf, **kw)
    (img.view(len(meshes), M, -1, S, S)[:, :, :3] * w).sum().backward()
    return leaf.grad


@pytest.mark.parametrize("shape", ["obj", "per_object", "per_vertex"])
@pytest.mark.parametrize("mode", ["list_hard", "list_soft_phong", "collated_hard", "collated_cuda_graph", "list_cache_geometry"])
def test_mvrenderer_colour_gradients(cuda_device, mode, shape):
    """MVRenderer(object_color="custom") with a colour of shape (3,), (B,1,3) or (B,maxV,3) that requires grad: the colour's
    gradient equals the ops-level one (atomics order aside) and azim / elev / dist still receive theirs."""
    dev = cuda_device
    M, S = 3, 48
    meshes = synth.make_meshes(2, 300, 61)
    B, nv = len(meshes), [v.shape[0] for v, _ in meshes]
    maxV = max(nv)
    base = torch.tensor([0.3, 0.6, 0.9])
    if shape == "obj":
        color = base.clone()
    elif shape == "per_object":
        color = torch.stack([base, base.flip(0)])[:, None, :].clone()
    else:
        color = torch.rand(B, maxV, 3, generator=torch.Generator().manual_seed(62))
    color = color.to(dev).requires_grad_()
    shader = "soft_phong" if "soft" in mode else "hard_phong"
    K = 4 if shader != "hard_phong" else 1
    r = MVRenderer(M, image_size=S, pc_rendering=False, object_color="custom", light_direction="fixed", shader=shader,
                   faces_per_pixel=K, blur_radius=2e-3 if shader != "hard_phong" else 0.0, blend_sigma=1e-3, blend_gamma=1e-2,
                   cuda_graph=True if "cuda_graph" in mode else None, cache_geometry="cache" in mode).to(dev)
    views = synth.learned_spherical_views(B, M, 63)
    w = torch.rand(B, M, 3, S, S, generator=torch.Generator().manual_seed(64)).to(dev)
    steps = 2 if ("cache" in mode or "graph" in mode) else 1      # a second step: a cached / captured state must not go stale
    mesh_in = [Meshes([v], [f]) for v, f in meshes]
    if mode.startswith("collated"):
        mesh_in = ops.collate_meshes(meshes, pin_memory=False)
    for step in range(steps):
        color.grad = None
        az, el, di = (t.to(dev).requires_grad_() for t in views)
        c_in = color * (1.0 + 0.1 * step)
        img, _ = r(mesh_in, None, az, el, di, color=c_in)
        (img[:, :, :3] * w).sum().backward()
        assert color.grad is not None and torch.isfinite(color.grad).all() and float(color.grad.abs().max()) > 0
        assert all(t.grad is not None and torch.isfinite(t.grad).all() and float(t.grad.abs().sum()) > 0 for t in (az, el, di))
        # the same through ops, with the colours the renderer was given
        c_det = c_in.detach()
        if shape == "obj":
            want = _ops_colour_grads_obj(meshes, az, el, di, M, S, w, shader, c_det, K) * (1.0 + 0.1 * step)
        else:
            per_v = torch.cat([torch.broadcast_to(c_det, (B, maxV, 3))[b, :n] for b, n in enumerate(nv)])
            gv = _ops_colour_grads(meshes, az, el, di, M, S, w, shader, per_v, K) * (1.0 + 0.1 * step)
            full = torch.zeros(B, maxV, 3, device=dev)
            off = 0
            for b, n in enumerate(nv):
                full[b, :n] = gv[off:off + n]
                off += n
            want = full.sum(1, keepdim=True) if shape == "per_object" else full
        err = rel(color.grad, want.cpu().numpy())
        print(f"[MVRenderer {mode} {shape} step {step}] colour grad vs ops level: {err:.1e}")
        assert err < 1e-5, err


def _ops_colour_grads_obj(meshes, az, el, di, M, S, w, shader, colour, K):
    dev = az.device
    R, T, C, _ = ops._LookAt.apply(*(t.detach() for t in (az, el, di)))
    vs = [v for v, _ in meshes]
    geom = ops.PackedMeshes.from_packed(torch.cat(vs).to(dev), torch.cat([f for _, f in meshes]).to(dev),
                                        [v.shape[0] for v in vs], [f.shape[0] for _, f in meshes])
    leaf = colour.detach().reshape(3).clone().requires_grad_()
    kw = dict(shader=shader, blur_radius=2e-3, sigma=1e-3, gamma=1e-2, faces_per_pixel=K) if shader != "hard_phong" else {}
    img, _ = ops.render_meshes(geom, M, R, T, C, torch.tensor([[0.0, 1.0, 0.0]], device=dev), leaf, WHITE.to(dev), S, **kw)
    (img.view(len(meshes), M, -1, S, S)[:, :, :3] * w).sum().backward()
    return leaf.grad


def test_mvrenderer_soft_silhouette_gives_no_colour_gradient(cuda_device):
    dev = cuda_device
    M, S = 2, 40
    meshes = synth.make_meshes(2, 200, 71)
    color = torch.tensor([0.2, 0.4, 0.6], device=dev, requires_grad=True)
    az, el, di = (t.to(dev).requires_grad_() for t in synth.learned_spherical_views(2, M, 72))
    r = MVRenderer(M, image_size=S, pc_rendering=False, object_color="custom", light_direction="fixed", shader="soft_silhouette",
                   faces_per_pixel=4, blur_radius=2e-3, blend_sigma=1e-3, keep_alpha=True).to(dev)
    img, _ = r([Meshes([v], [f]) for v, f in meshes], None, az, el, di, color=color)
    img[:, :, 3].sum().backward()
    assert color.grad is None
    assert all(t.grad is not None and torch.isfinite(t.grad).all() for t in (az, el, di))


@pytest.mark.parametrize("nb", [2, 8], ids=["graph_size_24_views", "eager_size_96_views"])
def test_mvrenderer_point_colour_gradient(cuda_device, nb):
    """A (3,) point colour that requires grad at <= 48 views (where the automatic CUDA graph would run) and > 48 views: its
    gradient equals ops.render_points_from_angles'."""
    dev = cuda_device
    M, S = 12, 64
    pts = synth.make_clouds(nb, 512, 81).to(dev)
    views = synth.learned_spherical_views(nb, M, 82)
    w = torch.rand(nb, M, 3, S, S, generator=torch.Generator().manual_seed(83)).to(dev)
    color = torch.tensor([0.2, 0.5, 0.8], device=dev, requires_grad=True)
    r = MVRenderer(M, image_size=S, pc_rendering=True, object_color="custom").to(dev)
    az, el, di = (t.to(dev).requires_grad_() for t in views)
    img, _ = r(None, pts, az, el, di, color=color)
    (img * w).sum().backward()
    assert color.grad is not None and float(color.grad.abs().max()) > 0
    leaf = color.detach().clone().requires_grad_()
    img2, _, _ = ops.render_points_from_angles(pts, leaf, M, *(t.detach().to(dev) for t in views), r.points_radius,
                                               WHITE.to(dev), S, points_per_pixel=r.points_per_pixel, compositor=r.compositor)
    assert torch.equal(img2.view_as(img), img.detach())
    (img2.view_as(img) * w).sum().backward()
    err = rel(color.grad, leaf.grad.cpu().numpy())
    print(f"[points {nb * M} views] colour grad vs ops level: {err:.1e}")
    assert err < 1e-5, err


# ------------------------------------------------------------------------------------------------- 6. the feature does its job
def test_per_vertex_colour_fit(cuda_device):
    """Texture fitting at a small size: per-vertex colours, started at grey, are fitted by Adam (lr 0.05, 50 steps) to four
    views of the same mesh rendered with known random colours under a fixed light; the loss falls at least tenfold."""
    dev = cuda_device
    v, f = synth.uv_sphere(16, 32)
    v, f = v.to(dev), f.to(dev)
    H = 64
    az = torch.tensor([0.0, 90.0, 180.0, 270.0], device=dev); el = torch.tensor([20.0, -30.0, 40.0, -10.0], device=dev)
    R, T, C, _ = ops._LookAt.apply(az, el, torch.full((4,), 2.5, device=dev))
    light = torch.tensor([[0.0, 1.0, 0.0]], device=dev); bg = torch.ones(3, device=dev)
    target_rgb = torch.rand(v.shape[0], 3, generator=torch.Generator().manual_seed(91)).to(dev)

    def render(rgb):
        geom = ops.PackedMeshes.from_packed(v, f, [v.shape[0]], [f.shape[0]], vert_rgb=rgb.detach())
        img, _ = ops.render_meshes(geom, 4, R, T, C, light, None, bg, H, rgb=rgb)
        return img

    with torch.no_grad():
        target = render(target_rgb)
    rgb = torch.full_like(target_rgb, 0.5).requires_grad_()
    opt = torch.optim.Adam([rgb], lr=0.05)
    losses = []
    for _ in range(50):
        opt.zero_grad()
        loss = ((render(rgb) - target) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    print(f"[colour fit] loss {losses[0]:.3e} -> {losses[-1]:.3e}")
    assert all(np.isfinite(losses))
    assert losses[-1] <= 0.1 * losses[0], losses
