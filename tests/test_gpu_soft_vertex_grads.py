"""GPU tests of the vertex gradients of the soft shaders (run on the B200 box with `-m gpu`).

render_meshes(shader="soft_phong" | "soft_silhouette", verts=v) and MVRenderer(shader=...) with meshes whose vertices require
grad: mesh_soft_backward_kernel<true> returns d/d positions (projection chain through every route a fragment's gradient takes:
colour, zbuf including the z_inv_max term, signed distance, clipped barycentrics, perspective correction, near-plane clipping)
and d/d unit normals (Phong), then mvr_mesh_normals_backward chains the normals to the positions (soft_phong only).

1. Against fp64 autograd of oracle/torch_ref.py (render_mesh_view_soft with the normals from vertex_normals) on every case of
   test_gpu_mesh_branches.SOFT and test_gpu_parity.SOFT_CASES, at VERT_GRAD_RTOL (the hard path's vertex bar).
2. The camera gradients are bit-identical with and without vertex gradients (the GV = false instance is today's kernel).
3. MVRenderer: list-of-meshes input, vertex gradients equal to the ops-level ones, angle gradients still present.
4. A seeded silhouette fit: the gradients are good enough to deform a sphere towards a target silhouette.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, Meshes, ops, synth
from test_gpu_branches import VERT_GRAD_RTOL, launches
from test_gpu_mesh_branches import BG, LIGHT, OBJ, SOFT, SOFT_PARAMS
from test_gpu_parity import K00, K11, SOFT_CASES, rel

pytestmark = pytest.mark.gpu


def _cases():
    """name -> (configuration in test_gpu_mesh_branches.SOFT's format, shader)."""
    out = {f"{n}-{s}": (SOFT[n], s) for n, s in SOFT_PARAMS}
    for n, c in SOFT_CASES.items():      # one mesh; views from learned_spherical_views(1, M, seed + 1) as the parity test
        out[f"parity_{n}"] = (dict(meshes=[(c["faces"], c["seed"])], M=c["M"], HW=(c["H"], c["H"]), K=c["K"], blur=c["blur"],
                                   sigma=c["sigma"], gamma=c["gamma"], clip=c.get("clip")), c["shader"])
    return out


CASES = _cases()


class Scene:
    """The inputs of one case: meshes, cameras (oracle look_at), colours, light, cotangent."""

    def __init__(self, oracle, c, shader):
        self.c, self.shader = c, shader
        self.meshes = [synth.make_mesh(nf, seed) for nf, seed in c["meshes"]]
        self.B, self.M, (self.H, self.W), self.K = len(self.meshes), c["M"], c["HW"], c["K"]
        self.persp, self.cull, self.near, self.clip = c.get("persp", True), c.get("cull", False), c.get("near", False), c.get("clip")
        self.views = c.get("views") or synth.learned_spherical_views(self.B, self.M, c["meshes"][0][1] + 1)
        self.R, self.T, self.Cc = oracle.look_at(*(t.numpy().ravel() for t in self.views))
        self.nv = [v.shape[0] for v, _ in self.meshes]
        self.nf = [f.shape[0] for _, f in self.meshes]
        self.voff = np.cumsum([0] + self.nv)
        self.vp = torch.cat([v for v, _ in self.meshes])
        self.vrgb = torch.rand(int(self.voff[-1]), 3, generator=torch.Generator().manual_seed(7)) if c.get("vrgb") else None
        self.light = torch.from_numpy(self.Cc.copy()) if c.get("light") == "camera" else torch.tensor(LIGHT)
        self.obj, self.bg = torch.tensor(OBJ), torch.tensor(BG)
        self.g = torch.randn(self.B * self.M, 4, self.H, self.W, generator=torch.Generator().manual_seed(5))
        self.z_clip = 0.5 if self.near else None

    def render(self, dev, verts=None, cameras=None):
        geom = ops.PackedMeshes.from_packed(self.vp.to(dev), torch.cat([f for _, f in self.meshes]).to(dev), self.nv, self.nf,
                                            vert_rgb=self.vrgb)
        Rd, Td, Cd = cameras or (torch.from_numpy(x).to(dev) for x in (self.R, self.T, self.Cc))
        c = self.c
        return ops.render_meshes(geom, self.M, Rd, Td, Cd, self.light.to(dev), None if self.vrgb is not None else self.obj.to(dev),
                                 self.bg.to(dev), (self.H, self.W), faces_per_pixel=self.K, shader=self.shader, blur_radius=c["blur"],
                                 sigma=c["sigma"], gamma=c["gamma"], perspective_correct=self.persp, cull_backfaces=self.cull,
                                 clip_barycentric_coords=self.clip, verts=verts)

    def reference(self, oracle, dtype):
        """Autograd of torch_ref in `dtype` on the reference rasterizer's fragments (bit-exact with the CUDA path's: compared by
        the caller) -> (d loss / d packed verts, fragment indices (n,H,W,K), clip stats)."""
        from oracle import torch_ref as tr
        c, H, W, K = self.c, self.H, self.W, self.K
        vd = self.vp.to(dtype, copy=True).requires_grad_()
        loss, p2fs = 0, []
        stats = dict(clip1=0, clip2=0)
        for b, (_, f) in enumerate(self.meshes):
            s = slice(int(self.voff[b]), int(self.voff[b + 1]))
            nrm = tr.vertex_normals(vd[s], f)
            rgb = (self.vrgb[s] if self.vrgb is not None else self.obj.expand(self.nv[b], 3)).to(dtype)
            for m in range(self.M):
                n = b * self.M + m
                v32 = self.vp[s].numpy()
                fv32 = torch.from_numpy(oracle.project_perspective(v32, self.R[n], self.T[n], K00, K11))[f]      # the oracle's IEEE projection
                rp2f, _, _, _, rp2c = tr.rasterize_meshes_soft(fv32, H, W, K, c["blur"], self.persp, self.clip, self.cull,
                                                               z_clip=self.z_clip, return_sub=True)
                p2fs.append(rp2f)
                if self.near:
                    nb_behind = (fv32[:, :, 2] < self.z_clip).sum(1)            # 1: two sub-triangles, 2: one
                    kind = torch.where(rp2f >= 0, nb_behind[rp2f.clamp_min(0)], torch.zeros_like(rp2f))
                    stats["clip2"] += int((kind == 1).sum()); stats["clip1"] += int((kind == 2).sum())
                light = self.light[n if self.light.shape[0] > 1 else 0]
                ref, _ = tr.render_mesh_view_soft(vd[s], f, nrm, rgb, *(torch.from_numpy(x[n]).to(dtype) for x in (self.R, self.T, self.Cc)),
                                                  light.to(dtype), self.bg.to(dtype), K00, K11, H, W, K, c["blur"], self.shader,
                                                  sigma=c["sigma"], gamma=c["gamma"], perspective_correct=self.persp, clip_bary=self.clip,
                                                  cull_backfaces=self.cull, p2f=None if self.near else rp2f, z_clip=self.z_clip,
                                                  p2c=rp2c if self.near else None)
                loss = loss + (ref * self.g[n].to(dtype)).sum()
        loss.backward()
        return vd.grad, torch.stack(p2fs), stats


# ------------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("case", list(CASES))
def test_soft_vertex_gradients_match_the_torch_restatement(oracle, cuda_device, case):
    """d loss / d verts of render_meshes(shader=soft_*, verts=vg) against fp64 autograd of the restatement, within
    VERT_GRAD_RTOL of the tensor's largest entry; every mesh of the batch gets a gradient; the backward runs
    mesh_soft_backward_kernel<true> once and the normals backward once (soft_phong) or not at all (soft_silhouette)."""
    c, shader = CASES[case]
    dev = cuda_device
    sc = Scene(oracle, c, shader)
    vg = sc.vp.to(dev).requires_grad_()
    img, frag = sc.render(dev, verts=vg)
    g = sc.g.to(dev)
    want = {"mesh_soft_backward_kernel<true>": 1, "mesh_soft_backward_kernel<false>": 0,
            "geom_normals_bwd_face_kernel": 1 if shader == "soft_phong" else 0}
    counts = {}
    for pfx in want:      # one backward per profiled prefix; the gradient of the last one is compared
        vg.grad = None
        _, counts[pfx] = launches(pfx, lambda: img.backward(g, retain_graph=True))
    assert counts == want, counts
    ref, rp2f, stats = sc.reference(oracle, torch.float64)
    assert torch.equal(frag["pix_to_face"].cpu().long(), rp2f), "fragments differ from the reference rasterizer"
    err = rel(vg.grad, ref.numpy())
    per_mesh = [float(vg.grad[int(sc.voff[b]):int(sc.voff[b + 1])].abs().max()) for b in range(sc.B)]
    print(f"[{case}] vertex grad err {err:.1e} (bar {VERT_GRAD_RTOL:.0e})  launches {counts}  max per mesh {per_mesh}  {stats}")
    assert torch.isfinite(vg.grad).all()
    assert err < VERT_GRAD_RTOL, err
    assert all(x > 0 for x in per_mesh), per_mesh
    if sc.near:                                          # one- and two-sub-triangle clips among the fragments
        assert stats["clip1"] > 0 and stats["clip2"] > 0, stats


# ------------------------------------------------------------------------------------------------- 2. cameras unchanged
@pytest.mark.parametrize("case", list(CASES))
def test_soft_camera_gradients_do_not_depend_on_vertex_gradients(oracle, cuda_device, case):
    """(gR, gT, gC) with `verts` requiring grad are bit-identical to those without; without, the backward runs
    mesh_soft_backward_kernel<false> and no normals backward."""
    c, shader = CASES[case]
    dev = cuda_device
    sc = Scene(oracle, c, shader)
    g = sc.g.to(dev)
    out = {}
    for with_verts in (False, True):
        cam = tuple(torch.from_numpy(x).to(dev).requires_grad_() for x in (sc.R, sc.T, sc.Cc))
        vg = sc.vp.to(dev).requires_grad_() if with_verts else None
        img, _ = sc.render(dev, verts=vg, cameras=cam)
        if not with_verts:
            want = {"mesh_soft_backward_kernel<false>": 1, "mesh_soft_backward_kernel<true>": 0, "geom_normals_bwd_face_kernel": 0}
            counts = {}
            for pfx in want:
                for t in cam:
                    t.grad = None
                _, counts[pfx] = launches(pfx, lambda: img.backward(g, retain_graph=True))
            assert counts == want, counts
        else:
            img.backward(g)
            assert vg.grad is not None
        out[with_verts] = [t.grad for t in cam]
    for name, a, b in zip(("gR", "gT", "gC"), out[False], out[True]):
        assert torch.equal(a, b), (name, float((a - b).abs().max()))


# ------------------------------------------------------------------------------------------------- 3. MVRenderer
def test_mvrenderer_soft_silhouette_vertex_gradients(cuda_device):
    """A list of Meshes whose vertices require grad, shader="soft_silhouette": every vertex tensor gets a finite, non-zero
    gradient equal (to the order of the atomics) to the ops-level gradient for the same angles, and azim / elev / dist still
    receive theirs.  normalize / bf16 output stay rejected with the soft shaders."""
    dev = cuda_device
    M, S, K = 3, 48, 6
    mesh_list = synth.make_meshes(2, 400, 41)
    views = synth.learned_spherical_views(2, M, 42)
    w = torch.rand(2, M, S, S, generator=torch.Generator().manual_seed(43)).to(dev)
    vs = [v.clone().requires_grad_() for v, _ in mesh_list]      # host tensors, as a data loader hands them over
    az, el, di = (t.to(dev).requires_grad_() for t in views)
    r = MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed", faces_per_pixel=K, shader="soft_silhouette",
                   blur_radius=2e-3, blend_sigma=1e-3, keep_alpha=True).to(dev)
    img, _ = r([Meshes([v], [f]) for v, (_, f) in zip(vs, mesh_list)], None, az, el, di)
    (img[:, :, 3] * w).sum().backward()
    for v in vs:
        assert v.grad is not None and torch.isfinite(v.grad).all() and float(v.grad.abs().max()) > 0
    assert all(t.grad is not None and torch.isfinite(t.grad).all() and float(t.grad.abs().sum()) > 0 for t in (az, el, di))
    # the same render through ops: look_at + render_meshes(verts=...)
    vg = torch.cat([v.detach() for v in vs]).to(dev).requires_grad_()
    R, T, C, _ = ops._LookAt.apply(*(t.detach() for t in (az, el, di)))
    geom = ops.PackedMeshes.from_packed(vg.detach(), torch.cat([f for _, f in mesh_list]).to(dev), [v.shape[0] for v in vs],
                                        [f.shape[0] for _, f in mesh_list])
    white = torch.ones(3, device=dev)
    img2, _ = ops.render_meshes(geom, M, R, T, C, torch.tensor([[0.0, 1.0, 0.0]], device=dev), white, white, S, faces_per_pixel=K,
                                shader="soft_silhouette", blur_radius=2e-3, sigma=1e-3, gamma=1e-4, verts=vg)
    assert torch.equal(img2.view(2, M, 4, S, S), img.detach())
    (img2.view(2, M, 4, S, S)[:, :, 3] * w).sum().backward()
    err = rel(torch.cat([v.grad for v in vs]), vg.grad.cpu().numpy())
    print(f"[MVRenderer soft_silhouette] vertex grads vs ops level: {err:.1e}")
    assert err < 1e-5, err
    with pytest.raises(ValueError):
        ops.render_meshes(geom, M, R, T, C, torch.tensor([[0.0, 1.0, 0.0]], device=dev), white, white, S, faces_per_pixel=K,
                          shader="soft_phong", blur_radius=2e-3, verts=vg, normalize=(0.5, 0.25))


# ------------------------------------------------------------------------------------------------- 4. the feature does its job
def test_soft_silhouette_fit_deforms_a_sphere(cuda_device):
    """PyTorch3D's mesh-fitting recipe at a small size: the unit sphere is deformed towards the silhouettes (4 views) of an
    ellipsoid (the sphere scaled by (1.3, 0.8, 1.0)) by Adam on per-vertex offsets for 50 steps on the L2 loss of the alpha
    channel (64x64, K = 16, sigma = 1e-3, blur = log(1 / 1e-4 - 1) sigma): the loss at least halves and stays finite."""
    dev = cuda_device
    v0, f = synth.uv_sphere(12, 24)
    v0, f = v0.to(dev), f.to(dev)
    H, K, sigma = 64, 16, 1e-3
    blur = float(np.log(1.0 / 1e-4 - 1.0)) * sigma
    az = torch.tensor([0.0, 90.0, 180.0, 270.0], device=dev); el = torch.tensor([20.0, -30.0, 40.0, -10.0], device=dev)
    R, T, C, _ = ops._LookAt.apply(az, el, torch.full((4,), 3.0, device=dev))
    light = torch.tensor([[0.0, 1.0, 0.0]], device=dev); white = torch.ones(3, device=dev)

    def alpha(v):
        geom = ops.PackedMeshes.from_packed(v.detach(), f, [v.shape[0]], [f.shape[0]])
        img, _ = ops.render_meshes(geom, 4, R, T, C, light, white, white, H, faces_per_pixel=K, shader="soft_silhouette",
                                   blur_radius=blur, sigma=sigma, verts=v)
        return img[:, 3]

    with torch.no_grad():
        target = alpha(v0 * torch.tensor([1.3, 0.8, 1.0], device=dev))
    off = torch.zeros_like(v0, requires_grad=True)
    opt = torch.optim.Adam([off], lr=1e-2)
    losses = []
    for _ in range(50):
        opt.zero_grad()
        loss = ((alpha(v0 + off) - target) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    print(f"[silhouette fit] loss {losses[0]:.3e} -> {losses[-1]:.3e}")
    assert all(np.isfinite(losses))
    assert losses[-1] <= 0.5 * losses[0], losses
