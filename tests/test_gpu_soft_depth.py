"""shader="soft_depth" on the GPU ([upstream] SoftDepthShader): the K fragments of the blurred rasterizer blended into one depth
plane by the cumulative sum of sigmoid(-dists / sigma) clamped at 1, depth_background taking what is left; differentiable
w.r.t. the cameras and the vertices across silhouette edges.

1. Parity on every case of test_gpu_mesh_branches.SOFT and test_gpu_parity.SOFT_CASES: fragments bit-exact against
   torch_ref.rasterize_meshes_soft, depth within 1e-5 of the largest |depth|, R / T gradients within 1e-4 and vertex gradients
   within VERT_GRAD_RTOL of fp64 autograd of tests/soft_depth_ref.py render_mesh_view_soft_depth on the kernels' fp32 projection
   (straight through, as tests/test_gpu_depth.py), gC exactly 0.  The clamp decision
   c <= 1 of a pixel whose cumulative sum lies within rounding of 1 can differ between the kernels' fp32 sum and the fp64
   reference; the reference takes that decision from the fp32 sum (mirrored on the host) and the test counts the pixels where
   it had to.
2. Determinism: camera gradients bit-identical over two runs and with / without vertex gradients.
3. The kernels that run, and those that must not.
4. The saturated limit (blur 0, tiny sigma): the nearest fragment's zbuf bit for bit, hard_depth's faces, the background.
5. What hard depth cannot do: an in-plane translation of a square facing the camera gets no gradient from hard_depth and one of
   the right sign from soft_depth.
6. MVRenderer(shader="soft_depth"): list and collated input, angle and vertex gradients equal to the ops-level chain,
   depth_background = 0, the rejected options.
7. A seeded fit of a mesh translation to target depth maps with an unmasked loss.
"""
import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, Meshes, ops, synth

import soft_depth_ref
from test_gpu_branches import VERT_GRAD_RTOL, expect_launches, launches
from test_gpu_mesh_branches import SOFT
from test_gpu_parity import K00, K11, SOFT_CASES

pytestmark = pytest.mark.gpu

GRAD_RTOL = 1e-4
DEPTH_RTOL = 1e-5
BGD = 4.0          # a background just behind the objects (dist ~2): the depth bar is then relative to the objects' depths
D = torch.float64


def rel(a, b):
    a, b = torch.as_tensor(a).detach().double().cpu(), torch.as_tensor(b).detach().double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-12))


def _cases():
    """name -> configuration in test_gpu_mesh_branches.SOFT's format (the shader there does not matter here)."""
    out = dict(SOFT)
    for n, c in SOFT_CASES.items():      # one mesh; views from learned_spherical_views(1, M, seed + 1) as the parity test
        out[f"parity_{n}"] = dict(meshes=[(c["faces"], c["seed"])], M=c["M"], HW=(c["H"], c["H"]), K=c["K"], blur=c["blur"],
                                  sigma=c["sigma"], gamma=c["gamma"], clip=c.get("clip"))
    return out


CASES = _cases()


def sigmoid_f32(d, sigma):
    """The kernels' fp32 sigmoidf_(-d / sigma) = 1 / (1 + expf(d / sigma)), on the host."""
    x = (-d.astype(np.float32) / np.float32(sigma)).astype(np.float32)
    with np.errstate(over="ignore"):
        return (np.float32(1.0) / (np.float32(1.0) + np.exp(-x).astype(np.float32))).astype(np.float32)


def live_f32(p2f, dists, sigma):
    """c_k <= 1 as the kernels decide it: the fp32 running sum over the valid entries, list order."""
    p = np.where(p2f >= 0, sigmoid_f32(dists, sigma), np.float32(0.0)).astype(np.float32)
    c = np.zeros(p.shape[:-1], np.float32)
    live = np.zeros(p.shape, bool)
    for k in range(p.shape[-1]):
        c = (c + p[..., k]).astype(np.float32)
        live[..., k] = c <= np.float32(1.0)
    return live


def blend_with_decision(p2f, zbuf, dists, sigma, background, live):
    """soft_depth_blend with min(c, 1) written as where(live, c, 1): with live = (c <= 1) it is the upstream formula (the clamp
    passes the gradient at equality too); with the kernels' fp32 decision it is the substitution described above."""
    prob = torch.sigmoid(-dists / sigma) * (p2f >= 0)
    c = prob.cumsum(-1)
    m = torch.where(live, c, torch.ones_like(c))
    w = m.diff(dim=-1, prepend=torch.zeros_like(m[..., :1]))
    return (w * zbuf).sum(-1) + (1 - m[..., -1]) * background


class Scene:
    def __init__(self, oracle, c, bg=BGD, meshes=None):
        """meshes: (verts, faces) pairs to use instead of c["meshes"]' synth.make_mesh ones (c must then give the views)."""
        self.c, self.bg = c, bg
        self.meshes = meshes or [synth.make_mesh(nf, seed) for nf, seed in c["meshes"]]
        self.B, self.M, (self.H, self.W), self.K = len(self.meshes), c["M"], c["HW"], c["K"]
        self.persp, self.cull, self.near, self.clip = c.get("persp", True), c.get("cull", False), c.get("near", False), c.get("clip")
        self.views = c.get("views") or synth.learned_spherical_views(self.B, self.M, c["meshes"][0][1] + 1)
        self.R, self.T, self.Cc = oracle.look_at(*(t.numpy().ravel() for t in self.views))
        self.nv = [v.shape[0] for v, _ in self.meshes]
        self.nf = [f.shape[0] for _, f in self.meshes]
        self.voff = np.cumsum([0] + self.nv)
        self.vp = torch.cat([v for v, _ in self.meshes])
        self.vrgb = torch.rand(int(self.voff[-1]), 3, generator=torch.Generator().manual_seed(7)) if c.get("vrgb") else None
        self.g = torch.randn(self.B * self.M, 1, self.H, self.W, generator=torch.Generator().manual_seed(5))
        self.z_clip = 0.5 if self.near else None

    def render(self, dev, verts=None, cameras=None, flags=0):
        geom = ops.PackedMeshes.from_packed(self.vp.to(dev), torch.cat([f for _, f in self.meshes]).to(dev), self.nv, self.nf,
                                            vert_rgb=self.vrgb)
        Rd, Td, Cd = cameras or (torch.from_numpy(x).to(dev) for x in (self.R, self.T, self.Cc))
        c = self.c
        return ops.render_meshes(geom, self.M, Rd, Td, Cd, torch.ones(1, 3, device=dev), torch.ones(3, device=dev),
                                 torch.zeros(3, device=dev), (self.H, self.W), faces_per_pixel=self.K, shader="soft_depth",
                                 blur_radius=c["blur"], sigma=c["sigma"], perspective_correct=self.persp, cull_backfaces=self.cull,
                                 clip_barycentric_coords=self.clip, verts=verts, depth_background=self.bg, _extra_flags=flags)

    def reference(self, oracle, gpu_dists):
        """fp64 autograd of render_mesh_view_soft_depth on the reference rasterizer's fragment lists, on the kernels' fp32 IEEE
        projection (the oracle's, straight through: the comparison measures the depth chain, not how a 1-ulp change of a projected
        corner moves an extrapolated or 1/area-conditioned fragment depth) ->
        depth (n,1,H,W), gR, gT, gV, fragment indices (n,H,W,K), (pixels whose clamp decision was substituted, the largest
        |c - 1| of the fp64 sum where fp32 and fp64 decide differently), clip stats."""
        from oracle import torch_ref as tr
        c, H, W, K, sigma = self.c, self.H, self.W, self.K, self.c["sigma"]
        vd = self.vp.to(D, copy=True).requires_grad_()
        Rr, Tr = (torch.from_numpy(x).to(D).requires_grad_() for x in (self.R, self.T))
        loss, p2fs, deps, subst, off1 = 0, [], [], 0, 0.0
        stats = dict(clip1=0, clip2=0)
        for b, (_, f) in enumerate(self.meshes):
            s = slice(int(self.voff[b]), int(self.voff[b + 1]))
            for m in range(self.M):
                n = b * self.M + m
                fv32 = torch.from_numpy(oracle.project_perspective(self.vp[s].numpy(), self.R[n], self.T[n], K00, K11))[f]
                rp2f, _, _, _, rp2c = tr.rasterize_meshes_soft(fv32, H, W, K, c["blur"], self.persp, self.clip, self.cull,
                                                               z_clip=self.z_clip, return_sub=True)
                p2fs.append(rp2f)
                if self.near:
                    nb_behind = (fv32[:, :, 2] < self.z_clip).sum(1)
                    kind = torch.where(rp2f >= 0, nb_behind[rp2f.clamp_min(0)], torch.zeros_like(rp2f))
                    stats["clip2"] += int((kind == 1).sum()); stats["clip1"] += int((kind == 2).sum())
                ndc = tr.project_perspective(vd[s], Rr[n], Tr[n], K00, K11)
                ndc = ndc + (torch.from_numpy(oracle.project_perspective(self.vp[s].numpy(), self.R[n], self.T[n], K00, K11)).to(D)
                             - ndc).detach()
                dep, frag = soft_depth_ref.render_mesh_view_soft_depth(None, f, None, None, K00, K11, H, W, K, c["blur"], sigma, self.bg,
                                                                  self.persp, self.clip, p2f=None if self.near else rp2f,
                                                                  cull_backfaces=self.cull, z_clip=self.z_clip,
                                                                  p2c=rp2c if self.near else None, ndc=ndc)
                p2f, zb, di = frag["pix_to_face"], frag["zbuf"], frag["dists"]
                with torch.no_grad():
                    c64 = (torch.sigmoid(-di / sigma) * (p2f >= 0)).cumsum(-1)
                live = torch.from_numpy(live_f32(p2f.numpy(), gpu_dists[n].numpy(), sigma))
                differ = (live != (c64 <= 1)) & (p2f >= 0)
                ns = int(differ.any(-1).sum())
                if ns:      # the clamp decision of these pixels from the kernels' fp32 sum
                    subst += ns
                    off1 = max(off1, float((c64[differ] - 1).abs().max()))
                    dep = blend_with_decision(p2f, zb, di, sigma, self.bg, live)
                deps.append(dep.detach())
                loss = loss + (dep * self.g[n, 0].to(D)).sum()
        loss.backward()
        return torch.stack(deps)[:, None], Rr.grad, Tr.grad, vd.grad, torch.stack(p2fs), (subst, off1), stats


# ------------------------------------------------------------------------------------------------- 1. parity, 3. launches
@pytest.mark.parametrize("case", list(CASES))
def test_soft_depth_matches_the_torch_restatement(oracle, cuda_device, case):
    c = CASES[case]
    dev = cuda_device
    sc = Scene(oracle, c)
    cam = tuple(torch.from_numpy(x).to(dev).requires_grad_() for x in (sc.R, sc.T, sc.Cc))
    vg = sc.vp.to(dev).requires_grad_()
    fwd = {"mesh_scatter": 1, "mesh_shade": 1, "mesh_soft_depth_kernel": 1, "mesh_soft_blend_kernel": 0}
    counts, out = {}, None
    for pfx in fwd:
        o, counts[pfx] = launches(pfx, lambda: sc.render(dev, verts=vg, cameras=cam))
        out = out or o
    expect_launches(counts, fwd, f"[{case}] forward")
    assert counts["mesh_soft_depth_kernel"] == 1
    depth, frag = out
    assert depth.shape == (sc.B * sc.M, 1, sc.H, sc.W) and depth.dtype == torch.float32
    g = sc.g.to(dev)
    back = {"mesh_soft_depth_backward_kernel<true>": 1, "mesh_soft_depth_backward_kernel<false>": 0,
            "mesh_backward_finish_kernel": 1, "mesh_soft_backward_kernel": 0, "geom_normals_bwd_face_kernel": 0}
    nb = {}
    for pfx in back:      # one backward per profiled prefix; the gradients of the last one are compared
        for t in (*cam, vg):
            t.grad = None
        _, nb[pfx] = launches(pfx, lambda: depth.backward(g, retain_graph=True))
    assert nb == back, nb
    ref, gRr, gTr, gVr, rp2f, subst, stats = sc.reference(oracle, frag["dists"].cpu())
    assert torch.equal(frag["pix_to_face"].cpu().long(), rp2f), "fragments differ from the reference rasterizer"
    e_d = rel(depth, ref)
    e_R, e_T, e_V = rel(cam[0].grad, gRr), rel(cam[1].grad, gTr), rel(vg.grad, gVr)
    covered = int((rp2f[..., 0] >= 0).sum())
    print(f"[{case}] depth {e_d:.1e}  R {e_R:.1e}  T {e_T:.1e}  verts {e_V:.1e}  clamp decisions taken from fp32: {subst[0]} of "
          f"{covered} covered pixels (fp64 sum within {subst[1]:.1e} of 1 there)  {stats}")
    assert e_d < DEPTH_RTOL, e_d
    assert e_R < GRAD_RTOL and e_T < GRAD_RTOL, (e_R, e_T)
    assert e_V < VERT_GRAD_RTOL, e_V
    assert torch.equal(cam[2].grad, torch.zeros_like(cam[2]))
    assert subst[1] < 1e-5, subst      # substituted only where the sum is 1 to fp32 rounding
    per_mesh = [float(vg.grad[int(sc.voff[b]):int(sc.voff[b + 1])].abs().max()) for b in range(sc.B)]
    assert all(x > 0 for x in per_mesh), per_mesh
    if sc.near:
        assert stats["clip1"] > 0 and stats["clip2"] > 0, stats


# ------------------------------------------------------------------------------------------------- 2. determinism
@pytest.mark.parametrize("case", ["ragged", "near_plane", "parity_silhouette"])
def test_soft_depth_camera_gradients_are_deterministic(oracle, cuda_device, case):
    dev = cuda_device
    sc = Scene(oracle, CASES[case])
    g = sc.g.to(dev)
    got = []
    for with_verts in (False, False, True):
        cam = tuple(torch.from_numpy(x).to(dev).requires_grad_() for x in (sc.R, sc.T, sc.Cc))
        vg = sc.vp.to(dev).requires_grad_() if with_verts else None
        depth, _ = sc.render(dev, verts=vg, cameras=cam)
        depth.backward(g)
        got.append((cam[0].grad, cam[1].grad))
    for gR, gT in got[1:]:
        assert torch.equal(gR, got[0][0]) and torch.equal(gT, got[0][1])


# ------------------------------------------------------------------------------------------------- 4. saturated limit
def test_soft_depth_saturated_limit_is_the_hard_depth(oracle, cuda_device):
    """blur 0 and sigma = 1e-7: every fragment lies inside its face, the nearest one's fp32 probability is 1 almost everywhere,
    and there the depth is its zbuf bit for bit; the nearest faces are hard_depth's; uncovered pixels hold depth_background."""
    dev = cuda_device
    meshes = [synth.make_mesh(900, 61), synth.make_mesh(400, 62)]
    M, H, K, bg = 3, 64, 4, 9.5
    views = synth.learned_spherical_views(2, M, 63)
    R, T, C = oracle.look_at(*(t.numpy().ravel() for t in views))
    Rd, Td, Cd = (torch.from_numpy(x).to(dev) for x in (R, T, C))
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    args = (geom, M, Rd, Td, Cd, torch.ones(1, 3, device=dev), torch.ones(3, device=dev), torch.zeros(3, device=dev), H)
    dep, frag = ops.render_meshes(*args, faces_per_pixel=K, shader="soft_depth", blur_radius=0.0, sigma=1e-7, depth_background=bg)
    hard, hfrag = ops.render_meshes(*args, shader="hard_depth", depth_background=bg)
    p2f0 = frag["pix_to_face"][..., 0]
    assert torch.equal(p2f0, hfrag["pix_to_face"][..., 0])
    prob0 = torch.from_numpy(sigmoid_f32(frag["dists"][..., 0].cpu().numpy(), 1e-7)).to(dev)
    sat = (p2f0 >= 0) & (prob0 == 1)
    assert int(sat.sum()) > 0.9 * int((p2f0 >= 0).sum())
    assert torch.equal(dep[:, 0][sat], frag["zbuf"][..., 0][sat])
    assert torch.equal(dep[:, 0][sat], hard[:, 0][sat])
    empty = p2f0 < 0
    assert int(empty.sum()) > 0 and bool((dep[:, 0][empty] == bg).all())


# ------------------------------------------------------------------------------------------------- 5. across the silhouette
def test_soft_depth_moves_a_square_that_hard_depth_cannot(cuda_device):
    """A two-triangle square in the plane z = 0 facing the camera (azim 0, elev 0): every corner has the same view depth.  The
    gradient of an L2 loss against the depth of the square shifted by +0.1 in x, w.r.t. a common x translation of its vertices,
    is exactly 0 under hard_depth (its backward uses only z differences) and negative under soft_depth (descent moves it toward
    the target)."""
    dev = cuda_device
    v0 = torch.tensor([[-0.5, -0.5, 0.0], [0.5, -0.5, 0.0], [0.5, 0.5, 0.0], [-0.5, 0.5, 0.0]], device=dev)
    f = torch.tensor([[0, 1, 2], [0, 2, 3]], device=dev)
    R, T, C, _ = ops._LookAt.apply(torch.zeros(1, device=dev), torch.zeros(1, device=dev), torch.full((1,), 2.5, device=dev))
    R, T, C = R.detach(), T.detach(), C.detach()
    light, white, black = torch.ones(1, 3, device=dev), torch.ones(3, device=dev), torch.zeros(3, device=dev)
    shift = torch.tensor([1.0, 0.0, 0.0], device=dev)

    def depth(shader, t):
        v = v0 + t * shift
        geom = ops.PackedMeshes.from_packed(v.detach(), f, [4], [2])
        kw = dict(faces_per_pixel=4, blur_radius=2e-3, sigma=2e-4) if shader == "soft_depth" else {}
        return ops.render_meshes(geom, 1, R, T, C, light, white, black, 64, shader=shader, verts=v, depth_background=6.0, **kw)[0]

    for shader in ("hard_depth", "soft_depth"):
        with torch.no_grad():
            target = depth(shader, torch.tensor(0.1, device=dev))
        t = torch.zeros((), device=dev, requires_grad=True)
        loss = ((depth(shader, t) - target) ** 2).sum()
        loss.backward()
        print(f"[{shader}] loss {float(loss.detach()):.4e}  d loss / d t {float(t.grad):.4e}")
        assert float(loss.detach()) > 0
        if shader == "hard_depth":
            assert float(t.grad) == 0.0
        else:
            assert float(t.grad) < 0.0


# ------------------------------------------------------------------------------------------------- 6. MVRenderer
def test_mvrenderer_soft_depth(cuda_device):
    dev = cuda_device
    B, M, H, K = 2, 3, 48, 6
    kw = dict(image_size=H, pc_rendering=False, light_direction="fixed", faces_per_pixel=K, shader="soft_depth", blur_radius=2e-3,
              blend_sigma=2e-4)
    meshes = [synth.make_mesh(500 + 200 * b, 70 + b) for b in range(B)]
    views = synth.learned_spherical_views(B, M, 72)
    # collated input, depth_background = 0
    r0 = MVRenderer(M, depth_background=0.0, **kw).eval()
    img0, cams0 = r0(ops.collate_meshes(meshes), None, *(t.to(dev) for t in views))
    assert img0.shape == (B, M, 1, H, H) and img0.dtype == torch.float32
    empty = r0.last_fragments["pix_to_face"][..., 0].reshape(B, M, H, H) < 0
    assert int(empty.sum()) > 0 and bool((img0[:, :, 0][empty] == 0).all())
    # list input with vertex gradients and angles that require grad (the general path)
    verts = [v.clone().to(dev).requires_grad_() for v, _ in meshes]
    faces = [f.to(dev) for _, f in meshes]
    a, e, d = (t.clone().to(dev).requires_grad_() for t in views)
    r = MVRenderer(M, depth_background=BGD, **kw).eval()
    img, _ = r([Meshes([v], [f]) for v, f in zip(verts, faces)], None, a, e, d)
    assert img.shape == (B, M, 1, H, H)
    g = torch.randn(B, M, 1, H, H, generator=torch.Generator().manual_seed(73)).to(dev)
    (img * g).sum().backward()
    assert all(v.grad is not None and torch.isfinite(v.grad).all() and float(v.grad.abs().max()) > 0 for v in verts)
    assert all(t.grad is not None and float(t.grad.abs().sum()) > 0 for t in (a, e, d))
    # the ops-level chain: look_at, render_meshes(verts=...), look_at backward
    Rk, Tk, Ck = ops.look_at_view_transform(d.detach(), e.detach(), a.detach(), return_centers=True)
    Rk, Tk = Rk.detach().requires_grad_(), Tk.detach().requires_grad_()
    vg = torch.cat([v.detach() for v in verts]).requires_grad_()
    geom = ops.PackedMeshes.from_packed(vg.detach(), torch.cat(faces), [v.shape[0] for v in verts], [f.shape[0] for f in faces])
    dep, _ = ops.render_meshes(geom, M, Rk, Tk, Ck, torch.ones(1, 3, device=dev), torch.ones(3, device=dev), torch.zeros(3, device=dev),
                               H, faces_per_pixel=K, shader="soft_depth", blur_radius=2e-3, sigma=2e-4, verts=vg, depth_background=BGD)
    assert torch.equal(dep.view(B, M, 1, H, H), img.detach())
    dep.backward(g.reshape(B * M, 1, H, H))
    ga, ge, gd = ops._look_at_backward_launch(*(t.detach().reshape(-1).float() for t in (a, e, d)), Rk.grad, Tk.grad, None)
    for got, want in ((a.grad, ga), (e.grad, ge), (d.grad, gd)):
        assert torch.allclose(got.reshape(-1), want, rtol=1e-6, atol=1e-6 * float(want.abs().max())), rel(got.reshape(-1), want)
    e_v = rel(torch.cat([v.grad for v in verts]), vg.grad)
    print(f"[MVRenderer soft_depth] vertex grads vs ops level: {e_v:.1e}")
    assert e_v < 1e-5, e_v
    # rejected options
    for bad in (dict(normalize=((0.5,) * 3, (0.2,) * 3)), dict(out_dtype=torch.bfloat16), dict(keep_alpha=True)):
        with pytest.raises(ValueError):
            MVRenderer(M, **kw, **bad)
    for bad in (dict(normalize=((0.5,) * 3, (0.2,) * 3)), dict(out_dtype=torch.bfloat16)):
        with pytest.raises(ValueError):
            ops.render_meshes(geom, M, Rk, Tk, Ck, torch.ones(1, 3, device=dev), torch.ones(3, device=dev), torch.zeros(3, device=dev),
                              H, faces_per_pixel=K, shader="soft_depth", blur_radius=2e-3, **bad)
    rp = MVRenderer(M, image_size=H, pc_rendering=True, shader="soft_depth")
    with pytest.raises(ValueError):
        rp(None, synth.make_clouds(B, 256, 74).to(dev), *(t.to(dev) for t in views))


# ------------------------------------------------------------------------------------------------- 7. seeded fit
def test_soft_depth_fit_of_a_translation_unmasked(cuda_device):
    """Adam on one offset added to every vertex of an asymmetric mesh, through MVRenderer(shader="soft_depth") with vertex
    gradients, against the depth maps of the mesh at the origin (4 views).  The start is offset by (0.25, -0.2, 0.15), where the
    silhouettes only partly overlap; the loss is the mean squared depth difference over EVERY pixel (no mask).  Loss below 20 %
    of its start, offset error below half of its start (DESIGN.md section 8 records the run)."""
    dev = cuda_device
    torch.manual_seed(0)
    M, H = 4, 96
    v, f = synth.make_mesh(2000, 17, amplitude=0.35)
    v, f = v.to(dev), f.to(dev)
    az = torch.tensor([[20.0, 110.0, 200.0, 290.0]], device=dev)
    el = torch.tensor([[15.0, -20.0, 30.0, 5.0]], device=dev)
    di = torch.full((1, M), 2.2, device=dev)
    sigma = 1e-4
    r = MVRenderer(M, image_size=H, pc_rendering=False, shader="soft_depth", light_direction="fixed", faces_per_pixel=8,
                   blur_radius=float(np.log(1.0 / 1e-4 - 1.0)) * sigma, blend_sigma=sigma, depth_background=BGD).eval()
    with torch.no_grad():
        target, _ = r([Meshes([v], [f])], None, az, el, di)
    off = torch.tensor([0.25, -0.2, 0.15], device=dev, requires_grad=True)
    with torch.no_grad():
        start, _ = r([Meshes([v + off], [f])], None, az, el, di)
        a, b = start < BGD - 1e-3, target < BGD - 1e-3
        iou = float((a & b).sum() / (a | b).sum())
    opt = torch.optim.Adam([off], lr=0.02)
    err0 = float(off.detach().norm())
    losses = []
    for _ in range(80):
        opt.zero_grad()
        dep, _ = r([Meshes([v + off], [f])], None, az, el, di)
        loss = ((dep - target) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    err = float(off.detach().norm())
    print(f"soft depth fit: silhouette IoU at the start {iou:.2f}; loss {losses[0]:.3e} -> {losses[-1]:.3e}, "
          f"offset error {err0:.3f} -> {err:.4f}")
    assert iou < 0.9
    assert all(np.isfinite(losses))
    assert losses[-1] < 0.2 * losses[0]
    assert err < 0.5 * err0
