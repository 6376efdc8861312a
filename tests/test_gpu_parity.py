"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C ABI
(mvtn_b200.ops -> libmvr_b200.so), against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star):
  * fragment indices (pix_to_face / idx): BIT-EXACT with the oracle given the same R, T (protocol stage A);
    exact depth ties are counted (the (z, index) rule makes them reproducible, so they must match too);
  * zbuf / barycentrics / dists2: bit-exact as well (same IEEE operation order, no FMA contraction);
  * images: |a-b| <= 1e-5 (values in [0,1]);
  * gradients: max|a-b| <= GRAD_RTOL * max|ref| per tensor, GRAD_RTOL = 1e-4 against the oracle's fp64-accumulated
    result (the CUDA chain is fp32 like PyTorch3D's; 1e-5 holds for the point path, the mesh shading chain has
    fp32 cancellation in the normalisations and is held to 1e-4);
  * look_at itself (sinf/cosf differ between CUDA and glibc): 2e-6 absolute on R/T (protocol stage B).
"""
import hashlib
import os

import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, Meshes, ops, synth
from mvtn_b200 import _lib as L
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

IMG_ATOL = 1e-5
GRAD_RTOL = 1e-4
POINT_GRAD_RTOL = 1e-5
K00, K11 = ops.fov_projection_scale()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def rel(a, b, floor=1e-6):
    a = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), floor))


def cams(oracle, views, dev):
    az, el, di = (t.numpy().ravel() for t in views)
    R, T, C = oracle.look_at(az, el, di)
    return R, T, C, tuple(torch.from_numpy(x).to(dev) for x in (R, T, C))


def pack_np(meshes):
    vp = torch.cat([v for v, _ in meshes]).numpy()
    fp = torch.cat([f for _, f in meshes]).numpy().astype(np.int32)
    voff = np.cumsum([0] + [v.shape[0] for v, _ in meshes]).astype(np.int32)
    foff = np.cumsum([0] + [f.shape[0] for _, f in meshes]).astype(np.int32)
    return vp, fp, voff, foff


# ------------------------------------------------------------------------------------------------ cameras
def test_look_at_forward_backward(oracle, cuda_device):
    g = torch.Generator().manual_seed(0)
    az = torch.rand(257, generator=g) * 360 - 180; el = torch.rand(257, generator=g) * 170 - 85; di = torch.rand(257, generator=g) * 2 + 1.2
    az[:4] = torch.tensor([0., 90., -90., 180.]); el[:4] = 0; di[:4] = 2.2
    a, e, d = (t.to(cuda_device).requires_grad_() for t in (az, el, di))
    R, T, C, bad = ops._LookAt.apply(a, e, d)
    Ro, To, Co = oracle.look_at(az.numpy(), el.numpy(), di.numpy())
    assert int(bad) == 0
    assert np.abs(R.detach().cpu().numpy() - Ro).max() < 2e-6
    assert np.abs(T.detach().cpu().numpy() - To).max() < 2e-6
    assert np.abs(C.detach().cpu().numpy() - Co).max() < 2e-6
    assert torch.allclose(R[0].cpu(), torch.diag(torch.tensor([-1.0, 1.0, -1.0])), atol=1e-6)
    gR, gT, gC = torch.randn(257, 3, 3, generator=g), torch.randn(257, 3, generator=g), torch.randn(257, 3, generator=g)
    ((R * gR.to(cuda_device)).sum() + (T * gT.to(cuda_device)).sum() + (C * gC.to(cuda_device)).sum()).backward()
    ga, ge, gd = oracle.look_at_backward(az.numpy(), el.numpy(), di.numpy(), gR.numpy(), gT.numpy(), gC.numpy())
    assert rel(a.grad, ga) < 1e-5 and rel(e.grad, ge) < 1e-5 and rel(d.grad, gd) < 1e-5


def test_camera_position_from_spherical_angles(oracle, cuda_device):
    """ViewGCN's graph vertices (Trainer_mvt.py:131-133) come from the same kernel as R and T."""
    az = torch.linspace(-180, 180, 13)[:-1].repeat(3, 1) - 90; el = torch.full((3, 12), 35.0); di = torch.full((3, 12), 2.2)
    d = di.to(cuda_device).requires_grad_()
    C = ops.camera_position_from_spherical_angles(d, el.to(cuda_device), az.to(cuda_device))
    _, _, Co = oracle.look_at(az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel())
    assert C.shape == (36, 3) and np.abs(C.detach().cpu().numpy() - Co).max() < 2e-6
    C.sum().backward()      # dC/d dist = C / dist
    assert torch.allclose(d.grad.reshape(-1).cpu(), torch.from_numpy(Co).sum(1) / 2.2, atol=1e-5)
    Cr = ops.camera_position_from_spherical_angles(di.to(cuda_device), torch.deg2rad(el).to(cuda_device),
                                                   torch.deg2rad(az).to(cuda_device), degrees=False)
    assert torch.allclose(Cr, C.detach(), atol=1e-5)


def test_rotation_guard_flag_matches_oracle(oracle, cuda_device):
    # nan / inf angles and zero distance give invalid matrices; the fused device check must count like util.py:403-420
    az = torch.tensor([0.0, 10.0, float("nan"), 30.0]); el = torch.tensor([0.0, 20.0, 0.0, 0.0]); di = torch.tensor([2.2, 0.0, 2.0, 2.0])
    R, T, C, bad = ops._LookAt.apply(az.to(cuda_device), el.to(cuda_device), di.to(cuda_device))
    Ro, _, _ = oracle.look_at(az.numpy(), el.numpy(), di.numpy())
    assert int(bad) == oracle.count_invalid_rotations(Ro) == 2


@pytest.mark.parametrize("n", [1, 300, 4096, 4097, 20000])
def test_rotation_flag_device_word_and_pinned_word_agree(cuda_device, n):
    """Up to 4096 views ONE CTA owns the count: no memset in front of the camera kernel, and with a FlagSink the kernel stores the
    count straight into the pinned host word (no copy behind it); above, the multi-CTA kernel + memset + copy.  Same cameras, same
    count, on the device word and on the host word, on both sides of the threshold and on repeated use of a pooled sink."""
    dev = cuda_device
    g = torch.Generator().manual_seed(n)
    az = torch.rand(n, generator=g) * 360 - 180; el = torch.rand(n, generator=g) * 160 - 80; di = torch.rand(n, generator=g) + 1.5
    bad_at = sorted(set(int(i) for i in torch.randint(0, n, (min(n, 5),), generator=g)))
    for k, i in enumerate(bad_at):
        if k % 2: di[i] = 0.0
        else: az[i] = float("nan")
    az, el, di = az.to(dev), el.to(dev), di.to(dev)
    a, e, d, R0, T0, C0, bad0 = ops._look_at_launch(az, el, di)
    assert int(bad0) == len(bad_at)
    for _ in range(3):
        sink = ops.FlagSink.get(dev)
        _, _, _, R1, T1, C1, bad1 = ops._look_at_launch(az, el, di, sink)
        assert sink.read() == len(bad_at) == int(bad1)
        assert torch.equal(R0.nan_to_num(7.0), R1.nan_to_num(7.0)) and torch.equal(T0.nan_to_num(7.0), T1.nan_to_num(7.0))
    # all-valid launch after an invalid one: the word is rewritten, not accumulated
    sink = ops.FlagSink.get(dev)
    ok = torch.ones(n, device=dev)
    ops._look_at_launch(ok * 30, ok * 20, ok * 2.2, sink)
    assert sink.read() == 0


# ------------------------------------------------------------------------------------------------- meshes
CUBE_V = torch.tensor([[-1, -1, -1], [1, -1, -1], [1, 1, -1], [-1, 1, -1], [-1, -1, 1], [1, -1, 1], [1, 1, 1], [-1, 1, 1]],
                      dtype=torch.float32) * 0.55
CUBE_F = torch.tensor([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [2, 3, 7], [2, 7, 6], [1, 2, 6], [1, 6, 5],
                       [0, 4, 7], [0, 7, 3]])


def mesh_case(name):
    if name == "small":
        return dict(meshes=synth.make_meshes(1, 300, 1), M=4, H=32, K=1, views=synth.circular_views(1, 4))
    if name == "spherical":
        return dict(meshes=synth.make_meshes(2, 2000, 2), M=4, H=64, K=1, views=synth.learned_spherical_views(2, 4, 9))
    if name == "ragged_k3":
        return dict(meshes=[synth.make_mesh(200, 4), synth.make_mesh(1200, 5), synth.make_mesh(60, 6)], M=2, H=50, K=3,
                    views=synth.learned_spherical_views(3, 2, 1))
    if name == "cube_big_faces":
        return dict(meshes=[(CUBE_V, CUBE_F)], M=4, H=96, K=2, views=synth.learned_spherical_views(1, 4, 3))
    if name == "cull_noperspective":
        return dict(meshes=synth.make_meshes(1, 800, 7), M=3, H=40, K=1, views=synth.learned_spherical_views(1, 3, 4), persp=False, cull=True)
    if name == "vertex_rgb":
        m = synth.make_meshes(1, 600, 8)
        return dict(meshes=m, M=3, H=48, K=1, views=synth.learned_spherical_views(1, 3, 5),
                    vert_rgb=torch.rand(m[0][0].shape[0], 3, generator=torch.Generator().manual_seed(1)))
    if name == "relative_light":
        return dict(meshes=synth.make_meshes(2, 500, 9), M=3, H=40, K=1, views=synth.learned_spherical_views(2, 3, 6), light="relative")
    if name == "close_camera_400":
        v = synth.learned_spherical_views(1, 2, 7)
        return dict(meshes=synth.make_meshes(1, 3000, 10), M=2, H=100, K=2, views=(v[0], v[1], v[2] * 0 + 1.25))
    if name == "c2_slice":
        return dict(meshes=synth.make_meshes(1, 10000, 12), M=2, H=224, K=1, views=synth.circular_views(1, 2))
    if name == "odd_width_k1":      # W % 4 != 0: the tile-per-CTA backward instead of the cp.async strip kernel; 97 px: partial tiles
        return dict(meshes=synth.make_meshes(2, 900, 14), M=3, H=97, K=1, views=synth.learned_spherical_views(2, 3, 11))
    if name == "c5_mesh_100k_400":  # BASELINE configs[4] shape: ~100k faces at 400x400 (two of the 20 spherical views; 3e10 oracle tests)
        return dict(meshes=synth.make_meshes(1, 100000, 15), M=2, H=400, K=1, views=tuple(t[:, 4:6].contiguous() for t in synth.spherical_views(1, 20)))
    if name == "dense_subpixel":
        return dict(meshes=synth.make_meshes(1, 20000, 13), M=2, H=64, K=1, views=synth.learned_spherical_views(1, 2, 8))
    raise KeyError(name)


MESH_CASES = ["small", "spherical", "ragged_k3", "cube_big_faces", "cull_noperspective", "vertex_rgb", "relative_light",
              "close_camera_400", "c2_slice", "dense_subpixel", "odd_width_k1", "c5_mesh_100k_400"]


def run_mesh(oracle, dev, cfg, backward=True, extra_flags=0):
    meshes, M, H, K = cfg["meshes"], cfg["M"], cfg["H"], cfg["K"]
    persp, cull = cfg.get("persp", True), cfg.get("cull", False)
    vert_rgb = cfg.get("vert_rgb")
    B = len(meshes)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev, vert_rgb=vert_rgb)
    R, T, C, (Rd, Td, Cd) = cams(oracle, cfg["views"], dev)
    light = C.copy() if cfg.get("light") == "relative" else np.array([cfg.get("light_dir", [0.3, 1.0, -0.5])], np.float32)
    obj = np.full(3, 0.99999, np.float32); bg = np.array([0.5, 0.25, 0.75], np.float32)
    Rg, Tg, Cg = (t.clone().requires_grad_() for t in (Rd, Td, Cd))
    flags_note = extra_flags
    img, frag = ops.render_meshes(geom, M, Rg, Tg, Cg, torch.from_numpy(light).to(dev), None if vert_rgb is not None else torch.from_numpy(obj).to(dev),
                                  torch.from_numpy(bg).to(dev), H, faces_per_pixel=K, cull_backfaces=cull, perspective_correct=persp,
                                  fragments=True, _extra_flags=flags_note, z_clip=cfg.get("z_clip"))
    vp, fp, voff, foff = pack_np(meshes)
    nrm = oracle.packed_vertex_normals(vp, fp, voff, foff)
    assert np.abs(geom.vertex_normals().cpu().numpy() - nrm).max() < 5e-7
    oflags = (oracle.PERSPECTIVE_CORRECT if persp else 0) | (oracle.CULL_BACKFACES if cull else 0)
    rgb = obj if vert_rgb is None else vert_rgb.numpy()
    z_clip = cfg.get("z_clip", 0.5 if persp else -1.0)
    o = oracle.mesh_forward(vp, fp, voff, foff, nrm, rgb, M, R, T, C, light, bg, K00, K11, z_clip, H, H, K, oflags)
    p2f = frag["pix_to_face"].cpu().numpy()
    res = dict(o=o, frag=frag, img=img, geom=geom, p2f=p2f)
    # exact depth ties inside a pixel's K-list (counted and reported, SURVEY 8d); they must still agree
    zb = o["zbuf"]
    res["ties"] = int(((zb[..., 1:] == zb[..., :-1]) & (o["pix_to_face"][..., 1:] >= 0)).sum()) if K > 1 else 0
    assert (p2f == o["pix_to_face"]).all(), f"{int((p2f != o['pix_to_face']).sum())} fragment index mismatches"
    assert (frag["zbuf"].cpu().numpy() == o["zbuf"]).all()
    assert (frag["bary_coords"].cpu().numpy() == o["bary"]).all()
    assert (frag["dists"].cpu().numpy() == o["dists"]).all()
    assert np.abs(img.detach().cpu().numpy() - o["images"]).max() <= IMG_ATOL
    assert int(frag["counters"][L.CNT_STRADDLE]) == o["straddle"]
    if backward:
        g = torch.randn(B * M, 3, H, H, generator=torch.Generator().manual_seed(5))
        img.backward(g.to(dev))
        ob = oracle.mesh_backward(vp, fp, voff, foff, nrm, rgb, M, R, T, C, light, K00, K11, H, H, K, oflags, p2f, g.numpy(), z_clip=z_clip)
        assert rel(Rg.grad, ob["gR"]) < GRAD_RTOL
        assert rel(Tg.grad, ob["gT"]) < GRAD_RTOL
        assert rel(Cg.grad, ob["gC"]) < GRAD_RTOL
    return res


@pytest.mark.parametrize("name", MESH_CASES)
def test_mesh_parity(oracle, cuda_device, name):
    res = run_mesh(oracle, cuda_device, mesh_case(name))
    cov = (res["p2f"][..., 0] >= 0).mean()
    assert 0.05 < cov <= 1.0
    print(f"[{name}] coverage {cov:.3f} exact-depth ties {res['ties']}")


def test_mesh_queue_overflow_fallbacks_are_exact(oracle, cuda_device):
    # 24-item / 5-candidate queues force the scatter kernel onto its in-place and whole-CTA fallbacks: same fragments
    for name in ("spherical", "cube_big_faces", "ragged_k3"):
        run_mesh(oracle, cuda_device, mesh_case(name), backward=False, extra_flags=L.TEST_TINY_QUEUES)


def test_mesh_forward_edge_cases_k1(oracle, cuda_device):
    """K = 1: a cube of faces spanning many pixels (walked by a whole CTA), near-plane clipping, a single triangle, a ragged batch
    and a non-square image.  (An object behind the camera at K = 1: test_mesh_edge_cases.)"""
    cube = dict(mesh_case("cube_big_faces"), K=1)
    res = run_mesh(oracle, cuda_device, cube, backward=False)
    assert int(res["frag"]["counters"][L.CNT_BIG_FACES]) > 0
    close = dict(mesh_case("close_camera_400"), K=1)
    res = run_mesh(oracle, cuda_device, close)
    assert res["o"]["straddle"] > 0
    tri_v = torch.tensor([[-0.5, -0.5, 0.0], [0.5, -0.5, 0.0], [0.0, 0.6, 0.0]]); tri_f = torch.tensor([[0, 1, 2]])
    run_mesh(oracle, cuda_device, dict(meshes=[(tri_v, tri_f)], M=2, H=33, K=1, views=(torch.tensor([[0.0, 40.0]]), torch.tensor([[10.0, 30.0]]),
                                       torch.tensor([[2.2, 2.0]])), light_dir=[0.3, 0.5, 0.8]), backward=False)
    run_mesh(oracle, cuda_device, dict(mesh_case("ragged_k3"), K=1))
    # non-square image
    dev = cuda_device
    H, W, M = 40, 104, 2
    meshes = synth.make_meshes(1, 700, 79)
    R, T, C, (Rd, Td, Cd) = cams(oracle, synth.learned_spherical_views(1, M, 6), dev)
    geom = ops.PackedMeshes([meshes[0][0]], [meshes[0][1]], dev)
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0.2, 1.0, 0.3]], device=dev)
    vp, fp, voff, foff = pack_np(meshes)
    o = oracle.mesh_forward(vp, fp, voff, foff, oracle.vertex_normals(vp, fp), np.full(3, 0.99999, np.float32), M, R, T, C,
                            np.array([[0.2, 1.0, 0.3]], np.float32), np.full(3, 0.499995, np.float32), K00, K11, 0.5, H, W, 1,
                            oracle.PERSPECTIVE_CORRECT)
    img, frag = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col * 0.5, (H, W), fragments=True)
    assert (frag["pix_to_face"].cpu().numpy() == o["pix_to_face"]).all() and (frag["zbuf"].cpu().numpy() == o["zbuf"]).all()
    assert np.abs(img.cpu().numpy() - o["images"]).max() <= IMG_ATOL


# ------------------------------------------------------------------------------------------------ soft shaders (8f N3)
SOFT_CASES = {
    "phong_default_blend": dict(faces=500, M=3, H=48, K=6, blur=9.2e-4, sigma=1e-4, gamma=1e-4, shader="soft_phong", seed=21),
    "phong_smooth_blend": dict(faces=300, M=2, H=40, K=8, blur=4e-3, sigma=2e-3, gamma=5e-2, shader="soft_phong", seed=22),
    "silhouette": dict(faces=400, M=3, H=56, K=12, blur=3e-3, sigma=1e-3, gamma=1e-4, shader="soft_silhouette", seed=23),
    "phong_no_clip": dict(faces=300, M=2, H=40, K=4, blur=2e-3, sigma=1e-3, gamma=1e-2, shader="soft_phong", seed=24, clip=False),
}


@pytest.mark.parametrize("name", list(SOFT_CASES))
def test_mesh_soft_shaders_match_the_torch_restatement(oracle, cuda_device, name):
    """blur_radius > 0, faces_per_pixel = K, SoftPhong / SoftSilhouette blending and their backward (grad_dists, grad_zbuf,
    clipped barycentrics) against oracle/torch_ref.py (the restatement of rasterize_meshes_cpu.cpp + blending.py; its forward is
    pinned to the C oracle at blur 0, its backward is autograd in fp64): fragment indices bit-exact, zbuf / bary / dists 1e-6,
    RGBA 1e-5 (5e-9 / gamma for sharper blends), camera gradients 1e-4 of the tensor's largest entry."""
    from oracle import torch_ref as tr
    c = SOFT_CASES[name]
    dev = cuda_device
    M, H, K = c["M"], c["H"], c["K"]
    v, f = synth.make_mesh(c["faces"], c["seed"])
    views = synth.learned_spherical_views(1, M, c["seed"] + 1)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    nrm = oracle.vertex_normals(v.numpy(), f.numpy())
    light = torch.tensor([[0.3, 1.0, -0.5]]); obj = torch.tensor([0.9, 0.7, 0.5]); bg = torch.tensor([0.5, 0.25, 0.75])
    geom = ops.PackedMeshes([v], [f], dev)
    Rg, Tg, Cg = (t.clone().requires_grad_() for t in (Rd, Td, Cd))
    clip = c.get("clip")
    img, frag = ops.render_meshes(geom, M, Rg, Tg, Cg, light.to(dev), obj.to(dev), bg.to(dev), H, faces_per_pixel=K, shader=c["shader"],
                                  blur_radius=c["blur"], sigma=c["sigma"], gamma=c["gamma"], clip_barycentric_coords=clip)
    assert img.shape == (M, 4, H, H)
    g = torch.randn(M, 4, H, H, generator=torch.Generator().manual_seed(5))
    img.backward(g.to(dev))
    p2f = frag["pix_to_face"].cpu()
    D = torch.float64
    Rr, Tr, Cr = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T, C))
    loss = 0
    n_out = 0
    for n in range(M):
        # forward reference in fp32 (fragments), backward reference in fp64 from the CUDA path's own fragment indices
        fv32 = torch.from_numpy(oracle.project_perspective(v.numpy(), R[n], T[n], K00, K11))[f]      # the oracle's IEEE projection
        rp2f, rz, rb, rd = tr.rasterize_meshes_soft(fv32, H, H, K, c["blur"], clip_bary=clip)
        assert (p2f[n].long() == rp2f).all(), f"view {n}: {int((p2f[n].long() != rp2f).sum())} fragment index mismatches"
        ok = rp2f >= 0
        n_out += int((rd[ok] > 0).sum())
        assert (frag["zbuf"][n].cpu() - rz).abs().max() <= 1e-6 and (frag["bary_coords"][n].cpu() - rb).abs().max() <= 2e-6
        assert (frag["dists"][n].cpu() - rd).abs().max() <= 1e-6
        ref, _ = tr.render_mesh_view_soft(v.to(D), f, torch.from_numpy(nrm).to(D), obj.to(D).expand(v.shape[0], 3), Rr[n], Tr[n], Cr[n],
                                          light[0].to(D), bg.to(D), K00, K11, H, H, K, c["blur"], c["shader"], sigma=c["sigma"],
                                          gamma=c["gamma"], clip_bary=clip, p2f=rp2f)
        # the blend weights are exp((z_inv - z_inv_max) / gamma): an fp32 ulp of z_inv (6e-8) is amplified by 1 / gamma, so against
        # the fp64 evaluation the fp32 image (PyTorch3D's included) is only good to ~5e-9 / gamma at BlendParams' default 1e-4
        img_tol = max(IMG_ATOL, 5e-9 / c["gamma"])
        assert (img[n].detach().cpu().to(D) - ref.detach()).abs().max() <= img_tol, (n, float((img[n].detach().cpu().to(D) - ref.detach()).abs().max()))
        loss = loss + (ref * g[n].to(D)).sum()
    assert n_out > 50                                   # fragments OUTSIDE their face (the blur) are really present
    loss.backward()
    assert rel(Rg.grad, Rr.grad.numpy()) < GRAD_RTOL and rel(Tg.grad, Tr.grad.numpy()) < GRAD_RTOL
    if c["shader"] == "soft_phong":
        assert rel(Cg.grad, Cr.grad.numpy()) < GRAD_RTOL
    else:
        assert float(Cg.grad.abs().max()) == 0.0


def test_mvrenderer_soft_shader_options(cuda_device):
    """MVRenderer(shader=..., blur_radius=..., faces_per_pixel=K): 3 channels as renderer.py:112 (4 with keep_alpha), gradients
    reach azim / elev / dist, the hard default is untouched."""
    dev = cuda_device
    M, S = 3, 48
    meshes = [Meshes([v], [f]) for v, f in synth.make_meshes(2, 400, 31)]
    az, el, di = (t.to(dev).requires_grad_() for t in synth.learned_spherical_views(2, M, 4))
    r = MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed", faces_per_pixel=6, shader="soft_silhouette",
                   blur_radius=2e-3, blend_sigma=1e-3, keep_alpha=True).to(dev)
    img, cams_ = r(meshes, None, az, el, di)
    assert img.shape == (2, M, 4, S, S) and 0.05 < float((img[:, :, 3] > 0.5).float().mean()) < 0.9
    img[:, :, 3].sum().backward()
    assert all(t.grad is not None and torch.isfinite(t.grad).all() and float(t.grad.abs().sum()) > 0 for t in (az, el, di))
    r3 = MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed", faces_per_pixel=4, shader="soft_phong", blur_radius=1e-3).to(dev)
    assert r3(meshes, None, az.detach(), el.detach(), di.detach())[0].shape == (2, M, 3, S, S)


def test_mesh_big_faces_take_the_cooperative_path(oracle, cuda_device):
    res = run_mesh(oracle, cuda_device, mesh_case("cube_big_faces"), backward=False)
    assert int(res["frag"]["counters"][L.CNT_BIG_FACES]) > 0


def test_mesh_duplicate_faces_tie_rule(oracle, cuda_device):
    v, f = synth.make_mesh(400, 3)
    f2 = torch.cat([f, f, f[:50]])                       # every face twice (some thrice): exact depth ties everywhere
    res = run_mesh(oracle, cuda_device, dict(meshes=[(v, f2)], M=3, H=48, K=3, views=synth.learned_spherical_views(1, 3, 2)), backward=False)
    assert res["ties"] > 100
    p = res["p2f"]
    hit = p[..., 1] >= 0
    assert (p[..., 0][hit] < p[..., 1][hit]).any()


def test_mesh_face_permutation_invariance(oracle, cuda_device):
    v, f = synth.make_mesh(1500, 21)
    views = synth.learned_spherical_views(1, 3, 4)
    perm = torch.randperm(f.shape[0], generator=torch.Generator().manual_seed(0))
    a = run_mesh(oracle, cuda_device, dict(meshes=[(v, f)], M=3, H=64, K=1, views=views), backward=False)
    b = run_mesh(oracle, cuda_device, dict(meshes=[(v, f[perm])], M=3, H=64, K=1, views=views), backward=False)
    pa, pb = a["p2f"][..., 0], b["p2f"][..., 0]
    assert ((pa >= 0) == (pb >= 0)).all()
    m = pa >= 0
    assert (perm.numpy()[pb[m]] == pa[m]).all()          # same winning face (no exact ties in this mesh)
    assert np.abs(a["img"].detach().cpu().numpy() - b["img"].detach().cpu().numpy()).max() <= 2e-6


def test_mesh_edge_cases(oracle, cuda_device):
    dev = cuda_device
    # single triangle facing the camera; and an object entirely behind the camera / off screen
    tri_v = torch.tensor([[-0.5, -0.5, 0.0], [0.5, -0.5, 0.0], [0.0, 0.6, 0.0]]); tri_f = torch.tensor([[0, 1, 2]])
    run_mesh(oracle, dev, dict(meshes=[(tri_v, tri_f)], M=2, H=33, K=2, views=(torch.tensor([[0.0, 40.0]]), torch.tensor([[10.0, 30.0]]), torch.tensor([[2.2, 2.0]])),
                           light_dir=[0.3, 0.5, 0.8]), backward=False)   # flat face, uniform normals: the true gradient is ~0
    far = tri_v + torch.tensor([0.0, 0.0, 50.0])
    res = run_mesh(oracle, dev, dict(meshes=[(far, tri_f)], M=1, H=16, K=1, views=(torch.tensor([[0.0]]), torch.tensor([[0.0]]), torch.tensor([[2.0]]))),
                   backward=False)
    assert (res["p2f"] == -1).all()
    # empty batch: a no-op, not an error
    geom = ops.PackedMeshes([], [], dev)
    z = torch.zeros(0, 3, device=dev)
    img, frag = ops.render_meshes(geom, 4, torch.zeros(0, 3, 3, device=dev), z, z, torch.tensor([[0, 1.0, 0]], device=dev),
                                  torch.ones(3, device=dev), torch.ones(3, device=dev), 32)
    assert img.shape == (0, 3, 32, 32)
    # camera/mesh count mismatch raises ValueError like upstream
    geom = ops.PackedMeshes([tri_v], [tri_f], dev)
    with pytest.raises(ValueError):
        ops.render_meshes(geom, 2, torch.zeros(3, 3, 3, device=dev), torch.zeros(3, 3, device=dev), torch.zeros(3, 3, device=dev),
                          torch.tensor([[0, 1.0, 0]], device=dev), torch.ones(3, device=dev), torch.ones(3, device=dev), 32)
    with pytest.raises(L.MVRError, match="faces_per_pixel"):
        Rd = torch.eye(3, device=dev)[None]
        ops.render_meshes(geom, 1, Rd, torch.tensor([[0, 0, 2.0]], device=dev), torch.tensor([[0, 0, 2.0]], device=dev),
                          torch.tensor([[0, 1.0, 0]], device=dev), torch.ones(3, device=dev), torch.ones(3, device=dev), 32, faces_per_pixel=100)


def test_mesh_near_plane_counters(oracle, cuda_device):
    # dist 1.1 with a unit-sphere object: faces cross z_clip = znear/2; they are culled / counted like the oracle
    m = synth.make_meshes(1, 2000, 31)
    v = (torch.tensor([[0.0, 90.0]]), torch.tensor([[0.0, 10.0]]), torch.tensor([[1.02, 1.05]]))
    res = run_mesh(oracle, cuda_device, dict(meshes=m, M=2, H=64, K=1, views=v), backward=False)
    assert res["o"]["straddle"] > 0


def _clipped_pixels(oracle, res, cfg, z_clip=0.5):
    """Pixels whose winning face crosses the near plane (recomputed from the oracle's projection)."""
    meshes, M = cfg["meshes"], cfg["M"]
    az, el, di = cfg["views"]
    R, T, _ = oracle.look_at(az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel())
    n_px = 0
    for b, (v, f) in enumerate(meshes):
        for m in range(M):
            n = b * M + m
            z = (v.numpy() @ R[n] + T[n])[:, 2][f.numpy()]              # (F,3) view depths
            strad = ((z < z_clip).sum(1) % 3) != 0
            p = res["p2f"][n, ..., 0]
            n_px += int(strad[p[p >= 0]].sum())
    return n_px


@pytest.mark.parametrize("variant", ["persp_k1", "persp_k2", "noperspective", "vertex_rgb_relative_light"])
def test_mesh_near_plane_clipping(oracle, cuda_device, variant):
    """Cameras 1.12 - 1.3 away from a unit-sphere object (mvtn.py:33 transform_distance reaches 1.1): faces crossing
    z = znear / 2 are clipped into one or two triangles ([upstream] clip.py) -- fragments bit-exact, images and camera
    gradients within the usual bars, for the pixels the clipped kernels own as for all the others."""
    m = synth.make_meshes(2, 1500, 61)
    views = (torch.tensor([[15.0, 140.0, -80.0], [200.0, 33.0, 77.0]]), torch.tensor([[10.0, -35.0, 50.0], [0.0, 20.0, -15.0]]),
             torch.tensor([[1.12, 1.2, 1.3], [1.15, 1.25, 1.18]]))
    cfg = dict(meshes=m, M=3, H=72, K=1, views=views)
    if variant == "persp_k2":
        cfg["K"] = 2
    if variant == "noperspective":
        cfg.update(persp=False, z_clip=0.5)
    if variant == "vertex_rgb_relative_light":
        cfg.update(meshes=m[:1], views=tuple(t[:1] for t in views), light="relative",
                   vert_rgb=torch.rand(m[0][0].shape[0], 3, generator=torch.Generator().manual_seed(3)))
    res = run_mesh(oracle, cuda_device, cfg)
    assert res["o"]["straddle"] > 0
    assert _clipped_pixels(oracle, res, cfg) > 200
    zb = res["o"]["zbuf"][res["o"]["pix_to_face"] >= 0]
    assert float(zb.min()) >= 0.5 - 1e-5      # nothing nearer than the plane survives


def test_mesh_clipping_vertex_gradients(oracle, cuda_device):
    from oracle import torch_ref as tr
    dev = cuda_device
    v, f = synth.make_mesh(400, 15)
    M, H = 3, 48
    views = (torch.tensor([[15.0, 140.0, -80.0]]), torch.tensor([[10.0, -35.0, 50.0]]), torch.tensor([[1.15, 1.22, 1.3]]))
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    vg = v.to(dev).requires_grad_()
    geom = ops.PackedMeshes.from_packed(vg.detach(), f.to(dev), [v.shape[0]], [f.shape[0]])
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0.3, 1.0, -0.5]], device=dev)
    img, frag = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col, H, verts=vg)
    assert int(frag["counters"][L.CNT_STRADDLE]) > 0
    g = torch.randn(M, 3, H, H, generator=torch.Generator().manual_seed(4))
    p2f = frag["pix_to_face"].cpu().numpy()
    D = torch.float64
    vd = v.to(D).requires_grad_()
    nd = tr.vertex_normals(vd, f)
    loss = 0
    for n in range(M):
        im, p2 = tr.render_mesh_view(vd, f, nd, torch.full((v.shape[0], 3), 0.99999, dtype=D), torch.from_numpy(R[n]).to(D), torch.from_numpy(T[n]).to(D),
                                     torch.from_numpy(C[n]).to(D), torch.tensor([0.3, 1.0, -0.5], dtype=D), torch.full((3,), 0.99999, dtype=D), K00, K11, H, H,
                                     z_clip=0.5)
        same = torch.from_numpy(p2f[n, ..., 0]).long() == p2       # fp64 restatement: drop pixels a rounding error away from an edge
        assert int((~same).sum()) <= 2
        g[n] *= same[None]
        loss = loss + (im * g[n].to(D)).sum()
    img.backward(g.to(dev))
    loss.backward()
    assert rel(vg.grad, vd.grad.numpy()) < 5e-4


def test_mesh_workspace_reuse_hints_are_exact(oracle, cuda_device):
    """The mesh path remembers what it left in its workspace (ops._ws_mesh): a forward after a same-layout forward skips
    the key-plane memset (the shade pass re-armed the plane, clipped pixels included), and a backward right after its
    forward skips the re-projection.  Results must be those of a cold workspace, bit for bit -- across changing views,
    layer peeling, near-plane clipping, out-of-order backwards and another renderer using the buffer."""
    dev = cuda_device
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0, 1.0, 0]], device=dev)
    key = (dev.index, ops._stream(dev))

    def render(geom, M, views, H, K, fragments):
        az, el, di = (t.to(dev).reshape(-1).requires_grad_() for t in views)
        R, T, C, _ = ops._LookAt.apply(az, el, di)
        img, fr = ops.render_meshes(geom, M, R, T, C, light, col, col, H, faces_per_pixel=K, fragments=fragments)
        return img, fr, (az, el, di)

    m = synth.make_meshes(2, 1500, 61)
    geom = ops.PackedMeshes([v for v, _ in m], [f for _, f in m], dev)
    far = (torch.tensor([[15.0, 140.0, -80.0], [200.0, 33.0, 77.0]]), torch.tensor([[10.0, -35.0, 50.0], [0.0, 20.0, -15.0]]),
           torch.tensor([[2.2, 2.0, 2.5], [1.9, 2.25, 3.0]]))
    near = (far[0] + 30.0, far[1], torch.tensor([[1.12, 1.2, 1.3], [1.15, 1.25, 1.18]]))      # faces cross the near plane
    armed_hits = 0
    for K in (1, 2):
        for H in (72, 40):
            for fragments in (True, False):
                ref = {}
                for name, views in (("far", far), ("near", near)):
                    ops._ws_mesh.pop(key, None)
                    img, fr, _ = render(geom, 3, views, H, K, fragments)
                    ref[name] = (img.clone(), {k: v.clone() for k, v in fr.items() if k != "counters"})
                if fragments:
                    assert int(fr["counters"][L.CNT_STRADDLE]) > 0
                ops._ws_mesh.pop(key, None)
                for i, name in enumerate(["far", "near", "near", "far", "far", "near"]):
                    st = ops._ws_mesh.get(key)
                    armed_hits += st is not None and st["armed"] is not None
                    img, fr, _ = render(geom, 3, far if name == "far" else near, H, K, fragments)
                    assert torch.equal(img, ref[name][0]), (K, H, i, name)
                    for k, v in ref[name][1].items():
                        assert torch.equal(fr[k], v), (K, H, i, name, k)
                    if i == 2:      # another user of the buffer: the hints must be dropped, not trusted
                        pts = torch.rand(2, 256, 3, device=dev) - 0.5
                        R, T, C, _ = ops._LookAt.apply(*(t.to(dev).reshape(-1) for t in far))
                        ops.render_points(pts, col, 3, R, T, None, 0.02, col * 0, H, dist=far[2].to(dev).reshape(-1))
                        assert ops._ws_mesh.get(key) is None
    assert armed_hits >= 8 * 4
    # gradients: warm (projection reused) == cold (re-projected), also when the backwards run out of order
    cot = torch.randn(6, 3, 72, 72, device=dev, generator=torch.Generator(device=dev).manual_seed(5))

    def grads(views, warm):
        if not warm:
            ops._ws_mesh.pop(key, None)
        img, _, leaves = render(geom, 3, views, 72, 1, False)
        if not warm:
            ops._ws_mesh.pop(key, None)
        else:
            assert ops._ws_mesh[key]["proj"] is not None
        img.backward(cot)
        return [t.grad.clone() for t in leaves]

    for views in (far, near):
        for a, b in zip(grads(views, False), grads(views, True)):
            assert torch.equal(a, b)
    img_a, _, la = render(geom, 3, far, 72, 1, False)
    img_b, _, lb = render(geom, 3, near, 72, 1, False)
    img_a.backward(cot)      # a's projection was overwritten by b's forward: a re-projects, which in turn invalidates b's
    assert ops._ws_mesh[key]["proj"] is None
    img_b.backward(cot)
    for a, b in zip(grads(far, False), [t.grad for t in la]):
        assert torch.equal(a, b)
    for a, b in zip(grads(near, False), [t.grad for t in lb]):
        assert torch.equal(a, b)


def test_mesh_golden_slice(cuda_device):
    g = np.load(os.path.join(GOLDEN, "mesh_c2_slice.npz"))
    dev = cuda_device
    geom = ops.PackedMeshes([torch.from_numpy(g["verts"])], [torch.from_numpy(g["faces"])], dev)
    R, T, C = (torch.from_numpy(g[k]).to(dev) for k in ("R", "T", "C"))
    col = torch.full((3,), 0.99999, device=dev)
    img, frag = ops.render_meshes(geom, 12, R, T, C, torch.tensor([[0, 1.0, 0]], device=dev), col, col, 224, fragments=True)
    assert sha(frag["pix_to_face"].cpu().numpy()) == str(g["p2f_sha256"])
    assert sha(frag["zbuf"].cpu().numpy()) == str(g["zbuf_sha256"])
    assert sha(frag["bary_coords"].cpu().numpy()) == str(g["bary_sha256"])
    assert ((frag["pix_to_face"][..., 0] >= 0).sum(dim=(1, 2)).cpu().numpy() == g["covered"]).all()
    assert np.abs(img.cpu().numpy()[:, :, ::16, ::16] - g["image_probe"]).max() <= IMG_ATOL
    assert np.allclose(img.double().sum(dim=(1, 2, 3)).cpu().numpy(), g["image_sum"], rtol=1e-6)


def test_mesh_golden_clip(cuda_device):
    """Committed golden of a close-up scene with 238 faces crossing the near plane (tests/golden/make_golden.py)."""
    g = np.load(os.path.join(GOLDEN, "mesh_clip.npz"))
    dev = cuda_device
    geom = ops.PackedMeshes([torch.from_numpy(g["verts"])], [torch.from_numpy(g["faces"])], dev)
    R, T, C = (torch.from_numpy(g[k]).to(dev) for k in ("R", "T", "C"))
    col = torch.full((3,), 0.99999, device=dev)
    img, frag = ops.render_meshes(geom, 3, R, T, C, torch.tensor([[0, 1.0, 0]], device=dev), col, col, 96, faces_per_pixel=2, fragments=True)
    assert int(frag["counters"][L.CNT_STRADDLE]) == int(g["straddle"])
    assert sha(frag["pix_to_face"].cpu().numpy()) == str(g["p2f_sha256"])
    assert sha(frag["zbuf"].cpu().numpy()) == str(g["zbuf_sha256"])
    assert sha(frag["bary_coords"].cpu().numpy()) == str(g["bary_sha256"])
    assert sha(frag["dists"].cpu().numpy()) == str(g["dists_sha256"])
    assert np.abs(img.cpu().numpy()[:, :, ::8, ::8] - g["image_probe"]).max() <= IMG_ATOL


def test_mesh_full_size_c2_properties(oracle, cuda_device):
    """BASELINE configs[1] at full size (32 x 12 views, ~10k faces, 224^2): size-independent properties +
    the oracle on two sampled objects."""
    dev = cuda_device
    B, M, H = 32, 12, 224
    meshes = synth.make_meshes(B, 10000, 1236)
    views = synth.learned_spherical_views(B, M, 17)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0, 1.0, 0]], device=dev)
    img1, f1 = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col, H)
    img2, f2 = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col, H)
    assert torch.equal(f1["pix_to_face"], f2["pix_to_face"]) and torch.equal(img1, img2)          # run-to-run determinism
    for b in (0, 19):                                                                              # object independence + oracle
        gb = ops.PackedMeshes([meshes[b][0]], [meshes[b][1]], dev)
        s = slice(b * M, (b + 1) * M)
        imgb, fb = ops.render_meshes(gb, M, Rd[s], Td[s], Cd[s], light, col, col, H)
        assert torch.equal(fb["pix_to_face"], f1["pix_to_face"][s]) and torch.equal(imgb, img1[s])
        vp, fp, voff, foff = pack_np([meshes[b]])
        o = oracle.mesh_forward(vp, fp, voff, foff, oracle.vertex_normals(vp, fp), np.full(3, 0.99999, np.float32), M, R[s], T[s], C[s],
                                np.array([[0, 1.0, 0]], np.float32), np.full(3, 0.99999, np.float32), K00, K11, 0.5, H, H, 1,
                                oracle.PERSPECTIVE_CORRECT, fragments=False)
        assert (fb["pix_to_face"].cpu().numpy() == o["pix_to_face"]).all()
        assert np.abs(imgb.cpu().numpy() - o["images"]).max() <= IMG_ATOL
    # backward determinism (fixed-order reductions, no float atomics on this path)
    g = torch.randn(B * M, 3, H, H, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    grads = []
    for _ in range(2):
        Rg, Tg, Cg = (t.clone().requires_grad_() for t in (Rd, Td, Cd))
        im, _ = ops.render_meshes(geom, M, Rg, Tg, Cg, light, col, col, H)
        im.backward(g)
        grads.append((Rg.grad, Tg.grad, Cg.grad))
    assert all(torch.equal(a, b) for a, b in zip(*grads))


# ------------------------------------------------------------------------------------------------- points
POINT_CASES = {
    "c1_k1_norm": dict(B=1, Np=2048, M=3, H=224, K=1, radius=0.006, mode="norm", views=synth.circular_views(1, 3)),
    "k4_alpha_rgb": dict(B=2, Np=500, M=3, H=64, K=4, radius=0.05, mode="alpha", views=synth.learned_spherical_views(2, 3, 2), per_point=True),
    "k3_norm_rgb": dict(B=2, Np=300, M=2, H=50, K=3, radius=0.04, mode="norm", views=synth.learned_spherical_views(2, 2, 3), per_point=True),
    "k1_alpha": dict(B=1, Np=1000, M=2, H=100, K=1, radius=0.02, mode="alpha", views=synth.circular_views(1, 2)),
    "k8_big_radius": dict(B=1, Np=400, M=2, H=40, K=8, radius=0.15, mode="alpha", views=synth.learned_spherical_views(1, 2, 5), per_point=True),
    "c5_16k_400_k4_alpha": dict(B=1, Np=16384, M=2, H=400, K=4, radius=0.006, mode="alpha", views=tuple(t[:, 7:9].contiguous() for t in synth.spherical_views(1, 20))),
    "c5_16k_400": dict(B=1, Np=16384, M=2, H=400, K=1, radius=0.006, mode="norm", views=tuple(t[:, 4:6].contiguous() for t in synth.spherical_views(1, 20))),
}


def run_points(oracle, dev, cfg, backward=True, pts=None):
    B, Np, M, H, K, radius, mode = (cfg[k] for k in ("B", "Np", "M", "H", "K", "radius", "mode"))
    pts = synth.make_clouds(B, Np, 11) if pts is None else pts
    R, T, C, (Rd, Td, Cd) = cams(oracle, cfg["views"], dev)
    inv = (1.0 / cfg["views"][2].reshape(-1)).contiguous()
    rgb = torch.rand(B, Np, 3, generator=torch.Generator().manual_seed(3)) if cfg.get("per_point") else torch.full((3,), 0.99999)
    bg = torch.tensor([0.1, 0.2, 0.3])
    Rg, Tg = Rd.clone().requires_grad_(), Td.clone().requires_grad_()
    sg, pg, fg = inv.to(dev).requires_grad_(), pts.to(dev).requires_grad_(), rgb.to(dev).requires_grad_()
    img, frag = ops.render_points(pg, fg, M, Rg, Tg, sg, radius, bg.to(dev), H, points_per_pixel=K, compositor=mode, fragments=True)
    flags = oracle.COMPOSITE_ALPHA if mode == "alpha" else 0
    o = oracle.points_forward(pts.numpy(), rgb.numpy(), M, R, T, inv.numpy(), radius, bg.numpy(), H, H, K, flags)
    idx = frag["idx"].cpu().numpy()
    assert (idx == o["idx"]).all(), f"{int((idx != o['idx']).sum())} point index mismatches"
    assert (frag["zbuf"].cpu().numpy() == o["zbuf"]).all()
    assert (frag["dists"].cpu().numpy() == o["dists2"]).all()
    assert np.abs(img.detach().cpu().numpy() - o["images"]).max() <= IMG_ATOL
    if backward:
        g = torch.randn(B * M, 3, H, H, generator=torch.Generator().manual_seed(6))
        img.backward(g.to(dev))
        ob = oracle.points_backward(pts.numpy(), rgb.numpy(), M, R, T, inv.numpy(), radius, H, H, K, flags, idx, g.numpy(),
                                    want_points=True, want_rgb=True)
        assert rel(Rg.grad, ob["gR"]) < POINT_GRAD_RTOL
        assert rel(Tg.grad, ob["gT"]) < POINT_GRAD_RTOL
        assert rel(sg.grad, ob["g_inv_dist"]) < POINT_GRAD_RTOL
        assert rel(pg.grad, ob["grad_points"]) < POINT_GRAD_RTOL
        assert rel(fg.grad, ob["grad_rgb"]) < POINT_GRAD_RTOL
    return dict(o=o, idx=idx, img=img)


@pytest.mark.parametrize("name", list(POINT_CASES))
def test_points_parity(oracle, cuda_device, name):
    res = run_points(oracle, cuda_device, POINT_CASES[name])
    assert (res["idx"][..., 0] >= 0).mean() > 0.005


def test_points_duplicates_and_behind_camera(oracle, cuda_device):
    pts = synth.make_clouds(1, 300, 4)
    pts = torch.cat([pts, pts[:, :100]], dim=1)                 # 100 exact duplicates: (z, idx) ties
    cfg = dict(B=1, Np=400, M=2, H=48, K=3, radius=0.06, mode="alpha", views=synth.learned_spherical_views(1, 2, 6))
    res = run_points(oracle, cuda_device, cfg, pts=pts)
    zb = res["o"]["zbuf"]
    assert ((zb[..., 1:] == zb[..., :-1]) & (res["idx"][..., 1:] >= 0)).sum() > 10
    # a cloud entirely behind the camera renders pure background
    far = pts * 0.01 + torch.tensor([0.0, 0.0, 10.0])
    cfg2 = dict(B=1, Np=400, M=1, H=32, K=2, radius=0.06, mode="norm", views=(torch.tensor([[0.0]]), torch.tensor([[0.0]]), torch.tensor([[2.0]])))
    res = run_points(oracle, cuda_device, cfg2, backward=False, pts=far)
    assert (res["idx"] == -1).all()
    assert np.allclose(res["img"].detach().cpu().numpy()[0, :, 3, 3], [0.1, 0.2, 0.3])


def test_points_golden(cuda_device):
    g = np.load(os.path.join(GOLDEN, "points_c1.npz"))
    dev = cuda_device
    pts = torch.from_numpy(g["points"]).to(dev)
    R, T, inv = (torch.from_numpy(g[k]).to(dev) for k in ("R", "T", "inv_dist"))
    col = torch.full((3,), 0.99999, device=dev)
    img, frag = ops.render_points(pts, col, 12, R, T, inv, 0.006, torch.zeros(3, device=dev), 224, fragments=True)
    assert sha(frag["idx"].cpu().numpy()) == str(g["idx_sha256"])
    assert sha(frag["zbuf"].cpu().numpy()) == str(g["zbuf_sha256"])
    assert sha(frag["dists"].cpu().numpy()) == str(g["d2_sha256"])
    assert np.allclose(img.double().sum(dim=(1, 2, 3)).cpu().numpy(), g["image_sum"], rtol=1e-6)
    img4, frag4 = ops.render_points(pts, col, 12, R, T, inv, 0.02, torch.zeros(3, device=dev), 224, points_per_pixel=4, compositor="alpha")
    assert sha(frag4["idx"].cpu().numpy()) == str(g["idx4_sha256"])
    assert np.allclose(img4.double().sum(dim=(1, 2, 3)).cpu().numpy(), g["image4_sum"], rtol=1e-5)


def test_mesh_full_size_c5_properties(oracle, cuda_device):
    """BASELINE configs[4] at full size (8 meshes x 20 views, ~100k faces, 400^2): properties that need no O(H W F) oracle pass --
    run-to-run determinism, object independence (an object rendered alone gives the slice of the batch: no cross-object term),
    invariance of the image under a permutation of the faces (ids map through the permutation), determinism of the backward.
    The oracle itself is run at this shape by test_mesh_parity[c5_mesh_100k_400] (two views) and by bench.py's parity gate."""
    dev = cuda_device
    B, M, H = 8, 20, 400
    meshes = synth.make_meshes(B, 100000, 1290)
    views = synth.spherical_views(B, M)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0, 1.0, 0]], device=dev)
    img1, f1 = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col, H)
    img2, f2 = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col, H)
    assert torch.equal(f1["pix_to_face"], f2["pix_to_face"]) and torch.equal(img1, img2)
    cov = float((f1["pix_to_face"] >= 0).float().mean())
    assert 0.2 < cov < 0.8
    b = 5
    s = slice(b * M, (b + 1) * M)
    gb = ops.PackedMeshes([meshes[b][0]], [meshes[b][1]], dev)
    imgb, fb = ops.render_meshes(gb, M, Rd[s], Td[s], Cd[s], light, col, col, H)
    assert torch.equal(fb["pix_to_face"], f1["pix_to_face"][s]) and torch.equal(imgb, img1[s])
    perm = torch.randperm(meshes[b][1].shape[0], generator=torch.Generator().manual_seed(3))
    gp = ops.PackedMeshes([meshes[b][0]], [meshes[b][1][perm]], dev)
    imgp, fpm = ops.render_meshes(gp, M, Rd[s], Td[s], Cd[s], light, col, col, H)
    ids = fpm["pix_to_face"][..., 0].long()
    mapped = torch.where(ids >= 0, perm.to(dev)[ids.clamp_min(0)], ids)
    same = mapped == fb["pix_to_face"][..., 0].long()
    # exact depth ties between two faces are resolved by the smaller index, which a permutation may change: count them
    assert float((~same).float().mean()) < 1e-4
    assert float(((imgp - imgb).abs() > 1e-5).float().mean()) < 1e-4
    g = torch.randn(B * M, 3, H, H, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    grads = []
    for _ in range(2):
        Rg, Tg, Cg = (t.clone().requires_grad_() for t in (Rd, Td, Cd))
        im, _ = ops.render_meshes(geom, M, Rg, Tg, Cg, light, col, col, H)
        im.backward(g)
        grads.append((Rg.grad, Tg.grad, Cg.grad))
    assert all(torch.equal(a_, b_) for a_, b_ in zip(*grads))


def test_points_full_size_c5_properties(oracle, cuda_device):
    """BASELINE configs[4] at full size (8 clouds x 20 views, 16384 points, 400^2, alpha K = 4): determinism, object independence,
    invariance under a permutation of the points (indices map through it), sorted layers; two views of one object against the
    oracle."""
    dev = cuda_device
    B, M, H, K = 8, 20, 400, 4
    pts = synth.make_clouds(B, 16384, 1291)
    views = synth.spherical_views(B, M)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    inv = (1.0 / views[2].reshape(-1)).to(dev)
    col = torch.full((3,), 0.99999, device=dev); bg = torch.zeros(3, device=dev)
    a = ops.render_points(pts.to(dev), col, M, Rd, Td, inv, 0.006, bg, H, points_per_pixel=K, compositor="alpha")
    b = ops.render_points(pts.to(dev), col, M, Rd, Td, inv, 0.006, bg, H, points_per_pixel=K, compositor="alpha")
    assert torch.equal(a[1]["idx"], b[1]["idx"]) and torch.equal(a[0], b[0])
    ob_ = 6
    s = slice(ob_ * M, (ob_ + 1) * M)
    im, fr = ops.render_points(pts[ob_:ob_ + 1].to(dev), col, M, Rd[s], Td[s], inv[s], 0.006, bg, H, points_per_pixel=K, compositor="alpha")
    assert torch.equal(fr["idx"], a[1]["idx"][s]) and torch.equal(im, a[0][s])
    perm = torch.randperm(16384, generator=torch.Generator().manual_seed(4))
    imp, frp = ops.render_points(pts[ob_:ob_ + 1][:, perm].to(dev), col, M, Rd[s], Td[s], inv[s], 0.006, bg, H, points_per_pixel=K, compositor="alpha")
    ids = frp["idx"].long()
    mapped = torch.where(ids >= 0, perm.to(dev)[ids.clamp_min(0)], ids)
    assert float((mapped != fr["idx"].long()).float().mean()) < 1e-4                  # (exact depth ties may swap)
    o = oracle.points_forward(pts[ob_:ob_ + 1].numpy(), np.full(3, 0.99999, np.float32), 2, R[s][:2], T[s][:2], inv[s][:2].cpu().numpy(), 0.006,
                              np.zeros(3, np.float32), H, H, K, oracle.COMPOSITE_ALPHA, fragments=False)
    assert (fr["idx"][:2].cpu().numpy() == o["idx"]).all() and np.abs(im[:2].cpu().numpy() - o["images"]).max() <= IMG_ATOL
    idx = a[1]["idx"]
    assert ((idx[..., 1:] != idx[..., :-1]) | (idx[..., 1:] < 0)).all()


def test_points_full_size_c3_properties(oracle, cuda_device):
    """BASELINE configs[2] at full size: 32 clouds x 12 learned_spherical views, alpha compositing, K=4."""
    dev = cuda_device
    B, M, H, K = 32, 12, 224, 4
    pts = synth.make_clouds(B, 2048, 1237)
    views = synth.learned_spherical_views(B, M, 23)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    inv = (1.0 / views[2].reshape(-1)).to(dev)
    col = torch.full((3,), 0.99999, device=dev); bg = torch.zeros(3, device=dev)
    a = ops.render_points(pts.to(dev), col, M, Rd, Td, inv, 0.006, bg, H, points_per_pixel=K, compositor="alpha")
    b = ops.render_points(pts.to(dev), col, M, Rd, Td, inv, 0.006, bg, H, points_per_pixel=K, compositor="alpha")
    assert torch.equal(a[1]["idx"], b[1]["idx"]) and torch.equal(a[0], b[0])
    for ob_ in (3, 30):
        s = slice(ob_ * M, (ob_ + 1) * M)
        im, fr = ops.render_points(pts[ob_:ob_ + 1].to(dev), col, M, Rd[s], Td[s], inv[s], 0.006, bg, H, points_per_pixel=K, compositor="alpha")
        assert torch.equal(fr["idx"], a[1]["idx"][s]) and torch.equal(im, a[0][s])
        o = oracle.points_forward(pts[ob_:ob_ + 1].numpy(), np.full(3, 0.99999, np.float32), M, R[s], T[s], inv[s].cpu().numpy(), 0.006,
                                  np.zeros(3, np.float32), H, H, K, oracle.COMPOSITE_ALPHA, fragments=False)
        assert (fr["idx"].cpu().numpy() == o["idx"]).all()
        assert np.abs(im.cpu().numpy() - o["images"]).max() <= IMG_ATOL
    # layers are sorted by depth and never repeat a point
    idx = a[1]["idx"]
    assert ((idx[..., 1:] != idx[..., :-1]) | (idx[..., 1:] < 0)).all()


def test_points_empty_cloud_and_tile_edges(oracle, cuda_device):
    """Zero points render pure background (tiled path with empty lists); a cloud concentrated on tile borders
    (x, y = multiples of 32 pixels) exercises points whose window straddles 2 or 4 tiles."""
    dev = cuda_device
    bg = torch.tensor([0.3, 0.6, 0.9], device=dev); col = torch.full((3,), 0.8, device=dev)
    R, T, C, (Rd, Td, Cd) = cams(oracle, (torch.tensor([[0.0, 40.0]]), torch.tensor([[0.0, 10.0]]), torch.tensor([[2.0, 2.0]])), dev)
    inv = torch.full((2,), 0.5, device=dev)
    img, fr = ops.render_points(torch.zeros(1, 0, 3, device=dev), col, 2, Rd, Td, inv, 0.02, bg, 70, points_per_pixel=4, compositor="alpha")
    assert (fr["idx"] == -1).all() and torch.allclose(img[0, :, 5, 5], bg)
    # points on a lattice whose projections fall near tile borders of a 96x96 image (3x3 tiles), large radius
    g = torch.linspace(-0.9, 0.9, 19)
    pts = torch.stack(torch.meshgrid(g, g, indexing="ij"), -1).reshape(1, -1, 2)
    pts = torch.cat([pts, 0.05 * torch.randn(1, pts.shape[1], 1, generator=torch.Generator().manual_seed(2))], -1)
    cfg = dict(B=1, Np=pts.shape[1], M=2, H=96, K=4, radius=0.09, mode="alpha",
               views=(torch.tensor([[0.0, 3.0]]), torch.tensor([[0.0, 2.0]]), torch.tensor([[2.0, 2.0]])))
    res = run_points(oracle, dev, cfg, pts=pts)
    assert (res["idx"][..., 3] >= 0).sum() > 100          # deep layers are populated across tile borders


def test_points_backward_without_hit_mask_matches(oracle, cuda_device):
    """The hit mask is an optional accelerator: mvr_points_backward(hit_mask=NULL) rebuilds the covered-pixel words
    from idx[..., 0] and must return the same partial sums bit for bit."""
    from mvtn_b200 import _lib as L
    dev = cuda_device
    B, Np, M, H, W, K = 2, 700, 3, 45, 70, 3          # W not a multiple of 32, H not a multiple of 32
    pts = synth.make_clouds(B, Np, 21).to(dev)
    R, T, C, (Rd, Td, Cd) = cams(oracle, synth.learned_spherical_views(B, M, 11), dev)
    inv = torch.full((B * M,), 1 / 1.5, device=dev)
    col = torch.full((3,), 0.9, device=dev)
    img, frag = ops.render_points(pts, col, M, Rd, Td, inv, 0.05, torch.zeros(3, device=dev), (H, W), points_per_pixel=K, compositor="alpha")
    idx = frag["idx"]
    g = torch.randn(B * M, 3, H, W, device=dev)
    lib = L.load()
    outs = []
    nwords = lib.mvr_points_hit_mask_words(B, M, H, W)
    assert nwords == B * M * H * ((W + 31) // 32)
    mask = torch.zeros(nwords, dtype=torch.int32, device=dev)
    covered = (idx[..., 0] >= 0)
    # rebuild the mask on the host and compare it with what the forward wrote (bit x%32 of word x/32)
    img2 = torch.empty_like(img); idx2 = torch.empty_like(idx)
    ws = ops.workspace(dev, lib.mvr_points_workspace_bytes(B, Np, M, H, W, K, 0.05))
    L.check(lib.mvr_points_forward(pts.data_ptr(), col.data_ptr(), B, Np, M, Rd.data_ptr(), Td.data_ptr(), inv.data_ptr(), 0.05,
                                   torch.zeros(3, device=dev).data_ptr(), H, W, K, L.COMPOSITE_ALPHA, None, img2.data_ptr(), idx2.data_ptr(),
                                   None, None, mask.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream), "fwd")
    assert torch.equal(idx2, idx) and torch.equal(img2, img)
    words = (W + 31) // 32
    cov = torch.zeros(B * M, H, words * 32, dtype=torch.bool, device=dev); cov[:, :, :W] = covered
    weights = (2 ** torch.arange(32, device=dev, dtype=torch.int64))
    expect = (cov.view(B * M, H, words, 32).to(torch.int64) * weights).sum(-1)
    got = mask.view(B * M, H, words).to(torch.int64) & 0xFFFFFFFF
    assert torch.equal(expect, got)
    for m_ptr in (mask.data_ptr(), None):
        gR = torch.empty(B * M, 3, 3, device=dev); gT = torch.empty(B * M, 3, device=dev); gs = torch.empty(B * M, device=dev)
        L.check(lib.mvr_points_backward(pts.data_ptr(), col.data_ptr(), B, Np, M, Rd.data_ptr(), Td.data_ptr(), inv.data_ptr(), 0.05, H, W, K,
                                        L.COMPOSITE_ALPHA, None, idx.data_ptr(), m_ptr, g.data_ptr(), gR.data_ptr(), gT.data_ptr(), gs.data_ptr(),
                                        None, None, ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream), "bwd")
        outs.append((gR, gT, gs))
    assert all(torch.equal(a, b) for a, b in zip(*outs))
    assert float(outs[0][0].abs().max()) > 0


def test_mesh_fast_shading_path_matches_exact(oracle, cuda_device):
    """fragments=False shades with two SFU reciprocals instead of six IEEE divisions: same pix_to_face, images within
    the 1e-5 bar of the oracle and a few 1e-6 of the exact path."""
    dev = cuda_device
    meshes = synth.make_meshes(2, 4000, 31)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    M, H = 4, 96
    R, T, C, (Rd, Td, Cd) = cams(oracle, synth.learned_spherical_views(2, M, 12), dev)
    light = torch.tensor([[0.3, 1.0, -0.5]], device=dev); col = torch.full((3,), 0.99999, device=dev); bg = torch.tensor([0.5, 0.25, 0.75], device=dev)
    img_e, fr_e = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, bg, H, fragments=True)
    img_f, fr_f = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, bg, H, fragments=False)
    assert torch.equal(fr_e["pix_to_face"], fr_f["pix_to_face"])
    assert float((img_e - img_f).abs().max()) <= 5e-6
    vp = torch.cat([v for v, _ in meshes]).numpy(); fp = torch.cat([f for _, f in meshes]).numpy().astype(np.int32)
    voff = np.array(geom.vert_off_host, np.int32); foff = np.array(geom.face_off_host, np.int32)
    o = oracle.mesh_forward(vp, fp, voff, foff, oracle.packed_vertex_normals(vp, fp, voff, foff), col.cpu().numpy(), M, R, T, C,
                            light.cpu().numpy(), bg.cpu().numpy(), K00, K11, 0.5, H, H, 1, oracle.PERSPECTIVE_CORRECT, fragments=False)
    assert np.abs(img_f.cpu().numpy() - o["images"]).max() <= IMG_ATOL


# ------------------------------------------------------------------------------------------ public API end-to-end
def test_mvrenderer_mesh_end_to_end(oracle, cuda_device):
    dev = cuda_device
    B, M, S = 3, 4, 64
    meshes = [synth.make_mesh(700, 40), synth.make_mesh(1500, 41), synth.make_mesh(300, 42)]
    ml = [Meshes([v], [f]) for v, f in meshes]
    az, el, di = synth.learned_spherical_views(B, M, 12)
    r = MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed").to(dev)
    a, e, d = (t.to(dev).requires_grad_() for t in (az, el, di))
    img, cams_ = r(ml, None, a, e, d)
    assert img.shape == (B, M, 3, S, S) and img.dtype == torch.float32 and img.device.type == "cuda"
    assert len(cams_) == B * M and cams_.R.shape == (B * M, 3, 3) and cams_.is_perspective()
    assert torch.allclose(cams_.get_camera_center().norm(dim=1), d.detach().reshape(-1), rtol=1e-5)
    # stage B: oracle fed with the GPU's own R, T, C reproduces the fragments; gradients flow to azim/elev/dist
    R, T, C = (x.detach().cpu().numpy() for x in (cams_.R, cams_.T, cams_._centers))
    vp, fp, voff, foff = pack_np(meshes)
    nrm = oracle.packed_vertex_normals(vp, fp, voff, foff)
    white = np.full(3, 1 / 1.00001, np.float32)
    o = oracle.mesh_forward(vp, fp, voff, foff, nrm, white, M, R, T, C, np.array([[0, 1.0, 0]], np.float32), white, K00, K11, 0.5, S, S, 1,
                            oracle.PERSPECTIVE_CORRECT)
    assert (r.last_fragments["pix_to_face"].cpu().numpy() == o["pix_to_face"]).all()
    assert np.abs(img.detach().cpu().numpy().reshape(B * M, 3, S, S) - o["images"]).max() <= IMG_ATOL
    g = torch.randn(B, M, 3, S, S, generator=torch.Generator().manual_seed(2))
    img.backward(g.to(dev))
    ob = oracle.mesh_backward(vp, fp, voff, foff, nrm, white, M, R, T, C, np.array([[0, 1.0, 0]], np.float32), K00, K11, S, S, 1,
                              oracle.PERSPECTIVE_CORRECT, o["pix_to_face"], g.numpy().reshape(B * M, 3, S, S))
    ga, ge, gd = oracle.look_at_backward(az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel(), ob["gR"], ob["gT"], ob["gC"])
    assert rel(a.grad.reshape(-1), ga) < GRAD_RTOL and rel(e.grad.reshape(-1), ge) < GRAD_RTOL and rel(d.grad.reshape(-1), gd) < GRAD_RTOL
    # a batched Meshes object and eval-mode "relative" light / no_grad also work (run_mvtn.py:517-533)
    r2 = MVRenderer(M, image_size=S, pc_rendering=False).to(dev).eval()
    with torch.no_grad():
        img2, _ = r2(Meshes([v for v, _ in meshes], [f for _, f in meshes]), None, az.to(dev), el.to(dev), di.to(dev))
    assert img2.shape == img.shape and float(img2.min()) >= 0 and float(img2.max()) <= 1.0 + 1e-6


def test_mvrenderer_accepts_collated_host_batch(cuda_device):
    """The loader-side collate (HostPackedMeshes) and the reference's python list render identically."""
    from mvtn_b200 import collate_meshes
    dev = cuda_device
    meshes = [synth.make_mesh(nf, 50 + i) for i, nf in enumerate((700, 90, 2500))]
    ml = [Meshes([v], [f]) for v, f in meshes]
    r = MVRenderer(3, image_size=48, pc_rendering=False, light_direction="fixed").to(dev).eval()
    az, el, di = (t.to(dev) for t in synth.learned_spherical_views(3, 3, 14))
    img_a, _ = r(ml, None, az, el, di)
    hp = collate_meshes(ml)
    assert hp.faces.dtype == torch.int16          # narrowed: every mesh has <= 65536 vertices (MVR_FACES_U16)
    img_b, _ = r(hp, None, az, el, di)
    assert torch.equal(img_a, img_b)
    img_b32, _ = r(collate_meshes(ml, narrow_faces=False), None, az, el, di)
    assert torch.equal(img_a, img_b32)
    a2 = az.clone().requires_grad_()
    img_c, _ = r(collate_meshes(ml), None, a2, el, di)
    img_c.square().mean().backward()
    assert a2.grad is not None and torch.isfinite(a2.grad).all()
    # the list path stages through mvr_host_stage_meshes_packed: uint16 ids + the offset table in the same call; a mesh with more
    # than 65536 vertices keeps int32 ids; both give the geometry of the already-packed device arrays
    g = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    assert g.faces.dtype == torch.int16
    assert g.vert_off.tolist() == [0] + list(np.cumsum([v.shape[0] for v, _ in meshes]))
    assert g.face_off.tolist() == [0] + list(np.cumsum([f.shape[0] for _, f in meshes]))
    g_dev = ops.PackedMeshes.from_packed(torch.cat([v for v, _ in meshes]).to(dev), torch.cat([f for _, f in meshes]).to(dev),
                                         [v.shape[0] for v, _ in meshes], [f.shape[0] for _, f in meshes])
    col = torch.tensor([0.8, 0.7, 0.6], device=dev); lt = torch.tensor([[0.0, 1.0, 0.3]], device=dev)

    def shot(gm):
        v = [t.to(dev) for t in synth.learned_spherical_views(gm.B, 3, 14)]
        with torch.no_grad():
            return ops.render_meshes_from_angles(gm, 3, v[0], v[1], v[2], lt, col, col * 0.5, 48)[0]
    assert torch.equal(shot(g), shot(g_dev)) and float(shot(g).std()) > 0
    big = synth.make_mesh(140000, 3)
    assert big[0].shape[0] > 65536
    g_big = ops.PackedMeshes([big[0], meshes[0][0]], [big[1], meshes[0][1]], dev)
    g_big_dev = ops.PackedMeshes.from_packed(torch.cat([big[0], meshes[0][0]]).to(dev), torch.cat([big[1], meshes[0][1]]).to(dev),
                                             [big[0].shape[0], meshes[0][0].shape[0]], [big[1].shape[0], meshes[0][1].shape[0]])
    assert g_big.faces.dtype == torch.int32 and torch.equal(shot(g_big), shot(g_big_dev))


@pytest.mark.parametrize("K", [1, 2])
def test_mvrenderer_pageable_collated_batch_matches_pinned(cuda_device, K):
    """A collated batch in pageable host memory (a DataLoader without pin_memory=True) is re-staged through pinned buffers by
    PackedMeshes.from_host_packed: a ragged batch gives the images, fragments and azim / elev / dist gradients of the pinned
    batch bit for bit."""
    from mvtn_b200 import collate_meshes
    dev = cuda_device
    meshes = [synth.make_mesh(nf, 70 + i) for i, nf in enumerate((700, 90, 2500, 300, 1200, 40))]
    ml = [Meshes([v], [f]) for v, f in meshes]
    B, M = len(ml), 3
    views = [t.to(dev) for t in synth.learned_spherical_views(B, M, 23)]
    cot = torch.randn(B, M, 3, 56, 56, device=dev)

    def run(pin):
        r = MVRenderer(M, image_size=56, pc_rendering=False, light_direction="relative", faces_per_pixel=K).to(dev).eval()
        a, e, d = (t.detach().clone().requires_grad_() for t in views)
        hp = collate_meshes(ml, pin_memory=pin)
        assert hp.is_pinned() == pin
        img, cams = r(hp, None, a, e, d)
        p2f = r.last_fragments["pix_to_face"].clone()
        img.backward(cot)
        return img.detach().clone(), p2f, a.grad.clone(), e.grad.clone(), d.grad.clone()

    ref, out = run(True), run(False)
    for x, y in zip(ref, out):
        assert torch.equal(x, y)
    assert int((ref[1] >= 0).sum()) > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_regularize_rendered_views_matches_reference(cuda_device, dtype):
    """mvtn_b200.regularize_rendered_views (one gather kernel + its adjoint) against ops.py:138-178 restated with the reference's
    own torch / torchvision calls on the GPU: same seeds -> the same views bit for bit; gradients against torch.autograd through
    dropout2d / flip / ReplicationPad2d / crop."""
    import mvtn_b200
    from oracle import torch_ref as tr
    dev = cuda_device
    B, M = 3, 4
    kinds = set()
    for seed in range(24):
        S = 40 if seed % 2 == 0 else 30      # (rows moved as 16-byte quads / element by element)
        p = [0, 0.3, 0.6][seed % 3]; aug = seed % 4 != 3; cr = [0.3, 0.5, 0.1][seed % 3]
        x0 = torch.rand(B, M, 3, S, S, generator=torch.Generator().manual_seed(seed)).to(dev).to(dtype)
        xr, xm = x0.clone().requires_grad_(), x0.clone().requires_grad_()
        torch.manual_seed(seed); ref = tr.regularize_rendered_views(xr, p, aug, cr)
        torch.manual_seed(seed); out = mvtn_b200.regualarize_rendered_views(xm, p, aug, cr)
        assert out.shape == ref.shape and out.dtype == ref.dtype
        assert torch.equal(out, ref), (seed, p, aug, cr)
        g = torch.randn(B, M, 3, S, S, generator=torch.Generator().manual_seed(100 + seed)).to(dev).to(dtype)
        if out.requires_grad:
            out.backward(g)
            if dtype is torch.float32:
                ref.backward(g)
                want = xr.grad
            else:
                # torch sums the folded edge gradients (up to (2 pad + 1)^2 terms per corner pixel) IN bf16; the kernel sums in
                # fp32 and rounds once: the bf16 check is against the fp32 adjoint of the same gather, to bf16 rounding
                from mvtn_b200.augment import draw_regularizer
                torch.manual_seed(seed); sc, fl, sy, sx = draw_regularizer(x0, p, aug, cr)
                x32 = x0.float().requires_grad_()
                tr.regularize_gather(x32, sc, fl, sy, sx).backward(g.float())
                want = x32.grad
            err = (xm.grad.float() - want.float()).abs().max() / want.float().abs().max().clamp_min(1e-6)
            # fp32: the folded sums differ from autograd's in order only
            assert float(err) < (1e-5 if dtype is torch.float32 else 5e-3), (seed, float(err))
        kinds.add((p > 0, aug))
    assert len(kinds) == 4
    with pytest.raises(ValueError):
        mvtn_b200.regularize_rendered_views(torch.zeros(1, 2, 3, 8, 12, device=dev), 0, True)


def test_cuda_graph_replay_matches_eager(cuda_device):
    """mvtn_b200.graphs: the captured forward / backward graphs reproduce the eager path bit for bit, and pick up
    in-place updates of the captured buffers (new points, moved vertices, new views)."""
    from mvtn_b200 import graphs
    dev = cuda_device
    B, M, S = 3, 4, 64
    views = [t.to(dev) for t in synth.learned_spherical_views(B, M, 17)]
    views2 = [t.to(dev) for t in synth.learned_spherical_views(B, M, 18)]
    cot = torch.randn(B * M, 3, S, S, device=dev)
    col = torch.full((3,), 0.9, device=dev); bg = torch.tensor([0.1, 0.2, 0.3], device=dev)

    def run(fn, vs):
        a, e, d = (t.detach().clone().requires_grad_() for t in vs)
        img = fn(a, e, d)
        img.backward(cot)
        return img.detach().clone(), a.grad.clone(), e.grad.clone(), d.grad.clone()

    # ---- points
    pts = synth.make_clouds(B, 800, 3).to(dev)
    pts2 = synth.make_clouds(B, 800, 4).to(dev)

    def eager_points(a, e, d):
        R, T, _, _ = ops._LookAt.apply(a.reshape(-1), e.reshape(-1), d.reshape(-1))
        return ops.render_points(pts, col, M, R, T, 1.0 / d.reshape(-1), 0.03, bg, S, points_per_pixel=4, compositor="alpha")[0]

    step = graphs.graphed_points_render(pts, col, M, 0.03, bg, S, views, points_per_pixel=4, compositor="alpha")
    for vs, newp in ((views, None), (views2, None), (views, pts2)):
        if newp is not None:
            pts.copy_(newp)
        got, want = run(step, vs), run(eager_points, vs)
        assert all(torch.equal(x, y) for x, y in zip(got, want))
    # ---- meshes (vertex positions updated in place: prepare is part of the graph)
    meshes = synth.make_meshes(B, 1500, 61)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    light = torch.tensor([[0.2, 1.0, -0.3]], device=dev)

    def eager_mesh(a, e, d):
        geom.refresh()
        R, T, C, _ = ops._LookAt.apply(a.reshape(-1), e.reshape(-1), d.reshape(-1))
        return ops.render_meshes(geom, M, R, T, C, light, col, bg, S)[0]

    mstep = graphs.graphed_mesh_render(geom, M, light, col, bg, S, views)
    for vs, scale in ((views, None), (views2, None), (views, 0.8)):
        if scale is not None:
            geom.verts.mul_(scale)
        got, want = run(mstep, vs), run(eager_mesh, vs)
        assert all(torch.equal(x, y) for x, y in zip(got, want))
    assert float(got[0].std()) > 0


def test_mvrenderer_points_end_to_end(oracle, cuda_device):
    dev = cuda_device
    B, M, S = 2, 4, 96
    pts = synth.make_clouds(B, 1024, 8)                        # CPU tensor, as the DataLoader hands it over
    az, el, di = synth.learned_spherical_views(B, M, 3)
    r = MVRenderer(M, image_size=S, pc_rendering=True, points_radius=0.02, points_per_pixel=3, background_color="black",
                   compositor="alpha").to(dev)
    a, e, d = (t.to(dev).requires_grad_() for t in (az, el, di))
    img, cams_ = r(None, pts, a, e, d)
    assert img.shape == (B, M, 3, S, S) and not cams_.is_perspective()
    R, T = cams_.R.detach().cpu().numpy(), cams_.T.detach().cpu().numpy()
    inv = (1.0 / di.reshape(-1)).numpy()
    white = np.full(3, 1 / 1.00001, np.float32)
    o = oracle.points_forward(pts.numpy(), white, M, R, T, inv, 0.02, np.zeros(3, np.float32), S, S, 3, oracle.COMPOSITE_ALPHA)
    assert (r.last_fragments["idx"].cpu().numpy() == o["idx"]).all()
    assert np.abs(img.detach().cpu().numpy().reshape(B * M, 3, S, S) - o["images"]).max() <= IMG_ATOL
    img.square().mean().backward()
    gimg = (2 * img.detach() / img.numel()).cpu().numpy().reshape(B * M, 3, S, S)
    ob = oracle.points_backward(pts.numpy(), white, M, R, T, inv, 0.02, S, S, 3, oracle.COMPOSITE_ALPHA, o["idx"], gimg)
    ga, ge, gd = oracle.look_at_backward(az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel(), ob["gR"], ob["gT"], None)
    gd = gd + ob["g_inv_dist"] * (-1.0 / di.numpy().ravel() ** 2)        # d(1/dist)/d dist
    assert rel(a.grad.reshape(-1), ga) < GRAD_RTOL and rel(e.grad.reshape(-1), ge) < GRAD_RTOL and rel(d.grad.reshape(-1), gd) < GRAD_RTOL
    assert a.grad.abs().max() > 0
    # default MVTN configuration (NormWeighted, K=1) gives ~zero view gradients -- SURVEY 3.4
    r1 = MVRenderer(M, image_size=S, pc_rendering=True, background_color="black").to(dev)
    a1 = az.to(dev).requires_grad_()
    im1, _ = r1(None, pts, a1, el.to(dev), di.to(dev))
    im1.sum().backward()
    assert a1.grad.abs().max() < 1e-3


def test_mvrenderer_rotation_guard_redraws(cuda_device):
    dev = cuda_device
    M = 2
    r = MVRenderer(M, image_size=32, pc_rendering=True, background_color="black").to(dev)
    az = torch.tensor([[0.0, 45.0]]); el = torch.tensor([[float("nan"), 10.0]]); di = torch.tensor([[2.0, 2.0]])
    with pytest.raises(SystemExit, match="Remedy did not work"):         # ops.py:163-164 semantics
        r(None, synth.make_clouds(1, 64, 1), az.to(dev), el.to(dev), di.to(dev))


def test_non_square_images(oracle, cuda_device):
    """H != W goes through the same kernels (PixToNonSquareNdc scales the longer side's NDC range)."""
    dev = cuda_device
    H, W, M = 48, 96, 3
    meshes = synth.make_meshes(1, 900, 77)
    views = synth.learned_spherical_views(1, M, 5)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    geom = ops.PackedMeshes([meshes[0][0]], [meshes[0][1]], dev)
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0.2, 1.0, 0.3]], device=dev)
    img, frag = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col * 0.5, (H, W), faces_per_pixel=2, fragments=True)
    vp, fp, voff, foff = pack_np(meshes)
    o = oracle.mesh_forward(vp, fp, voff, foff, oracle.vertex_normals(vp, fp), np.full(3, 0.99999, np.float32), M, R, T, C,
                            np.array([[0.2, 1.0, 0.3]], np.float32), np.full(3, 0.499995, np.float32), K00, K11, 0.5, H, W, 2,
                            oracle.PERSPECTIVE_CORRECT)
    assert img.shape == (M, 3, H, W)
    assert (frag["pix_to_face"].cpu().numpy() == o["pix_to_face"]).all() and (frag["zbuf"].cpu().numpy() == o["zbuf"]).all()
    assert np.abs(img.cpu().numpy() - o["images"]).max() <= IMG_ATOL
    pts = synth.make_clouds(1, 600, 78)
    inv = (1.0 / views[2].reshape(-1))
    imgp, fragp = ops.render_points(pts.to(dev), col, M, Rd, Td, inv.to(dev), 0.03, col * 0, (W, H), points_per_pixel=2, compositor="alpha", fragments=True)
    op = oracle.points_forward(pts.numpy(), np.full(3, 0.99999, np.float32), M, R, T, inv.numpy(), 0.03, np.zeros(3, np.float32), W, H, 2,
                               oracle.COMPOSITE_ALPHA)
    assert (fragp["idx"].cpu().numpy() == op["idx"]).all() and np.abs(imgp.cpu().numpy() - op["images"]).max() <= IMG_ATOL


def test_render_and_save(cuda_device, tmp_path):
    """renderer.py:200-207: image grid + camera plot (matplotlib is optional: falls back to an .npy of the wireframes)."""
    dev = cuda_device
    r = MVRenderer(4, image_size=64, pc_rendering=False, light_direction="fixed").to(dev)
    meshes = [Meshes([v], [f]) for v, f in synth.make_meshes(2, 400, 3)]
    az, el, di = (t.to(dev) for t in synth.circular_views(2, 4))
    img_path, cam_path = tmp_path / "views.png", tmp_path / "cams.png"
    r.render_and_save(meshes, None, az, el, di, str(img_path), str(cam_path))
    assert img_path.exists() and img_path.stat().st_size > 1000
    assert cam_path.exists() or (tmp_path / "cams.png.npy").exists()


def test_mesh_vertex_gradients(oracle, cuda_device):
    """Gradient scatter to the vertices (north_star (4)): projection + position paths from the kernel, the
    vertex-normal path chained in torch; checked against the oracle's separate outputs and, end to end, against
    torch.autograd of the independent restatement."""
    from oracle import torch_ref as tr
    dev = cuda_device
    v, f = synth.make_mesh(300, 5)
    M, H = 3, 40
    views = synth.learned_spherical_views(1, M, 2)
    R, T, C, (Rd, Td, Cd) = cams(oracle, views, dev)
    vg = v.to(dev).requires_grad_()
    geom = ops.PackedMeshes.from_packed(vg.detach(), f.to(dev), [v.shape[0]], [f.shape[0]])
    col = torch.full((3,), 0.99999, device=dev); light = torch.tensor([[0.3, 1.0, -0.5]], device=dev)
    img, frag = ops.render_meshes(geom, M, Rd, Td, Cd, light, col, col, H, verts=vg)
    g = torch.randn(M, 3, H, H, generator=torch.Generator().manual_seed(4))
    img.backward(g.to(dev))
    p2f = frag["pix_to_face"].cpu().numpy()
    D = torch.float64
    vd = v.to(D).requires_grad_()
    nd = tr.vertex_normals(vd, f)
    loss = 0
    for n in range(M):
        im, _ = tr.render_mesh_view(vd, f, nd, torch.full((v.shape[0], 3), 0.99999, dtype=D), torch.from_numpy(R[n]).to(D), torch.from_numpy(T[n]).to(D),
                                    torch.from_numpy(C[n]).to(D), torch.tensor([0.3, 1.0, -0.5], dtype=D), torch.full((3,), 0.99999, dtype=D), K00, K11, H, H,
                                    p2f=torch.from_numpy(p2f[n, ..., 0]).long())
        loss = loss + (im * g[n].to(D)).sum()
    loss.backward()
    assert rel(vg.grad, vd.grad.numpy()) < 5e-4
    # through the public module too: meshes whose vertices require grad
    r = MVRenderer(M, image_size=H, pc_rendering=False, light_direction="fixed").to(dev)
    v2 = v.clone().requires_grad_()
    im2, _ = r([Meshes([v2], [f])], None, *(t.to(dev) for t in views))
    im2.sum().backward()
    assert v2.grad is not None and v2.grad.abs().max() > 0


def test_training_step_example_runs(cuda_device):
    """BASELINE config 4 in miniature: selector -> renderer -> MVCNN -> loss.backward() reaches the selector."""
    import subprocess, sys as _sys
    from conftest import ROOT
    out = subprocess.run([_sys.executable, os.path.join(ROOT, "examples", "train_step.py"), "--batch", "2", "--views", "2",
                          "--image-size", "64", "--faces", "500", "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "views/s end to end" in out.stdout and "|grad| into the view selector" in out.stdout
    assert float(out.stdout.strip().split()[-1]) > 0


# ------------------------------------------------------------------------------------------ consumer-side fusion (8f N2)
NORM = ((0.456, 0.456, 0.456), (0.225, 0.225, 0.225))      # viewGCN/tools/Trainer_mvt.py:41-49


def _bf16_ulp_close(got_bf16, want_f32):
    """bf16 keeps 8 significant bits: round-to-nearest is within 2^-9 relative, and a value known only to ~1e-5 may
    land on the other neighbour -- allow one bf16 ulp (2^-8 relative) plus the fp32 tolerance."""
    got = got_bf16.to(torch.float32)
    return bool(((got - want_f32).abs() <= want_f32.abs() * 2.0 ** -8 + 1e-4).all())


def test_mesh_normalized_and_bf16_output_matches_oracle(oracle, cuda_device):
    """The shade kernel writes (image - mean) / std (and rounds to bf16 on request) instead of leaving a Normalize +
    cast pass to the consumer; the backward takes the cotangent of THAT tensor.  Checked against the oracle's fp32
    image pushed through the reference's own Normalize, and its gradients fed with g / std."""
    dev = cuda_device
    B, M, S = 2, 3, 80
    meshes = synth.make_meshes(B, 1500, 52)
    ml = [Meshes([v], [f]) for v, f in meshes]
    az, el, di = synth.learned_spherical_views(B, M, 5)
    mean = torch.tensor(NORM[0]).view(1, 3, 1, 1); std = torch.tensor(NORM[1]).view(1, 3, 1, 1)
    g = torch.randn(B, M, 3, S, S, generator=torch.Generator().manual_seed(4))
    grads = {}
    for dt in (torch.float32, torch.bfloat16):
        r = MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed", normalize=NORM, out_dtype=dt).to(dev)
        a, e, d = (t.to(dev).requires_grad_() for t in (az, el, di))
        img, cams_ = r(ml, None, a, e, d)
        assert img.dtype == dt and img.shape == (B, M, 3, S, S)
        R, T, C = (x.detach().cpu().numpy() for x in (cams_.R, cams_.T, cams_._centers))
        vp, fp, voff, foff = pack_np(meshes)
        nrm = oracle.packed_vertex_normals(vp, fp, voff, foff)
        white = np.full(3, 1 / 1.00001, np.float32)
        o = oracle.mesh_forward(vp, fp, voff, foff, nrm, white, M, R, T, C, np.array([[0, 1.0, 0]], np.float32), white, K00, K11, 0.5,
                                S, S, 1, oracle.PERSPECTIVE_CORRECT)
        assert (r.last_fragments["pix_to_face"].cpu().numpy() == o["pix_to_face"]).all()
        want = (torch.from_numpy(o["images"]) - mean) / std                     # Trainer_mvt.py:41-49 on the oracle image
        got = img.detach().cpu().reshape(B * M, 3, S, S)
        if dt is torch.float32:
            assert float((got - want).abs().max()) <= IMG_ATOL / min(NORM[1])
        else:
            assert _bf16_ulp_close(got, want)
        gd_ = g.to(dev).to(dt)
        img.backward(gd_)
        g_raw = (gd_.to(torch.float32).cpu().reshape(B * M, 3, S, S) / std).numpy()      # chain rule through Normalize
        ob = oracle.mesh_backward(vp, fp, voff, foff, nrm, white, M, R, T, C, np.array([[0, 1.0, 0]], np.float32), K00, K11, S, S, 1,
                                  oracle.PERSPECTIVE_CORRECT, o["pix_to_face"], g_raw)
        ga, ge, gdd = oracle.look_at_backward(az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel(), ob["gR"], ob["gT"], ob["gC"])
        assert rel(a.grad.reshape(-1), ga) < GRAD_RTOL and rel(e.grad.reshape(-1), ge) < GRAD_RTOL and rel(d.grad.reshape(-1), gdd) < GRAD_RTOL
        grads[dt] = a.grad.clone()
    assert float(grads[torch.float32].abs().max()) > 0


def test_points_normalized_and_bf16_output_matches_oracle(oracle, cuda_device):
    dev = cuda_device
    B, M, S, K = 2, 3, 96, 4
    pts = synth.make_clouds(B, 1024, 18)
    az, el, di = synth.learned_spherical_views(B, M, 6)
    mean = torch.tensor(NORM[0]).view(1, 3, 1, 1); std = torch.tensor(NORM[1]).view(1, 3, 1, 1)
    g = torch.randn(B, M, 3, S, S, generator=torch.Generator().manual_seed(5))
    for dt in (torch.float32, torch.bfloat16):
        r = MVRenderer(M, image_size=S, pc_rendering=True, points_radius=0.02, points_per_pixel=K, background_color="black",
                       compositor="alpha", normalize=NORM, out_dtype=dt).to(dev)
        a, e, d = (t.to(dev).requires_grad_() for t in (az, el, di))
        img, cams_ = r(None, pts, a, e, d)
        assert img.dtype == dt
        R, T = cams_.R.detach().cpu().numpy(), cams_.T.detach().cpu().numpy()
        inv = (1.0 / di.reshape(-1)).numpy()
        white = np.full(3, 1 / 1.00001, np.float32)
        o = oracle.points_forward(pts.numpy(), white, M, R, T, inv, 0.02, np.zeros(3, np.float32), S, S, K, oracle.COMPOSITE_ALPHA)
        assert (r.last_fragments["idx"].cpu().numpy() == o["idx"]).all()
        want = (torch.from_numpy(o["images"]) - mean) / std
        got = img.detach().cpu().reshape(B * M, 3, S, S)
        if dt is torch.float32:
            assert float((got - want).abs().max()) <= IMG_ATOL / min(NORM[1])
        else:
            assert _bf16_ulp_close(got, want)
        gd_ = g.to(dev).to(dt)
        img.backward(gd_)
        g_raw = (gd_.to(torch.float32).cpu().reshape(B * M, 3, S, S) / std).numpy()
        ob = oracle.points_backward(pts.numpy(), white, M, R, T, inv, 0.02, S, S, K, oracle.COMPOSITE_ALPHA, o["idx"], g_raw)
        ga, ge, gdd = oracle.look_at_backward(az.numpy().ravel(), el.numpy().ravel(), di.numpy().ravel(), ob["gR"], ob["gT"], None)
        gdd = gdd + ob["g_inv_dist"] * (-1.0 / di.numpy().ravel() ** 2)
        assert rel(a.grad.reshape(-1), ga) < GRAD_RTOL and rel(e.grad.reshape(-1), ge) < GRAD_RTOL and rel(d.grad.reshape(-1), gdd) < GRAD_RTOL


@pytest.mark.parametrize("workload", ["mesh", "points"])
def test_bench_line_carries_the_contract_keys_and_parity(cuda_device, workload, tmp_path):
    """One tiny `bench.py` run per workload: ONE JSON line with the contract's keys, and the parity object (SURVEY 8d)
    says what the parity tests say -- bit-exact fragment indices, images / gradients within the stated tolerances.
    --dump-outputs writes what the last timed step returned (6 views: all of them fit the dump)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--workload", workload, "--batch", "2", "--views", "3", "--image-size", "64",
           "--faces", "600", "--points", "512", "--steps", "2", "--warmup", "1", "--cpu-sample-objects", "2", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline", "parity"):
        assert k in d, k
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["gpu_launches"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["roofline"]["bound"] == "hbm" and 0 < d["roofline"]["frac"] < 1.5
    par = d["parity"]
    assert par["index_mismatches"] == 0
    assert par["image_max_abs_err"] <= par["tolerance"]["images_abs"]
    assert par["grad_camera_max_rel_err"] <= par["tolerance"]["gradients_rel"]
    assert par["look_at_max_abs_err"] <= par["tolerance"]["look_at_abs"]
    assert par["look_at_backward_max_rel_err"] <= 1e-4 and par["pass"]
    assert d["steps"] == 2
    index, K = ("pix_to_face", 1) if workload == "mesh" else ("idx", 4)
    want = {"images": ((6, 3, 64, 64), np.float32), index: ((6, 64, 64, K), np.float64), "R": ((6, 3, 3), np.float32),
            "T": ((6, 3), np.float32), "C": ((6, 3), np.float32), "grad_azim": ((2, 3), np.float32),
            "grad_elev": ((2, 3), np.float32), "grad_dist": ((2, 3), np.float32)}
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(k + ".npy" for k in want)
    got = {k: np.load(tmp_path / (k + ".npy")) for k in want}
    for k, (shape, dtype) in want.items():
        assert got[k].shape == shape and got[k].dtype == dtype and np.isfinite(got[k]).all(), k
    assert (got[index] >= -1).all() and (got[index] == np.round(got[index])).all() and (got[index] >= 0).any()
    assert np.abs(got["images"]).max() > 0 and np.abs(got["grad_azim"]).max() > 0


def test_bench_extra_records_carry_parity_baseline_and_roofline(cuda_device):
    """`bench.py --extras tiny`: the sub-records of BASELINE configs[0], [2] and both configs[4] shapes ride in the ONE JSON line,
    each with its own parity gates, CPU baseline (stated sub-sample) and roofline (SURVEY 8d)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--batch", "2", "--views", "3", "--image-size", "64", "--faces", "600",
           "--steps", "2", "--warmup", "1", "--cpu-sample-objects", "1", "--extras", "tiny"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert set(d["extra"]) == {"c1_points", "c3_points", "c5_mesh", "c5_points"}
    for name, rec in d["extra"].items():
        assert rec["value"] > 0 and rec["e2e"]["value"] > 0 and rec["gpu_launches"] > 0, name
        assert rec["parity"]["index_mismatches"] == 0 and rec["parity"]["pass"], (name, rec["parity"])
        assert rec["cpu_baseline"]["value"] > 0 and "sample" in rec["cpu_baseline"], name
        assert rec["roofline"]["bound"] == "hbm" and rec["roofline"]["step"]["frac"] > 0, name
        assert "workload" in rec["config"] and "l2" in rec["config"], name


def test_mvrenderer_points_cuda_graph_mode_matches_eager(cuda_device):
    """MVRenderer(cuda_graph=True): the point step replayed from CUDA graphs (one launch per direction) returns what the
    eager renderer returns -- images, cameras and the gradients w.r.t. azim / elev / dist -- across new clouds, new views,
    a second batch shape and a no-grad call."""
    dev = cuda_device
    M, S = 4, 64
    kw = dict(image_size=S, pc_rendering=True, points_per_pixel=4, points_radius=0.03, background_color="black", compositor="alpha")
    eager = MVRenderer(M, cuda_graph=False, **kw).to(dev).train()
    graph = MVRenderer(M, cuda_graph=True, **kw).to(dev).train()
    eager.object_color = graph.object_color = "white"

    def run(r, pts, views, grad=True):
        a, e, d = (t.to(dev).clone().requires_grad_(grad) for t in views)
        img, cams = r(None, pts, a, e, d)
        if not grad:
            return img.clone(), cams.R.clone()
        cot = torch.linspace(-1, 1, img.numel(), device=dev).view_as(img)
        img.backward(cot)
        return img.detach().clone(), cams.R.detach().clone(), cams.T.detach().clone(), a.grad.clone(), e.grad.clone(), d.grad.clone()

    for B, seeds in ((3, (3, 4, 5)), (2, (6, 7))):
        for i, sd in enumerate(seeds):
            pts = synth.make_clouds(B, 700, sd)                  # host tensor: copied straight into the captured buffer
            views = synth.learned_spherical_views(B, M, 20 + sd)
            got, want = run(graph, pts, views), run(eager, pts, views)
            for k, (x, y) in enumerate(zip(got, want)):
                assert torch.equal(x, y), (B, i, k)
        with torch.no_grad():
            got, want = run(graph, pts, views, grad=False), run(eager, pts, views, grad=False)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert len(graph._point_graphs) >= 2
    # one outstanding forward per captured backward: a second forward before the first result is back-propagated runs eagerly
    # and leaves the first one's gradients intact
    auto = MVRenderer(M, **kw).to(dev).train()                      # cuda_graph=None: automatic for <= 48 views
    auto.object_color = "white"
    pts = synth.make_clouds(2, 700, 3); v1 = synth.learned_spherical_views(2, M, 31); v2 = synth.learned_spherical_views(2, M, 32)
    a1, e1, d1 = (t.to(dev).clone().requires_grad_() for t in v1)
    a2, e2, d2 = (t.to(dev).clone().requires_grad_() for t in v2)
    auto(None, pts, a1, e1, d1)[0].sum().backward()                 # captures, replays, releases
    a1.grad = None
    img1, _ = auto(None, pts, a1, e1, d1)                           # replay: busy until img1 is back-propagated
    assert len(auto._point_graphs) == 1 and next(iter(auto._point_graphs.values()))["busy"]
    img2, _ = auto(None, pts, a2, e2, d2)                           # must not touch the buffers img1's backward reads
    cot = torch.linspace(-1, 1, img1.numel(), device=dev).view_as(img1)
    img1.backward(cot)
    assert not next(iter(auto._point_graphs.values()))["busy"]
    want = run(eager, pts, v1)
    assert torch.equal(a1.grad, want[3]) and torch.equal(img1.detach(), want[0]) and torch.equal(img2.detach(), run(eager, pts, v2)[0])
    # a degenerate elevation (rotation guard): the graphed step steps aside, the eager redraw loop answers
    views = [t.clone() for t in synth.learned_spherical_views(2, M, 9)]
    views[1][0, 0] = 90.0
    torch.manual_seed(0)
    img, cams = graph(None, synth.make_clouds(2, 700, 1), *[t.to(dev) for t in views])
    assert img.shape == (2, M, 3, S, S) and torch.isfinite(img).all()


def test_mvrenderer_mesh_cuda_graph_mode_matches_eager(cuda_device):
    """MVRenderer(cuda_graph=True) on the mesh path: collated host batches of a repeated SHAPE (per-mesh counts) are rendered by
    replaying the captured prepare + look_at + rasterizer + shader graphs, new vertices / faces / views / light copied into the
    captured buffers -- images, cameras, fragments and view gradients equal the eager renderer's bit for bit; a second shape gets
    its own capture; an outstanding forward and a python list of meshes take the eager path."""
    from mvtn_b200 import collate_meshes
    dev = cuda_device
    M, S = 3, 56
    kw = dict(image_size=S, pc_rendering=False, light_direction="relative")
    eager = MVRenderer(M, cuda_graph=False, **kw).to(dev).train()
    graph = MVRenderer(M, cuda_graph=True, **kw).to(dev).train()

    def batch(counts, seed):
        out = []
        for i, nf in enumerate(counts):
            v, f = synth.make_mesh(nf, 300 + i)                        # same topology / counts for every seed ...
            g = torch.Generator().manual_seed(seed * 10 + i)
            v = v * (1.0 + 0.05 * torch.randn(v.shape, generator=g))    # ... new vertex positions
            out.append(Meshes([v], [f.flip(1) if seed % 2 else f]))     # ... and (every other batch) re-wound faces
        return out

    def run(r, ml, views, collate=True):
        a, e, d = (t.to(dev).clone().requires_grad_() for t in views)
        img, cams = r(collate_meshes(ml) if collate else ml, None, a, e, d)
        p2f = r.last_fragments["pix_to_face"].clone()
        cot = torch.linspace(-1, 1, img.numel(), device=dev).view_as(img)
        img.backward(cot)
        return img.detach().clone(), cams.R.detach().clone(), cams.T.detach().clone(), p2f, a.grad.clone(), e.grad.clone(), d.grad.clone()

    for counts, seeds in (((300, 90, 700), (1, 2, 3)), ((120, 500), (4, 5))):
        for sd in seeds:
            ml = batch(counts, sd)
            views = synth.learned_spherical_views(len(counts), M, 40 + sd)
            got, want = run(graph, ml, views), run(eager, ml, views)
            for k, (x, y) in enumerate(zip(got, want)):
                assert torch.equal(x, y), (counts, sd, k)
    assert len(graph._mesh_graphs) == 2 and not any(s.get("failed") for s in graph._mesh_graphs.values())
    # python lists (no fixed host layout to copy from) stay eager
    ml = batch((300, 90, 700), 7)
    views = synth.learned_spherical_views(3, M, 50)
    got, want = run(graph, ml, views, collate=False), run(eager, ml, views, collate=False)
    assert all(torch.equal(x, y) for x, y in zip(got, want)) and len(graph._mesh_graphs) == 2
    # one outstanding forward per captured backward
    a1, e1, d1 = (t.to(dev).clone().requires_grad_() for t in views)
    img1, _ = graph(collate_meshes(ml), None, a1, e1, d1)
    st = graph._mesh_graphs[next(k for k in graph._mesh_graphs if len(k[0]) == 3)]
    assert st["busy"]
    v2 = synth.learned_spherical_views(3, M, 51)
    img2, _ = graph(collate_meshes(ml), None, *[t.to(dev) for t in v2])      # eager: must not touch what img1's backward reads
    img1.backward(torch.linspace(-1, 1, img1.numel(), device=dev).view_as(img1))
    assert not st["busy"]
    want = run(eager, ml, views)
    assert torch.equal(a1.grad, want[4]) and torch.equal(img1.detach(), want[0])
    assert torch.equal(img2.detach(), run(eager, ml, v2)[0])


def test_points_from_angles_fused_backward_equals_the_two_node_chain(cuda_device):
    """ops.render_points_from_angles ends its backward in mvr_points_backward_angles (rasterizer backward + reduction + camera backward
    + scale term in one call); ops.look_at_view_transform + ops.render_points(dist=...) runs the same chain as separate autograd nodes
    (mvr_points_backward, mvr_look_at_backward, torch adds): same gradients bit for bit; gradients sent through the cameras still
    take the unfused path and add up."""
    dev = cuda_device
    B, M, S = 3, 4, 64
    pts = synth.make_clouds(B, 900, 5).to(dev)
    col = torch.full((3,), 0.9, device=dev); bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    views = [t.to(dev) for t in synth.learned_spherical_views(B, M, 12)]
    cot = torch.randn(B * M, 3, S, S, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    for K, mode in ((4, "alpha"), (1, "norm"), (3, "alpha")):
        a1, e1, d1 = (t.clone().requires_grad_() for t in views)
        img1, cams1, _ = ops.render_points_from_angles(pts, col, M, a1, e1, d1, 0.03, bg, S, points_per_pixel=K, compositor=mode)
        img1.backward(cot)
        a2, e2, d2 = (t.clone().requires_grad_() for t in views)
        R, T, C, _bad = ops._LookAt.apply(a2, e2, d2)
        img2, _ = ops.render_points(pts, col, M, R, T, None, 0.03, bg, S, points_per_pixel=K, compositor=mode, dist=d2.reshape(-1))
        img2.backward(cot)
        assert torch.equal(img1, img2)
        for x, y in ((a1.grad, a2.grad), (e1.grad, e2.grad), (d1.grad, d2.grad)):
            assert torch.equal(x, y), (K, mode)
        # a loss that also reads the cameras: unfused path, contributions summed
        a3, e3, d3 = (t.clone().requires_grad_() for t in views)
        img3, (R3, T3, C3, _b), _ = ops.render_points_from_angles(pts, col, M, a3, e3, d3, 0.03, bg, S, points_per_pixel=K, compositor=mode)
        ((img3 * cot).sum() + T3.sum()).backward()
        a4, e4, d4 = (t.clone().requires_grad_() for t in views)
        R4, T4, C4, _b = ops._LookAt.apply(a4, e4, d4)
        img4, _ = ops.render_points(pts, col, M, R4, T4, None, 0.03, bg, S, points_per_pixel=K, compositor=mode, dist=d4.reshape(-1))
        ((img4 * cot).sum() + T4.sum()).backward()
        assert torch.allclose(a3.grad, a4.grad, rtol=1e-5, atol=1e-6) and torch.allclose(d3.grad, d4.grad, rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_mesh_from_angles_fused_backward_equals_the_two_node_chain(cuda_device):
    """ops.render_meshes_from_angles ends its backward in mvr_mesh_backward_angles (rasterizer/shader backward + per-view sums + camera
    backward in one call); ops._LookAt + ops.render_meshes runs the same chain as two autograd nodes (mvr_mesh_backward,
    mvr_look_at_backward): same gradients bit for bit, fixed and relative light;
    gradients sent through the cameras take the unfused path and add up."""
    dev = cuda_device
    B, M, S = 3, 4, 64
    ms = synth.make_meshes(B, 700, 41)
    geom = ops.PackedMeshes([m[0] for m in ms], [m[1] for m in ms], dev)
    col = torch.tensor([0.9, 0.5, 0.3], device=dev); bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    views = [t.to(dev) for t in synth.learned_spherical_views(B, M, 13)]
    cot = torch.randn(B * M, 3, S, S, device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    fixed = torch.tensor([[0.0, 1.0, 0.2]], device=dev)
    for K, light in ((1, None), (2, fixed), (1, fixed)):
        a1, e1, d1 = (t.clone().requires_grad_() for t in views)
        img1, cams1, _ = ops.render_meshes_from_angles(geom, M, a1, e1, d1, light, col, bg, S, faces_per_pixel=K)
        img1.backward(cot)
        a2, e2, d2 = (t.clone().requires_grad_() for t in views)
        R, T, C, _bad = ops._LookAt.apply(a2, e2, d2)
        img2 = ops.render_meshes(geom, M, R, T, C, C.detach() if light is None else light, col, bg, S, faces_per_pixel=K)
        img2 = img2[0] if isinstance(img2, tuple) else img2
        img2.backward(cot)
        assert torch.equal(img1, img2)
        for x, y in ((a1.grad, a2.grad), (e1.grad, e2.grad), (d1.grad, d2.grad)):
            assert torch.equal(x, y), (K, light is None)
        assert float(a1.grad.abs().sum()) > 0 and float(d1.grad.abs().sum()) > 0
        # a loss that also reads the cameras: unfused path, contributions summed
        a3, e3, d3 = (t.clone().requires_grad_() for t in views)
        img3, (R3, T3, C3, _b), _ = ops.render_meshes_from_angles(geom, M, a3, e3, d3, light, col, bg, S, faces_per_pixel=K)
        ((img3 * cot).sum() + T3.sum() + C3.sum()).backward()
        a4, e4, d4 = (t.clone().requires_grad_() for t in views)
        R4, T4, C4, _b = ops._LookAt.apply(a4, e4, d4)
        img4 = ops.render_meshes(geom, M, R4, T4, C4, C4.detach() if light is None else light, col, bg, S, faces_per_pixel=K)
        img4 = img4[0] if isinstance(img4, tuple) else img4
        ((img4 * cot).sum() + T4.sum() + C4.sum()).backward()
        assert torch.allclose(a3.grad, a4.grad, rtol=1e-5, atol=1e-6) and torch.allclose(d3.grad, d4.grad, rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
def test_two_overlapped_staging_jobs_do_not_share_buffers(cuda_device):
    """PackedMeshes.begin(overlap=True) twice before either finish(): one staging thread and one set of pinned buffers, so the second
    begin completes the first batch before it starts its own; both batches come out like the already-packed device arrays."""
    dev = cuda_device
    sets = [[synth.make_mesh(nf, 120 + i) for i, nf in enumerate((900, 4000, 150))], [synth.make_mesh(nf, 130 + i) for i, nf in enumerate((2500, 60))]]
    col = torch.tensor([0.8, 0.7, 0.6], device=dev); lt = torch.tensor([[0.0, 1.0, 0.3]], device=dev)

    def shot(gm):
        v = [t.to(dev) for t in synth.learned_spherical_views(gm.B, 2, 5)]
        with torch.no_grad():
            return ops.render_meshes_from_angles(gm, 2, v[0], v[1], v[2], lt, col, col * 0.5, 40)[0]
    for _ in range(3):
        a = ops.PackedMeshes.begin([v for v, _ in sets[0]], [f for _, f in sets[0]], dev, overlap=True)
        b = ops.PackedMeshes.begin([v for v, _ in sets[1]], [f for _, f in sets[1]], dev, overlap=True)
        assert a._pending is None and ops.PackedMeshes._inflight is b      # a was completed by b's begin
        imgs = [shot(b), shot(a)]                                           # (the node finishes b)
        assert ops.PackedMeshes._inflight is None
        for gm, ms, img in ((b, sets[1], imgs[0]), (a, sets[0], imgs[1])):
            ref = ops.PackedMeshes.from_packed(torch.cat([v for v, _ in ms]).to(dev), torch.cat([f for _, f in ms]).to(dev),
                                               [v.shape[0] for v, _ in ms], [f.shape[0] for _, f in ms])
            assert torch.equal(img, shot(ref)) and float(img.std()) > 0
