"""GPU tests of the mesh path's branches that MVTN's shapes do not reach (run on the B200 box with `-m gpu`).

1. The soft shaders (mvr_mesh_soft.cu, blurred rasterizer + SoftPhong / SoftSilhouette blend and backward) against the fp32 /
   fp64 torch restatement (oracle/torch_ref.py) beyond one mesh of one colour: a ragged batch, per-vertex colours, a light per
   view, a non-square image, no perspective correction with back-face culling, K above and at 1, saturated sigmoids, and
   faces crossing the near plane.  Bars of test_mesh_soft_shaders_match_the_torch_restatement.
2. Forward instances of the hard path against the CPU oracle (run_mesh's bars): the 128-thread scatter of meshes above 32768
   faces (layers, halved and tiny queues, big faces, clipped faces), the image-only shade kernel with per-vertex colours, and
   the three face-index types of geom_pack_faces_kernel.

Every case proves that it reached its kernel with the library's launch profiler (test_gpu_branches.launches), so a moved
threshold fails the case instead of moving it to another instance.
"""
import time

import numpy as np
import pytest
import torch

from mvtn_b200 import _lib as L
from mvtn_b200 import ops, synth
from test_gpu_branches import expect_launches, launches
from test_gpu_parity import CUBE_F, CUBE_V, GRAD_RTOL, IMG_ATOL, K00, K11, cams, rel, run_mesh

pytestmark = pytest.mark.gpu

LIGHT = [[0.3, 1.0, -0.5]]
OBJ = [0.9, 0.7, 0.5]
BG = [0.5, 0.25, 0.75]


def no_holes(p2f):
    """The invariant the soft backward relies on: in each pixel's K-list a -1 entry is never followed by a valid one."""
    p = torch.as_tensor(p2f)
    return int(((p[..., 1:] >= 0) & (p[..., :-1] < 0)).sum()) == 0


def saturated(d, sigma):
    """1 - sigmoid(-d / sigma) == 0 in fp32, evaluated as the kernels do (1 / (1 + exp(x)))."""
    x = (-d.numpy().astype(np.float32) / np.float32(sigma)).astype(np.float32)
    with np.errstate(over="ignore"):
        prob = np.float32(1.0) / (np.float32(1.0) + np.exp(-x).astype(np.float32))
    return (np.float32(1.0) - prob.astype(np.float32)) == 0


# ------------------------------------------------------------------------------------------------- 1. soft shaders
SOFT = {
    # name: meshes (target faces, seed), M, (H, W), K, blur, sigma, gamma, options
    "ragged": dict(meshes=[(60, 201), (400, 202), (900, 203)], M=2, HW=(40, 40), K=6, blur=3e-3, sigma=1e-3, gamma=1e-2),
    "vertex_rgb": dict(meshes=[(400, 211)], M=2, HW=(40, 40), K=6, blur=3e-3, sigma=1e-3, gamma=1e-2, vrgb=True, shaders=["soft_phong"]),
    "view_light": dict(meshes=[(300, 221), (500, 222)], M=2, HW=(40, 40), K=4, blur=2e-3, sigma=1e-3, gamma=1e-2, light="camera",
                       shaders=["soft_phong"]),
    "nonsquare_40x72": dict(meshes=[(500, 231)], M=2, HW=(40, 72), K=5, blur=3e-3, sigma=1e-3, gamma=1e-2),
    "noperspective_cull": dict(meshes=[(500, 241)], M=2, HW=(40, 40), K=5, blur=3e-3, sigma=1e-3, gamma=1e-2, persp=False, cull=True),
    "k16_sparse": dict(meshes=[(60, 251)], M=2, HW=(40, 40), K=16, blur=2e-3, sigma=1e-3, gamma=1e-2),
    "k1": dict(meshes=[(400, 261)], M=2, HW=(40, 40), K=1, blur=3e-3, sigma=1e-3, gamma=1e-2),
    "saturated": dict(meshes=[(80, 271)], M=2, HW=(64, 64), K=4, blur=2e-3, sigma=1e-4, gamma=1e-2),      # large faces: deep interiors
    "near_plane": dict(meshes=[(900, 281)], M=3, HW=(48, 48), K=6, blur=3e-3, sigma=1e-3, gamma=1e-2, near=True,
                       views=(torch.tensor([[15.0, 140.0, -80.0]]), torch.tensor([[10.0, -35.0, 50.0]]), torch.tensor([[1.12, 1.2, 1.3]]))),
}
SOFT_PARAMS = [(n, s) for n, c in SOFT.items() for s in c.get("shaders", ["soft_phong", "soft_silhouette"])]


@pytest.mark.parametrize("name,shader", SOFT_PARAMS)
def test_mesh_soft_shaders_branches(oracle, cuda_device, name, shader):
    """render_meshes(shader=soft_*) against torch_ref: fragments bit-exact (zbuf / dists 1e-6, bary 2e-6), RGBA within
    max(1e-5, 5e-9 / gamma), R / T / C gradients within 1e-4 of the tensor's largest entry (silhouette: C gradient exactly 0),
    no hole in any pixel's K-list.  Each view of each mesh of the batch is compared with the reference of its own mesh."""
    from oracle import torch_ref as tr
    c = SOFT[name]
    dev = cuda_device
    meshes = [synth.make_mesh(nf, seed) for nf, seed in c["meshes"]]
    B, M, (H, W), K = len(meshes), c["M"], c["HW"], c["K"]
    persp, cull, near = c.get("persp", True), c.get("cull", False), c.get("near", False)
    views = c.get("views") or synth.learned_spherical_views(B, M, c["meshes"][0][1] + 1)
    R, T, Cc, (Rd, Td, Cd) = cams(oracle, views, dev)
    nv = [v.shape[0] for v, _ in meshes]
    voff = np.cumsum([0] + nv)
    vrgb = torch.rand(int(voff[-1]), 3, generator=torch.Generator().manual_seed(7)) if c.get("vrgb") else None
    light = torch.from_numpy(Cc.copy()) if c.get("light") == "camera" else torch.tensor(LIGHT)
    obj, bg = torch.tensor(OBJ), torch.tensor(BG)
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev, vert_rgb=vrgb)
    Rg, Tg, Cg = (t.clone().requires_grad_() for t in (Rd, Td, Cd))

    def render():
        return ops.render_meshes(geom, M, Rg, Tg, Cg, light.to(dev), None if vrgb is not None else obj.to(dev), bg.to(dev), (H, W),
                                 faces_per_pixel=K, shader=shader, blur_radius=c["blur"], sigma=c["sigma"], gamma=c["gamma"],
                                 perspective_correct=persp, cull_backfaces=cull)

    counts = {}
    want = {"mesh_scatter_kernel<3, true>": 1, "mesh_soft_blend_kernel": 1, "mesh_scatter_kernel<4, false>": 0}
    if near:
        want["mesh_shade_clipped_kernel<true>"] = 1
    out = None
    for pfx in want:
        o, counts[pfx] = launches(pfx, render)
        out = out or o
    expect_launches(counts, want, f"[{name} {shader}] forward")
    img, frag = out
    assert img.shape == (B * M, 4, H, W)
    n_strad = int(frag["counters"][L.CNT_STRADDLE])
    assert (n_strad > 0) == near, n_strad
    g = torch.randn(B * M, 4, H, W, generator=torch.Generator().manual_seed(5))
    _, nb = launches("mesh_soft_backward_kernel", lambda: img.backward(g.to(dev)))
    assert nb == 1
    p2f = frag["pix_to_face"].cpu()
    assert no_holes(p2f), "a -1 entry in front of a valid one"
    D = torch.float64
    Rr, Tr, Cr = (torch.from_numpy(x).to(D).requires_grad_() for x in (R, T, Cc))
    z_clip = 0.5 if near else None
    loss, n_out, t_ref = 0, 0, 0.0
    stats = dict(sat1=0, sat2=0, clip1=0, clip2=0, twice=0, max_frags=0)
    for b, (v, f) in enumerate(meshes):
        nrm = torch.from_numpy(oracle.vertex_normals(v.numpy(), f.numpy())).to(D)
        rgb = (vrgb[voff[b]:voff[b + 1]] if vrgb is not None else obj.expand(v.shape[0], 3)).to(D)
        for m in range(M):
            n = b * M + m
            t0 = time.perf_counter()
            fv32 = torch.from_numpy(oracle.project_perspective(v.numpy(), R[n], T[n], K00, K11))[f]      # the oracle's IEEE projection
            rp2f, rz, rb, rd, rp2c = tr.rasterize_meshes_soft(fv32, H, W, K, c["blur"], persp, None, cull, z_clip=z_clip, return_sub=True)
            t_ref += time.perf_counter() - t0
            assert (p2f[n].long() == rp2f).all(), f"[{name}] view {n}: {int((p2f[n].long() != rp2f).sum())} fragment index mismatches"
            ok = rp2f >= 0
            n_out += int((rd[ok] > 0).sum())
            assert (frag["zbuf"][n].cpu() - rz).abs().max() <= 1e-6
            assert (frag["bary_coords"][n].cpu() - rb).abs().max() <= 2e-6
            assert (frag["dists"][n].cpu() - rd).abs().max() <= 1e-6
            assert no_holes(rp2f)
            stats["max_frags"] = max(stats["max_frags"], int(ok.sum(-1).max()))
            sat = torch.from_numpy(saturated(rd, c["sigma"])) & ok
            nsat = sat.sum(-1)
            stats["sat1"] += int((nsat == 1).sum()); stats["sat2"] += int((nsat >= 2).sum())
            if near:
                nb_behind = (fv32[:, :, 2] < z_clip).sum(1)            # 1: two sub-triangles, 2: one
                kind = torch.where(ok, nb_behind[rp2f.clamp_min(0)], torch.zeros_like(rp2f))
                stats["clip2"] += int((kind == 1).sum()); stats["clip1"] += int((kind == 2).sum())
                srt = rp2f.sort(-1).values
                stats["twice"] += int(((srt[..., 1:] == srt[..., :-1]) & (srt[..., 1:] >= 0)).sum())
            t0 = time.perf_counter()
            ref, rf = tr.render_mesh_view_soft(v.to(D), f, nrm, rgb, Rr[n], Tr[n], Cr[n], light[n if light.shape[0] > 1 else 0].to(D),
                                               bg.to(D), K00, K11, H, W, K, c["blur"], shader, sigma=c["sigma"], gamma=c["gamma"],
                                               perspective_correct=persp, cull_backfaces=cull, p2f=None if near else rp2f,
                                               z_clip=z_clip, p2c=rp2c if near else None)
            t_ref += time.perf_counter() - t0
            assert torch.equal(rf["pix_to_face"], rp2f)
            img_tol = max(IMG_ATOL, 5e-9 / c["gamma"])
            err = float((img[n].detach().cpu().to(D) - ref.detach()).abs().max())
            assert err <= img_tol, (name, n, err)
            loss = loss + (ref * g[n].to(D)).sum()
    t0 = time.perf_counter()
    loss.backward()
    t_ref += time.perf_counter() - t0
    errs = {"gR": rel(Rg.grad, Rr.grad.numpy()), "gT": rel(Tg.grad, Tr.grad.numpy())}
    if shader == "soft_phong":
        errs["gC"] = rel(Cg.grad, Cr.grad.numpy())
    print(f"[{name} {shader}] launches {counts} straddling faces {n_strad} blurred fragments {n_out} {stats} grad errs "
          + " ".join(f"{k} {e:.1e}" for k, e in errs.items()) + f"  reference {t_ref:.2f}s")
    assert n_out > 20                                    # fragments OUTSIDE their face (the blur) are really present
    assert errs["gR"] < GRAD_RTOL and errs["gT"] < GRAD_RTOL
    if shader == "soft_phong":
        assert errs["gC"] < GRAD_RTOL
    else:
        assert float(Cg.grad.abs().max()) == 0.0
    if name == "k16_sparse":
        assert stats["max_frags"] < K and (p2f[..., K - 1] < 0).all()
    if name == "saturated":                              # both branches of the alpha gradient's zero count
        assert stats["sat1"] > 0 and stats["sat2"] > 0, stats
    if near:                                             # one- and two-sub-triangle clips among the fragments
        assert stats["clip1"] > 0 and stats["clip2"] > 0, stats


# ------------------------------------------------------------------------------------------------- 2. hard forward instances
def big_mesh(n_faces, seed):
    """A synth mesh of n_faces (+-1 %) with the 12 faces of a cube (CUBE_V, half size 0.55) appended, shifted so that it sticks
    out of the mesh: its faces cover more than 1024 bbox pixels at H = 96 and are walked by the whole CTA."""
    v, f = synth.make_mesh(n_faces, seed)
    cube = CUBE_V + torch.tensor([0.45, 0.25, -0.3])
    return torch.cat([v, cube]), torch.cat([f, CUBE_F + v.shape[0]])


def scatter_forward_counts(mesh, cfg, want, extra_flags=0):
    """Forward launches of the scatter instances for the scene of cfg (same geometry, cameras and flags as run_mesh)."""
    dev = torch.device("cuda:0")
    geom = ops.PackedMeshes([mesh[0]], [mesh[1]], dev)
    from oracle import oracle as orc
    R, T, Cc, (Rd, Td, Cd) = cams(orc, cfg["views"], dev)
    col = torch.tensor(OBJ, device=dev)
    counts = {}
    for pfx in want:
        _, counts[pfx] = launches(pfx, lambda: ops.render_meshes(geom, cfg["M"], Rd, Td, Cd, torch.tensor(LIGHT, device=dev), col, col, cfg["H"],
                                                                 faces_per_pixel=cfg["K"], fragments=True, _extra_flags=extra_flags))
    return counts


SCATTER128 = {
    # name: (K, extra flags, camera distance, oracle backward)
    "k1": (1, 0, 2.2, True),
    "k3": (3, 0, 2.2, False),
    "tiny_queues": (2, L.TEST_TINY_QUEUES, 2.2, False),
    "close_camera": (1, 0, 1.1, True),
}


@pytest.mark.parametrize("name", list(SCATTER128))
def test_mesh_scatter_128_threads(oracle, cuda_device, name):
    """max_faces > 32768 selects mesh_scatter_kernel<8, false, 128> (128 faces per round, queue of SC_QCAP / 2): against the
    oracle at K = 1 and K = 3 (layer peeling), with 40-entry queues (the in-place fallback), and with a close camera (faces
    crossing the near plane, rasterized by the whole CTA, 4 warps striding the rows).  Big faces in every case."""
    K, flags, dist, bwd = SCATTER128[name]
    mesh = big_mesh(34000, 301)
    assert mesh[1].shape[0] > 32768
    views = synth.learned_spherical_views(1, 2, 302)
    cfg = dict(meshes=[mesh], M=2, H=96, K=K, views=(views[0], views[1], views[2] * 0 + dist))
    want = {"mesh_scatter_kernel<8, false, 128>": 1, "mesh_scatter_kernel<4, false>": 0}
    counts = scatter_forward_counts(mesh, cfg, want, flags)
    expect_launches(counts, want, f"[scatter128 {name}]")
    t0 = time.perf_counter()
    res = run_mesh(oracle, cuda_device, cfg, backward=bwd, extra_flags=flags)
    t_orc = time.perf_counter() - t0
    cnt = res["frag"]["counters"].cpu()
    nf = mesh[1].shape[0] - 12
    cube_px = int((res["p2f"] >= nf).sum())
    print(f"[scatter128 {name}] {counts} big faces {int(cnt[L.CNT_BIG_FACES])} straddling {int(cnt[L.CNT_STRADDLE])} "
          f"cube fragments {cube_px} oracle+run {t_orc:.2f}s")
    if dist < 1.5:
        assert int(cnt[L.CNT_STRADDLE]) > 0
    else:
        assert int(cnt[L.CNT_STRADDLE]) == 0 and int(cnt[L.CNT_BIG_FACES]) > 0 and cube_px > 500
    if K > 1:
        assert (res["p2f"][..., K - 1] >= 0).sum() > 100


def test_mesh_scatter_256_threads_below_the_threshold(oracle, cuda_device):
    """The control: at most 32768 faces (the same construction) stays on mesh_scatter_kernel<4, false>."""
    mesh = big_mesh(32000, 303)
    assert mesh[1].shape[0] <= 32768
    cfg = dict(meshes=[mesh], M=2, H=96, K=2, views=synth.learned_spherical_views(1, 2, 304))
    want = {"mesh_scatter_kernel<4, false>": 1, "mesh_scatter_kernel<8, false, 128>": 0}
    counts = scatter_forward_counts(mesh, cfg, want)
    expect_launches(counts, want, "[scatter256 control]")
    res = run_mesh(oracle, cuda_device, cfg, backward=False)
    assert int(res["frag"]["counters"][L.CNT_BIG_FACES]) > 0


def test_mesh_fast_shade_vertex_rgb_matches_oracle(oracle, cuda_device):
    """fragments=False with per-vertex colours: the image-only kernel mesh_shade_kernel<false, 4, 4, true> (MVRenderer's path for
    coloured meshes) against the oracle's images within 1e-5, and its pix_to_face equal to the exact path's."""
    dev = cuda_device
    meshes = [synth.make_mesh(900, 311), synth.make_mesh(300, 312)]
    vrgb = torch.rand(sum(v.shape[0] for v, _ in meshes), 3, generator=torch.Generator().manual_seed(313))
    M, H = 3, 72
    cfg = dict(meshes=meshes, M=M, H=H, K=1, views=synth.learned_spherical_views(2, M, 314), vert_rgb=vrgb)
    res = run_mesh(oracle, dev, cfg, backward=False)                           # exact path, fragments and images vs the oracle
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev, vert_rgb=vrgb)
    R, T, Cc, (Rd, Td, Cd) = cams(oracle, cfg["views"], dev)
    light = torch.tensor([[0.3, 1.0, -0.5]], device=dev); bg = torch.tensor([0.5, 0.25, 0.75], device=dev)

    def fast():
        return ops.render_meshes(geom, M, Rd, Td, Cd, light, None, bg, H)

    want = {"mesh_shade_kernel<false": 1, "mesh_shade_kernel<true": 0}
    counts, out = {}, None
    for pfx in want:
        o, counts[pfx] = launches(pfx, fast)
        out = out or o
    expect_launches(counts, want, "[fast shade vertex rgb]")
    img, frag = out
    assert torch.equal(frag["pix_to_face"].cpu(), torch.from_numpy(res["p2f"]))
    err = float(np.abs(img.cpu().numpy() - res["o"]["images"]).max())
    print(f"[fast shade vertex rgb] {counts} image err {err:.1e}")
    assert err <= IMG_ATOL


FACE_TYPES = {
    # name: (kernel instance, how the faces are given)
    "cpu_u16": "geom_pack_faces_kernel<unsigned short>",
    "cpu_padded_i32": "geom_pack_faces_kernel<int>",
    "cuda_i64": "geom_pack_faces_kernel<long long>",
    "cuda_i32": "geom_pack_faces_kernel<int>",
}


def test_mesh_face_index_types_agree(oracle, cuda_device):
    """One scene built four ways -- CPU int64 faces (narrowed to uint16 on the way), CPU faces of a mesh padded with 70000
    unreferenced vertices (int32), CUDA int64 and CUDA int32 faces -- takes the three instances of geom_pack_faces_kernel and
    gives the same images and fragments, bit for bit, and the oracle's."""
    dev = cuda_device
    meshes = [synth.make_mesh(700, 321), synth.make_mesh(1500, 322)]
    M, H, K = 2, 56, 2
    views = synth.learned_spherical_views(2, M, 323)
    R, T, Cc, (Rd, Td, Cd) = cams(oracle, views, dev)
    light = torch.tensor(LIGHT, device=dev); col = torch.full((3,), 0.99999, device=dev); bg = torch.tensor(BG, device=dev)
    pad = torch.full((70000, 3), 5.0)

    def build(kind):
        if kind == "cpu_u16":
            return ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
        if kind == "cpu_padded_i32":
            return ops.PackedMeshes([torch.cat([meshes[0][0], pad]), meshes[1][0]], [f for _, f in meshes], dev)
        dt = torch.int64 if kind == "cuda_i64" else torch.int32
        return ops.PackedMeshes([v.to(dev) for v, _ in meshes], [f.to(dt).to(dev) for _, f in meshes], dev)

    outs = {}
    for kind, kernel in FACE_TYPES.items():
        def go():
            geom = build(kind)
            return ops.render_meshes(geom, M, Rd, Td, Cd, light, col, bg, H, faces_per_pixel=K, fragments=True)
        (img, frag), n = launches(kernel, go)
        assert n == 1, (kind, kernel, n)
        outs[kind] = (img, frag)
    ref_img, ref = outs["cpu_u16"]
    for kind, (img, frag) in outs.items():
        assert torch.equal(img, ref_img), kind
        for k in ("pix_to_face", "zbuf", "bary_coords", "dists"):
            assert torch.equal(frag[k], ref[k]), (kind, k)
    res = run_mesh(oracle, dev, dict(meshes=meshes, M=M, H=H, K=K, views=views, light_dir=LIGHT[0]), backward=False)
    o = res["o"]      # run_mesh's colours, light and bg are the ones used here
    assert (ref["pix_to_face"].cpu().numpy() == o["pix_to_face"]).all() and (ref["zbuf"].cpu().numpy() == o["zbuf"]).all()
    assert (ref["bary_coords"].cpu().numpy() == o["bary"]).all() and (ref["dists"].cpu().numpy() == o["dists"]).all()
    assert np.abs(ref_img.cpu().numpy() - o["images"]).max() <= IMG_ATOL
