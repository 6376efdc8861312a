"""Tiny forward + backward of both paths (mesh: scatter + shade, strip and tile backward, K = 1 and 2, a clipped view, vertex
gradients with the warp-aggregated scatter, the soft shaders, a collated batch with uint16 faces; points: tiled and generic K,
the clustered binning (> 4096 points: DSMEM counters), point / colour gradients; the view regulariser; the one-node mesh path
from a python list of host meshes -- camera kernel that stores its flag into the pinned word, staging threads, backward ending in the angle gradients; the multi-CTA camera kernel) for compute-sanitizer:   compute-sanitizer --tool memcheck|racecheck python scripts/sanitize_small.py"""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import ops, synth

dev = torch.device("cuda:0")
col = torch.full((3,), 0.9, device=dev); bg = torch.tensor([0.1, 0.2, 0.3], device=dev); light = torch.tensor([[0.2, 1.0, -0.3]], device=dev)
meshes = synth.make_meshes(2, 700, 5)
geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
views = synth.learned_spherical_views(2, 3, 7)
near = (views[0], views[1], views[2] * 0 + 1.15)
for H, K, vs in ((64, 1, views), (50, 1, views), (40, 2, views), (64, 1, near), (64, 1, views)):
    a, e, d = (t.to(dev).reshape(-1).requires_grad_() for t in vs)
    R, T, C, _ = ops._LookAt.apply(a, e, d)
    img, fr = ops.render_meshes(geom, 3, R, T, C, light, col, bg, H, faces_per_pixel=K)
    img.backward(torch.ones_like(img))
    torch.cuda.synchronize()
    print("mesh", H, K, float(img.sum()), float(a.grad.abs().sum()))
v = geom.verts.detach().clone().requires_grad_()                      # vertex gradients: warp-aggregated atomic scatter + normals backward
a, e, d = (t.to(dev).reshape(-1) for t in views)
R, T, C, _ = ops._LookAt.apply(a, e, d)
img, fr = ops.render_meshes(geom, 3, R, T, C, light, col, bg, 64, verts=v)
img.backward(torch.ones_like(img))
torch.cuda.synchronize()
print("mesh vertex grads", float(v.grad.abs().sum()))
for shader, K in (("soft_phong", 4), ("soft_silhouette", 6)):          # blurred rasterizer + soft blend + backward
    a, e, d = (t.to(dev).reshape(-1).requires_grad_() for t in views)
    R, T, C, _ = ops._LookAt.apply(a, e, d)
    img, fr = ops.render_meshes(geom, 3, R, T, C, light, col, bg, 48, faces_per_pixel=K, shader=shader, blur_radius=2e-3, sigma=1e-3, gamma=1e-2)
    img.backward(torch.ones_like(img))
    torch.cuda.synchronize()
    print("mesh", shader, float(img.detach().sum()), float(a.grad.abs().sum()))
pts = synth.make_clouds(2, 600, 3).to(dev)
for K in (1, 4, 3):
    a, e, d = (t.to(dev).requires_grad_() for t in views)
    img, _, fr = ops.render_points_from_angles(pts, col, 3, a, e, d, 0.03, bg, 64, points_per_pixel=K, compositor="alpha")
    img.backward(torch.ones_like(img))
    torch.cuda.synchronize()
    print("points", K, float(img.sum()), float(d.grad.abs().sum()), int((fr["idx"] >= 0).sum()))
big = synth.make_clouds(1, 5000, 9).to(dev)                              # > 4096 points: 4-CTA cluster binning, DSMEM counters
for K, mode in ((4, "alpha"), (1, "norm")):
    a, e, d = (t[:1].to(dev).requires_grad_() for t in views)
    pg = big.clone().requires_grad_(); cg = col.clone().requires_grad_()      # per-point atomics + the single colour's gradient (partials)
    img, _, fr = ops.render_points_from_angles(pg, cg, 3, a, e, d, 0.02, bg, 96, points_per_pixel=K, compositor=mode)
    img.backward(torch.ones_like(img))
    torch.cuda.synchronize()
    print("points clustered", K, float(img.sum()), float(pg.grad.abs().sum()), float(cg.grad.abs().sum()))
from mvtn_b200 import MVRenderer, Meshes, collate_meshes
ml = [Meshes([v], [f]) for v, f in synth.make_meshes(4, 500, 21)]
r = MVRenderer(3, image_size=48, pc_rendering=False, light_direction="fixed").to(dev)
a, e, d = (t.to(dev).requires_grad_() for t in synth.learned_spherical_views(4, 3, 8))
img, _ = r(collate_meshes(ml), None, a, e, d)
img.backward(torch.ones_like(img))
torch.cuda.synchronize()
print("mesh collated (uint16 faces)", float(img.detach().sum()), float(a.grad.abs().sum()), collate_meshes(ml).faces.dtype)
from mvtn_b200 import regularize_rendered_views
for dt, S in ((torch.float32, 48), (torch.bfloat16, 48), (torch.float32, 30)):      # the view regulariser: gather + adjoint (quads / scalar rows)
    x = torch.rand(2, 3, 3, S, S, device=dev).to(dt).requires_grad_()
    torch.manual_seed(4)
    y = regularize_rendered_views(x, 0.4, True, 0.3)
    y.backward(torch.ones_like(y))
    torch.cuda.synchronize()
    print("regularize", dt, S, float(y.float().sum()), float(x.grad.float().abs().sum()))
# one-node path: camera kernel that owns its flag (stored into the pinned word by the kernel), list of host meshes staged on the
# library's threads (uint16 ids + offsets in one call), backward ending in the angle gradients (mesh_backward_finish_kernel + look_at)
from mvtn_b200 import MVRenderer, Meshes
r = MVRenderer(3, image_size=48, pc_rendering=False, light_direction="fixed").to(dev)
for near_cam in (False, True):
    a, e, d = (t.to(dev).clone().requires_grad_() for t in (near if near_cam else views))
    img, cams = r([Meshes([v_], [f_]) for v_, f_ in meshes], None, a, e, d)
    img.sum().backward()
    torch.cuda.synchronize()
    print("mesh from angles (list staging, fused camera backward)", near_cam, float(img.detach().sum()), float(a.grad.abs().sum()), float(d.grad.abs().sum()))
n_big = 5000                                                            # multi-CTA camera kernel (> 4096 views) + pooled sink
g_ = torch.Generator().manual_seed(3)
az_b = (torch.rand(n_big, generator=g_) * 360 - 180).to(dev); az_b[17] = float("nan")
sink = ops.FlagSink.get(dev)
ops._look_at_launch(az_b, az_b * 0 + 20, az_b * 0 + 2.2, sink)
print("cameras", n_big, "invalid:", sink.read())
