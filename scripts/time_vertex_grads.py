"""Backward of the C2 mesh workload WITH vertex gradients (d/d verts through projection, interpolated position and vertex
normals): per-kernel device time of the backward kernel."""
import ctypes, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import ops, synth
from mvtn_b200 import _lib as L

dev = torch.device("cuda:0")
B, M, S, NF = 32, 12, 224, 10000
meshes = synth.make_meshes(B, NF, 1236)
nv = [v.shape[0] for v, _ in meshes]; nf = [f.shape[0] for _, f in meshes]
verts = torch.cat([v for v, _ in meshes]).to(dev); faces = torch.cat([f for _, f in meshes]).to(dev)
az, el, di = (t.to(dev) for t in synth.circular_views(B, M))
cot = torch.randn(B * M, 3, S, S, device=dev) / (3 * S * S)
col = torch.tensor([0.99999] * 3, device=dev); light = torch.tensor([[0.0, 1.0, 0.0]], device=dev)
lib = L.load()

def step():
    v = verts.detach().requires_grad_()
    R, T, C, _ = ops._LookAt.apply(az, el, di)
    geom = ops.PackedMeshes.from_packed(v.detach(), faces, nv, nf)
    img, _ = ops.render_meshes(geom, M, R, T, C, light, col, col, S, verts=v)
    img.backward(cot)
    return v.grad

for _ in range(3):
    g = step()
torch.cuda.synchronize()
for nm in ("mesh_backward_kernel", "geom_normals_bwd"):
    lib.mvr_profile_enable(nm.encode())
    for _ in range(5):
        step()
    t, n = ctypes.c_double(0), ctypes.c_int(0)
    lib.mvr_profile_collect(ctypes.byref(t), ctypes.byref(n))
    print("%-28s %8.1f us per step (%d launches/step)" % (nm, 1e3 * t.value / 5, n.value // 5))
print("|grad_verts| sum %.6e" % float(g.abs().sum()))
