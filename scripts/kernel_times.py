"""Average device time of every kernel of the resident mesh step (mvr_profile_enable / collect: CUDA events on the
launching stream), plus the step time.  usage: python scripts/kernel_times.py"""
import ctypes, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import ops, synth
from mvtn_b200 import _lib as L

dev = torch.device("cuda:0")
B, M, S, NF = 32, 12, 224, 10000
if len(sys.argv) > 1 and sys.argv[1] == "c5":
    B, M, S, NF = 8, 20, 400, 100000
meshes = synth.make_meshes(B, NF, 1236)
nv = [v.shape[0] for v, _ in meshes]; nf = [f.shape[0] for _, f in meshes]
verts = torch.cat([v for v, _ in meshes]).to(dev); faces = torch.cat([f for _, f in meshes]).to(dev)
az, el, di = (t.to(dev) for t in (synth.circular_views(B, M) if S == 224 else synth.spherical_views(B, M)))
cot = torch.randn(B * M, 3, S, S, device=dev) / (3 * S * S)
col = torch.tensor([0.99999] * 3, device=dev); light = torch.tensor([[0.0, 1.0, 0.0]], device=dev)
lib = L.load()

def step():
    a = az.detach().requires_grad_(); e = el.detach().requires_grad_(); d = di.detach().requires_grad_()
    geom = ops.PackedMeshes.from_packed(verts, faces, nv, nf)
    img, _cams, _frag = ops.render_meshes_from_angles(geom, M, a, e, d, light, col, col, S)
    img.backward(cot)

for _ in range(5):
    step()
torch.cuda.synchronize()
names = ["look_at_forward_one_cta_kernel", "geom_pack_verts_kernel", "geom_pack_faces_kernel", "geom_finish_normals_kernel", "mesh_project_kernel",
         "mesh_scatter_kernel", "mesh_shade_kernel", "mesh_shade_clipped_kernel", "mesh_backward_kernel", "mesh_backward_finish_kernel", "look_at_backward_kernel"]
tot_all = 0.0
for nm in names:
    lib.mvr_profile_enable(nm.encode())
    for _ in range(5):
        step()
    t, n = ctypes.c_double(0), ctypes.c_int(0)
    lib.mvr_profile_collect(ctypes.byref(t), ctypes.byref(n))
    per_step = t.value / 5
    tot_all += per_step
    print("%-32s %8.1f us per step (%d launches/step)" % (nm, 1e3 * per_step, n.value // 5))
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
torch.cuda.synchronize(); e0.record()
for _ in range(30):
    step()
e1.record(); torch.cuda.synchronize()
print("sum of kernels %.1f us; step %.1f us" % (1e3 * tot_all, 1e3 * e0.elapsed_time(e1) / 30))
