"""GPU (CUDA events) and host (perf_counter) timeline of the C-ABI calls of one end-to-end mesh step from a collated batch.
usage: python scripts/trace_e2e_timeline.py"""
import os, sys, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import MVRenderer, Meshes, synth, collate_meshes
from mvtn_b200 import _lib as L
dev = torch.device("cuda:0")
B, M, S, NF = 32, 12, 224, 10000
ml = [Meshes([v], [f]) for v, f in synth.make_meshes(B, NF, 1236)]
host = collate_meshes(ml)
az, el, di = (t.contiguous().pin_memory() for t in synth.circular_views(B, M))
cot = torch.randn(B, M, 3, S, S, device=dev) / (3 * S * S)
g_host = torch.empty(3, B, M, pin_memory=True)
st = torch.cuda.current_stream()
lib = L.load()
marks = []
T0 = [0.0]
def mark(label, stream=None):
    ev = torch.cuda.Event(enable_timing=True); ev.record(stream or st); marks.append((label, ev, 1e6 * (time.perf_counter() - T0[0])))
def wrap(name):
    fn = getattr(lib, name)
    def w(*a):
        mark(name + " >"); rc = fn(*a); mark(name + " <"); return rc
    setattr(lib, name, w)
for n in ("mvr_mesh_prepare", "mvr_mesh_forward", "mvr_mesh_backward", "mvr_look_at_forward", "mvr_look_at_backward"):
    wrap(n)
r = MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed").to(dev).train()
def step(trace):
    T0[0] = time.perf_counter()
    if trace: mark("start")
    a = az.to(dev, non_blocking=True).requires_grad_(); e = el.to(dev, non_blocking=True).requires_grad_(); d = di.to(dev, non_blocking=True).requires_grad_()
    img, _ = r(host, None, a, e, d)
    if trace: mark("forward returned")
    img.backward(cot)
    if trace: mark("backward returned")
    g_host[0].copy_(a.grad, non_blocking=True); g_host[1].copy_(e.grad, non_blocking=True); g_host[2].copy_(d.grad, non_blocking=True)
    if trace: mark("end")
    st.synchronize()
for _ in range(10): step(False)
marks.clear()
torch.cuda.synchronize()
step(True)
torch.cuda.synchronize()
e0 = marks[0][1]
for label, ev, host_us in marks:
    print("  %-28s gpu %8.1f us   host %8.1f us" % (label, 1e3 * e0.elapsed_time(ev), host_us))
