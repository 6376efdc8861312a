"""Host-side timeline of one end-to-end MVRenderer step from the collated pinned batch: when (relative to the start of
the step) each C-ABI entry point is called and how long the call takes on the host.  No profiler, perf_counter only."""
import os, sys, time, statistics, collections
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import MVRenderer, Meshes, synth, collate_meshes
from mvtn_b200 import _lib as L

dev = torch.device("cuda:0")
B, M, S = 32, 12, 224
ml = [Meshes([v], [f]) for v, f in synth.make_meshes(B, 10000, 1236)]
host = ml if "list" in sys.argv[1:] else collate_meshes(ml)      # list: the reference's python list of per-object CPU meshes
az, el, di = (t.contiguous().pin_memory() for t in synth.circular_views(B, M))
r = MVRenderer(M, image_size=S, pc_rendering=False, light_direction="fixed", stage_overlap="overlap" in sys.argv[1:]).to(dev)
cot = torch.randn(B, M, 3, S, S, device=dev) / (3 * S * S)
g_host = torch.empty(3, B, M, pin_memory=True)
st = torch.cuda.current_stream()
lib = L.load()
log = collections.defaultdict(list)
T0 = [0.0]

def wrap(name):
    fn = getattr(lib, name)
    def w(*a):
        t = time.perf_counter()
        rc = fn(*a)
        t1 = time.perf_counter()
        log[name].append((1e6 * (t - T0[0]), 1e6 * (t1 - t)))
        return rc
    setattr(lib, name, w)

for n in ("mvr_host_stage_meshes_packed", "mvr_host_stage_meshes_packed_begin", "mvr_host_stage_meshes_end", "mvr_look_at_forward", "mvr_look_at_forward_flagged", "mvr_mesh_prepare", "mvr_mesh_forward", "mvr_mesh_backward", "mvr_mesh_backward_angles", "mvr_look_at_backward"):
    wrap(n)

def step(rec):
    T0[0] = time.perf_counter()
    a = az.to(dev, non_blocking=True).requires_grad_(); e = el.to(dev, non_blocking=True).requires_grad_(); d = di.to(dev, non_blocking=True).requires_grad_()
    t1 = time.perf_counter()
    img, _ = r(host, None, a, e, d)
    t2 = time.perf_counter()
    img.backward(cot.view_as(img))
    t3 = time.perf_counter()
    g_host[0].copy_(a.grad, non_blocking=True); g_host[1].copy_(e.grad, non_blocking=True); g_host[2].copy_(d.grad, non_blocking=True)
    t4 = time.perf_counter()
    st.synchronize()
    t5 = time.perf_counter()
    if rec is not None:
        rec.append([1e6 * (x - T0[0]) for x in (t1, t2, t3, t4, t5)])

for _ in range(10):
    step(None)
log.clear()
rec = []
for _ in range(40):
    step(rec)
names = ["views H2D enqueued", "forward returned", "backward returned", "D2H enqueued", "synchronized"]
for i, n in enumerate(names):
    print("%-22s at %8.1f us" % (n, statistics.median(x[i] for x in rec)))
for n, v in log.items():
    print("%-22s called at %8.1f us, host %6.1f us" % (n, statistics.median(x[0] for x in v), statistics.median(x[1] for x in v)))
