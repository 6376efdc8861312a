#!/usr/bin/env python
"""Device time of shader="soft_depth" against its nearest sibling, shader="soft_silhouette": the forward (blurred rasterizer
through mvr_mesh_forward, then mesh_soft_depth_kernel or mesh_soft_blend_kernel) and the backward (mvr_mesh_soft_depth_backward
or mvr_mesh_soft_backward, camera gradients only), each one render_meshes call / one backward of its autograd node, at the two
shapes of scripts/soft_times.py:

  (a) 8 meshes x 12 views, ~2.5 k faces each, 128x128, K = 8, blur 2e-3, sigma 1e-3;
  (b) PyTorch3D's mesh-fitting setup: 1 mesh of ~5 k faces x 20 views, 128x128, K = 50, sigma = 1e-4, blur = 9.2e-4.

Every call is timed with CUDA events around WARM calls, each timed window holding LAUNCHES back-to-back calls of one kind; the
windows of the kinds alternate, REPEATS times, and the median, min and max of the per-call means are printed.  As in
scripts/soft_times.py the fragment lists fit the 126 MB L2 of a B200 (warm-cache times).  The card's name and power limit are
printed with the numbers.

    python scripts/soft_depth_times.py
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import ops, synth         # noqa: E402

LAUNCHES, REPEATS = 30, 7
SHAPES = {
    "a: 8 meshes x 12 views, 2.5k faces, 128^2, K=8":
        dict(B=8, M=12, faces=2500, S=128, K=8, blur=2e-3, sigma=1e-3, dist=2.2, seed=51),
    "b: 1 mesh x 20 views, 5k faces, 128^2, K=50 (PyTorch3D fit)":
        dict(B=1, M=20, faces=5000, S=128, K=50, blur=9.2e-4, sigma=1e-4, dist=2.7, seed=52),
}
SHADERS = ("soft_depth", "soft_silhouette")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def calls(sh, dev):
    """-> {kind: callable}: '<shader> forward' (one render_meshes call) and '<shader> backward' (one backward of a retained graph)."""
    meshes = synth.make_meshes(sh["B"], sh["faces"], sh["seed"])
    nv, nf = [v.shape[0] for v, _ in meshes], [f.shape[0] for _, f in meshes]
    geom = ops.PackedMeshes.from_packed(torch.cat([v for v, _ in meshes]).to(dev), torch.cat([f for _, f in meshes]).to(dev), nv, nf)
    az, el, di = (t.to(dev) for t in synth.learned_spherical_views(sh["B"], sh["M"], sh["seed"] + 1, distance=sh["dist"]))
    R, T, C, _ = ops._LookAt.apply(az, el, di)
    R, T, C = (t.detach().contiguous().requires_grad_() for t in (R, T, C))
    light = torch.tensor([[0.3, 1.0, -0.5]], device=dev); col = torch.tensor([0.9, 0.7, 0.5], device=dev)
    bg = torch.tensor([0.5, 0.25, 0.75], device=dev)
    S, K, N = sh["S"], sh["K"], sh["B"] * sh["M"]
    out = {}
    for shader in SHADERS:
        def fwd(shader=shader):
            return ops.render_meshes(geom, sh["M"], R, T, C, light, col, bg, S, faces_per_pixel=K, shader=shader, blur_radius=sh["blur"],
                                     sigma=sh["sigma"], depth_background=100.0)[0]
        img = fwd()
        g = torch.randn(img.shape, generator=torch.Generator().manual_seed(sh["seed"])).to(dev)
        out[f"{shader} forward"] = fwd
        out[f"{shader} backward"] = lambda img=img, g=g: img.backward(g, retain_graph=True)
    return out, dict(views=N, faces=sum(nf))


def main():
    dev = torch.device("cuda:0")
    print(f"card: {card()}  (name, power limit, max SM clock)")
    print(f"CUDA events, {LAUNCHES} warm back-to-back calls per window, {REPEATS} alternating windows per kind: median [min, max] us per call")
    for name, sh in SHAPES.items():
        fns, info = calls(sh, dev)
        for f in fns.values():      # warm-up: module load, first touches, the workspace at its size
            for _ in range(5):
                f()
        torch.cuda.synchronize()
        per = {k: [] for k in fns}
        for _ in range(REPEATS):
            for k, f in fns.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(LAUNCHES):
                    f()
                e1.record()
                e1.synchronize()
                per[k].append(1e3 * e0.elapsed_time(e1) / LAUNCHES)
        print(f"\n({name})  " + "  ".join(f"{k} {v}" for k, v in info.items()))
        for k, v in per.items():
            print(f"  {k:28s} {np.median(v):9.1f} [{min(v):.1f}, {max(v):.1f}]")
        for d in ("forward", "backward"):
            a, b = np.median(per[f"soft_depth {d}"]), np.median(per[f"soft_silhouette {d}"])
            print(f"  {d}: soft_depth / soft_silhouette = {a / b:.2f}")


if __name__ == "__main__":
    main()
