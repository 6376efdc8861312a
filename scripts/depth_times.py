#!/usr/bin/env python
"""Device time of one forward + backward of the hard depth shader against the default render, at two shapes:

  (mesh)   BASELINE configs[1]: 32 meshes of ~10 k faces x 12 views, 224x224: shader="hard_depth" vs "hard_phong" (K = 1), both
           with camera gradients only (ops.render_meshes with R, T, C that require grad);
  (points) 32 clouds of 2048 points x 12 views, 224x224, radius 0.006: shader="hard_depth" vs the default render (norm compositor,
           K = 1), camera and dist gradients.

Each arm is forward + backward of the ops-level node on the same inputs.  Timed with CUDA events around WARM windows of LAUNCHES
back-to-back steps of one arm; the arms alternate, REPEATS times; median, min and max of the per-step means are printed with the
card's name and power limit.

    python scripts/depth_times.py [out.txt]
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import ops, synth         # noqa: E402

LAUNCHES, REPEATS = 20, 7


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def window(step):
    step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(LAUNCHES):
        step()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / LAUNCHES      # us per step


def alternate(arms):
    res = {k: [] for k in arms}
    for k, f in arms.items():      # warm every shape first
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    for _ in range(REPEATS):
        for k, f in arms.items():
            res[k].append(window(f))
    return {k: (float(np.median(v)), min(v), max(v)) for k, v in res.items()}


def mesh_arms(dev):
    B, M, H = 32, 12, 224
    meshes = synth.make_meshes(B, 10000, 0)
    az, el, di = synth.learned_spherical_views(B, M, 1)
    R, T, C = (t.detach() for t in ops.look_at_view_transform(di.to(dev), el.to(dev), az.to(dev), return_centers=True))
    geom = ops.PackedMeshes([v for v, _ in meshes], [f for _, f in meshes], dev)
    Rg, Tg, Cg = (t.clone().requires_grad_() for t in (R, T, C))
    light, col = torch.tensor([[0.0, 1.0, 0.0]], device=dev), torch.ones(3, device=dev)
    g3 = torch.randn(B * M, 3, H, H, device=dev)
    g1 = torch.randn(B * M, 1, H, H, device=dev)

    def phong():
        img, _ = ops.render_meshes(geom, M, Rg, Tg, Cg, light, col, col, H)
        img.backward(g3)

    def depth():
        d, _ = ops.render_meshes(geom, M, Rg, Tg, Cg, light, col, col, H, shader="hard_depth")
        d.backward(g1)

    return {"mesh hard_phong": phong, "mesh hard_depth": depth}


def point_arms(dev):
    B, Np, M, H = 32, 2048, 12, 224
    pts = synth.make_clouds(B, Np, 5).to(dev)
    az, el, di = synth.learned_spherical_views(B, M, 6)
    R, T = (t.detach() for t in ops.look_at_view_transform(di.to(dev), el.to(dev), az.to(dev)))
    Rg, Tg = R.clone().requires_grad_(), T.clone().requires_grad_()
    dg = di.reshape(-1).to(dev).requires_grad_()
    col, bg = torch.ones(3, device=dev), torch.zeros(3, device=dev)
    g3 = torch.randn(B * M, 3, H, H, device=dev)
    g1 = torch.randn(B * M, 1, H, H, device=dev)

    def composite():
        img, _ = ops.render_points(pts, col, M, Rg, Tg, None, 0.006, bg, H, dist=dg)
        img.backward(g3)

    def depth():
        d, _ = ops.render_points(pts, col, M, Rg, Tg, None, 0.006, bg, H, dist=dg, shader="hard_depth")
        d.backward(g1)

    return {"points composite": composite, "points hard_depth": depth}


def main():
    dev = torch.device("cuda:0")
    lines = [f"card: {card()}",
             f"forward + backward per step, us (median of {REPEATS} alternating windows of {LAUNCHES} warm steps; min, max)"]
    for arms in (mesh_arms(dev), point_arms(dev)):
        for k, (med, lo, hi) in alternate(arms).items():
            lines.append(f"{k:20s} {med:9.1f}  ({lo:.1f}, {hi:.1f})")
    text = "\n".join(lines)
    print(text)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
