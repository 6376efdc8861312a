#!/usr/bin/env python
"""Device time of the splat depth shader's forward and backward against the alpha colour path at the same K and against hard
depth, at two point shapes (radius 0.006, the renderer's default; K = 4 as bench.py's point records):

  configs[2]: 32 clouds of 2048 points x 12 learned spherical views, 224x224;
  configs[4]: 8 clouds of 16384 points x 20 spherical views, 400x400.

Each arm is the ops-level node with camera and dist gradients.  Forward: the node's call alone.  Backward: the node's backward on
a retained graph (one forward, then repeated backwards).  Timed with CUDA events around WARM windows of LAUNCHES back-to-back calls
of one arm; the arms alternate, REPEATS times; median, min and max of the per-call means are printed with the card's name and
power limit, read in the same run.

    python scripts/splat_depth_times.py [out.txt]
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
RADIUS, K = 0.006, 4


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
    return a.elapsed_time(b) * 1000.0 / LAUNCHES      # us per call


def alternate(arms):
    res = {k: [] for k in arms}
    for f in arms.values():      # warm every shape first
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    for _ in range(REPEATS):
        for k, f in arms.items():
            res[k].append(window(f))
    return {k: (float(np.median(v)), min(v), max(v)) for k, v in res.items()}


def arms(dev, B, Np, M, H, views):
    pts = synth.make_clouds(B, Np, 5).to(dev)
    az, el, di = views
    R, T = (t.detach() for t in ops.look_at_view_transform(di.to(dev), el.to(dev), az.to(dev)))
    Rg, Tg = R.clone().requires_grad_(), T.clone().requires_grad_()
    dg = di.reshape(-1).to(dev).requires_grad_()
    col, bg = torch.ones(3, device=dev), torch.zeros(3, device=dev)
    renders = {
        "alpha colour": (lambda: ops.render_points(pts, col, M, Rg, Tg, None, RADIUS, bg, H, points_per_pixel=K, compositor="alpha",
                                                   dist=dg)[0], 3),
        "splat_depth": (lambda: ops.render_points(pts, col, M, Rg, Tg, None, RADIUS, bg, H, points_per_pixel=K, dist=dg,
                                                  shader="splat_depth", depth_background=4.0)[0], 1),
        "hard_depth": (lambda: ops.render_points(pts, col, M, Rg, Tg, None, RADIUS, bg, H, dist=dg, shader="hard_depth",
                                                 depth_background=4.0)[0], 1),
    }
    fwd, bwd = {}, {}
    for name, (render, ch) in renders.items():
        g = torch.randn(B * M, ch, H, H, device=dev)
        out = render()

        def forward(render=render):
            with torch.no_grad():
                render()

        def backward(out=out, g=g):
            out.backward(g, retain_graph=True)

        fwd[f"{name} forward"] = forward
        bwd[f"{name} backward"] = backward
    return fwd, bwd


def main():
    dev = torch.device("cuda:0")
    lines = [f"card: {card()}",
             f"radius {RADIUS}, K = {K}; us per call (median of {REPEATS} alternating windows of {LAUNCHES} warm calls; min, max)"]
    shapes = [("configs[2] 32 x 2048 pts x 12 views, 224^2", 32, 2048, 12, 224, synth.learned_spherical_views(32, 12, 6)),
              ("configs[4] 8 x 16384 pts x 20 views, 400^2", 8, 16384, 20, 400, synth.spherical_views(8, 20))]
    for title, B, Np, M, H, views in shapes:
        lines.append(title)
        for group in arms(dev, B, Np, M, H, views):
            for k, (med, lo, hi) in alternate(group).items():
                lines.append(f"  {k:24s} {med:9.1f}  ({lo:.1f}, {hi:.1f})")
    text = "\n".join(lines)
    print(text)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
