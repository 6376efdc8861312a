#!/usr/bin/env python
"""Device time of the soft shaders' backward with and without vertex gradients (mvr_mesh_soft_backward: projection, the
per-fragment kernel mesh_soft_backward_kernel<false | true>, the partial-sum kernel) and of the normals chain that follows it for
soft_phong (mvr_mesh_normals_backward), at two shapes:

  (a) 8 meshes x 12 views, ~2.5 k faces each, 128x128, K = 8, soft_phong (a multi-view batch);
  (b) PyTorch3D's mesh-fitting setup: 1 mesh of ~5 k faces x 20 views, 128x128, K = 50, sigma = 1e-4, blur = 9.2e-4,
      soft_silhouette.

Every call is timed with CUDA events around WARM launches, each timed window holding LAUNCHES back-to-back calls of one kind;
the windows of the kinds alternate, REPEATS times, and the median, min and max of the per-call means are printed.  The
fragment list and the cotangent (75 / 71 MB at (a) / (b)) fit the 126 MB L2 of a B200: the times are those of a warm cache,
as inside a training step that has just run the forward.  The card's name and power limit are printed with the numbers.

    python scripts/soft_times.py
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mvtn_b200 import _lib as L          # noqa: E402
from mvtn_b200 import ops, synth         # noqa: E402

LAUNCHES, REPEATS = 50, 7
SHAPES = {
    "a: 8 meshes x 12 views, 2.5k faces, 128^2, K=8, soft_phong":
        dict(B=8, M=12, faces=2500, S=128, K=8, blur=2e-3, sigma=1e-3, gamma=1e-2, shader="soft_phong", dist=2.2, seed=51),
    "b: 1 mesh x 20 views, 5k faces, 128^2, K=50, soft_silhouette (PyTorch3D fit)":
        dict(B=1, M=20, faces=5000, S=128, K=50, blur=9.2e-4, sigma=1e-4, gamma=1e-4, shader="soft_silhouette", dist=2.7, seed=52),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def calls(sh, dev):
    """-> {kind: callable issuing one C call}, plus the setup for them (one soft forward through ops)."""
    meshes = synth.make_meshes(sh["B"], sh["faces"], sh["seed"])
    nv, nf = [v.shape[0] for v, _ in meshes], [f.shape[0] for _, f in meshes]
    geom = ops.PackedMeshes.from_packed(torch.cat([v for v, _ in meshes]).to(dev), torch.cat([f for _, f in meshes]).to(dev), nv, nf)
    az, el, di = (t.to(dev) for t in synth.learned_spherical_views(sh["B"], sh["M"], sh["seed"] + 1, distance=sh["dist"]))
    R, T, C, _ = ops._LookAt.apply(az, el, di)
    R, T, C = (t.detach().contiguous() for t in (R, T, C))
    light = torch.tensor([[0.3, 1.0, -0.5]], device=dev); col = torch.tensor([0.9, 0.7, 0.5], device=dev)
    bg = torch.tensor([0.5, 0.25, 0.75], device=dev)
    S, K, M, B = sh["S"], sh["K"], sh["M"], sh["B"]
    _, frag = ops.render_meshes(geom, M, R, T, C, light, col, bg, S, faces_per_pixel=K, shader=sh["shader"], blur_radius=sh["blur"],
                                sigma=sh["sigma"], gamma=sh["gamma"])
    p2f = frag["pix_to_face"]
    N = B * M
    g_rgba = torch.randn(N, 4, S, S, generator=torch.Generator().manual_seed(sh["seed"])).to(dev)
    gR, gT, gC = torch.empty(N, 3, 3, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, 3, device=dev)
    gV = torch.zeros(geom.total_verts, 3, device=dev)
    phong = sh["shader"] == "soft_phong"
    gN = torch.zeros(geom.total_verts, 3, device=dev) if phong else None
    lib = L.load()
    ws = ops.workspace(dev, lib.mvr_mesh_workspace_bytes(B, M, S, S, K, geom.total_verts, geom.total_faces))
    k00, k11 = ops.fov_projection_scale()
    flags = L.PERSPECTIVE_CORRECT | L.CLIP_BARYCENTRIC
    st = torch.cuda.current_stream(dev).cuda_stream
    p = lambda t: None if t is None else t.data_ptr()      # noqa: E731

    def soft(gv, gn):
        return lambda: L.check(lib.mvr_mesh_soft_backward(
            p(geom.geometry), p(geom.vert_off), p(geom.face_off), B, M, geom.total_verts, geom.total_faces, geom.max_verts, p(R), p(T),
            p(C), p(light), 0, p(col), p(bg), k00, k11, 0.5, sh["blur"], S, S, K, flags, ops.SOFT_SHADERS[sh["shader"]], sh["sigma"],
            sh["gamma"], 1.0, 100.0, p(p2f), p(g_rgba), p(gR), p(gT), p(gC), p(gv), p(gn), p(ws), ws.numel(), st), "mvr_mesh_soft_backward")

    out = {"soft_backward cameras only (<false>)": soft(None, None), "soft_backward + vertex grads (<true>)": soft(gV, gN)}
    if phong:      # (gN is consumed by the call; its values do not change the work done)
        out["normals_backward"] = lambda: L.check(lib.mvr_mesh_normals_backward(
            p(geom.geometry), p(geom.vert_off), p(geom.face_off), B, geom.total_verts, geom.total_faces, geom.max_faces, p(gN), p(gV), st),
            "mvr_mesh_normals_backward")
    frags = int((p2f >= 0).sum())
    return out, dict(views=N, faces=sum(nf), verts=geom.total_verts, fragments=frags, fragments_per_pixel=frags / (N * S * S))


def main():
    dev = torch.device("cuda:0")
    print(f"card: {card()}  (name, power limit, max SM clock)")
    print(f"CUDA events, {LAUNCHES} warm back-to-back calls per window, {REPEATS} alternating windows per kind: median [min, max] us per call")
    for name, sh in SHAPES.items():
        fns, info = calls(sh, dev)
        for f in fns.values():      # warm-up: module load, first touches
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
        print(f"\n({name})  " + "  ".join(f"{k} {v:.4g}" if isinstance(v, float) else f"{k} {v}" for k, v in info.items()))
        for k, v in per.items():
            print(f"  {k:40s} {np.median(v):9.1f} [{min(v):.1f}, {max(v):.1f}]")
        base = np.median(per["soft_backward cameras only (<false>)"])
        gv = np.median(per["soft_backward + vertex grads (<true>)"]) + (np.median(per["normals_backward"]) if "normals_backward" in per else 0.0)
        print(f"  vertex gradients cost (incl. normals chain): {gv:.1f} us vs {base:.1f} us = x{gv / base:.2f}")


if __name__ == "__main__":
    main()
