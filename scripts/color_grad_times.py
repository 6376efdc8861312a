#!/usr/bin/env python
"""Device time of the mesh backward with and without colour gradients, at two shapes:

  (hard) BASELINE configs[1]: 32 meshes of ~10 k faces x 12 views, 224x224, K = 1, HardPhong (mvr_mesh_backward vs
         mvr_mesh_backward_rgb; one object colour, and per-vertex colours);
  (soft) shape (a) of DESIGN section 8: 8 meshes x 12 views, ~2.5 k faces each, 128x128, K = 8, soft_phong
         (mvr_mesh_soft_backward vs mvr_mesh_soft_backward_rgb, one object colour).

Each call is the whole C call: projection, the per-pixel kernel, the partial-sum kernel (and, for one object colour, the sum
over the views).  Timed with CUDA events around WARM launches, each window holding LAUNCHES back-to-back calls of one kind;
the windows alternate, REPEATS times; median, min and max of the per-call means are printed with the card's name and power
limit.  The zero-filled per-vertex buffer is not re-zeroed between calls (the work does not depend on its values).

    python scripts/color_grad_times.py
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

LAUNCHES, REPEATS = 30, 7


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def _setup(B, M, faces, seed, dev, vrgb):
    meshes = synth.make_meshes(B, faces, seed)
    nv, nf = [v.shape[0] for v, _ in meshes], [f.shape[0] for _, f in meshes]
    rgb = torch.rand(sum(nv), 3, generator=torch.Generator().manual_seed(seed)).to(dev) if vrgb else None
    geom = ops.PackedMeshes.from_packed(torch.cat([v for v, _ in meshes]).to(dev), torch.cat([f for _, f in meshes]).to(dev), nv, nf,
                                        vert_rgb=rgb)
    az, el, di = (t.to(dev) for t in synth.learned_spherical_views(B, M, seed + 1))
    R, T, C, _ = ops._LookAt.apply(az, el, di)
    return geom, tuple(t.detach().contiguous() for t in (R, T, C))


def hard_calls(dev):
    B, M, S = 32, 12, 224
    lib = L.load()
    k00, k11 = ops.fov_projection_scale()
    st = torch.cuda.current_stream(dev).cuda_stream
    p = lambda t: None if t is None else t.data_ptr()      # noqa: E731
    light = torch.tensor([[0.3, 1.0, -0.5]], device=dev); col = torch.tensor([0.9, 0.7, 0.5], device=dev)
    out = {}
    for vrgb in (False, True):
        geom, (R, T, C) = _setup(B, M, 10000, 61, dev, vrgb)
        _, frag = ops.render_meshes(geom, M, R, T, C, light, None if vrgb else col, col, S)
        p2f = frag["pix_to_face"]
        N = B * M
        g = torch.randn(N, 3, S, S, generator=torch.Generator().manual_seed(62)).to(dev)
        gR, gT, gC = torch.empty(N, 3, 3, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, 3, device=dev)
        gRGB = torch.zeros(geom.total_verts, 3, device=dev) if vrgb else torch.empty(3, device=dev)
        ws = ops.workspace(dev, lib.mvr_mesh_workspace_bytes(B, M, S, S, 1, geom.total_verts, geom.total_faces))
        flags = L.PERSPECTIVE_CORRECT | (L.RGB_PER_ELEMENT if vrgb else 0)
        args = (p(geom.geometry), p(geom.vert_off), p(geom.face_off), B, M, geom.total_verts, geom.total_faces, geom.max_verts, p(R),
                p(T), p(C), p(light), 0, None if vrgb else p(col), k00, k11, 0.5, S, S, 1, flags, None, p(p2f), p(g), p(gR), p(gT),
                p(gC), None, None, p(ws), ws.numel(), st)
        tag = "per-vertex colours" if vrgb else "one object colour"
        out[f"hard {tag}: cameras only"] = (lambda a=args: L.check(lib.mvr_mesh_backward(*a), "mvr_mesh_backward"))
        out[f"hard {tag}: + colour gradient"] = (lambda a=args, gr=p(gRGB): L.check(lib.mvr_mesh_backward_rgb(*a, gr), "mvr_mesh_backward_rgb"))
        out[f"_keep {tag}"] = (geom, p2f, g, gR, gT, gC, gRGB, ws, R, T, C)
    return out


def soft_calls(dev):
    B, M, S, K, blur, sigma, gamma = 8, 12, 128, 8, 2e-3, 1e-3, 1e-2
    lib = L.load()
    k00, k11 = ops.fov_projection_scale()
    st = torch.cuda.current_stream(dev).cuda_stream
    p = lambda t: None if t is None else t.data_ptr()      # noqa: E731
    geom, (R, T, C) = _setup(B, M, 2500, 51, dev, False)
    light = torch.tensor([[0.3, 1.0, -0.5]], device=dev); col = torch.tensor([0.9, 0.7, 0.5], device=dev)
    bg = torch.tensor([0.5, 0.25, 0.75], device=dev)
    _, frag = ops.render_meshes(geom, M, R, T, C, light, col, bg, S, faces_per_pixel=K, shader="soft_phong", blur_radius=blur,
                                sigma=sigma, gamma=gamma)
    p2f = frag["pix_to_face"]
    N = B * M
    g = torch.randn(N, 4, S, S, generator=torch.Generator().manual_seed(51)).to(dev)
    gR, gT, gC = torch.empty(N, 3, 3, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, 3, device=dev)
    gRGB = torch.empty(3, device=dev)
    ws = ops.workspace(dev, lib.mvr_mesh_workspace_bytes(B, M, S, S, K, geom.total_verts, geom.total_faces))
    flags = L.PERSPECTIVE_CORRECT | L.CLIP_BARYCENTRIC
    args = (p(geom.geometry), p(geom.vert_off), p(geom.face_off), B, M, geom.total_verts, geom.total_faces, geom.max_verts, p(R), p(T),
            p(C), p(light), 0, p(col), p(bg), k00, k11, 0.5, blur, S, S, K, flags, 0, sigma, gamma, 1.0, 100.0, p(p2f), p(g), p(gR),
            p(gT), p(gC), None, None, p(ws), ws.numel(), st)
    return {"soft_phong one object colour: cameras only": lambda: L.check(lib.mvr_mesh_soft_backward(*args), "mvr_mesh_soft_backward"),
            "soft_phong one object colour: + colour gradient":
                lambda: L.check(lib.mvr_mesh_soft_backward_rgb(*args, p(gRGB)), "mvr_mesh_soft_backward_rgb"),
            "_keep": (geom, p2f, g, gR, gT, gC, gRGB, ws, R, T, C)}


def timed(fns):
    fns = {k: f for k, f in fns.items() if not k.startswith("_")}
    for f in fns.values():      # warm-up: module load, first touches
        for _ in range(3):
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
    return per


def main():
    dev = torch.device("cuda:0")
    print(f"card: {card()}  (name, power limit, max SM clock)")
    print(f"CUDA events, {LAUNCHES} warm back-to-back calls per window, {REPEATS} alternating windows per kind: median [min, max] us per call")
    for name, make in (("hard: BASELINE configs[1], 32 x 12 views, 10k faces, 224^2, K=1", hard_calls),
                       ("soft: DESIGN section 8 shape (a), 8 x 12 views, 2.5k faces, 128^2, K=8, soft_phong", soft_calls)):
        per = timed(make(dev))
        print(f"\n({name})")
        for k, v in per.items():
            print(f"  {k:52s} {np.median(v):9.1f} [{min(v):.1f}, {max(v):.1f}]")
        keys = list(per)
        for a, b in zip(keys[0::2], keys[1::2]):
            ma, mb = np.median(per[a]), np.median(per[b])
            print(f"  colour gradient overhead ({a.split(':')[0]}): {mb - ma:+.1f} us = x{mb / ma:.3f}")


if __name__ == "__main__":
    main()
