"""Differentiable torch restatements of the hard depth shader ([upstream] HardDepthShader), any dtype, built on the helpers of
oracle/torch_ref.py.  tests/test_depth_host.py pins them to the C oracle (zbuf, rasterizer backwards); tests/test_gpu_depth.py
compares the kernels with their fp64 autograd."""
import torch

from oracle import torch_ref as tr


def render_mesh_view_depth(verts, faces, R, T, k00, k11, H, W, perspective_correct=True, cull_backfaces=False, p2f=None,
                           z_clip=None, background=100.0, ndc=None):
    """Single-view hard depth: the nearest fragment's zbuf = sum_i b_i z_i of the (possibly near-plane clipped) face the K = 1
    rasterizer kept, `background` where no face covers the pixel.  p2f / z_clip as in torch_ref.render_mesh_view; ndc: the
    projected vertices to use instead of project_perspective(verts, R, T) (e.g. an fp64 projection whose values are replaced by
    the fp32 ones, straight through).  -> depth (H,W), p2f (H,W)."""
    if ndc is None:
        ndc = tr.project_perspective(verts, R, T, k00, k11)
    fv = ndc[faces]
    yf = tr.pix_centers(H, ndc.dtype)[:, None].expand(H, W)
    xf = tr.pix_centers(W, ndc.dtype)[None, :].expand(H, W)
    if z_clip is not None:
        assert p2f is None
        fvc, c2u, _ = tr.clip_faces(fv, z_clip, perspective_correct)
        with torch.no_grad():
            p2c, _, _ = tr.rasterize_meshes_naive(fvc, H, W, 1, perspective_correct, cull_backfaces)
        p2c = p2c[..., 0]
        sel = fvc[p2c.clamp_min(0)]
        z = (tr.bary_coords(xf, yf, sel, perspective_correct) * sel[..., 2]).sum(-1)
        p2f = torch.where(p2c >= 0, c2u[p2c.clamp_min(0)], torch.full_like(p2c, -1))
    else:
        if p2f is None:
            with torch.no_grad():
                p2f, _, _ = tr.rasterize_meshes_naive(fv, H, W, 1, perspective_correct, cull_backfaces)
            p2f = p2f[..., 0]
        sel = fv[p2f.clamp_min(0)]
        z = (tr.bary_coords(xf, yf, sel, perspective_correct) * sel[..., 2]).sum(-1)
    return torch.where(p2f >= 0, z, torch.full_like(z, background)), p2f


def render_points_view_depth(pts_world, R, T, inv_dist, radius, H, W, background=100.0, idx=None):
    """Single-view hard depth of a cloud: z of the nearest point ((X/d) R + T, orthographic), `background` where no point covers
    the pixel.  -> depth (H,W), idx (H,W,1)."""
    p = (pts_world * inv_dist) @ R + T
    if idx is None:
        with torch.no_grad():
            idx, _, _ = tr.rasterize_points_naive(p, radius, H, W, 1)
    z = p[idx[..., 0].clamp_min(0), 2]
    return torch.where(idx[..., 0] >= 0, z, torch.full_like(z, background)), idx
