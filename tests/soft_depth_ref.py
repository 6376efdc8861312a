"""Differentiable torch restatement of the soft depth shader ([upstream] SoftDepthShader), any dtype, built on the helpers of
oracle/torch_ref.py: soft_depth_blend (the upstream formula verbatim; tests/test_soft_depth_host.py pins it to the closed form
the kernels evaluate) and render_mesh_view_soft_depth (tests/test_gpu_soft_depth.py compares the kernels with its fp64
autograd)."""
import torch

from oracle import torch_ref as tr


def soft_depth_blend(p2f, zbuf, dists, sigma, background):
    """[upstream] SoftDepthShader on the fragments of the blurred rasterizer, verbatim: p2f / zbuf / dists (N,H,W,K) -> depth
    (N,H,W,1).  `background` is the shader's zfar."""
    N, H, W, K = p2f.shape
    prob = torch.sigmoid(-dists / sigma) * (p2f >= 0)
    d = torch.cat((zbuf, torch.full((N, H, W, 1), float(background), dtype=zbuf.dtype)), dim=3)
    p = torch.cat((prob, torch.ones((N, H, W, 1), dtype=prob.dtype)), dim=3)
    p = p.cumsum(dim=3).clamp(max=1)
    p = p.diff(dim=3, prepend=torch.zeros((N, H, W, 1), dtype=p.dtype))
    return (p * d).sum(dim=3, keepdim=True)


def render_mesh_view_soft_depth(verts, faces, R, T, k00, k11, H, W, K, blur_radius, sigma=1e-4, background=100.0,
                                perspective_correct=True, clip_bary=None, p2f=None, cull_backfaces=False, z_clip=None, p2c=None,
                                ndc=None):
    """Single-view soft depth: soft_depth_blend over the differentiable fragments of torch_ref.render_mesh_view_soft (zbuf and
    signed dists recomputed from the face ids, near-plane clipping included; p2f / z_clip / p2c as there).  ndc: the projected
    vertices to use instead of project_perspective(verts, R, T) (e.g. an fp64 projection whose values are replaced by the fp32
    ones, straight through); the fragments are then recomputed from them the way render_mesh_view_soft does.  -> depth (H,W),
    fragments dict."""
    if ndc is None:
        _, frag = tr.render_mesh_view_soft(verts, faces, None, None, R, T, None, None, None, k00, k11, H, W, K, blur_radius,
                                           "soft_silhouette", sigma=sigma, perspective_correct=perspective_correct,
                                           clip_bary=clip_bary, p2f=p2f, cull_backfaces=cull_backfaces, z_clip=z_clip, p2c=p2c)
    else:
        frag = _soft_fragments(ndc[faces], H, W, K, blur_radius, perspective_correct, clip_bary, p2f, cull_backfaces, z_clip, p2c)
    dep = soft_depth_blend(frag["pix_to_face"][None], frag["zbuf"][None], frag["dists"][None], sigma, background)
    return dep[0, ..., 0], frag


def _soft_fragments(fv, H, W, K, blur_radius, perspective_correct, clip_bary, p2f, cull_backfaces, z_clip, p2c):
    """The fragment part of torch_ref.render_mesh_view_soft on given projected face vertices fv (F,3,3)."""
    if clip_bary is None:
        clip_bary = blur_radius > 0
    dt = fv.dtype
    yf = tr.pix_centers(H, dt, W)[:, None, None].expand(H, W, K)
    xf = tr.pix_centers(W, dt, H)[None, :, None].expand(H, W, K)
    m1 = torch.full((), -1.0, dtype=dt)
    if z_clip is not None:
        assert p2f is None
        fvc, c2u, _ = tr.clip_faces(fv, z_clip, perspective_correct)
        if p2c is None:
            with torch.no_grad():
                p2c = tr.rasterize_meshes_soft(fv, H, W, K, blur_radius, perspective_correct, clip_bary, cull_backfaces, z_clip,
                                               return_sub=True)[4]
        valid = p2c >= 0
        _, _, pz, sd, _ = tr.soft_fragments(xf, yf, fvc[p2c.clamp_min(0)], perspective_correct, clip_bary)
        p2f = torch.where(valid, c2u[p2c.clamp_min(0)], torch.full_like(p2c, -1))
    else:
        if p2f is None:
            with torch.no_grad():
                p2f = tr.rasterize_meshes_soft(fv, H, W, K, blur_radius, perspective_correct, clip_bary, cull_backfaces)[0]
        valid = p2f >= 0
        _, _, pz, sd, _ = tr.soft_fragments(xf, yf, fv[p2f.clamp_min(0)], perspective_correct, clip_bary)
    return dict(pix_to_face=p2f, zbuf=torch.where(valid, pz, m1), dists=torch.where(valid, sd, m1))
