"""Differentiable torch restatement of the splat depth of point clouds (shader="splat_depth"), any dtype, built on the helpers of
oracle/torch_ref.py: splat_depth_blend (tests/test_splat_depth_host.py pins it to the per-pixel loop the kernels evaluate) and
render_points_view_splat_depth (tests/test_gpu_splat_depth.py compares the kernels with its fp64 autograd)."""
import torch

from oracle import torch_ref as tr


def splat_depth_blend(idx, zbuf, alpha, background, stopped=None):
    """[upstream] SoftDepthShader's blend with the splat weight alpha in place of sigmoid(-dists / sigma): idx / zbuf / alpha
    (N,H,W,K), valid entries a prefix of the list, nearest first -> depth (N,H,W,1).  c = cumsum(alpha), m_k = min(c_k, 1), the sum
    stopping after the first entry with c > 1 (later entries keep m = 1, as the kernels' loop ends there; alpha is not clamped, so
    without the stop a negative alpha could take c back under 1).  Where c <= 1, m = c passes the gradient (torch's clamp at
    equality).  stopped: the decision "this entry or an earlier one has c > 1" to use instead of the one taken from `alpha` (e.g.
    the kernels' fp32 one)."""
    valid = idx >= 0
    a = torch.where(valid, alpha, torch.zeros_like(alpha))
    c = a.cumsum(dim=3)
    if stopped is None:
        stopped = ((c > 1) & valid).cumsum(dim=3) > 0
    m = torch.where(stopped, torch.ones_like(c), c)
    w = m.diff(dim=3, prepend=torch.zeros_like(m[..., :1]))
    z = torch.where(valid, zbuf, torch.zeros_like(zbuf))
    return (w * z).sum(dim=3, keepdim=True) + (1 - m[..., -1:]) * background


def rasterize_points(p, radius, H, W, K):
    """torch_ref.rasterize_points_naive with the pixel centres of a non-square image ([upstream] PixToNonSquareNdc, as the
    kernels and the C oracle) -> idx (H,W,K) long, zbuf, dists2 (-1 where empty)."""
    dt = p.dtype
    yf = tr.pix_centers(H, dt, W)[:, None, None]
    xf = tr.pix_centers(W, dt, H)[None, :, None]
    d2 = (p[None, None, :, 0] - xf) ** 2 + (p[None, None, :, 1] - yf) ** 2
    r2 = torch.tensor(radius, dtype=dt) * torch.tensor(radius, dtype=dt)
    hit = (d2 < r2) & ~(p[None, None, :, 2] < 0)
    key = torch.where(hit, p[None, None, :, 2].expand_as(d2), torch.full_like(d2, float("inf")))
    order = torch.sort(key, dim=-1, stable=True)
    idx, zs = order.indices[..., :K], order.values[..., :K]
    if idx.shape[-1] < K:
        pad = K - idx.shape[-1]
        idx = torch.cat([idx, idx.new_zeros(H, W, pad)], -1)
        zs = torch.cat([zs, zs.new_full((H, W, pad), float("inf"))], -1)
    valid = torch.isfinite(zs)
    d2s = torch.gather(d2, 2, idx)
    m1 = torch.full_like(zs, -1.0)
    return torch.where(valid, idx, torch.full_like(idx, -1)), torch.where(valid, zs, m1), torch.where(valid, d2s, m1)


def render_points_view_splat_depth(pts_world, R, T, inv_dist, radius, H, W, K, background=100.0, idx=None, stopped=None, ndc=None):
    """Single-view splat depth of a cloud: (X/d) R + T (orthographic) as torch_ref.render_points_view, alpha = 1 - d2 / r^2 of
    the K nearest points, splat_depth_blend.  idx: the fragment list to use (H,W,K); stopped as in splat_depth_blend; ndc: the
    projected points to use instead of (X/d) R + T (e.g. an fp64 projection whose values are replaced by the fp32 ones, straight
    through).  -> depth (H,W), dict(idx, zbuf, alpha)."""
    p = (pts_world * inv_dist) @ R + T if ndc is None else ndc
    if idx is None:
        with torch.no_grad():
            idx = rasterize_points(p, radius, H, W, K)[0]
    # the pixel centres are fp32 numbers (the rasterizer's, [upstream] and the kernels'): in fp64 they would move d2 by up to
    # 2 r ulp(1), alpha by 2 ulp(1) / r -- 3e-6 at r = 0.02, far above what the comparison is meant to resolve
    yf = tr.pix_centers(H, torch.float32, W).to(p.dtype)[:, None, None]
    xf = tr.pix_centers(W, torch.float32, H).to(p.dtype)[None, :, None]
    sel = p[idx.clamp_min(0)]                       # (H,W,K,3)
    valid = idx >= 0
    d2 = (sel[..., 0] - xf) ** 2 + (sel[..., 1] - yf) ** 2
    alpha = torch.where(valid, 1 - d2 / (radius * radius), torch.zeros_like(d2))
    zbuf = torch.where(valid, sel[..., 2], torch.full_like(d2, -1.0))
    dep = splat_depth_blend(idx[None], zbuf[None], alpha[None], background, None if stopped is None else stopped[None])
    return dep[0, ..., 0], dict(idx=idx, zbuf=zbuf, alpha=alpha)
