"""Second, independent restatement of the MVRenderer arithmetic in plain torch (autograd-capable,
dtype-generic).  TEST INFRASTRUCTURE ONLY -- same import rules as oracle/oracle.py.

Purpose: (1) cross-check the C oracle (two independent restatements of an unpinned spec);
(2) validate every hand-derived backward (C oracle and CUDA) against torch.autograd, typically in
float64.  Follows the *python* layer of PyTorch3D v0.7 [upstream, not on disk]: renderer/cameras.py,
renderer/mesh/shading.py, renderer/lighting.py, renderer/blending.py, renderer/points/renderer.py,
renderer/compositing.py, structures/meshes.py -- as called from models/renderer.py:65-151.

Vectorised O(P*F) -- small sizes only.
"""
import math

import torch
import torch.nn.functional as F

K_EPS = 1e-8


def pix_centers(S, dtype=torch.float32, other=None):
    """NDC coordinate of pixel index i (0 = top row / left column): +Y up, +X left.  other: the image's other side -- the
    longer side of a non-square image spans 2 * (S // other) NDC units ([upstream] PixToNonSquareNdc)."""
    i = torch.arange(S, dtype=dtype)
    if other is None or S <= other:
        return -1.0 + (2.0 * (S - 1 - i) + 1.0) / S
    rng = 2.0 * (S // other)
    return -rng / 2 + (rng * (S - 1 - i) + rng / 2) / S


def look_at_view_transform(dist, elev, azim):
    """[upstream] cameras.look_at_view_transform with at=0, up=(0,1,0), degrees=True.  -> R, T, C"""
    e = math.pi / 180.0 * elev
    a = math.pi / 180.0 * azim
    C = torch.stack([dist * torch.cos(e) * torch.sin(a), dist * torch.sin(e), dist * torch.cos(e) * torch.cos(a)], dim=1)
    up = torch.zeros_like(C); up[:, 1] = 1
    z = F.normalize(-C, eps=1e-5)
    x = F.normalize(torch.cross(up, z, dim=1), eps=1e-5)
    y = F.normalize(torch.cross(z, x, dim=1), eps=1e-5)
    close = (x.abs() <= 5e-3).all(dim=1, keepdim=True)
    if close.any():
        x = torch.where(close, F.normalize(torch.cross(y, z, dim=1), eps=1e-5), x)
    R = torch.stack([x, y, z], dim=2)  # columns
    T = -torch.bmm(R.transpose(1, 2), C[:, :, None])[:, :, 0]
    return R, T, C


def look_at_backward_fp32(dist, elev, azim, gR, gT, gC):
    """fp32 autograd of look_at_view_transform under the cotangents (gR, gT, gC) -> (g_azim, g_elev, g_dist, cot), all (n,).
    cot[i] is the largest |cotangent| any node of view i's graph receives or passes on.  Near the poles the chain through
    the normalisations builds cotangents of 1e7 that cancel to an O(1) d elev, so an fp32 evaluation of it (this one, or the
    CUDA kernel) carries an absolute error of a few eps_fp32 * cot[i]: the conditioning bar of DESIGN.md 2."""
    n = dist.shape[0]
    d, e, a = (t.detach().float().clone().requires_grad_() for t in (dist, elev, azim))
    R, T, C = look_at_view_transform(d, e, a)
    loss = (R * gR.float()).sum() + (T * gT.float()).sum() + (C * gC.float()).sum()
    cot = torch.zeros(n)

    def hook(grad_inputs, grad_outputs):
        for g in grad_inputs + grad_outputs:
            if g is not None and g.dim() >= 1 and g.shape[0] == n:
                cot.copy_(torch.maximum(cot, g.detach().abs().reshape(n, -1).amax(1)))

    seen, todo = set(), [loss.grad_fn]
    while todo:
        node = todo.pop()
        if node is None or node in seen:
            continue
        seen.add(node)
        node.register_hook(hook)
        todo.extend(nx for nx, _ in node.next_functions)
    loss.backward()
    return a.grad, e.grad, d.grad, cot


def fov_k(fov_deg=60.0, znear=1.0, dtype=torch.float32):
    """[upstream] FoVPerspectiveCameras.compute_projection_matrix K00 = K11 (aspect 1), as fp32 ops."""
    fov = torch.tensor(fov_deg, dtype=dtype) * (math.pi / 180.0)
    max_y = torch.tan(fov / 2) * znear
    return float(2.0 * znear / (max_y - (-max_y)))


def project_perspective(verts, R, T, k00, k11):
    """verts (V,3), R (3,3), T (3) -> (V,3) = (x_ndc, y_ndc, z_view)."""
    p = verts @ R + T
    return torch.stack([p[:, 0] * k00 / p[:, 2], p[:, 1] * k11 / p[:, 2], p[:, 2]], dim=1)


def _edge(px, py, ax, ay, bx, by):
    return (px - ax) * (by - ay) - (py - ay) * (bx - ax)


def bary_coords(px, py, fv, perspective_correct):
    """px,py (...,) ; fv (...,3,3) -> bary (...,3) following geometry_utils.h."""
    x0, y0, z0 = fv[..., 0, 0], fv[..., 0, 1], fv[..., 0, 2]
    x1, y1, z1 = fv[..., 1, 0], fv[..., 1, 1], fv[..., 1, 2]
    x2, y2, z2 = fv[..., 2, 0], fv[..., 2, 1], fv[..., 2, 2]
    area = _edge(x2, y2, x0, y0, x1, y1) + K_EPS
    w0 = _edge(px, py, x1, y1, x2, y2) / area
    w1 = _edge(px, py, x2, y2, x0, y0) / area
    w2 = _edge(px, py, x0, y0, x1, y1) / area
    if perspective_correct:
        t0, t1, t2 = w0 * z1 * z2, w1 * z0 * z2, w2 * z0 * z1
        # forward: max(sum, kEpsilon).  [upstream] BarycentricPerspectiveCorrectionBackward differentiates the denominator as
        # the plain sum whether or not the clamp acted (it only acts OUTSIDE a face, i.e. for blurred fragments), so the clamp
        # is straight-through here: value kEpsilon exactly, gradient 1.
        ssum = t0 + t1 + t2
        den = torch.where(ssum < K_EPS, K_EPS + (ssum - ssum.detach()), ssum)
        w0, w1, w2 = t0 / den, t1 / den, t2 / den
    return torch.stack([w0, w1, w2], dim=-1)


def rasterize_meshes_naive(face_verts, H, W, K=1, perspective_correct=True, cull_backfaces=False):
    """One view.  face_verts (F,3,3) -> pix_to_face (H,W,K) long, zbuf (H,W,K), bary (H,W,K,3)."""
    dt = face_verts.dtype
    yf = pix_centers(H, dt)[:, None, None]
    xf = pix_centers(W, dt)[None, :, None]
    fv = face_verts[None, None]
    b = bary_coords(xf, yf, fv, perspective_correct)            # (H,W,F,3)
    x, y, z = face_verts[..., 0], face_verts[..., 1], face_verts[..., 2]
    area = _edge(x[:, 0], y[:, 0], x[:, 1], y[:, 1], x[:, 2], y[:, 2])
    ok = ~((area <= K_EPS) & (area >= -K_EPS))
    if cull_backfaces:
        ok &= ~(area < 0)
    ok &= ~(z.min(dim=1).values < K_EPS)
    inbox = (xf <= x.max(1).values) & (xf >= x.min(1).values) & (yf <= y.max(1).values) & (yf >= y.min(1).values)
    pz = (b * z[None, None]).sum(-1)
    hit = ok[None, None] & inbox & (b > 0).all(-1) & ~(pz < 0)
    key = torch.where(hit, pz, torch.full_like(pz, float("inf")))
    # stable sort by z then index == lexicographic (z, idx)
    order = torch.sort(key, dim=-1, stable=True)
    idx = order.indices[..., :K]
    zs = order.values[..., :K]
    if idx.shape[-1] < K:
        pad = K - idx.shape[-1]
        idx = torch.cat([idx, idx.new_zeros(H, W, pad)], -1)
        zs = torch.cat([zs, zs.new_full((H, W, pad), float("inf"))], -1)
    valid = torch.isfinite(zs)
    p2f = torch.where(valid, idx, torch.full_like(idx, -1))
    bsel = torch.gather(b, 2, idx.clamp_min(0)[..., None].expand(H, W, K, 3))
    zbuf = torch.where(valid, zs, torch.full_like(zs, -1.0))
    bary = torch.where(valid[..., None], bsel, torch.full_like(bsel, -1.0))
    return p2f, zbuf, bary


def vertex_normals(verts, faces):
    """[upstream] Meshes._compute_vertex_normals (v0.7 form)."""
    vf = verts[faces]
    vn = torch.zeros_like(verts)
    # one cross product per corner, three index_add passes in upstream's order (corner 1, 2, 0)
    vn = vn.index_add(0, faces[:, 1], torch.cross(vf[:, 2] - vf[:, 1], vf[:, 0] - vf[:, 1], dim=1))
    vn = vn.index_add(0, faces[:, 2], torch.cross(vf[:, 0] - vf[:, 2], vf[:, 1] - vf[:, 2], dim=1))
    vn = vn.index_add(0, faces[:, 0], torch.cross(vf[:, 1] - vf[:, 0], vf[:, 2] - vf[:, 0], dim=1))
    return F.normalize(vn, eps=1e-6, dim=1)


def phong_shade(bary, p2f, verts, faces, normals, vert_rgb, light_dir, cam_center, bg,
                ambient=0.5, diffuse=0.3, specular=0.2, shininess=64):
    """bary (H,W,3), p2f (H,W) for k=0.  -> (3,H,W).  phong_shading + hard_rgb_blend."""
    fg = p2f >= 0
    f = p2f.clamp_min(0)
    fvx = verts[faces][f]          # (H,W,3,3)
    fnr = normals[faces][f]
    fcl = vert_rgb[faces][f]
    P = (bary[..., None] * fvx).sum(-2)
    Nn = (bary[..., None] * fnr).sum(-2)
    tex = (bary[..., None] * fcl).sum(-2)
    n = F.normalize(Nn, p=2, dim=-1, eps=1e-6)
    l = F.normalize(light_dir.expand_as(n), p=2, dim=-1, eps=1e-6)
    cosang = (n * l).sum(-1)
    diff = F.relu(cosang)
    mask = (cosang > 0).to(bary.dtype)
    v = F.normalize(cam_center - P, p=2, dim=-1, eps=1e-6)
    r = -l + 2 * (cosang[..., None] * n)
    alpha = F.relu((v * r).sum(-1)) * mask
    col = (ambient + diffuse * diff)[..., None] * tex + (specular * torch.pow(alpha, shininess))[..., None]
    out = torch.where(fg[..., None], col, bg.expand_as(col))
    return out.permute(2, 0, 1)


def clip_faces(fv, z_clip, perspective_correct):
    """[upstream] renderer/mesh/clip.py clip_faces against the plane z = z_clip only (MeshRasterizer: cull_to_frustum
    False), written per face with differentiable tensor ops.  fv (F,3,3) = (x_ndc, y_ndc, z_view).
    -> fvc (Fc,3,3) clipped face list, c2u (Fc,) index of the unclipped face, conv (Fc,3,3) with conv[c][j][k] = barycentric
    weight of original vertex j in clipped vertex k (identity for untouched faces)."""
    out_v, out_u, out_c = [], [], []
    eye = torch.eye(3, dtype=fv.dtype)
    for f in range(fv.shape[0]):
        v = fv[f]
        behind = v[:, 2] < z_clip
        nb = int(behind.sum())
        if nb == 3:
            continue
        if nb == 0:
            out_v.append(v); out_u.append(f); out_c.append(eye); continue
        case4 = nb == 1
        i1 = int(torch.nonzero(behind if case4 else ~behind)[0])
        i2, i3 = (i1 + 1) % 3, (i1 + 2) % 3
        p1, p2, p3 = v[i1], v[i2], v[i3]
        w2 = (p1[2] - z_clip) / (p1[2] - p2[2])
        w3 = (p1[2] - z_clip) / (p1[2] - p3[2])
        p4 = p1 * (1 - w2) + p2 * w2
        p5 = p1 * (1 - w3) + p3 * w3
        if perspective_correct:      # interpolate the un-projected xy, re-project at the plane
            a1, a2, a3 = p1[:2] * p1[2], p2[:2] * p2[2], p3[:2] * p3[2]
            p4 = torch.cat([(a1 * (1 - w2) + a2 * w2) / z_clip, p4[2:]])
            p5 = torch.cat([(a1 * (1 - w3) + a3 * w3) / z_clip, p5[2:]])
        e = [eye[i1], eye[i2], eye[i3]]
        bc = [e[0], e[1], e[2], e[0] * (1 - w2) + e[1] * w2, e[0] * (1 - w3) + e[2] * w3]
        P = [p1, p2, p3, p4, p5]
        picks = [(3, 1, 4), (4, 1, 2)] if case4 else [(3, 4, 0)]
        for pk in picks:
            out_v.append(torch.stack([P[k] for k in pk]))
            out_u.append(f)
            out_c.append(torch.stack([bc[k] for k in pk], dim=1))
    if not out_v:
        return fv.new_zeros((0, 3, 3)), torch.zeros(0, dtype=torch.long), fv.new_zeros((0, 3, 3))
    return torch.stack(out_v), torch.tensor(out_u, dtype=torch.long), torch.stack(out_c)


def render_mesh_view(verts, faces, normals, vert_rgb, R, T, Cc, light_dir, bg, k00, k11, H, W,
                     perspective_correct=True, cull_backfaces=False, p2f=None, z_clip=None):
    """Differentiable single-view mesh render (K=1).  If p2f is given the raster step is skipped
    and barycentrics are recomputed differentiably from the face ids (that is what autograd does
    through _RasterizeFaceVerts: the index is a constant).  z_clip: near-plane cull + clip ([upstream] clip.py);
    with it the rasterizer always runs (on the clipped face list) and p2f must be None."""
    ndc = project_perspective(verts, R, T, k00, k11)
    fv = ndc[faces]
    yf = pix_centers(H, verts.dtype)[:, None].expand(H, W)
    xf = pix_centers(W, verts.dtype)[None, :].expand(H, W)
    if z_clip is not None:
        assert p2f is None
        fvc, c2u, conv = clip_faces(fv, z_clip, perspective_correct)
        with torch.no_grad():
            p2c, _, _ = rasterize_meshes_naive(fvc, H, W, 1, perspective_correct, cull_backfaces)
        p2c = p2c[..., 0]
        sel = p2c.clamp_min(0)
        bc = bary_coords(xf, yf, fvc[sel], perspective_correct)
        b = (conv[sel] * bc[..., None, :]).sum(-1)          # convert_clipped_rasterization_to_original_faces
        p2f = torch.where(p2c >= 0, c2u[sel], torch.full_like(p2c, -1))
        img = phong_shade(b, p2f, verts, faces, normals, vert_rgb, light_dir, Cc, bg)
        return img, p2f
    if p2f is None:
        with torch.no_grad():
            p2f, _, _ = rasterize_meshes_naive(fv, H, W, 1, perspective_correct, cull_backfaces)
        p2f = p2f[..., 0]
    b = bary_coords(xf, yf, fv[p2f.clamp_min(0)], perspective_correct)
    img = phong_shade(b, p2f, verts, faces, normals, vert_rgb, light_dir, Cc, bg)
    return img, p2f


def rasterize_points_naive(pts, radius, H, W, K):
    """One view.  pts (P,3) ndc -> idx (H,W,K) long, zbuf, dists2."""
    dt = pts.dtype
    yf = pix_centers(H, dt)[:, None, None]
    xf = pix_centers(W, dt)[None, :, None]
    dx = pts[None, None, :, 0] - xf
    dy = pts[None, None, :, 1] - yf
    d2 = dx * dx + dy * dy
    r2 = torch.tensor(radius, dtype=dt) * torch.tensor(radius, dtype=dt)
    hit = (d2 < r2) & ~(pts[None, None, :, 2] < 0)
    key = torch.where(hit, pts[None, None, :, 2].expand_as(d2), torch.full_like(d2, float("inf")))
    order = torch.sort(key, dim=-1, stable=True)
    idx = order.indices[..., :K]; zs = order.values[..., :K]
    if idx.shape[-1] < K:
        pad = K - idx.shape[-1]
        idx = torch.cat([idx, idx.new_zeros(H, W, pad)], -1)
        zs = torch.cat([zs, zs.new_full((H, W, pad), float("inf"))], -1)
    valid = torch.isfinite(zs)
    d2s = torch.gather(d2, 2, idx)
    return (torch.where(valid, idx, torch.full_like(idx, -1)), torch.where(valid, zs, torch.full_like(zs, -1.0)),
            torch.where(valid, d2s, torch.full_like(d2s, -1.0)))


def composite(idx, alphas, feats, alpha_mode):
    """idx/alphas (K,H,W), feats (3,P) -> (3,H,W).  [upstream] compositing.{norm_weighted_sum,alpha_composite}."""
    valid = (idx >= 0).to(alphas.dtype)
    f = feats[:, idx.clamp_min(0)]                  # (3,K,H,W)
    a = alphas * valid
    if alpha_mode:
        one_minus = torch.where(idx >= 0, 1 - alphas, torch.ones_like(alphas))
        cum = torch.cumprod(torch.cat([torch.ones_like(one_minus[:1]), one_minus[:-1]], 0), 0)
        return (f * (a * cum)[None]).sum(1)
    t = a.sum(0).clamp_min(1e-4)
    return (f * a[None]).sum(1) / t[None]


def render_points_view(pts_world, feats, R, T, inv_dist, radius, bg, H, W, K, alpha_mode, idx=None):
    """Differentiable single-view point render: (X/d) R + T, orthographic, compositor, background."""
    p = (pts_world * inv_dist) @ R + T
    if idx is None:
        with torch.no_grad():
            idx, _, _ = rasterize_points_naive(p, radius, H, W, K)
    yf = pix_centers(H, p.dtype)[:, None, None]
    xf = pix_centers(W, p.dtype)[None, :, None]
    sel = p[idx.clamp_min(0)]                       # (H,W,K,3)
    d2 = (sel[..., 0] - xf) ** 2 + (sel[..., 1] - yf) ** 2
    w = 1 - d2 / (radius * radius)
    img = composite(idx.permute(2, 0, 1), w.permute(2, 0, 1), feats, alpha_mode)
    fg = (idx[..., 0] >= 0)[None]
    return torch.where(fg, img, bg[:, None, None].expand_as(img)), idx


# --------------------------------------------------------------------------------------------------
# Soft rasterization (SURVEY 8f N3; renderer.py:4-6 imports SoftPhongShader / SoftSilhouetteShader, :91-92 blur_radius /
# faces_per_pixel).  [upstream] rasterize_meshes_cpu.cpp with blur_radius > 0 and clip_barycentric_coords, geometry_utils.h
# PointTriangleDistanceForward / BarycentricClipForward, renderer/blending.py softmax_rgb_blend / sigmoid_alpha_blend.
# --------------------------------------------------------------------------------------------------
def point_segment_dist2(px, py, ax, ay, bx, by):
    """[upstream] PointLineDistanceForward: squared distance to the SEGMENT a-b (degenerate: distance to b)."""
    dx, dy = bx - ax, by - ay
    l2 = dx * dx + dy * dy
    t = (dx * (px - ax) + dy * (py - ay)) / torch.where(l2 <= K_EPS, torch.ones_like(l2), l2)
    tt = t.clamp(0.0, 1.0)
    qx, qy = ax + tt * dx, ay + tt * dy
    d = (px - qx) * (px - qx) + (py - qy) * (py - qy)
    return torch.where(l2 <= K_EPS, (px - bx) * (px - bx) + (py - by) * (py - by), d)


def point_triangle_dist2(px, py, fv):
    """[upstream] PointTriangleDistanceForward: min over the edges (v0,v1), (v0,v2), (v1,v2)."""
    x0, y0, x1, y1, x2, y2 = fv[..., 0, 0], fv[..., 0, 1], fv[..., 1, 0], fv[..., 1, 1], fv[..., 2, 0], fv[..., 2, 1]
    e01 = point_segment_dist2(px, py, x0, y0, x1, y1)
    e02 = point_segment_dist2(px, py, x0, y0, x2, y2)
    e12 = point_segment_dist2(px, py, x1, y1, x2, y2)
    return torch.minimum(torch.minimum(e01, e02), e12)


def bary_clip(b):
    """[upstream] BarycentricClipForward: clamp below at 0, renormalise (sum floored at 1e-5)."""
    w = b.clamp_min(0.0)
    return w / w.sum(-1, keepdim=True).clamp_min(1e-5)


def soft_fragments(px, py, fv, perspective_correct, clip_bary):
    """Per (pixel, face) quantities of the blurred rasterizer: unclipped barycentrics (inside test), the barycentrics the
    fragment carries, depth and the SIGNED squared edge distance (negative inside)."""
    b = bary_coords(px, py, fv, perspective_correct)
    bc = bary_clip(b) if clip_bary else b
    pz = (bc * fv[..., 2]).sum(-1)
    d = point_triangle_dist2(px, py, fv)
    inside = (b > 0).all(-1)
    return b, bc, pz, torch.where(inside, -d, d), inside


def rasterize_meshes_soft(face_verts, H, W, K, blur_radius, perspective_correct=True, clip_bary=None, cull_backfaces=False,
                          z_clip=None, return_sub=False):
    """One view, blur_radius >= 0 (squared NDC units, as upstream).  -> p2f (H,W,K) long, zbuf, bary (H,W,K,3), dists (signed),
    all -1 padded.  A face is a fragment of a pixel when the pixel lies in its bbox grown by sqrt(blur_radius) and is inside it
    or closer than blur_radius (squared) to an edge; the K lexicographically smallest (z, face) win.
    z_clip: faces crossing the plane z = z_clip are clipped first (clip_faces, as the hard path) and their sub-triangles are
    rasterized with blur; bary is then converted back to the original face (after the clip of the sub-triangle's barycentrics),
    zbuf and the signed dists are the sub-triangle's.  A sub-triangle competes under its ORIGINAL face id by the same (z, id)
    rule as any candidate, so a pixel near the cut between the two halves of a quad may hold the face twice, nearer half first.
    That is the CUDA rasterizer's rule; upstream's rasterizer merges the two halves instead (clipped_faces_neighbor_idx),
    which is not reproduced.  return_sub: also -> p2c (H,W,K), the fragment's index in clip_faces' list (-1 padded)."""
    if clip_bary is None:
        clip_bary = blur_radius > 0
    dt = face_verts.dtype
    yf = pix_centers(H, dt, W)[:, None, None]
    xf = pix_centers(W, dt, H)[None, :, None]
    Fn0 = face_verts.shape[0]
    if z_clip is not None:
        face_verts, c2u, conv = clip_faces(face_verts, z_clip, perspective_correct)
    else:
        c2u, conv = torch.arange(Fn0), None
    fv = face_verts[None, None]
    b, bc, pz, sd, inside = soft_fragments(xf, yf, fv, perspective_correct, clip_bary)
    x, y, z = face_verts[..., 0], face_verts[..., 1], face_verts[..., 2]
    area = _edge(x[:, 0], y[:, 0], x[:, 1], y[:, 1], x[:, 2], y[:, 2])
    ok = ~((area <= K_EPS) & (area >= -K_EPS))
    if cull_backfaces:
        ok &= ~(area < 0)
    ok &= ~(z.min(dim=1).values < K_EPS)
    r = math.sqrt(blur_radius)
    inbox = (xf <= x.max(1).values + r) & (xf >= x.min(1).values - r) & (yf <= y.max(1).values + r) & (yf >= y.min(1).values - r)
    hit = ok[None, None] & inbox & ~(pz < 0) & (inside | (sd < blur_radius))
    key = torch.where(hit, pz, torch.full_like(pz, float("inf")))
    # stable sort by z: ties in clip_faces' order, i.e. by original face id (c2u is non-decreasing)
    order = torch.sort(key, dim=-1, stable=True)
    if z_clip is not None and order.values.shape[-1] > 1:
        # two sub-triangles of one face with the same depth make the same (z, id) key: one fragment
        oid = c2u[order.indices]
        dup = (order.values[..., 1:] == order.values[..., :-1]) & (oid[..., 1:] == oid[..., :-1]) & torch.isfinite(order.values[..., 1:])
        if dup.any():
            vals = order.values.clone()
            vals[..., 1:][dup] = float("inf")
            o2 = torch.sort(vals, dim=-1, stable=True)
            order = torch.return_types.sort((o2.values, torch.gather(order.indices, -1, o2.indices)))
    Fn = face_verts.shape[0]
    idx, zs = order.indices[..., :K], order.values[..., :K]
    if Fn < K:
        idx = torch.cat([idx, idx.new_zeros(H, W, K - Fn)], -1)
        zs = torch.cat([zs, zs.new_full((H, W, K - Fn), float("inf"))], -1)
    valid = torch.isfinite(zs)
    g = idx.clamp(0, max(Fn - 1, 0))
    p2f = torch.where(valid, c2u[g] if Fn else g, torch.full_like(idx, -1))
    zbuf = torch.where(valid, zs, torch.full_like(zs, -1.0))
    bsel = torch.gather(bc, 2, g[..., None].expand(H, W, K, 3)) if Fn else torch.zeros((H, W, K, 3), dtype=dt)
    if conv is not None and Fn:
        bsel = (conv[g] * bsel[..., None, :]).sum(-1)      # convert_clipped_rasterization_to_original_faces
    bary = torch.where(valid[..., None], bsel, torch.full((H, W, K, 3), -1.0, dtype=dt))
    dists = torch.where(valid, torch.gather(sd, 2, g), torch.full_like(zs, -1.0)) if Fn else torch.full_like(zs, -1.0)
    if return_sub:
        return p2f, zbuf, bary, dists, torch.where(valid, idx, torch.full_like(idx, -1))
    return p2f, zbuf, bary, dists


def phong_colors(bary, p2f, verts, faces, normals, vert_rgb, light_dir, cam_center, ambient=0.5, diffuse=0.3, specular=0.2, shininess=64):
    """[upstream] phong_shading for EVERY fragment: bary (H,W,K,3), p2f (H,W,K) -> colours (H,W,K,3); empty fragments
    interpolate zeros (interpolate_face_attributes masks them), which shades to 0."""
    fg = (p2f >= 0)[..., None]
    f = p2f.clamp_min(0)
    z3 = torch.zeros((), dtype=bary.dtype)
    P = torch.where(fg, (bary[..., None] * verts[faces][f]).sum(-2), z3)
    Nn = torch.where(fg, (bary[..., None] * normals[faces][f]).sum(-2), z3)
    tex = torch.where(fg, (bary[..., None] * vert_rgb[faces][f]).sum(-2), z3)
    n = F.normalize(Nn, p=2, dim=-1, eps=1e-6)
    l = F.normalize(light_dir.expand_as(n), p=2, dim=-1, eps=1e-6)
    cosang = (n * l).sum(-1)
    mask = (cosang > 0).to(bary.dtype)
    v = F.normalize(cam_center - P, p=2, dim=-1, eps=1e-6)
    r = -l + 2 * (cosang[..., None] * n)
    alpha = F.relu((v * r).sum(-1)) * mask
    return (ambient + diffuse * F.relu(cosang))[..., None] * tex + (specular * torch.pow(alpha, shininess))[..., None]


def softmax_rgb_blend(colors, p2f, zbuf, dists, bg, sigma=1e-4, gamma=1e-4, znear=1.0, zfar=100.0):
    """[upstream] blending.softmax_rgb_blend -> (H,W,4) RGBA."""
    eps = 1e-10
    mask = (p2f >= 0).to(colors.dtype)
    prob = torch.sigmoid(-dists / sigma) * mask
    alpha = torch.prod(1.0 - prob, dim=-1)
    z_inv = (zfar - zbuf) / (zfar - znear) * mask
    z_inv_max = torch.max(z_inv, dim=-1).values[..., None].clamp(min=eps)
    wnum = prob * torch.exp((z_inv - z_inv_max) / gamma)
    delta = torch.exp((eps - z_inv_max) / gamma).clamp(min=eps)
    denom = wnum.sum(-1)[..., None] + delta
    rgb = ((wnum[..., None] * colors).sum(-2) + delta * bg) / denom
    return torch.cat([rgb, (1.0 - alpha)[..., None]], -1)


def sigmoid_alpha_blend(colors, p2f, dists, sigma=1e-4):
    """[upstream] blending.sigmoid_alpha_blend -> (H,W,4): RGB of the nearest fragment, alpha = 1 - prod(1 - sigmoid(-d / sigma))."""
    mask = (p2f >= 0).to(colors.dtype)
    prob = torch.sigmoid(-dists / sigma) * mask
    alpha = torch.prod(1.0 - prob, dim=-1)
    return torch.cat([colors[..., 0, :], (1.0 - alpha)[..., None]], -1)


def render_mesh_view_soft(verts, faces, normals, vert_rgb, R, T, Cc, light_dir, bg, k00, k11, H, W, K, blur_radius, shader,
                          sigma=1e-4, gamma=1e-4, perspective_correct=True, clip_bary=None, p2f=None, cull_backfaces=False,
                          z_clip=None, p2c=None):
    """Differentiable single-view soft render -> (4,H,W) RGBA + fragments.  shader: "soft_phong" | "soft_silhouette".
    The raster step (which face is fragment k of a pixel) is not differentiated; barycentrics, depth and signed distances are
    recomputed differentiably from the face ids (what autograd does through _RasterizeFaceVerts).
    z_clip: near-plane clipping as rasterize_meshes_soft(z_clip=...); the fragments are then given (or found) as p2c, indices
    into clip_faces' list, and everything is recomputed on the sub-triangles and chained through the clipping ([upstream]
    clip.py under autograd); p2f must be None."""
    if clip_bary is None:
        clip_bary = blur_radius > 0
    ndc = project_perspective(verts, R, T, k00, k11)
    fv = ndc[faces]
    yf = pix_centers(H, verts.dtype, W)[:, None, None].expand(H, W, K)
    xf = pix_centers(W, verts.dtype, H)[None, :, None].expand(H, W, K)
    m1 = torch.full((), -1.0, dtype=verts.dtype)
    if z_clip is not None:
        assert p2f is None
        fvc, c2u, conv = clip_faces(fv, z_clip, perspective_correct)
        if p2c is None:
            with torch.no_grad():
                p2c = rasterize_meshes_soft(fv, H, W, K, blur_radius, perspective_correct, clip_bary, cull_backfaces, z_clip,
                                            return_sub=True)[4]
        assert int(p2c.max()) < fvc.shape[0]
        valid = p2c >= 0
        sel = p2c.clamp_min(0)
        _, bcs, pz, sd, _ = soft_fragments(xf, yf, fvc[sel], perspective_correct, clip_bary)
        bc = (conv[sel] * bcs[..., None, :]).sum(-1)
        p2f = torch.where(valid, c2u[sel], torch.full_like(p2c, -1))
    else:
        if p2f is None:
            with torch.no_grad():
                p2f, _, _, _ = rasterize_meshes_soft(fv, H, W, K, blur_radius, perspective_correct, clip_bary, cull_backfaces)
        valid = p2f >= 0
        _, bc, pz, sd, _ = soft_fragments(xf, yf, fv[p2f.clamp_min(0)], perspective_correct, clip_bary)
    bary = torch.where(valid[..., None], bc, m1); zbuf = torch.where(valid, pz, m1); dists = torch.where(valid, sd, m1)
    if shader == "soft_silhouette":
        img = sigmoid_alpha_blend(torch.ones_like(bary), p2f, dists, sigma)
    else:
        col = phong_colors(bary, p2f, verts, faces, normals, vert_rgb, light_dir, Cc)
        img = softmax_rgb_blend(col, p2f, zbuf, dists, bg, sigma, gamma)
    return img.permute(2, 0, 1), dict(pix_to_face=p2f, zbuf=zbuf, bary=bary, dists=dists)


# ---------------------------------------------------------------------------------------------------
# The regulariser behind the renderer: ops.py:138-178 restated with the same torch / torchvision calls in the same order (this
# one CAN be pinned: the reference's implementation is nothing but torch + torchvision library calls; the reference module itself
# does not import here only because of `torch._six`, ops.py:9).
def applied_transforms(images_batch, crop_ratio=0.3):
    """ops.py:138-146."""
    from torchvision.transforms import RandomCrop, RandomHorizontalFlip
    N, C, H, W = images_batch.shape
    padd = torch.nn.ReplicationPad2d(int((1 + crop_ratio) * H) - H)
    images_batch = RandomHorizontalFlip()(images_batch)
    images_batch = RandomCrop(H)(padd(images_batch))
    return images_batch


def regularize_rendered_views(rendered_images, dropout_p=0, augment_training=False, crop_ratio=0.3):
    """ops.py:168-176 regualarize_rendered_views: dropout2d on the 5-D (B, M, C, H, W) tensor, then the batchwise transforms on
    the views flattened to (B*M, C, H, W) (super_batched_op(1, ...), ops.py:149-153 with util.batch_tensor / unbatch_tensor)."""
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")      # torch >= 1.12 warns that a 5-D input makes dropout2d a feature dropout over dim 1
        rendered_images = F.dropout2d(rendered_images, p=dropout_p, training=True)
    if augment_training:
        B, M = rendered_images.shape[:2]
        flat = rendered_images.reshape(B * M, *rendered_images.shape[2:])
        rendered_images = applied_transforms(flat, crop_ratio=crop_ratio).reshape(B, M, *rendered_images.shape[2:])
    return rendered_images


def regularize_gather(x, scale, flip, sy, sx):
    """The composed form the CUDA kernel evaluates (mvtn_b200/csrc/mvr_augment.cu):
    out[n,c,y,x] = scale[n] * in[n,c,clamp(y+sy), fx(clamp(x+sx))], fx(u) = W-1-u under a flip."""
    B, M, C, H, W = x.shape
    yi = (torch.arange(H, device=x.device) + sy).clamp(0, H - 1)
    xi = (torch.arange(W, device=x.device) + sx).clamp(0, W - 1)
    if flip:
        xi = W - 1 - xi
    out = x[..., yi, :][..., xi]
    if scale is not None:
        out = out * scale.to(x.dtype).reshape(B, M, 1, 1, 1)
    return out
