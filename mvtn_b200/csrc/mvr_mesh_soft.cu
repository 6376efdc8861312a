// mvr_mesh_soft.cu -- soft shading of K rasterized fragments per pixel and its backward (SURVEY 8f N3; renderer.py:4-6
// imports SoftPhongShader / SoftSilhouetteShader, :91-92 exposes blur_radius / faces_per_pixel).
//
//   forward : the blurred rasterizer is the ordinary one (mesh_scatter_kernel + exact shade pass, K layers by peeling) with
//             blur_radius > 0 / clipped barycentrics (raster_soft); mesh_soft_blend_kernel then turns the K fragments of a
//             pixel into RGBA: [upstream] blending.softmax_rgb_blend over per-fragment Phong colours (SoftPhongShader) or
//             blending.sigmoid_alpha_blend (SoftSilhouetteShader).
//   backward: mesh_soft_backward_kernel -- per pixel, per fragment: recompute (barycentrics, depth, signed edge distance,
//             colour) from the projected vertices, then d RGBA -> blend weights -> (colour, zbuf, dists) -> Phong /
//             [upstream] RasterizeMeshesBackward (BarycentricClipBackward, perspective correction, edge functions,
//             PointTriangleDistanceBackward) -> NDC vertices -> (dR, dT, dC); per-warp partials, fixed-order sum (deterministic).
//             <GV = true> also returns, per fragment, d/d position of the three vertices of its ORIGINAL face (projection
//             chain through R, plus Phong's interpolated-position term) and d/d their unit normals (Phong, soft_phong only),
//             scattered with one plain atomicAdd per value (as [upstream] RasterizeMeshesBackward): the vertex gradients are
//             tolerance-level, their summation order is not fixed.  The camera arithmetic is the same in both instances.
// Tolerance-compared against the torch restatement (oracle/torch_ref.py render_mesh_view_soft + vertex_normals, autograd): not
// on MVTN's default path, written for clarity rather than tuned.
#include "mvr_mesh.cuh"

namespace mvr {

struct SoftParams {
  int mode;                // 0 = softmax_rgb_blend over Phong colours, 1 = sigmoid_alpha_blend (silhouette)
  float sigma, gamma, znear, zfar, blur;
  const float* zbuf; const float* bary; const float* dists;      // forward: the rasterizer's fragments (n, H, W, K[, 3])
  float* rgba;             // forward out: (n, 4, H, W)
  const float* grad_rgba;  // backward in
  float* grad_verts; float* grad_normals;      // backward out (GV): (Vtot,3) accumulated, either may be NULL
};

constexpr float SOFT_EPS = 1e-10f;

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// colour of one fragment (soft_phong) from its face and barycentrics
__device__ __forceinline__ void fragment_colour(const MeshParams& p, int voff, const int4 fi, const float bb[3], const ShadeCtx& sc,
                                                float out[3]) {
  float4 X0, X1, X2, N0, N1, N2, c0, c1, c2;
  gather_xn(p.xn8, voff + fi.x, X0, N0); gather_xn(p.xn8, voff + fi.y, X1, N1); gather_xn(p.xn8, voff + fi.z, X2, N2);
  if (p.flags & MVR_RGB_PER_ELEMENT) { c0 = __ldg(p.rgb4 + voff + fi.x); c1 = __ldg(p.rgb4 + voff + fi.y); c2 = __ldg(p.rgb4 + voff + fi.z); }
  else { c0 = c1 = c2 = make_float4(__ldg(p.obj_rgb), __ldg(p.obj_rgb + 1), __ldg(p.obj_rgb + 2), 0.f); }
  phong_pixel<true>(bb, X0, X1, X2, N0, N1, N2, c0, c1, c2, sc, out);
}

// grid: x = 256-pixel chunks of the image, y = view m, z = object b
__global__ void __launch_bounds__(MVR_THREADS) mesh_soft_blend_kernel(const MeshParams p, const SoftParams sp) {
  const int b = blockIdx.z, m = blockIdx.y, n = b * p.M + m;
  const int HW = p.H * p.W, pix = blockIdx.x * MVR_THREADS + threadIdx.x;
  if (pix >= HW) return;
  const int K = p.K;
  const size_t fo = ((size_t)n * HW + pix) * K;
  const int f0 = p.face_off[b], voff = p.vert_off[b];
  const float zscale = 1.0f / (sp.zfar - sp.znear);
  float zmax = 0.f;
  for (int k = 0; k < K; ++k)
    if (p.pix_to_face[fo + k] >= 0) zmax = fmaxf(zmax, (sp.zfar - sp.zbuf[fo + k]) * zscale);
  zmax = fmaxf(zmax, SOFT_EPS);
  const ShadeCtx sc = load_shade_ctx(p.light, p.light_stride, p.Cc, n);
  float num[3] = {0.f, 0.f, 0.f}, den = 0.f, keep = 1.0f, first[3] = {1.f, 1.f, 1.f};
  for (int k = 0; k < K; ++k) {
    const int fid = p.pix_to_face[fo + k];
    if (fid < 0) continue;
    const float prob = sigmoidf_(-sp.dists[fo + k] / sp.sigma);
    keep *= 1.0f - prob;
    if (sp.mode == 0) {
      const float bb[3] = {sp.bary[3 * (fo + k)], sp.bary[3 * (fo + k) + 1], sp.bary[3 * (fo + k) + 2]};
      float col[3];
      fragment_colour(p, voff, __ldg(p.faces4 + f0 + fid), bb, sc, col);
      const float w = prob * expf(((sp.zfar - sp.zbuf[fo + k]) * zscale - zmax) / sp.gamma);
      num[0] += w * col[0]; num[1] += w * col[1]; num[2] += w * col[2];
      den += w;
    }
  }
  float* o = sp.rgba + (size_t)n * 4 * HW + pix;
  if (sp.mode == 0) {
    const float delta = fmaxf(expf((SOFT_EPS - zmax) / sp.gamma), SOFT_EPS);
    const float inv = 1.0f / (den + delta);
    o[0] = (num[0] + delta * __ldg(p.bg_rgb)) * inv;
    o[(size_t)HW] = (num[1] + delta * __ldg(p.bg_rgb + 1)) * inv;
    o[2 * (size_t)HW] = (num[2] + delta * __ldg(p.bg_rgb + 2)) * inv;
  } else {      // SoftSilhouetteShader: colours = ones
    o[0] = first[0]; o[(size_t)HW] = first[1]; o[2 * (size_t)HW] = first[2];
  }
  o[3 * (size_t)HW] = 1.0f - keep;
}

// [upstream] PointLineDistanceBackward: d (squared distance of p to segment a-b) -> (ga, gb), scaled by g
__device__ __forceinline__ void point_line_dist2_bwd(float px, float py, float ax, float ay, float bx, float by, float g,
                                                     float& gax, float& gay, float& gbx, float& gby) {
  const float dx = bx - ax, dy = by - ay;
  const float l2 = dx * dx + dy * dy;
  if (l2 <= MVR_K_EPS) { gax = 0.f; gay = 0.f; gbx = -2.f * (px - bx) * g; gby = -2.f * (py - by) * g; return; }
  const float t = (dx * (px - ax) + dy * (py - ay)) / l2;
  const float tt = fminf(fmaxf(t, 0.f), 1.f);
  const float qx = ax + tt * dx, qy = ay + tt * dy;
  // d = |p - q|^2, q = (1 - tt) a + tt b; the dependence through tt vanishes (optimal or clamped)
  const float ex = 2.f * (qx - px) * g, ey = 2.f * (qy - py) * g;
  gax = (1.f - tt) * ex; gay = (1.f - tt) * ey; gbx = tt * ex; gby = tt * ey;
}

// One fragment of a pixel, recomputed from the projected vertices: raster_soft on its face, or -- a face crossing the near
// plane (p.z_clip, while the projection has found a vertex behind it) -- on the sub-triangle the forward's scatter kept
// (pick_sub_soft), with the barycentrics mapped back to the face (conv_bary) as mvr_mesh_shade_clipped_kernel writes them.
struct SoftFrag {
  Face g;            // the triangle rasterized: the face, or sub-triangle s of its clipping
  int s;             // -1: not clipped
  SoftHit h;         // barycentrics (raw, carried), depth and signed distance on g
  float bb[3];       // barycentrics on the original face (colour)
};
// rank: how many entries of the same face precede this one in the pixel's K-list (a clipped face may hold two)
__device__ __forceinline__ bool soft_fragment(const MeshParams& p, const Face& fc, bool persp, bool clipb, bool clip_on, float xf,
                                              float yf, int rank, ClipSub& cs, SoftFrag& fr) {
  fr.s = -1;
  if (clip_on && face_straddles(fc, p.z_clip)) {
    clip_face(fc, p.z_clip, persp, cs);
    fr.s = pick_sub_soft(cs, p.flags, persp, clipb, p.blur_radius, p.blur_r, xf, yf, 0u, rank, fr.h);
    if (fr.s < 0) return false;
    fr.g = cs.f[fr.s];
    conv_bary(cs.conv[fr.s], fr.h.bc, fr.bb);
    return true;
  }
  fr.g = fc;
  raster_soft(fc, face_edges(fc), persp, clipb, xf, yf, fr.h.bu, fr.h.bc, fr.h.pz, fr.h.sd, fr.h.inside);
  fr.bb[0] = fr.h.bc[0]; fr.bb[1] = fr.h.bc[1]; fr.bb[2] = fr.h.bc[2];
  return true;
}

__device__ __forceinline__ int rank_in_list(const int* list, int k, int fid) {
  int r = 0;
  for (int j = 0; j < k; ++j) r += list[j] == fid;
  return r;
}

// One fragment of view n: push (g_colour, g_zbuf, g_sdist) back to the camera accumulators acc[15]; GV: also to the vertices
// of the original face (sp.grad_verts: projection chain + Phong's interpolated position; sp.grad_normals: Phong's normal term).
template <bool GV>
__device__ __forceinline__ void soft_fragment_backward(const MeshParams& p, const SoftParams& sp, int n, int voff, const int4 fi, const Face& fc,
                                                       const SoftFrag& fr, const ClipSub& cs, bool persp, bool clipb, float xf, float yf,
                                                       const ShadeCtx& sc, const float gcol[3], float gz, float gsd, bool with_colour,
                                                       float acc[16]) {
  const Face& g = fr.g;
  float4 X0, X1, X2, N0, N1, N2;
  gather_xn(p.xn8, voff + fi.x, X0, N0); gather_xn(p.xn8, voff + fi.y, X1, N1); gather_xn(p.xn8, voff + fi.z, X2, N2);
  const int vid[3] = {fi.x, fi.y, fi.z};
  float gbb[3] = {0.f, 0.f, 0.f};      // w.r.t. the barycentrics on the original face
  float gP[3] = {0.f, 0.f, 0.f};       // GV: w.r.t. the interpolated position P = sum_i bb_i X_i (= -d/d camera centre)
  if (with_colour) {
    float4 c0, c1, c2;
    if (p.flags & MVR_RGB_PER_ELEMENT) { c0 = __ldg(p.rgb4 + voff + fi.x); c1 = __ldg(p.rgb4 + voff + fi.y); c2 = __ldg(p.rgb4 + voff + fi.z); }
    else { c0 = c1 = c2 = make_float4(__ldg(p.obj_rgb), __ldg(p.obj_rgb + 1), __ldg(p.obj_rgb + 2), 0.f); }
    float gv[3], gN[3];
    phong_backward(fr.bb, X0, X1, X2, N0, N1, N2, c0, c1, c2, sc, gcol[0], gcol[1], gcol[2], gbb, gv, gN);
    acc[12] += gv[0]; acc[13] += gv[1]; acc[14] += gv[2];      // dC
    if (GV) {
      gP[0] = -gv[0]; gP[1] = -gv[1]; gP[2] = -gv[2];
      if (sp.grad_normals)      // Nn = sum_i bb_i N_i
        for (int i = 0; i < 3; ++i) {
          float* o = sp.grad_normals + 3 * (size_t)(voff + vid[i]);
          atomicAdd(o + 0, fr.bb[i] * gN[0]); atomicAdd(o + 1, fr.bb[i] * gN[1]); atomicAdd(o + 2, fr.bb[i] * gN[2]);
        }
    }
  }
  // w.r.t. the barycentrics carried on g: through the conversion bb_j = sum_k conv[3 j + k] bc_k for a sub-triangle
  float gbc[3] = {gbb[0], gbb[1], gbb[2]};
  if (fr.s >= 0) {
    const float* cv = cs.conv[fr.s];
    for (int k = 0; k < 3; ++k) gbc[k] = cv[k] * gbb[0] + cv[3 + k] * gbb[1] + cv[6 + k] * gbb[2];
  }
  // zbuf = bc . z
  float gq[9];
  gbc[0] += gz * g.z0; gbc[1] += gz * g.z1; gbc[2] += gz * g.z2;
  float gb[3] = {gbc[0], gbc[1], gbc[2]};
  bool orth = false;
  const float* bu = fr.h.bu;
  const float* bc = fr.h.bc;
  if (clipb) {      // [upstream] BarycentricClipBackward: bc = w / s, w = max(b, 0), s = max(sum w, 1e-5)
    const float w0 = fmaxf(bu[0], 0.f), w1 = fmaxf(bu[1], 0.f), w2 = fmaxf(bu[2], 0.f);
    const float ssum = (w0 + w1) + w2;
    const float s = fmaxf(ssum, 1e-5f), is = 1.0f / s;
    const float dot = ssum > 1e-5f ? (gbc[0] * bc[0] + gbc[1] * bc[1] + gbc[2] * bc[2]) : 0.f;
    gb[0] = bu[0] > 0.f ? (gbc[0] - dot) * is : 0.f;
    gb[1] = bu[1] > 0.f ? (gbc[1] - dot) * is : 0.f;
    gb[2] = bu[2] > 0.f ? (gbc[2] - dot) * is : 0.f;
    orth = ssum > 1e-5f;      // sum_i bu_i gb_i = dot - dot sum(bc) = 0
  }
  raster_backward(g, persp, xf, yf, gb, gq, orth);
  gq[2] += gz * bc[0]; gq[5] += gz * bc[1]; gq[8] += gz * bc[2];
  // signed distance: sd = inside ? -d : d over the nearest edge ([upstream] PointTriangleDistanceBackward)
  if (gsd != 0.f) {
    const float gs = fr.h.inside ? -gsd : gsd;
    const float e01 = point_line_dist2(xf, yf, g.x0, g.y0, g.x1, g.y1);
    const float e02 = point_line_dist2(xf, yf, g.x0, g.y0, g.x2, g.y2);
    const float e12 = point_line_dist2(xf, yf, g.x1, g.y1, g.x2, g.y2);
    float ax, ay, bx, by;
    if (e01 <= e02 && e01 <= e12) { point_line_dist2_bwd(xf, yf, g.x0, g.y0, g.x1, g.y1, gs, ax, ay, bx, by); gq[0] += ax; gq[1] += ay; gq[3] += bx; gq[4] += by; }
    else if (e02 <= e01 && e02 <= e12) { point_line_dist2_bwd(xf, yf, g.x0, g.y0, g.x2, g.y2, gs, ax, ay, bx, by); gq[0] += ax; gq[1] += ay; gq[6] += bx; gq[7] += by; }
    else { point_line_dist2_bwd(xf, yf, g.x1, g.y1, g.x2, g.y2, gs, ax, ay, bx, by); gq[3] += ax; gq[4] += ay; gq[6] += bx; gq[7] += by; }
  }
  if (fr.s >= 0) {      // sub-triangle -> original face ([upstream] clip.py under autograd), as the hard path's clipped pixels
    float gfv[9];
    clip_face_backward(fc, p.z_clip, persp, cs.info, fr.s, gq, gbb, bc, gfv);
    for (int i = 0; i < 9; ++i) gq[i] = gfv[i];
  }
  // projection backward + X R + T backward
  const float xn[3] = {fc.x0, fc.x1, fc.x2}, yn[3] = {fc.y0, fc.y1, fc.y2}, zv[3] = {fc.z0, fc.z1, fc.z2};
  const float4 Xs[3] = {X0, X1, X2};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float iz = 1.0f / zv[i];
    const float gpx = gq[3 * i] * p.k00 * iz, gpy = gq[3 * i + 1] * p.k11 * iz;
    const float gpz = gq[3 * i + 2] - (gq[3 * i] * xn[i] + gq[3 * i + 1] * yn[i]) * iz;
    acc[0] += Xs[i].x * gpx; acc[1] += Xs[i].x * gpy; acc[2] += Xs[i].x * gpz;
    acc[3] += Xs[i].y * gpx; acc[4] += Xs[i].y * gpy; acc[5] += Xs[i].y * gpz;
    acc[6] += Xs[i].z * gpx; acc[7] += Xs[i].z * gpy; acc[8] += Xs[i].z * gpz;
    acc[9] += gpx; acc[10] += gpy; acc[11] += gpz;
    if (GV && sp.grad_verts) {      // X_view = X R + T: d/d X = R (gpx, gpy, gpz); P = sum_i bb_i X_i
      const float* r = p.R + 9 * (size_t)n;
      float* o = sp.grad_verts + 3 * (size_t)(voff + vid[i]);
      atomicAdd(o + 0, (__ldg(r + 0) * gpx + __ldg(r + 1) * gpy + __ldg(r + 2) * gpz) + fr.bb[i] * gP[0]);
      atomicAdd(o + 1, (__ldg(r + 3) * gpx + __ldg(r + 4) * gpy + __ldg(r + 5) * gpz) + fr.bb[i] * gP[1]);
      atomicAdd(o + 2, (__ldg(r + 6) * gpx + __ldg(r + 7) * gpy + __ldg(r + 8) * gpz) + fr.bb[i] * gP[2]);
    }
  }
}

// grid: x = 32x32-pixel tiles, y = view m, z = object b; thread (lane, warp) owns pixels (x0 + lane, y0 + warp + 8 j); one
// 16-float partial per warp at partials[(n * parts_per_view + tile * NWARPS + warp) * 16] (mesh_backward_finish_kernel sums them)
// GV: vertex gradients too (soft_fragment_backward<true>)
template <bool GV>
__global__ void __launch_bounds__(MVR_THREADS) mesh_soft_backward_kernel(const MeshParams p, const SoftParams sp, float* __restrict__ partials,
                                                                         int parts_per_view, int tiles_x) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.z, m = blockIdx.y, n = b * p.M + m, cta = blockIdx.x;
  int tyb, txb;
  tile_rc(cta, tiles_x, tyb, txb);
  const int xi = txb * 32 + lane;
  const int HW = p.H * p.W, K = p.K;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT, clipb = p.flags & MVR_CLIP_BARYCENTRIC;
  const bool clip_on = may_clip(p.wsflags);      // some vertex lies behind the near plane: faces may straddle it
  const ShadeCtx sc = load_shade_ctx(p.light, p.light_stride, p.Cc, n);
  const float zscale = 1.0f / (sp.zfar - sp.znear);
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  for (int j = 0; j < 4; ++j) {
    const int yi = tyb * 32 + warp + 8 * j;
    if (xi >= p.W || yi >= p.H) continue;
    const int pix = yi * p.W + xi;
    const float xf = __ldg(p.tab + xi), yf = __ldg(p.tab + p.W + yi);
    const size_t fo = ((size_t)n * HW + pix) * K;
    const int* list = p.pix_to_face + fo;
    const float* g = sp.grad_rgba + (size_t)n * 4 * HW + pix;
    const float g0 = g[0], g1 = g[(size_t)HW], g2 = g[2 * (size_t)HW], ga = g[3 * (size_t)HW];
    if (g0 == 0.f && g1 == 0.f && g2 == 0.f && ga == 0.f) continue;
    // every loop below skips -1 entries, as mesh_soft_blend_kernel does
    // pass 1: z_inv_max (and which fragment holds it), the product of (1 - prob) with its zeros counted
    float zmax = 0.f, keep_nz = 1.0f;
    int kmax = -1, nzero = 0, kzero = -1;
    for (int k = 0; k < K; ++k) {
      const int fid = list[k];
      if (fid < 0) continue;
      const Face fc = gather_face(pvn, __ldg(p.faces4 + f0 + fid));
      ClipSub cs; SoftFrag fr;
      if (!soft_fragment(p, fc, persp, clipb, clip_on, xf, yf, clip_on ? rank_in_list(list, k, fid) : 0, cs, fr)) continue;
      const float zi = (sp.zfar - fr.h.pz) * zscale;
      if (zi > zmax) { zmax = zi; kmax = k; }
      const float q = 1.0f - sigmoidf_(-fr.h.sd / sp.sigma);
      if (q == 0.f) { ++nzero; kzero = k; } else keep_nz *= q;
    }
    const bool zmax_live = zmax >= SOFT_EPS;
    zmax = fmaxf(zmax, SOFT_EPS);
    // pass 2 (soft_phong): numerator / denominator of the blend
    float num[3] = {0.f, 0.f, 0.f}, den = 0.f, delta = 0.f, inv = 0.f, rgb[3] = {0.f, 0.f, 0.f};
    bool delta_live = false;
    if (sp.mode == 0) {
      for (int k = 0; k < K; ++k) {
        const int fid = list[k];
        if (fid < 0) continue;
        const int4 fi = __ldg(p.faces4 + f0 + fid);
        const Face fc = gather_face(pvn, fi);
        ClipSub cs; SoftFrag fr;
        if (!soft_fragment(p, fc, persp, clipb, clip_on, xf, yf, clip_on ? rank_in_list(list, k, fid) : 0, cs, fr)) continue;
        float col[3];
        fragment_colour(p, voff, fi, fr.bb, sc, col);
        const float w = sigmoidf_(-fr.h.sd / sp.sigma) * expf(((sp.zfar - fr.h.pz) * zscale - zmax) / sp.gamma);
        num[0] += w * col[0]; num[1] += w * col[1]; num[2] += w * col[2]; den += w;
      }
      const float dr = expf((SOFT_EPS - zmax) / sp.gamma);
      delta_live = dr >= SOFT_EPS;
      delta = fmaxf(dr, SOFT_EPS);
      inv = 1.0f / (den + delta);
      rgb[0] = (num[0] + delta * __ldg(p.bg_rgb)) * inv; rgb[1] = (num[1] + delta * __ldg(p.bg_rgb + 1)) * inv; rgb[2] = (num[2] + delta * __ldg(p.bg_rgb + 2)) * inv;
    }
    // pass 3: per-fragment gradients.  g_zmax collects what flows into the maximum and is handed to fragment kmax at the end.
    float gzmax = 0.f;
    if (sp.mode == 0 && delta_live)
      gzmax -= (g0 * (__ldg(p.bg_rgb) - rgb[0]) + g1 * (__ldg(p.bg_rgb + 1) - rgb[1]) + g2 * (__ldg(p.bg_rgb + 2) - rgb[2])) * inv * delta / sp.gamma;
    for (int pass = 0; pass < 2; ++pass) {      // pass 0: every fragment (its own terms); pass 1: fragment kmax gets g_zmax
      for (int k = 0; k < K; ++k) {
        const int fid = list[k];
        if (fid < 0) continue;
        if (pass == 1 && k != kmax) continue;
        const int4 fi = __ldg(p.faces4 + f0 + fid);
        const Face fc = gather_face(pvn, fi);
        ClipSub cs; SoftFrag fr;
        if (!soft_fragment(p, fc, persp, clipb, clip_on, xf, yf, clip_on ? rank_in_list(list, k, fid) : 0, cs, fr)) continue;
        if (pass == 1) {      // z_inv_max = z_inv of this fragment
          if (zmax_live && gzmax != 0.f) {
            const float gcz[3] = {0.f, 0.f, 0.f};
            soft_fragment_backward<GV>(p, sp, n, voff, fi, fc, fr, cs, persp, clipb, xf, yf, sc, gcz, -gzmax * zscale, 0.f, false, acc);
          }
          continue;
        }
        const float prob = sigmoidf_(-fr.h.sd / sp.sigma);
        float gprob = 0.f, gzi = 0.f, gcol[3] = {0.f, 0.f, 0.f};
        // alpha = 1 - prod(1 - prob): d alpha / d prob_k = prod over the others
        {
          const float q = 1.0f - prob;
          float others;
          if (nzero == 0) others = keep_nz / q;
          else if (nzero == 1) others = (k == kzero) ? keep_nz : 0.f;
          else others = 0.f;
          gprob += ga * others;
        }
        if (sp.mode == 0) {
          float col[3];
          fragment_colour(p, voff, fi, fr.bb, sc, col);
          const float E = expf(((sp.zfar - fr.h.pz) * zscale - zmax) / sp.gamma);
          const float w = prob * E;
          gcol[0] = g0 * w * inv; gcol[1] = g1 * w * inv; gcol[2] = g2 * w * inv;
          const float gw = (g0 * (col[0] - rgb[0]) + g1 * (col[1] - rgb[1]) + g2 * (col[2] - rgb[2])) * inv;
          gprob += gw * E;
          const float gE = gw * prob;
          gzi = gE * E / sp.gamma;
          gzmax -= gzi;
        }
        const float gsd = gprob * (-1.0f / sp.sigma) * prob * (1.0f - prob);
        soft_fragment_backward<GV>(p, sp, n, voff, fi, fc, fr, cs, persp, clipb, xf, yf, sc, gcol, -gzi * zscale, gsd, sp.mode == 0, acc);
      }
    }
  }
  float* out = partials + ((size_t)n * parts_per_view + (size_t)cta * NWARPS + warp) * 16;
  const float mine = warp_sum16_transposed(acc);
  if (!(lane & 1)) out[lane >> 1] = mine;
}

}  // namespace mvr

using namespace mvr;

static int fill_params(MeshParams& p, const void* geometry, const int* vert_off, const int* face_off, int B, int M, int64_t total_verts,
                       int64_t total_faces, const float* R, const float* T, const float* Cc, const float* light, int light_stride,
                       const float* obj_rgb, const float* bg_rgb, float k00, float k11, int H, int W, int K, int flags, const int* pix_to_face) {
  const GeomLayout g = geom_layout(total_verts, total_faces);
  const char* gb = (const char*)geometry;
  p.verts4 = (const float4*)(gb + g.verts4); p.normals4 = (const float4*)(gb + g.normals4);
  p.rgb4 = (const float4*)(gb + g.rgb4); p.faces4 = (const int4*)(gb + g.faces4); p.xn8 = (const float4*)(gb + g.xn8);
  p.vert_off = vert_off; p.face_off = face_off;
  p.R = R; p.T = T; p.Cc = Cc; p.light = light; p.light_stride = light_stride; p.obj_rgb = obj_rgb; p.bg_rgb = bg_rgb;
  p.k00 = k00; p.k11 = k11; p.z_clip = -1.f; p.blur_radius = 0.f; p.blur_r = 0.f;
  p.B = B; p.M = M; p.H = H; p.W = W; p.K = K; p.flags = flags; p.layer = 0;
  p.pix_to_face = const_cast<int*>(pix_to_face);
  p.images = nullptr; p.zbuf = nullptr; p.bary = nullptr; p.dists = nullptr; p.counters = nullptr; p.keys = nullptr; p.prev = nullptr;
  p.onorm = make_out_norm(nullptr); p.wsflags = nullptr; p.pv = nullptr; p.tab = nullptr;
  return 0;
}

extern "C" int mvr_mesh_soft_blend_forward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                           int64_t total_verts, int64_t total_faces, const float* Cc, const float* light, int light_stride,
                                           const float* obj_rgb, const float* bg_rgb, int H, int W, int K, int flags, int mode, float sigma,
                                           float gamma, float znear, float zfar, const int* pix_to_face, const float* zbuf, const float* bary,
                                           const float* dists, float* rgba, void* stream) {
  int rc = check_mesh_common("mvr_mesh_soft_blend_forward", B, M, H, W, K, total_verts, total_faces, 0);
  if (rc) return rc;
  if ((int64_t)B * M == 0) return 0;
  if (!geometry || !vert_off || !face_off || !Cc || !light || !bg_rgb || !pix_to_face || !zbuf || !bary || !dists || !rgba) { set_error("mvr_mesh_soft_blend_forward: null pointer"); return -5; }
  if (!(flags & MVR_RGB_PER_ELEMENT) && !obj_rgb) { set_error("mvr_mesh_soft_blend_forward: obj_rgb is NULL"); return -6; }
  if (mode < 0 || mode > 1 || !(sigma > 0.f) || !(gamma > 0.f) || !(zfar > znear)) { set_error("mvr_mesh_soft_blend_forward: bad mode / sigma / gamma / z range"); return -7; }
  MeshParams p;
  fill_params(p, geometry, vert_off, face_off, B, M, total_verts, total_faces, nullptr, nullptr, Cc, light, light_stride, obj_rgb, bg_rgb, 0.f, 0.f, H, W, K, flags, pix_to_face);
  SoftParams sp = {mode, sigma, gamma, znear, zfar, 0.f, zbuf, bary, dists, rgba, nullptr, nullptr, nullptr};
  const dim3 grid((unsigned)(((size_t)H * W + MVR_THREADS - 1) / MVR_THREADS), (unsigned)M, (unsigned)B);
  MVR_LAUNCH(mesh_soft_blend_kernel, grid, MVR_THREADS, 0, (cudaStream_t)stream, p, sp);
  return check_launch("mesh_soft_blend_kernel");
}

extern "C" int mvr_mesh_soft_backward(const void* geometry, const int* vert_off, const int* face_off, int B, int M, int64_t total_verts,
                                      int64_t total_faces, int max_verts, const float* R, const float* T, const float* Cc, const float* light,
                                      int light_stride, const float* obj_rgb, const float* bg_rgb, float k00, float k11, float z_clip,
                                      float blur_radius, int H, int W, int K, int flags, int mode, float sigma, float gamma, float znear,
                                      float zfar, const int* pix_to_face,
                                      const float* grad_rgba, float* gR, float* gT, float* gC, float* grad_verts, float* grad_normals,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_mesh_common("mvr_mesh_soft_backward", B, M, H, W, K, total_verts, total_faces, max_verts);
  if (rc) return rc;
  const int64_t N = (int64_t)B * M;
  if (N == 0) return 0;
  if (!geometry || !vert_off || !face_off || !R || !T || !Cc || !light || !bg_rgb || !pix_to_face || !grad_rgba || !gR || !gT || !gC || !workspace) { set_error("mvr_mesh_soft_backward: null pointer"); return -5; }
  if (!(flags & MVR_RGB_PER_ELEMENT) && !obj_rgb) { set_error("mvr_mesh_soft_backward: obj_rgb is NULL"); return -6; }
  if (mode < 0 || mode > 1 || !(sigma > 0.f) || !(gamma > 0.f) || !(zfar > znear)) { set_error("mvr_mesh_soft_backward: bad mode / sigma / gamma / z range"); return -7; }
  if (!(blur_radius >= 0.f)) { set_error("mvr_mesh_soft_backward: blur_radius must be >= 0"); return -9; }
  const WsLayout w = ws_layout(B, M, H, W, K, total_verts, total_faces);
  if (workspace_bytes < w.total) { set_error("mvr_mesh_soft_backward: workspace too small (%zu < %zu)", workspace_bytes, w.total); return -8; }
  const GeomLayout g = geom_layout(total_verts, total_faces);
  cudaStream_t st = (cudaStream_t)stream;
  char* wb = (char*)workspace;
  // project again, with the forward's z_clip: the projection clears the workspace flag WSF_CLIP when a vertex lies behind the
  // plane, and the fragments of faces crossing it are then recomputed on their clipped sub-triangles (soft_fragment)
  rc = launch_project("mesh_project_kernel", g, w, geometry, vert_off, R, T, B, M, H, W, max_verts, k00, k11, z_clip, true, workspace, st);
  if (rc) return rc;
  MeshParams p;
  fill_params(p, geometry, vert_off, face_off, B, M, total_verts, total_faces, R, T, Cc, light, light_stride, obj_rgb, bg_rgb, k00, k11, H, W, K, flags, pix_to_face);
  p.pv = (float4*)(wb + w.pv); p.tab = (float*)(wb + w.tab); p.wsflags = (int*)(wb + w.flags);
  p.z_clip = z_clip;
  p.blur_radius = blur_radius > 0.f ? blur_radius : 0.f; p.blur_r = sqrtf(p.blur_radius);      // as mvr_mesh_forward
  SoftParams sp = {mode, sigma, gamma, znear, zfar, 0.f, nullptr, nullptr, nullptr, nullptr, grad_rgba, grad_verts, grad_normals};
  const int tiles_x = (W + 31) / 32;
  const dim3 grid((unsigned)w.bwd_ctas_per_view, (unsigned)M, (unsigned)B);
  if (grad_verts || grad_normals)
    MVR_LAUNCH((mesh_soft_backward_kernel<true>), grid, MVR_THREADS, 0, st, p, sp, (float*)(wb + w.partials), w.bwd_parts_per_view, tiles_x);
  else
    MVR_LAUNCH((mesh_soft_backward_kernel<false>), grid, MVR_THREADS, 0, st, p, sp, (float*)(wb + w.partials), w.bwd_parts_per_view, tiles_x);
  rc = check_launch("mesh_soft_backward_kernel");
  if (rc) return rc;
  MeshBwdParams q;
  q.azim = q.elev = q.dist = nullptr; q.g_azim = q.g_elev = q.g_dist = nullptr;
  // the finish kernel only sums the partials here: its hard clipped-pixel pass is kept off by pointing its flag at a word of the
  // armed flag block that the projection never clears (word WSF_CLIP may be cleared above)
  q.partials = (float*)(wb + w.partials); q.parts_per_view = w.bwd_parts_per_view; q.wsflags = (int*)(wb + w.flags) + WSF_CLIP + 1;
  q.B = B; q.M = M; q.H = H; q.W = W; q.K = K; q.flags = flags; q.z_clip = -1.f; q.grad_verts = nullptr; q.grad_normals = nullptr;
  return launch_mesh_backward_finish(q, (int)N, gR, gT, gC, st);
}
