// mvr_mesh_clip.cu -- pixels won by a face that crosses the near clip plane ([upstream] renderer/mesh/clip.py).
//
// PyTorch3D >= 0.5 clips such a face against z = znear / 2 into one or two sub-triangles before rasterizing and maps
// the fragments back to the original face (barycentric conversion).  MVTN only meets them when transform_distance pulls
// a camera closer than 1.5 to a unit-sphere object (mvtn.py:33), so the hot kernels stay as they are and merely step
// aside: mesh_project_kernel raises a flag in the workspace when any vertex lies behind the plane, mesh_scatter_kernel
// rasterizes the sub-triangles of a straddling face (whole CTA per face), mesh_shade_kernel / mesh_backward_kernel skip a
// pixel whose winning face straddles the plane, and the two kernels below -- which exit at once while the flag is down
// -- redo exactly those pixels with the clipped geometry.
// Compiled with -fmad=false like the forward unit: which sub-triangle owns a pixel is a fragment decision.
#include "mvr_mesh.cuh"
#include "mvr_camera.cuh"

namespace mvr {

// The sub-triangle the rasterizer kept for pixel (xf, yf): inside, smallest (pz, index).  want_z_bits != 0: the one
// whose depth is the recorded key (forward); bcl = its barycentrics, pz its depth.  Returns -1 if none.
__device__ __forceinline__ int pick_sub(const ClipSub& cs, int flags, bool persp, float xf, float yf, unsigned int want_z_bits,
                                        float bcl[3], float& pz_out) {
  int best = -1;
  float bz = 0.f;
  for (int s = 0; s < cs.ns; ++s) {
    const Face sf = cs.f[s];
    if (!sub_face_ok(sf, flags)) continue;
    float w[3], b[3], pz;
    if (!raster_test(sf, face_edges(sf), persp, xf, yf, w, b, pz)) continue;
    if (want_z_bits && __float_as_uint(pz + 0.0f) != want_z_bits) continue;
    if (best < 0 || pz < bz) { best = s; bz = pz; bcl[0] = b[0]; bcl[1] = b[1]; bcl[2] = b[2]; }
  }
  pz_out = bz;
  return best;
}

// SOFT: the blurred rasterizer (blur_radius > 0 / clipped barycentrics) -- the sub-triangle is picked by its soft test
// (pick_sub_soft), the fragment carries its (clipped) barycentrics converted to the original face and its SIGNED edge distance
template <bool SOFT>
__device__ __forceinline__ void shade_clipped_pixel(const MeshParams& p, int b, int m, int n, int pix) {
  const int HW = p.H * p.W;
  const int yi = pix / p.W, xi = pix - yi * p.W;
  const int k = p.layer;
  // the shade pass has already handed this layer's keys to `prev` when another layer follows
  const unsigned long long key = (k + 1 < p.K) ? p.prev[(size_t)n * HW + pix] : p.keys[(size_t)n * HW + pix];
  if (key == MVR_EMPTY_KEY) return;
  // the shade pass re-armed every key it consumed (MVR_WS_REARM_KEYS) except those of the pixels handled here
  if ((p.flags & MVR_WS_REARM_KEYS) && k + 1 == p.K) p.keys[(size_t)n * HW + pix] = MVR_EMPTY_KEY;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  const int fid = (int)(unsigned int)(key & 0xffffffffull);
  const int4 fi = __ldg(p.faces4 + f0 + fid);
  const Face fc = gather_face(p.pv + (size_t)p.M * voff + (size_t)m * V, fi);
  if (!face_straddles(fc, p.z_clip)) return;
  ClipSub cs;
  clip_face(fc, p.z_clip, persp, cs);
  const float xf = __ldg(p.tab + xi), yf = __ldg(p.tab + p.W + yi);
  float bcl[3], pz;
  float bb[3] = {-1.f, -1.f, -1.f}, dd = -1.f;
  int s;
  if (SOFT) {
    SoftHit h;
    s = pick_sub_soft(cs, p.flags, persp, p.flags & MVR_CLIP_BARYCENTRIC, p.blur_radius, p.blur_r, xf, yf, (unsigned int)(key >> 32), 0, h);
    if (s >= 0) { bcl[0] = h.bc[0]; bcl[1] = h.bc[1]; bcl[2] = h.bc[2]; dd = h.sd; }
  } else {
    s = pick_sub(cs, p.flags, persp, xf, yf, (unsigned int)(key >> 32), bcl, pz);
    if (s < 0) s = pick_sub(cs, p.flags, persp, xf, yf, 0u, bcl, pz);
  }
  float out[3] = {__ldg(p.bg_rgb), __ldg(p.bg_rgb + 1), __ldg(p.bg_rgb + 2)};
  if (s >= 0) {
    conv_bary(cs.conv[s], bcl, bb);
    if (!SOFT) {
      const Face sf = cs.f[s];
      const float e01 = point_line_dist2(xf, yf, sf.x0, sf.y0, sf.x1, sf.y1);
      const float e02 = point_line_dist2(xf, yf, sf.x0, sf.y0, sf.x2, sf.y2);
      const float e12 = point_line_dist2(xf, yf, sf.x1, sf.y1, sf.x2, sf.y2);
      dd = -fminf(fminf(e01, e02), e12);
    }
    if (k == 0) {
      const float4 X0 = __ldg(p.verts4 + voff + fi.x), X1 = __ldg(p.verts4 + voff + fi.y), X2 = __ldg(p.verts4 + voff + fi.z);
      const float4 N0 = __ldg(p.normals4 + voff + fi.x), N1 = __ldg(p.normals4 + voff + fi.y), N2 = __ldg(p.normals4 + voff + fi.z);
      float4 c0, c1, c2;
      if (p.flags & MVR_RGB_PER_ELEMENT) { c0 = __ldg(p.rgb4 + voff + fi.x); c1 = __ldg(p.rgb4 + voff + fi.y); c2 = __ldg(p.rgb4 + voff + fi.z); }
      else { c0 = c1 = c2 = make_float4(__ldg(p.obj_rgb), __ldg(p.obj_rgb + 1), __ldg(p.obj_rgb + 2), 0.f); }
      const ShadeCtx sc = load_shade_ctx(p.light, p.light_stride, p.Cc, n);
      phong_pixel(bb, X0, X1, X2, N0, N1, N2, c0, c1, c2, sc, out);
    }
  }
  const size_t po = ((size_t)n * HW + pix) * p.K + k;
  p.pix_to_face[po] = s >= 0 ? fid : -1;
  if (p.zbuf) p.zbuf[po] = s >= 0 ? __uint_as_float((unsigned int)(key >> 32)) : -1.f;
  if (p.dists) p.dists[po] = dd;
  if (p.bary) { p.bary[3 * po] = bb[0]; p.bary[3 * po + 1] = bb[1]; p.bary[3 * po + 2] = bb[2]; }
  if (k == 0) store_rgb(p.images, p.flags & MVR_IMAGES_BF16, (size_t)n * 3 * HW + pix, (size_t)HW, out[0], out[1], out[2], p.onorm);
}

// Hard depth (K = 1) of a pixel won by a face crossing the near plane: the depth is the key's z -- the z of the sub-triangle
// the scatter kept -- unless no sub-triangle passes the forward's own test at this pixel (then background, as shade_clipped_pixel).
__device__ __forceinline__ void depth_clipped_pixel(const MeshParams& p, int b, int m, int n, int pix) {
  const int HW = p.H * p.W;
  const int yi = pix / p.W, xi = pix - yi * p.W;
  const unsigned long long key = p.keys[(size_t)n * HW + pix];
  if (key == MVR_EMPTY_KEY) return;
  if (p.flags & MVR_WS_REARM_KEYS) p.keys[(size_t)n * HW + pix] = MVR_EMPTY_KEY;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  const int fid = (int)(unsigned int)(key & 0xffffffffull);
  const Face fc = gather_face(p.pv + (size_t)p.M * voff + (size_t)m * V, __ldg(p.faces4 + f0 + fid));
  if (!face_straddles(fc, p.z_clip)) return;
  ClipSub cs;
  clip_face(fc, p.z_clip, persp, cs);
  const float xf = __ldg(p.tab + xi), yf = __ldg(p.tab + p.W + yi);
  float bcl[3], pz;
  int s = pick_sub(cs, p.flags, persp, xf, yf, (unsigned int)(key >> 32), bcl, pz);
  if (s < 0) s = pick_sub(cs, p.flags, persp, xf, yf, 0u, bcl, pz);
  p.pix_to_face[(size_t)n * HW + pix] = s >= 0 ? fid : -1;
  reinterpret_cast<float*>(p.images)[(size_t)n * HW + pix] = s >= 0 ? __uint_as_float((unsigned int)(key >> 32)) : p.depth_bg;
}

// grid: one CTA per view, striding over its pixels (the common case is "flag down": N tiny CTAs that exit at once).
// Writes EVERY output of a pixel whose winning face straddles the plane (mesh_shade_kernel left it untouched).
// DEPTH: the hard depth instance (depth_clipped_pixel).
template <bool SOFT, bool DEPTH = false>
__global__ void __launch_bounds__(MVR_THREADS) mesh_shade_clipped_kernel(const MeshParams p) {
  pdl_enter();
  if (!may_clip(p.wsflags)) return;
  const int n = blockIdx.x, b = n / p.M, m = n - b * p.M;
  const int HW = p.H * p.W;
  for (int pix = threadIdx.x; pix < HW; pix += MVR_THREADS) {
    if (DEPTH) depth_clipped_pixel(p, b, m, n, pix);
    else shade_clipped_pixel<SOFT>(p, b, m, n, pix);
  }
}


// ------------------------------------------------------------------------------------------------
// backward of one clipped pixel: d image -> Phong -> unclipped barycentrics -> (conversion, clipped barycentrics) ->
// clipped triangle -> original (x_ndc, y_ndc, z_view) (clip_face_backward, mvr_mesh.cuh), then the projection as usual.
// Same derivation as oracle/mvr_oracle.c clip_face_bwd / raster_bwd_one / phong_pixel_bwd, in fp32.
// ------------------------------------------------------------------------------------------------
// The clipped-face pixels of view n (those mesh_backward_kernel skipped), accumulated by the whole CTA into acc (per thread).
// GC: colour gradients too -- per-vertex colours into p.grad_rgb (atomics), one object colour into gcol (per thread).
template <bool GC>
__device__ __forceinline__ void backward_clipped_view(const MeshBwdParams& p, int n, float (&acc)[16], float (&gcol)[3]) {
  const int tid = threadIdx.x;
  const int b = n / p.M, m = n - b * p.M;
  const int HW = p.H * p.W;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  const bool per_vertex_rgb = p.flags & MVR_RGB_PER_ELEMENT;
  const ShadeCtx sc = load_shade_ctx(p.light, p.light_stride, p.Cc, n);
  float4 ucol = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!per_vertex_rgb) ucol = make_float4(__ldg(p.obj_rgb), __ldg(p.obj_rgb + 1), __ldg(p.obj_rgb + 2), 0.f);
  for (int pix = tid; pix < HW; pix += MVR_THREADS) {
    const int fid = __ldg(p.pix_to_face + ((size_t)n * HW + pix) * p.K);
    if (fid < 0) continue;
    const int4 fi = __ldg(p.faces4 + f0 + fid);
    const Face fc = gather_face(pvn, fi);
    if (!face_straddles(fc, p.z_clip)) continue;
    float g0, g1, g2;
    load_grad_rgb(p.grad_images, p.flags & MVR_IMAGES_BF16, (size_t)n * 3 * HW + pix, (size_t)HW, p.onorm, g0, g1, g2);
    if (g0 == 0.f && g1 == 0.f && g2 == 0.f) continue;
    const int yi = pix / p.W, xi = pix - yi * p.W;
    const float xf = __ldg(p.tab + xi), yf = __ldg(p.tab + p.W + yi);
    ClipSub cs;
    clip_face(fc, p.z_clip, persp, cs);
    float bcl[3], pz;
    const int s = pick_sub(cs, p.flags, persp, xf, yf, 0u, bcl, pz);
    if (s < 0) continue;
    float bb[3];
    conv_bary(cs.conv[s], bcl, bb);
    const float4 X[3] = {__ldg(p.verts4 + voff + fi.x), __ldg(p.verts4 + voff + fi.y), __ldg(p.verts4 + voff + fi.z)};
    const float4 N0 = __ldg(p.normals4 + voff + fi.x), N1 = __ldg(p.normals4 + voff + fi.y), N2 = __ldg(p.normals4 + voff + fi.z);
    float4 c0 = ucol, c1 = ucol, c2 = ucol;
    if (per_vertex_rgb) { c0 = __ldg(p.rgb4 + voff + fi.x); c1 = __ldg(p.rgb4 + voff + fi.y); c2 = __ldg(p.rgb4 + voff + fi.z); }
    float gb[3], gv[3], gN[3], gt[3];
    phong_backward(bb, X[0], X[1], X[2], N0, N1, N2, c0, c1, c2, sc, g0, g1, g2, gb, gv, gN, GC ? gt : nullptr);
    acc[12] += gv[0]; acc[13] += gv[1]; acc[14] += gv[2];      // dC
    if (GC) {      // texel = sum_i bb_i c_i
      if (per_vertex_rgb) {
        for (int i = 0; i < 3; ++i) {
          float* o = p.grad_rgb + 3 * (size_t)(voff + (i == 0 ? fi.x : i == 1 ? fi.y : fi.z));
          atomicAdd(o + 0, bb[i] * gt[0]); atomicAdd(o + 1, bb[i] * gt[1]); atomicAdd(o + 2, bb[i] * gt[2]);
        }
      } else {
        const float sb = bb[0] + bb[1] + bb[2];
        gcol[0] += sb * gt[0]; gcol[1] += sb * gt[1]; gcol[2] += sb * gt[2];
      }
    }
    float gbeta[3], gq[9], gfv[9];
    for (int k = 0; k < 3; ++k) gbeta[k] = cs.conv[s][k] * gb[0] + cs.conv[s][3 + k] * gb[1] + cs.conv[s][6 + k] * gb[2];
    raster_backward(cs.f[s], persp, xf, yf, gbeta, gq);
    clip_face_backward(fc, p.z_clip, persp, cs.info, s, gq, gb, bcl, gfv);
    // projection backward + X R + T backward: x_ndc = (px k00) / pz, so px k00 = x_ndc pz
    const float xn[3] = {fc.x0, fc.x1, fc.x2}, yn[3] = {fc.y0, fc.y1, fc.y2}, zv[3] = {fc.z0, fc.z1, fc.z2};
    const int vid[3] = {fi.x, fi.y, fi.z};
    for (int i = 0; i < 3; ++i) {
      const float iz = 1.0f / zv[i];
      const float gpx = gfv[3 * i] * p.k00 * iz;
      const float gpy = gfv[3 * i + 1] * p.k11 * iz;
      const float gpz = gfv[3 * i + 2] - (gfv[3 * i] * xn[i] + gfv[3 * i + 1] * yn[i]) * iz;
      acc[0] += X[i].x * gpx; acc[1] += X[i].x * gpy; acc[2] += X[i].x * gpz;
      acc[3] += X[i].y * gpx; acc[4] += X[i].y * gpy; acc[5] += X[i].y * gpz;
      acc[6] += X[i].z * gpx; acc[7] += X[i].z * gpy; acc[8] += X[i].z * gpz;
      acc[9] += gpx; acc[10] += gpy; acc[11] += gpz;
      if (p.grad_verts) {
        const float* r = p.R + 9 * (size_t)n;
        float* o = p.grad_verts + 3 * (size_t)(voff + vid[i]);
        atomicAdd(o + 0, (__ldg(r + 0) * gpx + __ldg(r + 1) * gpy + __ldg(r + 2) * gpz) - bb[i] * gv[0]);
        atomicAdd(o + 1, (__ldg(r + 3) * gpx + __ldg(r + 4) * gpy + __ldg(r + 5) * gpz) - bb[i] * gv[1]);
        atomicAdd(o + 2, (__ldg(r + 6) * gpx + __ldg(r + 7) * gpy + __ldg(r + 8) * gpz) - bb[i] * gv[2]);
      }
      if (p.grad_normals) {
        float* o = p.grad_normals + 3 * (size_t)(voff + vid[i]);
        atomicAdd(o + 0, bb[i] * gN[0]); atomicAdd(o + 1, bb[i] * gN[1]); atomicAdd(o + 2, bb[i] * gN[2]);
      }
    }
  }
}

// Hard depth: the clipped-face pixels of view n (those mesh_depth_backward_kernel skipped) -> acc (dR, dT; dC stays 0).  The pixel's
// depth is the sub-triangle's bcl . z_sub: d/d its barycentrics = g z_sub (raster_backward), d/d z_sub = g bcl, and nothing reaches
// the converted (original-face) barycentrics; then clip_face_backward and the projection as backward_clipped_view.
__device__ __forceinline__ void backward_clipped_view_depth(const MeshBwdParams& p, int n, float (&acc)[16]) {
  const int b = n / p.M, m = n - b * p.M;
  const int HW = p.H * p.W;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  const float* gd = reinterpret_cast<const float*>(p.grad_images);
  for (int pix = threadIdx.x; pix < HW; pix += MVR_THREADS) {
    const int fid = __ldg(p.pix_to_face + (size_t)n * HW + pix);
    if (fid < 0) continue;
    const int4 fi = __ldg(p.faces4 + f0 + fid);
    const Face fc = gather_face(pvn, fi);
    if (!face_straddles(fc, p.z_clip)) continue;
    const float g = __ldg(gd + (size_t)n * HW + pix);
    if (g == 0.f) continue;
    const int yi = pix / p.W, xi = pix - yi * p.W;
    const float xf = __ldg(p.tab + xi), yf = __ldg(p.tab + p.W + yi);
    ClipSub cs;
    clip_face(fc, p.z_clip, persp, cs);
    float bcl[3], pz;
    const int s = pick_sub(cs, p.flags, persp, xf, yf, 0u, bcl, pz);
    if (s < 0) continue;
    const Face sf = cs.f[s];
    const float gbeta[3] = {g * sf.z0, g * sf.z1, g * sf.z2}, gb0[3] = {0.f, 0.f, 0.f};
    float gq[9], gfv[9];
    raster_backward(sf, persp, xf, yf, gbeta, gq);
    gq[2] += g * bcl[0]; gq[5] += g * bcl[1]; gq[8] += g * bcl[2];
    clip_face_backward(fc, p.z_clip, persp, cs.info, s, gq, gb0, bcl, gfv);
    const float4 X[3] = {__ldg(p.verts4 + voff + fi.x), __ldg(p.verts4 + voff + fi.y), __ldg(p.verts4 + voff + fi.z)};
    const float xn[3] = {fc.x0, fc.x1, fc.x2}, yn[3] = {fc.y0, fc.y1, fc.y2}, zv[3] = {fc.z0, fc.z1, fc.z2};
    const int vid[3] = {fi.x, fi.y, fi.z};
    for (int i = 0; i < 3; ++i) {
      const float iz = 1.0f / zv[i];
      const float gpx = gfv[3 * i] * p.k00 * iz;
      const float gpy = gfv[3 * i + 1] * p.k11 * iz;
      const float gpz = gfv[3 * i + 2] - (gfv[3 * i] * xn[i] + gfv[3 * i + 1] * yn[i]) * iz;
      acc[0] += X[i].x * gpx; acc[1] += X[i].x * gpy; acc[2] += X[i].x * gpz;
      acc[3] += X[i].y * gpx; acc[4] += X[i].y * gpy; acc[5] += X[i].y * gpz;
      acc[6] += X[i].z * gpx; acc[7] += X[i].z * gpy; acc[8] += X[i].z * gpz;
      acc[9] += gpx; acc[10] += gpy; acc[11] += gpz;
      if (p.grad_verts) {
        const float* r = p.R + 9 * (size_t)n;
        float* o = p.grad_verts + 3 * (size_t)(voff + vid[i]);
        atomicAdd(o + 0, __ldg(r + 0) * gpx + __ldg(r + 1) * gpy + __ldg(r + 2) * gpz);
        atomicAdd(o + 1, __ldg(r + 3) * gpx + __ldg(r + 4) * gpy + __ldg(r + 5) * gpz);
        atomicAdd(o + 2, __ldg(r + 6) * gpx + __ldg(r + 7) * gpy + __ldg(r + 8) * gpz);
      }
    }
  }
}

// grid: one CTA per view -> gR, gT, gC.  (1) when some vertex lies behind the near plane (WSF_CLIP), the pixels of
// straddling faces, which mesh_backward_kernel skipped, are redone with the clipped geometry; (2) fixed-order sum of the
// per-warp partials of mesh_backward_kernel: thread t owns value t & 15 of the parts congruent to t >> 4 modulo 16
// (coalesced 64-byte rows), then 16 threads add the 16 group sums (and the clipped part) in a fixed order.
// GC (p.grad_rgb set): also the colour gradient -- the clipped pixels' share and, for one object colour, the view's total of
// the colour partials in fp64 (rgb_views; mesh_rgb_grad_sum_kernel adds the views).
// DEPTH: the partials are mesh_depth_backward_kernel's and the clipped pixels go through backward_clipped_view_depth.
template <bool GC, bool DEPTH = false>
__global__ void __launch_bounds__(MVR_THREADS) mesh_backward_finish_kernel(const MeshBwdParams p, float* __restrict__ gR,
                                                                           float* __restrict__ gT, float* __restrict__ gC) {
  __shared__ double s_sum[MVR_THREADS];
  __shared__ float s_red[(MVR_THREADS / 32) * 16];
  __shared__ float s_cred[GC ? (MVR_THREADS / 32) * 3 : 1];
  pdl_enter();
  const int n = blockIdx.x, tid = threadIdx.x;
  const bool clip = may_clip(p.wsflags);      // block-uniform
  const bool one_rgb = GC && !(p.flags & MVR_RGB_PER_ELEMENT);
  if (clip) {
    float acc[16], gcol[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    if (DEPTH) backward_clipped_view_depth(p, n, acc);
    else backward_clipped_view<GC>(p, n, acc, gcol);
    block_sum<16>(acc, s_red);                // s_red[0..15] = the clipped pixels' totals
    if (one_rgb) block_sum<3>(gcol, s_cred);  // s_cred[0..2]: their colour gradient
  }
  // the per-warp partials (tens to hundreds per view, of mixed sign) are summed in fp64: free here, and it removes the
  // one accumulation level whose operands are large next to the result
  const int v = tid & 15, grp = tid >> 4;
  double s = 0.0;
  for (int t = grp; t < p.parts_per_view; t += MVR_THREADS / 16) s += (double)p.partials[((size_t)n * p.parts_per_view + t) * 16 + v];
  s_sum[tid] = s;
  __syncthreads();
  if (tid < 16) {
    double tot = clip ? (double)s_red[tid] : 0.0;
#pragma unroll
    for (int g = 0; g < MVR_THREADS / 16; ++g) tot += s_sum[g * 16 + tid];
    const float out = (float)tot;
    if (tid < 9) { if (gR) gR[9 * (size_t)n + tid] = out; }
    else if (tid < 12) { if (gT) gT[3 * (size_t)n + tid - 9] = out; }
    else if (tid < 15) { if (gC) gC[3 * (size_t)n + tid - 12] = out; }
    s_red[tid] = out;
  }
  if (one_rgb) {      // block-uniform: the view's colour partials, value tid & 3 of the parts congruent to tid >> 2 modulo 64
    __syncthreads();
    const int c = tid & 3, cg = tid >> 2;
    double t = 0.0;
    if (c < 3)
      for (int q = cg; q < p.parts_per_view; q += MVR_THREADS / 4) t += (double)p.rgb_partials[((size_t)n * p.parts_per_view + q) * 4 + c];
    s_sum[tid] = t;
    __syncthreads();
    if (tid < 3) {
      double tot = clip ? (double)s_cred[tid] : 0.0;
      for (int g = 0; g < MVR_THREADS / 4; ++g) tot += s_sum[g * 4 + tid];
      p.rgb_views[3 * (size_t)n + tid] = tot;
    }
  }
  if (p.azim) {      // mvr_mesh_backward_angles: (dR, dT, dC) -> (d azim, d elev, d dist) of this view, same launch (block-uniform)
    __syncthreads();
    if (tid == 0) {
      float ga, ge, gd;
      look_at_backward_view(__ldg(p.azim + n), __ldg(p.elev + n), __ldg(p.dist + n), s_red, s_red + 9, s_red + 12, ga, ge, gd);
      p.g_azim[n] = ga; p.g_elev[n] = ge; p.g_dist[n] = gd;
    }
  }
}

// One object colour: grad_rgb[c] = the sum of the N per-view fp64 totals in a fixed order (thread t: views congruent to t >> 2
// modulo 64, then thread c adds the 64 group sums in order) -- bit-reproducible, as the camera gradients are.
__global__ void __launch_bounds__(MVR_THREADS) mesh_rgb_grad_sum_kernel(const double* __restrict__ views, int N, float* __restrict__ grad_rgb) {
  __shared__ double s_sum[MVR_THREADS];
  pdl_enter();
  const int tid = threadIdx.x, c = tid & 3, g = tid >> 2;
  double t = 0.0;
  if (c < 3)
    for (int n = g; n < N; n += MVR_THREADS / 4) t += views[3 * (size_t)n + c];
  s_sum[tid] = t;
  __syncthreads();
  if (tid < 3) {
    double tot = 0.0;
    for (int q = 0; q < MVR_THREADS / 4; ++q) tot += s_sum[q * 4 + tid];
    grad_rgb[tid] = (float)tot;
  }
}

}  // namespace mvr

using namespace mvr;

int launch_mesh_shade_clipped(const MeshParams& p, int N, bool soft, cudaStream_t st, bool depth) {
  if (depth) MVR_LAUNCH_PDL((mesh_shade_clipped_kernel<false, true>), (unsigned)N, MVR_THREADS, 0, st, p);
  else if (soft) MVR_LAUNCH_PDL(mesh_shade_clipped_kernel<true>, (unsigned)N, MVR_THREADS, 0, st, p);
  else MVR_LAUNCH_PDL(mesh_shade_clipped_kernel<false>, (unsigned)N, MVR_THREADS, 0, st, p);
  return check_launch("mesh_shade_clipped_kernel");
}

int launch_mesh_backward_finish(const MeshBwdParams& p, int N, float* gR, float* gT, float* gC, cudaStream_t st, bool depth) {
  if (depth) {
    MVR_LAUNCH_PDL((mesh_backward_finish_kernel<false, true>), (unsigned)N, MVR_THREADS, 0, st, p, gR, gT, gC);
    return check_launch("mesh_backward_finish_kernel");
  }
  if (!p.grad_rgb) {
    MVR_LAUNCH_PDL(mesh_backward_finish_kernel<false>, (unsigned)N, MVR_THREADS, 0, st, p, gR, gT, gC);
    return check_launch("mesh_backward_finish_kernel");
  }
  MVR_LAUNCH_PDL(mesh_backward_finish_kernel<true>, (unsigned)N, MVR_THREADS, 0, st, p, gR, gT, gC);
  int rc = check_launch("mesh_backward_finish_kernel");
  if (rc || (p.flags & MVR_RGB_PER_ELEMENT)) return rc;
  MVR_LAUNCH_PDL(mesh_rgb_grad_sum_kernel, 1u, MVR_THREADS, 0, st, p.rgb_views, N, p.grad_rgb);
  return check_launch("mesh_rgb_grad_sum_kernel");
}
