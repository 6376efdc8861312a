// mvr_mesh_fwd.cuh -- device code of the mesh path's forward rasterizer, the bin-free scatter onto a global key plane
// (mvr_mesh.cu): face setup, the scanline candidate spans and the exact per-(face, pixel) test.  mvr_mesh.cu is compiled
// with -fmad=false: everything here that decides a fragment is IEEE fp32 in the written order.
#pragma once
#include "mvr_mesh.cuh"

namespace mvr {

// ------------------------------------------------------------------------------------------------
// shared device code: projection, face setup and the per-(face, pixel) test
// ------------------------------------------------------------------------------------------------
// Face-level rejection ([upstream] clip.py near cull, CheckPointOutsideBoundingBox z_invalid,
// RasterizeMeshesNaiveCpu zero-area / back-face tests) and the exact pixel bbox (inclusive ranges).
__device__ __forceinline__ bool face_pixel_bbox(const Face& f, const MeshParams& p, const float* s_xf, const float* s_yf,
                                                int& xi_lo, int& xi_hi, int& yi_lo, int& yi_hi) {
  if (p.z_clip >= 0.f && f.z0 < p.z_clip && f.z1 < p.z_clip && f.z2 < p.z_clip) return false;
  const float zmin = fminf(fminf(f.z0, f.z1), f.z2);
  if (zmin < MVR_K_EPS) return false;
  const float face_area = (f.x0 - f.x1) * (f.y2 - f.y1) - (f.y0 - f.y1) * (f.x2 - f.x1);
  if ((p.flags & MVR_CULL_BACKFACES) && face_area < 0.f) return false;
  if (face_area <= MVR_K_EPS && face_area >= -1.0f * MVR_K_EPS) return false;
  const float xmin = fminf(fminf(f.x0, f.x1), f.x2) - p.blur_r, xmax = fmaxf(fmaxf(f.x0, f.x1), f.x2) + p.blur_r;
  const float ymin = fminf(fminf(f.y0, f.y1), f.y2) - p.blur_r, ymax = fmaxf(fmaxf(f.y0, f.y1), f.y2) + p.blur_r;
  pixel_range(xmin, xmax, p.W, p.H, 0, p.W - 1, s_xf, xi_lo, xi_hi);
  if (xi_lo > xi_hi) return false;
  pixel_range(ymin, ymax, p.H, p.W, 0, p.H - 1, s_yf, yi_lo, yi_hi);
  return yi_lo <= yi_hi;
}

// conservative range of pixel indices whose centre can lie in [vmin, vmax] (superset of pixel_range's exact answer: the
// float estimate of the inverse pixel map is widened by 4e-3 pixel, ~6x its worst rounding error at S1 = 4096)
__device__ __forceinline__ bool pixel_range_conservative(float vmin, float vmax, int S1, float scale, float off, int& ilo, int& ihi) {
  const float jhi = floorf(fmaf(vmax, scale, off) + 4e-3f);
  const float jlo = ceilf(fmaf(vmin, scale, off) - 4e-3f);
  if (!(jlo <= jhi) || jhi < 0.f || jlo > (float)(S1 - 1)) return false;
  const int jh = (int)fminf(jhi, (float)(S1 - 1)), jl = (int)fmaxf(jlo, 0.f);
  ilo = S1 - 1 - jh; ihi = S1 - 1 - jl;
  return true;
}

// The rasterizer's face-level rejections (as face_pixel_bbox) with a CONSERVATIVE pixel bbox: no table look-ups, no fix-up
// loops.  The exact bbox test of the oracle (CheckPointOutsideBoundingBox) is then applied per candidate, in
// resolve_pixel_with, as the four float compares it is.
__device__ __forceinline__ bool face_pixel_bbox_conservative(const Face& f, const MeshParams& p, int& xi_lo, int& xi_hi, int& yi_lo, int& yi_hi) {
  if (p.z_clip >= 0.f && f.z0 < p.z_clip && f.z1 < p.z_clip && f.z2 < p.z_clip) return false;
  const float zmin = fminf(fminf(f.z0, f.z1), f.z2);
  if (zmin < MVR_K_EPS) return false;
  const float face_area = (f.x0 - f.x1) * (f.y2 - f.y1) - (f.y0 - f.y1) * (f.x2 - f.x1);
  if ((p.flags & MVR_CULL_BACKFACES) && face_area < 0.f) return false;
  if (face_area <= MVR_K_EPS && face_area >= -1.0f * MVR_K_EPS) return false;
  const float r = p.blur_r;      // [upstream] CheckPointOutsideBoundingBox grows the bbox by sqrt(blur_radius)
  if (!pixel_range_conservative(fminf(fminf(f.x0, f.x1), f.x2) - r, fmaxf(fmaxf(f.x0, f.x1), f.x2) + r, p.W, p.jx_scale, p.jx_off, xi_lo, xi_hi)) return false;
  return pixel_range_conservative(fminf(fminf(f.y0, f.y1), f.y2) - r, fmaxf(fmaxf(f.y0, f.y1), f.y2) + r, p.H, p.jy_scale, p.jy_off, yi_lo, yi_hi);
}

// ------------------------------------------------------------------------------------------------
// scatter pass
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned int smem_addr_pinned(const void* ptr) {
  unsigned int a;
  asm volatile("{ .reg .u64 t; cvta.to.shared.u64 t, %1; cvt.u32.u64 %0, t; }" : "=r"(a) : "l"(ptr));
  return a;
}
__device__ __forceinline__ void sts_u32(unsigned int a, unsigned int v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}

// exact test of one (face, pixel) candidate and the keyed min on the global key plane
// soft: blur_radius (squared), its root, and whether the fragment carries clipped barycentrics (all 0 / false: the hard rasterizer)
struct SoftMode {
  float blur, blur_r;
  bool clipb;
  __device__ __forceinline__ bool on() const { return blur > 0.f || clipb; }
};
__device__ __forceinline__ SoftMode soft_mode(const MeshParams& p) {
  SoftMode m;
  m.blur = p.blur_radius; m.blur_r = p.blur_r; m.clipb = p.flags & MVR_CLIP_BARYCENTRIC;
  return m;
}
// SOFT is a template parameter: the hard rasterizer's instantiation (MVTN's configuration) carries none of the blur code
template <bool SOFT = false>
__device__ __forceinline__ void resolve_pixel_with(const Face& fc, const FaceEdges& fe, int fid, unsigned int zmin_bits,
                                                   bool persp, float xf, float yf, unsigned long long* key_ptr,
                                                   const unsigned long long* prev_ptr, const unsigned long long cur,
                                                   const SoftMode sm = SoftMode{0.f, 0.f, false});
template <bool SOFT = false>
__device__ __forceinline__ void resolve_pixel(const Face& fc, const FaceEdges& fe, int fid, unsigned int zmin_bits,
                                              bool persp, float xf, float yf, unsigned long long* key_ptr,
                                              const unsigned long long* prev_ptr, const SoftMode sm = SoftMode{0.f, 0.f, false}) {
  resolve_pixel_with<SOFT>(fc, fe, fid, zmin_bits, persp, xf, yf, key_ptr, prev_ptr, __ldcg(key_ptr), sm);
}
// cur: a snapshot of *key_ptr taken earlier (keys only decrease, so a stale snapshot is merely less effective)
template <bool SOFT>
__device__ __forceinline__ void resolve_pixel_with(const Face& fc, const FaceEdges& fe, int fid, unsigned int zmin_bits,
                                                   bool persp, float xf, float yf, unsigned long long* key_ptr,
                                                   const unsigned long long* prev_ptr, const unsigned long long cur, const SoftMode sm) {
  // early depth reject: pz is a convex combination of the vertex depths up to a few ulp (perspective-corrected
  // barycentrics sum to 1 unless their 1e-8 denominator clamp acts, which needs z ~ 1e-4; plain barycentrics sum
  // to area/(area+1e-8), so zmin_bits is 0 for them), hence a face whose nearest vertex is clearly behind the
  // pixel's current winner cannot produce a smaller key.  A stale `cur` only makes the test less effective.
  if (zmin_bits > (unsigned int)(cur >> 32)) return;
  // [upstream] CheckPointOutsideBoundingBox (blur 0): the candidate generators only guarantee a superset of the bbox pixels
  const float grow = SOFT ? sm.blur_r : 0.f;
  if (SOFT) {
    if (xf > fmaxf(fmaxf(fc.x0, fc.x1), fc.x2) + grow || xf < fminf(fminf(fc.x0, fc.x1), fc.x2) - grow ||
        yf > fmaxf(fmaxf(fc.y0, fc.y1), fc.y2) + grow || yf < fminf(fminf(fc.y0, fc.y1), fc.y2) - grow) return;
  } else if (xf > fmaxf(fmaxf(fc.x0, fc.x1), fc.x2) || xf < fminf(fminf(fc.x0, fc.x1), fc.x2) || yf > fmaxf(fmaxf(fc.y0, fc.y1), fc.y2) ||
             yf < fminf(fminf(fc.y0, fc.y1), fc.y2)) return;
  float w[3], b[3], pz;
  if (SOFT) {      // [upstream] blur_radius > 0: inside, or closer than blur_radius (squared) to an edge
    float bc[3], sd;
    bool inside;
    raster_soft(fc, fe, persp, sm.clipb, xf, yf, b, bc, pz, sd, inside);
    if (pz < 0.f) return;
    if (!inside && !(sd < sm.blur)) return;
  } else if (!raster_test(fc, fe, persp, xf, yf, w, b, pz)) return;
  const unsigned long long key = make_key(pz, fid);
  if (key >= cur) return;
  if (prev_ptr && key <= __ldcg(prev_ptr)) return;
  atomicMin(key_ptr, key);      // result unused: RED.MIN.64 resolved in L2
}

// The pixel filter in FMA form.  Edge function i of the oracle, e_i = (px - xa) A - (py - ya) B (five IEEE
// operations), is evaluated as fma(px, A, fma(-py, B, C)) with C = ya B - xa A: two instructions.  The two differ by
// rounding only: with u = 2^-24, |px|, |py| <= pmax (1, or the aspect ratio of a non-square image) and
// S = (pmax + |xa|) |A| + (pmax + |ya|) |B|, the IEEE sequence is within
// 3 u S of the real value and the FMA form within 4 u S, so adding 16 u S to C makes "fma form > 0" a NECESSARY condition
// for "IEEE form > 0": the filter never drops a pixel the exact test (resolve_pixel_with) would accept, it only lets a few
// pixels within 2^-20 S of an edge through to be rejected there.  The sign of the area is folded into (A, B, C) first
// (negation is exact).
// span_edges keeps the filter in registers -- the thread that set a face up also walks its rows: per edge the
// coefficients (B, C' = C + 2^-20 S) of t(y) = fma(-y, B, C'), the reciprocal of A, and its class (flat / lower bound /
// upper bound)
struct SpanEdges {
  float B[3], C[3], rA[3];
  int cls;      // 2 bits per edge: 0 = no x dependence, 1 = lower bound on x (A > 0), 2 = upper bound (A < 0)
};
__device__ __forceinline__ SpanEdges span_edges(const Face& f, float pmax) {
  SpanEdges se;
  float A[3] = {f.y2 - f.y1, f.y0 - f.y2, f.y1 - f.y0};
  float B[3] = {f.x2 - f.x1, f.x0 - f.x2, f.x1 - f.x0};
  const float xa[3] = {f.x1, f.x2, f.x0}, ya[3] = {f.y1, f.y2, f.y0};
  const float area_p = ((f.x2 - f.x0) * A[2] - (f.y2 - f.y0) * B[2]) + MVR_K_EPS;
  const bool flip = !(area_p > 0.f);
  se.cls = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (flip) { A[i] = -A[i]; B[i] = -B[i]; }
    const float C = ya[i] * B[i] - xa[i] * A[i];
    const float S = (pmax + fabsf(xa[i])) * fabsf(A[i]) + (pmax + fabsf(ya[i])) * fabsf(B[i]);
    se.B[i] = B[i];
    se.C[i] = C + 9.5367431640625e-07f * S;      // 2^-20
    const bool flat = fabsf(A[i]) < 1e-30f;
    se.rA[i] = flat ? 0.f : rcp_fast(A[i]);
    se.cls |= (flat ? 0 : (A[i] > 0.f ? 1 : 2)) << (2 * i);
  }
  return se;
}

// The filter as a SCANLINE: the pixels of one bbox row that can pass it form an interval, and its end points come from the
// three filter inequalities  fma(xf, A_i, t_i) > 0,  t_i = fma(-yf, B_i, C_i')  (span_edges) solved for xf:
// xf > -t_i / A_i where A_i > 0, xf < -t_i / A_i where A_i < 0 (fma(xf, A, t) > 0 implies xf A + t > 0 in the reals: rounding
// to nearest never changes the sign of a non-zero value, and a real value <= 0 never rounds above 0).  An edge with no x
// dependence passes or fails the row as a whole.  The bounds are evaluated with an SFU reciprocal (<= 2 ulp on -t / A) and
// mapped to pixel columns (flipped column j grows with x; pixel index i = W - 1 - j) through the inverse pixel map widened
// by 8e-3 pixel -- an order of magnitude above the accumulated rounding (bound, map, pixel-centre table: ~1e-3 pixel at
// 4096 columns) -- so the interval is a SUPERSET of the filter's pixels, themselves a superset of the oracle's.  Which of
// them are fragments is the exact test's decision.  A face of 17 bbox pixels has ~4.6 inside (C2): a per-pixel filter loop
// spends 3/4 of its lanes on pixels this closed form excludes.
// Returns the number of candidate columns; xs = the first one (pixel index, xl <= xs, xs + count - 1 <= xl + bw - 1).
__device__ __forceinline__ int row_span_regs(const SpanEdges& se, float yf, int xl, int bw, int W, float jx_scale, float jx_off, int& xs) {
  float lo = -3.0e38f, hi = 3.0e38f;
  bool empty = false;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float t = fmaf(-yf, se.B[i], se.C[i]);
    const int c = (se.cls >> (2 * i)) & 3;
    const float bnd = -t * se.rA[i];
    if (c == 0) empty = empty || !(t > 0.f);
    else if (c == 1) lo = fmaxf(lo, bnd);
    else hi = fminf(hi, bnd);
  }
  float jlo = ceilf(fmaf(lo, jx_scale, jx_off) - 8e-3f), jhi = floorf(fmaf(hi, jx_scale, jx_off) + 8e-3f);
  jlo = fminf(fmaxf(jlo, -1.0f), (float)W); jhi = fminf(fmaxf(jhi, -1.0f), (float)W);      // (NaN -> -1)
  const int i_lo = max(W - 1 - (int)jhi, xl), i_hi = min(W - 1 - (int)jlo, xl + bw - 1);
  xs = i_lo;
  return empty ? 0 : max(i_hi - i_lo + 1, 0);
}

// Barycentrics of a pixel KNOWN to be inside its face, for shading only (images are compared at 1e-5): the edge
// functions come from the same projected vertices as the scatter pass, so they are bit-identical to the rasterizer's;
// only the six IEEE divisions are replaced by two SFU reciprocals (a few ulp on b, ~1e-7 on the colour).  The exact
// sequence (raster_test) is used whenever the caller asks for the barycentrics themselves.
__device__ __forceinline__ void shading_barycentrics(const Face& f, const FaceEdges& e, bool persp, float xf, float yf,
                                                     float b[3]) {
  const float e0 = (xf - f.x1) * e.A0 - (yf - f.y1) * e.B0;
  const float e1 = (xf - f.x2) * e.A1 - (yf - f.y2) * e.B1;
  const float e2 = (xf - f.x0) * e.A2 - (yf - f.y0) * e.B2;
  const float ia = rcp_fast(e.area_p);
  b[0] = e0 * ia; b[1] = e1 * ia; b[2] = e2 * ia;
  if (persp) {
    const float t0 = b[0] * f.z1 * f.z2, t1 = b[1] * f.z0 * f.z2, t2 = b[2] * f.z0 * f.z1;
    const float id = rcp_fast(fmaxf(t0 + t1 + t2, MVR_K_EPS));
    b[0] = t0 * id; b[1] = t1 * id; b[2] = t2 * id;
  }
}

}  // namespace mvr
