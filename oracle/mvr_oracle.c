/*
 * mvr_oracle.c -- CPU ORACLE for the MVRenderer hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library.  The product (mvtn_b200/) never links, imports or calls it.
 *
 * PARITY UNPINNED: the arithmetic of this path lives in PyTorch3D, a third-party dependency of
 * the reference (README.md:38 `conda install pytorch3d -c pytorch3d`, version unpinned) whose
 * sources are NOT under /root/reference and which cannot be installed here (no network).  The
 * reference itself holds no tests, golden images or known-answer vectors.  This file restates
 * the published algorithm of PyTorch3D v0.7.x's CPU path (the path every CPU tensor takes:
 * RasterizeMeshesNaiveCpu / RasterizePointsNaiveCpu / weightedSumNormCpu* / alphaCompositeCpu*)
 * and anchors on the reference's call sites:
 *     models/renderer.py:65-114   render_meshes  (Meshes.extend, look_at, FoVPerspective,
 *                                 MeshRasterizer, HardPhongShader, hard_rgb_blend)
 *     models/renderer.py:116-151  render_points  (Pointclouds.extend/scale_, FoVOrthographic,
 *                                 PointsRasterizer, NormWeightedCompositor)
 *     models/renderer.py:162-171  light_direction, :153-160 rendering_color
 *     util.py:403-420             check_valid_rotation_matrix
 * Each function below cites the upstream file it follows ([upstream], from the published source).
 *
 * Arithmetic contract: fp32, IEEE, operations in the written order, NO fused multiply-add
 * (build with -ffp-contract=off; upstream wheels are generic x86-64 builds without FMA).
 * Per-view gradient reductions are accumulated in double so that the oracle is the more exact
 * side of every tolerance comparison.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define K_EPS 1e-8f /* [upstream] csrc/utils/geometry_utils.h kEpsilon */
#define ORC_MAX_K 160 /* >= [upstream] kMaxPointsPerPixel = 150 */

/* Phong constants: DirectionalLights / Materials defaults used by renderer.py:190-191
 * ([upstream] renderer/lighting.py, renderer/materials.py). */
#define AMBIENT 0.5f
#define DIFFUSE 0.3f
#define SPECULAR 0.2f
#define SHININESS 64.0f

#define ORC_PERSPECTIVE_CORRECT 1
#define ORC_CULL_BACKFACES 2
#define ORC_COMPOSITE_ALPHA 4 /* AlphaCompositor instead of NormWeightedCompositor */
#define ORC_RGB_PER_ELEMENT 8 /* rgb is (total_elems,3) instead of a single 3-vector */

int orc_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}
void orc_set_num_threads(int n) {
#ifdef _OPENMP
  if (n > 0) omp_set_num_threads(n);
#else
  (void)n;
#endif
}

/* ------------------------------------------------------------------------------------------ */
/* Pixel grid: [upstream] csrc/utils/pixel_utils / rasterization_utils.h PixToNonSquareNdc     */
/* ------------------------------------------------------------------------------------------ */
static inline float pix_to_ndc(int i, int S1, int S2) {
  float range = 2.0f;
  if (S1 > S2) range = ((float)(S1 / S2)) * range;
  const float offset = range / 2.0f;
  return -offset + (range * (float)i + offset) / (float)S1;
}

/* ------------------------------------------------------------------------------------------ */
/* Cameras: [upstream] renderer/cameras.py camera_position_from_spherical_angles,              */
/* look_at_rotation, look_at_view_transform (called at renderer.py:79,122,168; ops.py:160)     */
/* ------------------------------------------------------------------------------------------ */
/* F.normalize: v / max(||v||_2, eps).  Returns whether the norm, not eps, divided. */
static inline int normalize3(const float v[3], float eps, float out[3]) {
  float n = sqrtf((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
  float d = n > eps ? n : eps;
  out[0] = v[0] / d; out[1] = v[1] / d; out[2] = v[2] / d;
  return n > eps;
}
static inline void cross3(const float a[3], const float b[3], float o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}

/* The branch decisions of one view's fp32 forward: which of F.normalize's eps clamps bound and whether the x axis was
 * replaced.  orc_look_at_backward differentiates the branches these name, so that near the poles, where the fp32 and the
 * double forward part ways, it differentiates the function the fp32 forward computed. */
typedef struct { int z_norm, x_norm, y_norm, xr_norm, replaced; } LookAtBranches;

static void look_at_view(float azim, float elev, float dist, float R[9], float T[3], float C[3], LookAtBranches* b) {
  const float deg = (float)(M_PI / 180.0);
  const float e = deg * elev, a = deg * azim, d = dist;
  float c[3];
  c[0] = (d * cosf(e)) * sinf(a);
  c[1] = d * sinf(e);
  c[2] = (d * cosf(e)) * cosf(a);
  const float up[3] = {0.f, 1.f, 0.f};
  float mz[3] = {0.f - c[0], 0.f - c[1], 0.f - c[2]}; /* at - camera_position */
  float x[3], y[3], z[3], t[3];
  b->z_norm = normalize3(mz, 1e-5f, z);
  cross3(up, z, t); b->x_norm = normalize3(t, 1e-5f, x);
  cross3(z, x, t); b->y_norm = normalize3(t, 1e-5f, y);
  /* isclose(x_axis, 0, atol=5e-3).all() -> x = normalize(cross(y, z)) */
  b->replaced = fabsf(x[0]) <= 5e-3f && fabsf(x[1]) <= 5e-3f && fabsf(x[2]) <= 5e-3f;
  b->xr_norm = 1;
  if (b->replaced) {
    cross3(y, z, t); b->xr_norm = normalize3(t, 1e-5f, x);
  }
  for (int r = 0; r < 3; ++r) { R[3 * r + 0] = x[r]; R[3 * r + 1] = y[r]; R[3 * r + 2] = z[r]; }
  /* T = -bmm(R^T, C) */
  for (int j = 0; j < 3; ++j)
    T[j] = -((R[0 + j] * c[0] + R[3 + j] * c[1]) + R[6 + j] * c[2]);
  C[0] = c[0]; C[1] = c[1]; C[2] = c[2];
}

void orc_look_at(const float* azim, const float* elev, const float* dist, int n,
                 float* R, float* T, float* C) {
  for (int i = 0; i < n; ++i) {
    float c[3];
    LookAtBranches b;
    look_at_view(azim[i], elev[i], dist[i], R + 9 * i, T + 3 * i, c, &b);
    if (C) { C[3 * i] = c[0]; C[3 * i + 1] = c[1]; C[3 * i + 2] = c[2]; }
  }
}

/* util.py:403-420 check_valid_rotation_matrix: allclose(R R^T, I, atol=1e-6) (rtol 1e-5 default)
 * and allclose(det R, 1) (rtol 1e-5, atol 1e-8).  Returns the number of INVALID matrices. */
int orc_count_invalid_rotations(const float* R, int n) {
  int bad = 0;
  for (int i = 0; i < n; ++i) {
    const float* r = R + 9 * i;
    int ok = 1;
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) {
        float s = (r[3 * a] * r[3 * b] + r[3 * a + 1] * r[3 * b + 1]) + r[3 * a + 2] * r[3 * b + 2];
        float I = a == b ? 1.f : 0.f;
        if (!(fabsf(s - I) <= 1e-6f + 1e-5f * fabsf(I))) ok = 0;
      }
    float det = r[0] * (r[4] * r[8] - r[5] * r[7]) - r[1] * (r[3] * r[8] - r[5] * r[6]) +
                r[2] * (r[3] * r[7] - r[4] * r[6]);
    if (!(fabsf(det - 1.f) <= 1e-8f + 1e-5f * 1.f)) ok = 0;
    bad += !ok;
  }
  return bad;
}

/* Backward of orc_look_at in double: (gR, gT, gC) -> (g_azim, g_elev, g_dist) per view.  Every branch (the eps clamps of the
 * four normalisations, the x-axis replacement) is the one the fp32 forward took (LookAtBranches): at elevation +-90 the fp32
 * cos is -4.4e-8 where the double one is 6e-17, and only the fp32 branches give fp32 PyTorch3D's gradient (DESIGN.md 2). */
static void normalize_bwd_d(const double v[3], double eps, int above, const double g[3], double gv[3]) {
  double n = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  if (above) {
    double u[3] = {v[0] / n, v[1] / n, v[2] / n};
    double d = u[0] * g[0] + u[1] * g[1] + u[2] * g[2];
    for (int i = 0; i < 3; ++i) gv[i] = (g[i] - u[i] * d) / n;
  } else {
    for (int i = 0; i < 3; ++i) gv[i] = g[i] / eps;
  }
}
static void cross_d(const double a[3], const double b[3], double o[3]) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
void orc_look_at_backward(const float* azim, const float* elev, const float* dist, int n,
                          const float* gR, const float* gT, const float* gC,
                          float* g_azim, float* g_elev, float* g_dist) {
  const double deg = M_PI / 180.0;
  const float degf = (float)(M_PI / 180.0);
  for (int i = 0; i < n; ++i) {
    float Rf[9], Tf[3], Cf[3];
    LookAtBranches b;
    look_at_view(azim[i], elev[i], dist[i], Rf, Tf, Cf, &b);
    /* Where the fp32 x axis is clamped (within 6e-4 deg of a pole) x = (up x z) / 1e-5 depends on cos(elev) itself, which the
     * fp32 rounding of the angle sets: fp32(pi/180) 90 lies 4.4e-8 rad past the pole, so there the camera sits on the other
     * side of it.  There the angles are taken as the fp32 forward rounds them; elsewhere that rounding is a 6e-8 relative
     * perturbation like any other and the exact angles are kept. */
    const double e = b.x_norm ? deg * elev[i] : (double)(degf * elev[i]);
    const double a = b.x_norm ? deg * azim[i] : (double)(degf * azim[i]);
    const double d = dist[i];
    const double ce = cos(e), se = sin(e), ca = cos(a), sa = sin(a);
    double c[3] = {d * ce * sa, d * se, d * ce * ca};
    double up[3] = {0, 1, 0}, mz[3] = {-c[0], -c[1], -c[2]};
    double nz = sqrt(mz[0] * mz[0] + mz[1] * mz[1] + mz[2] * mz[2]);
    double dz = b.z_norm ? nz : 1e-5;
    double z[3] = {mz[0] / dz, mz[1] / dz, mz[2] / dz};
    double tx[3]; cross_d(up, z, tx);
    double nx = sqrt(tx[0] * tx[0] + tx[1] * tx[1] + tx[2] * tx[2]);
    double dx = b.x_norm ? nx : 1e-5;
    double x[3] = {tx[0] / dx, tx[1] / dx, tx[2] / dx};
    double ty[3]; cross_d(z, x, ty);
    double ny = sqrt(ty[0] * ty[0] + ty[1] * ty[1] + ty[2] * ty[2]);
    double dy = b.y_norm ? ny : 1e-5;
    double y[3] = {ty[0] / dy, ty[1] / dy, ty[2] / dy};
    const int replaced = b.replaced;
    double x0[3] = {x[0], x[1], x[2]}; /* x before replacement: y depends on this one */
    double txr[3];
    if (replaced) {
      cross_d(y, z, txr);
      double nr = sqrt(txr[0] * txr[0] + txr[1] * txr[1] + txr[2] * txr[2]);
      double dr = b.xr_norm ? nr : 1e-5;
      for (int k = 0; k < 3; ++k) x[k] = txr[k] / dr;
    }
    /* upstream grads: R[r][0]=x[r], R[r][1]=y[r], R[r][2]=z[r];  T_j = -sum_r R[r][j] c_r */
    double gx[3] = {0, 0, 0}, gy[3] = {0, 0, 0}, gz[3] = {0, 0, 0}, gc[3] = {0, 0, 0};
    for (int r = 0; r < 3; ++r) {
      double g0 = gR ? gR[9 * i + 3 * r + 0] : 0, g1 = gR ? gR[9 * i + 3 * r + 1] : 0,
             g2 = gR ? gR[9 * i + 3 * r + 2] : 0;
      if (gT) {
        g0 += -gT[3 * i + 0] * c[r]; g1 += -gT[3 * i + 1] * c[r]; g2 += -gT[3 * i + 2] * c[r];
        gc[r] += -(gT[3 * i + 0] * x[r] + gT[3 * i + 1] * y[r] + gT[3 * i + 2] * z[r]);
      }
      gx[r] += g0; gy[r] += g1; gz[r] += g2;
      if (gC) gc[r] += gC[3 * i + r];
    }
    double gt[3], tmp[3];
    if (replaced) { /* x = normalize(cross(y, z)) */
      normalize_bwd_d(txr, 1e-5, b.xr_norm, gx, gt);
      cross_d(z, gt, tmp); for (int k = 0; k < 3; ++k) gy[k] += tmp[k];  /* d cross(y,z)/dy */
      cross_d(gt, y, tmp); for (int k = 0; k < 3; ++k) gz[k] += tmp[k];  /* d cross(y,z)/dz */
      gx[0] = gx[1] = gx[2] = 0;
    }
    /* y = normalize(cross(z, x0)) */
    normalize_bwd_d(ty, 1e-5, b.y_norm, gy, gt);
    cross_d(x0, gt, tmp); for (int k = 0; k < 3; ++k) gz[k] += tmp[k];
    cross_d(gt, z, tmp);  for (int k = 0; k < 3; ++k) gx[k] += tmp[k];
    /* x0 = normalize(cross(up, z)) */
    normalize_bwd_d(tx, 1e-5, b.x_norm, gx, gt);
    cross_d(gt, up, tmp); for (int k = 0; k < 3; ++k) gz[k] += tmp[k];
    /* z = normalize(-c) */
    normalize_bwd_d(mz, 1e-5, b.z_norm, gz, gt);
    for (int k = 0; k < 3; ++k) gc[k] -= gt[k];
    /* c(d, e, a) */
    double gd = gc[0] * ce * sa + gc[1] * se + gc[2] * ce * ca;
    double ge = gc[0] * (-d * se * sa) + gc[1] * (d * ce) + gc[2] * (-d * se * ca);
    double ga = gc[0] * (d * ce * ca) + gc[2] * (-d * ce * sa);
    if (g_dist) g_dist[i] = (float)gd;
    if (g_elev) g_elev[i] = (float)(ge * deg);
    if (g_azim) g_azim[i] = (float)(ga * deg);
  }
}

/* ------------------------------------------------------------------------------------------ */
/* Projection.  [upstream] Transform3d.transform_points with the 4x4 [[R,0],[T,1]] matrix,     */
/* FoVPerspectiveCameras.compute_projection_matrix (K00 = 2 znear/(max_x-min_x)), NDC z := view */
/* z (MeshRasterizer.transform / PointsRasterizer.transform).  Normative op order, SURVEY 8c.3  */
/* ------------------------------------------------------------------------------------------ */
static inline void world_to_view(const float X[3], const float* R, const float* T, float p[3]) {
  for (int j = 0; j < 3; ++j) p[j] = ((X[0] * R[0 + j] + X[1] * R[3 + j]) + X[2] * R[6 + j]) + T[j];
}
/* verts (V,3) world -> out (V,3) = (x_ndc, y_ndc, z_view) for ONE view. */
void orc_project_perspective(const float* verts, int V, const float* R, const float* T,
                             float k00, float k11, float* out) {
  for (int v = 0; v < V; ++v) {
    float p[3]; world_to_view(verts + 3 * v, R, T, p);
    out[3 * v + 0] = (p[0] * k00) / p[2];
    out[3 * v + 1] = (p[1] * k11) / p[2];
    out[3 * v + 2] = p[2];
  }
}
/* renderer.py:141-143: cloud scaled by 1/dist, then FoVOrthographic (x_ndc=x_v, y_ndc=y_v). */
void orc_project_orthographic(const float* pts, int P, const float* R, const float* T,
                              float inv_dist, float* out) {
  for (int p = 0; p < P; ++p) {
    float X[3] = {pts[3 * p] * inv_dist, pts[3 * p + 1] * inv_dist, pts[3 * p + 2] * inv_dist};
    world_to_view(X, R, T, out + 3 * p);
  }
}

/* ------------------------------------------------------------------------------------------ */
/* Mesh rasterizer: [upstream] csrc/rasterize_meshes/rasterize_meshes_cpu.cpp                  */
/* RasterizeMeshesNaiveCpu + csrc/utils/geometry_utils.h (blur_radius = 0, no bary clipping)   */
/* ------------------------------------------------------------------------------------------ */
static inline float edge_fn(float px, float py, float ax, float ay, float bx, float by) {
  return (px - ax) * (by - ay) - (py - ay) * (bx - ax);
}
static inline float point_line_dist2(float px, float py, float ax, float ay, float bx, float by) {
  const float dx = bx - ax, dy = by - ay;
  const float l2 = dx * dx + dy * dy;
  if (l2 <= K_EPS) return (px - bx) * (px - bx) + (py - by) * (py - by);
  const float t = (dx * (px - ax) + dy * (py - ay)) / l2;
  const float tt = fminf(fmaxf(t, 0.00f), 1.00f);
  const float qx = ax + tt * dx, qy = ay + tt * dy;
  return (px - qx) * (px - qx) + (py - qy) * (py - qy);
}
static inline void bary_forward(float px, float py, const float* fv, float w[3]) {
  const float area = edge_fn(fv[6], fv[7], fv[0], fv[1], fv[3], fv[4]) + K_EPS;
  w[0] = edge_fn(px, py, fv[3], fv[4], fv[6], fv[7]) / area;
  w[1] = edge_fn(px, py, fv[6], fv[7], fv[0], fv[1]) / area;
  w[2] = edge_fn(px, py, fv[0], fv[1], fv[3], fv[4]) / area;
}
static inline void bary_persp_forward(const float w[3], float z0, float z1, float z2, float b[3]) {
  const float t0 = w[0] * z1 * z2, t1 = w[1] * z0 * z2, t2 = w[2] * z0 * z1;
  const float denom = fmaxf(t0 + t1 + t2, K_EPS);
  b[0] = t0 / denom; b[1] = t1 / denom; b[2] = t2 / denom;
}

/* [upstream] renderer/mesh/clip.py clip_faces / _find_verts_intersecting_clipping_plane (z plane only: MeshRasterizer
 * passes cull_to_frustum=False).  A face with one or two vertices behind z = c is replaced by one (case 3: two
 * behind) or two (case 4: one behind) triangles:
 *     p1 = the lone vertex (in front for case 3, behind for case 4), p2, p3 = the next two in cyclic order,
 *     w2 = (p1.z - c) / (p1.z - p2.z), w3 = (p1.z - c) / (p1.z - p3.z),
 *     p4 = p1 (1 - w2) + p2 w2, p5 = p1 (1 - w3) + p3 w3 -- with perspective_correct the xy are interpolated
 *     un-projected: ((p1.xy p1.z)(1 - w) + (p2.xy p2.z) w) / c,
 *     case 3 -> (p4, p5, p1);  case 4 -> (p4, p2, p5), (p5, p2, p3)  (consecutive in the clipped face list).
 * conv[s][3 j + k] = barycentric weight of ORIGINAL vertex j in clipped vertex k of sub-triangle s
 * (convert_clipped_rasterization_to_original_faces: bary_unclipped = conv . bary_clipped).
 * Returns the number of sub-triangles (1 or 2), or 0 when the face does not straddle the plane.
 * info: i1 | case4 << 2 (for the backward). */
static int clip_face(const float* v, float c, int persp, float sub[2][9], float conv[2][9], int* info) {
  const int b0 = v[2] < c, b1 = v[5] < c, b2 = v[8] < c;
  const int nb = b0 + b1 + b2;
  if (nb == 0 || nb == 3) return 0;
  const int case4 = nb == 1;
  int i1;
  if (case4) i1 = b0 ? 0 : (b1 ? 1 : 2);       /* the vertex behind */
  else i1 = !b0 ? 0 : (!b1 ? 1 : 2);           /* the vertex in front */
  const int i2 = (i1 + 1) % 3, i3 = (i1 + 2) % 3;
  const float* p1 = v + 3 * i1; const float* p2 = v + 3 * i2; const float* p3 = v + 3 * i3;
  const float w2 = (p1[2] - c) / (p1[2] - p2[2]);
  const float w3 = (p1[2] - c) / (p1[2] - p3[2]);
  const float om2 = 1.0f - w2, om3 = 1.0f - w3;
  float p4[3], p5[3];
  for (int d = 0; d < 3; ++d) { p4[d] = p1[d] * om2 + p2[d] * w2; p5[d] = p1[d] * om3 + p3[d] * w3; }
  if (persp) {
    for (int d = 0; d < 2; ++d) {
      const float a1 = p1[d] * p1[2], a2 = p2[d] * p2[2], a3 = p3[d] * p3[2];
      p4[d] = (a1 * om2 + a2 * w2) / c;
      p5[d] = (a1 * om3 + a3 * w3) / c;
    }
  }
  float bc[5][3];                                /* barycentrics of p1..p5 in the original triangle */
  memset(bc, 0, sizeof(bc));
  bc[0][i1] = 1.f; bc[1][i2] = 1.f; bc[2][i3] = 1.f;
  bc[3][i1] = om2; bc[3][i2] = w2;
  bc[4][i1] = om3; bc[4][i3] = w3;
  const float* P[5] = {p1, p2, p3, p4, p5};
  int pick[2][3];
  int ns;
  if (!case4) { ns = 1; pick[0][0] = 3; pick[0][1] = 4; pick[0][2] = 0; }
  else { ns = 2; pick[0][0] = 3; pick[0][1] = 1; pick[0][2] = 4; pick[1][0] = 4; pick[1][1] = 1; pick[1][2] = 2; }
  for (int s2 = 0; s2 < ns; ++s2)
    for (int k = 0; k < 3; ++k) {
      memcpy(sub[s2] + 3 * k, P[pick[s2][k]], 12);
      for (int j = 0; j < 3; ++j) conv[s2][3 * j + k] = bc[pick[s2][k]][j];
    }
  if (info) *info = i1 | (case4 << 2);
  return ns;
}
static inline void conv_bary(const float* conv, const float bc[3], float bo[3]) {
  for (int j = 0; j < 3; ++j) bo[j] = (conv[3 * j] * bc[0] + conv[3 * j + 1] * bc[1]) + conv[3 * j + 2] * bc[2];
}

typedef struct { float z; int idx; float d; float b0, b1, b2; } frag_t;
static inline int frag_less(const frag_t* a, const frag_t* b) {
  /* std::tuple<float,int,...> operator< : lexicographic; idx is unique so (z, idx) decides */
  if (a->z < b->z) return 1;
  if (b->z < a->z) return 0;
  return a->idx < b->idx;
}
/* keep the K lexicographically smallest, ascending (== priority_queue push / pop-when->K) */
static inline void frag_insert(frag_t* q, int* n, int K, const frag_t* f) {
  int i = *n;
  if (i == K) { if (!frag_less(f, &q[K - 1])) return; i = K - 1; } else { (*n)++; }
  while (i > 0 && frag_less(f, &q[i - 1])) { q[i] = q[i - 1]; --i; }
  q[i] = *f;
}

/*
 * face_verts (F_total,3,3): (x_ndc, y_ndc, z_view) per face corner; first_idx/num_faces (N).
 * face_skip (F_total) optional: faces removed before rasterization (near-plane cull).
 * Outputs (N,H,W,K): pix_to_face int32 PACKED index (-1 pad), zbuf, dists (-1 pad),
 * bary (N,H,W,K,3) (-1 pad).  zbuf/bary/dists may be NULL.
 */
void orc_rasterize_meshes(const float* face_verts, const int* first_idx, const int* num_faces,
                          const unsigned char* face_skip, int N, int H, int W, int K, int flags,
                          int* pix_to_face, float* zbuf, float* bary, float* dists) {
  const int persp = flags & ORC_PERSPECTIVE_CORRECT, cull = flags & ORC_CULL_BACKFACES;
  int Ftot = 0;
  for (int n = 0; n < N; ++n) if (first_idx[n] + num_faces[n] > Ftot) Ftot = first_idx[n] + num_faces[n];
  /* ComputeFaceBoundingBoxes / ComputeFaceAreas */
  float* bbox = (float*)malloc(sizeof(float) * 5 * (size_t)(Ftot > 0 ? Ftot : 1));
  float* area = (float*)malloc(sizeof(float) * (size_t)(Ftot > 0 ? Ftot : 1));
#pragma omp parallel for schedule(static)
  for (int f = 0; f < Ftot; ++f) {
    const float* v = face_verts + 9 * (size_t)f;
    bbox[5 * f + 0] = fminf(fminf(v[0], v[3]), v[6]);
    bbox[5 * f + 1] = fminf(fminf(v[1], v[4]), v[7]);
    bbox[5 * f + 2] = fmaxf(fmaxf(v[0], v[3]), v[6]);
    bbox[5 * f + 3] = fmaxf(fmaxf(v[1], v[4]), v[7]);
    bbox[5 * f + 4] = fminf(fminf(v[2], v[5]), v[8]);
    area[f] = edge_fn(v[0], v[1], v[3], v[4], v[6], v[7]); /* EdgeFunctionForward(v0, v1, v2) */
  }
#pragma omp parallel for collapse(2) schedule(dynamic, 4)
  for (int n = 0; n < N; ++n) {
    for (int yi = 0; yi < H; ++yi) {
      frag_t q[ORC_MAX_K];
      const int f0 = first_idx[n], f1 = first_idx[n] + num_faces[n];
      const float yf = pix_to_ndc(H - 1 - yi, H, W);
      for (int xi = 0; xi < W; ++xi) {
        const float xf = pix_to_ndc(W - 1 - xi, W, H);
        int nq = 0;
        for (int f = f0; f < f1; ++f) {
          if (face_skip && face_skip[f]) continue;
          const float fa = area[f];
          if (cull && fa < 0.f) continue;
          if (fa <= K_EPS && fa >= -1.0f * K_EPS) continue;
          const float* bb = bbox + 5 * (size_t)f;
          /* CheckPointOutsideBoundingBox, blur 0; z_invalid = zmin < kEpsilon */
          if (xf > bb[2] || xf < bb[0] || yf > bb[3] || yf < bb[1] || bb[4] < K_EPS) continue;
          const float* v = face_verts + 9 * (size_t)f;
          float w[3], b[3];
          bary_forward(xf, yf, v, w);
          if (persp) bary_persp_forward(w, v[2], v[5], v[8], b);
          else { b[0] = w[0]; b[1] = w[1]; b[2] = w[2]; }
          const float pz = b[0] * v[2] + b[1] * v[5] + b[2] * v[8];
          if (pz < 0) continue;
          const int inside = b[0] > 0.0f && b[1] > 0.0f && b[2] > 0.0f;
          if (!inside) continue; /* !inside && dist >= blur_radius(=0) */
          const float e01 = point_line_dist2(xf, yf, v[0], v[1], v[3], v[4]);
          const float e02 = point_line_dist2(xf, yf, v[0], v[1], v[6], v[7]);
          const float e12 = point_line_dist2(xf, yf, v[3], v[4], v[6], v[7]);
          const float d = fminf(fminf(e01, e02), e12);
          frag_t fr = {pz, f, -d, b[0], b[1], b[2]};
          frag_insert(q, &nq, K, &fr);
        }
        const size_t o = (((size_t)n * H + yi) * W + xi) * K;
        for (int k = 0; k < K; ++k) {
          const int ok = k < nq;
          pix_to_face[o + k] = ok ? q[k].idx : -1;
          if (zbuf) zbuf[o + k] = ok ? q[k].z : -1.f;
          if (dists) dists[o + k] = ok ? q[k].d : -1.f;
          if (bary) {
            bary[3 * (o + k) + 0] = ok ? q[k].b0 : -1.f;
            bary[3 * (o + k) + 1] = ok ? q[k].b1 : -1.f;
            bary[3 * (o + k) + 2] = ok ? q[k].b2 : -1.f;
          }
        }
      }
    }
  }
  free(bbox); free(area);
}

/* [upstream] geometry_utils.h BarycentricPerspectiveCorrectionBackward, BarycentricCoordsBackward,
 * EdgeFunctionBackward; rasterize_meshes_cpu.cpp RasterizeMeshesBackwardCpu (grad_dists omitted:
 * HardPhongShader never produces one, SURVEY 3.4).  grad_face_verts (F_total,3,3) accumulated in
 * double then cast.  Per pixel/k helper shared with the fused pipeline below. */
static void raster_bwd_one(float xf, float yf, const float* v, int persp, const double gb_in[3],
                           double gz_up, double gfv[9]) {
  double w[3], area, e[3];
  {
    area = (double)edge_fn(v[6], v[7], v[0], v[1], v[3], v[4]) + (double)K_EPS;
    e[0] = edge_fn(xf, yf, v[3], v[4], v[6], v[7]);
    e[1] = edge_fn(xf, yf, v[6], v[7], v[0], v[1]);
    e[2] = edge_fn(xf, yf, v[0], v[1], v[3], v[4]);
    for (int i = 0; i < 3; ++i) w[i] = e[i] / area;
  }
  const double z0 = v[2], z1 = v[5], z2 = v[8];
  double b[3] = {w[0], w[1], w[2]};
  double t[3] = {0, 0, 0}, denom = 1;
  if (persp) {
    t[0] = w[0] * z1 * z2; t[1] = w[1] * z0 * z2; t[2] = w[2] * z0 * z1;
    denom = t[0] + t[1] + t[2]; if (denom < (double)K_EPS) denom = K_EPS;
    for (int i = 0; i < 3; ++i) b[i] = t[i] / denom;
  }
  /* grad_bary_f_sum = grad_bary_upstream + grad_zbuf_upstream * (z0,z1,z2) */
  double gb[3] = {gb_in[0] + gz_up * z0, gb_in[1] + gz_up * z1, gb_in[2] + gz_up * z2};
  double dz[3] = {0, 0, 0};
  if (persp) {
    const double gden_top = gb[0] * t[0] + gb[1] * t[1] + gb[2] * t[2];
    const double gden = -gden_top / (denom * denom);
    const double gt0 = gden + gb[0] / denom, gt1 = gden + gb[1] / denom, gt2 = gden + gb[2] / denom;
    gb[0] = gt0 * z1 * z2; gb[1] = gt1 * z0 * z2; gb[2] = gt2 * z0 * z1;
    dz[0] = gt1 * w[1] * z2 + gt2 * w[2] * z1;
    dz[1] = gt0 * w[0] * z2 + gt2 * w[2] * z0;
    dz[2] = gt0 * w[0] * z1 + gt1 * w[1] * z0;
  }
  /* BarycentricCoordsBackward: w_i = e_i / area */
  const double x0 = v[0], y0 = v[1], x1 = v[3], y1 = v[4], x2 = v[6], y2 = v[7];
  const double ge[3] = {gb[0] / area, gb[1] / area, gb[2] / area};
  const double garea = -(gb[0] * e[0] + gb[1] * e[1] + gb[2] * e[2]) / (area * area);
  double g[6] = {0, 0, 0, 0, 0, 0}; /* x0 y0 x1 y1 x2 y2 */
  /* E(p,a,b) = (px-ax)(by-ay) - (py-ay)(bx-ax): dE/da = (py-by, bx-px), dE/db = (ay-py, px-ax) */
#define EDGE_BWD(G, PX, PY, AX, AY, BX, BY, IA, IB)                       \
  g[2 * IA] += (G) * ((PY) - (BY)); g[2 * IA + 1] += (G) * ((BX) - (PX)); \
  g[2 * IB] += (G) * ((AY) - (PY)); g[2 * IB + 1] += (G) * ((PX) - (AX));
  EDGE_BWD(ge[0], xf, yf, x1, y1, x2, y2, 1, 2)
  EDGE_BWD(ge[1], xf, yf, x2, y2, x0, y0, 2, 0)
  EDGE_BWD(ge[2], xf, yf, x0, y0, x1, y1, 0, 1)
  /* area = E(v2, v0, v1): p = v2, a = v0, b = v1; dE/dp = (by-ay, ax-bx) */
  EDGE_BWD(garea, x2, y2, x0, y0, x1, y1, 0, 1)
  g[4] += garea * (y1 - y0); g[5] += garea * (x0 - x1);
#undef EDGE_BWD
  for (int i = 0; i < 3; ++i) {
    gfv[3 * i + 0] += g[2 * i];
    gfv[3 * i + 1] += g[2 * i + 1];
    gfv[3 * i + 2] += gz_up * b[i] + dz[i];
  }
}

/* Backward of clip_face + conv_bary for one pixel of sub-triangle s2 (autograd of [upstream] clip.py, whose tensor
 * ops are all differentiable): gq (3,3) = gradient w.r.t. the clipped triangle's (x, y, z) from raster_bwd_one,
 * gb (3) = gradient w.r.t. the UNCLIPPED barycentrics, bcl = the clipped barycentrics.  Accumulates into gfv (3,3),
 * the gradient w.r.t. the original face's (x_ndc, y_ndc, z_view). */
static void clip_face_bwd(const float* v, float c, int persp, int info, int s2, const double gq[9],
                          const double gb[3], const float bcl[3], double gfv[9]) {
  const int i1 = info & 3, case4 = (info >> 2) & 1;
  const int i2 = (i1 + 1) % 3, i3 = (i1 + 2) % 3;
  const double p1[3] = {v[3 * i1], v[3 * i1 + 1], v[3 * i1 + 2]};
  const double p2[3] = {v[3 * i2], v[3 * i2 + 1], v[3 * i2 + 2]};
  const double p3[3] = {v[3 * i3], v[3 * i3 + 1], v[3 * i3 + 2]};
  const double w2 = (p1[2] - c) / (p1[2] - p2[2]), w3 = (p1[2] - c) / (p1[2] - p3[2]);
  int pick[3];
  if (!case4) { pick[0] = 3; pick[1] = 4; pick[2] = 0; }
  else if (s2 == 0) { pick[0] = 3; pick[1] = 1; pick[2] = 4; }
  else { pick[0] = 4; pick[1] = 1; pick[2] = 2; }
  double gP[5][3];
  memset(gP, 0, sizeof(gP));
  double gw2 = 0, gw3 = 0;
  for (int k = 0; k < 3; ++k) {
    for (int d = 0; d < 3; ++d) gP[pick[k]][d] += gq[3 * k + d];
    /* conv[:, k] = barycentrics of clipped vertex k: p4 -> (1 - w2) e_i1 + w2 e_i2, p5 -> (1 - w3) e_i1 + w3 e_i3 */
    if (pick[k] == 3) gw2 += (double)bcl[k] * (gb[i2] - gb[i1]);
    if (pick[k] == 4) gw3 += (double)bcl[k] * (gb[i3] - gb[i1]);
  }
  double g1[3] = {gP[0][0], gP[0][1], gP[0][2]}, g2[3] = {gP[1][0], gP[1][1], gP[1][2]}, g3[3] = {gP[2][0], gP[2][1], gP[2][2]};
  /* p4 = f(p1, p2, w2), p5 = f(p1, p3, w3) */
  for (int q = 0; q < 2; ++q) {
    const double* gp = q == 0 ? gP[3] : gP[4];
    const double* po = q == 0 ? p2 : p3;
    double* go = q == 0 ? g2 : g3;
    const double w = q == 0 ? w2 : w3;
    double* gw = q == 0 ? &gw2 : &gw3;
    for (int d = 0; d < 2; ++d) {
      if (persp) {     /* p.xy = ((p1.xy p1.z)(1 - w) + (po.xy po.z) w) / c */
        const double A = p1[d] * p1[2], Bq = po[d] * po[2];
        const double gA = gp[d] * (1 - w) / c, gB = gp[d] * w / c;
        *gw += gp[d] * (Bq - A) / c;
        g1[d] += gA * p1[2]; g1[2] += gA * p1[d];
        go[d] += gB * po[2]; go[2] += gB * po[d];
      } else {
        g1[d] += gp[d] * (1 - w); go[d] += gp[d] * w; *gw += gp[d] * (po[d] - p1[d]);
      }
    }
    g1[2] += gp[2] * (1 - w); go[2] += gp[2] * w; *gw += gp[2] * (po[2] - p1[2]);
  }
  /* w2 = (z1 - c) / (z1 - z2) */
  {
    const double d2 = p1[2] - p2[2], d3 = p1[2] - p3[2];
    g1[2] += gw2 * (c - p2[2]) / (d2 * d2); g2[2] += gw2 * (p1[2] - c) / (d2 * d2);
    g1[2] += gw3 * (c - p3[2]) / (d3 * d3); g3[2] += gw3 * (p1[2] - c) / (d3 * d3);
  }
  for (int d = 0; d < 3; ++d) { gfv[3 * i1 + d] += g1[d]; gfv[3 * i2 + d] += g2[d]; gfv[3 * i3 + d] += g3[d]; }
}

/* Which sub-triangle of a clipped face owns pixel (xf, yf): the one the rasterizer keeps, i.e. the inside one with the
 * smallest (pz, index).  Returns -1 if none (cannot happen for a pixel whose pix_to_face is this face). */
static int clip_pick_sub(float xf, float yf, float sub[2][9], int ns, int persp, float bcl[3]) {
  int best = -1; float bz = 0.f;
  for (int s2 = 0; s2 < ns; ++s2) {
    const float* tv = sub[s2];
    const float fa = edge_fn(tv[0], tv[1], tv[3], tv[4], tv[6], tv[7]);
    if (fa <= K_EPS && fa >= -1.0f * K_EPS) continue;
    float w[3], b[3];
    bary_forward(xf, yf, tv, w);
    if (persp) bary_persp_forward(w, tv[2], tv[5], tv[8], b); else { b[0] = w[0]; b[1] = w[1]; b[2] = w[2]; }
    const float pz = b[0] * tv[2] + b[1] * tv[5] + b[2] * tv[8];
    if (pz < 0 || !(b[0] > 0.0f && b[1] > 0.0f && b[2] > 0.0f)) continue;
    if (best < 0 || pz < bz) { best = s2; bz = pz; memcpy(bcl, b, 12); }
  }
  return best;
}

void orc_rasterize_meshes_backward(const float* face_verts, const int* pix_to_face,
                                   const float* grad_zbuf, const float* grad_bary, int N, int H,
                                   int W, int K, int Ftot, int flags, float* grad_face_verts) {
  const int persp = flags & ORC_PERSPECTIVE_CORRECT;
  double* acc = (double*)calloc((size_t)9 * (Ftot > 0 ? Ftot : 1), sizeof(double));
  for (int n = 0; n < N; ++n)
    for (int yi = 0; yi < H; ++yi) {
      const float yf = pix_to_ndc(H - 1 - yi, H, W);
      for (int xi = 0; xi < W; ++xi) {
        const float xf = pix_to_ndc(W - 1 - xi, W, H);
        for (int k = 0; k < K; ++k) {
          const size_t o = (((size_t)n * H + yi) * W + xi) * K + k;
          const int f = pix_to_face[o];
          if (f < 0) continue;
          double gb[3] = {0, 0, 0};
          if (grad_bary) { gb[0] = grad_bary[3 * o]; gb[1] = grad_bary[3 * o + 1]; gb[2] = grad_bary[3 * o + 2]; }
          raster_bwd_one(xf, yf, face_verts + 9 * (size_t)f, persp, gb, grad_zbuf ? grad_zbuf[o] : 0.0,
                         acc + 9 * (size_t)f);
        }
      }
    }
  for (size_t i = 0; i < (size_t)9 * Ftot; ++i) grad_face_verts[i] = (float)acc[i];
  free(acc);
}

/* ------------------------------------------------------------------------------------------ */
/* Vertex normals: [upstream] structures/meshes.py Meshes._compute_vertex_normals              */
/* ------------------------------------------------------------------------------------------ */
void orc_vertex_normals(const float* verts, const int* faces, int V, int F, float* normals) {
  memset(normals, 0, sizeof(float) * 3 * (size_t)V);
  /* upstream runs three successive index_add passes in face order, one per CORNER, each with that corner's own
   * cross product (equal in exact arithmetic, ~1 ulp apart in fp32):
   *   faces[:,1] += (v2 - v1) x (v0 - v1);  faces[:,2] += (v0 - v2) x (v1 - v2);  faces[:,0] += (v1 - v0) x (v2 - v0) */
  static const int corner[3] = {1, 2, 0};
  for (int pass = 0; pass < 3; ++pass) {
    const int c = corner[pass], n = (c + 1) % 3, pr = (c + 2) % 3;
    for (int f = 0; f < F; ++f) {
      const float* vc = verts + 3 * (size_t)faces[3 * f + c];
      const float* vn = verts + 3 * (size_t)faces[3 * f + n];
      const float* vp = verts + 3 * (size_t)faces[3 * f + pr];
      const float a[3] = {vn[0] - vc[0], vn[1] - vc[1], vn[2] - vc[2]};
      const float b[3] = {vp[0] - vc[0], vp[1] - vc[1], vp[2] - vc[2]};
      float fn[3]; cross3(a, b, fn);
      float* o = normals + 3 * (size_t)faces[3 * f + c];
      o[0] += fn[0]; o[1] += fn[1]; o[2] += fn[2];
    }
  }
  for (int v = 0; v < V; ++v) { float t[3]; normalize3(normals + 3 * v, 1e-6f, t); memcpy(normals + 3 * v, t, 12); }
}

/* ------------------------------------------------------------------------------------------ */
/* Phong shading + hard blend for one pixel.  [upstream] renderer/mesh/shading.py phong_shading, */
/* renderer/lighting.py diffuse/specular, renderer/blending.py hard_rgb_blend,                  */
/* csrc/interp_face_attrs (b0*a0 + b1*a1 + b2*a2).                                              */
/* ------------------------------------------------------------------------------------------ */
static inline void interp3(const float b[3], const float* a0, const float* a1, const float* a2, float o[3]) {
  for (int d = 0; d < 3; ++d) o[d] = (b[0] * a0[d] + b[1] * a1[d]) + b[2] * a2[d];
}
static void phong_pixel(const float b[3], const float* X[3], const float* Nv[3], const float* col[3],
                        const float* L, const float* Cc, float rgb[3]) {
  float P[3], Nn[3], tex[3], n[3], l[3], vv[3], v[3], r[3];
  interp3(b, X[0], X[1], X[2], P);
  interp3(b, Nv[0], Nv[1], Nv[2], Nn);
  interp3(b, col[0], col[1], col[2], tex);
  normalize3(Nn, 1e-6f, n);
  normalize3(L, 1e-6f, l);
  const float cosang = (n[0] * l[0] + n[1] * l[1]) + n[2] * l[2];
  const float diff = cosang > 0.f ? cosang : 0.f; /* relu */
  const float mask = cosang > 0.f ? 1.f : 0.f;
  vv[0] = Cc[0] - P[0]; vv[1] = Cc[1] - P[1]; vv[2] = Cc[2] - P[2];
  normalize3(vv, 1e-6f, v);
  for (int d = 0; d < 3; ++d) r[d] = -l[d] + 2.f * (cosang * n[d]);
  float dt = (v[0] * r[0] + v[1] * r[1]) + v[2] * r[2];
  float alpha = (dt > 0.f ? dt : 0.f) * mask;
  const float spec = SPECULAR * powf(alpha, SHININESS);
  for (int c = 0; c < 3; ++c) rgb[c] = (AMBIENT + DIFFUSE * diff) * tex[c] + spec;
}

/* Backward of phong_pixel in double: g (3) -> gb (3), gC (3); optionally gX/gN/gcol (3x3 each). */
static void phong_pixel_bwd(const float bf[3], const float* X[3], const float* Nv[3],
                            const float* col[3], const float* L, const float* Cc, const double g[3],
                            double gb[3], double gC[3], double* gX, double* gN, double* gcol) {
  double b[3] = {bf[0], bf[1], bf[2]}, P[3], Nn[3], tex[3];
  for (int d = 0; d < 3; ++d) {
    P[d] = b[0] * X[0][d] + b[1] * X[1][d] + b[2] * X[2][d];
    Nn[d] = b[0] * Nv[0][d] + b[1] * Nv[1][d] + b[2] * Nv[2][d];
    tex[d] = b[0] * col[0][d] + b[1] * col[1][d] + b[2] * col[2][d];
  }
  double nn = sqrt(Nn[0] * Nn[0] + Nn[1] * Nn[1] + Nn[2] * Nn[2]);
  double dn = nn > 1e-6 ? nn : 1e-6;
  double n[3] = {Nn[0] / dn, Nn[1] / dn, Nn[2] / dn};
  double ln = sqrt((double)L[0] * L[0] + (double)L[1] * L[1] + (double)L[2] * L[2]);
  double dl = ln > 1e-6 ? ln : 1e-6;
  double l[3] = {L[0] / dl, L[1] / dl, L[2] / dl};
  double cosang = n[0] * l[0] + n[1] * l[1] + n[2] * l[2];
  double diff = cosang > 0 ? cosang : 0;
  double vv[3] = {Cc[0] - P[0], Cc[1] - P[1], Cc[2] - P[2]};
  double vn = sqrt(vv[0] * vv[0] + vv[1] * vv[1] + vv[2] * vv[2]);
  double dv = vn > 1e-6 ? vn : 1e-6;
  double v[3] = {vv[0] / dv, vv[1] / dv, vv[2] / dv};
  double r[3]; for (int d = 0; d < 3; ++d) r[d] = -l[d] + 2.0 * cosang * n[d];
  double dt = v[0] * r[0] + v[1] * r[1] + v[2] * r[2];
  int lit = cosang > 0;
  double alpha = (dt > 0 && lit) ? dt : 0;
  /* color_c = (amb + dif*diff) * tex_c + spec*alpha^64 */
  double gtex[3], gdiff = 0, gs = 0;
  for (int c = 0; c < 3; ++c) {
    gtex[c] = g[c] * ((double)AMBIENT + (double)DIFFUSE * diff);
    gdiff += g[c] * tex[c] * (double)DIFFUSE;
    gs += g[c] * (double)SPECULAR;
  }
  double galpha = gs * 64.0 * pow(alpha, 63.0);
  double gdt = (dt > 0 && lit) ? galpha : 0;
  double gv[3], gr[3];
  for (int d = 0; d < 3; ++d) { gv[d] = gdt * r[d]; gr[d] = gdt * v[d]; }
  double gcos = (lit ? gdiff : 0) + 2.0 * (gr[0] * n[0] + gr[1] * n[1] + gr[2] * n[2]);
  double gn[3]; for (int d = 0; d < 3; ++d) gn[d] = 2.0 * cosang * gr[d] + gcos * l[d];
  double gNn[3], gvv[3];
  if (nn > 1e-6) { double dd = n[0] * gn[0] + n[1] * gn[1] + n[2] * gn[2]; for (int d = 0; d < 3; ++d) gNn[d] = (gn[d] - n[d] * dd) / nn; }
  else for (int d = 0; d < 3; ++d) gNn[d] = gn[d] / 1e-6;
  if (vn > 1e-6) { double dd = v[0] * gv[0] + v[1] * gv[1] + v[2] * gv[2]; for (int d = 0; d < 3; ++d) gvv[d] = (gv[d] - v[d] * dd) / vn; }
  else for (int d = 0; d < 3; ++d) gvv[d] = gv[d] / 1e-6;
  for (int d = 0; d < 3; ++d) gC[d] = gvv[d];
  for (int i = 0; i < 3; ++i) {
    double s = 0;
    for (int d = 0; d < 3; ++d) s += gtex[d] * col[i][d] + gNn[d] * Nv[i][d] - gvv[d] * X[i][d];
    gb[i] = s;
    if (gX) for (int d = 0; d < 3; ++d) gX[3 * i + d] += -b[i] * gvv[d];
    if (gN) for (int d = 0; d < 3; ++d) gN[3 * i + d] += b[i] * gNn[d];
    if (gcol) for (int d = 0; d < 3; ++d) gcol[3 * i + d] += b[i] * gtex[d];
  }
}

/* ------------------------------------------------------------------------------------------ */
/* Fused mesh pipeline (renderer.py:65-114 for B objects x M views).                           */
/*  verts (Vtot,3), faces (Ftot,3) int32 mesh-local vertex ids, vert_off/face_off (B+1),       */
/*  normals (Vtot,3) from orc_vertex_normals, rgb: (3) or (Vtot,3) [ORC_RGB_PER_ELEMENT],      */
/*  R (B*M,3,3), T, C (B*M,3); light (1,3) if light_stride==0 else (B*M,3); bg (3).            */
/*  out images (B*M,3,H,W); pix_to_face (B*M,H,W,K) VIEW-LOCAL face ids (-1 pad);               */
/*  optional zbuf (..K), bary (..K,3), dists (..K).  counters[0] += faces straddling z_clip     */
/*  (they are clipped against it as [upstream] clip.py does; z_clip < 0 disables cull and clip). */
/* ------------------------------------------------------------------------------------------ */
void orc_mesh_forward(const float* verts, const int* faces, const int* vert_off, const int* face_off,
                      const float* normals, const float* rgb, int B, int M, const float* R,
                      const float* T, const float* C, const float* light, int light_stride,
                      const float* bg, float k00, float k11, float z_clip, int H, int W, int K,
                      int flags, float* images, int* pix_to_face, float* zbuf, float* bary,
                      float* dists, long long* counters) {
  long long straddle = 0;
  const int persp = flags & ORC_PERSPECTIVE_CORRECT;
  for (int n = 0; n < B * M; ++n) {
    const int b = n / M;
    const int V = vert_off[b + 1] - vert_off[b], F = face_off[b + 1] - face_off[b];
    const float* vw = verts + 3 * (size_t)vert_off[b];
    const int* fc = faces + 3 * (size_t)face_off[b];
    const size_t Fa = (size_t)(F > 0 ? F : 1);
    float* ndc = (float*)malloc(sizeof(float) * 3 * (size_t)(V > 0 ? V : 1));
    /* the CLIPPED face list ([upstream] clip.py ClippedFaces): unclipped faces in their original order, culled faces
     * removed, clipped faces replaced in place by their one or two sub-triangles */
    float* fvc = (float*)malloc(sizeof(float) * 9 * 2 * Fa);
    float* cnv = (float*)malloc(sizeof(float) * 9 * 2 * Fa);
    int* c2u = (int*)malloc(sizeof(int) * 2 * Fa);
    unsigned char* has_conv = (unsigned char*)calloc(2 * Fa, 1);
    int Fc = 0;
    orc_project_perspective(vw, V, R + 9 * n, T + 3 * n, k00, k11, ndc);
    for (int f = 0; f < F; ++f) {
      float fv[9];
      int nb = 0;
      for (int i = 0; i < 3; ++i) {
        memcpy(fv + 3 * i, ndc + 3 * (size_t)fc[3 * f + i], 12);
        nb += (z_clip >= 0.f && fv[3 * i + 2] < z_clip);
      }
      if (nb == 3) continue;                     /* entirely behind the plane: culled */
      if (nb == 0) { memcpy(fvc + 9 * (size_t)Fc, fv, 36); c2u[Fc++] = f; continue; }
      straddle++;
      float sub[2][9], conv[2][9];
      const int ns = clip_face(fv, z_clip, persp, sub, conv, NULL);
      for (int s2 = 0; s2 < ns; ++s2) {
        memcpy(fvc + 9 * (size_t)Fc, sub[s2], 36);
        memcpy(cnv + 9 * (size_t)Fc, conv[s2], 36);
        has_conv[Fc] = 1; c2u[Fc++] = f;
      }
    }
    const int first = 0;
    const size_t po = (size_t)n * H * W * K;
    const size_t npk = (size_t)H * W * K;
    int* p2c = (int*)malloc(sizeof(int) * npk);            /* clipped-list ids */
    float* bc = (float*)malloc(sizeof(float) * 3 * npk);   /* barycentrics w.r.t. the clipped faces */
    orc_rasterize_meshes(fvc, &first, &Fc, NULL, 1, H, W, K, flags, p2c, zbuf ? zbuf + po : NULL, bc,
                         dists ? dists + po : NULL);
    /* [upstream] convert_clipped_rasterization_to_original_faces: ids and barycentrics back to the unclipped faces
     * (zbuf and dists stay those of the clipped triangle) */
    for (size_t i = 0; i < npk; ++i) {
      const int c = p2c[i];
      pix_to_face[po + i] = c < 0 ? -1 : c2u[c];
      if (c >= 0 && has_conv[c]) { float bo[3]; conv_bary(cnv + 9 * (size_t)c, bc + 3 * i, bo); memcpy(bc + 3 * i, bo, 12); }
      if (bary) memcpy(bary + 3 * (po + i), bc + 3 * i, 12);
    }
    /* shade k = 0 (hard_rgb_blend uses colors[..., 0, :]) */
    const float* Ln = light + (size_t)light_stride * n;
    float* img = images + (size_t)n * 3 * H * W;
#pragma omp parallel for schedule(static)
    for (int yi = 0; yi < H; ++yi) {
      for (int xi = 0; xi < W; ++xi) {
        const size_t o = ((size_t)yi * W + xi) * K;
        const int f = pix_to_face[po + o];
        float out[3] = {bg[0], bg[1], bg[2]};
        if (f >= 0) {
          const float *X[3], *Nv[3], *col[3];
          for (int i = 0; i < 3; ++i) {
            const int vi = fc[3 * f + i];
            X[i] = vw + 3 * (size_t)vi;
            Nv[i] = normals + 3 * ((size_t)vert_off[b] + vi);
            col[i] = (flags & ORC_RGB_PER_ELEMENT) ? rgb + 3 * ((size_t)vert_off[b] + vi) : rgb;
          }
          phong_pixel(bc + 3 * o, X, Nv, col, Ln, C + 3 * n, out);
        }
        for (int c = 0; c < 3; ++c) img[((size_t)c * H + yi) * W + xi] = out[c];
      }
    }
    free(ndc); free(fvc); free(cnv); free(c2u); free(has_conv); free(p2c); free(bc);
  }
  if (counters) counters[0] += straddle;
}

/* Backward of orc_mesh_forward w.r.t. R, T, C (per view) and optionally world vertices
 * (grad_verts (Vtot,3): contributions through projection and through the interpolated position;
 * the vertex-normal and colour paths are reported separately in grad_normals / grad_rgb when
 * given).  Chain: d images -> Phong -> bary -> RasterizeMeshesBackwardCpu -> projection ->
 * X R + T  (SURVEY 3.4). */
void orc_mesh_backward(const float* verts, const int* faces, const int* vert_off, const int* face_off,
                       const float* normals, const float* rgb, int B, int M, const float* R,
                       const float* T, const float* C, const float* light, int light_stride,
                       float k00, float k11, float z_clip, int H, int W, int K, int flags, const int* pix_to_face,
                       const float* grad_images, float* gR, float* gT, float* gC, float* grad_verts,
                       float* grad_normals) {
  int Vtot = vert_off[B];
  double* gv_acc = grad_verts ? (double*)calloc((size_t)3 * (Vtot > 0 ? Vtot : 1), sizeof(double)) : NULL;
  double* gn_acc = grad_normals ? (double*)calloc((size_t)3 * (Vtot > 0 ? Vtot : 1), sizeof(double)) : NULL;
  for (int n = 0; n < B * M; ++n) {
    const int b = n / M;
    const int V = vert_off[b + 1] - vert_off[b];
    const float* vw = verts + 3 * (size_t)vert_off[b];
    const int* fc = faces + 3 * (size_t)face_off[b];
    const float *Rn = R + 9 * n, *Tn = T + 3 * n, *Ln = light + (size_t)light_stride * n;
    float* ndc = (float*)malloc(sizeof(float) * 3 * (size_t)(V > 0 ? V : 1));
    orc_project_perspective(vw, V, Rn, Tn, k00, k11, ndc);
    double aR[9] = {0}, aT[3] = {0}, aC[3] = {0};
    const int persp = flags & ORC_PERSPECTIVE_CORRECT;
    const float* gimg = grad_images + (size_t)n * 3 * H * W;
    for (int yi = 0; yi < H; ++yi) {
      const float yf = pix_to_ndc(H - 1 - yi, H, W);
      for (int xi = 0; xi < W; ++xi) {
        const int f = pix_to_face[((size_t)n * H * W + (size_t)yi * W + xi) * K];
        if (f < 0) continue;
        const float xf = pix_to_ndc(W - 1 - xi, W, H);
        float v[9]; const float *X[3], *Nv[3], *col[3]; int vi[3];
        for (int i = 0; i < 3; ++i) {
          vi[i] = fc[3 * f + i];
          memcpy(v + 3 * i, ndc + 3 * (size_t)vi[i], 12);
          X[i] = vw + 3 * (size_t)vi[i];
          Nv[i] = normals + 3 * ((size_t)vert_off[b] + vi[i]);
          col[i] = (flags & ORC_RGB_PER_ELEMENT) ? rgb + 3 * ((size_t)vert_off[b] + vi[i]) : rgb;
        }
        float w[3], bb[3];
        /* a face straddling z_clip was rasterized as its clipped sub-triangle(s) (orc_mesh_forward) */
        float sub[2][9], conv[2][9], bcl[3];
        int info = 0, s2 = -1;
        const int ns = z_clip >= 0.f ? clip_face(v, z_clip, persp, sub, conv, &info) : 0;
        if (ns > 0) {
          s2 = clip_pick_sub(xf, yf, sub, ns, persp, bcl);
          if (s2 < 0) continue;
          conv_bary(conv[s2], bcl, bb);
        } else {
          bary_forward(xf, yf, v, w);
          if (persp) bary_persp_forward(w, v[2], v[5], v[8], bb);
          else { bb[0] = w[0]; bb[1] = w[1]; bb[2] = w[2]; }
        }
        double g[3], gb[3], gCp[3], gX[9] = {0}, gN[9] = {0};
        for (int c = 0; c < 3; ++c) g[c] = gimg[((size_t)c * H + yi) * W + xi];
        phong_pixel_bwd(bb, X, Nv, col, Ln, C + 3 * n, g, gb, gCp, gv_acc ? gX : NULL, gn_acc ? gN : NULL, NULL);
        for (int d = 0; d < 3; ++d) aC[d] += gCp[d];
        double gfv[9] = {0};
        if (ns > 0) {
          double gbeta[3], gq[9] = {0};
          for (int k = 0; k < 3; ++k)
            gbeta[k] = (double)conv[s2][k] * gb[0] + (double)conv[s2][3 + k] * gb[1] + (double)conv[s2][6 + k] * gb[2];
          raster_bwd_one(xf, yf, sub[s2], persp, gbeta, 0.0, gq);
          clip_face_bwd(v, z_clip, persp, info, s2, gq, gb, bcl, gfv);
        } else {
          raster_bwd_one(xf, yf, v, persp, gb, 0.0, gfv);
        }
        for (int i = 0; i < 3; ++i) {
          /* projection backward: xn = xv*k00/zv, yn = yv*k11/zv, z = zv */
          float pv[3]; world_to_view(X[i], Rn, Tn, pv);
          const double zv = pv[2];
          double gp[3];
          gp[0] = gfv[3 * i] * k00 / zv;
          gp[1] = gfv[3 * i + 1] * k11 / zv;
          gp[2] = gfv[3 * i + 2] - gfv[3 * i] * ((double)pv[0] * k00) / (zv * zv) -
                  gfv[3 * i + 1] * ((double)pv[1] * k11) / (zv * zv);
          for (int r = 0; r < 3; ++r)
            for (int j = 0; j < 3; ++j) aR[3 * r + j] += (double)X[i][r] * gp[j];
          for (int j = 0; j < 3; ++j) aT[j] += gp[j];
          if (gv_acc) {
            double* o = gv_acc + 3 * ((size_t)vert_off[b] + vi[i]);
            for (int r = 0; r < 3; ++r)
              o[r] += Rn[3 * r] * gp[0] + Rn[3 * r + 1] * gp[1] + Rn[3 * r + 2] * gp[2] + gX[3 * i + r];
          }
          if (gn_acc) {
            double* o = gn_acc + 3 * ((size_t)vert_off[b] + vi[i]);
            for (int r = 0; r < 3; ++r) o[r] += gN[3 * i + r];
          }
        }
      }
    }
    for (int i = 0; i < 9; ++i) gR[9 * n + i] = (float)aR[i];
    for (int i = 0; i < 3; ++i) { gT[3 * n + i] = (float)aT[i]; gC[3 * n + i] = (float)aC[i]; }
    free(ndc);
  }
  if (gv_acc) { for (size_t i = 0; i < (size_t)3 * Vtot; ++i) grad_verts[i] = (float)gv_acc[i]; free(gv_acc); }
  if (gn_acc) { for (size_t i = 0; i < (size_t)3 * Vtot; ++i) grad_normals[i] = (float)gn_acc[i]; free(gn_acc); }
}

/* ------------------------------------------------------------------------------------------ */
/* Point rasterizer: [upstream] csrc/rasterize_points/rasterize_points_cpu.cpp                 */
/* RasterizePointsNaiveCpu / RasterizePointsBackwardCpu                                         */
/* ------------------------------------------------------------------------------------------ */
void orc_rasterize_points(const float* points, const int* first_idx, const int* num_points,
                          const float* radius, int N, int H, int W, int K, int* idx, float* zbuf,
                          float* dists2) {
#pragma omp parallel for collapse(2) schedule(dynamic, 4)
  for (int n = 0; n < N; ++n) {
    for (int yi = 0; yi < H; ++yi) {
      frag_t q[ORC_MAX_K];
      const int p0 = first_idx[n], p1 = first_idx[n] + num_points[n];
      const float yf = pix_to_ndc(H - 1 - yi, H, W);
      for (int xi = 0; xi < W; ++xi) {
        const float xf = pix_to_ndc(W - 1 - xi, W, H);
        int nq = 0;
        for (int p = p0; p < p1; ++p) {
          const float px = points[3 * (size_t)p], py = points[3 * (size_t)p + 1], pz = points[3 * (size_t)p + 2];
          const float r = radius[p];
          const float radius2 = r * r;
          if (pz < 0) continue;
          const float dx = px - xf, dy = py - yf;
          const float dist2 = dx * dx + dy * dy;
          if (dist2 < radius2) {
            frag_t fr = {pz, p, dist2, 0, 0, 0};
            frag_insert(q, &nq, K, &fr);
          }
        }
        const size_t o = (((size_t)n * H + yi) * W + xi) * K;
        for (int k = 0; k < K; ++k) {
          const int ok = k < nq;
          idx[o + k] = ok ? q[k].idx : -1;
          if (zbuf) zbuf[o + k] = ok ? q[k].z : -1.f;
          if (dists2) dists2[o + k] = ok ? q[k].d : -1.f;
        }
      }
    }
  }
}

void orc_rasterize_points_backward(const float* points, const int* idx, const float* grad_zbuf,
                                   const float* grad_dists, int N, int H, int W, int K, int Ptot,
                                   float* grad_points) {
  double* acc = (double*)calloc((size_t)3 * (Ptot > 0 ? Ptot : 1), sizeof(double));
  for (int n = 0; n < N; ++n)
    for (int yi = 0; yi < H; ++yi) {
      const float yf = pix_to_ndc(H - 1 - yi, H, W);
      for (int xi = 0; xi < W; ++xi) {
        const float xf = pix_to_ndc(W - 1 - xi, W, H);
        for (int k = 0; k < K; ++k) {
          const size_t o = (((size_t)n * H + yi) * W + xi) * K + k;
          const int p = idx[o];
          if (p < 0) break;
          const float gd = grad_dists ? grad_dists[o] : 0.f;
          const float dx = points[3 * (size_t)p] - xf, dy = points[3 * (size_t)p + 1] - yf;
          acc[3 * (size_t)p + 0] += 2.0f * gd * dx;
          acc[3 * (size_t)p + 1] += 2.0f * gd * dy;
          acc[3 * (size_t)p + 2] += grad_zbuf ? grad_zbuf[o] : 0.f;
        }
      }
    }
  for (size_t i = 0; i < (size_t)3 * Ptot; ++i) grad_points[i] = (float)acc[i];
  free(acc);
}

/* ------------------------------------------------------------------------------------------ */
/* Compositors: [upstream] csrc/compositing/norm_weighted_sum_cpu.cpp (kEps 1e-4),             */
/* alpha_composite_cpu.cpp (kEps 1e-9).  features (C,P), alphas/idx (N,K,H,W), out (N,C,H,W).   */
/* ------------------------------------------------------------------------------------------ */
void orc_composite_forward(const float* features, const float* alphas, const int* idx, int N, int K,
                           int H, int W, int Cn, int P, int alpha_mode, float* out) {
  const size_t HW = (size_t)H * W;
  memset(out, 0, sizeof(float) * (size_t)N * Cn * HW);
#pragma omp parallel for schedule(static)
  for (int n = 0; n < N; ++n)
    for (int c = 0; c < Cn; ++c)
      for (size_t px = 0; px < HW; ++px) {
        float* o = out + ((size_t)n * Cn + c) * HW + px;
        if (alpha_mode) {
          float cum = 1.f;
          for (int k = 0; k < K; ++k) {
            const int p = idx[((size_t)n * K + k) * HW + px];
            if (p < 0) continue;
            const float a = alphas[((size_t)n * K + k) * HW + px];
            *o += cum * a * features[(size_t)c * P + p];
            cum = cum * (1 - a);
          }
        } else {
          float t = 0.f;
          for (int k = 0; k < K; ++k) {
            const int p = idx[((size_t)n * K + k) * HW + px];
            if (p < 0) continue;
            t += alphas[((size_t)n * K + k) * HW + px];
          }
          t = fmaxf(t, 1e-4f);
          for (int k = 0; k < K; ++k) {
            const int p = idx[((size_t)n * K + k) * HW + px];
            if (p < 0) continue;
            const float a = alphas[((size_t)n * K + k) * HW + px];
            *o += a * features[(size_t)c * P + p] / t;
          }
        }
      }
}

void orc_composite_backward(const float* grad_out, const float* features, const float* alphas,
                            const int* idx, int N, int K, int H, int W, int Cn, int P,
                            int alpha_mode, float* grad_features, float* grad_alphas) {
  const size_t HW = (size_t)H * W;
  double* gf = (double*)calloc((size_t)Cn * (P > 0 ? P : 1), sizeof(double));
  double* ga = (double*)calloc((size_t)N * K * HW, sizeof(double));
  for (int n = 0; n < N; ++n)
    for (int c = 0; c < Cn; ++c)
      for (size_t px = 0; px < HW; ++px) {
        const float go = grad_out[((size_t)n * Cn + c) * HW + px];
#define AL(k) alphas[((size_t)n * K + (k)) * HW + px]
#define ID(k) idx[((size_t)n * K + (k)) * HW + px]
#define GA(k) ga[((size_t)n * K + (k)) * HW + px]
        if (alpha_mode) {
          float cum = 1.f;
          for (int k = 0; k < K; ++k) {
            const int p = ID(k);
            if (p < 0) continue;
            const float a = AL(k), f = features[(size_t)c * P + p];
            GA(k) += go * f * cum;
            gf[(size_t)c * P + p] += go * cum * a;
            for (int t = 0; t < k; ++t) {
              if (ID(t) < 0) continue;
              const float at = AL(t);
              GA(t) -= go * f * cum * a / (1 - at + 1e-9f);
            }
            cum = cum * (1 - a);
          }
        } else {
          float t_alpha = 0.f, t_af = 0.f;
          for (int k = 0; k < K; ++k) {
            const int p = ID(k);
            if (p < 0) continue;
            t_alpha += AL(k);
            t_af += AL(k) * features[(size_t)c * P + p];
          }
          t_alpha = fmaxf(t_alpha, 1e-4f);
          for (int k = 0; k < K; ++k) {
            const int p = ID(k);
            if (p < 0) continue;
            const float a = AL(k);
            GA(k) += go * (t_alpha * features[(size_t)c * P + p] - t_af) / (t_alpha * t_alpha);
            gf[(size_t)c * P + p] += go * a / t_alpha;
          }
        }
#undef AL
#undef ID
#undef GA
      }
  if (grad_features) for (size_t i = 0; i < (size_t)Cn * P; ++i) grad_features[i] = (float)gf[i];
  if (grad_alphas) for (size_t i = 0; i < (size_t)N * K * HW; ++i) grad_alphas[i] = (float)ga[i];
  free(gf); free(ga);
}

/* ------------------------------------------------------------------------------------------ */
/* Fused point pipeline (renderer.py:116-151).  points (B,Np,3); rgb (3) or (B*Np,3);           */
/* inv_dist (B*M); radius scalar; out images (B*M,3,H,W); idx (B*M,H,W,K) CLOUD-LOCAL ids.      */
/* weights = 1 - dists2/(r*r) with r*r evaluated in double and rounded ([upstream]             */
/* renderer/points/renderer.py: python-float r*r), raster test uses float r*r.                  */
/* ------------------------------------------------------------------------------------------ */
void orc_points_forward(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                        const float* T, const float* inv_dist, double radius, const float* bg,
                        int H, int W, int K, int flags, float* images, int* idx, float* zbuf,
                        float* dists2) {
  const size_t HW = (size_t)H * W;
  const float r2w = (float)(radius * radius);
  for (int n = 0; n < B * M; ++n) {
    const int b = n / M;
    float* ndc = (float*)malloc(sizeof(float) * 3 * (size_t)(Np > 0 ? Np : 1));
    float* rad = (float*)malloc(sizeof(float) * (size_t)(Np > 0 ? Np : 1));
    float* feat = (float*)malloc(sizeof(float) * 3 * (size_t)(Np > 0 ? Np : 1));
    int* lidx = idx + (size_t)n * HW * K;
    float* lz = (float*)malloc(sizeof(float) * HW * K);
    float* ld = (float*)malloc(sizeof(float) * HW * K);
    float* al = (float*)malloc(sizeof(float) * HW * K);
    int* kidx = (int*)malloc(sizeof(int) * HW * K);
    orc_project_orthographic(points + 3 * (size_t)b * Np, Np, R + 9 * n, T + 3 * n, inv_dist[n], ndc);
    for (int p = 0; p < Np; ++p) {
      rad[p] = (float)radius;
      for (int c = 0; c < 3; ++c)
        feat[(size_t)c * Np + p] = (flags & ORC_RGB_PER_ELEMENT) ? rgb[3 * ((size_t)b * Np + p) + c] : rgb[c];
    }
    const int first = 0;
    orc_rasterize_points(ndc, &first, &Np, rad, 1, H, W, K, lidx, lz, ld);
    /* permute (H,W,K)->(K,H,W); weights = 1 - dists2 / (r*r) */
    for (size_t px = 0; px < HW; ++px)
      for (int k = 0; k < K; ++k) {
        kidx[(size_t)k * HW + px] = lidx[px * K + k];
        al[(size_t)k * HW + px] = 1 - ld[px * K + k] / r2w;
      }
    float* img = images + (size_t)n * 3 * HW;
    orc_composite_forward(feat, al, kidx, 1, K, H, W, 3, Np, flags & ORC_COMPOSITE_ALPHA, img);
    /* _add_background_color_to_images: pixels with idx[:,0] < 0 */
    for (size_t px = 0; px < HW; ++px)
      if (kidx[px] < 0) for (int c = 0; c < 3; ++c) img[(size_t)c * HW + px] = bg[c];
    if (zbuf) memcpy(zbuf + (size_t)n * HW * K, lz, sizeof(float) * HW * K);
    if (dists2) memcpy(dists2 + (size_t)n * HW * K, ld, sizeof(float) * HW * K);
    free(ndc); free(rad); free(feat); free(lz); free(ld); free(al); free(kidx);
  }
}

/* Backward: grad_images -> gR, gT (B*M), g_inv_dist (B*M), optional grad_points (B,Np,3) (summed
 * over the M views), optional grad_rgb (B*Np,3 or 3). */
void orc_points_backward(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                         const float* T, const float* inv_dist, double radius, int H, int W, int K,
                         int flags, const int* idx, const float* grad_images, float* gR, float* gT,
                         float* g_inv_dist, float* grad_points, float* grad_rgb) {
  const size_t HW = (size_t)H * W;
  const float r2w = (float)(radius * radius);
  double* gp_acc = grad_points ? (double*)calloc((size_t)3 * B * (Np > 0 ? Np : 1), sizeof(double)) : NULL;
  const int per = flags & ORC_RGB_PER_ELEMENT;
  double* grgb = grad_rgb ? (double*)calloc(per ? (size_t)3 * B * Np : 3, sizeof(double)) : NULL;
  for (int n = 0; n < B * M; ++n) {
    const int b = n / M;
    const float* pw = points + 3 * (size_t)b * Np;
    const float *Rn = R + 9 * n, *Tn = T + 3 * n;
    const float s = inv_dist[n];
    float* ndc = (float*)malloc(sizeof(float) * 3 * (size_t)(Np > 0 ? Np : 1));
    float* feat = (float*)malloc(sizeof(float) * 3 * (size_t)(Np > 0 ? Np : 1));
    float* al = (float*)malloc(sizeof(float) * HW * K);
    float* gal = (float*)malloc(sizeof(float) * HW * K);
    float* gfeat = (float*)malloc(sizeof(float) * 3 * (size_t)(Np > 0 ? Np : 1));
    int* kidx = (int*)malloc(sizeof(int) * HW * K);
    float* gd = (float*)malloc(sizeof(float) * HW * K);
    float* gndc = (float*)malloc(sizeof(float) * 3 * (size_t)(Np > 0 ? Np : 1));
    float* gimg = (float*)malloc(sizeof(float) * 3 * HW);
    orc_project_orthographic(pw, Np, Rn, Tn, s, ndc);
    for (int p = 0; p < Np; ++p)
      for (int c = 0; c < 3; ++c)
        feat[(size_t)c * Np + p] = per ? rgb[3 * ((size_t)b * Np + p) + c] : rgb[c];
    const int* lidx = idx + (size_t)n * HW * K;
    for (int yi = 0; yi < H; ++yi) {
      const float yf = pix_to_ndc(H - 1 - yi, H, W);
      for (int xi = 0; xi < W; ++xi) {
        const float xf = pix_to_ndc(W - 1 - xi, W, H);
        const size_t px = (size_t)yi * W + xi;
        for (int k = 0; k < K; ++k) {
          const int p = lidx[px * K + k];
          kidx[(size_t)k * HW + px] = p;
          float d2 = -1.f;
          if (p >= 0) { const float dx = ndc[3 * p] - xf, dy = ndc[3 * p + 1] - yf; d2 = dx * dx + dy * dy; }
          al[(size_t)k * HW + px] = 1 - d2 / r2w;
        }
        /* masked_scatter background: no gradient reaches the compositor there */
        for (int c = 0; c < 3; ++c)
          gimg[(size_t)c * HW + px] = lidx[px * K] < 0 ? 0.f : grad_images[((size_t)n * 3 + c) * HW + px];
      }
    }
    orc_composite_backward(gimg, feat, al, kidx, 1, K, H, W, 3, Np, flags & ORC_COMPOSITE_ALPHA, gfeat, gal);
    for (size_t px = 0; px < HW; ++px)
      for (int k = 0; k < K; ++k) gd[px * K + k] = gal[(size_t)k * HW + px] * (-1.f / r2w);
    orc_rasterize_points_backward(ndc, lidx, NULL, gd, 1, H, W, K, Np, gndc);
    double aR[9] = {0}, aT[3] = {0}, as = 0;
    for (int p = 0; p < Np; ++p) {
      const double g[3] = {gndc[3 * p], gndc[3 * p + 1], gndc[3 * p + 2]};
      const double Xs[3] = {(double)pw[3 * p] * s, (double)pw[3 * p + 1] * s, (double)pw[3 * p + 2] * s};
      for (int r = 0; r < 3; ++r) {
        double gx = Rn[3 * r] * g[0] + Rn[3 * r + 1] * g[1] + Rn[3 * r + 2] * g[2]; /* d/d(Xs_r) */
        for (int j = 0; j < 3; ++j) aR[3 * r + j] += Xs[r] * g[j];
        as += gx * pw[3 * p + r];
        if (gp_acc) gp_acc[3 * ((size_t)b * Np + p) + r] += gx * s;
      }
      for (int j = 0; j < 3; ++j) aT[j] += g[j];
      if (grgb) for (int c = 0; c < 3; ++c) {
        if (per) grgb[3 * ((size_t)b * Np + p) + c] += gfeat[(size_t)c * Np + p];
        else grgb[c] += gfeat[(size_t)c * Np + p];
      }
    }
    for (int i = 0; i < 9; ++i) gR[9 * n + i] = (float)aR[i];
    for (int i = 0; i < 3; ++i) gT[3 * n + i] = (float)aT[i];
    g_inv_dist[n] = (float)as;
    free(ndc); free(feat); free(al); free(gal); free(gfeat); free(kidx); free(gd); free(gndc); free(gimg);
  }
  if (gp_acc) { for (size_t i = 0; i < (size_t)3 * B * Np; ++i) grad_points[i] = (float)gp_acc[i]; free(gp_acc); }
  if (grgb) { size_t nn = per ? (size_t)3 * B * Np : 3; for (size_t i = 0; i < nn; ++i) grad_rgb[i] = (float)grgb[i]; free(grgb); }
}
