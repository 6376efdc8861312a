// mvr_mesh_bwd.cu -- backward of the mesh path (see mvr_mesh.cu for the forward).  Compiled WITH FMA contraction
// (build.py: no -fmad=false for this file): everything here is compared with the oracle at a tolerance, and the exact
// part it depends on -- the projected vertices -- comes from mesh_project_kernel, whose arithmetic is written with
// non-contractable intrinsics.  Contraction removes ~120 of the ~480 floating-point instructions per covered pixel.
//
//   mesh_backward_kernel -- per pixel recompute (no fragment traffic), chain
//             d image -> Phong -> barycentrics -> NDC verts -> view verts -> (dR, dT, dC), warp-reduced to one partial
//             per warp; mesh_backward_finish_kernel (mvr_mesh_clip.cu) sums them in fixed order (deterministic, no
//             float atomics on the camera gradients).
#include <cstdint>

#include "mvr_mesh.cuh"

namespace mvr {

// One covered pixel: forward recompute from the projected vertices, then the chain
// d image -> Phong -> barycentrics -> NDC vertices -> view-space vertices -> acc = (dR 9, dT 3, dC 3).
// GV (vertex gradients wanted): the contributions to d/d verts and d/d normals of the pixel's three vertices are returned
// in gvn[18] (vertex i: gvn[6 i .. 6 i + 2] = d/d position, gvn[6 i + 3 .. 6 i + 5] = d/d unit normal) and vids, and the
// caller scatters them with warp-aggregated atomics (scatter_vertex_grads); returns false when nothing was produced.
// GC (colour gradient wanted): with VRGB, gcol[3 i .. 3 i + 2] = d/d colour of vertex i (= bb_i d/d texel; vids set as for GV,
// scattered by scatter_vertex9<true>); with one object colour, gcol[0..2] += sum(bb) d/d texel (the thread's running sum).
template <bool VRGB, bool GV, bool GC = false>
__device__ __forceinline__ bool mesh_backward_pixel(const MeshBwdParams& p, int n, int f0, int voff, const float4* __restrict__ pvn,
                                                    bool persp, const ShadeCtx& sc, const float4 ucol, int fid, float g0, float g1,
                                                    float g2, float xf, int yi, float acc[16], float* gvn = nullptr, int* vids = nullptr,
                                                    float* gcol = nullptr) {
  const int4 fi = __ldg(p.faces4 + f0 + fid);
  // ---- forward recompute from the projected vertices (exact IEEE projection, done once per view by
  // mesh_project_kernel: for small faces the barycentrics amplify a 1-ulp change of a vertex by |xy| / area);
  // everything downstream is well conditioned and uses fast reciprocals ----
  const Face fc = gather_face(pvn, fi);
  // (two 16-byte gathers per vertex here: the 32-byte record of the shade kernel needs 8 aligned registers per load,
  // which this register-bound kernel pays for in spills -- measured 369 vs 362 us)
  const float4 X0 = __ldg(p.verts4 + voff + fi.x), X1 = __ldg(p.verts4 + voff + fi.y), X2 = __ldg(p.verts4 + voff + fi.z);
  const float4 N0 = __ldg(p.normals4 + voff + fi.x), N1 = __ldg(p.normals4 + voff + fi.y), N2 = __ldg(p.normals4 + voff + fi.z);
  float4 c0 = ucol, c1 = ucol, c2 = ucol;
  if (VRGB) { c0 = __ldg(p.rgb4 + voff + fi.x); c1 = __ldg(p.rgb4 + voff + fi.y); c2 = __ldg(p.rgb4 + voff + fi.z); }
  // (after every load of the pixel has been issued) a face crossing the near plane: mesh_backward_clipped_kernel owns the pixel
  // (the flag -- some vertex lies behind the plane, never in MVTN's default setups -- is re-read per pixel: an L1 hit
  // is cheaper than a register kept live across this loop)
  if (may_clip(p.wsflags) && face_straddles(fc, p.z_clip)) return false;
  const FaceEdges fe = face_edges(fc);
  const float yf = __ldg(p.tab + p.W + yi);
  const float e0 = (xf - fc.x1) * fe.A0 - (yf - fc.y1) * fe.B0;
  const float e1 = (xf - fc.x2) * fe.A1 - (yf - fc.y2) * fe.B1;
  const float e2 = (xf - fc.x0) * fe.A2 - (yf - fc.y0) * fe.B2;
  const float inv_area = rcp_fast(fe.area_p);
  const float w0 = e0 * inv_area, w1 = e1 * inv_area, w2 = e2 * inv_area;
  float bb[3] = {w0, w1, w2};
  float t0 = 0.f, t1 = 0.f, t2 = 0.f, id = 1.f;
  bool clamped = false;
  if (persp) {
    t0 = w0 * fc.z1 * fc.z2; t1 = w1 * fc.z0 * fc.z2; t2 = w2 * fc.z0 * fc.z1;
    const float st = t0 + t1 + t2;
    clamped = st < MVR_K_EPS;
    id = rcp_fast(fmaxf(st, MVR_K_EPS));
    bb[0] = t0 * id; bb[1] = t1 * id; bb[2] = t2 * id;
  }
  // ---- Phong backward ----
  const float3 P = interp(bb, X0, X1, X2);
  const float3 Nn = interp(bb, N0, N1, N2);
  float3 tex;
  float sb = 0.f;
  if (VRGB) tex = interp(bb, c0, c1, c2);
  else { sb = bb[0] + bb[1] + bb[2]; tex = make_float3(ucol.x * sb, ucol.y * sb, ucol.z * sb); }
  const float in = inv_norm_clamped(Nn.x, Nn.y, Nn.z, 1e-6f);
  const float nx = Nn.x * in, ny = Nn.y * in, nz = Nn.z * in;
  const float cosang = fmaf(nx, sc.lx, fmaf(ny, sc.ly, nz * sc.lz));
  const float diff = fmaxf(cosang, 0.f);
  const float vx = sc.cx - P.x, vy = sc.cy - P.y, vz = sc.cz - P.z;
  const float iv = inv_norm_clamped(vx, vy, vz, 1e-6f);
  const float vhx = vx * iv, vhy = vy * iv, vhz = vz * iv;
  const float rx = fmaf(2.f * cosang, nx, -sc.lx), ry = fmaf(2.f * cosang, ny, -sc.ly), rz = fmaf(2.f * cosang, nz, -sc.lz);
  const float dt = fmaf(vhx, rx, fmaf(vhy, ry, vhz * rz));
  const bool lit = cosang > 0.f;
  const float alpha = (dt > 0.f && lit) ? dt : 0.f;
  const float kd = fmaf(MVR_DIFFUSE, diff, MVR_AMBIENT);
  const float gtx = g0 * kd, gty = g1 * kd, gtz = g2 * kd;
  if (GC) {      // the texel is linear in the colours: d colour = bb_i d texel (per vertex) / sum(bb) d texel (one colour)
    if (VRGB) {
#pragma unroll
      for (int i = 0; i < 3; ++i) { gcol[3 * i] = bb[i] * gtx; gcol[3 * i + 1] = bb[i] * gty; gcol[3 * i + 2] = bb[i] * gtz; }
      vids[0] = fi.x; vids[1] = fi.y; vids[2] = fi.z;
    } else {
      gcol[0] = fmaf(sb, gtx, gcol[0]); gcol[1] = fmaf(sb, gty, gcol[1]); gcol[2] = fmaf(sb, gtz, gcol[2]);
    }
  }
  const float gdiff = MVR_DIFFUSE * fmaf(g0, tex.x, fmaf(g1, tex.y, g2 * tex.z));
  const float gs = MVR_SPECULAR * (g0 + g1 + g2);
  const float a2 = alpha * alpha, a4 = a2 * a2, a8 = a4 * a4, a16 = a8 * a8, a32 = a16 * a16;
  const float a63 = a32 * a16 * a8 * a4 * a2 * alpha;
  const float gdt = (dt > 0.f && lit) ? gs * 64.f * a63 : 0.f;
  const float gvhx = gdt * rx, gvhy = gdt * ry, gvhz = gdt * rz;
  const float grx = gdt * vhx, gry = gdt * vhy, grz = gdt * vhz;
  const float gcos = (lit ? gdiff : 0.f) + 2.f * fmaf(grx, nx, fmaf(gry, ny, grz * nz));
  const float gnx = fmaf(2.f * cosang, grx, gcos * sc.lx), gny = fmaf(2.f * cosang, gry, gcos * sc.ly), gnz = fmaf(2.f * cosang, grz, gcos * sc.lz);
  float gNx, gNy, gNz, gvx, gvy, gvz;
  normalize_bwd3(Nn.x, Nn.y, Nn.z, 1e-6f, gnx, gny, gnz, gNx, gNy, gNz);
  normalize_bwd3(vx, vy, vz, 1e-6f, gvhx, gvhy, gvhz, gvx, gvy, gvz);
  acc[12] += gvx; acc[13] += gvy; acc[14] += gvz;   // dC
  // d bary_i = gtex.col_i + gN.n_i + gP.X_i  with gP = -gv
  float gb0, gb1, gb2;
  // ---- [upstream] BarycentricPerspectiveCorrectionBackward ----
  float dz0 = 0.f, dz1 = 0.f, dz2 = 0.f;
  if (persp && !clamped) {
    // b = t / sum(t) is invariant to a common shift of d/db (its Jacobian annihilates constants): the gradient only depends on
    // gb_i - k, k = sum_j b_j gb_j, i.e. on sum_j b_j (gb_i - gb_j) (sum b = 1) -- and the differences gb_i - gb_j are formed from
    // ATTRIBUTE differences, gN.(N_i - N_j) - gv.(X_i - X_j) (+ gtex.(c_i - c_j)), never from the gb themselves.  The three gb are
    // nearly equal (one object colour: the common part is gtex.colour ~ 0.5, the differences ~ 1e-5), the Jacobian behind them is
    // ~ 1/area, and a sliver's vertex gradients are a small residual of its terms: forming gb_i first rounds them at 6e-8, which a
    // sliver of NDC area 3e-6 amplifies to a 3..26 % error of the pixel's camera gradient, jumping with single ulps anywhere
    // upstream (scripts/fuzz_parity.py, soup case 5421; PyTorch3D's own fp32 chain rounds d/db the same way).  From attribute
    // differences the error stays relative to the differences.  (Without perspective correction sum w = area / (area + eps) is
    // only nearly constant and the plain chain below is kept, with upstream's conditioning.)
    const float n01x = N0.x - N1.x, n01y = N0.y - N1.y, n01z = N0.z - N1.z, n02x = N0.x - N2.x, n02y = N0.y - N2.y, n02z = N0.z - N2.z;
    const float x01x = X0.x - X1.x, x01y = X0.y - X1.y, x01z = X0.z - X1.z, x02x = X0.x - X2.x, x02y = X0.y - X2.y, x02z = X0.z - X2.z;
    float d01 = fmaf(gNx, n01x, fmaf(gNy, n01y, gNz * n01z)) - fmaf(gvx, x01x, fmaf(gvy, x01y, gvz * x01z));
    float d02 = fmaf(gNx, n02x, fmaf(gNy, n02y, gNz * n02z)) - fmaf(gvx, x02x, fmaf(gvy, x02y, gvz * x02z));
    if (VRGB) {
      d01 += fmaf(gtx, c0.x - c1.x, fmaf(gty, c0.y - c1.y, gtz * (c0.z - c1.z)));
      d02 += fmaf(gtx, c0.x - c2.x, fmaf(gty, c0.y - c2.y, gtz * (c0.z - c2.z)));
    }
    const float d12 = d02 - d01;
    gb0 = fmaf(bb[1], d01, bb[2] * d02);
    gb1 = fmaf(bb[2], d12, -bb[0] * d01);
    gb2 = -fmaf(bb[0], d02, bb[1] * d12);
  } else {
    const float gc0 = fmaf(gtx, c0.x, fmaf(gty, c0.y, gtz * c0.z));
    const float gc1 = VRGB ? fmaf(gtx, c1.x, fmaf(gty, c1.y, gtz * c1.z)) : gc0;
    const float gc2 = VRGB ? fmaf(gtx, c2.x, fmaf(gty, c2.y, gtz * c2.z)) : gc0;
    gb0 = gc0 + fmaf(gNx, N0.x, fmaf(gNy, N0.y, gNz * N0.z)) - fmaf(gvx, X0.x, fmaf(gvy, X0.y, gvz * X0.z));
    gb1 = gc1 + fmaf(gNx, N1.x, fmaf(gNy, N1.y, gNz * N1.z)) - fmaf(gvx, X1.x, fmaf(gvy, X1.y, gvz * X1.z));
    gb2 = gc2 + fmaf(gNx, N2.x, fmaf(gNy, N2.y, gNz * N2.z)) - fmaf(gvx, X2.x, fmaf(gvy, X2.y, gvz * X2.z));
  }
  if (persp) {
    const float gden = clamped ? -(gb0 * t0 + gb1 * t1 + gb2 * t2) * id * id : 0.f;
    const float gt0 = fmaf(gb0, id, gden), gt1 = fmaf(gb1, id, gden), gt2 = fmaf(gb2, id, gden);
    gb0 = gt0 * fc.z1 * fc.z2; gb1 = gt1 * fc.z0 * fc.z2; gb2 = gt2 * fc.z0 * fc.z1;
    dz0 = gt1 * w1 * fc.z2 + gt2 * w2 * fc.z1;
    dz1 = gt0 * w0 * fc.z2 + gt2 * w2 * fc.z0;
    dz2 = gt0 * w0 * fc.z1 + gt1 * w1 * fc.z0;
  }
  // ---- [upstream] BarycentricCoordsBackward / EdgeFunctionBackward ----
  const float ge0 = gb0 * inv_area, ge1 = gb1 * inv_area, ge2 = gb2 * inv_area;
  // (perspective-corrected barycentrics do not depend on a common factor of the w_i: d/d area vanishes identically there --
  // computed, it is rounding noise times 1/area^2)
  const float garea = (persp && !clamped) ? 0.f : -(gb0 * e0 + gb1 * e1 + gb2 * e2) * inv_area * inv_area;
  float gx0, gy0, gx1, gy1, gx2, gy2;
  // E(p,a,b): dE/da = (py-by, bx-px), dE/db = (ay-py, px-ax)
  gx1 = ge0 * (yf - fc.y2); gy1 = ge0 * (fc.x2 - xf); gx2 = ge0 * (fc.y1 - yf); gy2 = ge0 * (xf - fc.x1);          // e0 = E(p,v1,v2)
  gx2 += ge1 * (yf - fc.y0); gy2 += ge1 * (fc.x0 - xf); gx0 = ge1 * (fc.y2 - yf); gy0 = ge1 * (xf - fc.x2);        // e1 = E(p,v2,v0)
  gx0 += ge2 * (yf - fc.y1); gy0 += ge2 * (fc.x1 - xf); gx1 += ge2 * (fc.y0 - yf); gy1 += ge2 * (xf - fc.x0);      // e2 = E(p,v0,v1)
  // area = E(v2, v0, v1)
  gx0 += garea * (fc.y2 - fc.y1); gy0 += garea * (fc.x1 - fc.x2);
  gx1 += garea * (fc.y0 - fc.y2); gy1 += garea * (fc.x2 - fc.x0);
  gx2 += garea * (fc.y1 - fc.y0); gy2 += garea * (fc.x0 - fc.x1);
  // ---- projection backward + X R + T backward: x_ndc = (px k00) / pz, so px k00 = x_ndc pz ----
  const float gxn[3] = {gx0, gx1, gx2}, gyn[3] = {gy0, gy1, gy2}, gzn[3] = {dz0, dz1, dz2};
  const float xn[3] = {fc.x0, fc.x1, fc.x2}, yn[3] = {fc.y0, fc.y1, fc.y2}, zv[3] = {fc.z0, fc.z1, fc.z2};
  const float4 Xs[3] = {X0, X1, X2};
  const int vid[3] = {fi.x, fi.y, fi.z};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float iz = rcp_fast(zv[i]);
    const float gpx = gxn[i] * p.k00 * iz;
    const float gpy = gyn[i] * p.k11 * iz;
    const float gpz = gzn[i] - (gxn[i] * xn[i] + gyn[i] * yn[i]) * iz;
    acc[0] = fmaf(Xs[i].x, gpx, acc[0]); acc[1] = fmaf(Xs[i].x, gpy, acc[1]); acc[2] = fmaf(Xs[i].x, gpz, acc[2]);
    acc[3] = fmaf(Xs[i].y, gpx, acc[3]); acc[4] = fmaf(Xs[i].y, gpy, acc[4]); acc[5] = fmaf(Xs[i].y, gpz, acc[5]);
    acc[6] = fmaf(Xs[i].z, gpx, acc[6]); acc[7] = fmaf(Xs[i].z, gpy, acc[7]); acc[8] = fmaf(Xs[i].z, gpz, acc[8]);
    acc[9] += gpx; acc[10] += gpy; acc[11] += gpz;
    if (GV) {
      const float* r = p.R + 9 * (size_t)n;
      gvn[6 * i + 0] = fmaf(__ldg(r + 0), gpx, fmaf(__ldg(r + 1), gpy, __ldg(r + 2) * gpz)) - bb[i] * gvx;
      gvn[6 * i + 1] = fmaf(__ldg(r + 3), gpx, fmaf(__ldg(r + 4), gpy, __ldg(r + 5) * gpz)) - bb[i] * gvy;
      gvn[6 * i + 2] = fmaf(__ldg(r + 6), gpx, fmaf(__ldg(r + 7), gpy, __ldg(r + 8) * gpz)) - bb[i] * gvz;
      gvn[6 * i + 3] = bb[i] * gNx; gvn[6 * i + 4] = bb[i] * gNy; gvn[6 * i + 5] = bb[i] * gNz;
      vids[i] = vid[i];
    }
  }
  return true;
}

// Warp-aggregated gradient scatter (north_star (4)): neighbouring pixels share faces -- an 8x4-pixel block of the strip
// kernel touches ~5 of them at C2, a large triangle fills whole warps -- so the lanes of a warp that hold the SAME face sum
// their 18 per-vertex values first (__match_any_sync on the face id, then one pass over the group's members by shuffles)
// and ONE lane per face issues the 18 atomicAdds: 6x fewer L2 atomics at C2, 32x fewer on large faces.  Must be called by
// all 32 lanes (fid < 0: nothing to add).
__device__ __forceinline__ void scatter_vertex_grads(const MeshBwdParams& p, int voff, int fid, const float gvn[18], const int vids[3]) {
  const unsigned int full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned int grp = __match_any_sync(full, fid);
  unsigned int peers = fid >= 0 ? grp : 0u;
  const bool leader = fid >= 0 && (int)(__ffs(grp) - 1) == lane;
  float sum[18];
#pragma unroll
  for (int i = 0; i < 18; ++i) sum[i] = 0.f;
  while (__any_sync(full, peers != 0u)) {      // warp-uniform: max group size iterations
    const int src = peers ? __ffs(peers) - 1 : lane;
#pragma unroll
    for (int i = 0; i < 18; ++i) {
      const float t = __shfl_sync(full, gvn[i], src);
      if (peers) sum[i] += t;
    }
    peers &= peers - 1u;
  }
  if (leader) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (p.grad_verts) {
        float* o = p.grad_verts + 3 * (size_t)(voff + vids[i]);
        atomicAdd(o + 0, sum[6 * i + 0]); atomicAdd(o + 1, sum[6 * i + 1]); atomicAdd(o + 2, sum[6 * i + 2]);
      }
      if (p.grad_normals) {
        float* o = p.grad_normals + 3 * (size_t)(voff + vids[i]);
        atomicAdd(o + 0, sum[6 * i + 3]); atomicAdd(o + 1, sum[6 * i + 4]); atomicAdd(o + 2, sum[6 * i + 5]);
      }
    }
  }
}

// scatter_vertex_grads for 9 per-vertex values of a pixel: the colour gradients (RGB: gcol of mesh_backward_pixel<true, GV, true>, into
// p.grad_rgb) or the hard depth's position gradients (into p.grad_verts): lanes that hold the same face sum first, one lane per face
// issues the atomics.  Must be called by all 32 lanes (fid < 0: nothing to add).
template <bool RGB>
__device__ __forceinline__ void scatter_vertex9(const MeshBwdParams& p, int voff, int fid, const float gcol[9], const int vids[3]) {
  const unsigned int full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned int grp = __match_any_sync(full, fid);
  unsigned int peers = fid >= 0 ? grp : 0u;
  const bool leader = fid >= 0 && (int)(__ffs(grp) - 1) == lane;
  float sum[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) sum[i] = 0.f;
  while (__any_sync(full, peers != 0u)) {
    const int src = peers ? __ffs(peers) - 1 : lane;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const float t = __shfl_sync(full, gcol[i], src);
      if (peers) sum[i] += t;
    }
    peers &= peers - 1u;
  }
  if (leader) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float* o = (RGB ? p.grad_rgb : p.grad_verts) + 3 * (size_t)(voff + vids[i]);
      atomicAdd(o + 0, sum[3 * i + 0]); atomicAdd(o + 1, sum[3 * i + 1]); atomicAdd(o + 2, sum[3 * i + 2]);
    }
  }
}

// GC && !VRGB: the warp's colour partial (d r, d g, d b, 0) next to its camera partial (fixed-order sum in the finish kernel).
// Must be called by all 32 lanes.
__device__ __forceinline__ void store_rgb_partial(const MeshBwdParams& p, size_t part, const float gcol[3]) {
  const float r = warp_sum(gcol[0]), g = warp_sum(gcol[1]), b = warp_sum(gcol[2]);
  if ((threadIdx.x & 31) == 0) *reinterpret_cast<float4*>(p.rgb_partials + 4 * part) = make_float4(r, g, b, 0.f);
}

// VRGB: per-vertex colours (object_color == "custom"); otherwise ONE object colour: the texel is c * sum(b) and its
// cotangent one dot product -- six registers and ~13 floating-point instructions less per covered pixel.
// GC: colour gradients too (mesh_backward_pixel's gcol): per vertex through scatter_vertex9<true>, one object colour through the
// per-warp partials rgb_partials.
template <int MINB, bool VRGB, bool GV, bool GC = false>
__global__ void __launch_bounds__(MVR_THREADS, MINB) mesh_backward_kernel(const MeshBwdParams p) {
  pdl_enter();
  const int tid = threadIdx.x;
  // grid: x = 32x32-pixel tiles, y = view m, z = object b; thread (lane, warp) owns pixels (x0+lane, y0+warp+8j)
  const int b = blockIdx.z, m = blockIdx.y, n = b * p.M + m, cta = blockIdx.x;
  int tyb, txb;
  tile_rc(cta, p.tiles_x, tyb, txb);
  const int xi = txb * 32 + (tid & 31), yi0 = tyb * 32 + (tid >> 5);
  const int HW = p.H * p.W;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  // issue every load of this thread's pixels first (memory-level parallelism), then do the math
  int fids[BWD_PIX_PER_THREAD];
  float gin[BWD_PIX_PER_THREAD][3];
#pragma unroll
  for (int j = 0; j < BWD_PIX_PER_THREAD; ++j) {
    const int yi = yi0 + 8 * j;
    fids[j] = (xi < p.W && yi < p.H) ? __ldg(p.pix_to_face + ((size_t)n * HW + (size_t)yi * p.W + xi) * p.K) : -1;
  }
#pragma unroll
  for (int j = 0; j < BWD_PIX_PER_THREAD; ++j) {
    const int pix = (yi0 + 8 * j) * p.W + xi;
    if (fids[j] >= 0) {
      load_grad_rgb(p.grad_images, p.flags & MVR_IMAGES_BF16, (size_t)n * 3 * HW + pix, (size_t)HW, p.onorm, gin[j][0], gin[j][1], gin[j][2]);
    } else {
      gin[j][0] = gin[j][1] = gin[j][2] = 0.f;
    }
  }
  float acc[16];                                      // BWD_VALS used, [15] stays 0
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  bool any = false;
  const ShadeCtx sc = load_shade_ctx(p.light, p.light_stride, p.Cc, n);
  const float xf = xi < p.W ? __ldg(p.tab + xi) : 0.f;
  float4 ucol = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!VRGB) ucol = make_float4(__ldg(p.obj_rgb), __ldg(p.obj_rgb + 1), __ldg(p.obj_rgb + 2), 0.f);
  constexpr bool SCAT = GV || (GC && VRGB);      // a warp-aggregated scatter follows every pixel
  float gcol[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};      // GC: per-vertex (VRGB) or the running sum (one colour)
#pragma unroll 1
  for (int j = 0; j < BWD_PIX_PER_THREAD; ++j) {
    const int fid = fids[j];
    const float g0 = gin[j][0], g1 = gin[j][1], g2 = gin[j][2];
    const bool live = !(fid < 0 || (g0 == 0.f && g1 == 0.f && g2 == 0.f));
    const int yi = yi0 + 8 * j;
    if (SCAT) {      // all lanes stay together for the warp-aggregated scatter
      float gvn[18];
      int vids[3] = {0, 0, 0};
      bool done = false;
      if (live) { any = true; done = mesh_backward_pixel<VRGB, GV, GC>(p, n, f0, voff, pvn, persp, sc, ucol, fid, g0, g1, g2, xf, yi, acc, gvn, vids, gcol); }
      if (GV) scatter_vertex_grads(p, voff, done ? fid : -1, gvn, vids);
      if (GC && VRGB) scatter_vertex9<true>(p, voff, done ? fid : -1, gcol, vids);
      continue;
    }
    if (!live) continue;
    any = true;
    mesh_backward_pixel<VRGB, false, GC>(p, n, f0, voff, pvn, persp, sc, ucol, fid, g0, g1, g2, xf, yi, acc, nullptr, nullptr, gcol);
  }
  // one partial per WARP, no block barrier: a warp retires as soon as its own pixels are done
  const size_t part = (size_t)n * p.parts_per_view + (size_t)cta * NWARPS + (tid >> 5);
  if (GC && !VRGB) store_rgb_partial(p, part, gcol);
  float* out = p.partials + part * 16;
  const int lane = tid & 31;
  if (!__any_sync(0xffffffffu, any)) {   // background-only warp
    if (lane < 16) out[lane] = 0.f;
    return;
  }
  const float mine = warp_sum16_transposed(acc);      // lanes 2i, 2i+1: total of value i
  if (!(lane & 1)) out[lane >> 1] = mine;
}

// ---- strip variant: one CTA walks a ROW of 32x32-pixel tiles with a two-stage cp.async pipeline ----
// The face ids and the cotangent of tile t + 1 (16 KB) travel to shared memory while tile t is being processed, so the
// two dependent DRAM trips every thread of mesh_backward_kernel starts with (pix_to_face, then the cotangent of its
// covered pixels) leave the critical path, the per-thread staging arrays (local memory) disappear, and a warp reduces
// and writes ONE partial per strip instead of one per tile.  Requirements (else mesh_backward_kernel runs):
// K == 1, fp32 cotangent, W % 4 == 0 (16-byte chunks never straddle the image edge).
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned int a = (unsigned int)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(a), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int MINB, bool VRGB, bool GV, bool GC = false>
__global__ void __launch_bounds__(MVR_THREADS, MINB) mesh_backward_kernel_strip(const MeshBwdParams p) {
  pdl_enter();
  // Every WARP stages its own pixels: the four 8x4-pixel blocks it owns in a 32x32 tile (128 pixels x 4 planes = 2 KB per
  // stage, two stages), one 16-byte cp.async per lane and plane -- so the pipeline needs __syncwarp only.  The kernel has
  // no CTA barrier at all: a warp whose blocks are background runs ahead through the strip instead of waiting for the
  // warp that holds the silhouette (22 % of the stall samples of the CTA-staged version were barrier waits).
  // Layout of a warp's stage: pixel (block j, row r, column c) of plane q at [q][(4 j + r) * 8 + c]: the lanes of a block
  // read consecutive words.
  __shared__ __align__(16) int s_fid[NWARPS][2][128];
  __shared__ __align__(16) float s_g[NWARPS][2][3][128];
  __shared__ unsigned char s_list[NWARPS][128];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // grid: x = tile row, y = view m, z = object b
  const int b = blockIdx.z, m = blockIdx.y, n = b * p.M + m, tyb = blockIdx.x;
  const int HW = p.H * p.W;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  const int* fid_base = p.pix_to_face + (size_t)n * HW;
  const float* g_base = reinterpret_cast<const float*>(p.grad_images) + (size_t)n * 3 * HW;
  // block q = warp + 8 j of the tile (4 across, 8 down): column (warp & 3), rows (warp >> 2) + 2 j
  const int bx0 = (warp & 3) << 3, by0 = (warp >> 2) << 2;
  // this lane's 16-byte chunk of every plane: block cj, row cr of the block, half ch (pixels 4 ch .. 4 ch + 3)
  const int cj = lane >> 3, cr = (lane >> 1) & 3, ch = lane & 1;
  const int cy = tyb * 32 + by0 + 8 * cj + cr;                 // image row of the chunk
  const int so = (cj * 4 + cr) * 8 + ch * 4;                    // word offset in the warp's stage
  auto issue = [&](int txb, int buf) {
    const int x0 = txb * 32 + bx0 + ch * 4;
    if (cy < p.H && x0 < p.W) {
      const size_t pix = (size_t)cy * p.W + x0;
      cp_async16(&s_fid[warp][buf][so], fid_base + pix);
      cp_async16(&s_g[warp][buf][0][so], g_base + pix);
      cp_async16(&s_g[warp][buf][1][so], g_base + (size_t)HW + pix);
      cp_async16(&s_g[warp][buf][2][so], g_base + 2 * (size_t)HW + pix);
    } else {
      *reinterpret_cast<int4*>(&s_fid[warp][buf][so]) = make_int4(-1, -1, -1, -1);      // outside the image: background
    }
    cp_async_commit();
  };
  issue(0, 0);
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  bool any = false;
  const ShadeCtx sc = load_shade_ctx(p.light, p.light_stride, p.Cc, n);
  float4 ucol = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!VRGB) ucol = make_float4(__ldg(p.obj_rgb), __ldg(p.obj_rgb + 1), __ldg(p.obj_rgb + 2), 0.f);
  constexpr bool SCAT = GV || (GC && VRGB);      // as mesh_backward_kernel
  float gcol[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  // Pixels -> lanes: a warp takes 8x4-pixel BLOCKS (lane = 8 r + c) instead of 32x1 rows.  A face covers ~2.5 x 2.5 pixels
  // at C2: a block touches ~5 faces where a row touches ~13, and every gather instruction of the warp (face record, 3 + 6
  // vertex records) splits into that many fewer L1 wavefronts.
#pragma unroll 1
  for (int t = 0; t < p.tiles_x; ++t) {
    const int buf = t & 1;
    if (t + 1 < p.tiles_x) { issue(t + 1, buf ^ 1); cp_async_wait<1>(); }
    else cp_async_wait<0>();
    __syncwarp();                                      // tile t has landed for every lane of this warp
    // the warp's covered pixels (of its four blocks) compacted into a list: the chain below then runs in
    // ceil(covered / 32) rounds with every lane busy instead of four rounds with the background lanes idle
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool cov = s_fid[warp][buf][j * 32 + lane] >= 0;      // block j, pixel (lane >> 3, lane & 7)
      const unsigned int mk = __ballot_sync(0xffffffffu, cov);
      if (cov) s_list[warp][cnt + __popc(mk & ((1u << lane) - 1u))] = (unsigned char)((j << 5) | lane);
      cnt += __popc(mk);
    }
    __syncwarp();
#pragma unroll 1
    for (int base = 0; base < cnt; base += 32) {
      const bool has = base + lane < cnt;
      if (!SCAT && !has) continue;
      const int o = has ? s_list[warp][base + lane] : 0;          // = 32 j + 8 r + c: the pixel's offset in the stage
      const int x = bx0 + (o & 7), y = by0 + ((o >> 5) << 3) + ((o >> 3) & 3);
      const int fid = s_fid[warp][buf][o];
      float g0 = s_g[warp][buf][0][o], g1 = s_g[warp][buf][1][o], g2 = s_g[warp][buf][2][o];
      const bool live = has && !(g0 == 0.f && g1 == 0.f && g2 == 0.f);
      if (!SCAT && !live) continue;
      if (p.onorm.on) { g0 *= p.onorm.s0; g1 *= p.onorm.s1; g2 *= p.onorm.s2; }
      if (SCAT) {      // all lanes stay together for the warp-aggregated scatter
        float gvn[18];
        int vids[3] = {0, 0, 0};
        bool done = false;
        if (live) {
          any = true;
          done = mesh_backward_pixel<VRGB, GV, GC>(p, n, f0, voff, pvn, persp, sc, ucol, fid, g0, g1, g2, __ldg(p.tab + t * 32 + x), tyb * 32 + y, acc, gvn, vids, gcol);
        }
        if (GV) scatter_vertex_grads(p, voff, done ? fid : -1, gvn, vids);
        if (GC && VRGB) scatter_vertex9<true>(p, voff, done ? fid : -1, gcol, vids);
        continue;
      }
      any = true;
      const float xf = __ldg(p.tab + t * 32 + x);      // covered => inside the image
      mesh_backward_pixel<VRGB, false, GC>(p, n, f0, voff, pvn, persp, sc, ucol, fid, g0, g1, g2, xf, tyb * 32 + y, acc, nullptr, nullptr, gcol);
    }
    __syncwarp();                                      // the list and stage `buf` are free again (tile t + 2 overwrites it)
  }
  const size_t part = (size_t)n * p.parts_per_view + (size_t)tyb * NWARPS + warp;
  if (GC && !VRGB) store_rgb_partial(p, part, gcol);
  float* out = p.partials + part * 16;
  if (!__any_sync(0xffffffffu, any)) {
    if (lane < 16) out[lane] = 0.f;
    return;
  }
  const float mine = warp_sum16_transposed(acc);
  if (!(lane & 1)) out[lane >> 1] = mine;
}

// ---- hard depth: d depth -> barycentrics / z_i -> perspective correction -> edge functions -> NDC -> view space ----
// One covered pixel of mesh_depth_backward_kernel, depth = sum_i b_i z_i (the key's z), cotangent g: acc += (dR 9, dT 3); GV: the
// d/d position of its three vertices in gv[9] (R . d view position), vids set.  Returns false for a pixel of a face crossing the near
// plane (mesh_backward_finish_kernel<false, true> owns it).
// The per-vertex d/d b_i = g z_i are nearly equal (their common part g depth is ~1e3 times their differences on a 10 k-face mesh
// at 224^2), and the Jacobian behind them is ~1/area: they are never formed.  With perspective correction b = t / sum(t) annihilates
// a common shift, so only g (z_i - z_j) enters (the difference form of mesh_backward_pixel with z as the attribute); without it,
// depth = z0 S + w1 (z1 - z0) + w2 (z2 - z0) with S = sum w = A / (A + eps) identically, whose only dependence on the vertices is
// through the area, d S = eps / (A + eps)^2 d A.
template <bool GV>
__device__ __forceinline__ bool mesh_depth_backward_pixel(const MeshBwdParams& p, int n, int f0, int voff, const float4* __restrict__ pvn,
                                                          bool persp, int fid, float g, float xf, int yi, float acc[16], float gv[9],
                                                          int vids[3]) {
  const int4 fi = __ldg(p.faces4 + f0 + fid);
  const Face fc = gather_face(pvn, fi);
  if (may_clip(p.wsflags) && face_straddles(fc, p.z_clip)) return false;
  const FaceEdges fe = face_edges(fc);
  const float yf = __ldg(p.tab + p.W + yi);
  const float e0 = (xf - fc.x1) * fe.A0 - (yf - fc.y1) * fe.B0;
  const float e1 = (xf - fc.x2) * fe.A1 - (yf - fc.y2) * fe.B1;
  const float e2 = (xf - fc.x0) * fe.A2 - (yf - fc.y0) * fe.B2;
  const float inv_area = rcp_fast(fe.area_p);
  const float w0 = e0 * inv_area, w1 = e1 * inv_area, w2 = e2 * inv_area;
  const float d10 = g * (fc.z1 - fc.z0), d20 = g * (fc.z2 - fc.z0);      // g (z_i - z_0)
  float gb0, gb1, gb2, dz0, dz1, dz2, garea;
  if (persp) {
    const float t0 = w0 * fc.z1 * fc.z2, t1 = w1 * fc.z0 * fc.z2, t2 = w2 * fc.z0 * fc.z1;
    const float st = t0 + t1 + t2;
    const bool clamped = st < MVR_K_EPS;
    const float id = rcp_fast(fmaxf(st, MVR_K_EPS));
    const float b0 = t0 * id, b1 = t1 * id, b2 = t2 * id;
    dz0 = g * b0; dz1 = g * b1; dz2 = g * b2;
    float gden = 0.f;
    if (!clamped) {      // gb_i - sum_j b_j gb_j = sum_j b_j g (z_i - z_j)
      const float d01 = -d10, d02 = -d20, d12 = d02 - d01;
      gb0 = fmaf(b1, d01, b2 * d02);
      gb1 = fmaf(b2, d12, -b0 * d01);
      gb2 = -fmaf(b0, d02, b1 * d12);
    } else {
      gb0 = g * fc.z0; gb1 = g * fc.z1; gb2 = g * fc.z2;
      gden = -(gb0 * t0 + gb1 * t1 + gb2 * t2) * id * id;
    }
    const float gt0 = fmaf(gb0, id, gden), gt1 = fmaf(gb1, id, gden), gt2 = fmaf(gb2, id, gden);
    gb0 = gt0 * fc.z1 * fc.z2; gb1 = gt1 * fc.z0 * fc.z2; gb2 = gt2 * fc.z0 * fc.z1;
    dz0 += gt1 * w1 * fc.z2 + gt2 * w2 * fc.z1;
    dz1 += gt0 * w0 * fc.z2 + gt2 * w2 * fc.z0;
    dz2 += gt0 * w0 * fc.z1 + gt1 * w1 * fc.z0;
    garea = clamped ? -(gb0 * e0 + gb1 * e1 + gb2 * e2) * inv_area * inv_area : 0.f;
  } else {
    gb0 = 0.f; gb1 = d10; gb2 = d20;
    dz0 = g * w0; dz1 = g * w1; dz2 = g * w2;
    garea = (g * fc.z0 * MVR_K_EPS - (d10 * e1 + d20 * e2)) * inv_area * inv_area;
  }
  const float ge0 = gb0 * inv_area, ge1 = gb1 * inv_area, ge2 = gb2 * inv_area;
  float gx0, gy0, gx1, gy1, gx2, gy2;
  gx1 = ge0 * (yf - fc.y2); gy1 = ge0 * (fc.x2 - xf); gx2 = ge0 * (fc.y1 - yf); gy2 = ge0 * (xf - fc.x1);          // e0 = E(p,v1,v2)
  gx2 += ge1 * (yf - fc.y0); gy2 += ge1 * (fc.x0 - xf); gx0 = ge1 * (fc.y2 - yf); gy0 = ge1 * (xf - fc.x2);        // e1 = E(p,v2,v0)
  gx0 += ge2 * (yf - fc.y1); gy0 += ge2 * (fc.x1 - xf); gx1 += ge2 * (fc.y0 - yf); gy1 += ge2 * (xf - fc.x0);      // e2 = E(p,v0,v1)
  gx0 += garea * (fc.y2 - fc.y1); gy0 += garea * (fc.x1 - fc.x2);                                                  // area = E(v2,v0,v1)
  gx1 += garea * (fc.y0 - fc.y2); gy1 += garea * (fc.x2 - fc.x0);
  gx2 += garea * (fc.y1 - fc.y0); gy2 += garea * (fc.x0 - fc.x1);
  const float gxn[3] = {gx0, gx1, gx2}, gyn[3] = {gy0, gy1, gy2}, gzn[3] = {dz0, dz1, dz2};
  const float xn[3] = {fc.x0, fc.x1, fc.x2}, yn[3] = {fc.y0, fc.y1, fc.y2}, zv[3] = {fc.z0, fc.z1, fc.z2};
  const int vid[3] = {fi.x, fi.y, fi.z};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const float4 X = __ldg(p.verts4 + voff + vid[i]);
    const float iz = rcp_fast(zv[i]);
    const float gpx = gxn[i] * p.k00 * iz;
    const float gpy = gyn[i] * p.k11 * iz;
    const float gpz = gzn[i] - (gxn[i] * xn[i] + gyn[i] * yn[i]) * iz;
    acc[0] = fmaf(X.x, gpx, acc[0]); acc[1] = fmaf(X.x, gpy, acc[1]); acc[2] = fmaf(X.x, gpz, acc[2]);
    acc[3] = fmaf(X.y, gpx, acc[3]); acc[4] = fmaf(X.y, gpy, acc[4]); acc[5] = fmaf(X.y, gpz, acc[5]);
    acc[6] = fmaf(X.z, gpx, acc[6]); acc[7] = fmaf(X.z, gpy, acc[7]); acc[8] = fmaf(X.z, gpz, acc[8]);
    acc[9] += gpx; acc[10] += gpy; acc[11] += gpz;
    if (GV) {
      const float* r = p.R + 9 * (size_t)n;
      gv[3 * i + 0] = fmaf(__ldg(r + 0), gpx, fmaf(__ldg(r + 1), gpy, __ldg(r + 2) * gpz));
      gv[3 * i + 1] = fmaf(__ldg(r + 3), gpx, fmaf(__ldg(r + 4), gpy, __ldg(r + 5) * gpz));
      gv[3 * i + 2] = fmaf(__ldg(r + 6), gpx, fmaf(__ldg(r + 7), gpy, __ldg(r + 8) * gpz));
      vids[i] = vid[i];
    }
  }
  return true;
}

// grid: x = 32x32-pixel tiles, y = view m, z = object b; thread (lane, warp) owns pixels (x0 + lane, y0 + warp + 8 j), as
// mesh_backward_kernel.  grad_images = the cotangent of the (n,1,H,W) depth plane.  One 16-float camera partial per warp (dC = 0) in
// the layout mesh_backward_finish_kernel sums in fixed order.  GV: d/d vertex positions into p.grad_verts (warp-aggregated atomics).
template <bool GV>
__global__ void __launch_bounds__(MVR_THREADS) mesh_depth_backward_kernel(const MeshBwdParams p) {
  pdl_enter();
  const int tid = threadIdx.x;
  const int b = blockIdx.z, m = blockIdx.y, n = b * p.M + m, cta = blockIdx.x;
  int tyb, txb;
  tile_rc(cta, p.tiles_x, tyb, txb);
  const int xi = txb * 32 + (tid & 31), yi0 = tyb * 32 + (tid >> 5);
  const int HW = p.H * p.W;
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  const float* gd = reinterpret_cast<const float*>(p.grad_images) + (size_t)n * HW;
  int fids[BWD_PIX_PER_THREAD];
  float gin[BWD_PIX_PER_THREAD];
#pragma unroll
  for (int j = 0; j < BWD_PIX_PER_THREAD; ++j) {
    const int yi = yi0 + 8 * j;
    fids[j] = (xi < p.W && yi < p.H) ? __ldg(p.pix_to_face + (size_t)n * HW + (size_t)yi * p.W + xi) : -1;
  }
#pragma unroll
  for (int j = 0; j < BWD_PIX_PER_THREAD; ++j) gin[j] = fids[j] >= 0 ? __ldg(gd + (size_t)(yi0 + 8 * j) * p.W + xi) : 0.f;
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  bool any = false;
  const float xf = xi < p.W ? __ldg(p.tab + xi) : 0.f;
#pragma unroll 1
  for (int j = 0; j < BWD_PIX_PER_THREAD; ++j) {
    const int fid = fids[j];
    const bool live = fid >= 0 && gin[j] != 0.f;
    if (GV) {      // all lanes stay together for the warp-aggregated scatter
      float gv[9];
      int vids[3] = {0, 0, 0};
      bool done = false;
      if (live) { any = true; done = mesh_depth_backward_pixel<true>(p, n, f0, voff, pvn, persp, fid, gin[j], xf, yi0 + 8 * j, acc, gv, vids); }
      scatter_vertex9<false>(p, voff, done ? fid : -1, gv, vids);
      continue;
    }
    if (!live) continue;
    any = true;
    mesh_depth_backward_pixel<false>(p, n, f0, voff, pvn, persp, fid, gin[j], xf, yi0 + 8 * j, acc, nullptr, nullptr);
  }
  float* out = p.partials + ((size_t)n * p.parts_per_view + (size_t)cta * NWARPS + (tid >> 5)) * 16;
  const int lane = tid & 31;
  if (!__any_sync(0xffffffffu, any)) {
    if (lane < 16) out[lane] = 0.f;
    return;
  }
  const float mine = warp_sum16_transposed(acc);
  if (!(lane & 1)) out[lane >> 1] = mine;
}

}  // namespace mvr

using namespace mvr;

extern "C" int mvr_mesh_depth_backward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                       int64_t total_verts, int64_t total_faces, int max_verts, const float* R, const float* T,
                                       float k00, float k11, float z_clip, int H, int W, int flags, const int* pix_to_face,
                                       const float* grad_depth, float* gR, float* gT, float* grad_verts, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  int rc = check_mesh_common("mvr_mesh_depth_backward", B, M, H, W, 1, total_verts, total_faces, max_verts);
  if (rc) return rc;
  const int64_t N = (int64_t)B * M;
  if (N == 0) return 0;
  if (!geometry || !vert_off || !face_off || !R || !T || !pix_to_face || !grad_depth || !gR || !gT || !workspace) {
    set_error("mvr_mesh_depth_backward: null pointer"); return -5;
  }
  const WsLayout w = ws_layout(B, M, H, W, 1, total_verts, total_faces);
  if (workspace_bytes < w.total) { set_error("mvr_mesh_depth_backward: workspace too small (%zu < %zu)", workspace_bytes, w.total); return -7; }
  const GeomLayout g = geom_layout(total_verts, total_faces);
  const char* gb = (const char*)geometry;
  char* wb = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  if (!(flags & MVR_WS_PROJECTED)) rc = launch_project("mesh_project_kernel", g, w, geometry, vert_off, R, T, B, M, H, W, max_verts, k00, k11, z_clip, true, workspace, st);
  if (rc) return rc;
  MeshBwdParams p = {};
  p.verts4 = (const float4*)(gb + g.verts4); p.normals4 = (const float4*)(gb + g.normals4);
  p.rgb4 = (const float4*)(gb + g.rgb4); p.faces4 = (const int4*)(gb + g.faces4); p.xn8 = (const float4*)(gb + g.xn8);
  p.vert_off = vert_off; p.face_off = face_off;
  p.R = R; p.T = T;
  p.k00 = k00; p.k11 = k11;
  p.B = B; p.M = M; p.H = H; p.W = W; p.K = 1; p.flags = flags; p.ctas_per_view = w.bwd_ctas_per_view; p.tiles_x = (W + 31) / 32;
  p.pv = (const float4*)(wb + w.pv); p.tab = (const float*)(wb + w.tab);
  p.pix_to_face = pix_to_face; p.grad_images = grad_depth;
  p.partials = (float*)(wb + w.partials); p.grad_verts = grad_verts;
  p.z_clip = z_clip; p.wsflags = (int*)(wb + w.flags); p.parts_per_view = w.bwd_parts_per_view;
  const dim3 bgrid((unsigned)w.bwd_ctas_per_view, (unsigned)M, (unsigned)B);
  if (grad_verts) MVR_LAUNCH_PDL(mesh_depth_backward_kernel<true>, bgrid, MVR_THREADS, 0, st, p);
  else MVR_LAUNCH_PDL(mesh_depth_backward_kernel<false>, bgrid, MVR_THREADS, 0, st, p);
  rc = check_launch("mesh_depth_backward_kernel");
  if (rc) return rc;
  // clipped-face pixels (if any) + the fixed-order sum of the per-warp partials -> gR, gT
  return launch_mesh_backward_finish(p, (int)N, gR, gT, nullptr, st, true);
}

static int mesh_backward_impl(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                              int64_t total_verts, int64_t total_faces, int max_verts, const float* R,
                              const float* T, const float* Cc, const float* light, int light_stride,
                              const float* obj_rgb, float k00, float k11, float z_clip, int H, int W, int K, int flags,
                              const float* out_mean_std, const int* pix_to_face, const void* grad_images, float* gR, float* gT, float* gC,
                              float* grad_verts, float* grad_normals, void* workspace, size_t workspace_bytes,
                              void* stream, const float* azim, const float* elev, const float* dist, float* g_azim, float* g_elev,
                              float* g_dist, float* grad_rgb) {
  int rc = check_mesh_common("mvr_mesh_backward", B, M, H, W, K, total_verts, total_faces, max_verts);
  if (rc) return rc;
  const int64_t N = (int64_t)B * M;
  if (N == 0) return 0;
  if (!geometry || !vert_off || !face_off || !R || !T || !Cc || !light || !pix_to_face || !grad_images || !workspace ||
      (!azim && (!gR || !gT || !gC)) || (azim && (!elev || !dist || !g_azim || !g_elev || !g_dist))) {
    set_error("mvr_mesh_backward: null pointer"); return -5;
  }
  if (!(flags & MVR_RGB_PER_ELEMENT) && !obj_rgb) { set_error("mvr_mesh_backward: obj_rgb is NULL"); return -6; }
  if (!out_norm_valid(out_mean_std)) { set_error("mvr_mesh_backward: out_mean_std needs std > 0"); return -9; }
  const WsLayout w = ws_layout(B, M, H, W, K, total_verts, total_faces);
  if (workspace_bytes < w.total) { set_error("mvr_mesh_backward: workspace too small (%zu < %zu)", workspace_bytes, w.total); return -7; }
  const GeomLayout g = geom_layout(total_verts, total_faces);
  const char* gb = (const char*)geometry;
  char* wb = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  // the workspace is scratch (it may have served another render since the forward): project again, 1% of the step,
  // unless the caller vouches that it has not (MVR_WS_PROJECTED)
  if (!(flags & MVR_WS_PROJECTED)) rc = launch_project("mesh_project_kernel", g, w, geometry, vert_off, R, T, B, M, H, W, max_verts, k00, k11, z_clip, true, workspace, st);
  if (rc) return rc;
  MeshBwdParams p;
  p.verts4 = (const float4*)(gb + g.verts4); p.normals4 = (const float4*)(gb + g.normals4);
  p.rgb4 = (const float4*)(gb + g.rgb4); p.faces4 = (const int4*)(gb + g.faces4); p.xn8 = (const float4*)(gb + g.xn8);
  p.vert_off = vert_off; p.face_off = face_off;
  p.R = R; p.T = T; p.Cc = Cc; p.light = light; p.light_stride = light_stride; p.obj_rgb = obj_rgb;
  p.k00 = k00; p.k11 = k11;
  p.B = B; p.M = M; p.H = H; p.W = W; p.K = K; p.flags = flags; p.ctas_per_view = w.bwd_ctas_per_view; p.tiles_x = (W + 31) / 32;
  p.pv = (const float4*)(wb + w.pv); p.tab = (const float*)(wb + w.tab);
  p.pix_to_face = pix_to_face; p.grad_images = grad_images;
  p.partials = (float*)(wb + w.partials); p.grad_verts = grad_verts; p.grad_normals = grad_normals;
  p.onorm = make_out_norm(out_mean_std);
  p.z_clip = z_clip; p.wsflags = (int*)(wb + w.flags); p.parts_per_view = w.bwd_parts_per_view;
  p.azim = azim; p.elev = elev; p.dist = dist; p.g_azim = g_azim; p.g_elev = g_elev; p.g_dist = g_dist;
  p.grad_rgb = grad_rgb; p.rgb_partials = (float*)(wb + w.rgb_partials); p.rgb_views = (double*)(wb + w.rgb_views);
  const dim3 bgrid((unsigned)w.bwd_ctas_per_view, (unsigned)M, (unsigned)B);
  const bool vrgb = flags & MVR_RGB_PER_ELEMENT;
  const bool strip = K == 1 && !(flags & MVR_IMAGES_BF16) && W % 4 == 0 &&
                     ((uintptr_t)pix_to_face % 16 == 0) && ((uintptr_t)grad_images % 16 == 0);
  const bool gv = grad_verts || grad_normals;
  if (grad_rgb) {      // colour gradients: instances of their own (GC), so that the ones above stay as they are
    if (strip) {
      p.parts_per_view = ((H + 31) / 32) * NWARPS;
      const dim3 sgrid((unsigned)((H + 31) / 32), (unsigned)M, (unsigned)B);
      if (gv) {
        if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel_strip<2, true, true, true>), sgrid, MVR_THREADS, 0, st, p);
        else MVR_LAUNCH_PDL((mesh_backward_kernel_strip<2, false, true, true>), sgrid, MVR_THREADS, 0, st, p);
      }
      else if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel_strip<2, true, false, true>), sgrid, MVR_THREADS, 0, st, p);
      else MVR_LAUNCH_PDL((mesh_backward_kernel_strip<3, false, false, true>), sgrid, MVR_THREADS, 0, st, p);
    }
    else if (gv) { if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel<2, true, true, true>), bgrid, MVR_THREADS, 0, st, p); else MVR_LAUNCH_PDL((mesh_backward_kernel<2, false, true, true>), bgrid, MVR_THREADS, 0, st, p); }
    else if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel<2, true, false, true>), bgrid, MVR_THREADS, 0, st, p);
    else MVR_LAUNCH_PDL((mesh_backward_kernel<3, false, false, true>), bgrid, MVR_THREADS, 0, st, p);
  }
  else if (strip) {
    p.parts_per_view = ((H + 31) / 32) * NWARPS;      // one partial per warp of every tile ROW
    const dim3 sgrid((unsigned)((H + 31) / 32), (unsigned)M, (unsigned)B);
    if (gv) {      // vertex gradients: the variant with the warp-aggregated atomic scatter (its 18 extra live values cost occupancy)
      if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel_strip<2, true, true>), sgrid, MVR_THREADS, 0, st, p);
      else MVR_LAUNCH_PDL((mesh_backward_kernel_strip<2, false, true>), sgrid, MVR_THREADS, 0, st, p);
    }
    else if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel_strip<3, true, false>), sgrid, MVR_THREADS, 0, st, p);
    else MVR_LAUNCH_PDL((mesh_backward_kernel_strip<3, false, false>), sgrid, MVR_THREADS, 0, st, p);
  }
  else if (gv) { if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel<2, true, true>), bgrid, MVR_THREADS, 0, st, p); else MVR_LAUNCH_PDL((mesh_backward_kernel<2, false, true>), bgrid, MVR_THREADS, 0, st, p); }
  else if (vrgb) MVR_LAUNCH_PDL((mesh_backward_kernel<3, true, false>), bgrid, MVR_THREADS, 0, st, p);
  else MVR_LAUNCH_PDL((mesh_backward_kernel<3, false, false>), bgrid, MVR_THREADS, 0, st, p);
  rc = check_launch("mesh_backward_kernel");
  if (rc) return rc;
  // clipped-face pixels (if any) + the fixed-order sum of the per-warp partials -> gR, gT, gC (and the colour gradient)
  return launch_mesh_backward_finish(p, (int)N, gR, gT, gC, st);
}

extern "C" int mvr_mesh_backward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                 int64_t total_verts, int64_t total_faces, int max_verts, const float* R,
                                 const float* T, const float* Cc, const float* light, int light_stride,
                                 const float* obj_rgb, float k00, float k11, float z_clip, int H, int W, int K, int flags,
                                 const float* out_mean_std, const int* pix_to_face, const void* grad_images, float* gR, float* gT, float* gC,
                                 float* grad_verts, float* grad_normals, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  return mesh_backward_impl(geometry, vert_off, face_off, B, M, total_verts, total_faces, max_verts, R, T, Cc, light, light_stride, obj_rgb,
                            k00, k11, z_clip, H, W, K, flags, out_mean_std, pix_to_face, grad_images, gR, gT, gC, grad_verts, grad_normals,
                            workspace, workspace_bytes, stream, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

// mvr_mesh_backward that also returns the colour gradient: grad_rgb (Vtot, 3), accumulated, for per-vertex colours
// (MVR_RGB_PER_ELEMENT), else (3) for the one object colour, written (fixed-order sum, bit-reproducible).
extern "C" int mvr_mesh_backward_rgb(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                     int64_t total_verts, int64_t total_faces, int max_verts, const float* R,
                                     const float* T, const float* Cc, const float* light, int light_stride,
                                     const float* obj_rgb, float k00, float k11, float z_clip, int H, int W, int K, int flags,
                                     const float* out_mean_std, const int* pix_to_face, const void* grad_images, float* gR, float* gT, float* gC,
                                     float* grad_verts, float* grad_normals, void* workspace, size_t workspace_bytes,
                                     void* stream, float* grad_rgb) {
  return mesh_backward_impl(geometry, vert_off, face_off, B, M, total_verts, total_faces, max_verts, R, T, Cc, light, light_stride, obj_rgb,
                            k00, k11, z_clip, H, W, K, flags, out_mean_std, pix_to_face, grad_images, gR, gT, gC, grad_verts, grad_normals,
                            workspace, workspace_bytes, stream, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, grad_rgb);
}

// mvr_mesh_backward for cameras that came from mvr_look_at_forward(azim, elev, dist): the kernel that sums the per-warp partials of a
// view also applies its camera backward (look_at_backward_view), so the chain ends in (d azim, d elev, d dist) with one launch less.
extern "C" int mvr_mesh_backward_angles(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                        int64_t total_verts, int64_t total_faces, int max_verts, const float* R,
                                        const float* T, const float* Cc, const float* light, int light_stride,
                                        const float* obj_rgb, float k00, float k11, float z_clip, int H, int W, int K, int flags,
                                        const float* out_mean_std, const int* pix_to_face, const void* grad_images,
                                        const float* azim, const float* elev, const float* dist, float* g_azim, float* g_elev,
                                        float* g_dist, float* gR, float* gT, float* gC, float* grad_verts, float* grad_normals,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  if (!azim) { set_error("mvr_mesh_backward_angles: null pointer"); return -5; }
  return mesh_backward_impl(geometry, vert_off, face_off, B, M, total_verts, total_faces, max_verts, R, T, Cc, light, light_stride, obj_rgb,
                            k00, k11, z_clip, H, W, K, flags, out_mean_std, pix_to_face, grad_images, gR, gT, gC, grad_verts, grad_normals,
                            workspace, workspace_bytes, stream, azim, elev, dist, g_azim, g_elev, g_dist, nullptr);
}
