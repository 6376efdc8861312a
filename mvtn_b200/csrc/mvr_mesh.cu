// mvr_mesh.cu -- mesh path of MVRenderer (renderer.py:65-114) for sm_100a.
//
//   prepare : pack verts/normals/colours to float4 and faces to int4; area-weighted vertex normals
//             ([upstream] Meshes._compute_vertex_normals) once per OBJECT, not per view.
//   project : mesh_project_kernel -- every vertex of every view is projected exactly ONCE (world -> view -> NDC,
//             IEEE order) into a float4 (x_ndc, y_ndc, z_view) plane that stays L2-resident (30 MB at C2); the
//             scatter, shade and backward kernels gather it instead of re-projecting three vertices per
//             face / pixel.  The same launch writes the table of exact pixel-centre NDC coordinates.
//   scatter : mesh_scatter_kernel -- each face of each view is set up exactly ONCE (project, cull, exact pixel
//             bbox) by the CTA that owns its 1024-face chunk.  No bins: the work is flattened inside the CTA
//             through shared-memory queues so that every phase runs on full warps --
//               A  setup    thread per face   -> record + runs of <= 32 bbox pixels ("sub-items")
//               B  filter   thread per run    -> edge-function sign test  -> per-warp candidate queues
//               C  resolve  thread per candidate: exact barycentrics / depth -> 64-bit (z, face) RED.MIN on the
//                           pixel's key in a global (L2-resident) key plane
//             so a 3-pixel sliver and a large triangle cost their threads the same, and the IEEE divisions run
//             only on dense warps of pixels that are inside their face.  Triangles covering > 1024 pixels are
//             walked by the whole CTA.  K > 1 peels layers (pass k keeps keys > layer k-1).
//   shade   : mesh_shade_kernel -- one thread per pixel: winning key -> face, exact barycentrics recomputed with the
//             same operation sequence, Phong shading + hard background blend, planar (n,3,H,W) image and
//             pix_to_face (+ optional zbuf / bary / dists) written with fully coalesced stores.
//   backward: mesh_backward_kernel -- per pixel recompute (no fragment traffic), chain
//             d image -> Phong -> barycentrics -> NDC verts -> view verts -> (dR, dT, dC), block-reduced to
//             one partial per CTA and summed in fixed order (deterministic, no float atomics).
#include "mvr_mesh_fwd.cuh"

namespace mvr {

// ------------------------------------------------------------------------------------------------
// prepare
// ------------------------------------------------------------------------------------------------
__global__ void geom_pack_verts_kernel(const float* __restrict__ verts, const float* __restrict__ rgb, int64_t tv,
                                       float4* __restrict__ verts4, float4* __restrict__ rgb4, double* __restrict__ nacc) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= tv) return;
  verts4[v] = make_float4(verts[3 * v], verts[3 * v + 1], verts[3 * v + 2], 0.f);
  if (rgb) rgb4[v] = make_float4(rgb[3 * v], rgb[3 * v + 1], rgb[3 * v + 2], 0.f);
  nacc[3 * v] = 0.0; nacc[3 * v + 1] = 0.0; nacc[3 * v + 2] = 0.0;
}

template <typename IdxT>
__global__ void geom_pack_faces_kernel(const IdxT* __restrict__ faces, const int* __restrict__ vert_off,
                                       const int* __restrict__ face_off, const float4* __restrict__ verts4,
                                       int4* __restrict__ faces4, double* __restrict__ nacc) {
  pdl_enter();
  const int b = blockIdx.y;
  const int f0 = face_off[b], F = face_off[b + 1] - f0;
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const int voff = vert_off[b], V = vert_off[b + 1] - voff;
  const IdxT* fp = faces + 3 * (size_t)(f0 + f);
  int i0 = (int)fp[0], i1 = (int)fp[1], i2 = (int)fp[2];
  // out-of-range ids would fault later: clamp (garbage in, bounded garbage out)
  i0 = min(max(i0, 0), V - 1); i1 = min(max(i1, 0), V - 1); i2 = min(max(i2, 0), V - 1);
  faces4[f0 + f] = make_int4(i0, i1, i2, 0);
  const float4 v0 = verts4[voff + i0], v1 = verts4[voff + i1], v2 = verts4[voff + i2];
  // [upstream] Meshes._compute_vertex_normals: one area-weighted cross product PER CORNER -- corner c adds
  // (v_next - v_c) x (v_prev - v_c) to its vertex (the three are equal in exact arithmetic, ~1 ulp apart in fp32).
  // double accumulation: order-independent to ~1e-16, i.e. run-to-run identical after rounding to fp32
  const float4 vc[3] = {v0, v1, v2};
  const int id[3] = {i0, i1, i2};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float4 o = vc[c], a = vc[(c + 1) % 3], b = vc[(c + 2) % 3];
    const float ax = a.x - o.x, ay = a.y - o.y, az = a.z - o.z;
    const float bx = b.x - o.x, by = b.y - o.y, bz = b.z - o.z;
    double* dst = nacc + 3 * (size_t)(voff + id[c]);
    atomicAdd(dst, (double)(ay * bz - az * by)); atomicAdd(dst + 1, (double)(az * bx - ax * bz)); atomicAdd(dst + 2, (double)(ax * by - ay * bx));
  }
}

// ---- backward of the vertex normals (only when mesh vertices require grad): d/d unit normals -> d/d verts ----
// n_v = s_v / max(|s_v|, 1e-6), s_v = sum over the corners at v of (v_next - v_c) x (v_prev - v_c).
// pass 1 (thread / vertex): g_s = normalize_bwd(s, g_n), in place over grad_normals;
// pass 2 (thread / face):   per corner with a = v_next - v_c, b = v_prev - v_c: g_a = b x g_s, g_b = g_s x a,
//                           v_next += g_a, v_prev += g_b, v_c -= g_a + g_b  (float atomics: tolerance-compared).
__global__ void geom_normals_bwd_vertex_kernel(const double* __restrict__ nacc, int64_t tv, float* __restrict__ gn) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= tv) return;
  const float x = (float)nacc[3 * v], y = (float)nacc[3 * v + 1], z = (float)nacc[3 * v + 2];
  const float gx = gn[3 * v], gy = gn[3 * v + 1], gz = gn[3 * v + 2];
  const float n = sqrtf((x * x + y * y) + z * z);
  float ox, oy, oz;
  if (n > 1e-6f) {
    const float inv = 1.0f / n, ux = x * inv, uy = y * inv, uz = z * inv;
    const float d = ux * gx + uy * gy + uz * gz;
    ox = (gx - ux * d) * inv; oy = (gy - uy * d) * inv; oz = (gz - uz * d) * inv;
  } else {
    ox = gx * 1e6f; oy = gy * 1e6f; oz = gz * 1e6f;
  }
  gn[3 * v] = ox; gn[3 * v + 1] = oy; gn[3 * v + 2] = oz;
}

__global__ void geom_normals_bwd_face_kernel(const int4* __restrict__ faces4, const int* __restrict__ vert_off,
                                             const int* __restrict__ face_off, const float4* __restrict__ verts4,
                                             const float* __restrict__ gs, float* __restrict__ grad_verts) {
  const int b = blockIdx.y;
  const int f0 = face_off[b], F = face_off[b + 1] - f0;
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const int voff = vert_off[b];
  const int4 fi = faces4[f0 + f];
  const int id[3] = {fi.x, fi.y, fi.z};
  const float4 vc[3] = {verts4[voff + fi.x], verts4[voff + fi.y], verts4[voff + fi.z]};
  float acc[3][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int nx = (c + 1) % 3, pr = (c + 2) % 3;
    const float* g = gs + 3 * (size_t)(voff + id[c]);
    const float gx = g[0], gy = g[1], gz = g[2];
    const float ax = vc[nx].x - vc[c].x, ay = vc[nx].y - vc[c].y, az = vc[nx].z - vc[c].z;
    const float bx = vc[pr].x - vc[c].x, by = vc[pr].y - vc[c].y, bz = vc[pr].z - vc[c].z;
    const float gax = by * gz - bz * gy, gay = bz * gx - bx * gz, gaz = bx * gy - by * gx;      // b x g
    const float gbx = gy * az - gz * ay, gby = gz * ax - gx * az, gbz = gx * ay - gy * ax;      // g x a
    acc[nx][0] += gax; acc[nx][1] += gay; acc[nx][2] += gaz;
    acc[pr][0] += gbx; acc[pr][1] += gby; acc[pr][2] += gbz;
    acc[c][0] -= gax + gbx; acc[c][1] -= gay + gby; acc[c][2] -= gaz + gbz;
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float* o = grad_verts + 3 * (size_t)(voff + id[c]);
    atomicAdd(o, acc[c][0]); atomicAdd(o + 1, acc[c][1]); atomicAdd(o + 2, acc[c][2]);
  }
}

__global__ void geom_finish_normals_kernel(const double* __restrict__ nacc, int64_t tv, const float4* __restrict__ verts4,
                                           float4* __restrict__ normals4, float4* __restrict__ xn8) {
  pdl_enter();
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= tv) return;
  const float x = (float)nacc[3 * v], y = (float)nacc[3 * v + 1], z = (float)nacc[3 * v + 2];
  const float n = sqrtf((x * x + y * y) + z * z);
  const float d = n > 1e-6f ? n : 1e-6f;
  const float4 nn = make_float4(x / d, y / d, z / d, 0.f);
  normals4[v] = nn;
  xn8[2 * v] = verts4[v]; xn8[2 * v + 1] = nn;      // the interleaved copy the per-pixel kernels gather
}

__global__ void geom_get_normals_kernel(const float4* __restrict__ normals4, int64_t tv, float* __restrict__ out) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= tv) return;
  const float4 n = normals4[v];
  out[3 * v] = n.x; out[3 * v + 1] = n.y; out[3 * v + 2] = n.z;
}

constexpr int SC_REC_WORDS = 13;      // x0 y0 z0 x1 y1 z1 x2 y2 z2 fid zmin_bits | rect_xy rect_wh (big faces only)
constexpr int SC_QCAP = 3072;         // candidates per round (256 faces x ~4.6 inside pixels at C2)

template <int MINB, bool SOFT, int NT = MVR_THREADS>      // NT: threads (= faces per round) of a CTA
__global__ void __launch_bounds__(NT, MINB) mesh_scatter_kernel(const MeshParams p) {
  __shared__ float s_rec[SC_REC_WORDS][NT];  // SoA face records of the current round
  __shared__ int s_q[SC_QCAP * NT / 256];                         // candidates of the round: slot | x << 8 | y << 20
  __shared__ int s_big[NT];
  __shared__ int s_cnt2[2][2];                         // per round parity: [0] candidates, [1] big faces
  pdl_enter();
  __shared__ __align__(16) int4 s_faces[2][NT];      // face records of two rounds: TMA bulk-copy destinations
  __shared__ __align__(8) unsigned long long s_mbar[2];
  extern __shared__ float s_tab[];                     // pixel centres: xf[W], yf[H]
  const float* s_xf = s_tab;
  const float* s_yf = s_tab + p.W;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // grid: x = chunk of faces, y = view m, z = object b (no integer divisions in the prologue)
  const int chunk = blockIdx.x, m = blockIdx.y, b = blockIdx.z, n = b * p.M + m;
  const int f0 = p.face_off[b], F = p.face_off[b + 1] - f0;
  const int fbeg = chunk * FACES_PER_CTA, fend = min(F, fbeg + FACES_PER_CTA);
  if (fbeg >= fend) return;
  const int voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;     // this view's projected vertices
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  unsigned long long* keys = p.keys + (size_t)n * p.H * p.W;
  const unsigned long long* prev = p.layer > 0 ? p.prev + (size_t)n * p.H * p.W : nullptr;
  const int qcap = p.wcap;      // SC_QCAP, or a handful under MVR_TEST_TINY_QUEUES
  const SoftMode sm = SOFT ? soft_mode(p) : SoftMode{0.f, 0.f, false};
  constexpr bool soft = SOFT;   // blur_radius > 0 / clipped barycentrics: every pixel of the (grown) bbox is a candidate

  // The chunk's face records (int4 vertex ids) are CONTIGUOUS: each round's 256 records (4 KB) are staged by a 1-D TMA bulk
  // copy (cp.async.bulk + mbarrier), round r + 1 in flight while round r is rasterized -- the first of the two dependent trips of
  // the setup (face record -> projected vertices) leaves the critical path of every round but the first.
  const unsigned int mbar_a = smem_addr_pinned(&s_mbar[0]);
  const unsigned int fstage_a = smem_addr_pinned(&s_faces[0][0]);
  auto issue_faces = [&](int r) {      // one thread; 16-byte records: source aligned, size a multiple of 16
    const int start = fbeg + r * NT;
    const unsigned int bytes = (unsigned int)(min(NT, fend - start) * 16);
    const unsigned int mb = mbar_a + 8u * (r & 1);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     fstage_a + 16u * NT * (r & 1)),
                 "l"(p.faces4 + f0 + start), "r"(bytes), "r"(mb)
                 : "memory");
  };
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_a) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_a + 8u) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    issue_faces(0);
  }
  for (int i = tid; i < p.W + p.H; i += NT) s_tab[i] = __ldg(p.tab + i);
  if (tid < 4) (&s_cnt2[0][0])[tid] = 0;
  __syncthreads();
  const unsigned int q_a = smem_addr_pinned(&s_q[0]);

  int n_straddle = 0, n_big = 0;
  for (int rbeg = fbeg, rpar = 0, round = 0; rbeg < fend; rbeg += NT, rpar ^= 1, ++round) {
    int* s_cnt = s_cnt2[rpar];
    if (tid == 0 && rbeg + NT < fend) issue_faces(round + 1);      // its stage was released by the barrier that ended round - 1
    {
      const unsigned int mb = mbar_a + 8u * (round & 1), parity = (unsigned int)((round >> 1) & 1);
      asm volatile(
          "{\n.reg .pred p;\nWAITF_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONEF_%=;\nbra WAITF_%=;\nDONEF_%=:\n}\n" ::"r"(mb),
          "r"(parity)
          : "memory");
    }
    // ---------------- phase A: setup + scanline spans, one thread per face ----------------
    // gather, cull, exact bbox, then ROW BY ROW the interval of pixels that can pass the edge filter (row_span_regs): its
    // pixels go straight to the round's candidate queue.  The filter coefficients never leave the registers.
    const int fid = rbeg + tid;
    int xl = 0, yl = 0, bw = 0, bh = 0;
    SpanEdges se;
    if (fid < fend) {
      const Face fc = gather_face(pvn, s_faces[round & 1][tid]);
      int xh, yh;
      const bool straddles = face_straddles(fc, p.z_clip);
      if (straddles || face_pixel_bbox_conservative(fc, p, xl, xh, yl, yh)) {
        s_rec[0][tid] = fc.x0; s_rec[1][tid] = fc.y0; s_rec[2][tid] = fc.z0;
        s_rec[3][tid] = fc.x1; s_rec[4][tid] = fc.y1; s_rec[5][tid] = fc.z1;
        s_rec[6][tid] = fc.x2; s_rec[7][tid] = fc.y2; s_rec[8][tid] = fc.z2;
        s_rec[9][tid] = __int_as_float(fid);
        const float zmin = fminf(fminf(fc.z0, fc.z1), fc.z2);
        s_rec[10][tid] = __uint_as_float((persp && zmin > 1e-3f && !soft) ? __float_as_uint(zmin * 0.999999f) : 0u);
        if (straddles) {
          // crosses the near clip plane ([upstream] clip.py): counted, visible or not (as the oracle does), and handed to
          // the whole CTA below, which rasterizes its one or two clipped sub-triangles
          n_straddle += p.layer == 0;
          s_big[atomicAdd(&s_cnt[1], 1)] = tid | 0x100;
        } else {
          bw = xh - xl + 1; bh = yh - yl + 1;
          if (bw * bh > BIG_FACE_PIX) {      // walked by the whole CTA below
            s_rec[11][tid] = __int_as_float(xl | (yl << 16));
            s_rec[12][tid] = __int_as_float(bw | (bh << 16));
            s_big[atomicAdd(&s_cnt[1], 1)] = tid;
            bh = 0;
          } else if (!soft) {
            se = span_edges(fc, p.ndc_max);
          }
        }
      }
    }
    {
      const int maxr = __reduce_max_sync(0xffffffffu, bh);
      for (int row = 0; row < maxr; ++row) {      // warp-uniform trip count
        int cnt = 0, xs = 0;
        const int yy = yl + row;
        if (row < bh) {
          if (soft) { cnt = bw; xs = xl; }
          else cnt = row_span_regs(se, s_yf[yy], xl, bw, p.W, p.jx_scale, p.jx_off, xs);
        }
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        if (total == 0) continue;
        int base = 0;
        if (lane == 31) base = atomicAdd(&s_cnt[0], total);
        base = __shfl_sync(0xffffffffu, base, 31) + incl - cnt;
        const unsigned int word0 = (unsigned)tid | ((unsigned)xs << 8) | ((unsigned)yy << 20);
        const int maxc = __reduce_max_sync(0xffffffffu, cnt);
        for (int c = 0; c < maxc; ++c) {
          if (c < cnt) {
            const int at = base + c;
            if (at < qcap) {
              sts_u32(q_a + 4u * (unsigned)at, word0 + ((unsigned)c << 8));
            } else {                                                  // queue full: resolve in place
              const int xx = xs + c;
              Face fc;
              fc.x0 = s_rec[0][tid]; fc.y0 = s_rec[1][tid]; fc.z0 = s_rec[2][tid];
              fc.x1 = s_rec[3][tid]; fc.y1 = s_rec[4][tid]; fc.z1 = s_rec[5][tid];
              fc.x2 = s_rec[6][tid]; fc.y2 = s_rec[7][tid]; fc.z2 = s_rec[8][tid];
              resolve_pixel<SOFT>(fc, face_edges(fc), fid, 0u, persp, s_xf[xx], s_yf[yy], keys + (size_t)yy * p.W + xx,
                            prev ? prev + (size_t)yy * p.W + xx : nullptr, sm);
            }
          }
        }
      }
    }
    __syncthreads();
    // ---------------- phase C: exact resolve, the round's candidates spread over all threads ----------------
    const int total_c = min(s_cnt[0], qcap);
    const int n_bigf = s_cnt[1];
    if (tid < 2) s_cnt2[rpar ^ 1][tid] = 0;      // the next round's counters (last read before the barrier that ended the previous round)
    {
      // the key of the NEXT candidate is fetched before the current one is resolved: its trip to L2 overlaps the
      // divisions instead of stalling the early depth test (a thread resolves ~4-5 candidates per round)
      int cd_next = 0;
      unsigned long long cur_next = 0ull;
      if (tid < total_c) {
        cd_next = s_q[tid];
        cur_next = __ldcg(keys + (size_t)((cd_next >> 20) & 4095) * p.W + ((cd_next >> 8) & 4095));
      }
      for (int j = tid; j < total_c; j += NT) {
        const int cd = cd_next;
        const unsigned long long cur = cur_next;
        if (j + NT < total_c) {
          cd_next = s_q[j + NT];
          cur_next = __ldcg(keys + (size_t)((cd_next >> 20) & 4095) * p.W + ((cd_next >> 8) & 4095));
        }
        const int slot = cd & 255, xx = (cd >> 8) & 4095, yy = (cd >> 20) & 4095;
        const unsigned int zmin_bits = __float_as_uint(s_rec[10][slot]);
        if (zmin_bits > (unsigned int)(cur >> 32)) continue;      // hidden: before the face record is even read
        Face fc;
        fc.x0 = s_rec[0][slot]; fc.y0 = s_rec[1][slot]; fc.z0 = s_rec[2][slot];
        fc.x1 = s_rec[3][slot]; fc.y1 = s_rec[4][slot]; fc.z1 = s_rec[5][slot];
        fc.x2 = s_rec[6][slot]; fc.y2 = s_rec[7][slot]; fc.z2 = s_rec[8][slot];
        resolve_pixel_with<SOFT>(fc, face_edges(fc), __float_as_int(s_rec[9][slot]), zmin_bits, persp, s_xf[xx], s_yf[yy],
                           keys + (size_t)yy * p.W + xx, prev ? prev + (size_t)yy * p.W + xx : nullptr, cur, sm);
      }
    }
    // ---------------- large faces: the whole CTA walks the bbox ----------------
    int n_clipf = 0;
    for (int q = 0; q < n_bigf; ++q) {
      const int ent = s_big[q], slot = ent & 255;
      Face fc;
      fc.x0 = s_rec[0][slot]; fc.y0 = s_rec[1][slot]; fc.z0 = s_rec[2][slot];
      fc.x1 = s_rec[3][slot]; fc.y1 = s_rec[4][slot]; fc.z1 = s_rec[5][slot];
      fc.x2 = s_rec[6][slot]; fc.y2 = s_rec[7][slot]; fc.z2 = s_rec[8][slot];
      const int bfid = __float_as_int(s_rec[9][slot]);
      if (ent & 0x100) {      // near-plane clipping: the sub-triangles compete under the ORIGINAL face id
        ++n_clipf;
        ClipSub cs;
        clip_face(fc, p.z_clip, persp, cs);
        for (int s = 0; s < cs.ns; ++s) {
          const Face sf = cs.f[s];
          int cxl, cxh, cyl, cyh;
          if (!face_pixel_bbox(sf, p, s_xf, s_yf, cxl, cxh, cyl, cyh)) continue;
          const FaceEdges sfe = face_edges(sf);
          for (int yy = cyl + warp; yy <= cyh; yy += (NT / 32))
            for (int xx = cxl + lane; xx <= cxh; xx += 32)
              resolve_pixel<SOFT>(sf, sfe, bfid, 0u, persp, s_xf[xx], s_yf[yy], keys + (size_t)yy * p.W + xx,
                            prev ? prev + (size_t)yy * p.W + xx : nullptr, sm);
        }
        continue;
      }
      const FaceEdges fe = face_edges(fc);
      const int rxy = __float_as_int(s_rec[11][slot]), rwh = __float_as_int(s_rec[12][slot]);
      const int bxl = rxy & 0xffff, byl = rxy >> 16, bbw = rwh & 0xffff, bbh = rwh >> 16;
      const unsigned int zmin_bits = __float_as_uint(s_rec[10][slot]);
      for (int y = warp; y < bbh; y += (NT / 32))
        for (int x = lane; x < bbw; x += 32) {
          const int xx = bxl + x, yy = byl + y;
          resolve_pixel<SOFT>(fc, fe, bfid, zmin_bits, persp, s_xf[xx], s_yf[yy], keys + (size_t)yy * p.W + xx,
                        prev ? prev + (size_t)yy * p.W + xx : nullptr, sm);
        }
    }
    n_big += (tid == 0) ? n_bigf - n_clipf : 0;
    __syncthreads();
  }
  if (p.counters) {
    if (n_straddle) atomicAdd((unsigned long long*)(p.counters + MVR_CNT_STRADDLE), (unsigned long long)n_straddle);
    if (n_big) atomicAdd((unsigned long long*)(p.counters + MVR_CNT_BIG_FACES), (unsigned long long)n_big);
  }
}

// ------------------------------------------------------------------------------------------------
// shading ([upstream] shading.py phong_shading, lighting.py diffuse/specular, blending.py hard_rgb_blend)
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// shade pass: one thread per pixel
// ------------------------------------------------------------------------------------------------
// grid: x = 32 x (8 PPT)-pixel tiles of the image, y = view m, z = object b.  EXACT: the caller wants zbuf / bary / dists.
// PPT pixels per thread (rows yi0 + 8 j): the keys -- the one operand that comes from DRAM -- of all of them are
// loaded before the first is shaded, so a thread pays the DRAM trip once instead of once per pixel; the dependent L2
// trips (face -> vertex records) of pixel j then overlap with those of the other warps only.
// DEPTH (hard depth, K = 1): the winning key's z -- the nearest fragment's depth, bit for bit -- or p.depth_bg into the
// (n,1,H,W) plane `images`, and pix_to_face; no vertex / normal / colour gathers, no shading, no 3-channel stores.
template <bool EXACT, int MINB, int PPT, bool VRGB, bool DEPTH = false>
__global__ void __launch_bounds__(MVR_THREADS, MINB) mesh_shade_kernel(const MeshParams p, int tiles_x) {
  pdl_enter();
  const int b = blockIdx.z, m = blockIdx.y, n = b * p.M + m;
  int ty, tx;
  tile_rc(blockIdx.x, tiles_x, ty, tx);
  const int xi = tx * 32 + (threadIdx.x & 31), yi0 = ty * (8 * PPT) + (threadIdx.x >> 5);
  const int HW = p.H * p.W;
  if (xi >= p.W || yi0 >= p.H) return;
  const int k = p.layer;
  unsigned long long* const kp0 = p.keys + (size_t)n * HW + (size_t)yi0 * p.W + xi;
  unsigned long long keys[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) keys[j] = (j == 0 || yi0 + 8 * j < p.H) ? __ldcs(kp0 + (size_t)(8 * j) * p.W) : MVR_EMPTY_KEY;
  const float xf = __ldg(p.tab + xi);
  const int f0 = p.face_off[b], voff = p.vert_off[b], V = p.vert_off[b + 1] - voff;
  const float4* pvn = p.pv + (size_t)p.M * voff + (size_t)m * V;
  const bool persp = p.flags & MVR_PERSPECTIVE_CORRECT;
  float bg[3] = {0.f, 0.f, 0.f};
  if (k == 0 && !DEPTH) { bg[0] = __ldg(p.bg_rgb); bg[1] = __ldg(p.bg_rgb + 1); bg[2] = __ldg(p.bg_rgb + 2); }
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const int yi = yi0 + 8 * j;
    if (j > 0 && yi >= p.H) break;
    const int pix = yi * p.W + xi;
    const unsigned long long key = keys[j];
    if (DEPTH) {
      int fid = -1;
      float z = p.depth_bg;
      if (key != MVR_EMPTY_KEY) {
        fid = (int)(unsigned int)(key & 0xffffffffull);
        // a face crossing the near plane: mesh_shade_clipped_kernel<false, true> owns the pixel (the face is read only then)
        if (may_clip(p.wsflags) && face_straddles(gather_face(pvn, __ldg(p.faces4 + f0 + fid)), p.z_clip)) continue;
        if (p.flags & MVR_WS_REARM_KEYS) p.keys[(size_t)n * HW + pix] = MVR_EMPTY_KEY;
        z = __uint_as_float((unsigned int)(key >> 32));
      }
      p.pix_to_face[(size_t)n * HW + pix] = fid;
      reinterpret_cast<float*>(p.images)[(size_t)n * HW + pix] = z;
      continue;
    }
    if (k + 1 < p.K) {            // hand the layer to the next peeling pass
      p.prev[(size_t)n * HW + pix] = key;
      p.keys[(size_t)n * HW + pix] = MVR_EMPTY_KEY;
    }
    int fid = -1;
    float w[3] = {-1.f, -1.f, -1.f}, bb[3] = {-1.f, -1.f, -1.f}, pz = -1.f, dd = -1.f;
    float out[3] = {bg[0], bg[1], bg[2]};
    if (key != MVR_EMPTY_KEY) {
      fid = (int)(unsigned int)(key & 0xffffffffull);
      const int4 fi = __ldg(p.faces4 + f0 + fid);
      // every gather of this pixel is issued before the first use (one round trip to L2 instead of three)
      const Face fc = gather_face(pvn, fi);
      // rasterized as clipped sub-triangles: mesh_shade_clipped_kernel owns this pixel (flag: see WSF_CLIP)
      if (may_clip(p.wsflags) && face_straddles(fc, p.z_clip)) continue;
      // last layer: leave the plane armed for the next forward (background keys are EMPTY already; clipped pixels are
      // re-armed by mesh_shade_clipped_kernel, which still needs their keys)
      if ((p.flags & MVR_WS_REARM_KEYS) && k + 1 == p.K) p.keys[(size_t)n * HW + pix] = MVR_EMPTY_KEY;
      float4 X0, X1, X2, N0, N1, N2, c0, c1, c2;
      if (k == 0) {
        gather_xn(p.xn8, voff + fi.x, X0, N0); gather_xn(p.xn8, voff + fi.y, X1, N1); gather_xn(p.xn8, voff + fi.z, X2, N2);
        if (VRGB) { c0 = __ldg(p.rgb4 + voff + fi.x); c1 = __ldg(p.rgb4 + voff + fi.y); c2 = __ldg(p.rgb4 + voff + fi.z); }
        else { c0 = c1 = c2 = make_float4(__ldg(p.obj_rgb), __ldg(p.obj_rgb + 1), __ldg(p.obj_rgb + 2), 0.f); }
      }
      const float yf = __ldg(p.tab + p.W + yi);
      const FaceEdges fe = face_edges(fc);
      if (EXACT && soft_mode(p).on()) {      // blurred rasterizer: (clipped) barycentrics and the SIGNED edge distance
        float bu[3];
        bool inside;
        raster_soft(fc, fe, persp, p.flags & MVR_CLIP_BARYCENTRIC, xf, yf, bu, bb, pz, dd, inside);
      } else if (EXACT) {
        // The barycentrics are recomputed with the SAME exact operation sequence as the scatter (from the same
        // projected vertices), so the fragments returned to the caller are the rasterizer's, bit for bit.
        raster_test(fc, fe, persp, xf, yf, w, bb, pz);
        if (p.dists) {
          const float e01 = point_line_dist2(xf, yf, fc.x0, fc.y0, fc.x1, fc.y1);
          const float e02 = point_line_dist2(xf, yf, fc.x0, fc.y0, fc.x2, fc.y2);
          const float e12 = point_line_dist2(xf, yf, fc.x1, fc.y1, fc.x2, fc.y2);
          dd = -fminf(fminf(e01, e02), e12);
        }
      } else {
        shading_barycentrics(fc, fe, persp, xf, yf, bb);
      }
      pz = __uint_as_float((unsigned int)(key >> 32));
      if (k == 0) {
        const ShadeCtx sc = load_shade_ctx(p.light, p.light_stride, p.Cc, n);
        phong_pixel<VRGB>(bb, X0, X1, X2, N0, N1, N2, c0, c1, c2, sc, out);
      }
    }
    const size_t po = ((size_t)n * HW + pix) * p.K + k;
    p.pix_to_face[po] = fid;
    if (EXACT) {
      if (p.zbuf) p.zbuf[po] = pz;
      if (p.dists) p.dists[po] = dd;
      if (p.bary) { p.bary[3 * po] = bb[0]; p.bary[3 * po + 1] = bb[1]; p.bary[3 * po + 2] = bb[2]; }
    }
    if (k == 0) store_rgb(p.images, p.flags & MVR_IMAGES_BF16, (size_t)n * 3 * HW + pix, (size_t)HW, out[0], out[1], out[2], p.onorm);
  }
}

}  // namespace mvr

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
using namespace mvr;

extern "C" size_t mvr_mesh_geometry_bytes(int64_t total_verts, int64_t total_faces) {
  if (total_verts < 0 || total_faces < 0) return 0;
  return geom_layout(total_verts, total_faces).total;
}

extern "C" int mvr_mesh_prepare(const float* verts, const void* faces, const int* vert_off, const int* face_off,
                                int B, int64_t total_verts, int64_t total_faces, int max_faces,
                                const float* vert_rgb, int flags, void* geometry, size_t geometry_bytes,
                                void* stream) {
  if (B < 0 || total_verts < 0 || total_faces < 0 || max_faces < 0) { set_error("mvr_mesh_prepare: negative size"); return -1; }
  if (total_verts > 0x7fffffffLL || total_faces > 0x7fffffffLL) { set_error("mvr_mesh_prepare: more than 2^31-1 packed verts/faces"); return -2; }
  const GeomLayout g = geom_layout(total_verts, total_faces);
  if (geometry_bytes < g.total) { set_error("mvr_mesh_prepare: geometry buffer too small (%zu < %zu)", geometry_bytes, g.total); return -3; }
  if (B == 0 || total_verts == 0) return 0;
  if (!verts || !vert_off || !face_off || !geometry || (total_faces > 0 && !faces)) { set_error("mvr_mesh_prepare: null pointer"); return -4; }
  if ((flags & MVR_RGB_PER_ELEMENT) && !vert_rgb) { set_error("mvr_mesh_prepare: MVR_RGB_PER_ELEMENT without vert_rgb"); return -5; }
  if ((flags & MVR_FACES_I64) && (flags & MVR_FACES_U16)) { set_error("mvr_mesh_prepare: MVR_FACES_I64 and MVR_FACES_U16 are exclusive"); return -7; }
  char* base = (char*)geometry;
  cudaStream_t st = (cudaStream_t)stream;
  float4* verts4 = (float4*)(base + g.verts4);
  float4* normals4 = (float4*)(base + g.normals4);
  float4* rgb4 = (float4*)(base + g.rgb4);
  int4* faces4 = (int4*)(base + g.faces4);
  double* nacc = (double*)(base + g.nacc);
  const int tb = 256;
  MVR_LAUNCH(geom_pack_verts_kernel, (unsigned)((total_verts + tb - 1) / tb), tb, 0, st, verts,
             (flags & MVR_RGB_PER_ELEMENT) ? vert_rgb : nullptr, total_verts, verts4, rgb4, nacc);
  if (total_faces > 0 && max_faces > 0) {
    dim3 grid((max_faces + tb - 1) / tb, B);
    if (flags & MVR_FACES_I64) MVR_LAUNCH_PDL(geom_pack_faces_kernel<long long>, grid, tb, 0, st, (const long long*)faces, vert_off, face_off, verts4, faces4, nacc);
    else if (flags & MVR_FACES_U16) MVR_LAUNCH_PDL(geom_pack_faces_kernel<unsigned short>, grid, tb, 0, st, (const unsigned short*)faces, vert_off, face_off, verts4, faces4, nacc);
    else MVR_LAUNCH_PDL(geom_pack_faces_kernel<int>, grid, tb, 0, st, (const int*)faces, vert_off, face_off, verts4, faces4, nacc);
  }
  MVR_LAUNCH_PDL(geom_finish_normals_kernel, (unsigned)((total_verts + tb - 1) / tb), tb, 0, st, nacc, total_verts, verts4, normals4,
                 (float4*)(base + g.xn8));
  return check_launch("mvr_mesh_prepare");
}

extern "C" int mvr_mesh_get_normals(const void* geometry, int64_t total_verts, int64_t total_faces, float* normals, void* stream) {
  if (total_verts <= 0) return 0;
  if (!geometry || !normals) { set_error("mvr_mesh_get_normals: null pointer"); return -1; }
  const GeomLayout g = geom_layout(total_verts, total_faces);
  MVR_LAUNCH(geom_get_normals_kernel, (unsigned)((total_verts + 255) / 256), 256, 0, (cudaStream_t)stream, (const float4*)((const char*)geometry + g.normals4), total_verts, normals);
  return check_launch("mvr_mesh_get_normals");
}

extern "C" int mvr_mesh_normals_backward(const void* geometry, const int* vert_off, const int* face_off, int B,
                                         int64_t total_verts, int64_t total_faces, int max_faces, float* grad_normals,
                                         float* grad_verts, void* stream) {
  if (B < 0 || total_verts < 0 || total_faces < 0 || max_faces < 0) { set_error("mvr_mesh_normals_backward: negative size"); return -1; }
  if (B == 0 || total_verts == 0) return 0;
  if (!geometry || !vert_off || !face_off || !grad_normals || !grad_verts) { set_error("mvr_mesh_normals_backward: null pointer"); return -2; }
  const GeomLayout g = geom_layout(total_verts, total_faces);
  const char* gb = (const char*)geometry;
  cudaStream_t st = (cudaStream_t)stream;
  const int tb = 256;
  MVR_LAUNCH(geom_normals_bwd_vertex_kernel, (unsigned)((total_verts + tb - 1) / tb), tb, 0, st, (const double*)(gb + g.nacc), total_verts, grad_normals);
  if (total_faces > 0 && max_faces > 0) {
    dim3 grid((max_faces + tb - 1) / tb, B);
    MVR_LAUNCH(geom_normals_bwd_face_kernel, grid, tb, 0, st, (const int4*)(gb + g.faces4), vert_off, face_off, (const float4*)(gb + g.verts4), (const float*)grad_normals, grad_verts);
  }
  return check_launch("mvr_mesh_normals_backward");
}

extern "C" size_t mvr_mesh_workspace_bytes(int B, int M, int H, int W, int K, int64_t total_verts, int64_t total_faces) {
  if (B < 0 || M < 0 || H <= 0 || W <= 0 || K < 1 || total_verts < 0 || total_faces < 0) return 0;
  return ws_layout(B, M, H, W, K, total_verts, total_faces).total;
}

// Threads (= faces per round) of a scatter CTA: 256 (4 CTAs per SM), or 128 (8 per SM) for large meshes -- twice as many
// independent CTAs to cover each other's two barriers per round: 706 -> 663 us at 100 k faces x 160 views (r3z), but 340 -> 358 us at
// 10 k faces x 384 views, where the rounds are too few to fill.
static int scatter_nt(int max_faces) { return max_faces > 32768 ? 128 : 256; }

// depth: mvr_mesh_depth_forward -- `images` is the (n,1,H,W) depth plane, K = 1, no shading inputs, no optional fragments
static int mesh_forward_impl(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                             int64_t total_verts, int64_t total_faces, int max_verts, int max_faces,
                             const float* R, const float* T, const float* Cc, const float* light,
                             int light_stride, const float* obj_rgb, const float* bg_rgb, float k00, float k11,
                             float z_clip, float blur_radius, int H, int W, int K, int flags, const float* out_mean_std, void* images,
                             int* pix_to_face, float* zbuf, float* bary, float* dists, int64_t* counters,
                             void* workspace, size_t workspace_bytes, void* stream, bool depth, float depth_bg) {
  int rc = check_mesh_common("mvr_mesh_forward", B, M, H, W, K, total_verts, total_faces, max_verts);
  if (rc) return rc;
  const int64_t N = (int64_t)B * M;
  if (counters && N == 0) {           // the call owns the counters: zeroed by mesh_project_kernel, in front of the kernels that count
    cudaError_t ce = cudaMemsetAsync(counters, 0, MVR_NUM_COUNTERS * sizeof(int64_t), (cudaStream_t)stream);
    if (ce != cudaSuccess) { set_error("mvr_mesh_forward: cudaMemsetAsync: %s", cudaGetErrorString(ce)); return (int)ce; }
  }
  if (N == 0) return 0;
  if (!geometry || !vert_off || !face_off || !R || !T || (!depth && (!Cc || !light || !bg_rgb)) || !images || !pix_to_face || !workspace) {
    set_error("mvr_mesh_forward: null pointer"); return -5;
  }
  if (!depth && !(flags & MVR_RGB_PER_ELEMENT) && !obj_rgb) { set_error("mvr_mesh_forward: obj_rgb is NULL and the geometry has no per-vertex colours"); return -6; }
  if (!out_norm_valid(out_mean_std)) { set_error("mvr_mesh_forward: out_mean_std needs std > 0"); return -9; }
  if (!(blur_radius >= 0.f)) { set_error("mvr_mesh_forward: blur_radius must be >= 0"); return -10; }
  const WsLayout w = ws_layout(B, M, H, W, K, total_verts, total_faces);
  if (workspace_bytes < w.total) { set_error("mvr_mesh_forward: workspace too small (%zu < %zu)", workspace_bytes, w.total); return -7; }
  const int chunks_per_view = max_faces > 0 ? (max_faces + FACES_PER_CTA - 1) / FACES_PER_CTA : 0;
  if (N * (int64_t)(chunks_per_view + 1) > 0x7fffffffLL) { set_error("mvr_mesh_forward: too many face chunks"); return -8; }
  const GeomLayout g = geom_layout(total_verts, total_faces);
  const char* gb = (const char*)geometry;
  char* wb = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  MeshParams p;
  p.verts4 = (const float4*)(gb + g.verts4); p.normals4 = (const float4*)(gb + g.normals4);
  p.rgb4 = (const float4*)(gb + g.rgb4); p.faces4 = (const int4*)(gb + g.faces4); p.xn8 = (const float4*)(gb + g.xn8);
  p.vert_off = vert_off; p.face_off = face_off;
  p.R = R; p.T = T; p.Cc = Cc; p.light = light; p.light_stride = light_stride;
  p.obj_rgb = obj_rgb; p.bg_rgb = bg_rgb;
  p.k00 = k00; p.k11 = k11; p.z_clip = z_clip;
  p.blur_radius = blur_radius > 0.f ? blur_radius : 0.f; p.blur_r = sqrtf(p.blur_radius);
  p.B = B; p.M = M; p.H = H; p.W = W; p.K = K; p.flags = flags;
  p.chunks_per_view = chunks_per_view; p.layer = 0;
  p.ndc_max = W > H ? (float)((W + H - 1) / H) : (float)((H + W - 1) / W);      // bound on |pixel-centre NDC| (>= aspect ratio)
  {
    const float rx = W > H ? 2.0f * (float)(W / H) : 2.0f;
    const float ry = H > W ? 2.0f * (float)(H / W) : 2.0f;
    p.jx_scale = (float)W / rx; p.jx_off = (0.5f * rx * (float)W - 0.5f * rx) / rx;
    p.jy_scale = (float)H / ry; p.jy_off = (0.5f * ry * (float)H - 0.5f * ry) / ry;
  }
  p.wcap = (flags & MVR_TEST_TINY_QUEUES) ? 40 : SC_QCAP;      // candidate queue of a round (scatter kernel)
  p.pv = (float4*)(wb + w.pv); p.tab = (float*)(wb + w.tab);
  p.keys = (unsigned long long*)(wb + w.keys); p.prev = (unsigned long long*)(wb + w.prev);
  p.images = images; p.pix_to_face = pix_to_face; p.zbuf = zbuf; p.bary = bary; p.dists = dists;
  p.counters = (long long*)counters;
  p.onorm = make_out_norm(out_mean_std);
  p.wsflags = (int*)(wb + w.flags);
  p.depth_bg = depth_bg;
  const size_t HW = (size_t)H * W;
  const bool soft_raster = p.blur_radius > 0.f || (flags & MVR_CLIP_BARYCENTRIC);
  // every key = EMPTY, and the workspace flags right in front of the plane armed (WSF_CLIP)
  const size_t plane_bytes = (flags & MVR_WS_KEYS_ARMED) ? 0 : (size_t)N * HW * 8;
  cudaError_t e = cudaMemsetAsync(wb + w.flags, 0xFF, (w.keys - w.flags) + plane_bytes, st);
  if (e != cudaSuccess) { set_error("mvr_mesh_forward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return (int)e; }
  rc = launch_project("mesh_project_kernel", g, w, geometry, vert_off, R, T, B, M, H, W, max_verts, k00, k11, z_clip, false, workspace, st, (long long*)counters);
  if (rc) return rc;
  const size_t tab_smem = ((size_t)W + H) * sizeof(float);
  const int tiles_x = (W + 31) / 32;
  const dim3 shade_grid((unsigned)(tiles_x * ((H + 7) / 8)), (unsigned)M, (unsigned)B);           // 1 pixel per thread
  const dim3 shade_fast_grid((unsigned)(tiles_x * ((H + 31) / 32)), (unsigned)M, (unsigned)B);     // 4 pixels per thread
  for (int k = 0; k < K; ++k) {
    p.layer = k;
    if (chunks_per_view > 0) {
      const dim3 scatter_grid((unsigned)chunks_per_view, (unsigned)M, (unsigned)B);
      if (soft_raster) MVR_LAUNCH_PDL((mesh_scatter_kernel<3, true>), scatter_grid, MVR_THREADS, tab_smem, st, p);
      else if (scatter_nt(max_faces) == 128) { MeshParams q = p; q.wcap = p.wcap < SC_QCAP ? p.wcap : SC_QCAP / 2; MVR_LAUNCH_PDL((mesh_scatter_kernel<8, false, 128>), scatter_grid, 128, tab_smem, st, q); }
      else MVR_LAUNCH_PDL((mesh_scatter_kernel<4, false>), scatter_grid, MVR_THREADS, tab_smem, st, p);
      rc = check_launch("mesh_scatter_kernel");
      if (rc) return rc;
    }
    const bool vrgb = flags & MVR_RGB_PER_ELEMENT;
    if (depth) MVR_LAUNCH_PDL((mesh_shade_kernel<false, 4, 4, false, true>), shade_fast_grid, MVR_THREADS, 0, st, p, tiles_x);
    else if (zbuf || bary || dists) {
      if (vrgb) MVR_LAUNCH_PDL((mesh_shade_kernel<true, 3, 1, true>), shade_grid, MVR_THREADS, 0, st, p, tiles_x);
      else MVR_LAUNCH_PDL((mesh_shade_kernel<true, 3, 1, false>), shade_grid, MVR_THREADS, 0, st, p, tiles_x);
    } else if (vrgb) MVR_LAUNCH_PDL((mesh_shade_kernel<false, 4, 4, true>), shade_fast_grid, MVR_THREADS, 0, st, p, tiles_x);
    else MVR_LAUNCH_PDL((mesh_shade_kernel<false, 4, 4, false>), shade_fast_grid, MVR_THREADS, 0, st, p, tiles_x);
    rc = check_launch("mesh_shade_kernel");
    if (rc) return rc;
    if (z_clip >= 0.f) {      // pixels won by a face crossing the near plane (none in MVTN's default configurations: the kernel exits at once)
      rc = launch_mesh_shade_clipped(p, (int)N, soft_raster, st, depth);
      if (rc) return rc;
    }
  }
  return 0;
}

extern "C" int mvr_mesh_forward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                int64_t total_verts, int64_t total_faces, int max_verts, int max_faces,
                                const float* R, const float* T, const float* Cc, const float* light,
                                int light_stride, const float* obj_rgb, const float* bg_rgb, float k00, float k11,
                                float z_clip, float blur_radius, int H, int W, int K, int flags, const float* out_mean_std, void* images,
                                int* pix_to_face, float* zbuf, float* bary, float* dists, int64_t* counters,
                                void* workspace, size_t workspace_bytes, void* stream) {
  return mesh_forward_impl(geometry, vert_off, face_off, B, M, total_verts, total_faces, max_verts, max_faces, R, T, Cc, light,
                           light_stride, obj_rgb, bg_rgb, k00, k11, z_clip, blur_radius, H, W, K, flags, out_mean_std, images,
                           pix_to_face, zbuf, bary, dists, counters, workspace, workspace_bytes, stream, false, 0.f);
}

extern "C" int mvr_mesh_depth_forward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                      int64_t total_verts, int64_t total_faces, int max_verts, int max_faces,
                                      const float* R, const float* T, float k00, float k11, float z_clip, float depth_background,
                                      int H, int W, int flags, float* depth, int* pix_to_face, int64_t* counters,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  if (flags & (MVR_IMAGES_BF16 | MVR_CLIP_BARYCENTRIC)) { set_error("mvr_mesh_depth_forward: the depth is fp32 from the hard rasterizer"); return -11; }
  return mesh_forward_impl(geometry, vert_off, face_off, B, M, total_verts, total_faces, max_verts, max_faces, R, T, nullptr, nullptr,
                           0, nullptr, nullptr, k00, k11, z_clip, 0.f, H, W, 1, flags & ~MVR_RGB_PER_ELEMENT, nullptr, depth, pix_to_face,
                           nullptr, nullptr, nullptr, counters, workspace, workspace_bytes, stream, true, depth_background);
}

