// mvr_points.cu -- point-cloud path of MVRenderer (renderer.py:116-151) for sm_100a.
//
//   forward : ONE pass whatever K (= points_per_pixel) is --
//               points_scatter_kernel -- one thread per (view, point): p = (X / dist) R + T is computed ONCE per
//                 view, the handful of pixel centres inside the point's radius are tested exactly
//                 (dist2 < r^2, IEEE fp32) and the 64-bit (z, point) key is inserted into the pixel's K sorted
//                 slots by a chain of 64-bit atomic mins: slot k keeps min(old, key) and the larger of the two
//                 moves on to slot k+1.  Every key but the k smallest passes slot k exactly once, so slot k ends
//                 up holding the (k+1)-th smallest (z, index) key whatever the order of arrival: the oracle's
//                 priority-queue result, deterministically.  K = 1 degenerates to a fire-and-forget RED.MIN.64;
//               points_resolve_kernel -- one thread per pixel: the pixel's K keys (one 32-byte sector for K = 4)
//                 -> idx / zbuf / dists2 of every layer, norm-weighted or alpha compositing, background, planar
//                 (n,3,H,W) rows, and one bit per pixel in a hit mask (the images are ~90 % background).
//   backward: points_backward_kernel -- one CTA per column of 8 32x32-pixel tiles: the hit-mask words of the tiles are
//             compacted into one dense list of covered pixels (warp scans + shared memory) and only those touch
//             idx / grad_images, with all threads busy: compositor backward -> d dist2 -> d ndc.xy ->
//             (dR, dT, d(1/dist)) reduced to one partial per CTA, summed in fixed order; optional
//             per-point / colour gradients via atomics.
#include <cooperative_groups.h>
#include <cstdlib>

#include "mvr_camera.cuh"

namespace mvr {

constexpr int PB_VALS = 13;            // dR 9, dT 3, d inv_dist 1

struct PointsParams {
  const float* points; const float* rgb;
  const float* R; const float* T; const float* inv_dist; const float* bg_rgb;
  float radius, r2_raster, r2_weight;
  int B, Np, M, H, W, K, flags, mask_words;
  unsigned long long* keys;      // (n, H*W, K): the K smallest (z, point) keys of every pixel, ascending
  const float* tab;              // pixel-centre NDC coordinates: xf[W] then yf[H]
  // tiled path (K in {1,2,4,8}): per-(view, point) projection + pixel window, per-(view, tile) point lists
  float4* pp; int2* pw; int* tile_cnt; int* tile_off; int* tile_cur; int* list;
  int tiles_x, tiles_y, ntiles, list_cap;
  int vec_bg;                    // W % 4 == 0 and 16-byte aligned images: the tile kernel paints the background 4 pixels per store
  void* images; int* idx; float* zbuf; float* dists2; unsigned int* hit_mask;
  OutNorm onorm;
};

__device__ __forceinline__ void project_point(const float* __restrict__ pts, int pi, float s, const Camera& cam,
                                              float& px, float& py, float& pz) {
  const float x = __ldg(pts + 3 * (size_t)pi) * s, y = __ldg(pts + 3 * (size_t)pi + 1) * s, z = __ldg(pts + 3 * (size_t)pi + 2) * s;
  world_to_view(cam, x, y, z, px, py, pz);
}

// per-view scale of the cloud (renderer.py:142 point_cloud.scale_(1 / dist)): the caller passes 1/dist, or dist itself
// with MVR_SCALE_IS_DIST -- then the reciprocal is the IEEE division torch's `1.0 / dist` performs, bit for bit, and the
// backward returns d/d dist instead of d/d (1/dist) (two elementwise launches and their autograd nodes less per step)
__device__ __forceinline__ float view_scale(const float* __restrict__ scale, int flags, int n) {
  const float v = __ldg(scale + n);
  return (flags & MVR_SCALE_IS_DIST) ? __fdiv_rn(1.0f, v) : v;
}

__global__ void pixel_table_kernel(float* __restrict__ tab, int H, int W) { fill_pixel_table(tab, H, W, threadIdx.x, blockDim.x); }

// insertion of one (z, point) key into the K ascending slots of a pixel (see the file header)
__device__ __forceinline__ void insert_key(unsigned long long* slot, unsigned long long key, int K) {
  if (K == 1) {
    if (key < __ldcg(slot)) atomicMin(slot, key);      // result unused: RED.MIN.64 resolved in L2
    return;
  }
  for (int k = 0; k < K; ++k) {
    // Deeper slots are first read: keys never grow, so key >= (possibly stale, i.e. larger) snapshot means the slot
    // keeps its value and `key` moves on unchanged -- a plain load instead of an atomic.  Slot 0 is hit directly:
    // most pixels of a point cloud receive a single fragment, and the load would double the L2 transactions.
    if (k > 0 && key >= __ldcg(slot + k)) continue;
    const unsigned long long old = atomicMin(slot + k, key);
    key = old > key ? old : key;                         // the displaced (or rejected) key goes one slot deeper
    if (key == MVR_EMPTY_KEY) break;
  }
}

// exclusive prefix sum of one int per thread over the CTA (MVR_THREADS threads); total returned to every thread.
// s_w: shared int[MVR_THREADS / 32 + 1].  Contains two block barriers.
__device__ __forceinline__ int block_exclusive_scan(int v, int* s_w, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  int base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < MVR_THREADS / 32; ++w) {
    const int x = s_w[w];
    base += w < warp ? x : 0;
    tot += x;
  }
  __syncthreads();
  total = tot;
  return base + inc - v;
}

constexpr int PS_CAP = 4096;      // (point, pixel) candidates queued per CTA; beyond that they are inserted in place

// grid: x = blocks of 256 points, y = view m, z = object b.
// Phase 1 (thread per point): project once, walk the few pixel centres around the point, queue the ones inside the
// radius.  Phase 2 (thread per queued fragment): the atomic-min chain, with every lane busy and its L2 round trips
// overlapped -- a point covers 1 to ~30 pixels depending on radius and resolution, so inserting from phase 1 would leave
// most lanes of a warp waiting on the slowest one.
__global__ void __launch_bounds__(MVR_THREADS) points_scatter_kernel(const PointsParams p) {
  __shared__ unsigned int s_cand[PS_CAP];       // local point << 24 | y << 12 | x
  __shared__ unsigned long long s_key[MVR_THREADS];
  __shared__ int s_w[MVR_THREADS / 32 + 1];
  const int b = blockIdx.z, n = b * p.M + blockIdx.y;
  const int tid = threadIdx.x;
  const int pi = blockIdx.x * MVR_THREADS + tid;
  const size_t HW = (size_t)p.H * p.W;
  unsigned long long* keys = p.keys + (size_t)n * HW * p.K;
  const float* tx = p.tab;
  const float* ty = p.tab + p.W;
  float px = 0.f, py = 0.f;
  int xl = 1, xh = 0, yl = 1, yh = 0, cnt = 0;
  unsigned long long key = MVR_EMPTY_KEY;
  if (pi < p.Np) {
    const Camera cam = load_camera(p.R, p.T, n);
    const float s = view_scale(p.inv_dist, p.flags, n);
    float pz;
    project_point(p.points + 3 * (size_t)b * p.Np, pi, s, cam, px, py, pz);
    if (!(pz < 0.f)) {
      key = make_key(pz, pi);
      // conservative search window for candidate pixel centres (the exact test is dist2 < r2 below)
      const float rr = p.radius * 1.0001f + 1e-7f;
      pixel_range(py - rr, py + rr, p.H, p.W, 0, p.H - 1, ty, yl, yh);
      pixel_range(px - rr, px + rr, p.W, p.H, 0, p.W - 1, tx, xl, xh);
      if (yl > yh || xl > xh) { xl = 1; xh = 0; yl = 1; yh = 0; }
      for (int yy = yl; yy <= yh; ++yy) {          // pass 1: count the pixel centres inside the radius
        const float dy = py - __ldg(ty + yy);
        for (int xx = xl; xx <= xh; ++xx) {
          const float dx = px - __ldg(tx + xx);
          cnt += (dx * dx + dy * dy < p.r2_raster) ? 1 : 0;
        }
      }
    }
  }
  s_key[tid] = key;
  int total;
  int at = block_exclusive_scan(cnt, s_w, total);      // queue slots without atomics (and in a deterministic order)
  if (cnt > 0) {
    for (int yy = yl; yy <= yh; ++yy) {            // pass 2: same tests, write the queue
      const float dy = py - __ldg(ty + yy);
      for (int xx = xl; xx <= xh; ++xx) {
        const float dx = px - __ldg(tx + xx);
        if (!(dx * dx + dy * dy < p.r2_raster)) continue;
        if (at < PS_CAP) s_cand[at] = ((unsigned int)tid << 24) | ((unsigned int)yy << 12) | (unsigned int)xx;
        else insert_key(keys + ((size_t)yy * p.W + xx) * p.K, key, p.K);
        ++at;
      }
    }
  }
  __syncthreads();
  const int nc = min(total, PS_CAP);
  for (int c = tid; c < nc; c += MVR_THREADS) {
    const unsigned int cd = s_cand[c];
    const int xx = cd & 4095, yy = (cd >> 12) & 4095;
    insert_key(keys + ((size_t)yy * p.W + xx) * p.K, s_key[cd >> 24], p.K);
  }
}

// A pixel no point covers: empty fragment slots and the background colour.
template <int KT>
__device__ __forceinline__ void store_background_pixel(const PointsParams& p, int n, int xi, int yi) {
  const int K = KT > 0 ? KT : p.K;
  const size_t HW = (size_t)p.H * p.W;
  const size_t pix = (size_t)yi * p.W + xi;
  const size_t po = ((size_t)n * HW + pix) * K;
  if (KT == 4) {
    *reinterpret_cast<int4*>(p.idx + po) = make_int4(-1, -1, -1, -1);
  } else {
    for (int l = 0; l < K; ++l) p.idx[po + l] = -1;
  }
  if (p.zbuf || p.dists2)
    for (int l = 0; l < K; ++l) {
      if (p.zbuf) p.zbuf[po + l] = -1.f;
      if (p.dists2) p.dists2[po + l] = -1.f;
    }
  store_rgb(p.images, p.flags & MVR_IMAGES_BF16, (size_t)n * 3 * HW + pix, HW, __ldg(p.bg_rgb), __ldg(p.bg_rgb + 1),
            __ldg(p.bg_rgb + 2), p.onorm);
}

// A covered pixel, its K ascending keys known (kreg: in registers, KT > 0; kp: their address, KT == 0): idx / zbuf /
// dists2 of every layer, norm-weighted or alpha compositing ([upstream] norm_weighted_sum / alpha_composite), planar
// image stores.
// PP: the view's projected points are in the workspace (tiled path: p.pp, written by the binning kernel with the very
// project_point below, so the values are the same bits) -- one 16-byte load instead of three loads and the transform.
template <int KT, bool PP = false>
__device__ __forceinline__ void composite_hit_pixel(const PointsParams& p, const unsigned long long* kreg,
                                                    const unsigned long long* kp, const Camera& cam, float s, int b, int n,
                                                    int xi, int yi) {
  const int K = KT > 0 ? KT : p.K;
  const size_t HW = (size_t)p.H * p.W;
  const size_t pix = (size_t)yi * p.W + xi;
  const size_t po = ((size_t)n * HW + pix) * K;
  const float xf = pix_to_ndc(p.W - 1 - xi, p.W, p.H);
  const float yf = pix_to_ndc(p.H - 1 - yi, p.H, p.W);
  const float* pts = p.points + 3 * (size_t)b * p.Np;
  const bool per_point_rgb = p.flags & MVR_RGB_PER_ELEMENT;
  const bool alpha_mode = p.flags & MVR_COMPOSITE_ALPHA;
  const float* feat = per_point_rgb ? p.rgb + 3 * (size_t)b * p.Np : p.rgb;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, aw = alpha_mode ? 1.f : 0.f;
  int ids[KT > 0 ? KT : 1];
  bool open = true;      // layers are contiguous: the first EMPTY key ends them
#pragma unroll
  for (int l = 0; l < K; ++l) {
    const unsigned long long key = KT > 0 ? kreg[KT > 0 ? l : 0] : kp[l];
    open = open && key != MVR_EMPTY_KEY;
    int q = -1;
    float z = -1.f, d2 = -1.f;
    if (open) {
      q = (int)(unsigned int)(key & 0xffffffffull);
      float px, py, pz;
      if (PP) { const float4 P = __ldg(p.pp + (size_t)n * p.Np + q); px = P.x; py = P.y; }
      else project_point(pts, q, s, cam, px, py, pz);
      const float dx = px - xf, dy = py - yf;
      d2 = dx * dx + dy * dy;
      z = __uint_as_float((unsigned int)(key >> 32));
      const float a = 1.f - d2 / p.r2_weight;
      const float* f = feat + (per_point_rgb ? 3 * (size_t)q : 0);
      const float f0 = __ldg(f), f1 = __ldg(f + 1), f2 = __ldg(f + 2);
      if (alpha_mode) {   // out += cum * alpha * f ; cum *= (1 - alpha)
        const float ca = aw * a;
        a0 += ca * f0; a1 += ca * f1; a2 += ca * f2;
        aw = aw * (1.f - a);
      } else {            // numerators and the alpha sum
        a0 += a * f0; a1 += a * f1; a2 += a * f2;
        aw += a;
      }
    }
    if (KT == 4) ids[KT > 0 ? l : 0] = q; else p.idx[po + l] = q;
    if (p.zbuf) p.zbuf[po + l] = z;
    if (p.dists2) p.dists2[po + l] = d2;
  }
  if (KT == 4) *reinterpret_cast<int4*>(p.idx + po) = make_int4(ids[0], ids[KT > 1 ? 1 : 0], ids[KT > 2 ? 2 : 0], ids[KT > 3 ? 3 : 0]);
  float o0 = a0, o1 = a1, o2 = a2;
  if (!alpha_mode) { const float t = fmaxf(aw, 1e-4f); o0 = a0 / t; o1 = a1 / t; o2 = a2 / t; }
  store_rgb(p.images, p.flags & MVR_IMAGES_BF16, (size_t)n * 3 * HW + pix, HW, o0, o1, o2, p.onorm);
}

// Everything that happens to ONE pixel once its K ascending keys are known: hit-mask bit (warp ballot: call with all
// 32 lanes, lane = x within a 32-pixel row word `mask_word`), then the background or the composited pixel.
template <int KT>
__device__ __forceinline__ void composite_and_store(const PointsParams& p, const unsigned long long* kreg,
                                                    const unsigned long long* kp, int b, int n, int xi, int yi,
                                                    int mask_word, bool inside) {
  const unsigned long long key0 = inside ? (KT > 0 ? kreg[0] : kp[0]) : MVR_EMPTY_KEY;
  const bool hit = key0 != MVR_EMPTY_KEY;      // first-layer hit decides foreground ([upstream] _add_background_color_to_images)
  if (p.hit_mask) {
    const unsigned int mword = __ballot_sync(0xffffffffu, hit);
    if ((threadIdx.x & 31) == 0 && yi < p.H) p.hit_mask[((size_t)n * p.H + yi) * p.mask_words + mask_word] = mword;
  }
  if (!inside) return;
  if (!hit) { store_background_pixel<KT>(p, n, xi, yi); return; }
  const Camera cam = load_camera(p.R, p.T, n);
  composite_hit_pixel<KT>(p, kreg, kp, cam, view_scale(p.inv_dist, p.flags, n), b, n, xi, yi);
}

// grid: x = 32x8-pixel tiles, y = view m, z = object b.  KT = K when K <= PK_MAX_REG (keys in registers), 0 = generic
template <int KT>
__global__ void __launch_bounds__(MVR_THREADS) points_resolve_kernel(const PointsParams p, int tiles_x) {
  const int b = blockIdx.z, n = b * p.M + blockIdx.y;
  const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
  const int xi = tx * 32 + (threadIdx.x & 31), yi = ty * 8 + (threadIdx.x >> 5);
  const int K = KT > 0 ? KT : p.K;
  const bool inside = xi < p.W && yi < p.H;
  const size_t HW = (size_t)p.H * p.W;
  const size_t pix = (size_t)yi * p.W + xi;
  const size_t po = ((size_t)n * HW + pix) * K;
  const unsigned long long* kp = p.keys + po;
  // ---- the pixel's keys: ascending, EMPTY-padded ----
  unsigned long long kreg[KT > 0 ? KT : 1];
  kreg[0] = MVR_EMPTY_KEY;
  if (inside) {
    if (KT == 0) {
    } else if (KT % 2 == 0) {
#pragma unroll
      for (int l = 0; l < KT; l += 2) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(kp + l);
        kreg[l] = v.x; kreg[l + 1] = v.y;
      }
    } else {
#pragma unroll
      for (int l = 0; l < KT; ++l) kreg[l] = kp[l];
    }
  }
  composite_and_store<KT>(p, kreg, kp, b, n, xi, yi, tx, inside);
}

// ------------------------------------------------------------------------------------------------
// tiled forward (K in {1, 2, 4, 8}): bin the points of every view into 32x32-pixel tiles, then ONE CTA per
// (view, tile) keeps the tile's K-slot key planes in shared memory, inserts its points with shared-memory atomics and
// writes idx / zbuf / dists2 / image / hit mask directly -- no global key plane, no memset, no global atomics.
// ------------------------------------------------------------------------------------------------
constexpr int PT_QCAP = 2048;      // (point, pixel) candidates queued per round

// grid: x = blocks of 256 points, y = view m, z = object b.  FILL = false: project, window, count per tile;
// FILL = true: append the point to the lists of the tiles its window touches.
template <bool FILL>
__global__ void __launch_bounds__(MVR_THREADS) points_bin_kernel(const PointsParams p) {
  const int b = blockIdx.z, n = b * p.M + blockIdx.y;
  const int pi = blockIdx.x * MVR_THREADS + threadIdx.x;
  if (pi >= p.Np) return;
  const size_t o = (size_t)n * p.Np + pi;
  int xl, xh, yl, yh;
  if (!FILL) {
    const Camera cam = load_camera(p.R, p.T, n);
    const float s = view_scale(p.inv_dist, p.flags, n);
    float px, py, pz;
    project_point(p.points + 3 * (size_t)b * p.Np, pi, s, cam, px, py, pz);
    xl = 1; xh = 0; yl = 1; yh = 0;                       // empty window
    if (!(pz < 0.f)) {
      // conservative search window for candidate pixel centres (the exact test is dist2 < r2 in the tile kernel)
      const float rr = p.radius * 1.0001f + 1e-7f;
      pixel_range(py - rr, py + rr, p.H, p.W, 0, p.H - 1, p.tab + p.W, yl, yh);
      if (yl <= yh) pixel_range(px - rr, px + rr, p.W, p.H, 0, p.W - 1, p.tab, xl, xh);
      if (yl > yh || xl > xh) { xl = 1; xh = 0; yl = 1; yh = 0; }
    }
    p.pp[o] = make_float4(px, py, pz, 0.f);
    p.pw[o] = make_int2(xl | (xh << 16), yl | (yh << 16));
  } else {
    const int2 w = p.pw[o];
    xl = w.x & 0xffff; xh = w.x >> 16; yl = w.y & 0xffff; yh = w.y >> 16;
  }
  if (xl > xh) return;
  int* cnt = (FILL ? p.tile_cur : p.tile_cnt) + (size_t)n * p.ntiles;
  for (int ty = yl >> 5; ty <= (yh >> 5); ++ty)
    for (int tx = xl >> 5; tx <= (xh >> 5); ++tx) {
      const int at = atomicAdd(cnt + ty * p.tiles_x + tx, 1);
      if (FILL && at < p.list_cap) p.list[(size_t)n * p.list_cap + at] = pi;      // at < list_cap by construction
    }
}

// one CTA per view: exclusive scan of the per-tile counts -> list offsets (tile_off) and fill cursors (tile_cur)
__global__ void __launch_bounds__(MVR_THREADS) points_bin_scan_kernel(const PointsParams p) {
  __shared__ int s_part[MVR_THREADS];
  const int n = blockIdx.x, tid = threadIdx.x;
  const int per = (p.ntiles + MVR_THREADS - 1) / MVR_THREADS;
  const int beg = min(tid * per, p.ntiles), end = min(beg + per, p.ntiles);
  const int* cnt = p.tile_cnt + (size_t)n * p.ntiles;
  int sum = 0;
  for (int t = beg; t < end; ++t) sum += cnt[t];
  s_part[tid] = sum;
  __syncthreads();
  if (tid == 0) {
    int acc = 0;
    for (int i = 0; i < MVR_THREADS; ++i) { const int v = s_part[i]; s_part[i] = acc; acc += v; }
  }
  __syncthreads();
  int acc = s_part[tid];
  for (int t = beg; t < end; ++t) {
    p.tile_off[(size_t)n * p.ntiles + t] = acc;
    p.tile_cur[(size_t)n * p.ntiles + t] = acc;
    acc += cnt[t];
  }
}

// The three binning launches (+ the pixel-table launch and the counter memset) as ONE kernel for clouds of up to
// BIN_FUSED_MAX_POINTS points and images of up to BIN_FUSED_MAX_TILES tiles: one CTA per view counts into shared
// memory, scans, and fills its lists.  At MVTN's sizes (2048 points, 49 tiles) the point path is launch-bound: five
// launches of 5-18 us of work each become one.  grid: x = view m, y = object b; dynamic smem: (W + H) floats.
constexpr int BIN_FUSED_MAX_TILES = 1024;
constexpr int BIN_FUSED_MAX_POINTS = 16384;
// A view is binned by a thread-block CLUSTER of `cs` CTAs (1 for small clouds: a plain launch; 4 above 4096 points): each CTA
// takes every cs-th 256-point slab of the cloud and counts into its own shared memory; after a cluster barrier every CTA reads
// the other CTAs' counters through distributed shared memory (DSMEM) to get, per tile, the total and the number of points the
// lower-ranked CTAs will write -- its private write cursor -- and fills its share of the lists.  At configs[4] (16384 points x
// 160 views) one CTA per view left the GPU at 13 % occupancy for 127 us: the cluster gives 4x the CTAs without a second
// launch or a global-memory hand-off.
__global__ void __launch_bounds__(MVR_THREADS) points_bin_kernel_fused(const PointsParams p, float* __restrict__ tab_out, int cs) {
  __shared__ int s_cnt[BIN_FUSED_MAX_TILES];
  __shared__ int s_cur[BIN_FUSED_MAX_TILES];
  __shared__ int s_w[MVR_THREADS / 32 + 1];
  extern __shared__ float s_ptab[];                          // xf[W], yf[H]
  namespace cg = cooperative_groups;
  const int rank = cs > 1 ? (int)cg::this_cluster().block_rank() : 0;
  const int b = blockIdx.y, n = b * p.M + (int)(blockIdx.x / cs), tid = threadIdx.x;
  fill_pixel_table(s_ptab, p.H, p.W, tid, MVR_THREADS);
  for (int t = tid; t < p.ntiles; t += MVR_THREADS) s_cnt[t] = 0;
  __syncthreads();
  if (n == 0 && rank == 0) for (int i = tid; i < p.W + p.H; i += MVR_THREADS) tab_out[i] = s_ptab[i];      // the tile / backward kernels read it
  const Camera cam = load_camera(p.R, p.T, n);
  const float s = view_scale(p.inv_dist, p.flags, n);
  const float rr = p.radius * 1.0001f + 1e-7f;               // conservative window (the exact test is dist2 < r2 in the tile kernel)
  const int pstep = MVR_THREADS * cs;
  for (int pi = rank * MVR_THREADS + tid; pi < p.Np; pi += pstep) {
    const size_t o = (size_t)n * p.Np + pi;
    float px, py, pz;
    project_point(p.points + 3 * (size_t)b * p.Np, pi, s, cam, px, py, pz);
    int xl = 1, xh = 0, yl = 1, yh = 0;                      // empty window
    if (!(pz < 0.f)) {
      pixel_range(py - rr, py + rr, p.H, p.W, 0, p.H - 1, s_ptab + p.W, yl, yh);
      if (yl <= yh) pixel_range(px - rr, px + rr, p.W, p.H, 0, p.W - 1, s_ptab, xl, xh);
      if (yl > yh || xl > xh) { xl = 1; xh = 0; yl = 1; yh = 0; }
    }
    p.pp[o] = make_float4(px, py, pz, 0.f);
    p.pw[o] = make_int2(xl | (xh << 16), yl | (yh << 16));
    if (xl > xh) continue;
    for (int ty = yl >> 5; ty <= (yh >> 5); ++ty)
      for (int tx = xl >> 5; tx <= (xh >> 5); ++tx) atomicAdd(&s_cnt[ty * p.tiles_x + tx], 1);
  }
  __syncthreads();
  // exclusive scan of the per-tile counts (of the whole cluster): `per` consecutive tiles per thread
  const int per = (p.ntiles + MVR_THREADS - 1) / MVR_THREADS;
  const int beg = min(tid * per, p.ntiles), end = min(beg + per, p.ntiles);
  if (cs > 1) {
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();                                          // every CTA of the view has finished counting
    // s_cur[t] := points the lower-ranked CTAs hold for tile t; s_w-free temporaries: totals go through registers below
    int sum = 0;
    for (int t = beg; t < end; ++t) {
      int tot = 0, before = 0;
      for (int c = 0; c < cs; ++c) {
        const int v = cluster.map_shared_rank(s_cnt, c)[t];  // DSMEM read
        tot += v;
        before += c < rank ? v : 0;
      }
      s_cur[t] = before;
      sum += tot;
    }
    int total;
    int acc = block_exclusive_scan(sum, s_w, total);
    for (int t = beg; t < end; ++t) {
      int tot = 0;
      for (int c = 0; c < cs; ++c) tot += cluster.map_shared_rank(s_cnt, c)[t];
      s_cur[t] += acc;                                       // this CTA's first slot in tile t's list
      if (rank == 0) {
        p.tile_off[(size_t)n * p.ntiles + t] = acc;
        p.tile_cur[(size_t)n * p.ntiles + t] = acc + tot;    // where the cluster's fill ends
      }
      acc += tot;
    }
    cluster.sync();                                          // nobody leaves (or reuses s_cnt) while its counters are being read
  } else {
    int sum = 0;
    for (int t = beg; t < end; ++t) sum += s_cnt[t];
    int total;
    int acc = block_exclusive_scan(sum, s_w, total);
    for (int t = beg; t < end; ++t) {
      const int c = s_cnt[t];
      s_cur[t] = acc;
      p.tile_off[(size_t)n * p.ntiles + t] = acc;
      p.tile_cur[(size_t)n * p.ntiles + t] = acc + c;        // where the fill below ends
      acc += c;
    }
    __syncthreads();
  }
  for (int pi = rank * MVR_THREADS + tid; pi < p.Np; pi += pstep) {
    const int2 w = p.pw[(size_t)n * p.Np + pi];              // this thread's own store
    const int xl = w.x & 0xffff, xh = w.x >> 16, yl = w.y & 0xffff, yh = w.y >> 16;
    if (xl > xh) continue;
    for (int ty = yl >> 5; ty <= (yh >> 5); ++ty)
      for (int tx = xl >> 5; tx <= (xh >> 5); ++tx) {
        const int at = atomicAdd(&s_cur[ty * p.tiles_x + tx], 1);
        if (at < p.list_cap) p.list[(size_t)n * p.list_cap + at] = pi;
      }
  }
}

// slot-major shared key planes: slot k of local pixel q at s_keys[k * 1024 + q]
template <int KT>
__device__ __forceinline__ void insert_key_smem(unsigned long long* s_keys, int q, unsigned long long key) {
#pragma unroll
  for (int k = 0; k < KT; ++k) {
    unsigned long long* slot = s_keys + k * 1024 + q;
    if (key >= *(volatile unsigned long long*)slot) continue;      // keys never grow: a stale snapshot is conservative
    const unsigned long long old = atomicMin(slot, key);
    key = old > key ? old : key;
    if (key == MVR_EMPTY_KEY) break;
  }
}

// grid: x = tile (ty * tiles_x + tx), y = view m, z = object b; dynamic shared memory: KT * 1024 keys
// MINB: minimum CTAs per SM for the register allocator; 0 = unconstrained
template <int KT, int MINB>
__global__ void __launch_bounds__(MVR_THREADS, MINB) points_tile_kernel(const PointsParams p) {
  pdl_enter();
  extern __shared__ unsigned long long s_keys[];              // [KT][1024]
  __shared__ unsigned int s_cand[PT_QCAP];                    // local point << 10 | local pixel
  __shared__ unsigned long long s_key[MVR_THREADS];
  __shared__ __align__(16) int s_ids[2][MVR_THREADS + 8];     // the tile's point list, a round per stage: TMA bulk-copy destinations
  __shared__ __align__(8) unsigned long long s_mbar[2];
  __shared__ int s_n;
  const int b = blockIdx.z, n = b * p.M + blockIdx.y, t = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int ty, tx;
  { ty = (int)__fdividef((float)t + 0.5f, (float)p.tiles_x); tx = t - ty * p.tiles_x; }
  const int x0 = tx * 32, y0 = ty * 32;
  const int beg = p.Np > 0 ? p.tile_off[(size_t)n * p.ntiles + t] : 0;
  const int end = p.Np > 0 ? min(p.tile_cur[(size_t)n * p.ntiles + t], p.list_cap) : 0;
  if (beg < end) {                                            // block-uniform
    // The tile's point list is CONTIGUOUS in global memory: it is staged by 1-D TMA bulk copies (cp.async.bulk + mbarrier),
    // round r + 1 in flight while round r is rasterized, and round 0 issued before the CTA initialises its key planes -- the
    // first of the three dependent trips a tile starts with (tile range -> list -> projected point) overlaps the set-up.
    const unsigned int mbar_a = (unsigned int)__cvta_generic_to_shared(&s_mbar[0]);
    const unsigned int ids_a = (unsigned int)__cvta_generic_to_shared(&s_ids[0][0]);
    const int* lst = p.list + (size_t)n * p.list_cap;
    auto issue_ids = [&](int r) {      // one thread: 16-byte aligned source (the list buffer is), size a multiple of 16
      const int start = beg + r * MVR_THREADS, cnt = min(MVR_THREADS, end - start);
      const size_t g = (size_t)n * p.list_cap + start, a0 = g & ~(size_t)3;
      const unsigned int bytes = (unsigned int)((((int)(g - a0) + cnt + 3) & ~3) * 4);
      const unsigned int mb = mbar_a + 8u * (r & 1);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       ids_a + 4u * (MVR_THREADS + 8) * (r & 1)),
                   "l"(p.list + a0), "r"(bytes), "r"(mb)
                   : "memory");
    };
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_a) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_a + 8u) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      issue_ids(0);
      s_n = 0;
    }
    (void)lst;
    for (int i = tid; i < KT * 1024; i += MVR_THREADS) s_keys[i] = MVR_EMPTY_KEY;
    __syncthreads();
    const float* tabx = p.tab;
    const float* taby = p.tab + p.W;
    int round = 0;
    for (int base = beg; base < end; base += MVR_THREADS, ++round) {
      // phase 1: thread per point -- pixel centres of the window (clipped to this tile) inside the radius go to the
      // queue (one shared atomic per hit: measured faster here than count + block scan + second pass)
      if (tid == 0 && base + MVR_THREADS < end) issue_ids(round + 1);      // (its stage was released by the barrier that ended round - 1)
      {
        const unsigned int mb = mbar_a + 8u * (round & 1), parity = (unsigned int)((round >> 1) & 1);
        asm volatile(
            "{\n.reg .pred p;\nWAITP_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONEP_%=;\nbra WAITP_%=;\nDONEP_%=:\n}\n" ::"r"(mb),
            "r"(parity)
            : "memory");
      }
      const int i = base + tid;
      if (i < end) {
        const int pi = s_ids[round & 1][(int)(((size_t)n * p.list_cap + base) & 3) + tid];
        const size_t o = (size_t)n * p.Np + pi;
        const float4 P = p.pp[o];
        const int2 w = p.pw[o];
        const int xl = max(w.x & 0xffff, x0), xh = min(w.x >> 16, x0 + 31);
        const int yl = max(w.y & 0xffff, y0), yh = min(w.y >> 16, y0 + 31);
        const unsigned long long key = make_key(P.z, pi);
        s_key[tid] = key;
        for (int yy = yl; yy <= yh; ++yy) {
          const float dy = P.y - __ldg(taby + yy);
          for (int xx = xl; xx <= xh; ++xx) {
            const float dx = P.x - __ldg(tabx + xx);
            const float d2 = dx * dx + dy * dy;
            if (!(d2 < p.r2_raster)) continue;
            const int q = ((yy - y0) << 5) | (xx - x0);
            const int at = atomicAdd(&s_n, 1);
            if (at < PT_QCAP) s_cand[at] = ((unsigned int)tid << 10) | (unsigned int)q;
            else insert_key_smem<KT>(s_keys, q, key);          // queue full: insert in place
          }
        }
      }
      __syncthreads();
      // phase 2: thread per queued fragment -- all lanes busy in the atomic chain
      const int nc = min(s_n, PT_QCAP);
      for (int c = tid; c < nc; c += MVR_THREADS) {
        const unsigned int cd = s_cand[c];
        insert_key_smem<KT>(s_keys, cd & 1023, s_key[cd >> 10]);
      }
      __syncthreads();
      if (tid == 0) s_n = 0;
      __syncthreads();
    }
  }
  // resolve.  The images are sparse (~10 % of the pixels are covered) and a covered pixel costs ~10x a background one,
  // so the two are separated: pass 1 -- thread (lane, warp) owns pixels (x0 + lane, y0 + warp + 8 j) -- writes the hit
  // mask and the background pixels (full coalesced rows) and compacts the covered pixels into a list in shared memory;
  // pass 2 walks that list with every lane busy.
  unsigned short* s_hits = reinterpret_cast<unsigned short*>(s_cand);      // the candidate queue is free by now
  const bool have = beg < end;
  if (tid == 0) s_n = 0;
  __syncthreads();
  {
    // per-view bases and the (normalised) background colour once per thread: the loop body is then 32-bit index
    // arithmetic and stores
    const size_t HW = (size_t)p.H * p.W;
    const size_t frag_o = (size_t)n * HW * KT;      // (the zbuf / dists2 pointers are formed only where a caller asked for them)
    int* idx_v = p.idx + frag_o;
    unsigned int* mask_v = p.hit_mask ? p.hit_mask + (size_t)n * p.H * p.mask_words + tx : nullptr;
    const bool bf16 = p.flags & MVR_IMAGES_BF16;
    const bool sparse_idx = (p.flags & MVR_IDX_SPARSE) && mask_v;
    float* img_f = reinterpret_cast<float*>(p.images) + (size_t)n * 3 * HW;
    __nv_bfloat16* img_h = reinterpret_cast<__nv_bfloat16*>(p.images) + (size_t)n * 3 * HW;
    float g0 = __ldg(p.bg_rgb), g1 = __ldg(p.bg_rgb + 1), g2 = __ldg(p.bg_rgb + 2);
    if (p.onorm.on) { g0 = (g0 - p.onorm.m0) * p.onorm.s0; g1 = (g1 - p.onorm.m1) * p.onorm.s1; g2 = (g2 - p.onorm.m2) * p.onorm.s2; }
    const __nv_bfloat16 h0 = __float2bfloat16_rn(g0), h1 = __float2bfloat16_rn(g1), h2 = __float2bfloat16_rn(g2);
    const int hw = (int)HW, xi = x0 + lane;
    if (p.vec_bg) {
      // the background colour of the WHOLE tile first, four pixels per store (thread = row tid / 8, pixels 4 (tid % 8) ..+3):
      // 3 stores per thread instead of 12; the covered pixels are overwritten by pass 2, behind the barrier below
      const int yv = y0 + (tid >> 3), xv = x0 + ((tid & 7) << 2);
      if (yv < p.H && xv < p.W) {
        const int pv = yv * p.W + xv;
        if (bf16) {
          const unsigned int u0 = __bfloat16_as_ushort(h0), u1 = __bfloat16_as_ushort(h1), u2 = __bfloat16_as_ushort(h2);
          *reinterpret_cast<uint2*>(img_h + pv) = make_uint2(u0 | (u0 << 16), u0 | (u0 << 16));
          *reinterpret_cast<uint2*>(img_h + pv + hw) = make_uint2(u1 | (u1 << 16), u1 | (u1 << 16));
          *reinterpret_cast<uint2*>(img_h + pv + 2 * hw) = make_uint2(u2 | (u2 << 16), u2 | (u2 << 16));
        } else {
          *reinterpret_cast<float4*>(img_f + pv) = make_float4(g0, g0, g0, g0);
          *reinterpret_cast<float4*>(img_f + pv + hw) = make_float4(g1, g1, g1, g1);
          *reinterpret_cast<float4*>(img_f + pv + 2 * hw) = make_float4(g2, g2, g2, g2);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int row = warp + 8 * j, yi = y0 + row;
      const bool inside = xi < p.W && yi < p.H;
      const bool hit = inside && have && s_keys[(row << 5) + lane] != MVR_EMPTY_KEY;      // slot 0 decides foreground
      const unsigned int mword = __ballot_sync(0xffffffffu, hit);
      if (lane == 0 && mask_v && yi < p.H) mask_v[yi * p.mask_words] = mword;
      if (mword) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_n, __popc(mword));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (hit) s_hits[base + __popc(mword & ((1u << lane) - 1u))] = (unsigned short)((row << 5) | lane);
      }
      if (inside && !hit) {                              // background pixel: empty fragment slots + background colour
        const int pix = yi * p.W + xi;
        if (sparse_idx) {
          // MVR_IDX_SPARSE: the hit mask already says "empty"; 4 K bytes per background pixel (~90 % of the image) stay unwritten
        } else if (KT == 4) {
          *reinterpret_cast<int4*>(idx_v + 4 * pix) = make_int4(-1, -1, -1, -1);
        } else if (KT == 2) {
          *reinterpret_cast<int2*>(idx_v + 2 * pix) = make_int2(-1, -1);
        } else {
#pragma unroll
          for (int l = 0; l < KT; ++l) idx_v[KT * pix + l] = -1;
        }
        if (p.zbuf) {
#pragma unroll
          for (int l = 0; l < KT; ++l) p.zbuf[frag_o + KT * pix + l] = -1.f;
        }
        if (p.dists2) {
#pragma unroll
          for (int l = 0; l < KT; ++l) p.dists2[frag_o + KT * pix + l] = -1.f;
        }
        if (!p.vec_bg) {
          if (bf16) { img_h[pix] = h0; img_h[pix + hw] = h1; img_h[pix + 2 * hw] = h2; }
          else { img_f[pix] = g0; img_f[pix + hw] = g1; img_f[pix + 2 * hw] = g2; }
        }
      }
    }
  }
  __syncthreads();
  const int nhit = s_n;
  if (nhit > 0) {
    const Camera cam = load_camera(p.R, p.T, n);
    const float s = view_scale(p.inv_dist, p.flags, n);
    for (int i = tid; i < nhit; i += MVR_THREADS) {
      const int q = s_hits[i];
      unsigned long long kreg[KT];
#pragma unroll
      for (int k = 0; k < KT; ++k) kreg[k] = s_keys[k * 1024 + q];
      composite_hit_pixel<KT, true>(p, kreg, nullptr, cam, s, b, n, x0 + (q & 31), y0 + (q >> 5));
    }
  }
}

// ------------------------------------------------------------------------------------------------
struct PointsBwdParams {
  const float* points; const float* rgb;
  const float* R; const float* T; const float* inv_dist;
  float r2_weight;
  int B, Np, M, H, W, K, flags, tiles_x, tiles_y, ctas_per_view, mask_words;
  const int* idx; const void* grad_images; const unsigned int* hit_mask;
  float* partials;        // (N, ctas_per_view, 16): one per 32x32 tile
  float* grad_points; float* grad_rgb;
  OutNorm onorm;
};

// (dR, dT, d scale) contributions of one fragment layer whose d out / d alpha is `ga`
template <bool GU>      // GU: the gradient of the single point colour is wanted (it rides in acc[13..15])
__device__ __forceinline__ void points_backward_layer(const PointsBwdParams& p, const Camera& cam, float s, float inv_r2, int b, int pid,
                                                      bool per_point_rgb, float X0, float X1, float X2, float dx, float dy, float ga, float gf,
                                                      float g0, float g1, float g2, float (&acc)[16]) {
  const float gd2 = -ga * inv_r2;
  const float gpx = 2.f * gd2 * dx, gpy = 2.f * gd2 * dy;
  const float Xs0 = X0 * s, Xs1 = X1 * s, Xs2 = X2 * s;
  acc[0] = fmaf(Xs0, gpx, acc[0]); acc[1] = fmaf(Xs0, gpy, acc[1]);
  acc[3] = fmaf(Xs1, gpx, acc[3]); acc[4] = fmaf(Xs1, gpy, acc[4]);
  acc[6] = fmaf(Xs2, gpx, acc[6]); acc[7] = fmaf(Xs2, gpy, acc[7]);
  acc[9] += gpx; acc[10] += gpy;
  const float gx0 = cam.r[0] * gpx + cam.r[1] * gpy, gx1 = cam.r[3] * gpx + cam.r[4] * gpy, gx2 = cam.r[6] * gpx + cam.r[7] * gpy;
  acc[12] += gx0 * X0 + gx1 * X1 + gx2 * X2;
  if (p.grad_points) {
    float* o = p.grad_points + 3 * ((size_t)b * p.Np + pid);
    atomicAdd(o, gx0 * s); atomicAdd(o + 1, gx1 * s); atomicAdd(o + 2, gx2 * s);
  }
  if (p.grad_rgb) {
    if (per_point_rgb) {
      float* o = p.grad_rgb + 3 * ((size_t)b * p.Np + pid);
      atomicAdd(o, g0 * gf); atomicAdd(o + 1, g1 * gf); atomicAdd(o + 2, g2 * gf);
    } else if (GU) {
      // ONE colour for every point: its gradient is a sum over every fragment of the batch.  It rides in the three spare slots
      // of the per-thread partials (-> one partial per CTA -> one atomicAdd per view in the reduce kernel) instead of three
      // atomics per fragment on the same three words (serialised in L2, and an fp32 sum of ~10^5 terms in arrival order)
      acc[13] = fmaf(g0, gf, acc[13]); acc[14] = fmaf(g1, gf, acc[14]); acc[15] = fmaf(g2, gf, acc[15]);
    }
  }
}

// grid: x = groups of `nw` (= 8) vertically adjacent 32x32-pixel tiles, y = view m, z = object b.
// The images are sparse (~10 % of the pixels are covered) and unevenly so: a tile holds anything from 0 to 1024 covered
// pixels.  Each warp COMPACTS the covered pixels of one tile -- lane r owns row r: one hit-mask word, its set bits go to a
// list in shared memory at the exclusive prefix of the per-row counts -- and the CTA then walks the JOINT list of its tiles
// with every thread busy, whichever tile the pixels came from (one warp per tile left the warps of the dense tiles running
// alone at 16 % occupancy).  Per covered pixel the chain idx -> point -> weights is a string of dependent loads, so (i) the
// pixel's K point ids arrive as ONE vector load and its cotangent as raw bits, both fetched one iteration ahead, and (ii) for
// KT in {1, 2, 4} the K layers (point, offset, alpha) stay in registers between the compositor-total pass and the gradient
// pass instead of being re-read and re-projected.  KT = 0 serves any other K with the layers re-read.
template <int KT, bool VRGB, bool GU>
__global__ void __launch_bounds__(MVR_THREADS) points_backward_kernel(const PointsBwdParams p) {
  __shared__ unsigned short s_list[8 * 1024];     // warp << 10 | row << 5 | x of every covered pixel of the CTA's tiles
  __shared__ int s_wtot[8];
  __shared__ float s_part[8][16];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.z, n = b * p.M + blockIdx.y;
  const int nw = blockDim.x >> 5;                    // warps (= tiles) per CTA (8; MVR_PBWD_WPC for profiling)
  const int tgy = blockIdx.x / p.tiles_x, txb = blockIdx.x - tgy * p.tiles_x;
  const int tyb = tgy * nw + warp;                   // the tile row this warp compacts
  const bool alpha_mode = p.flags & MVR_COMPOSITE_ALPHA;
  const bool bf16 = p.flags & MVR_IMAGES_BF16;
  const float* pts = p.points + 3 * (size_t)b * p.Np;
  const float* feat = VRGB ? p.rgb + 3 * (size_t)b * p.Np : p.rgb;
  const size_t plane = (size_t)p.H * p.W;
  // ---- covered pixels of row (tile row * 32 + lane) ----
  unsigned int word = 0u;
  if (tyb < p.tiles_y) {                             // warp-uniform
    const int yi = tyb * 32 + lane;
    if (p.hit_mask) {
      if (yi < p.H) word = __ldg(p.hit_mask + ((size_t)n * p.H + yi) * p.mask_words + txb);
    } else {                                         // no mask: first-layer idx >= 0, one coalesced row per step
      const int xi = txb * 32 + lane;
      for (int r = 0; r < 32; ++r) {
        const int yr = tyb * 32 + r;
        const bool h = yr < p.H && xi < p.W && __ldg(p.idx + ((size_t)n * plane + (size_t)yr * p.W + xi) * p.K) >= 0;
        const unsigned int wr = __ballot_sync(0xffffffffu, h);
        if (lane == r) word = wr;
      }
    }
  }
  const int cnt = __popc(word);
  int pre = cnt;                                     // inclusive warp scan of the per-row counts
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, pre, o);
    if (lane >= o) pre += v;
  }
  if (lane == 31) s_wtot[warp] = pre;
  __syncthreads();
  int base = 0, total = 0;
  for (int w = 0; w < nw; ++w) { const int c = s_wtot[w]; if (w < warp) base += c; total += c; }
  float* out = p.partials + ((size_t)n * p.ctas_per_view + blockIdx.x) * 16;      // one partial per CTA
  if (total == 0) {                                  // background only (block-uniform)
    if (tid < 16) out[tid] = 0.f;
    return;
  }
  {
    int at = base + pre - cnt;
    unsigned int wv = word;
    while (wv) {
      const int x = __ffs(wv) - 1;
      wv &= wv - 1u;
      s_list[at++] = (unsigned short)((warp << 10) | (lane << 5) | x);
    }
  }
  __syncthreads();
  float acc[16];                                      // PB_VALS camera values + [13..15]: gradient of the single point colour
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  const Camera cam = load_camera(p.R, p.T, n);
  const float s = view_scale(p.inv_dist, p.flags, n);
  const float inv_r2 = 1.f / p.r2_weight;
  float uf0 = 0.f, uf1 = 0.f, uf2 = 0.f;             // the one colour of all points (!VRGB)
  if (!VRGB) { uf0 = __ldg(feat); uf1 = __ldg(feat + 1); uf2 = __ldg(feat + 2); }
  constexpr int KR = KT > 0 ? KT : 1;
  const int step = blockDim.x;
  auto pixel_of = [&](int i, int& xi, int& yi) {
    const int code = s_list[i];
    yi = (tgy * nw + (code >> 10)) * 32 + ((code >> 5) & 31); xi = txb * 32 + (code & 31);
  };
  auto fetch = [&](int i, int (&pid)[KR], GradRaw& gr) {
    int xi, yi; pixel_of(i, xi, yi);
    const size_t pix = ((size_t)n * p.H + yi) * p.W + xi;
    if (KT == 4) { const int4 v = __ldg(reinterpret_cast<const int4*>(p.idx) + pix); pid[0] = v.x; pid[1 % KR] = v.y; pid[2 % KR] = v.z; pid[3 % KR] = v.w; }
    else if (KT == 2) { const int2 v = __ldg(reinterpret_cast<const int2*>(p.idx) + pix); pid[0] = v.x; pid[1 % KR] = v.y; }
    else if (KT == 1) pid[0] = __ldg(p.idx + pix);
    gr = load_grad_raw(p.grad_images, bf16, ((size_t)n * 3 * p.H + yi) * p.W + xi, plane);
  };
  int pid_n[KR] = {}; GradRaw gr_n = {0u, 0u, 0u};
  if (tid < total) fetch(tid, pid_n, gr_n);
  for (int it = tid; it < total; it += step) {
    int pid[KR];
#pragma unroll
    for (int k = 0; k < KR; ++k) pid[k] = pid_n[k];
    const GradRaw gr = gr_n;
    int xi, yi; pixel_of(it, xi, yi);
    if (it + step < total) fetch(it + step, pid_n, gr_n);
    float g0, g1, g2;
    grad_from_raw(gr, bf16, p.onorm, g0, g1, g2);
    if (g0 == 0.f && g1 == 0.f && g2 == 0.f) continue;
    const float xf = pix_to_ndc(p.W - 1 - xi, p.W, p.H), yf = pix_to_ndc(p.H - 1 - yi, p.H, p.W);
    if (KT > 0) {
      // ---- the K layers in registers: all point loads issued together, one projection per layer ----
      int nk = 0;
#pragma unroll
      for (int k = 0; k < KR; ++k) if (nk == k && pid[k] >= 0) nk = k + 1;      // the filled slots are a prefix
      float X[KR][3], f[KR][3], a[KR], dx[KR], dy[KR];
#pragma unroll
      for (int k = 0; k < KR; ++k) {
        const size_t q = k < nk ? (size_t)pid[k] : 0;      // (slot 0 is filled: the pixel is covered)
        X[k][0] = __ldg(pts + 3 * q); X[k][1] = __ldg(pts + 3 * q + 1); X[k][2] = __ldg(pts + 3 * q + 2);
        if (VRGB) { f[k][0] = __ldg(feat + 3 * q); f[k][1] = __ldg(feat + 3 * q + 1); f[k][2] = __ldg(feat + 3 * q + 2); }
        else { f[k][0] = uf0; f[k][1] = uf1; f[k][2] = uf2; }
      }
      float t_alpha = 0.f, tf0 = 0.f, tf1 = 0.f, tf2 = 0.f;   // norm: sum a, sum a f ; alpha: out_c
      {
        float cum = 1.f;
#pragma unroll
        for (int k = 0; k < KR; ++k) {
          float px, py, pz; world_to_view(cam, X[k][0] * s, X[k][1] * s, X[k][2] * s, px, py, pz);
          dx[k] = px - xf; dy[k] = py - yf;
          a[k] = 1.f - (dx[k] * dx[k] + dy[k] * dy[k]) / p.r2_weight;   // exactly the forward's alpha: it is clamped at 1e-4 below
          if (k < nk) {
            const float wgt = alpha_mode ? cum * a[k] : a[k];
            tf0 = fmaf(wgt, f[k][0], tf0); tf1 = fmaf(wgt, f[k][1], tf1); tf2 = fmaf(wgt, f[k][2], tf2);
            t_alpha += a[k]; cum *= (1.f - a[k]);
          }
        }
      }
      const float t = fmaxf(t_alpha, 1e-4f);
      float cum = 1.f, pre0 = 0.f, pre1 = 0.f, pre2 = 0.f;
#pragma unroll
      for (int k = 0; k < KR; ++k) {
        if (k < nk) {
          float ga, gf;   // d/d alpha_k ; d/d f_k (per unit grad_out, same for all channels)
          if (alpha_mode) {
            // out_c = sum_j f_jc cum_j a_j ;  d/da_k = f_kc cum_k - (sum_{j>k} f_jc cum_j a_j) / (1 - a_k + 1e-9)
            const float w = cum * a[k];
            pre0 = fmaf(w, f[k][0], pre0); pre1 = fmaf(w, f[k][1], pre1); pre2 = fmaf(w, f[k][2], pre2);
            const float inv1m = 1.f / (1.f - a[k] + 1e-9f);
            ga = g0 * (f[k][0] * cum - (tf0 - pre0) * inv1m) + g1 * (f[k][1] * cum - (tf1 - pre1) * inv1m) + g2 * (f[k][2] * cum - (tf2 - pre2) * inv1m);
            gf = w;
            cum *= (1.f - a[k]);
          } else {
            const float it2 = 1.f / (t * t);
            ga = (g0 * (t * f[k][0] - tf0) + g1 * (t * f[k][1] - tf1) + g2 * (t * f[k][2] - tf2)) * it2;
            gf = a[k] / t;
          }
          points_backward_layer<GU>(p, cam, s, inv_r2, b, pid[k], VRGB, X[k][0], X[k][1], X[k][2], dx[k], dy[k], ga, gf, g0, g1, g2, acc);
        }
      }
    } else {
      // ---- any K: the layers are re-read (L1) and re-projected by the second pass ----
      const int* ip = p.idx + (((size_t)n * p.H + yi) * p.W + xi) * p.K;
      float t_alpha = 0.f, tf0 = 0.f, tf1 = 0.f, tf2 = 0.f;
      {
        float cum = 1.f;
        for (int k = 0; k < p.K; ++k) {
          const int q = __ldg(ip + k);
          if (q < 0) break;
          float px, py, pz; project_point(pts, q, s, cam, px, py, pz);
          const float ddx = px - xf, ddy = py - yf;
          const float al = 1.f - (ddx * ddx + ddy * ddy) / p.r2_weight;
          const float* ff = feat + (VRGB ? 3 * (size_t)q : 0);
          const float wgt = alpha_mode ? cum * al : al;
          tf0 = fmaf(wgt, __ldg(ff), tf0); tf1 = fmaf(wgt, __ldg(ff + 1), tf1); tf2 = fmaf(wgt, __ldg(ff + 2), tf2);
          t_alpha += al; cum *= (1.f - al);
        }
      }
      const float t = fmaxf(t_alpha, 1e-4f);
      float cum = 1.f, pre0 = 0.f, pre1 = 0.f, pre2 = 0.f;
      for (int k = 0; k < p.K; ++k) {
        const int q = __ldg(ip + k);
        if (q < 0) break;
        const float X0 = __ldg(pts + 3 * (size_t)q), X1 = __ldg(pts + 3 * (size_t)q + 1), X2 = __ldg(pts + 3 * (size_t)q + 2);
        float px, py, pz; world_to_view(cam, X0 * s, X1 * s, X2 * s, px, py, pz);
        const float ddx = px - xf, ddy = py - yf;
        const float al = 1.f - (ddx * ddx + ddy * ddy) / p.r2_weight;
        const float* ff = feat + (VRGB ? 3 * (size_t)q : 0);
        const float f0 = __ldg(ff), f1 = __ldg(ff + 1), f2 = __ldg(ff + 2);
        float ga, gf;
        if (alpha_mode) {
          const float w = cum * al;
          pre0 = fmaf(w, f0, pre0); pre1 = fmaf(w, f1, pre1); pre2 = fmaf(w, f2, pre2);
          const float inv1m = 1.f / (1.f - al + 1e-9f);
          ga = g0 * (f0 * cum - (tf0 - pre0) * inv1m) + g1 * (f1 * cum - (tf1 - pre1) * inv1m) + g2 * (f2 * cum - (tf2 - pre2) * inv1m);
          gf = w;
          cum *= (1.f - al);
        } else {
          const float it2 = 1.f / (t * t);
          ga = (g0 * (t * f0 - tf0) + g1 * (t * f1 - tf1) + g2 * (t * f2 - tf2)) * it2;
          gf = al / t;
        }
        points_backward_layer<GU>(p, cam, s, inv_r2, b, q, VRGB, X0, X1, X2, ddx, ddy, ga, gf, g0, g1, g2, acc);
      }
    }
  }
  // one partial per CTA: warp totals, then the warps in fixed order; the reduce kernel sums the CTAs in fixed order
  const float mine = warp_sum16_transposed(acc);      // lanes 2i, 2i+1: total of value i
  if (!(lane & 1)) s_part[warp][lane >> 1] = mine;
  __syncthreads();
  if (tid < 16) {
    float v = 0.f;
    for (int w = 0; w < nw; ++w) v += s_part[w][tid];
    out[tid] = v;
  }
}

// grad_rgb_uniform: the (3,) gradient of the single point colour, or NULL (per-point colours / not wanted)
__global__ void points_backward_reduce_kernel(const float* __restrict__ partials, int N, int n_parts,
                                              float* __restrict__ gR, float* __restrict__ gT, float* __restrict__ gs,
                                              const float* __restrict__ scale, int flags, float* __restrict__ grad_rgb_uniform) {
  pdl_enter();
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  const int v = lane & 15, par = lane >> 4;
  float s = 0.f;
  for (int t = par; t < n_parts; t += 2) s += partials[((size_t)n * n_parts + t) * 16 + v];
  s += __shfl_xor_sync(0xffffffffu, s, 16);
  if (lane < 9) gR[9 * (size_t)n + lane] = s;
  else if (lane < 12) gT[3 * (size_t)n + lane - 9] = s;
  else if (lane == 12) {
    if (flags & MVR_SCALE_IS_DIST) {      // d(1/dist)/d dist = -(1/dist)^2
      const float inv = __fdiv_rn(1.0f, __ldg(scale + n));
      s = -s * (inv * inv);
    }
    gs[n] = s;
  }
  else if (lane < 16 && grad_rgb_uniform) atomicAdd(grad_rgb_uniform + (lane - 13), s);      // N terms per channel
}

// The same reduction with the camera backward of the view behind it: (dR, dT) -> (d azim, d elev, d dist) by look_at_backward_view,
// plus the cloud-scale term of d dist -- the path MVRenderer takes (angles in, images out) then ends its backward with ONE launch
// instead of a reduction and a camera kernel, and the host with one call instead of two (the point step is bound by the host).
// gR / gT: optional copies of the camera gradients (NULL: not stored).  `dist` is the scale array (MVR_SCALE_IS_DIST).
__global__ void points_backward_reduce_angles_kernel(const float* __restrict__ partials, int N, int n_parts, const float* __restrict__ azim,
                                                     const float* __restrict__ elev, const float* __restrict__ dist, float* __restrict__ gR,
                                                     float* __restrict__ gT, float* __restrict__ g_azim, float* __restrict__ g_elev,
                                                     float* __restrict__ g_dist, float* __restrict__ grad_rgb_uniform) {
  pdl_enter();
  const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  const int v = lane & 15, par = lane >> 4;
  float s = 0.f;
  for (int t = par; t < n_parts; t += 2) s += partials[((size_t)n * n_parts + t) * 16 + v];
  s += __shfl_xor_sync(0xffffffffu, s, 16);
  if (gR && lane < 9) gR[9 * (size_t)n + lane] = s;
  else if (gT && lane >= 9 && lane < 12) gT[3 * (size_t)n + lane - 9] = s;
  else if (lane >= 13 && lane < 16 && grad_rgb_uniform) atomicAdd(grad_rgb_uniform + (lane - 13), s);
  float g[13];
#pragma unroll
  for (int i = 0; i < 13; ++i) g[i] = __shfl_sync(0xffffffffu, s, i);
  if (lane == 0) {
    const float d = __ldg(dist + n);
    float ga, ge, gd;
    look_at_backward_view(__ldg(azim + n), __ldg(elev + n), d, g, g + 9, nullptr, ga, ge, gd);
    const float inv = __fdiv_rn(1.0f, d);      // d(1/dist)/d dist = -(1/dist)^2, as points_backward_reduce_kernel
    g_azim[n] = ga; g_elev[n] = ge; g_dist[n] = gd + (-g[12] * (inv * inv));
  }
}

}  // namespace mvr

using namespace mvr;

static int check_points_common(const char* who, int B, int Np, int M, int H, int W, int K, double radius) {
  if (B < 0 || Np < 0 || M < 0) { set_error("%s: negative size", who); return -1; }
  if (H <= 0 || W <= 0 || H > 4096 || W > 4096) { set_error("%s: image size %dx%d outside [1, 4096]", who, H, W); return -2; }
  if (K < 1 || K > 64) { set_error("%s: points_per_pixel %d outside [1, 64]", who, K); return -3; }
  if (!(radius > 0.0)) { set_error("%s: radius must be positive", who); return -4; }
  if ((int64_t)B * M > 0x7fffffffLL / (H + 1) || B > 65535 || M > 65535) { set_error("%s: too many views", who); return -5; }
  return 0;
}

struct PointsWs {
  size_t keys, tab, pp, pw, tile_cnt, tile_off, tile_cur, list, partials, total;
  int tiles_x, tiles_y, ntiles, list_cap, ctas_per_view, mask_words;
  bool tiled;
};
static bool points_use_tiles(int K) {
  static const bool off = [] { const char* e = getenv("MVR_POINTS_TILED"); return e && atoi(e) == 0; }();   // profiling knob
  return !off && (K == 1 || K == 2 || K == 4 || K == 8);
}
static PointsWs points_ws(int B, int Np, int M, int H, int W, int K, double radius) {
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  PointsWs w;
  const size_t N = (size_t)B * M;
  w.tiles_x = (W + 31) / 32;
  w.tiles_y = (H + 31) / 32;
  w.ntiles = w.tiles_x * w.tiles_y;
  w.ctas_per_view = w.ntiles;
  w.mask_words = w.tiles_x;
  w.tiled = points_use_tiles(K);
  // a window of wpx consecutive pixels touches at most (wpx - 1) / 32 + 2 tiles per axis; the window holds the pixel
  // centres within +-rr of the point, at most floor(2 rr / pitch) + 1 with pitch >= 2 / max(H, W)
  const double rr = radius * 1.0001 + 1e-7;
  const long long wpx = (long long)(rr * (H > W ? H : W)) + 2;
  long long span = (wpx - 1) / 32 + 2;
  if (span > w.tiles_x && span > w.tiles_y) span = w.tiles_x > w.tiles_y ? w.tiles_x : w.tiles_y;
  const long long sx = span < w.tiles_x ? span : w.tiles_x, sy = span < w.tiles_y ? span : w.tiles_y;
  const long long cap = (long long)Np * sx * sy;
  w.list_cap = cap > 0x7fffffffLL ? 0x7fffffff : (int)cap;
  size_t o = 0;
  w.tab = o; o = al(o + ((size_t)W + H) * sizeof(float));
  w.keys = w.pp = w.pw = w.tile_cnt = w.tile_off = w.tile_cur = w.list = o;
  if (w.tiled) {
    w.pp = o; o = al(o + N * Np * sizeof(float4));
    w.pw = o; o = al(o + N * Np * sizeof(int2));
    w.tile_cnt = o; o = al(o + N * w.ntiles * sizeof(int));
    w.tile_off = o; o = al(o + N * w.ntiles * sizeof(int));
    w.tile_cur = o; o = al(o + N * w.ntiles * sizeof(int));
    w.list = o; o = al(o + N * (size_t)w.list_cap * sizeof(int) + 16);      // + 16: the tile kernel's bulk copies round a list's end up to 16 bytes
  } else {
    w.keys = o; o = al(o + N * H * W * K * 8);
  }
  const size_t fwd = o;
  w.partials = 0;                                  // the backward reuses the front of the workspace
  const size_t bwd = al(N * w.ctas_per_view * 16 * sizeof(float));
  w.total = fwd > bwd ? fwd : bwd;
  return w;
}

extern "C" size_t mvr_points_workspace_bytes(int B, int Np, int M, int H, int W, int K, double radius) {
  if (B < 0 || Np < 0 || M < 0 || H <= 0 || W <= 0 || K < 1 || !(radius > 0.0)) return 0;
  return points_ws(B, Np, M, H, W, K, radius).total;
}

extern "C" size_t mvr_points_hit_mask_words(int B, int M, int H, int W) {
  if (B < 0 || M < 0 || H <= 0 || W <= 0) return 0;
  return (size_t)B * M * H * ((W + 31) / 32);
}

static int points_tile_minb_k1() {
  static const int v = [] { const char* e = getenv("MVR_TILE_MINB_K1"); return (e && atoi(e) == 5) ? 5 : 4; }();
  return v;
}
// profiling knob: MVR_TILE_MINB=4 asks for four instead of five tile CTAs per SM at K = 4
static int points_tile_minb() {
  static const int v = [] { const char* e = getenv("MVR_TILE_MINB"); return (e && atoi(e) == 4) ? 4 : 5; }();
  return v;
}
// profiling knob: MVR_POINTS_BIN_FUSED=0 keeps the three-launch binning everywhere
static bool points_bin_fused() {
  static const bool v = [] { const char* e = getenv("MVR_POINTS_BIN_FUSED"); return !(e && atoi(e) == 0); }();
  return v;
}

extern "C" int mvr_points_forward(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                                  const float* T, const float* inv_dist, double radius, const float* bg_rgb,
                                  int H, int W, int K, int flags, const float* out_mean_std, void* images, int* idx,
                                  float* zbuf, float* dists2, uint32_t* hit_mask, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  int rc = check_points_common("mvr_points_forward", B, Np, M, H, W, K, radius);
  if (rc) return rc;
  const int64_t N = (int64_t)B * M;
  if (N == 0) return 0;
  if ((Np > 0 && !points) || !rgb || !R || !T || !inv_dist || !bg_rgb || !images || !idx || !workspace) { set_error("mvr_points_forward: null pointer"); return -6; }
  // K = 2 / 4: the kernels store a pixel's K ids as one int2 / int4 (a slice of a larger int32 buffer may not be aligned for that)
  if ((K == 2 || K == 4) && ((uintptr_t)idx & (uintptr_t)(4 * K - 1))) { set_error("mvr_points_forward: idx must be aligned to 4*K = %d bytes", 4 * K); return -10; }
  if (!out_norm_valid(out_mean_std)) { set_error("mvr_points_forward: out_mean_std needs std > 0"); return -9; }
  const PointsWs w = points_ws(B, Np, M, H, W, K, radius);
  const size_t HW = (size_t)H * W;
  if (workspace_bytes < w.total) { set_error("mvr_points_forward: workspace too small (%zu < %zu)", workspace_bytes, w.total); return -7; }
  if (w.tiled && (long long)Np * 1 > 0 && (long long)w.list_cap >= 0x7fffffffLL) { set_error("mvr_points_forward: point lists too large"); return -8; }
  char* wb = (char*)workspace;
  PointsParams p;
  p.points = points; p.rgb = rgb; p.R = R; p.T = T; p.inv_dist = inv_dist; p.bg_rgb = bg_rgb;
  p.radius = (float)radius;
  p.r2_raster = p.radius * p.radius;            // [upstream] rasterize_points_cpu.cpp: float radius * radius
  p.r2_weight = (float)(radius * radius);       // [upstream] points/renderer.py: python-float r * r
  p.B = B; p.Np = Np; p.M = M; p.H = H; p.W = W; p.K = K; p.flags = flags; p.mask_words = w.mask_words;
  p.keys = (unsigned long long*)(wb + w.keys);
  p.tab = (const float*)(wb + w.tab);
  p.pp = (float4*)(wb + w.pp); p.pw = (int2*)(wb + w.pw);
  p.tile_cnt = (int*)(wb + w.tile_cnt); p.tile_off = (int*)(wb + w.tile_off); p.tile_cur = (int*)(wb + w.tile_cur);
  p.list = (int*)(wb + w.list);
  p.tiles_x = w.tiles_x; p.tiles_y = w.tiles_y; p.ntiles = w.ntiles; p.list_cap = w.list_cap;
  p.vec_bg = (W % 4 == 0) && ((uintptr_t)images % 16 == 0);
  p.images = images; p.idx = idx; p.zbuf = zbuf; p.dists2 = dists2; p.hit_mask = hit_mask;
  p.onorm = make_out_norm(out_mean_std);
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 point_grid((unsigned)((Np + MVR_THREADS - 1) / MVR_THREADS), (unsigned)M, (unsigned)B);
  const bool bin_fused = w.tiled && Np > 0 && Np <= BIN_FUSED_MAX_POINTS && w.ntiles <= BIN_FUSED_MAX_TILES && points_bin_fused();
  if (Np > 0 && !bin_fused) MVR_LAUNCH(pixel_table_kernel, 1, MVR_THREADS, 0, st, (float*)(wb + w.tab), H, W);
  if (w.tiled) {
    if (bin_fused) {
      static const int cs_knob = [] { const char* e = getenv("MVR_BIN_CLUSTER"); return e ? atoi(e) : 0; }();      // profiling knob: 1 / 2 / 4 / 8
      // a cluster of 4 CTAs per view for large clouds, and whenever there are fewer views than SMs (configs[0]: 12 views -- one CTA per
      // view leaves 136 SMs idle while 12 CTAs walk 2048 points each: 24 -> 16 us, a fifth of that graph-replayed step)
      const int cs = (cs_knob == 1 || cs_knob == 2 || cs_knob == 4 || cs_knob == 8) ? cs_knob : ((Np > 4096 || (N < 148 && Np >= 512)) ? 4 : 1);
      if (cs == 1) {
        MVR_LAUNCH(points_bin_kernel_fused, dim3((unsigned)M, (unsigned)B), MVR_THREADS, ((size_t)W + H) * sizeof(float), st, p, (float*)(wb + w.tab), 1);
      } else {      // thread-block cluster of cs CTAs per view (distributed shared memory)
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(M * cs), (unsigned)B); cfg.blockDim = dim3(MVR_THREADS);
        cfg.dynamicSmemBytes = ((size_t)W + H) * sizeof(float); cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        mvr::prof_begin("points_bin_kernel_fused", st);
        cudaError_t le = cudaLaunchKernelEx(&cfg, points_bin_kernel_fused, p, (float*)(wb + w.tab), cs);
        mvr::prof_end("points_bin_kernel_fused", st);
        if (le != cudaSuccess) { set_error("mvr_points_forward: cudaLaunchKernelEx: %s", cudaGetErrorString(le)); return (int)le; }
      }
      rc = check_launch("points_bin_kernel_fused");
      if (rc) return rc;
    } else if (Np > 0) {
      cudaError_t e = cudaMemsetAsync(p.tile_cnt, 0, (size_t)N * w.ntiles * sizeof(int), st);
      if (e != cudaSuccess) { set_error("mvr_points_forward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return (int)e; }
      MVR_LAUNCH(points_bin_kernel<false>, point_grid, MVR_THREADS, 0, st, p);
      MVR_LAUNCH(points_bin_scan_kernel, (unsigned)N, MVR_THREADS, 0, st, p);
      MVR_LAUNCH(points_bin_kernel<true>, point_grid, MVR_THREADS, 0, st, p);
      rc = check_launch("points_bin_kernel");
      if (rc) return rc;
    }
    const dim3 tile_grid((unsigned)w.ntiles, (unsigned)M, (unsigned)B);
    const size_t smem = (size_t)K * 1024 * sizeof(unsigned long long);
    cudaError_t e = cudaSuccess;
    switch (K) {
      // Occupancy is what hides the start-up latency of these short CTAs (r2t, same box, K = 1: 40 registers / unconstrained
      // 0.094 ms, 47 registers / 5 CTAs 0.102 ms, 55 registers / 4 CTAs 0.110 ms): K = 1 / 2 compile to 40 / 46 registers when
      // left alone (MINB = 0), K = 4 is held to five CTAs per SM (48 registers instead of 56, no spills: 0.131 vs 0.133 ms),
      // K = 8 to three (74 KB of shared memory per CTA).
      case 1:
        if (points_tile_minb_k1() == 5) MVR_LAUNCH_PDL((points_tile_kernel<1, 5>), tile_grid, MVR_THREADS, smem, st, p);
        else MVR_LAUNCH_PDL((points_tile_kernel<1, 0>), tile_grid, MVR_THREADS, smem, st, p);
        break;
      case 2: MVR_LAUNCH_PDL((points_tile_kernel<2, 0>), tile_grid, MVR_THREADS, smem, st, p); break;
      case 4:
        if (points_tile_minb() == 4) MVR_LAUNCH_PDL((points_tile_kernel<4, 0>), tile_grid, MVR_THREADS, smem, st, p);
        else MVR_LAUNCH_PDL((points_tile_kernel<4, 5>), tile_grid, MVR_THREADS, smem, st, p);
        break;
      default: {
        // 64 KB of dynamic shared memory needs the opt-in (per device; the call is a few hundred nanoseconds)
        e = cudaFuncSetAttribute(points_tile_kernel<8, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("mvr_points_forward: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return (int)e; }
        MVR_LAUNCH_PDL((points_tile_kernel<8, 3>), tile_grid, MVR_THREADS, smem, st, p);
      }
    }
    return check_launch("points_tile_kernel");
  }
  // ---- generic K: global key plane (memset + scatter with global atomics + resolve) ----
  const size_t need = (size_t)N * HW * K * 8;
  cudaError_t e = cudaMemsetAsync(p.keys, 0xFF, need, st);      // every key = EMPTY
  if (e != cudaSuccess) { set_error("mvr_points_forward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return (int)e; }
  const int tiles_x = (W + 31) / 32, tiles_y = (H + 7) / 8;
  const dim3 resolve_grid((unsigned)(tiles_x * tiles_y), (unsigned)M, (unsigned)B);
  if (Np > 0) {
    MVR_LAUNCH(points_scatter_kernel, point_grid, MVR_THREADS, 0, st, p);
    rc = check_launch("points_scatter_kernel");
    if (rc) return rc;
  }
  switch (K) {
    case 1: MVR_LAUNCH(points_resolve_kernel<1>, resolve_grid, MVR_THREADS, 0, st, p, tiles_x); break;
    case 2: MVR_LAUNCH(points_resolve_kernel<2>, resolve_grid, MVR_THREADS, 0, st, p, tiles_x); break;
    case 4: MVR_LAUNCH(points_resolve_kernel<4>, resolve_grid, MVR_THREADS, 0, st, p, tiles_x); break;
    case 8: MVR_LAUNCH(points_resolve_kernel<8>, resolve_grid, MVR_THREADS, 0, st, p, tiles_x); break;
    default: MVR_LAUNCH(points_resolve_kernel<0>, resolve_grid, MVR_THREADS, 0, st, p, tiles_x); break;
  }
  return check_launch("points_resolve_kernel");
}

static int points_backward_impl(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                                const float* T, const float* inv_dist, double radius, int H, int W, int K,
                                int flags, const float* out_mean_std, const int* idx, const uint32_t* hit_mask,
                                const void* grad_images,
                                float* gR, float* gT, float* g_inv_dist, float* grad_points, float* grad_rgb,
                                void* workspace, size_t workspace_bytes, void* stream,
                                const float* azim, const float* elev, float* g_azim, float* g_elev, float* g_dist) {
  const bool angles = azim != nullptr;
  int rc = check_points_common("mvr_points_backward", B, Np, M, H, W, K, radius);
  if (rc) return rc;
  const int64_t N = (int64_t)B * M;
  if (N == 0) return 0;
  if ((Np > 0 && !points) || !rgb || !R || !T || !inv_dist || !idx || !grad_images || !workspace ||
      (!angles && (!gR || !gT || !g_inv_dist)) || (angles && (!elev || !g_azim || !g_elev || !g_dist))) {
    set_error("mvr_points_backward: null pointer"); return -6;
  }
  if (angles && !(flags & MVR_SCALE_IS_DIST)) { set_error("mvr_points_backward_angles: needs MVR_SCALE_IS_DIST (the scale array is dist)"); return -10; }
  if (!out_norm_valid(out_mean_std)) { set_error("mvr_points_backward: out_mean_std needs std > 0"); return -9; }
  const PointsWs w = points_ws(B, Np, M, H, W, K, radius);
  const size_t need = (size_t)N * w.ctas_per_view * 16 * sizeof(float);
  if (workspace_bytes < need) { set_error("mvr_points_backward: workspace too small (%zu < %zu)", workspace_bytes, need); return -7; }
  PointsBwdParams p;
  p.points = points; p.rgb = rgb; p.R = R; p.T = T; p.inv_dist = inv_dist;
  p.r2_weight = (float)(radius * radius);
  p.B = B; p.Np = Np; p.M = M; p.H = H; p.W = W; p.K = K; p.flags = flags;
  p.tiles_x = w.tiles_x; p.tiles_y = (H + 31) / 32; p.ctas_per_view = w.ctas_per_view; p.mask_words = w.mask_words;
  p.idx = idx; p.grad_images = grad_images; p.hit_mask = hit_mask;
  p.partials = (float*)((char*)workspace + w.partials);
  p.grad_points = grad_points; p.grad_rgb = grad_rgb;
  p.onorm = make_out_norm(out_mean_std);
  cudaStream_t st = (cudaStream_t)stream;
  static const int wpc = [] { const char* e = getenv("MVR_PBWD_WPC"); const int x = e ? atoi(e) : 8; return (x == 1 || x == 2 || x == 4 || x == 8) ? x : 8; }();      // profiling knob
  const int groups_y = (p.tiles_y + wpc - 1) / wpc;
  p.ctas_per_view = w.tiles_x * groups_y;             // one partial per CTA (<= one per tile: the workspace is sized for that)
  const dim3 grid((unsigned)p.ctas_per_view, (unsigned)M, (unsigned)B);
  const bool vrgb = flags & MVR_RGB_PER_ELEMENT;
  const bool gu = grad_rgb && !vrgb;      // gradient of the single point colour: through the partials (acc[13..15])
  // the register-resident variants read a pixel's K ids as one vector: they need the fragment tensor aligned to K ints
  const int kt = ((K == 1 || K == 2 || K == 4) && ((uintptr_t)idx & (size_t)(4 * K - 1)) == 0) ? K : 0;
#define MVR_PBWD(KT_) do { if (vrgb) MVR_LAUNCH((points_backward_kernel<KT_, true, false>), grid, 32 * wpc, 0, st, p); \
                           else if (gu) MVR_LAUNCH((points_backward_kernel<KT_, false, true>), grid, 32 * wpc, 0, st, p); \
                           else MVR_LAUNCH((points_backward_kernel<KT_, false, false>), grid, 32 * wpc, 0, st, p); } while (0)
  switch (kt) {
    case 1: MVR_PBWD(1); break;
    case 2: MVR_PBWD(2); break;
    case 4: MVR_PBWD(4); break;
    default: MVR_PBWD(0); break;
  }
#undef MVR_PBWD
  rc = check_launch("points_backward_kernel");
  if (rc) return rc;
  const int wpb = 8;
  if (angles) {
    MVR_LAUNCH_PDL(points_backward_reduce_angles_kernel, (unsigned)((N + wpb - 1) / wpb), wpb * 32, 0, st, (const float*)p.partials, (int)N, p.ctas_per_view,
               azim, elev, inv_dist, gR, gT, g_azim, g_elev, g_dist, gu ? grad_rgb : (float*)nullptr);
    return check_launch("points_backward_reduce_angles_kernel");
  }
  MVR_LAUNCH_PDL(points_backward_reduce_kernel, (unsigned)((N + wpb - 1) / wpb), wpb * 32, 0, st, (const float*)p.partials, (int)N, p.ctas_per_view, gR, gT, g_inv_dist, inv_dist, flags,
             gu ? grad_rgb : (float*)nullptr);
  return check_launch("points_backward_reduce_kernel");
}

extern "C" int mvr_points_backward(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                                   const float* T, const float* inv_dist, double radius, int H, int W, int K,
                                   int flags, const float* out_mean_std, const int* idx, const uint32_t* hit_mask,
                                   const void* grad_images,
                                   float* gR, float* gT, float* g_inv_dist, float* grad_points, float* grad_rgb,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  return points_backward_impl(points, rgb, B, Np, M, R, T, inv_dist, radius, H, W, K, flags, out_mean_std, idx, hit_mask, grad_images, gR, gT,
                              g_inv_dist, grad_points, grad_rgb, workspace, workspace_bytes, stream, nullptr, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int mvr_points_backward_angles(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                                          const float* T, const float* azim, const float* elev, const float* dist, double radius,
                                          int H, int W, int K, int flags, const float* out_mean_std, const int* idx,
                                          const uint32_t* hit_mask, const void* grad_images, float* g_azim, float* g_elev,
                                          float* g_dist, float* gR, float* gT, float* grad_points, float* grad_rgb, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  if (!azim) { set_error("mvr_points_backward_angles: null pointer"); return -6; }
  return points_backward_impl(points, rgb, B, Np, M, R, T, dist, radius, H, W, K, flags, out_mean_std, idx, hit_mask, grad_images, gR, gT,
                              nullptr, grad_points, grad_rgb, workspace, workspace_bytes, stream, azim, elev, g_azim, g_elev, g_dist);
}
