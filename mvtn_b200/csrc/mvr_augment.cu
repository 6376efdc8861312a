// mvr_augment.cu -- the regulariser the training loops apply to the rendered views right behind the renderer
// (ops.py:138-178 regualarize_rendered_views -> run_mvtn.py:186,244, viewGCN/tools/Trainer_mvt.py:104), as ONE pass:
//
//   reference: dropout2d over (B, M, 3, H, W) -- feature dropout: a whole VIEW is zeroed or scaled by 1 / (1 - p) --, then, batchwise
//   (one decision for all B*M views): RandomHorizontalFlip, ReplicationPad2d(pad) with pad = int((1 + crop_ratio) H) - H, RandomCrop(H).
//   Four full-size passes (one of them over the (H + 2 pad)^2 padded copy: 3.0x the image bytes written at crop_ratio 0.3).
//
//   here: the three steps compose into one gather,
//       out[n, c, y, x] = scale[n] * in[n, c, clamp(y + sy, 0, H-1), fx(clamp(x + sx, 0, W-1))],   fx(u) = flip ? W-1-u : u,
//   with (sy, sx) = crop offset - pad in [-pad, pad]: 1 read + 1 write of the images (HBM-bound streaming; SURVEY 8f N2).
//   The random decisions are drawn by the caller with the very torch calls the reference makes (mvtn_b200/augment.py), so the
//   result is the reference's bit for bit under the same seeds.
//
//   backward: the gather's adjoint.  An interior input pixel feeds exactly one output pixel; an input pixel of the first / last row
//   (column) also receives every output row (column) the clamp folded onto it -- up to 2 pad + 1 of them.  One WARP per (view,
//   channel, input row) (one CTA above W = 1024): the column sums of the contributing output rows go to shared memory (coalesced row
//   reads), then each thread adds up the columns folded onto its input column.
#include <cstdint>
#include <cuda_bf16.h>

#include "mvr_common.cuh"

namespace mvr {

struct AugParams {
  const void* in; void* out;
  const float* scale;      // (N) per-view factor (0 or 1 / (1 - p)), or NULL
  int N, C, H, W, flip, sy, sx, bf16;
};

__device__ __forceinline__ float aug_load(const void* base, bool bf16, size_t i) {
  if (bf16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[i]);
  return __ldg(reinterpret_cast<const float*>(base) + i);
}
__device__ __forceinline__ void aug_store(void* base, bool bf16, size_t i, float v) {
  if (bf16) reinterpret_cast<__nv_bfloat16*>(base)[i] = __float2bfloat16_rn(v);
  else reinterpret_cast<float*>(base)[i] = v;
}

// grid: x = chunks of 256 QUADS (4 consecutive output pixels of a row), y = (view, channel) plane.  VEC: W % 4 == 0 and 16-byte
// (bf16: 8-byte) aligned planes -- one vector store per quad; the four source pixels are consecutive (or the clamp repeats one)
template <bool VEC>
__global__ void __launch_bounds__(MVR_THREADS) images_regularize_kernel(const AugParams p) {
  const int qpr = (p.W + 3) >> 2;
  const int q = blockIdx.x * MVR_THREADS + threadIdx.x, plane = blockIdx.y;
  if (q >= p.H * qpr) return;
  const int y = q / qpr, x0 = (q - y * qpr) << 2;
  const float s = p.scale ? __ldg(p.scale + plane / p.C) : 1.f;
  const int yi = min(max(y + p.sy, 0), p.H - 1);
  const size_t base = (size_t)plane * p.H * p.W;
  const size_t row_in = base + (size_t)yi * p.W, o = base + (size_t)y * p.W + x0;
  float v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int xi = min(max(x0 + k + p.sx, 0), p.W - 1);
    if (p.flip) xi = p.W - 1 - xi;
    // (a dropped view is written as zeros without being read: the reference's `input * 0` is 0 for the finite images a renderer emits)
    v[k] = (s == 0.f || x0 + k >= p.W) ? 0.f : aug_load(p.in, p.bf16, row_in + xi) * s;
  }
  if (VEC) {
    if (p.bf16) {
      const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + o) = make_uint2(*reinterpret_cast<const unsigned int*>(&a), *reinterpret_cast<const unsigned int*>(&b));
    } else {
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + o) = make_float4(v[0], v[1], v[2], v[3]);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) if (x0 + k < p.W) aug_store(p.out, p.bf16, o + k, v[k]);
  }
}

// the output rows (columns) whose clamped source is input row (column) u: [lo, hi], empty when lo > hi
__device__ __forceinline__ void folded_range(int u, int shift, int S, int& lo, int& hi) {
  lo = hi = u - shift;                                  // the unclamped preimage
  if (u == 0) lo = 0;                                   // everything the clamp folded onto the first ...
  if (u == S - 1) hi = S - 1;                           // ... / last row
  lo = max(lo, 0); hi = min(hi, S - 1);
  if (u == 0 && u == S - 1) { lo = 0; hi = S - 1; }
}

// grid: x = input row, y = (view, channel) plane; dynamic shared memory: W floats (column sums of the contributing output rows)
__global__ void __launch_bounds__(MVR_THREADS) images_regularize_backward_kernel(const AugParams p) {
  extern __shared__ float s_col[];
  const int yi = blockIdx.x, plane = blockIdx.y, tid = threadIdx.x;
  const int n = plane / p.C;
  const float s = p.scale ? __ldg(p.scale + n) : 1.f;
  const size_t base = (size_t)plane * p.H * p.W;
  int ylo, yhi;
  folded_range(yi, p.sy, p.H, ylo, yhi);
  for (int x = tid; x < p.W; x += MVR_THREADS) {
    float a = 0.f;
    if (s != 0.f)
      for (int y = ylo; y <= yhi; ++y) a += aug_load(p.in, p.bf16, base + (size_t)y * p.W + x);      // p.in = grad_out here
    s_col[x] = a;
  }
  __syncthreads();
  for (int x = tid; x < p.W; x += MVR_THREADS) {      // x: input column; its source index before the flip
    const int u = p.flip ? p.W - 1 - x : x;
    int xlo, xhi;
    folded_range(u, p.sx, p.W, xlo, xhi);
    float a = 0.f;
    for (int xo = xlo; xo <= xhi; ++xo) a += s_col[xo];
    aug_store(p.out, p.bf16, base + (size_t)yi * p.W + x, a * s);                                     // p.out = grad_in
  }
}

// The same with one WARP per input row (W <= 1024: eight rows' column sums fit in shared memory): only the first and the last row
// of a plane loop over more than one output row, so a CTA per row spends most of its time launching.
// grid: x = groups of 8 input rows, y = plane; dynamic shared memory: 8 W floats
template <bool VEC>      // VEC: W % 4 == 0 and aligned planes -- the rows move as 16-byte (bf16: 8-byte) quads
__global__ void __launch_bounds__(MVR_THREADS) images_regularize_backward_rows_kernel(const AugParams p) {
  extern __shared__ float s_rows[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int yi = blockIdx.x * 8 + warp, plane = blockIdx.y;
  if (yi >= p.H) return;                              // warp-uniform; no CTA barrier below
  float* s_col = s_rows + (size_t)warp * p.W;
  const float s = p.scale ? __ldg(p.scale + plane / p.C) : 1.f;
  const size_t base = (size_t)plane * p.H * p.W;
  int ylo, yhi;
  folded_range(yi, p.sy, p.H, ylo, yhi);
  if (VEC) {
    for (int x = lane << 2; x < p.W; x += 128) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      if (s != 0.f)
        for (int y = ylo; y <= yhi; ++y) {
          const size_t i = base + (size_t)y * p.W + x;
          if (p.bf16) {
            const uint2 r = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p.in) + i));
            a0 += __uint_as_float(r.x << 16); a1 += __uint_as_float(r.x & 0xffff0000u);
            a2 += __uint_as_float(r.y << 16); a3 += __uint_as_float(r.y & 0xffff0000u);
          } else {
            const float4 r = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.in) + i));
            a0 += r.x; a1 += r.y; a2 += r.z; a3 += r.w;
          }
        }
      *reinterpret_cast<float4*>(s_col + x) = make_float4(a0, a1, a2, a3);
    }
  } else {
    for (int x = lane; x < p.W; x += 32) {
      float a = 0.f;
      if (s != 0.f)
        for (int y = ylo; y <= yhi; ++y) a += aug_load(p.in, p.bf16, base + (size_t)y * p.W + x);
      s_col[x] = a;
    }
  }
  __syncwarp();
  auto folded = [&](int x) {      // x: input column; u: its source index before the flip
    const int u = p.flip ? p.W - 1 - x : x;
    int xlo, xhi;
    folded_range(u, p.sx, p.W, xlo, xhi);
    float a = 0.f;
    for (int xo = xlo; xo <= xhi; ++xo) a += s_col[xo];
    return a * s;
  };
  if (VEC) {
    for (int x = lane << 2; x < p.W; x += 128) {
      const float v0 = folded(x), v1 = folded(x + 1), v2 = folded(x + 2), v3 = folded(x + 3);
      const size_t o = base + (size_t)yi * p.W + x;
      if (p.bf16) {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v0, v1), b = __floats2bfloat162_rn(v2, v3);
        *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + o) = make_uint2(*reinterpret_cast<const unsigned int*>(&a), *reinterpret_cast<const unsigned int*>(&b));
      } else {
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + o) = make_float4(v0, v1, v2, v3);
      }
    }
  } else {
    for (int x = lane; x < p.W; x += 32) aug_store(p.out, p.bf16, base + (size_t)yi * p.W + x, folded(x));
  }
}

}  // namespace mvr

using namespace mvr;

static int check_aug(const char* who, const void* in, const void* out, int N, int C, int H, int W, int sy, int sx) {
  if (N < 0 || C <= 0 || C > 65535 || H <= 0 || W <= 0 || H > 65535 || W > 65535 || (int64_t)N * C > 0x7fffffffLL) { set_error("%s: bad shape (%d, %d, %d, %d)", who, N, C, H, W); return -1; }
  if (N == 0) return 0;
  if (!in || !out) { set_error("%s: null pointer", who); return -2; }
  if (in == out) { set_error("%s: in-place is not supported (the gather reads what another thread writes)", who); return -3; }
  if (sy <= -H || sy >= H || sx <= -W || sx >= W) { set_error("%s: shift (%d, %d) outside the image", who, sy, sx); return -4; }
  return 0;
}

extern "C" int mvr_images_regularize_forward(const void* images, int N, int C, int H, int W, const float* view_scale, int flip,
                                             int shift_y, int shift_x, int flags, void* out, void* stream) {
  int rc = check_aug("mvr_images_regularize_forward", images, out, N, C, H, W, shift_y, shift_x);
  if (rc || N == 0) return rc;
  AugParams p{images, out, view_scale, N, C, H, W, flip ? 1 : 0, shift_y, shift_x, (flags & MVR_IMAGES_BF16) ? 1 : 0};
  const int64_t planes = (int64_t)N * C;
  const bool vec = W % 4 == 0 && ((uintptr_t)out % 16 == 0);
  const unsigned gx = (unsigned)(((int64_t)H * ((W + 3) / 4) + MVR_THREADS - 1) / MVR_THREADS);
  const int64_t chunk = (int64_t)(65535 / C) * C;      // grid.y limit, in whole views: a chunk's planes start at view z0 / C
  for (int64_t z0 = 0; z0 < planes; z0 += chunk) {
    const int nz = (int)((planes - z0) < chunk ? (planes - z0) : chunk);
    AugParams q = p;
    const size_t off = (size_t)z0 * H * W * (p.bf16 ? 2 : 4);
    q.in = (const char*)images + off; q.out = (char*)out + off;
    q.scale = view_scale ? view_scale + z0 / C : nullptr;
    if (vec) MVR_LAUNCH(images_regularize_kernel<true>, dim3(gx, (unsigned)nz), MVR_THREADS, 0, (cudaStream_t)stream, q);
    else MVR_LAUNCH(images_regularize_kernel<false>, dim3(gx, (unsigned)nz), MVR_THREADS, 0, (cudaStream_t)stream, q);
  }
  return check_launch("images_regularize_kernel");
}

extern "C" int mvr_images_regularize_backward(const void* grad_out, int N, int C, int H, int W, const float* view_scale, int flip,
                                              int shift_y, int shift_x, int flags, void* grad_in, void* stream) {
  int rc = check_aug("mvr_images_regularize_backward", grad_out, grad_in, N, C, H, W, shift_y, shift_x);
  if (rc || N == 0) return rc;
  if ((size_t)W * sizeof(float) > 48 * 1024) { set_error("mvr_images_regularize_backward: W > 12288"); return -6; }
  AugParams p{grad_out, grad_in, view_scale, N, C, H, W, flip ? 1 : 0, shift_y, shift_x, (flags & MVR_IMAGES_BF16) ? 1 : 0};
  const int64_t planes = (int64_t)N * C;
  const int64_t chunk = (int64_t)(65535 / C) * C;      // grid.y limit, in whole views
  for (int64_t z0 = 0; z0 < planes; z0 += chunk) {
    const int nz = (int)((planes - z0) < chunk ? (planes - z0) : chunk);
    AugParams q = p;
    const size_t off = (size_t)z0 * H * W * (p.bf16 ? 2 : 4);
    q.in = (const char*)grad_out + off; q.out = (char*)grad_in + off;
    q.scale = view_scale ? view_scale + z0 / C : nullptr;
    const bool vec = W % 4 == 0 && ((uintptr_t)grad_out % 16 == 0) && ((uintptr_t)grad_in % 16 == 0);
    if (W <= 1024 && vec) MVR_LAUNCH(images_regularize_backward_rows_kernel<true>, dim3((unsigned)((H + 7) / 8), (unsigned)nz), MVR_THREADS, (size_t)8 * W * sizeof(float), (cudaStream_t)stream, q);
    else if (W <= 1024) MVR_LAUNCH(images_regularize_backward_rows_kernel<false>, dim3((unsigned)((H + 7) / 8), (unsigned)nz), MVR_THREADS, (size_t)8 * W * sizeof(float), (cudaStream_t)stream, q);
    else MVR_LAUNCH(images_regularize_backward_kernel, dim3((unsigned)H, (unsigned)nz), MVR_THREADS, (size_t)W * sizeof(float), (cudaStream_t)stream, q);
  }
  return check_launch("images_regularize_backward_kernel");
}
