"""GPU tests of the view regulariser (mvtn_b200/csrc/mvr_augment.cu) at the shapes its fast paths do not cover: widths above
1024 (the one-CTA-per-row backward), widths that are not a multiple of 4 and misaligned buffers (the element-by-element
forward and backward), one-row / one-column images, shifts of a whole image side, dropped views, no views, and more than
65535 (view, channel) planes (the launches are chunked at the grid.y limit, in whole views).

Called through the C ABI and through mvtn_b200.regularize_rendered_views, against the plain fp64 gather written here,
    out[n, c, y, x] = scale[n] * in[n, c, clamp(y + sy), fx(clamp(x + sx))],   fx(u) = flip ? W-1-u : u,
and its adjoint (every output pixel's gradient added to its source pixel).  Bars:
  * forward, fp32: bit-exact (one fp32 product with the view's factor: the fp64 product of two fp32 values rounded once);
  * forward, bf16: bit-exact with that fp32 product rounded once to bf16;
  * backward, fp32: 1e-5 relative to the summed magnitudes (the fp64 adjoint of |grad_out|, times |scale|) per pixel;
  * backward, bf16: within one bf16 ulp of the fp64 adjoint (plus the same fp32 summation allowance).
Every case asserts the kernel that ran with the library's launch profiler (test_gpu_branches.launches).
"""
import numpy as np
import pytest
import torch

import mvtn_b200
from mvtn_b200 import _lib as L
from mvtn_b200.augment import draw_regularizer
from test_gpu_branches import launches

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.bfloat16]
P_DROP = 0.3


def ref_forward(x, scale, flip, sy, sx):
    """x (N, C, H, W) -> the gather in fp64 (products of two fp32 values are exact there)."""
    N, C, H, W = x.shape
    yi = (torch.arange(H, device=x.device) + sy).clamp(0, H - 1)
    xi = (torch.arange(W, device=x.device) + sx).clamp(0, W - 1)
    if flip:
        xi = W - 1 - xi
    out = x.double()[:, :, yi][:, :, :, xi]
    if scale is not None:
        out = out * scale.double().reshape(N, 1, 1, 1)
    return out


def ref_backward(g, scale, flip, sy, sx):
    """The adjoint of ref_forward in fp64: grad_out (N, C, H, W) -> grad_in."""
    N, C, H, W = g.shape
    yi = (torch.arange(H, device=g.device) + sy).clamp(0, H - 1)
    xi = (torch.arange(W, device=g.device) + sx).clamp(0, W - 1)
    if flip:
        xi = W - 1 - xi
    rows = torch.zeros(N, C, H, W, dtype=torch.float64, device=g.device).index_add_(2, yi, g.double())
    out = torch.zeros_like(rows).index_add_(3, xi, rows)
    if scale is not None:
        out = out * scale.double().reshape(N, 1, 1, 1)
    return out


def expected_forward(x, scale, flip, sy, sx):
    """What the kernel must write: the fp32 product, and for bf16 that product rounded once more."""
    return ref_forward(x, scale, flip, sy, sx).float().to(x.dtype)


def check_backward(gi, g, scale, flip, sy, sx):
    want = ref_backward(g, scale, flip, sy, sx)
    mag = ref_backward(g.abs(), None if scale is None else scale.abs(), flip, sy, sx)
    err = (gi.double() - want).abs()
    if gi.dtype is torch.float32:
        bar = 1e-5 * mag
    else:
        # one bf16 ulp of the reference (8 significant bits), floored at the smallest normal; plus fp32 summation rounding
        e = torch.floor(torch.log2(want.abs().clamp_min(2.0 ** -126)))
        bar = torch.exp2(e - 7) + 2.0 ** -20 * mag
    worst = float((err - bar).max())
    assert worst <= 0, f"backward off by {worst} beyond the bar"


def view_scale(N, dev, seed):
    """Per-view factors 0 (dropped) or 1 / (1 - p), as dropout2d draws them, with both present."""
    g = torch.Generator().manual_seed(seed)
    s = (torch.rand(N, generator=g) >= P_DROP).float() / (1 - P_DROP)
    s[0] = 0.0
    if N > 1:
        s[-1] = 1.0 / (1 - P_DROP)
    return s.to(dev)


def buffer(shape, dtype, dev, seed, offset=0):
    """A contiguous (N, C, H, W) tensor of normal values whose data starts `offset` elements into its allocation."""
    n = int(np.prod(shape))
    flat = torch.randn(n + offset, generator=torch.Generator().manual_seed(seed)).to(dtype).to(dev)
    return flat[offset:].view(shape)


def stream():
    return torch.cuda.current_stream().cuda_stream


def abi_forward(x, scale, flip, sy, sx, out):
    N, C, H, W = x.shape
    flags = L.IMAGES_BF16 if x.dtype is torch.bfloat16 else 0
    return L.load().mvr_images_regularize_forward(x.data_ptr() if N else None, N, C, H, W, None if scale is None else scale.data_ptr(),
                                                  int(flip), sy, sx, flags, out.data_ptr() if N else None, stream())


def abi_backward(g, scale, flip, sy, sx, gi):
    N, C, H, W = g.shape
    flags = L.IMAGES_BF16 if g.dtype is torch.bfloat16 else 0
    return L.load().mvr_images_regularize_backward(g.data_ptr() if N else None, N, C, H, W, None if scale is None else scale.data_ptr(),
                                                   int(flip), sy, sx, flags, gi.data_ptr() if N else None, stream())


def fwd_kernel(W, out):
    vec = W % 4 == 0 and out.data_ptr() % 16 == 0
    return f"images_regularize_kernel<{'true' if vec else 'false'}>"


def bwd_kernel(W, g, gi):
    if W > 1024:
        return "images_regularize_backward_kernel"
    vec = W % 4 == 0 and g.data_ptr() % 16 == 0 and gi.data_ptr() % 16 == 0
    return f"images_regularize_backward_rows_kernel<{'true' if vec else 'false'}>"


def run_abi_case(dev, dtype, N, C, H, W, flip, sy, sx, scaled=True, in_off=0, out_off=0, seed=0, chunks=1):
    """Forward and backward through the C ABI, each checked against the fp64 reference and for the kernel it launched."""
    x = buffer((N, C, H, W), dtype, dev, seed, in_off)
    out = buffer((N, C, H, W), dtype, dev, seed + 1, out_off)
    scale = view_scale(N, dev, seed + 2) if scaled else None
    rc, n = launches(fwd_kernel(W, out), lambda: abi_forward(x, scale, flip, sy, sx, out))
    L.check(rc, "mvr_images_regularize_forward")
    assert n == chunks, (fwd_kernel(W, out), n)
    torch.cuda.synchronize()
    assert torch.equal(out, expected_forward(x, scale, flip, sy, sx))
    g = buffer((N, C, H, W), dtype, dev, seed + 3, out_off)         # the gradient arrives where the output was written
    gi = buffer((N, C, H, W), dtype, dev, seed + 4, in_off)
    rc, n = launches(bwd_kernel(W, g, gi), lambda: abi_backward(g, scale, flip, sy, sx, gi))
    L.check(rc, "mvr_images_regularize_backward")
    assert n == chunks, (bwd_kernel(W, g, gi), n)
    torch.cuda.synchronize()
    check_backward(gi, g, scale, flip, sy, sx)


# (N, C, H, W, flip, sy, sx, scaled): W > 1024 reaches the one-CTA-per-row backward; W % 4 != 0 the element-by-element paths
CASES = {
    "w1025_flip_shift": (2, 3, 3, 1025, 1, 1, -7, True),
    "w1031_shift": (3, 2, 2, 1031, 0, -1, 5, True),
    "w1025_c1_edge_shift": (3, 1, 2, 1025, 1, 1, -1024, True),
    "w1031_c4_edge_shift": (2, 4, 3, 1031, 0, -2, 1030, True),
    "w_mod4_1": (2, 3, 5, 13, 1, 2, -3, True),
    "w_mod4_2": (2, 3, 5, 14, 0, -4, 13, False),
    "w_mod4_3": (3, 4, 6, 15, 1, 5, -14, True),
    "h1": (3, 3, 1, 16, 1, 0, -5, True),
    "h1_w7": (2, 4, 1, 7, 0, 0, 6, True),
    "w1": (3, 3, 7, 1, 1, -6, 0, True),
    "h_ne_w": (2, 3, 12, 20, 0, 3, -4, True),
    "h_ne_w_flip": (4, 1, 20, 12, 1, -19, 11, True),
    "edge_shift_pos": (2, 3, 9, 12, 1, 8, 11, True),
    "edge_shift_neg": (2, 3, 9, 12, 0, -8, -11, True),
    "no_scale": (2, 3, 8, 8, 1, 2, 3, False),
}


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp32", "bf16"])
@pytest.mark.parametrize("case", list(CASES))
def test_regularizer_abi_matches_fp64_gather(cuda_device, case, dtype):
    N, C, H, W, flip, sy, sx, scaled = CASES[case]
    run_abi_case(cuda_device, dtype, N, C, H, W, flip, sy, sx, scaled, seed=len(case))


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp32", "bf16"])
@pytest.mark.parametrize("in_off,out_off", [(1, 0), (0, 1), (1, 1)])
def test_regularizer_misaligned_buffers(cuda_device, dtype, in_off, out_off):
    """W % 4 == 0 but a buffer one element off its allocation: the forward takes its element-by-element instance when the
    output is misaligned (a misaligned input is read element by element by either), the backward when either is."""
    run_abi_case(cuda_device, dtype, 3, 3, 16, 16, 1, -3, 2, True, in_off, out_off, seed=5)


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp32", "bf16"])
def test_regularizer_no_views(cuda_device, dtype):
    """N = 0: nothing to do, no launch, null pointers accepted."""
    empty = torch.empty(0, 3, 8, 8, dtype=dtype, device=cuda_device)
    rc, n = launches("images_regularize", lambda: (abi_forward(empty, None, 1, 2, 2, empty), abi_backward(empty, None, 1, 2, 2, empty)))
    assert rc == (0, 0) and n == 0


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp32", "bf16"])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_regularizer_more_than_65535_planes(cuda_device, dtype, C):
    """N C > 65535 planes at 8 x 8 (17 MB in fp32): two launches, split between views, so each plane still finds its view's
    factor -- also when C does not divide 65535 (C = 4: the soft shaders' RGBA views)."""
    N = 66000 // C + 1
    run_abi_case(cuda_device, dtype, N, C, 8, 8, 1, -2, 3, True, seed=40 + C, chunks=2)


@pytest.mark.parametrize("dtype", DTYPES, ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape,seed", [((1, 2, 1, 1025, 1025), 3), ((4200, 4, 4, 4, 4), 8), ((2, 3, 3, 13, 13), 21)])
def test_regularize_rendered_views_edges(cuda_device, dtype, shape, seed):
    """mvtn_b200.regularize_rendered_views with dropout and the flip / crop draw: 1025 x 1025 views (one CTA per row in the
    backward), 67200 RGBA planes (chunked between views), 13 x 13 views (element by element); against the fp64 gather under
    the decisions draw_regularizer makes from the same seed."""
    dev = cuda_device
    B, M, C, H, W = shape
    x = torch.randn(shape, generator=torch.Generator().manual_seed(seed)).to(dtype).to(dev).requires_grad_()
    torch.manual_seed(seed)
    scale, flip, sy, sx = draw_regularizer(x, P_DROP, True, 0.3)
    torch.manual_seed(seed)
    out = mvtn_b200.regularize_rendered_views(x, P_DROP, True, 0.3)
    xs = x.detach().reshape(B * M, C, H, W)
    assert torch.equal(out.detach().reshape(B * M, C, H, W), expected_forward(xs, scale, flip, sy, sx))
    g = torch.randn(shape, generator=torch.Generator().manual_seed(seed + 1)).to(dtype).to(dev)
    chunks = -(-(B * M * C) // ((65535 // C) * C))
    want = bwd_kernel(W, g, x) if W > 1024 else "images_regularize_backward_rows_kernel"
    _, n = launches(want, lambda: out.backward(g))
    assert n == chunks, (want, n)
    check_backward(x.grad.reshape(B * M, C, H, W), g.reshape(B * M, C, H, W), scale, flip, sy, sx)
