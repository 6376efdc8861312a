"""shader="soft_depth" at the edges test_gpu_soft_depth.py's cases do not reach.  Parity cases use its Scene, reference and
bars: fragments bit-exact against torch_ref.rasterize_meshes_soft, depth within 1e-5 of the largest |depth|, R / T gradients
within 1e-4 and vertex gradients within VERT_GRAD_RTOL of fp64 autograd of tests/soft_depth_ref.py on the kernels' fp32
projection.  Every case named after a branch asserts, from the launch profiler or the forward's counters, that it ran there.

1. blur_radius = 0 (PyTorch3D's default): the hard scatter with K-layer peeling and the exact shade pass in front of the blend,
   the hard clipped pass at the near plane, and the soft scatter selected by clipped barycentrics alone; every fragment lies
   inside its face (p >= 1/2), so the running sum passes 1 early and the forward's break is taken.
2. The blurred scatter's fallbacks: the whole-CTA walk of faces larger than BIG_FACE_PIX, and the in-place resolve of a full
   candidate queue (MVR_TEST_TINY_QUEUES), both with the previous layer's keys at K > 1.
3. K = 64 and 50 on three nested shells: lists full to the last entry, running sums that pass 1 past entry 16.
4. Odd and tall images: 1x1, 7x13, 33x31, 72x40 (H > W), 17x96.
5. Views that see nothing, zero cotangents, cotangents on empty pixels only (NaN included), expanded and strided cotangents.
6. depth_background 0, -3 and +-1e30; sigma = 1e-2 (well above the blur) and sigma = 1e-37, where the backward once formed
   inf * 0 = NaN; sigma = 1e8, where every p is exactly 1/2 and running sums of exactly 1 are everywhere; a subnormal sigma
   is refused by the entry points (9).
7. The mesh workspace's reuse hints with soft depth next to the other shaders, and the order of backwards.
8. MVRenderer(shader="soft_depth"): the redraw loop near the poles, cuda_graph=True, a per-vertex colour that requires grad.
9. (host, no GPU) the argument checks of mvr_mesh_soft_depth_forward / _backward, and B * M = 0.
10. mesh_soft_depth_kernel on hand-made fragment lists: exact probabilities 0, 1/2, 1 bit for bit against an fp32 emulation of
    its loop, random ones against the fp64 closed form.
"""

import numpy as np
import pytest
import torch

from mvtn_b200 import MVRenderer, _lib as L, ops, synth

from test_gpu_branches import VERT_GRAD_RTOL, expect_launches, launches
from test_gpu_depth_edges import pole_angles
from test_gpu_mesh_branches import SOFT
from test_gpu_parity import CUBE_F, CUBE_V
from test_gpu_soft_depth import BGD, DEPTH_RTOL, GRAD_RTOL, Scene, live_f32, rel, sigmoid_f32
from test_soft_depth_host import closed_form

gpu = pytest.mark.gpu
D = torch.float64
FWD_SOFT = {"mesh_scatter_kernel<3, true>": 1, "mesh_scatter_kernel<4, false>": 0}
FWD_HARD = {"mesh_scatter_kernel<4, false>": 1, "mesh_scatter_kernel<3, true>": 0}


def case(name, **kw):
    c = dict(SOFT[name])
    c.update(kw)
    return c


def run(sc, dev, g=None, flags=0, want=None, tag=""):
    """Forward (one per prefix of `want`, launches asserted) and backward to R, T and the vertices with cotangent g (default
    sc.g; "sum": depth.sum()) -> dict of detached results."""
    cam = tuple(torch.from_numpy(x).to(dev).requires_grad_() for x in (sc.R, sc.T, sc.Cc))
    vg = sc.vp.to(dev).requires_grad_()
    want = {"mesh_soft_depth_kernel": 1, **(want or {})}
    counts, out = {}, None
    for pfx in want:
        o, counts[pfx] = launches(pfx, lambda: sc.render(dev, verts=vg, cameras=cam, flags=flags))
        out = out or o
    expect_launches(counts, want, f"[{tag}] forward")
    depth, frag = out
    if isinstance(g, str):
        depth.sum().backward()
    else:
        depth.backward(sc.g.to(dev) if g is None else g)
    assert torch.equal(cam[2].grad, torch.zeros_like(cam[2]))
    return dict(depth=depth.detach(), frag=frag, gR=cam[0].grad, gT=cam[1].grad, gV=vg.grad, counts=counts)


def parity(oracle, dev, sc, tag, bars=("depth", "R", "T", "V"), **kw):
    """run() and the fp64 reference: fragments bit-exact, then the errors named in `bars` within their bars -> run's dict +
    reference and errors."""
    res = run(sc, dev, tag=tag, **kw)
    ref, gRr, gTr, gVr, rp2f, subst, stats = sc.reference(oracle, res["frag"]["dists"].cpu())
    assert torch.equal(res["frag"]["pix_to_face"].cpu().long(), rp2f), f"[{tag}] fragments differ from the reference rasterizer"
    errs = dict(depth=rel(res["depth"], ref), R=rel(res["gR"], gRr), T=rel(res["gT"], gTr), V=rel(res["gV"], gVr))
    covered = int((rp2f[..., 0] >= 0).sum())
    print(f"[{tag}] launches {res['counts']}  " + "  ".join(f"{k} {e:.1e}" for k, e in errs.items())
          + f"  clamp decisions taken from fp32: {subst[0]} of {covered} covered pixels  {stats}")
    bar = dict(depth=DEPTH_RTOL, R=GRAD_RTOL, T=GRAD_RTOL, V=VERT_GRAD_RTOL)
    for k in bars:
        assert errs[k] < bar[k], (tag, k, errs)
    assert subst[1] < 1e-5, subst
    res.update(ref=ref, gRr=gRr, gTr=gTr, gVr=gVr, errs=errs, stats=stats)
    return res


def host_lists(frag, sigma):
    """-> p2f, fp32 dists (numpy), valid, the kernels' c <= 1 decision, index of the first entry with c > 1 (-1: none)."""
    p2f, di = frag["pix_to_face"].cpu().numpy(), frag["dists"].cpu().numpy()
    valid = p2f >= 0
    live = live_f32(p2f, di, sigma)
    dead = valid & ~live
    return p2f, di, valid, live, np.where(dead.any(-1), dead.argmax(-1), -1)


# ------------------------------------------------------------------------------------------------- 1. blur 0
BLUR0 = {
    "ragged_k4": (case("ragged", K=4, blur=0.0),
                  {**FWD_HARD, "mesh_shade_kernel<true, 3, 1, false>": 1, "mesh_shade_clipped_kernel<true>": 0}),
    "near_plane_k6": (case("near_plane", K=6, blur=0.0),
                      {**FWD_HARD, "mesh_shade_kernel<true, 3, 1, false>": 1, "mesh_shade_clipped_kernel<false>": 1,
                       "mesh_shade_clipped_kernel<true>": 0}),
    "ragged_k4_clipped_bary": (case("ragged", K=4, blur=0.0, clip=True), {**FWD_SOFT, "mesh_shade_clipped_kernel<true>": 1}),
}


@gpu
@pytest.mark.parametrize("name", list(BLUR0))
def test_soft_depth_blur0(oracle, cuda_device, name):
    c, want = BLUR0[name]
    sc = Scene(oracle, c)
    res = parity(oracle, cuda_device, sc, f"blur 0 {name}", want=want)
    p2f, di, valid, live, first = host_lists(res["frag"], c["sigma"])
    assert (di[valid] <= 0).all(), "a fragment outside its face at blur 0"
    early = int(((valid & ~live).sum(-1) >= 2).sum())      # entries left after the one where the forward stops
    print(f"[blur 0 {name}] pixels stopping before their last valid entry: {early}")
    assert early > 0
    if sc.near:
        assert res["stats"]["clip1"] > 0 and res["stats"]["clip2"] > 0, res["stats"]


# ------------------------------------------------------------------------------------------------- 2. scatter fallbacks
CUBE_VIEWS = (torch.tensor([[30.0, 200.0]]), torch.tensor([[20.0, -40.0]]), torch.tensor([[1.7, 3.0]]))


def cube_scene(oracle, K):
    return Scene(oracle, dict(M=2, HW=(96, 96), K=K, blur=3e-3, sigma=1e-3, views=CUBE_VIEWS), meshes=[(CUBE_V, CUBE_F)])


@gpu
def test_soft_depth_big_face_walk(oracle, cuda_device):
    """The cube at 96^2 from 1.7 and 3.0: its faces' bboxes exceed BIG_FACE_PIX and the whole CTA walks them."""
    res = parity(oracle, cuda_device, cube_scene(oracle, 4), "cube big faces", want=FWD_SOFT)
    nbig = int(res["frag"]["counters"][L.CNT_BIG_FACES])
    print(f"[cube big faces] faces walked by the whole CTA: {nbig}")
    assert nbig > 0


@gpu
@pytest.mark.parametrize("name", ["ragged_k6", "cube_k6"])
def test_soft_depth_tiny_queues(oracle, cuda_device, name):
    """MVR_TEST_TINY_QUEUES: a round's candidate queue holds 40 pixels, the rest are resolved in place (with the previous
    layer's keys at K = 6); parity, and the fragments, depth and camera gradients of the run without the flag bit for bit."""
    dev = cuda_device
    sc = Scene(oracle, SOFT["ragged"]) if name == "ragged_k6" else cube_scene(oracle, 6)
    tiny = parity(oracle, dev, sc, f"tiny queues {name}", flags=L.TEST_TINY_QUEUES, want=FWD_SOFT)
    plain = run(sc, dev, tag=name)
    for k in ("pix_to_face", "zbuf", "dists", "bary_coords"):
        assert torch.equal(tiny["frag"][k], plain["frag"][k]), k
    for k in ("depth", "gR", "gT"):
        assert torch.equal(tiny[k], plain[k]), k
    if name == "cube_k6":
        assert int(tiny["frag"]["counters"][L.CNT_BIG_FACES]) > 0


# ------------------------------------------------------------------------------------------------- 3. K at the bound
def shells(nf, seed):
    """Three nested synth.make_mesh shells (scales 1, 0.8, 0.6) as one mesh: six surfaces behind the centre pixels."""
    vs, fs, off = [], [], 0
    for i, s in enumerate((1.0, 0.8, 0.6)):
        v, f = synth.make_mesh(nf, seed + i)
        vs.append(v * s)
        fs.append(f + off)
        off += v.shape[0]
    return torch.cat(vs), torch.cat(fs)


@gpu
@pytest.mark.parametrize("K", [64, 50])
def test_soft_depth_long_lists(oracle, cuda_device, K):
    """~3000 faces at 48^2, blur 1e-2 (2.4 px), sigma 1e-3: lists full to entry K, and running sums that first pass 1 past
    entry 16 -- where the forward's break and the backward's Z_stop search act."""
    c = dict(M=2, HW=(48, 48), K=K, blur=1e-2, sigma=1e-3, views=synth.learned_spherical_views(1, 2, 302))
    sc = Scene(oracle, c, meshes=[shells(1000, 301)])
    res = parity(oracle, cuda_device, sc, f"K={K} shells")
    _, _, valid, _, first = host_lists(res["frag"], c["sigma"])
    full, late = int(valid.all(-1).sum()), int((first > 16).sum())
    print(f"[K={K} shells] pixels with all {K} entries valid: {full}; first c > 1 past entry 16: {late} (deepest {first.max()})")
    assert full > 0 and late > 0


# ------------------------------------------------------------------------------------------------- 4. odd and tall shapes
@gpu
@pytest.mark.parametrize("H,W", [(1, 1), (7, 13), (33, 31), (72, 40), (17, 96)])
def test_soft_depth_odd_shapes(oracle, cuda_device, H, W):
    c = dict(meshes=[(400, 401)], M=2, HW=(H, W), K=4, blur=3e-3, sigma=1e-3)
    sc = Scene(oracle, c)
    res = parity(oracle, cuda_device, sc, f"{H}x{W}")
    assert (res["frag"]["pix_to_face"][:, H // 2, W // 2, 0] >= 0).all(), "the object does not cover the centre pixel"


# ------------------------------------------------------------------------------------------------- 5. empty and degenerate
@gpu
def test_soft_depth_nothing_in_view(oracle, cuda_device):
    """The ragged batch with mesh 1's two views turned away (the object 40 units aside, 40 units below): depth_background everywhere,
    pix_to_face -1, R / T gradients and mesh 1's vertex gradients exactly 0; the other meshes match the reference."""
    dev = cuda_device
    sc = Scene(oracle, SOFT["ragged"])
    sc.T = sc.T.copy()
    sc.T[2] = (40.0, 0.0, 2.2)
    sc.T[3] = (0.0, -40.0, 2.2)
    res = parity(oracle, dev, sc, "nothing in view")
    for n in (2, 3):
        assert torch.equal(res["depth"][n], torch.full_like(res["depth"][n], BGD)), n
        assert (res["frag"]["pix_to_face"][n] == -1).all(), n
        assert not res["gR"][n].any() and not res["gT"][n].any(), n
    v1 = slice(int(sc.voff[1]), int(sc.voff[2]))
    assert not res["gV"][v1].any() and res["gV"][: int(sc.voff[1])].any()
    assert all(bool((res["frag"]["pix_to_face"][n] >= 0).any()) for n in (0, 1, 4, 5))


@gpu
def test_soft_depth_degenerate_cotangents(oracle, cuda_device):
    """All-zero cotangent -> exactly zero gradients; a cotangent only on pixels without a fragment (NaN on some) -> exactly
    zero, and added to a full cotangent it leaves the camera gradients unchanged bit for bit; expanded (depth.sum(), expand)
    and strided (transposed, every other column) cotangents give the bits of their contiguous copies."""
    dev = cuda_device
    sc = Scene(oracle, SOFT["ragged"])
    full = run(sc, dev, tag="full")
    shape = full["depth"].shape
    zero = run(sc, dev, g=torch.zeros(shape, device=dev))
    for k in ("gR", "gT", "gV"):
        assert not zero[k].any(), k
    empty = (full["frag"]["pix_to_face"] < 0).all(-1)[:, None]
    assert int(empty.sum()) > 0
    ge = torch.where(empty, torch.randn(shape, device=dev, generator=torch.Generator(device=dev).manual_seed(9)), 0.0)
    ge.view(-1)[torch.nonzero(empty.view(-1))[::3, 0]] = float("nan")
    assert torch.isnan(ge).any()
    on_empty = run(sc, dev, g=ge)
    for k in ("gR", "gT", "gV"):
        assert torch.equal(on_empty[k], torch.zeros_like(on_empty[k])), k
    both = run(sc, dev, g=sc.g.to(dev) + ge)
    assert torch.equal(both["gR"], full["gR"]) and torch.equal(both["gT"], full["gT"])
    N, _, H, W = shape
    base = torch.randn(N, 1, W, 2 * H, device=dev, generator=torch.Generator(device=dev).manual_seed(10))
    for what, g in (("sum", "sum"), ("expand", torch.randn(1, 1, 1, 1, device=dev).expand(shape)),
                    ("transposed", base[..., :H].transpose(-1, -2)), ("strided", base.transpose(-1, -2)[:, :, ::2])):
        contiguous = torch.ones(shape, device=dev) if what == "sum" else g.contiguous()
        assert what == "sum" or not g.is_contiguous()
        a, b = run(sc, dev, g=g), run(sc, dev, g=contiguous)
        assert torch.equal(a["gR"], b["gR"]) and torch.equal(a["gT"], b["gT"]), what
        assert rel(a["gV"], b["gV"]) < 1e-5, what


# ------------------------------------------------------------------------------------------------- 6. sigma and background
@gpu
@pytest.mark.parametrize("bg", [0.0, -3.0])
def test_soft_depth_background_parity(oracle, cuda_device, bg):
    parity(oracle, cuda_device, Scene(oracle, SOFT["ragged"], bg=bg), f"background {bg}")


@gpu
@pytest.mark.parametrize("bg", [1e30, -1e30])
def test_soft_depth_huge_background(oracle, cuda_device, bg):
    """Uncovered pixels hold the background exactly, everything is finite, pixels whose background weight is 0 (fp64 sum
    >= 1 + 1e-5, clear of rounding) have the depth of the run with a background of 4 bit for bit, R / T within 1e-4."""
    dev = cuda_device
    c = SOFT["ragged"]
    res = parity(oracle, dev, Scene(oracle, c, bg=bg), f"background {bg:.0e}", bars=("depth", "R", "T"))
    bg4 = run(Scene(oracle, c, bg=BGD), dev)
    for k in ("depth", "gR", "gT", "gV"):
        assert torch.isfinite(res[k]).all(), k
    p2f, di = res["frag"]["pix_to_face"], res["frag"]["dists"]
    empty = (p2f < 0).all(-1)
    assert int(empty.sum()) > 0 and bool((res["depth"][:, 0][empty] == bg).all())
    c64 = (torch.sigmoid(-di.double() / c["sigma"]) * (p2f >= 0)).sum(-1)
    saturated = c64 >= 1 + 1e-5
    assert int(saturated.sum()) > 0
    assert torch.equal(res["depth"][:, 0][saturated], bg4["depth"][:, 0][saturated])


@gpu
def test_soft_depth_large_sigma(oracle, cuda_device):
    """sigma = 1e-2, well above the blur (3e-3): every p is close to 1/2, and the two faces of a shared edge, one inside and
    one outside at the same distance, sum to 1 up to rounding.  Pixels whose
    fp64 running sum comes within 1e-6 of 1 get a zero cotangent (the kernels' expf and the host mirror's exp may decide the
    clamp differently there, and the kernels skip a zero cotangent); parity on the rest."""
    dev = cuda_device
    c = case("ragged", sigma=1e-2)
    sc = Scene(oracle, c)
    frag = run(sc, dev)["frag"]
    p2f, di = frag["pix_to_face"].cpu(), frag["dists"].cpu()
    cs = (torch.sigmoid(-di.double() / c["sigma"]) * (p2f >= 0)).cumsum(-1)
    tie = (((cs - 1).abs() < 1e-6) & (p2f >= 0)).any(-1)
    covered = int((p2f[..., 0] >= 0).sum())
    sc.g = torch.where(tie[:, None], 0.0, sc.g)
    print(f"[sigma 1e-2] cotangent masked on {int(tie.sum())} of {covered} covered pixels")
    assert int(tie.sum()) < 0.5 * covered
    parity(oracle, dev, sc, "sigma 1e-2")


@gpu
def test_soft_depth_tiny_sigma(oracle, cuda_device):
    """sigma = 1e-37 (a normal float) at the default background of 100: every p is 0 or 1, and g (z - Z_stop) / sigma overflows.
    Multiplied by p (1 - p) = 0 only after that, the backward gave NaN; the gradients are finite and match the reference."""
    dev = cuda_device
    res = parity(oracle, dev, Scene(oracle, case("ragged", sigma=1e-37), bg=100.0), "sigma 1e-37")
    for k in ("gR", "gT", "gV"):
        assert torch.isfinite(res[k]).all(), k
    assert res["gR"].abs().max() > 0


@gpu
def test_soft_depth_exact_ties(oracle, cuda_device):
    """sigma = 1e8: every |dists| / sigma is below 1e-9, so expf(dists / sigma) is exactly 1 and every fragment has p = 1/2
    exactly, in the kernels and on the host alike.  Every pixel with two or more fragments then reaches a running sum of exactly
    1 at its second entry, where torch's clamp passes the gradient (the backward's c <= 1): that fragment's distance term
    g (z - Z_stop) p (1 - p) / sigma counts.  With a background of 4e8 the term is of the order of g, and at a pixel with exactly
    two fragments it balances the first fragment's term across their shared edge; without it the camera and vertex gradients
    move by about 1e-2 of their largest entry.  Parity on the ragged batch, with the clamp decisions identical on both sides."""
    c = case("ragged", sigma=1e8)
    res = parity(oracle, cuda_device, Scene(oracle, c, bg=4e8), "exact ties")
    p2f, di, valid, _, _ = host_lists(res["frag"], c["sigma"])
    p = np.where(valid, sigmoid_f32(di, c["sigma"]), np.float32(0.0))
    assert (p[valid] == 0.5).all()
    ties = int(((np.cumsum(p, -1, dtype=np.float32) == 1.0) & valid).any(-1).sum())
    only_two = int((valid.sum(-1) == 2).sum())
    print(f"[exact ties] pixels whose running sum is exactly 1 at a valid entry: {ties}; with exactly two fragments: {only_two}")
    assert ties > 100 and only_two > 0


# ------------------------------------------------------------------------------------------------- 7. workspace reuse
@gpu
def test_soft_depth_workspace_reuse(oracle, cuda_device):
    """ops._ws_mesh's hints are keyed by the layout (B, M, H, W, K, total_verts), not by the shader: soft depth at K = 1 shares
    the layout of hard Phong and hard depth, at K = 2 that of soft Phong.  A fixed interleaving with a point render, far and
    near-plane views, gives every output and fragment of its cold-workspace reference bit for bit, and takes the armed hint into
    soft depth and out of it.  The soft depth backward re-projects into the shared buffer (a non-owner workspace() call): right
    after its forward, behind a forward of other views, and a hard Phong backward issued behind it must re-project too."""
    dev = cuda_device
    key = (dev.index, ops._stream(dev))
    H, M = 48, 3
    m = synth.make_meshes(2, 1500, 61)
    geom = ops.PackedMeshes([v for v, _ in m], [f for _, f in m], dev)
    far = (torch.tensor([[15.0, 140.0, -80.0], [200.0, 33.0, 77.0]]), torch.tensor([[10.0, -35.0, 50.0], [0.0, 20.0, -15.0]]),
           torch.tensor([[2.2, 2.0, 2.5], [1.9, 2.25, 3.0]]))
    near = (far[0] + 30.0, far[1], torch.tensor([[1.12, 1.2, 1.3], [1.15, 1.25, 1.18]]))
    cam = {}
    for name, (a, e, d) in (("far", far), ("near", near)):
        R, T, C = oracle.look_at(*(t.numpy().ravel() for t in (a, e, d)))
        cam[name] = tuple(torch.from_numpy(x).to(dev) for x in (R, T, C))
    col = torch.full((3,), 0.99999, device=dev)
    light = torch.tensor([[0, 1.0, 0]], device=dev)
    pts = synth.make_clouds(2, 256, 62).to(dev)
    K_OF = {"phong": 1, "depth": 1, "soft_depth1": 1, "soft_depth2": 2, "soft_phong": 2}

    def render(shader, views, R=None, T=None):
        Rv, Tv, Cv = cam[views]
        R, T = (Rv if R is None else R), (Tv if T is None else T)
        if shader == "phong":
            return ops.render_meshes(geom, M, R, T, Cv, light, col, col, H, fragments=True)
        if shader == "depth":
            return ops.render_meshes(geom, M, R, T, Cv, light, col, col, H, shader="hard_depth", depth_background=BGD)
        if shader == "soft_phong":
            return ops.render_meshes(geom, M, R, T, Cv, light, col, col, H, faces_per_pixel=2, shader="soft_phong", blur_radius=1e-4)
        return ops.render_meshes(geom, M, R, T, Cv, light, col, col, H, faces_per_pixel=K_OF[shader], shader="soft_depth",
                                 blur_radius=1e-4, sigma=1e-4, depth_background=BGD)

    def snapshot(img, fr):
        return [img.detach().clone()] + [v.clone() for k, v in sorted(fr.items()) if k != "counters" and v is not None]

    ref = {}
    for shader in K_OF:
        for views in ("far", "near"):
            ops._ws_mesh.pop(key, None)
            img, fr = render(shader, views)
            ref[shader, views] = snapshot(img, fr)
            if views == "near":
                assert int(fr["counters"][L.CNT_STRADDLE]) > 0, shader
    ops._ws_mesh.pop(key, None)
    seq = [("soft_depth1", "near"), ("phong", "far"), ("soft_depth1", "far"), ("depth", "near"), ("soft_depth1", "near"),
           ("points", "far"), ("soft_depth2", "far"), ("soft_phong", "near"), ("soft_depth2", "near"), ("soft_phong", "far"),
           ("soft_depth1", "far"), ("phong", "near"), ("soft_depth2", "far"), ("soft_depth1", "near"), ("depth", "far"),
           ("soft_depth2", "near")]
    taken, prev = {}, None
    for i, (shader, views) in enumerate(seq):
        if shader == "points":
            Rv, Tv, _ = cam[views]
            ops.render_points(pts, col, M, Rv, Tv, None, 0.02, col * 0, H, dist=far[2].to(dev).reshape(-1))
            assert ops._ws_mesh.get(key) is None
            prev = shader
            continue
        st = ops._ws_mesh.get(key)
        ws = ops._workspaces.get(key)
        layout = (geom.B, M, H, H, K_OF[shader], geom.total_verts)
        hit = isinstance(st, dict) and ws is not None and st.get("armed") == (ws.data_ptr(), layout)
        taken[prev, shader] = taken.get((prev, shader), 0) + int(hit)
        out = snapshot(*render(shader, views))
        for j, (a, b) in enumerate(zip(out, ref[shader, views])):
            assert torch.equal(a, b), (i, shader, views, j)
        prev = shader
    print(f"armed hints taken: {taken}")
    into = sum(n for (a, b), n in taken.items() if b.startswith("soft_depth") and not str(a).startswith("soft_depth"))
    out_of = sum(n for (a, b), n in taken.items() if str(a).startswith("soft_depth") and not b.startswith("soft_depth"))
    assert into >= 1 and out_of >= 1, taken
    other = {"near": "far", "far": "near"}
    cot = torch.randn(2 * M, 1, H, H, device=dev, generator=torch.Generator(device=dev).manual_seed(5))

    def soft_depth_grads(views, mode):
        Rg, Tg = (t.clone().requires_grad_() for t in cam[views][:2])
        if mode == "cold":
            ops._ws_mesh.pop(key, None)
        dep, _ = render("soft_depth2", views, Rg, Tg)
        if mode == "cold":
            ops._ws_mesh.pop(key, None)
        elif mode == "behind_other_views":
            render("phong", other[views])
        _, n = launches("mesh_project_kernel", lambda: dep.backward(cot))
        assert n == 1, (views, mode, n)
        return Rg.grad, Tg.grad

    cot_img = torch.randn(2 * M, 3, H, H, device=dev, generator=torch.Generator(device=dev).manual_seed(6))

    def phong_grads(views, behind_soft_depth):
        Rg, Tg = (t.clone().requires_grad_() for t in cam[views][:2])
        if behind_soft_depth:
            Rs, Ts = (t.clone().requires_grad_() for t in cam[other[views]][:2])
            dep, _ = render("soft_depth1", other[views], Rs, Ts)
        else:
            ops._ws_mesh.pop(key, None)
        img, _ = render("phong", views, Rg, Tg)
        if behind_soft_depth:
            dep.backward(cot)      # re-projects the other views into the shared buffer
        else:
            ops._ws_mesh.pop(key, None)
        _, n = launches("mesh_project_kernel", lambda: img.backward(cot_img))
        assert n == 1, (views, behind_soft_depth, n)
        return Rg.grad, Tg.grad

    for views in ("near", "far"):
        cold = soft_depth_grads(views, "cold")
        assert float(cold[0].abs().max()) > 0
        for mode in ("warm", "behind_other_views"):
            got = soft_depth_grads(views, mode)
            assert torch.equal(got[0], cold[0]) and torch.equal(got[1], cold[1]), (views, mode)
        cold = phong_grads(views, False)
        got = phong_grads(views, True)
        assert torch.equal(got[0], cold[0]) and torch.equal(got[1], cold[1]), (views, "phong behind soft depth")


# ------------------------------------------------------------------------------------------------- 8. MVRenderer
RKW = dict(pc_rendering=False, light_direction="fixed", faces_per_pixel=4, shader="soft_depth", blur_radius=2e-3, blend_sigma=2e-4,
           depth_background=BGD)


def ops_soft_depth(geom, M, R, T, C, H):
    dev = geom.device
    return ops.render_meshes(geom, M, R, T, C, torch.ones(1, 3, device=dev), None, torch.zeros(3, device=dev), H, faces_per_pixel=4,
                             shader="soft_depth", blur_radius=2e-3, sigma=2e-4, depth_background=BGD)[0]


@gpu
def test_soft_depth_mvrenderer_redraw_loop(cuda_device):
    """Views at and next to the poles: the redraw loop renders again; the depth is the ops-level depth of the returned cameras
    bit for bit, and the angle gradients are finite."""
    dev = cuda_device
    torch.manual_seed(0)
    B, M, H = 2, 6, 48
    az, el, di = (t.to(dev).requires_grad_() for t in pole_angles(B, M))
    r = MVRenderer(M, image_size=H, **RKW).eval()
    obj = [(v.to(dev), f.to(dev)) for v, f in synth.make_meshes(B, 800, 72)]
    (img, cameras), k = launches("look_at_forward", lambda: r(obj, None, az, el, di))
    assert k >= 2, "the redraw loop did not run"
    geom = ops.PackedMeshes([v for v, _ in obj], [f for _, f in obj], dev)
    ref = ops_soft_depth(geom, M, cameras.R.detach(), cameras.T.detach(), cameras.get_camera_center().detach(), H)
    assert torch.equal(img.detach().reshape(B * M, 1, H, H), ref)
    assert (ref < BGD - 1e-3).sum() > 100
    g = torch.randn(B, M, 1, H, H, generator=torch.Generator().manual_seed(3)).to(dev)
    (img * g).sum().backward()
    for t in (az, el, di):
        assert t.grad is not None and torch.isfinite(t.grad).all()
    assert float(el.grad.abs().max()) > 0


@gpu
def test_soft_depth_mvrenderer_cuda_graph_and_colour(cuda_device):
    """cuda_graph=True with a collated batch: the soft depth step stays eager (the full fragments are kept) and gives the bits
    of cuda_graph=False, angle gradients included.  A per-vertex colour that requires grad leaves the depth unchanged bit for
    bit and gets no gradient (its .grad stays None: the depth does not depend on it); so does one object colour."""
    dev = cuda_device
    B, M, H = 2, 3, 40
    meshes = [synth.make_mesh(500 + 200 * b, 80 + b) for b in range(B)]
    views = synth.learned_spherical_views(B, M, 82)
    g = torch.randn(B, M, 1, H, H, generator=torch.Generator().manual_seed(83)).to(dev)
    out = {}
    for graph in (False, True, True):
        r = MVRenderer(M, image_size=H, cuda_graph=graph, **RKW).eval()
        a, e, d = (t.clone().to(dev).requires_grad_() for t in views)
        img, _ = r(ops.collate_meshes(meshes), None, a, e, d)
        assert "dists" in r.last_fragments, "the soft depth step was replayed from a CUDA graph"
        (img * g).sum().backward()
        out.setdefault(graph, []).append((img.detach(), a.grad, e.grad, d.grad))
    for got in out[True]:
        for x, y in zip(got, out[False][0]):
            assert torch.equal(x, y)
    # per-vertex colours that require grad
    nv = max(v.shape[0] for v, _ in meshes)
    colour = torch.rand(B, nv, 3, generator=torch.Generator().manual_seed(84)).to(dev).requires_grad_()
    r = MVRenderer(M, image_size=H, object_color="custom", **RKW).eval()
    a, e, d = (t.clone().to(dev).requires_grad_() for t in views)
    img, _ = r([(v.to(dev), f.to(dev)) for v, f in meshes], None, a, e, d, color=colour)
    assert torch.equal(img.detach(), out[False][0][0])
    (img * g).sum().backward()
    assert colour.grad is None
    assert torch.equal(a.grad, out[False][0][1])
    # one object colour that requires grad
    colour = torch.tensor([0.3, 0.6, 0.9], device=dev, requires_grad=True)
    a, e, d = (t.clone().to(dev).requires_grad_() for t in views)
    img, _ = r([(v.to(dev), f.to(dev)) for v, f in meshes], None, a, e, d, color=colour)
    assert torch.equal(img.detach(), out[False][0][0])
    (img * g).sum().backward()
    assert colour.grad is None
    assert torch.equal(a.grad, out[False][0][1])


# ------------------------------------------------------------------------------------------------- 9. host: argument checks
FAKE = 1 << 20      # never dereferenced: every call below is refused before any CUDA call


def _fwd_args(**kw):
    a = dict(B=1, M=2, H=16, W=16, K=4, sigma=1e-3, bg=100.0, p2f=FAKE, zbuf=FAKE, dists=FAKE, depth=FAKE, stream=None)
    a.update(kw)
    return list(a.values())


def _bwd_args(lib, **kw):
    a = dict(geometry=FAKE, vert_off=FAKE, face_off=FAKE, B=1, M=2, tv=30, tf=40, max_verts=30, R=FAKE, T=FAKE, k00=1.7, k11=1.7,
             z_clip=0.5, blur=1e-3, H=16, W=16, K=4, flags=0, sigma=1e-3, bg=100.0, p2f=FAKE, grad_depth=FAKE, gR=FAKE, gT=FAKE,
             grad_verts=None, ws=FAKE, ws_bytes=None, stream=None)
    a.update(kw)
    if a["ws_bytes"] is None:
        a["ws_bytes"] = lib.mvr_mesh_workspace_bytes(a["B"], a["M"], a["H"], a["W"], a["K"], a["tv"], a["tf"])
    return list(a.values())


NAN, INF = float("nan"), float("inf")
COMMON = [(dict(sigma=0.0), -7, b"sigma"), (dict(sigma=-1.0), -7, b"sigma"), (dict(sigma=NAN), -7, b"sigma"),
          (dict(sigma=1e-40), -7, b"sigma"), (dict(bg=INF), -7, b"depth_background"), (dict(bg=-INF), -7, b"depth_background"),
          (dict(bg=NAN), -7, b"depth_background"), (dict(K=0), -3, b"faces_per_pixel"), (dict(K=65), -3, b"faces_per_pixel"),
          (dict(H=0), -2, b"image size"), (dict(W=0), -2, b"image size"), (dict(H=4097), -2, b"image size"),
          (dict(W=4097), -2, b"image size")]
FWD_ONLY = [(dict(p2f=None), -5, b"null pointer"), (dict(zbuf=None), -5, b"null pointer"), (dict(dists=None), -5, b"null pointer"),
            (dict(depth=None), -5, b"null pointer")]
BWD_ONLY = [(dict(blur=-1e-3), -9, b"blur_radius"), (dict(blur=NAN), -9, b"blur_radius"), (dict(flags=L.IMAGES_BF16), -11, b"fp32"),
            (dict(geometry=None), -5, b"null pointer"), (dict(R=None), -5, b"null pointer"), (dict(grad_depth=None), -5, b"null pointer"),
            (dict(gT=None), -5, b"null pointer"), (dict(ws=None), -5, b"null pointer")]


@pytest.mark.skipif(torch.cuda.is_available(), reason="the pointers are fake: they must never reach a device")
@pytest.mark.parametrize("entry", ["forward", "backward"])
def test_soft_depth_argument_checks(entry):
    """Each bad argument alone: a negative status, the message naming it, no launch.  A subnormal sigma (1e-40) is refused
    like 0: 1 / sigma overflows.  B * M = 0 is a no-op that returns 0 before looking at any pointer."""
    lib = L.load()
    fn = lib.mvr_mesh_soft_depth_forward if entry == "forward" else lib.mvr_mesh_soft_depth_backward
    cases = COMMON + (FWD_ONLY if entry == "forward" else BWD_ONLY)
    if entry == "backward":
        cases = cases + [(dict(ws_bytes=lib.mvr_mesh_workspace_bytes(1, 2, 16, 16, 4, 30, 40) - 1), -8, b"workspace too small")]
    for kw, code, what in cases:
        args = _fwd_args(**kw) if entry == "forward" else _bwd_args(lib, **kw)
        n0 = lib.mvr_launch_count()
        rc = fn(*args)
        msg = lib.mvr_last_error_string()
        assert rc == code, (entry, kw, rc, msg)
        assert what in msg and f"mvr_mesh_soft_depth_{entry}".encode() in msg, (entry, kw, msg)
        assert lib.mvr_launch_count() == n0
    for B, M in ((0, 2), (1, 0)):
        n0 = lib.mvr_launch_count()
        none = dict(p2f=None, zbuf=None, dists=None, depth=None) if entry == "forward" else \
            dict(geometry=None, vert_off=None, face_off=None, R=None, T=None, p2f=None, grad_depth=None, gR=None, gT=None, ws=None, ws_bytes=0)
        args = _fwd_args(B=B, M=M, **none) if entry == "forward" else _bwd_args(lib, B=B, M=M, **none)
        assert fn(*args) == 0 and lib.mvr_launch_count() == n0


@pytest.mark.skipif(torch.cuda.is_available(), reason="the pointers are fake: they must never reach a device")
def test_soft_blend_entry_points_refuse_a_subnormal_sigma():
    """mvr_mesh_soft_blend_forward / mvr_mesh_soft_backward: a subnormal (1e-40) or zero sigma is refused with -7 and a message
    naming sigma; FLT_MIN passes the sigma check -- the same call is then refused for its gamma of 0 (-7, a message naming gamma
    and not sigma), so no valid call is ever made here."""
    lib = L.load()
    for sigma, sigma_ok in ((1e-40, False), (0.0, False), (1.1754944e-38, True)):
        n0 = lib.mvr_launch_count()
        rc = lib.mvr_mesh_soft_blend_forward(FAKE, FAKE, FAKE, 1, 1, 3, 1, FAKE, FAKE, 0, FAKE, FAKE, 16, 16, 4, 0, 1, sigma, 0.0,
                                             1.0, 100.0, FAKE, FAKE, FAKE, FAKE, FAKE, None)
        msg = lib.mvr_last_error_string()
        assert rc == -7 and lib.mvr_launch_count() == n0, (sigma, rc)
        assert (b"sigma" not in msg and b"gamma" in msg) if sigma_ok else b"sigma must be a normal float" in msg, (sigma, msg)
        rc = lib.mvr_mesh_soft_backward(FAKE, FAKE, FAKE, 1, 1, 3, 1, 3, FAKE, FAKE, FAKE, FAKE, 0, FAKE, FAKE, 1.7, 1.7, 0.5, 1e-3,
                                        16, 16, 4, 0, 1, sigma, 1e-4, 1.0, 100.0, FAKE, FAKE, FAKE, FAKE, FAKE, None, None,
                                        FAKE, 0, None)
        msg = lib.mvr_last_error_string()
        # with a normal sigma the zero workspace size is what is refused
        assert rc == (-8 if sigma_ok else -7) and lib.mvr_launch_count() == n0, (sigma, rc)
        assert (b"workspace too small" if sigma_ok else b"sigma must be a normal float") in msg, (sigma, msg)


# ------------------------------------------------------------------------------------------------- 10. synthetic fragments
def emulate_f32(p2f, zbuf, dists, sigma, bg):
    """mesh_soft_depth_kernel's loop in numpy fp32 (exact for p in {0, 1/2, 1}: every product is exact, FMA or not)."""
    p = sigmoid_f32(dists, sigma)
    N, H, W, K = p2f.shape
    out = np.empty((N, 1, H, W), np.float32)
    one, f = np.float32(1.0), np.float32
    for n, y, x in np.ndindex(N, H, W):
        c = mprev = d = f(0.0)
        for k in range(K):
            if p2f[n, y, x, k] < 0:
                continue
            c = f(c + p[n, y, x, k])
            m = min(c, one)
            d = f(d + f((m - mprev) * zbuf[n, y, x, k]))
            mprev = m
            if c > one:
                break
        out[n, 0, y, x] = f(d + f((one - mprev) * f(bg)))
    return out


def synthetic(K, seed, exact, sigma, B=2, M=3, H=7, W=9):
    """Hand-made lists, -1 holes anywhere (30 %).  exact: dists in {0, +-1e3 sigma} (p = 1/2, 0, 1); the entries past the first
    with c > 1 are poisoned with NaN (the forward must not read them).  Otherwise dists ~ 2 sigma N(0, 1)."""
    rs = np.random.RandomState(seed)
    shape = (B * M, H, W, K)
    p2f = np.where(rs.rand(*shape) < 0.3, -1, rs.randint(0, 1000, shape)).astype(np.int32)
    zbuf = np.sort(1 + 3 * rs.rand(*shape), -1).astype(np.float32)
    if exact:
        dists = (np.float32(1e3 * sigma) * rs.choice(np.array([0, 0, 1, -1], np.float32), shape)).astype(np.float32)
        p = np.where(p2f >= 0, sigmoid_f32(dists, sigma), 0).astype(np.float32)
        assert set(np.unique(p)) <= {0.0, 0.5, 1.0}
        past = np.cumsum(np.cumsum(p, -1) > 1, -1) > 1      # strictly past the first entry with c > 1 (sums of halves: exact)
        zbuf[past & (p2f >= 0)] = np.nan
        dists[past & (p2f >= 0)] = np.nan
    else:
        dists = (2 * sigma * rs.randn(*shape)).astype(np.float32)
    dists[p2f < 0] = -1.0
    zbuf[p2f < 0] = -1.0
    return p2f, zbuf, dists


def soft_depth_forward(dev, p2f, zbuf, dists, sigma, bg, M=3):
    lib = L.load()
    N, H, W, K = p2f.shape
    t = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (p2f, zbuf, dists)]
    out = torch.full((N, 1, H, W), -7.0, device=dev)
    L.check(lib.mvr_mesh_soft_depth_forward(N // M, M, H, W, K, sigma, bg, *(x.data_ptr() for x in t), out.data_ptr(),
                                            torch.cuda.current_stream(dev).cuda_stream), "mvr_mesh_soft_depth_forward")
    return out.cpu().numpy()


@gpu
@pytest.mark.parametrize("K", [1, 2, 3, 17, 64])
def test_soft_depth_forward_exact_probabilities(cuda_device, K):
    sigma, bg = 1e-3, 7.5
    p2f, zbuf, dists = synthetic(K, 500 + K, True, sigma)
    got = soft_depth_forward(cuda_device, p2f, zbuf, dists, sigma, bg)
    want = emulate_f32(p2f, zbuf, dists, sigma, bg)
    p = np.where(p2f >= 0, sigmoid_f32(np.nan_to_num(dists), sigma), 0)
    cs = np.cumsum(p, -1)
    ties = int(((cs == 1) & (p2f >= 0)).any(-1).sum())
    print(f"[K={K}] pixels whose running sum is exactly 1 at a valid entry: {ties}; empty pixels: {int((p2f < 0).all(-1).sum())}")
    if K > 1:
        assert ties > 0
    assert np.isfinite(got).all()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@gpu
@pytest.mark.parametrize("K", [1, 2, 3, 17, 64])
def test_soft_depth_forward_random_probabilities(cuda_device, K):
    sigma, bg = 1e-3, 7.5
    p2f, zbuf, dists = synthetic(K, 600 + K, False, sigma)
    got = soft_depth_forward(cuda_device, p2f, zbuf, dists, sigma, bg)
    t = lambda x: torch.from_numpy(x)
    g = torch.zeros(p2f.shape[:3] + (1,), dtype=D)
    ref = closed_form(t(p2f).long(), t(zbuf).to(D), t(dists).to(D), sigma, bg, g)[0][..., 0].numpy()
    err = float(np.abs(got[:, 0] - ref).max() / np.abs(ref).max())
    print(f"[K={K}] random probabilities: depth {err:.1e}")
    assert err < 1e-6
