"""Randomised parity sweep on the GPU: many small random mesh / point configurations (random image sizes incl. odd ones, K, radius,
camera distances down to the near plane, triangle soups with slivers / duplicates / huge faces, perspective on / off, culling,
both forward rasterizers) through tests/test_gpu_parity.py's run_mesh / run_points, i.e. bit-exact fragments and toleranced images /
gradients against the C oracle.  Prints the failing seeds.   usage: python scripts/fuzz_parity.py [cases] [first_seed] [soup|smooth|mix]

Fragments, depths, barycentrics and images are held to the tests' bars (bit-exact / 1e-5).  Gradients: smooth meshes and clouds to
2e-4 of the largest entry; a triangle soup with slivers is far worse conditioned than anything the renderer is fed (d bary / d vertex
~ 1 / area), so there the error is compared with the fp32 FLOOR of the case -- the same formulas under torch.autograd in fp32 vs fp64
(oracle/torch_ref.py, as scripts/fp32_gradient_floor.py does) -- and a case fails when it is more than 30x above it."""
import os, sys, traceback
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_gpu_parity as T
from mvtn_b200 import synth
from oracle import oracle as orc

orc.build()
dev = torch.device("cuda:0")
# gradient errors are RECORDED (the worst relative error of a case is printed) and judged here, not by the tests' fixed bars: a random
# soup of slivers is far worse conditioned than anything the renderer is fed, and the sweep should say by how much
_rel, _seen = T.rel, []
def _rec(a, b, floor=1e-6):
    # Recorded as (largest error, largest reference entry) per tensor and judged per CASE (_worst below): a tensor is compared with its
    # own largest entry, but never with less than 0.5, nor with less than 1e-3 of the largest gradient entry of the case.  Two kinds of
    # tensors would otherwise compare rounding noise with rounding noise: an analytically vanishing gradient (every visible face unlit
    # under one object colour, one point colour under the norm compositor: the image is a constant), and a sum that happens to cancel
    # (d loss / d scale = 0.56 next to d loss / d T = 1970 in the same view: 3e-4 of absolute error is 1.6e-7 of its terms).
    a64 = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, np.float64); b64 = np.asarray(b, np.float64)
    _seen.append((float(np.abs(a64 - b64).max()), float(np.abs(b64).max())))
    return 0.0


def _worst():
    scale = max((m for _, m in _seen), default=0.0)
    return max((e / max(m, 0.5, 1e-3 * scale) for e, m in _seen), default=0.0)


T.rel = _rec
T.GRAD_RTOL = T.POINT_GRAD_RTOL = float("inf")
T.IMG_ATOL = float("inf")      # (checked below, so that a failure says by how much and where)
GRAD_BAR = 2e-4
n_cases = int(sys.argv[1]) if len(sys.argv) > 1 else 120
seed0 = int(sys.argv[2]) if len(sys.argv) > 2 else 0
kind_of_mesh = sys.argv[3] if len(sys.argv) > 3 else "mix"
from oracle import torch_ref as tr


def fp32_floor(cfg):
    """max over (gR, gT, gC) of |fp32 autograd - fp64 autograd| / max|fp64| for a K = 1 perspective case, fragments from the oracle."""
    meshes, M, H = cfg["meshes"], cfg["M"], cfg["H"]
    R, Tt, C = orc.look_at(*(t.numpy().ravel() for t in cfg["views"]))
    vp, fp, voff, foff = T.pack_np(meshes)
    nrm = orc.packed_vertex_normals(vp, fp, voff, foff)
    light = C.copy() if cfg.get("light") == "relative" else np.array([cfg.get("light_dir", [0.3, 1.0, -0.5])], np.float32)
    bg = np.array([0.5, 0.25, 0.75], np.float32)
    rgb = np.full(3, 0.99999, np.float32)
    flags = orc.PERSPECTIVE_CORRECT | (orc.CULL_BACKFACES if cfg["cull"] else 0)
    o = orc.mesh_forward(vp, fp, voff, foff, nrm, rgb, M, R, Tt, C, light, bg, T.K00, T.K11, 0.5, H, H, 1, flags)
    gimg = torch.randn(len(meshes) * M, 3, H, H, generator=torch.Generator().manual_seed(5)).numpy()
    out = []
    for dtype in (torch.float32, torch.float64):
        Rd, Td, Cd = (torch.from_numpy(x).to(dtype).requires_grad_() for x in (R, Tt, C))
        loss = 0
        for b, (v, f) in enumerate(meshes):
            nb = torch.from_numpy(nrm[voff[b]:voff[b + 1]]).to(dtype)
            col = torch.from_numpy(np.broadcast_to(rgb, (v.shape[0], 3)).copy()).to(dtype)
            for m in range(M):
                n = b * M + m
                img, _ = tr.render_mesh_view(v.to(dtype), f, nb, col, Rd[n], Td[n], Cd[n], torch.from_numpy(light[n if light.shape[0] > 1 else 0]).to(dtype),
                                             torch.from_numpy(bg).to(dtype), T.K00, T.K11, H, H, p2f=torch.from_numpy(o["pix_to_face"][n, ..., 0]).long())
                loss = loss + (img * torch.from_numpy(gimg[n]).to(dtype)).sum()
        loss.backward()
        out.append([t.grad.double().numpy() for t in (Rd, Td, Cd)])
    return max(float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-6)) for a, b in zip(*out))


def soup(rng, nf):
    """Random triangle soup in the unit ball: a share of slivers, tiny, huge and duplicated faces."""
    v = rng.normal(size=(3 * nf, 3)).astype(np.float32)
    v /= np.maximum(np.linalg.norm(v, axis=1, keepdims=True), 1e-6)
    v *= rng.uniform(0.05, 1.0, size=(3 * nf, 1)).astype(np.float32)
    f = np.arange(3 * nf, dtype=np.int64).reshape(nf, 3)
    kind = rng.integers(0, 5, nf)
    for i in np.nonzero(kind == 0)[0]:      # sliver: third vertex almost on the first edge
        t = rng.uniform(0, 1)
        v[3 * i + 2] = v[3 * i] * (1 - t) + v[3 * i + 1] * t + rng.normal(size=3).astype(np.float32) * 1e-4
    for i in np.nonzero(kind == 1)[0]:      # tiny (sub-pixel) face
        v[3 * i + 1] = v[3 * i] + rng.normal(size=3).astype(np.float32) * 5e-3
        v[3 * i + 2] = v[3 * i] + rng.normal(size=3).astype(np.float32) * 5e-3
    if nf > 4:                              # exact duplicates (the (z, face) tie rule) and a degenerate face
        f[1] = f[0]
        f[2] = np.array([f[3][0], f[3][0], f[3][1]])
    return torch.from_numpy(v), torch.from_numpy(f)


def views(rng, B, M, near):
    az = torch.from_numpy(rng.uniform(-180, 180, (B, M)).astype(np.float32))
    el = torch.from_numpy(rng.uniform(-80, 80, (B, M)).astype(np.float32))
    lo = 0.7 if near else 1.6
    di = torch.from_numpy(rng.uniform(lo, 3.0, (B, M)).astype(np.float32))
    return az, el, di


def mesh_case(rng, kind):
    """One random mesh configuration -> (cfg for run_mesh, near, any_soup)."""
    B, M = int(rng.integers(1, 4)), int(rng.integers(1, 4))
    H = int(rng.choice([8, 17, 31, 32, 33, 48, 50, 64, 97, 128]))
    K = int(rng.choice([1, 1, 1, 2, 3]))
    near = bool(rng.integers(0, 3) == 0)
    meshes, any_soup = [], False
    for b in range(B):
        is_soup = bool(rng.integers(0, 2)) if kind == "mix" else kind == "soup"
        any_soup = any_soup or is_soup
        if is_soup:
            meshes.append(soup(rng, int(rng.integers(1, 400))))
        else:
            meshes.append(synth.make_mesh(int(rng.integers(20, 5000)), int(rng.integers(0, 1 << 30)), amplitude=float(rng.uniform(0, 0.5))))
    cfg = dict(meshes=meshes, M=M, H=H, K=K, views=views(rng, B, M, near), persp=bool(rng.integers(0, 4) != 0),
               cull=bool(rng.integers(0, 4) == 0))
    if rng.integers(0, 2):
        cfg["light"] = "relative"      # lit from the camera: the visible faces are lit, the gradients are not ~0
    else:
        cfg["light_dir"] = [float(x) for x in rng.normal(size=3)]
    return cfg, near, any_soup


fails, n_highlight = [], 0
for case in (range(seed0, seed0 + n_cases) if __name__ == "__main__" else ()):
    rng = np.random.default_rng(10_000 + case)
    try:
        if case % 3 != 2:
            cfg, near, any_soup = mesh_case(rng, kind_of_mesh)
            meshes, B, M, H, K = cfg["meshes"], len(cfg["meshes"]), cfg["M"], cfg["H"], cfg["K"]
            res = T.run_mesh(orc, dev, cfg, backward=True)
            d = np.abs(res["img"].detach().cpu().numpy() - res["o"]["images"])
            hl = ""
            if 1e-5 < d.max() <= 1.5e-5 and int((d > 1e-5).sum()) <= 6 and res["o"]["images"][d > 1e-5].min() > 0.9:
                # one or two saturated highlight pixels: alpha^64 multiplies the rounding differences of two fp32 evaluation orders by 64 --
                # the oracle itself is 6e-6 away from an fp64 evaluation there (DESIGN.md section 2); counted, not failed
                hl = f" [highlight pixel {d.max():.3e}]"; n_highlight += 1
            elif d.max() > 1e-5:
                n, c, y, x = np.unravel_index(d.argmax(), d.shape)
                raise AssertionError(f"image error {d.max():.3e} at view {n} channel {c} pixel ({y}, {x}): got {float(res['img'][n, c, y, x]):.7f} "
                                     f"want {res['o']['images'][n, c, y, x]:.7f}, face {int(res['p2f'][n, y, x, 0])}, {int((d > 1e-5).sum())} values over 1e-5")
            what = f"mesh soup={any_soup} light={cfg.get('light', 'fixed')} B={B} M={M} H={H} K={K} near={near} persp={cfg['persp']} cull={cfg['cull']} F={[int(f.shape[0]) for _, f in meshes]}"
        else:
            B, M = int(rng.integers(1, 3)), int(rng.integers(1, 4))
            Np = int(rng.choice([2, 7, 100, 900, 3000, 5000]))
            H = int(rng.choice([8, 31, 32, 40, 64, 100, 130]))
            K = int(rng.choice([1, 2, 3, 4, 8]))
            radius = float(rng.choice([0.003, 0.006, 0.02, 0.06, 0.2]))
            pts = synth.make_clouds(B, Np, int(rng.integers(0, 1 << 30))) * float(rng.uniform(0.3, 1.0))
            cfg = dict(B=B, Np=Np, M=M, H=H, K=K, radius=radius, mode=str(rng.choice(["norm", "alpha"])), views=views(rng, B, M, False),
                       per_point=bool(rng.integers(0, 2)))
            if cfg["mode"] == "norm":      # one colour under the norm compositor: the image is that colour wherever covered, every
                cfg["per_point"] = True    # camera gradient is identically zero and a RELATIVE error means nothing
            any_soup = False
            res = T.run_points(orc, dev, cfg, backward=True, pts=pts)
            d = np.abs(res["img"].detach().cpu().numpy() - res["o"]["images"])
            if d.max() > 1e-5:
                raise AssertionError(f"image error {d.max():.3e}, {int((d > 1e-5).sum())} values over 1e-5")
            what = f"points B={B} M={M} Np={Np} H={H} K={K} r={radius} {cfg['mode']} per_point={cfg['per_point']}"
        worst = _worst()
        _seen.clear()
        note = ""
        if worst > GRAD_BAR:
            if case % 3 != 2 and K == 1 and cfg["persp"] and not near:
                floor = fp32_floor(cfg)
                note = f" (fp32 floor of the case {floor:.2e})"
                if worst > 30 * floor:
                    raise AssertionError(f"gradient rel err {worst:.3e} > 30 x fp32 floor {floor:.2e}: {what}")
            elif any_soup:
                note = " (soup: no floor available for this configuration)"
            else:
                raise AssertionError(f"gradient rel err {worst:.3e} > {GRAD_BAR}: {what}")
        print(f"case {case}: ok   grad rel err {worst:.2e}{note}{hl if case % 3 != 2 else ''}   {what}", flush=True)
    except Exception as e:      # noqa: BLE001
        msg = traceback.format_exc().strip().splitlines()
        print(f"case {case}: FAIL {type(e).__name__}: {str(e)[:200]}  @ {msg[-3].strip() if len(msg) > 2 else ''} | cfg: "
              + ", ".join(f"{k}={v}" for k, v in cfg.items() if k not in ("meshes", "views")) + f" views={[t.tolist() for t in cfg['views']]}", flush=True)
        fails.append(case); _seen.clear()
if __name__ == "__main__":
    print(f"{n_cases - len(fails)} / {n_cases} cases passed ({n_highlight} with one or two highlight pixels between 1e-5 and 1.5e-5); failing seeds: {fails}")
