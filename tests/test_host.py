"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol (no compute calls
without a GPU), host helpers keep the reference's semantics, and the product refuses to run without CUDA
instead of falling back."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import mvtn_b200
from mvtn_b200 import _lib, cameras, parallel, structures, synth, util
from mvtn_b200.renderer import MVRenderer
from conftest import ROOT


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "mvr_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(mvr_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    names = declared_symbols()
    assert len(names) >= 15 and "mvr_mesh_forward" in names and "mvr_points_backward" in names
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"libmvr_b200.so does not export {n}"
    assert set(names) == set(_lib.SIGNATURES), "ctypes signatures and header declarations differ"


def test_ctypes_signatures_follow_the_header_argument_by_argument():
    """Every prototype of include/mvr_b200.h against mvtn_b200/_lib.py SIGNATURES: same number of arguments, and each argument in
    the same class (pointer / int / int64 / size_t / float / double / uint32) -- a swapped or missing argument in the hand-written
    ctypes table would otherwise only show up as garbage on the GPU."""
    import ctypes as C
    hdr = open(os.path.join(ROOT, "include", "mvr_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    protos = re.findall(r"([A-Za-z_][A-Za-z0-9_ \*]*?)\b(mvr_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", hdr, flags=re.S)
    assert {p[1] for p in protos} == set(_lib.SIGNATURES)
    scalar = {"int": "int", "int64_t": "i64", "long long": "i64", "size_t": "size", "float": "f32", "double": "f64", "uint32_t": "u32"}

    def header_class(param):
        param = param.strip()
        if param in ("void", ""):
            return None
        if "*" in param:
            return "ptr"
        ctype = re.sub(r"\b[a-zA-Z_][a-zA-Z0-9_]*$", "", param).replace("const", "").strip()      # drop the parameter name
        return scalar[ctype]

    def ctypes_class(t):
        if t in (C.c_void_p, C.c_char_p) or hasattr(t, "contents"):
            return "ptr"
        return {C.c_int: "int", C.c_int64: "i64", C.c_size_t: "size", C.c_float: "f32", C.c_double: "f64", C.c_uint32: "u32"}[t]

    for _ret, name, args in protos:
        want = [c for c in (header_class(a) for a in args.split(",")) if c is not None]
        got = [ctypes_class(t) for t in _lib.SIGNATURES[name][1]]
        assert want == got, f"{name}: header {want} != ctypes {got}"


def test_library_loads_and_answers_host_queries():
    lib = _lib.load()
    assert lib.mvr_abi_version() == _lib.ABI_VERSION
    assert lib.mvr_launch_count() >= 0
    # size queries are pure host arithmetic
    ws = lib.mvr_mesh_workspace_bytes(32, 12, 224, 224, 1, 160000, 320000)
    assert 8 * 384 * 224 * 224 <= ws < 1 << 30          # one 64-bit (z, face) key per pixel and view
    assert ws >= 8 * 384 * 224 * 224 + 16 * 12 * 160000    # + the projected vertices of every view
    assert lib.mvr_mesh_workspace_bytes(32, 12, 224, 224, 2, 160000, 320000) >= 2 * 8 * 384 * 224 * 224   # + previous layer when peeling
    assert lib.mvr_mesh_geometry_bytes(5000, 10000) >= 5000 * 48 + 10000 * 16
    assert lib.mvr_mesh_geometry_bytes(-1, 0) == 0
    assert lib.mvr_points_workspace_bytes(32, 2048, 12, 224, 224, 3, 0.006) >= 3 * 8 * 384 * 224 * 224   # generic K: key plane


def test_argument_validation_returns_status_not_crash():
    lib = _lib.load()
    # invalid arguments are rejected before any CUDA call: status < 0 and a message, never an exception/abort
    rc = lib.mvr_points_forward(None, None, 1, 16, 1, None, None, None, 0.01, None, 0, 64, 1, 0, None, None, None, None, None, None, None, 0, None)
    assert rc < 0 and b"image size" in lib.mvr_last_error_string()
    rc = lib.mvr_points_forward(None, None, 1, 16, 1, None, None, None, 0.01, None, 64, 64, 200, 0, None, None, None, None, None, None, None, 0, None)
    assert rc < 0 and b"points_per_pixel" in lib.mvr_last_error_string()
    rc = lib.mvr_points_forward(None, None, 1, 16, 1, None, None, None, -1.0, None, 64, 64, 1, 0, None, None, None, None, None, None, None, 0, None)
    assert rc < 0 and b"radius" in lib.mvr_last_error_string()
    rc = lib.mvr_mesh_forward(None, None, None, 1, 1, 3, 1, 3, 1, None, None, None, None, 0, None, None, 1.7, 1.7, 0.5, 0.0, 64, 64, 1, 0,
                              None, None, None, None, None, None, None, None, 0, None)
    assert rc < 0 and b"null pointer" in lib.mvr_last_error_string()
    rc = lib.mvr_mesh_soft_blend_forward(None, None, None, 1, 1, 3, 1, None, None, 0, None, None, 64, 64, 4, 0, 7, 1e-4, 1e-4, 1.0, 100.0,
                                         None, None, None, None, None, None)
    assert rc < 0 and b"null pointer" in lib.mvr_last_error_string()
    rc = lib.mvr_mesh_prepare(None, None, None, None, 1, 10, 10, 10, None, 0, None, 16, None)
    assert rc < 0 and b"too small" in lib.mvr_last_error_string()
    with pytest.raises(_lib.MVRError):
        _lib.check(rc, "mvr_mesh_prepare")
    # empty batches are a no-op
    assert lib.mvr_look_at_forward(None, None, None, 0, None, None, None, None, None) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="the pointers are fake: they must never reach a device")
def test_points_forward_rejects_misaligned_idx_before_any_launch():
    """K = 2 / 4: the forward stores a pixel's ids as one int2 / int4, so an idx not aligned to 4 K bytes is refused on the host
    (status -10, a message naming the alignment) before any CUDA call -- here with fake, otherwise valid, pointers."""
    lib = _lib.load()
    fake = 1 << 20
    for K in (2, 4):
        for off in range(4, 4 * K, 4):
            n0 = lib.mvr_launch_count()
            rc = lib.mvr_points_forward(fake, fake, 1, 16, 1, fake, fake, fake, 0.01, fake, 64, 64, K, 0, None, fake, fake + off, None, None,
                                        None, fake, 1 << 30, None)
            assert rc == -10, (K, off, rc)
            assert b"idx must be aligned to 4*K = %d bytes" % (4 * K) in lib.mvr_last_error_string()
            assert lib.mvr_launch_count() == n0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    r = MVRenderer(nb_views=2, image_size=32)
    az = torch.zeros(1, 2)
    with pytest.raises(_lib.MVRError, match="no CPU path"):
        r(None, torch.zeros(1, 8, 3), az, az, az + 2.0)
    with pytest.raises(_lib.MVRError):
        mvtn_b200.PackedMeshes([torch.zeros(3, 3)], [torch.zeros(1, 3, dtype=torch.int64)], "cpu")


def test_constructor_matches_reference_signature():
    import inspect
    sig = inspect.signature(MVRenderer.__init__)
    names = list(sig.parameters)[1:11]
    assert names == ["nb_views", "image_size", "pc_rendering", "object_color", "background_color", "faces_per_pixel",
                     "points_radius", "points_per_pixel", "light_direction", "cull_backfaces"]      # renderer.py:52
    d = {k: v.default for k, v in sig.parameters.items()}
    assert (d["image_size"], d["pc_rendering"], d["object_color"], d["background_color"]) == (224, True, "white", "white")
    assert (d["faces_per_pixel"], d["points_radius"], d["points_per_pixel"], d["light_direction"], d["cull_backfaces"]) == \
        (1, 0.006, 1, "random", False)
    r = MVRenderer(12)
    assert len(r.state_dict()) == 0 and len(list(r.parameters())) == 0      # stateless: old checkpoints load
    fwd = list(inspect.signature(MVRenderer.forward).parameters)
    assert fwd == ["self", "meshes", "points", "azim", "elev", "dist", "color"]
    assert list(inspect.signature(MVRenderer.render_and_save).parameters)[1:] == \
        ["meshes", "points", "azim", "elev", "dist", "images_path", "cameras_path", "color"]


def test_color_and_light_policy():
    torch.manual_seed(0); np.random.seed(0)
    assert torch.allclose(util.torch_color("white", max_lightness=True), torch.full((3,), 1 / 1.00001))   # util.py:314-334
    assert torch.equal(util.torch_color("black", max_lightness=True), torch.zeros(3))
    assert torch.allclose(util.torch_color("red", max_lightness=True), torch.tensor([1 / 1.00001, 0, 0]))
    r = MVRenderer(4, object_color="random", light_direction="random")
    r.train()
    c = r.rendering_color()
    assert c.max() == pytest.approx(1 / 1.00001, rel=1e-5) and c.min() >= 0
    l = r.light_direction(None, None, None)
    assert len(l) == 1 and len(l[0]) == 3 and all(-1 <= x <= 1 for x in l[0])
    r.eval()
    assert torch.equal(r.rendering_color(), torch.ones(3))                    # eval + "random" -> plain white
    assert r.light_direction(None, None, None) is None                        # -> relative (camera) light
    assert MVRenderer(4, light_direction="fixed").light_direction(None, None, None) == ((0, 1.0, 0),)
    assert MVRenderer(4, object_color="custom").rendering_color((0.1, 0.2, 0.3)) == (0.1, 0.2, 0.3)


def test_batch_tensor_flat_order():
    B, M = 3, 4
    x = torch.arange(B * M).reshape(B, M)
    flat = util.batch_tensor(x.T, dim=1, squeeze=True)       # renderer.py:79: view n = b*M + m
    assert torch.equal(flat, x.reshape(-1))
    imgs = torch.arange(B * M * 2 * 2 * 3).reshape(B * M, 2, 2, 3)
    un = util.unbatch_tensor(imgs, batch_size=M, dim=1, unsqueeze=True).transpose(0, 1)   # renderer.py:109-110
    assert torch.equal(un, imgs.reshape(B, M, 2, 2, 3))


def test_check_valid_rotation_matrix():
    assert util.check_valid_rotation_matrix(torch.eye(3)[None])
    assert not util.check_valid_rotation_matrix(torch.diag(torch.tensor([1.0, 1.0, -1.0]))[None])
    assert not util.check_valid_rotation_matrix(torch.zeros(1, 3, 3))


def test_meshes_container_and_unpack():
    v, f = synth.make_mesh(100, 0)
    ms = [structures.Meshes([v], [f]), structures.Meshes([v * 2], [f])]
    verts, faces = structures.unpack_mesh_list(ms)
    assert len(verts) == 2 and torch.equal(verts[1], v * 2)
    batched = structures.Meshes([v, v * 2], [f, f])
    verts2, _ = structures.unpack_mesh_list(batched)            # run_mvtn.py:517-533 passes a batched object
    assert len(verts2) == 2 and len(batched) == 2 and len(batched[0:1]) == 1
    ext = batched.extend(3)
    assert len(ext) == 6 and torch.equal(ext.verts_list()[2], v) and torch.equal(ext.verts_list()[3], v * 2)


def test_camera_shim_transforms():
    from oracle import oracle as orc
    R, T, C = orc.look_at([30.0, -70.0], [20.0, 45.0], [2.2, 1.7])
    cam = cameras.FoVPerspectiveCameras(torch.from_numpy(R), torch.from_numpy(T))
    assert len(cam) == 2 and cam.is_perspective()
    assert torch.allclose(cam.get_camera_center(), torch.from_numpy(C), atol=1e-5)
    w2v = cam.get_world_to_view_transform()
    p = torch.randn(2, 5, 3)
    assert torch.allclose(w2v.transform_points(p), p @ torch.from_numpy(R) + torch.from_numpy(T)[:, None], atol=1e-6)
    assert torch.allclose(w2v.inverse().transform_points(w2v.transform_points(p)), p, atol=1e-5)
    from mvtn_b200.viz import camera_wireframes_world
    wires = camera_wireframes_world(cam, 0.22)
    assert wires.shape == (2, 12, 3) and torch.allclose(wires[:, 5], torch.from_numpy(C), atol=1e-5)   # apex = centre


def test_synthetic_inputs_follow_the_normalisation_contract():
    v, f = synth.make_mesh(10000, 1236)
    assert abs(f.shape[0] - 10000) < 300 and f.max() < v.shape[0] and f.min() == 0
    assert v.norm(dim=1).max() == pytest.approx(1.0, abs=1e-5) and v.mean(0).abs().max() < 1e-5
    e = torch.cat([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    key = e[:, 0] * v.shape[0] + e[:, 1]; rev = e[:, 1] * v.shape[0] + e[:, 0]
    assert key.unique().numel() == key.numel() and set(key.tolist()) == set(rev.tolist())   # closed, consistently wound
    p = synth.make_clouds(2, 2048, 5)
    assert p.shape == (2, 2048, 3) and p[0].norm(dim=1).max() == pytest.approx(1.0, abs=1e-5)
    assert torch.equal(synth.make_clouds(2, 64, 5), synth.make_clouds(2, 64, 5))
    az, el, di = synth.circular_views(2, 12)
    assert az.shape == (2, 12) and az[0, 0] == -270 and (el == 30).all() and (di == 2.2).all()   # mvtn.py:22-24
    a, e2, _ = synth.learned_spherical_views(3, 12, 0)
    assert a.shape == (3, 12) and e2.abs().max() <= 89.0


def test_shard_ranges_partition_objects():
    for n in (0, 1, 7, 32, 33, 256):
        for w in (1, 2, 4, 8):
            r = [parallel.shard_range(n, i, w) for i in range(w)]
            assert r[0][0] == 0 and r[-1][1] == n and all(r[i][1] == r[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in r]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        parallel.shard_range(4, 4, 4)
    parts = parallel.shard_by_weight([10, 1, 1, 1, 1, 10, 1, 1, 1, 1], 2)
    assert parts == [(0, 5), (5, 10)]
    parts = parallel.shard_by_weight([1] * 3, 8)
    assert parts[0][0] == 0 and parts[-1][1] == 3 and all(a <= b for a, b in parts)


def test_async_mesh_staging_worker_matches_torch_cat():
    """mvr_host_stage_meshes_begin/_end (host-only use: device pointers NULL, no CUDA call): gathers ragged meshes on
    the worker thread, narrows int64 faces, refuses a second job while one is in flight, and rejects stale job ids."""
    import ctypes as C
    from mvtn_b200 import synth
    lib = _lib.load()
    meshes = [synth.make_mesh(nf, 40 + i) for i, nf in enumerate((300, 5000, 60, 2200))]
    vs = [v for v, _ in meshes]; fs = [f for _, f in meshes]
    tv = sum(v.shape[0] for v in vs); tf = sum(f.shape[0] for f in fs)
    vd = torch.empty(tv * 3); fd = torch.empty(tf * 3, dtype=torch.int32)
    n = len(vs)
    vp = (C.c_void_p * n)(*[t.data_ptr() for t in vs]); vc = (C.c_int64 * n)(*[t.numel() for t in vs])
    fp = (C.c_void_p * n)(*[t.data_ptr() for t in fs]); fc = (C.c_int64 * n)(*[t.numel() for t in fs])
    for _ in range(3):
        vd.zero_(); fd.zero_()
        job = lib.mvr_host_stage_meshes_begin(vp, vc, fp, fc, n, 8, vd.data_ptr(), fd.data_ptr(), None, None, 0, None)
        assert job > 0
        assert lib.mvr_host_stage_meshes_begin(vp, vc, fp, fc, n, 8, vd.data_ptr(), fd.data_ptr(), None, None, 0, None) == -10
        assert lib.mvr_host_stage_meshes_end(job) == 0
        assert lib.mvr_host_stage_meshes_end(job) == -11 and b"unknown job" in lib.mvr_last_error_string()
        assert torch.equal(torch.cat(vs).reshape(-1), vd)
        assert torch.equal(torch.cat(fs).reshape(-1).to(torch.int32), fd)
    # synchronous entry point, int32 faces
    f32 = [f.to(torch.int32) for f in fs]
    fp32 = (C.c_void_p * n)(*[t.data_ptr() for t in f32])
    fd.zero_()
    assert lib.mvr_host_stage_meshes(vp, vc, fp32, fc, n, 4, vd.data_ptr(), fd.data_ptr(), None, None, None) == 0
    assert torch.equal(torch.cat(f32).reshape(-1), fd)
    assert lib.mvr_host_stage_meshes(vp, vc, fp32, fc, n, 2, vd.data_ptr(), fd.data_ptr(), None, None, None) == -2
    # uint16 ids, from int64 and from int32 sources; out-of-range ids saturate (mvr_mesh_prepare clamps them to the mesh afterwards)
    fs_bad = [f.clone() for f in fs]
    fs_bad[1][0, 0] = -7; fs_bad[1][1, 2] = 70000; fs_bad[3][5, 1] = 65535
    want = torch.cat(fs_bad).reshape(-1).clamp(0, 65535)
    for srcs, eb in ((fs_bad, 8), ([f.to(torch.int32) for f in fs_bad], 4)):
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in srcs])
        f16 = torch.zeros(tf * 3, dtype=torch.int16)
        offs = torch.zeros(2 * n + 2, dtype=torch.int32)
        assert lib.mvr_host_stage_meshes_packed(vp, vc, ptrs, fc, n, eb, 2, vd.data_ptr(), f16.data_ptr(), offs.data_ptr(), None, None, None, None) == 0
        assert torch.equal(f16.to(torch.int64) & 0xFFFF, want) and torch.equal(torch.cat(vs).reshape(-1), vd)
        assert offs.tolist() == [0] + list(np.cumsum([v.shape[0] for v in vs])) + [0] + list(np.cumsum([f.shape[0] for f in fs]))
    f32o = torch.zeros(tf * 3, dtype=torch.int32)
    assert lib.mvr_host_stage_meshes_packed(vp, vc, fp32, fc, n, 4, 4, vd.data_ptr(), f32o.data_ptr(), None, None, None, None, None) == 0
    assert torch.equal(torch.cat(f32).reshape(-1), f32o)
    assert lib.mvr_host_stage_meshes_packed(vp, vc, fp32, fc, n, 4, 3, vd.data_ptr(), f32o.data_ptr(), None, None, None, None, None) == -2


def test_collate_meshes_packs_like_torch_cat():
    from mvtn_b200 import HostPackedMeshes, Meshes, collate_meshes, synth
    meshes = [synth.make_mesh(nf, 7 + i) for i, nf in enumerate((500, 80, 3000))]
    hp = collate_meshes([Meshes([v], [f]) for v, f in meshes], pin_memory=False)
    assert isinstance(hp, HostPackedMeshes) and len(hp) == 3
    assert hp.num_verts == [v.shape[0] for v, _ in meshes] and hp.num_faces == [f.shape[0] for _, f in meshes]
    assert torch.equal(hp.verts, torch.cat([v for v, _ in meshes])) and hp.faces.dtype == torch.int16      # (<= 65536 vertices: uint16 ids)
    assert torch.equal(torch.cat(hp.faces_list()), torch.cat([f for _, f in meshes]).to(torch.int32))
    hp32 = collate_meshes([Meshes([v], [f]) for v, f in meshes], pin_memory=False, narrow_faces=False)
    assert hp32.faces.dtype == torch.int32 and torch.equal(hp32.faces, torch.cat([f for _, f in meshes]).to(torch.int32))
    assert all(torch.equal(a, b) for a, (b, _) in zip(hp.verts_list(), meshes))
    with pytest.raises(ValueError):
        HostPackedMeshes(hp.verts, hp.faces, [1, 2, 3], hp.num_faces)
    with pytest.raises(ValueError):
        HostPackedMeshes(hp.verts, hp.faces.to(torch.int64), hp.num_verts, hp.num_faces)
    empty = collate_meshes([], pin_memory=False)
    assert len(empty) == 0 and empty.verts.shape == (0, 3)


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` (the oracle port on the host cores) needs no GPU: one tiny step, one JSON line."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "1", "--views", "2",
                          "--image-size", "32", "--faces", "200", "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["value"] > 0 and d["unit"] == "views/s" and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0


def test_point_fragments_complete_the_sparse_idx_lazily():
    """ops._PointFragments: with MVR_IDX_SPARSE the kernels leave idx unwritten at background pixels; the dict handed to the
    caller fills those with -1 from the 1-bit hit mask (bit x & 31 of word x >> 5 of row y) on first access."""
    import torch
    from mvtn_b200 import ops
    g = torch.Generator().manual_seed(0)
    N, H, W, K = 2, 5, 70, 2                                   # 3 mask words per row, the last one partial
    hit = torch.rand(N, H, W, generator=g) < 0.3
    idx = torch.randint(0, 1000, (N, H, W, K), dtype=torch.int32, generator=g)      # "uninitialised" background included
    mw = (W + 31) // 32
    bits = torch.zeros(N, H, mw * 32, dtype=torch.int64)
    bits[:, :, :W] = hit.long()
    words = (bits.view(N, H, mw, 32) << torch.arange(32)).sum(-1)
    words = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)   # bit 31 set = negative int32
    mask = torch.cat([words.reshape(-1), torch.full((7,), -1, dtype=torch.int32)])  # the buffer may be longer than needed
    fr = ops._PointFragments(idx, mask, H, W)
    assert list(fr.keys()) == ["idx"]
    dense = fr["idx"]
    assert torch.equal(dense[hit], idx[hit])
    assert (dense[~hit] == -1).all()
    assert fr.get("idx") is dense and dict(fr.items())["idx"] is dense


def test_mesh_workspace_hint_bookkeeping(monkeypatch):
    """ops._ws_mesh: what the mesh path may assume about its workspace between calls (MVR_WS_* flags).  Pure host logic:
    the stream accessor and the capture query are stubbed, the "workspace" is a CPU tensor."""
    import torch
    from mvtn_b200 import ops
    L = _lib
    monkeypatch.setattr(ops, "_stream", lambda device: 1234)
    capturing = {"on": False}
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: capturing["on"])
    dev = torch.device("cuda", 0)
    key = (0, 1234)
    ws = torch.empty(1 << 12, dtype=torch.uint8)
    monkeypatch.setitem(ops._workspaces, key, ws)
    ops._ws_mesh.pop(key, None)
    layout = (2, 3, 64, 64, 1, 1000)
    # cold: re-arm only; nothing is known while the call is in flight (it may raise before commit)
    flags, commit = ops._ws_mesh_flags_forward(dev, ws, layout)
    assert flags == L.WS_REARM_KEYS and key not in ops._ws_mesh
    t1 = commit()
    assert ops._ws_mesh_flags_backward(dev, ws, t1) == L.WS_PROJECTED
    # warm, same layout: the memset is skipped
    flags, commit = ops._ws_mesh_flags_forward(dev, ws, layout)
    assert flags == L.WS_REARM_KEYS | L.WS_KEYS_ARMED
    t2 = commit()
    assert t2 != t1
    # the backward of the OLDER forward re-projects and thereby invalidates the newer projection
    assert ops._ws_mesh_flags_backward(dev, ws, t1) == 0
    assert ops._ws_mesh_flags_backward(dev, ws, t2) == 0
    # another layout, another buffer, a failed call, another user of the buffer: all cold again
    flags, commit = ops._ws_mesh_flags_forward(dev, ws, (2, 3, 64, 64, 2, 1000)); commit()
    assert flags == L.WS_REARM_KEYS
    flags, commit = ops._ws_mesh_flags_forward(dev, torch.empty(1 << 12, dtype=torch.uint8), (2, 3, 64, 64, 2, 1000)); commit()
    assert flags == L.WS_REARM_KEYS
    flags, _no_commit = ops._ws_mesh_flags_forward(dev, ws, layout)            # the C call raised: commit never ran
    flags, commit = ops._ws_mesh_flags_forward(dev, ws, layout); commit()
    assert flags == L.WS_REARM_KEYS
    assert ops.workspace(dev, 16, _mesh_owner=True) is ws and key in ops._ws_mesh
    assert ops.workspace(dev, 16) is ws and key not in ops._ws_mesh             # e.g. the point path
    # a stream that has been captured into a CUDA graph is never trusted again (replays bypass this bookkeeping)
    flags, commit = ops._ws_mesh_flags_forward(dev, ws, layout); commit()
    capturing["on"] = True
    flags, commit = ops._ws_mesh_flags_forward(dev, ws, layout)
    assert flags == 0 and commit() is None
    capturing["on"] = False
    flags, commit = ops._ws_mesh_flags_forward(dev, ws, layout)
    assert flags == 0 and commit() is None and ops._ws_mesh_flags_backward(dev, ws, 7) == 0
    ops._ws_mesh.pop(key, None)


def test_flag_constants_match_the_header():
    """Every `#define MVR_<NAME> <int>` flag / counter slot of include/mvr_b200.h that the ctypes layer mirrors carries the
    same value there (mvtn_b200/_lib.py), and the flag bits are pairwise disjoint."""
    hdr = open(os.path.join(ROOT, "include", "mvr_b200.h")).read()
    defs = {m.group(1): int(m.group(2), 0) for m in re.finditer(r"#define\s+MVR_([A-Z0-9_]+)\s+(0x[0-9a-fA-F]+|\d+)\b", hdr)}
    assert defs["ABI_VERSION"] == _lib.ABI_VERSION
    mirrored = [n for n in defs if hasattr(_lib, n) and n != "ABI_VERSION"]
    assert {"PERSPECTIVE_CORRECT", "CULL_BACKFACES", "COMPOSITE_ALPHA", "RGB_PER_ELEMENT", "FACES_I64", "IMAGES_BF16", "SCALE_IS_DIST",
            "WS_KEYS_ARMED", "WS_REARM_KEYS", "WS_PROJECTED", "IDX_SPARSE", "FACES_U16", "CLIP_BARYCENTRIC", "TEST_TINY_QUEUES", "NUM_COUNTERS"} <= set(mirrored)
    for n in mirrored:
        assert getattr(_lib, n) == defs[n], n
    flags = [defs[n] for n in mirrored if n not in ("NUM_COUNTERS", "CNT_STRADDLE", "CNT_BIG_FACES")]
    assert all(f & (f - 1) == 0 for f in flags)                   # single bits
    assert len(set(flags)) == len(flags)                          # no two flags share a bit


def test_collate_meshes_narrows_faces_to_uint16_when_it_can():
    """collate_meshes sends the faces as uint16 (in an int16 tensor) when every mesh has at most 65536 vertices -- ids above 32767
    included -- and as int32 otherwise; faces_list() gives the ids back either way."""
    import torch
    from mvtn_b200 import Meshes, collate_meshes
    g = torch.Generator().manual_seed(3)
    big = torch.rand(40000, 3, generator=g)
    fbig = torch.randint(0, 40000, (500, 3), generator=g)
    fbig[0] = torch.tensor([39999, 32768, 32767])
    small = torch.rand(50, 3, generator=g)
    fsmall = torch.randint(0, 50, (80, 3), generator=g)
    ml = [Meshes([big], [fbig]), Meshes([small], [fsmall])]
    hp = collate_meshes(ml, pin_memory=False)
    assert hp.faces.dtype == torch.int16 and hp.faces.shape == (580, 3)
    got = hp.faces_list()
    assert torch.equal(got[0].long(), fbig) and torch.equal(got[1].long(), fsmall)
    hp32 = collate_meshes(ml, pin_memory=False, narrow_faces=False)
    assert hp32.faces.dtype == torch.int32 and torch.equal(hp32.faces_list()[0].long(), fbig)
    huge = torch.rand(70000, 3, generator=g)
    fhuge = torch.randint(0, 70000, (10, 3), generator=g)
    hp2 = collate_meshes([Meshes([huge], [fhuge])], pin_memory=False)
    assert hp2.faces.dtype == torch.int32 and torch.equal(hp2.faces_list()[0].long(), fhuge)
    import pytest
    with pytest.raises(ValueError):
        collate_meshes([Meshes([huge], [fhuge])], pin_memory=False, narrow_faces=True)


def test_async_packed_staging_on_the_helper_pool_matches_the_synchronous_call():
    """mvr_host_stage_meshes_packed_begin/_end: the gather runs on the staging thread + its private helper pool (no OpenMP team);
    same bytes as the synchronous call for ragged batches, repeated jobs (pool reuse), a single tiny mesh (fewer items than
    threads) and an empty batch."""
    import ctypes as C
    from mvtn_b200 import synth
    lib = _lib.load()
    cases = [[synth.make_mesh(nf, 60 + i) for i, nf in enumerate((300, 50000, 60, 2200, 9000))], [synth.make_mesh(12, 3)],
             [synth.make_mesh(nf, 80 + i) for i, nf in enumerate((40000, 40000, 40000))]]
    for rep in range(3):
        for meshes in cases:
            vs = [v for v, _ in meshes]; fs = [f for _, f in meshes]
            n = len(vs); tv = sum(v.shape[0] for v in vs); tf = sum(f.shape[0] for f in fs)
            vp = (C.c_void_p * n)(*[t.data_ptr() for t in vs]); vc = (C.c_int64 * n)(*[t.numel() for t in vs])
            fp = (C.c_void_p * n)(*[t.data_ptr() for t in fs]); fc = (C.c_int64 * n)(*[t.numel() for t in fs])
            for out_bytes, dt in ((2, torch.int16), (4, torch.int32)):
                got, want = [], []
                for sync in (False, True):
                    vd = torch.zeros(tv * 3); fd = torch.zeros(tf * 3, dtype=dt); offs = torch.zeros(2 * n + 2, dtype=torch.int32)
                    if sync:
                        assert lib.mvr_host_stage_meshes_packed(vp, vc, fp, fc, n, 8, out_bytes, vd.data_ptr(), fd.data_ptr(), offs.data_ptr(),
                                                                None, None, None, None) == 0
                    else:
                        job = lib.mvr_host_stage_meshes_packed_begin(vp, vc, fp, fc, n, 8, out_bytes, vd.data_ptr(), fd.data_ptr(),
                                                                     offs.data_ptr(), None, None, None, 0, None)
                        assert job > 0 and lib.mvr_host_stage_meshes_end(job) == 0
                    (want if sync else got).extend([vd, fd, offs])
                assert all(torch.equal(a, b) for a, b in zip(got, want))
                assert torch.equal(got[0], torch.cat(vs).reshape(-1)) and torch.equal(got[1].to(torch.int64) & (0xFFFF if out_bytes == 2 else -1),
                                                                                         torch.cat(fs).reshape(-1))
    assert lib.mvr_host_stage_meshes_packed_begin(None, None, None, None, 0, 8, 3, None, None, None, None, None, None, 0, None) == -2


def test_async_staging_survives_fork():
    """The staging thread and its helper pool do not exist in a forked child (a DataLoader worker): the library starts fresh ones
    there instead of waiting for threads that are gone."""
    import ctypes as C
    import os
    from mvtn_b200 import synth
    lib = _lib.load()
    meshes = [synth.make_mesh(nf, 90 + i) for i, nf in enumerate((3000, 50000, 700))]
    vs = [v for v, _ in meshes]; fs = [f for _, f in meshes]
    n = len(vs); tv = sum(v.shape[0] for v in vs); tf = sum(f.shape[0] for f in fs)
    vp = (C.c_void_p * n)(*[t.data_ptr() for t in vs]); vc = (C.c_int64 * n)(*[t.numel() for t in vs])
    fp = (C.c_void_p * n)(*[t.data_ptr() for t in fs]); fc = (C.c_int64 * n)(*[t.numel() for t in fs])

    def job():
        vd = torch.zeros(tv * 3); fd = torch.zeros(tf * 3, dtype=torch.int16); offs = torch.zeros(2 * n + 2, dtype=torch.int32)
        j = lib.mvr_host_stage_meshes_packed_begin(vp, vc, fp, fc, n, 8, 2, vd.data_ptr(), fd.data_ptr(), offs.data_ptr(), None, None, None, 0, None)
        return j > 0 and lib.mvr_host_stage_meshes_end(j) == 0 and torch.equal(vd, torch.cat(vs).reshape(-1)) and torch.equal(fd.to(torch.int64) & 0xFFFF, torch.cat(fs).reshape(-1))

    assert job()                      # threads exist in the parent now
    pid = os.fork()
    if pid == 0:
        ok = False
        try:
            import signal
            signal.alarm(60)          # a hang (waiting for threads that do not exist) must not outlive the test
            torch.set_num_threads(1)  # (libgomp's own team does not survive fork either: keep torch's checks below serial)
            ok = job() and job()
        finally:
            os._exit(0 if ok else 1)
    _, status = os.waitpid(pid, 0)
    assert os.WIFEXITED(status) and os.WEXITSTATUS(status) == 0
    assert job()                      # and the parent's threads are untouched
