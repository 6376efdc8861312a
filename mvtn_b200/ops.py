"""Torch-facing operators over the C ABI (include/mvr_b200.h): device memory, streams and autograd
plumbing only -- every arithmetic step of the path runs in libmvr_b200.so.

Operator surface (mirrors what renderer.py reaches in PyTorch3D):
    look_at_view_transform(dist, elev, azim)         renderer.py:79,122
    PackedMeshes                                     renderer.py:67-77 (Meshes / Textures / normals)
    render_meshes(...)                               renderer.py:89-107 (MeshRenderer + HardPhong)
    render_points(...)                               renderer.py:129-145 (PointsRenderer + compositor)
"""
import functools
import math
from typing import Optional, Sequence

import torch

from . import _lib as L

_workspaces = {}


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(device):
    """Raw cudaStream_t of torch's current stream on `device` (the C-level accessor when this torch has it: the python
    Stream object costs several microseconds per call, and the hot path asks a dozen times per step)."""
    if _raw_stream is not None:
        idx = device.index if isinstance(device, torch.device) else torch.device(device).index
        return _raw_stream(torch.cuda.current_device() if idx is None else idx)
    return torch.cuda.current_stream(device).cuda_stream


class _NoCtx:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NOCTX = _NoCtx()


def _on(device):
    """Context making `device` current for a C-ABI call; free when it already is (the usual case)."""
    idx = device.index
    if idx is None or idx == torch.cuda.current_device():
        return _NOCTX
    return torch.cuda.device(device)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise L.MVRError(f"{name} must be a CUDA tensor: mvtn_b200 has no CPU path")


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype is torch.float32 and t.is_contiguous():
        return t.detach()
    return t.detach().to(torch.float32).contiguous()


def workspace(device, nbytes: int, _mesh_owner: bool = False) -> torch.Tensor:
    """Per-(device, stream) scratch reused across calls (stream order makes reuse safe).  Any user other than the mesh
    path invalidates what the mesh path remembers about the buffer's contents (see _ws_mesh_state)."""
    key = (torch.device(device).index, _stream(device))
    w = _workspaces.get(key)
    if w is None or w.numel() < nbytes:
        w = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = w
        if _ws_mesh.get(key) is not _WS_POISON:
            _ws_mesh.pop(key, None)
    if not _mesh_owner and _ws_mesh.get(key) is not _WS_POISON:
        _ws_mesh.pop(key, None)
    return w


# What the mesh path knows about a workspace between its own calls (SURVEY 8f N1/N4: no redundant passes per step):
#   "armed": (data_ptr, layout) -- the key plane was left all-EMPTY by the last forward (MVR_WS_REARM_KEYS), so the next
#            forward with the same layout skips its 154 MB memset (C2);
#   "proj":  token of the forward whose projected vertices / pixel table / clip flag still sit in the buffer, so its
#            backward skips the re-projection.
# Cleared by any other user of the buffer (workspace()), by reallocation, and never used on a stream that has been
# captured into a CUDA graph (replays touch the buffer behind python's back).
_ws_mesh = {}
_WS_POISON = object()
_ws_token = [0]


def _ws_mesh_flags_forward(dev, ws, layout):
    """-> (extra flags for mvr_mesh_forward, commit(): call after a successful launch, returns the projection token)."""
    key = (torch.device(dev).index, _stream(dev))
    if torch.cuda.is_current_stream_capturing():
        _ws_mesh[key] = _WS_POISON
    st = _ws_mesh.get(key)
    if st is _WS_POISON:
        return 0, lambda: None
    flags = L.WS_REARM_KEYS
    if st is not None and st.get("armed") == (ws.data_ptr(), layout):
        flags |= L.WS_KEYS_ARMED
    _ws_mesh.pop(key, None)          # nothing is known while the call is being made (it may raise)

    def commit():
        _ws_token[0] += 1
        _ws_mesh[key] = {"armed": (ws.data_ptr(), layout), "proj": (ws.data_ptr(), _ws_token[0])}
        return _ws_token[0]

    return flags, commit


def _ws_mesh_flags_backward(dev, ws, token):
    key = (torch.device(dev).index, _stream(dev))
    st = _ws_mesh.get(key)
    if token is None or st is None or st is _WS_POISON or torch.cuda.is_current_stream_capturing():
        return 0
    if st.get("proj") == (ws.data_ptr(), token):
        return L.WS_PROJECTED
    st["proj"] = None      # this backward re-projects ITS views over whatever a later forward left there
    return 0


_staging_bufs = {}
_copy_streams = {}


def _staging(tag, device, numel: int, dtype) -> torch.Tensor:
    """Reusable pinned host buffer for one async H2D copy; reuse waits for the previous copy's event."""
    key = (tag, torch.device(device).index, dtype)
    buf, ev = _staging_bufs.get(key, (None, None))
    if ev is not None:
        ev.synchronize()
    if buf is None or buf.numel() < numel:
        buf = torch.empty(max(numel, 1), dtype=dtype, pin_memory=True)
    _staging_bufs[key] = (buf, None)
    return buf[:numel]


def _staging_done(device):
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(device))
    for key, (buf, old) in list(_staging_bufs.items()):
        if key[1] == torch.device(device).index and old is None:
            _staging_bufs[key] = (buf, ev)


def _out_norm(normalize):
    """(mean, std) -> ctypes float[6] for the C ABI's HOST out_mean_std argument (None = identity)."""
    if normalize is None:
        return None
    import ctypes as C
    mean, std = normalize
    mean = [float(x) for x in (mean if hasattr(mean, "__len__") else (mean,) * 3)]
    std = [float(x) for x in (std if hasattr(std, "__len__") else (std,) * 3)]
    if len(mean) != 3 or len(std) != 3:
        raise ValueError("normalize must be (mean, std) with 3 channels each")
    if not all(x > 0 for x in std):
        raise ValueError("normalize: std must be positive")
    return (C.c_float * 6)(*mean, *std)


def _image_dtype(out_dtype):
    if out_dtype in (None, torch.float32):
        return torch.float32, 0
    if out_dtype is torch.bfloat16:
        return torch.bfloat16, L.IMAGES_BF16
    raise ValueError("out_dtype must be torch.float32 or torch.bfloat16")


def _grad_like_images(g, flags):
    """Cotangent of the images in the dtype the forward wrote (fp32, or bf16 under IMAGES_BF16), contiguous."""
    want = torch.bfloat16 if flags & L.IMAGES_BF16 else torch.float32
    g = g.detach()
    if g.dtype is not want:
        g = g.to(want)
    return g if g.is_contiguous() else g.contiguous()


def _hw(image_size):
    """int -> (S, S); (H, W) tuple as in PyTorch3D's RasterizationSettings.image_size."""
    if isinstance(image_size, (tuple, list)):
        return int(image_size[0]), int(image_size[1])
    return int(image_size), int(image_size)


def _host_array(t: torch.Tensor, dtype) -> torch.Tensor:
    """Contiguous CPU view of `t` in `dtype`; the common case (already so) costs three attribute reads."""
    if t.dtype == dtype and t.is_cpu and t.is_contiguous():
        return t
    return t.detach().to(device="cpu", dtype=dtype).contiguous()


def _host_gather(srcs, dst: torch.Tensor, elem_bytes: int, narrow: bool):
    import ctypes as C
    n = len(srcs)
    if n == 0:
        return
    ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in srcs])
    counts = (C.c_int64 * n)(*[t.numel() for t in srcs])
    L.check(L.load().mvr_host_gather(ptrs, counts, n, dst.data_ptr(), elem_bytes, 1 if narrow else 0), "mvr_host_gather")


def _stage_meshes(v_src, f_src, face_elem_bytes, v_host, f_host, v_dev, f_dev, device, overlap, offs_host=None, offs_dev=None):
    """Parallel gather of every mesh into the pinned buffers with the vertices' H2D copy already in flight while the
    faces are gathered (mvr_host_stage_meshes_packed: offsets written + copied by the same call, ids as wide as f_host -- an int16
    tensor = uint16 ids).  overlap=True runs it on the library's worker thread and returns (job, keep-alive); the caller joins
    with mvr_host_stage_meshes_end."""
    import ctypes as C
    lib = L.load()
    n = len(v_src)
    vp = (C.c_void_p * n)(*[t.data_ptr() for t in v_src])
    vc = (C.c_int64 * n)(*[3 * t.shape[0] for t in v_src])
    fp = (C.c_void_p * n)(*[t.data_ptr() for t in f_src])
    fc = (C.c_int64 * n)(*[3 * t.shape[0] for t in f_src])
    keep = (vp, vc, fp, fc, v_src, f_src, v_host, f_host)
    if overlap:
        job = lib.mvr_host_stage_meshes_packed_begin(vp, vc, fp, fc, n, face_elem_bytes, f_host.element_size(), v_host.data_ptr(),
                                                     f_host.data_ptr(), _ptr(offs_host), v_dev.data_ptr(), f_dev.data_ptr(),
                                                     _ptr(offs_dev), torch.device(device).index or 0, _stream(device))
        if job > 0:
            return job, keep
        if job != -10:          # -10: the worker is busy with another batch -> stage synchronously
            L.check(job, "mvr_host_stage_meshes_packed_begin")
    with _on(torch.device(device)):
        L.check(lib.mvr_host_stage_meshes_packed(vp, vc, fp, fc, n, face_elem_bytes, f_host.element_size(), v_host.data_ptr(),
                                                 f_host.data_ptr(), _ptr(offs_host), v_dev.data_ptr(), f_dev.data_ptr(),
                                                 _ptr(offs_dev), _stream(device)), "mvr_host_stage_meshes_packed")
    return None, keep


@functools.lru_cache(maxsize=16)
def fov_projection_scale(fov_deg: float = 60.0, znear: float = 1.0, aspect: float = 1.0):
    """K00, K11 of [upstream] FoVPerspectiveCameras.compute_projection_matrix, evaluated with the same
    fp32 tensor ops (fov*pi/180, tan(fov/2)*znear, 2*znear/(max-min))."""
    fov = torch.tensor(fov_deg, dtype=torch.float32) * (math.pi / 180.0)
    max_y = torch.tan(fov / 2) * znear
    min_y = -max_y
    max_x = max_y * aspect
    min_x = -max_x
    return float(2.0 * znear / (max_x - min_x)), float(2.0 * znear / (max_y - min_y))


# --------------------------------------------------------------------------------------------------
# cameras
# --------------------------------------------------------------------------------------------------
class FlagSink:
    """Where the rotation-validity flag of a look_at launch lands on the host: a pinned word the camera kernel stores the count
    into (up to 4096 views; an asynchronous copy above) + an event the LIBRARY records behind it (mvr_look_at_forward_flagged), so
    the caller neither issues a copy nor records an event in front of the rasterizer launch.  read() waits for that event only --
    i.e. for the camera kernel, not for the rasterizer behind it.  Pooled per device."""
    _pool = {}

    def __init__(self, device):
        self.device = device
        self.host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.event = torch.cuda.Event()
        self.event.record(torch.cuda.current_stream(device))      # (torch creates the cudaEvent_t on first record)
        self.armed = False

    @classmethod
    def get(cls, device):
        pool = cls._pool.setdefault(device.index, [])
        return pool.pop() if pool else cls(device)

    def read(self) -> int:
        """The flag (number of invalid rotations); returns the sink to the pool."""
        self.event.synchronize()
        v = int(self.host[0])
        self.armed = False
        FlagSink._pool.setdefault(self.device.index, []).append(self)
        return v


def _look_at_launch(azim, elev, dist, sink: "Optional[FlagSink]" = None):
    """Flat fp32 copies of the angles + one mvr_look_at_forward launch -> (a, e, d, R, T, C, invalid flag).
    sink: a FlagSink that receives the flag on the host (copy + event issued by the library call itself)."""
    _require_cuda(azim, "azim")
    a, e, d = _f32c(azim).reshape(-1), _f32c(elev).reshape(-1), _f32c(dist).reshape(-1)
    n = a.numel()
    if e.numel() != n or d.numel() != n:
        raise ValueError("azim, elev and dist must have the same number of elements")
    dev = a.device
    buf = torch.empty(15 * n, dtype=torch.float32, device=dev)      # one allocation: R | T | C
    R, T, Cc = buf[: 9 * n].view(n, 3, 3), buf[9 * n: 12 * n].view(n, 3), buf[12 * n:].view(n, 3)
    bad = torch.empty(1, dtype=torch.int32, device=dev)      # zeroed by mvr_look_at_forward
    with _on(dev):
        if sink is not None:
            L.check(L.load().mvr_look_at_forward_flagged(_ptr(a), _ptr(e), _ptr(d), n, _ptr(R), _ptr(T), _ptr(Cc), _ptr(bad),
                                                         sink.host.data_ptr(), sink.event.cuda_event, _stream(dev)),
                    "mvr_look_at_forward_flagged")
            sink.armed = True
        else:
            L.check(L.load().mvr_look_at_forward(_ptr(a), _ptr(e), _ptr(d), n, _ptr(R), _ptr(T), _ptr(Cc), _ptr(bad),
                                                 _stream(dev)), "mvr_look_at_forward")
    return a, e, d, R, T, Cc, bad


def _look_at_backward_launch(a, e, d, gR, gT, gC):
    n = a.numel()
    dev = a.device
    gR = None if gR is None else _f32c(gR)
    gT = None if gT is None else _f32c(gT)
    gC = None if gC is None else _f32c(gC)
    g = torch.empty(3 * n, dtype=torch.float32, device=dev)
    ga, ge, gd = g[:n], g[n: 2 * n], g[2 * n:]
    with _on(dev):
        L.check(L.load().mvr_look_at_backward(_ptr(a), _ptr(e), _ptr(d), n, _ptr(gR), _ptr(gT), _ptr(gC), _ptr(ga),
                                              _ptr(ge), _ptr(gd), _stream(dev)), "mvr_look_at_backward")
    return ga, ge, gd


class _LookAt(torch.autograd.Function):
    @staticmethod
    def forward(ctx, azim, elev, dist):
        a, e, d, R, T, Cc, bad = _look_at_launch(azim, elev, dist)
        ctx.save_for_backward(a, e, d)
        ctx.set_materialize_grads(False)
        ctx.shapes = (azim.shape, elev.shape, dist.shape)
        ctx.mark_non_differentiable(bad)
        return R, T, Cc, bad

    @staticmethod
    def backward(ctx, gR, gT, gC, _gbad):
        a, e, d = ctx.saved_tensors
        if gR is None and gT is None and gC is None:
            return None, None, None
        ga, ge, gd = _look_at_backward_launch(a, e, d, gR, gT, gC)
        sa, se, sd = ctx.shapes
        return ga.reshape(sa), ge.reshape(se), gd.reshape(sd)


def look_at_view_transform(dist, elev, azim, return_centers=False, return_invalid=False):
    """PyTorch3D's look_at_view_transform(dist, elev, azim) (degrees, at=0, up=+Y) on device, differentiable.
    Returns R (n,3,3), T (n,3) [, C (n,3)] [, invalid-count int32 tensor]."""
    R, T, Cc, bad = _LookAt.apply(azim, elev, dist)
    out = [R, T]
    if return_centers:
        out.append(Cc)
    if return_invalid:
        out.append(bad)
    return tuple(out)


def camera_position_from_spherical_angles(distance, elevation, azimuth, degrees: bool = True):
    """[upstream] cameras.py camera_position_from_spherical_angles(distance, elevation, azimuth) -> (n,3) camera
    centres, as used for the "relative" light (renderer.py:168) and for ViewGCN's graph vertices
    (viewGCN/tools/Trainer_mvt.py:131-133).  Same kernel as look_at_view_transform (SURVEY 8f N4: one launch yields
    R, T and C), differentiable w.r.t. all three inputs.  Inputs may be (B, M): the result is in flat order b*M + m."""
    if not degrees:
        k = 180.0 / math.pi
        elevation, azimuth = elevation * k, azimuth * k
    return _LookAt.apply(azimuth, elevation, distance)[2]


# --------------------------------------------------------------------------------------------------
# packed geometry
# --------------------------------------------------------------------------------------------------
class HostPackedMeshes:
    """A batch of meshes packed on the HOST into pinned memory: verts (Vtot,3) f32, faces (Ftot,3) int32 (mesh-local
    ids) -- or int16 holding UNSIGNED 16-bit ids (torch has no uint16 arithmetic; collate_meshes narrows to it when every mesh
    has at most 65536 vertices: half the faces' bytes on the host-to-device copy, MVR_FACES_U16) --, per-mesh counts.  This is what a DataLoader collate_fn should hand to MVRenderer (SURVEY 8f N1: the
    reference's collate keeps python lists, custom_dataset.py:149-188, and re-packs them on every forward,
    renderer.py:67-77): the packing then runs in the loader's workers, off the training step, and the step itself only
    pays two H2D copies.  Build with collate_meshes()."""

    def __init__(self, verts: torch.Tensor, faces: torch.Tensor, num_verts: Sequence[int], num_faces: Sequence[int],
                 vert_rgb: Optional[torch.Tensor] = None):
        if verts.dim() != 2 or verts.shape[1] != 3 or faces.dim() != 2 or faces.shape[1] != 3:
            raise ValueError("verts must be (Vtot,3) and faces (Ftot,3)")
        if verts.is_cuda or faces.is_cuda:
            raise ValueError("HostPackedMeshes holds host tensors; use PackedMeshes.from_packed for device arrays")
        if verts.dtype != torch.float32 or faces.dtype not in (torch.int32, torch.int16):
            raise ValueError("verts must be float32 and faces int32 (or int16 holding uint16 ids)")
        if faces.dtype == torch.int16 and max(num_verts, default=0) > 65536:
            raise ValueError("16-bit faces need meshes of at most 65536 vertices")
        if sum(num_verts) != verts.shape[0] or sum(num_faces) != faces.shape[0]:
            raise ValueError("packed arrays do not match the per-mesh counts")
        self.verts, self.faces = verts.contiguous(), faces.contiguous()
        self.num_verts, self.num_faces = [int(x) for x in num_verts], [int(x) for x in num_faces]
        self.vert_rgb = vert_rgb
        # per-batch metadata the step would otherwise rebuild on every forward: prefix offsets (one small pinned tensor,
        # [vert_off | face_off]) and the totals / maxima that size the grids
        self.vert_off_host, self.face_off_host = [0], [0]
        for a in self.num_verts:
            self.vert_off_host.append(self.vert_off_host[-1] + a)
        for a in self.num_faces:
            self.face_off_host.append(self.face_off_host[-1] + a)
        offs = torch.tensor(self.vert_off_host + self.face_off_host, dtype=torch.int32)
        self.offs = offs.pin_memory() if verts.is_pinned() else offs

    def __len__(self):
        return len(self.num_verts)

    def is_pinned(self):
        return self.verts.is_pinned() and self.faces.is_pinned() and self.offs.is_pinned()

    def pin_memory(self):
        """Pinned copy (or self when already pinned).  torch's DataLoader(pin_memory=True) calls this on the batch in its
        pin thread of the MAIN process: batches collated in forked workers come back through shared memory, un-pinned
        (workers must not touch CUDA), and are pinned here, off the training step."""
        if self.is_pinned():
            return self
        hp = HostPackedMeshes.__new__(HostPackedMeshes)
        hp.__dict__.update(self.__dict__)
        hp.verts, hp.faces, hp.offs = self.verts.pin_memory(), self.faces.pin_memory(), self.offs.pin_memory()
        return hp

    def verts_list(self):
        return list(torch.split(self.verts, self.num_verts))

    def faces_list(self):
        f = self.faces if self.faces.dtype == torch.int32 else self.faces.to(torch.int32) & 0xFFFF
        return list(torch.split(f, self.num_faces))


def _in_loader_worker() -> bool:
    try:
        from torch.utils.data import get_worker_info
        return get_worker_info() is not None
    except Exception:
        return False


def collate_meshes(meshes, pin_memory: Optional[bool] = None, vert_rgb: Optional[torch.Tensor] = None,
                   narrow_faces: Optional[bool] = None) -> HostPackedMeshes:
    """Pack a list of meshes (objects with verts_list()/faces_list(), or (verts, faces) pairs) into one
    HostPackedMeshes with the library's multi-threaded gather (int64 faces are narrowed to int32).  Host only: usable
    as a DataLoader collate_fn.
    pin_memory=None (default): pinned when called in the main process with CUDA available, pageable inside a DataLoader
    worker -- a forked worker must not initialise CUDA (run_mvtn.py:110 uses num_workers=6), and its batch travels back
    through shared memory anyway; DataLoader(pin_memory=True) then pins it via HostPackedMeshes.pin_memory() in the main
    process, and PackedMeshes.from_host_packed stages whatever is still pageable through a reusable pinned buffer.
    narrow_faces=None (default): the faces travel as uint16 when every mesh has at most 65536 vertices (3.8 -> 1.9 MB for 32
    ModelNet-sized meshes), as int32 otherwise; True insists (ValueError when a mesh is too large), False keeps int32."""
    from .structures import unpack_mesh_list
    verts, faces = unpack_mesh_list(meshes)
    if len(verts) != len(faces):
        raise ValueError("verts and faces lists differ in length")
    for v, f in zip(verts, faces):
        if v.dim() != 2 or v.shape[1] != 3 or f.dim() != 2 or f.shape[1] != 3:
            raise ValueError("verts must be (V,3) and faces (F,3)")
    nv = [int(v.shape[0]) for v in verts]
    nf = [int(f.shape[0]) for f in faces]
    if pin_memory is None:
        pin_memory = not _in_loader_worker()
    pin = bool(pin_memory) and not _in_loader_worker() and torch.cuda.is_available()
    small = max(nv, default=0) <= 65536
    if narrow_faces and not small:
        raise ValueError("narrow_faces=True needs meshes of at most 65536 vertices")
    narrow = small if narrow_faces is None else bool(narrow_faces)
    v_host = torch.empty((sum(nv), 3), dtype=torch.float32, pin_memory=pin)
    f_host = torch.empty((sum(nf), 3), dtype=torch.int16 if narrow else torch.int32, pin_memory=pin)
    if len(verts):
        import ctypes as C
        fdt = torch.int32 if all(f.dtype == torch.int32 for f in faces) else torch.int64
        v_src = [_host_array(v, torch.float32) for v in verts]
        f_src = [_host_array(f, fdt) for f in faces]
        n = len(v_src)
        vp = (C.c_void_p * n)(*[t.data_ptr() for t in v_src]); vc = (C.c_int64 * n)(*[t.numel() for t in v_src])
        fp = (C.c_void_p * n)(*[t.data_ptr() for t in f_src]); fc = (C.c_int64 * n)(*[t.numel() for t in f_src])
        lib = L.load()      # narrow: ids saturated to [0, 65535] on the way (out-of-range ids are clamped by mvr_mesh_prepare either way)
        L.check(lib.mvr_host_stage_meshes_packed(vp, vc, fp, fc, n, 8 if fdt == torch.int64 else 4, 2 if narrow else 4, v_host.data_ptr(),
                                                 f_host.data_ptr(), None, None, None, None, None), "mvr_host_stage_meshes_packed")
    return HostPackedMeshes(v_host, f_host, nv, nf, vert_rgb=vert_rgb)


class PackedMeshes:
    """Device-resident packed batch of meshes: float4 vertices / unit vertex normals / colours and
    int4 faces, built by mvr_mesh_prepare.  Replaces Meshes(verts, faces) + Textures(verts_rgb) +
    verts_normals_packed() (renderer.py:67-77); can be cached across iterations (SURVEY 8f N1)."""

    _pending = None
    _inflight = None      # the instance whose staging job is running on the library's thread (at most one)

    def __init__(self, verts: Sequence[torch.Tensor], faces: Sequence[torch.Tensor], device,
                 vert_rgb: Optional[torch.Tensor] = None):
        """verts: list of (V_b,3) float tensors, faces: list of (F_b,3) int tensors (any device).  Host lists
        are gathered by native threads into one pinned buffer per array and copied with ONE async H2D each
        instead of the reference's 2B small copies (renderer.py:67-68)."""
        self._pending = None
        self._begin(verts, faces, device, vert_rgb, overlap=False)
        self.finish()

    @classmethod
    def begin(cls, verts: Sequence[torch.Tensor], faces: Sequence[torch.Tensor], device,
              vert_rgb: Optional[torch.Tensor] = None, overlap: bool = False):
        """Deferred construction: validate now, stage + build the device geometry in .finish().  MVRenderer uses it to
        enqueue the camera kernel and build its constants BEFORE the meshes are staged, so that the rasterizer launch
        follows mvr_mesh_prepare with as little host work in between as possible.
        overlap=True additionally starts the gather + H2D at once on the library's staging thread and its private helper pool
        (mvr_host_stage_meshes_packed_begin); finish() joins it.  MVRenderer's default since the pool no longer runs an OpenMP team
        (two teams, the caller's spinning, cost 1.92 vs 1.30 ms per end-to-end step at BASELINE configs[1]; the pool: 1.26)."""
        self = cls.__new__(cls)
        self._pending = None
        self._begin(verts, faces, device, vert_rgb, overlap=overlap, defer=not overlap)
        return self

    def _begin(self, verts, faces, device, vert_rgb, overlap, defer=False):
        device = torch.device(device)
        if device.type != "cuda":
            raise L.MVRError("PackedMeshes needs a CUDA device: mvtn_b200 has no CPU path")
        if len(verts) != len(faces):
            raise ValueError("verts and faces lists differ in length")
        for v, f in zip(verts, faces):
            if v.dim() != 2 or v.shape[1] != 3 or f.dim() != 2 or f.shape[1] != 3:
                raise ValueError("verts must be (V,3) and faces (F,3)")
        self.B = len(verts)                   # known before finish(): MVRenderer validates against them early
        self.per_vertex_rgb = vert_rgb is not None
        self.device = device
        if defer:
            self._pending = ("deferred", list(verts), list(faces), device, vert_rgb)
            return
        if overlap and PackedMeshes._inflight is not None:
            # one staging thread and one set of pinned buffers: a batch that is still in flight is completed before the next one starts
            PackedMeshes._inflight.finish()
        self._pending = self._stage(verts, faces, device, vert_rgb, overlap)
        if self._pending[6] is not None:      # (a job id: the gather runs on the library's thread until finish() joins it)
            PackedMeshes._inflight = self

    @staticmethod
    def _stage(verts, faces, device, vert_rgb, overlap):
        nv = [int(v.shape[0]) for v in verts]
        nf = [int(f.shape[0]) for f in faces]
        tv, tf = sum(nv), sum(nf)
        job = None
        keep = None
        offs = None
        if len(verts) == 0:
            v_dev = torch.zeros((0, 3), dtype=torch.float32, device=device)
            f_dev = torch.zeros((0, 3), dtype=torch.int64, device=device)
        else:
            fdt = torch.int32 if faces[0].dtype == torch.int32 and all(f.dtype == torch.int32 for f in faces) else torch.int64
            if verts[0].is_cuda and all(v.is_cuda for v in verts) and all(f.is_cuda for f in faces):
                v_dev = torch.cat([v.detach().to(torch.float32) for v in verts], 0)
                f_dev = torch.cat([f.detach().to(fdt) for f in faces], 0)
            else:
                # multi-threaded gather into pinned memory (faces narrowed int64 -> int32 on the way) with the
                # vertices' H2D copy in flight while the faces are gathered: one native call
                v_src = [_host_array(v, torch.float32) for v in verts]
                f_src = [_host_array(f, fdt) for f in faces]
                # ... and to uint16 when every mesh has at most 65536 vertices (MVR_FACES_U16): 5.8 -> 3.8 MB at BASELINE configs[1]
                narrow = max(nv) <= 65536
                fdev_t = torch.int16 if narrow else torch.int32
                v_host = _staging("verts", device, tv * 3, torch.float32)
                f_host = _staging("faces16" if narrow else "faces", device, tf * 3, fdev_t)
                v_dev = torch.empty((tv, 3), dtype=torch.float32, device=device)
                f_dev = torch.empty((tf, 3), dtype=fdev_t, device=device)
                # the offset table travels with the same call (2B + 2 words, first on the wire)
                offs_h = _staging("offs", device, 2 * len(nv) + 2, torch.int32)
                offs = torch.empty(2 * len(nv) + 2, dtype=torch.int32, device=device)
                job, keep = _stage_meshes(v_src, f_src, 8 if fdt == torch.int64 else 4, v_host, f_host, v_dev, f_dev, device,
                                          overlap, offs_h, offs)
        return (v_dev, f_dev, nv, nf, device, vert_rgb, job, keep, offs)

    def finish(self):
        """Stage (if deferred) or join the staging job (if overlapped), then build the packed device geometry
        (mvr_mesh_prepare).  Idempotent."""
        if self._pending is None:
            return self
        pending, self._pending = self._pending, None
        if PackedMeshes._inflight is self:
            PackedMeshes._inflight = None
        if pending[0] == "deferred":
            _, verts, faces, device, vert_rgb = pending
            pending = self._stage(verts, faces, device, vert_rgb, overlap=False)
        v_dev, f_dev, nv, nf, device, vert_rgb, job, keep, offs = pending
        offsets = None
        if offs is not None:
            from itertools import accumulate
            offsets = (list(accumulate(nv, initial=0)), list(accumulate(nf, initial=0)), offs)
        # everything that does not read the staged bytes happens BEFORE the join: while the staging thread still gathers, this one
        # is idle anyway
        self._init_packed(v_dev, f_dev, nv, nf, device, vert_rgb, offsets, prepare=False)
        if job is not None:
            L.check(L.load().mvr_host_stage_meshes_end(job), "mvr_host_stage_meshes_end")
        if keep is not None:
            _staging_done(device)
        del keep
        self.refresh()
        return self

    @classmethod
    def from_host_packed(cls, hp: "HostPackedMeshes", device, vert_rgb: Optional[torch.Tensor] = None, copy_stream: bool = False):
        """Two async H2D copies of an already packed (ideally pinned) host batch + mvr_mesh_prepare.
        copy_stream=True: the copies go through a dedicated stream (the compute stream waits on an event), so that in a
        loop that does not synchronise every step they overlap with the previous step's kernels instead of queueing
        behind them (5.8 MB = 0.11 ms per step at C2)."""
        device = torch.device(device)
        if device.type != "cuda":
            raise L.MVRError("PackedMeshes needs a CUDA device: mvtn_b200 has no CPU path")
        self = cls.__new__(cls)
        if not hp.is_pinned():
            # a batch that came out of a DataLoader worker without DataLoader(pin_memory=True): copy it into reusable pinned
            # staging buffers first, so that the H2D below is still asynchronous (a pageable source would block the host)
            src = hp
            hp = HostPackedMeshes.__new__(HostPackedMeshes)
            hp.__dict__.update(src.__dict__)
            v_st = _staging("hp_verts", device, src.verts.numel(), torch.float32).view(-1, 3)
            f_st = _staging("hp_faces16" if src.faces.dtype == torch.int16 else "hp_faces", device, src.faces.numel(), src.faces.dtype).view(-1, 3)
            o_st = _staging("hp_offs", device, src.offs.numel(), torch.int32)
            v_st.copy_(src.verts); f_st.copy_(src.faces); o_st.copy_(src.offs)
            hp.verts, hp.faces, hp.offs = v_st, f_st, o_st
            staged = True
        else:
            staged = False
        if copy_stream:
            cur = torch.cuda.current_stream(device)
            cs = _copy_streams.get(device.index)
            if cs is None:
                cs = _copy_streams[device.index] = torch.cuda.Stream(device)
            with torch.cuda.stream(cs):
                v_dev = hp.verts.to(device, non_blocking=True)
                f_dev = hp.faces.to(device, non_blocking=True)
                offs = hp.offs.to(device, non_blocking=True)
            cur.wait_stream(cs)
            for t in (v_dev, f_dev, offs):
                t.record_stream(cur)
        else:
            v_dev = hp.verts.to(device, non_blocking=True)
            f_dev = hp.faces.to(device, non_blocking=True)
            offs = hp.offs.to(device, non_blocking=True)
        if staged:
            _staging_done(device)
        self._init_packed(v_dev, f_dev, hp.num_verts, hp.num_faces, device,
                          vert_rgb if vert_rgb is not None else hp.vert_rgb,
                          offsets=(hp.vert_off_host, hp.face_off_host, offs))
        return self

    @classmethod
    def from_packed(cls, verts: torch.Tensor, faces: torch.Tensor, num_verts: Sequence[int], num_faces: Sequence[int],
                    vert_rgb: Optional[torch.Tensor] = None):
        """Already-packed device arrays: verts (Vtot,3) f32, faces (Ftot,3) int32/int64 (mesh-local ids)."""
        self = cls.__new__(cls)
        _require_cuda(verts, "verts")
        _require_cuda(faces, "faces")
        self._init_packed(verts, faces, list(num_verts), list(num_faces), verts.device, vert_rgb)
        return self

    def _init_packed(self, v_dev, f_dev, nv, nf, device, vert_rgb, offsets=None, prepare=True):
        lib = L.load()
        self.B = len(nv)
        self.num_verts, self.num_faces = nv, nf
        if offsets is not None:          # precomputed at collate time (HostPackedMeshes), already on their way to the device
            voff, foff, offs = offsets
        else:
            voff, foff = [0], [0]
            for a in nv:
                voff.append(voff[-1] + a)
            for a in nf:
                foff.append(foff[-1] + a)
            offs_h = _staging("offs", device, 2 * self.B + 2, torch.int32)
            offs_h.copy_(torch.tensor(voff + foff, dtype=torch.int32))
            offs = offs_h.to(device, non_blocking=True)
            _staging_done(device)
        self.total_verts, self.total_faces = voff[-1], foff[-1]
        self.max_faces = max(nf) if nf else 0
        self.max_verts = max(nv) if nv else 0
        if v_dev.shape[0] != self.total_verts or f_dev.shape[0] != self.total_faces:
            raise ValueError("packed arrays do not match the per-mesh counts")
        self.vert_off_host, self.face_off_host = voff, foff
        self.device = device
        self.per_vertex_rgb = vert_rgb is not None
        self.verts = _f32c(v_dev)
        if f_dev.dtype not in (torch.int32, torch.int64, torch.int16):      # (int16: uint16 ids of a narrowed host batch)
            f_dev = f_dev.to(torch.int64)
        if f_dev.dtype == torch.int16 and self.max_verts > 65536:
            raise ValueError("16-bit faces need meshes of at most 65536 vertices")
        self.faces = f_dev if f_dev.is_contiguous() else f_dev.contiguous()
        self.vert_off, self.face_off = offs[: self.B + 1], offs[self.B + 1:]
        flags = L.FACES_I64 if self.faces.dtype == torch.int64 else (L.FACES_U16 if self.faces.dtype == torch.int16 else 0)
        rgb = None
        if vert_rgb is not None:
            rgb = _f32c(vert_rgb.to(device)).reshape(-1, 3)
            if rgb.shape[0] != self.total_verts:
                raise ValueError("vert_rgb must hold one colour per packed vertex")
            flags |= L.RGB_PER_ELEMENT
        nbytes = lib.mvr_mesh_geometry_bytes(self.total_verts, self.total_faces)
        self.geometry = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=device)
        self._rgb, self._prep_flags = rgb, flags
        if prepare:
            self.refresh()

    def refresh(self):
        """(Re)build the packed float4 / int4 geometry and the vertex normals from self.verts / self.faces
        (mvr_mesh_prepare): call it after updating self.verts in place.  Pure device work on the current stream."""
        if self.B == 0:
            return self
        with _on(self.device):
            L.check(L.load().mvr_mesh_prepare(_ptr(self.verts), _ptr(self.faces), _ptr(self.vert_off), _ptr(self.face_off),
                                              self.B, self.total_verts, self.total_faces, self.max_faces, _ptr(self._rgb),
                                              self._prep_flags, _ptr(self.geometry), self.geometry.numel(),
                                              _stream(self.device)), "mvr_mesh_prepare")
        return self

    def faces_global(self) -> torch.Tensor:
        """(Ftot,3) int64 faces indexing the PACKED vertex array (mesh-local id + the mesh's vertex offset)."""
        if getattr(self, "_faces_global", None) is None:
            counts = torch.tensor(self.num_faces, device=self.device)
            off = torch.repeat_interleave(self.vert_off[:-1].to(torch.int64), counts)
            f = self.faces.to(torch.int64)
            if self.faces.dtype == torch.int16:
                f = f & 0xFFFF
            self._faces_global = f + off[:, None]
        return self._faces_global

    def vertex_normals(self) -> torch.Tensor:
        out = torch.empty((self.total_verts, 3), dtype=torch.float32, device=self.device)
        with _on(self.device):
            L.check(L.load().mvr_mesh_get_normals(_ptr(self.geometry), self.total_verts, self.total_faces, _ptr(out),
                                                  _stream(self.device)), "mvr_mesh_get_normals")
        return out


# --------------------------------------------------------------------------------------------------
# mesh rendering
# --------------------------------------------------------------------------------------------------
def _mesh_forward_launch(geom: "PackedMeshes", M, R, T, Cc, light, obj_rgb, bg_rgb, k00, k11, z_clip, H, W, K, flags,
                         want_fragments, out_norm, out_dtype, blur_radius=0.0):
    """Argument normalisation, output allocation and ONE mvr_mesh_forward call.  Returns (saved, images, extras): `saved` is
    what the matching backward launch needs."""
    lib = L.load()
    dev = geom.device
    R, T, Cc = _f32c(R), _f32c(T), _f32c(Cc)
    N = geom.B * M
    if R.shape[0] != N:
        raise ValueError(f"expected {N} cameras (B*M), got {R.shape[0]}")
    light = _f32c(light).reshape(-1, 3)
    if light.shape[0] not in (1, N):
        raise ValueError("light direction must be (1,3) or (B*M,3)")
    light_stride = 0 if light.shape[0] == 1 else 3
    obj_rgb = None if obj_rgb is None else _f32c(obj_rgb)
    bg_rgb = _f32c(bg_rgb)
    if geom.per_vertex_rgb:
        flags |= L.RGB_PER_ELEMENT
    img_dtype, dt_flag = _image_dtype(out_dtype)
    flags |= dt_flag
    images = torch.empty((N, 3, H, W), dtype=img_dtype, device=dev)
    p2f = torch.empty((N, H, W, K), dtype=torch.int32, device=dev)
    zbuf = bary = dists = None
    if want_fragments:
        zbuf = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
        bary = torch.empty((N, H, W, K, 3), dtype=torch.float32, device=dev)
        dists = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
    geom.finish()
    counters = torch.empty(L.NUM_COUNTERS, dtype=torch.int64, device=dev)      # zeroed by mvr_mesh_forward
    ws_bytes = lib.mvr_mesh_workspace_bytes(geom.B, M, H, W, K, geom.total_verts, geom.total_faces)
    ws = workspace(dev, ws_bytes, _mesh_owner=True)
    ws_flags, ws_commit = _ws_mesh_flags_forward(dev, ws, (geom.B, M, H, W, K, geom.total_verts))
    with _on(dev):
        L.check(lib.mvr_mesh_forward(_ptr(geom.geometry), _ptr(geom.vert_off), _ptr(geom.face_off), geom.B, M,
                                     geom.total_verts, geom.total_faces, geom.max_verts, geom.max_faces, _ptr(R), _ptr(T), _ptr(Cc),
                                     _ptr(light), light_stride, _ptr(obj_rgb), _ptr(bg_rgb), k00, k11, z_clip, float(blur_radius), H, W,
                                     K, flags | ws_flags, out_norm, _ptr(images), _ptr(p2f), _ptr(zbuf), _ptr(bary), _ptr(dists),
                                     _ptr(counters), _ptr(ws), ws.numel(), _stream(dev)), "mvr_mesh_forward")
    cfg = (k00, k11, H, W, K, flags, out_norm, light_stride, z_clip, ws_commit())
    saved = (R, T, Cc, light, obj_rgb if obj_rgb is not None else bg_rgb, p2f)
    extras = [p2f, counters]
    if want_fragments:
        extras += [zbuf, bary, dists]
    return cfg, saved, images, extras


def _mesh_backward_launch(geom: "PackedMeshes", M, cfg, saved, g_images, want_verts, angles=None):
    """ONE mvr_mesh_backward call -> (gR, gT, gC, gV | None) (gV includes the chain through the vertex normals).  angles =
    (azim, elev, dist) flat fp32: mvr_mesh_backward_angles instead, whose last kernel also applies the camera backward ->
    (g_azim, g_elev, g_dist, gV | None)."""
    lib = L.load()
    R, T, Cc, light, obj_rgb, p2f = saved
    k00, k11, H, W, K, flags, out_norm, light_stride, z_clip, ws_token = cfg
    dev = geom.device
    N = geom.B * M
    g_images = _grad_like_images(g_images, flags)
    if angles is None:
        g = torch.empty(15 * N, dtype=torch.float32, device=dev)
        gR, gT, gC = g[: 9 * N].view(N, 3, 3), g[9 * N: 12 * N].view(N, 3), g[12 * N:].view(N, 3)
    else:
        g = torch.empty(3 * N, dtype=torch.float32, device=dev)
        ga, ge, gd = g[:N], g[N: 2 * N], g[2 * N:]
    gV = gN = None
    if want_verts:
        gV = torch.zeros((geom.total_verts, 3), dtype=torch.float32, device=dev)
        gN = torch.zeros((geom.total_verts, 3), dtype=torch.float32, device=dev)
    ws_bytes = lib.mvr_mesh_workspace_bytes(geom.B, M, H, W, K, geom.total_verts, geom.total_faces)
    ws = workspace(dev, ws_bytes, _mesh_owner=True)
    flags = flags | _ws_mesh_flags_backward(dev, ws, ws_token)
    if angles is not None:
        az, el, di = angles
        with _on(dev):
            L.check(lib.mvr_mesh_backward_angles(_ptr(geom.geometry), _ptr(geom.vert_off), _ptr(geom.face_off), geom.B, M,
                                                 geom.total_verts, geom.total_faces, geom.max_verts, _ptr(R), _ptr(T), _ptr(Cc),
                                                 _ptr(light), light_stride, _ptr(obj_rgb), k00, k11, z_clip, H, W, K, flags, out_norm,
                                                 _ptr(p2f), _ptr(g_images), _ptr(az), _ptr(el), _ptr(di), _ptr(ga), _ptr(ge), _ptr(gd),
                                                 None, None, None, _ptr(gV), _ptr(gN), _ptr(ws), ws.numel(),
                                                 _stream(dev)), "mvr_mesh_backward_angles")
    else:
        with _on(dev):
            L.check(lib.mvr_mesh_backward(_ptr(geom.geometry), _ptr(geom.vert_off), _ptr(geom.face_off), geom.B, M,
                                          geom.total_verts, geom.total_faces, geom.max_verts, _ptr(R), _ptr(T), _ptr(Cc), _ptr(light),
                                          light_stride, _ptr(obj_rgb), k00, k11, z_clip, H, W, K, flags, out_norm, _ptr(p2f),
                                          _ptr(g_images), _ptr(gR), _ptr(gT), _ptr(gC), _ptr(gV), _ptr(gN), _ptr(ws),
                                          ws.numel(), _stream(dev)), "mvr_mesh_backward")
    if gV is not None:
        # the kernel returned d/d verts through projection + interpolated position, and d/d unit normals; the
        # normals -> verts chain ([upstream] Meshes._compute_vertex_normals) is mvr_mesh_normals_backward
        with _on(dev):
            L.check(lib.mvr_mesh_normals_backward(_ptr(geom.geometry), _ptr(geom.vert_off), _ptr(geom.face_off), geom.B,
                                                  geom.total_verts, geom.total_faces, geom.max_faces, _ptr(gN), _ptr(gV),
                                                  _stream(dev)), "mvr_mesh_normals_backward")
    if angles is not None:
        return ga, ge, gd, gV
    return gR, gT, gC, gV


class _MeshRender(torch.autograd.Function):
    @staticmethod
    def forward(ctx, R, T, Cc, verts, geom: PackedMeshes, M, light, obj_rgb, bg_rgb, k00, k11, z_clip, H, W, K, flags,
                want_fragments, out_norm=None, out_dtype=None):
        # `verts` (packed (Vtot,3), same values as geom.verts) only carries autograd history for vertex gradients
        cfg, saved, images, extras = _mesh_forward_launch(geom, M, R, T, Cc, light, obj_rgb, bg_rgb, k00, k11, z_clip, H, W, K,
                                                          flags, want_fragments, out_norm, out_dtype)
        ctx.set_materialize_grads(False)      # no zero-filled "gradients" for pix_to_face & co (77 MB at C2)
        ctx.geom, ctx.M, ctx.cfg = geom, M, cfg
        ctx.save_for_backward(*saved)
        ctx.mark_non_differentiable(*extras)
        return (images, *extras)

    @staticmethod
    def backward(ctx, g_images, *_unused):
        if g_images is None:
            return (None,) * 19
        gR, gT, gC, gV = _mesh_backward_launch(ctx.geom, ctx.M, ctx.cfg, ctx.saved_tensors, g_images, ctx.needs_input_grad[3])
        return (gR, gT, gC, gV) + (None,) * 15


class _MeshRenderFromAngles(torch.autograd.Function):
    """look_at + mesh render as ONE autograd node: (azim, elev, dist) -> images (+ R, T, C, pix_to_face, counters).
    Same two C-ABI launches as _LookAt followed by _MeshRender, without the second Function.apply and the tensor
    plumbing between them -- on the end-to-end step the GPU has the geometry before the host has reached
    mvr_mesh_forward, so host microseconds in front of that call are step time (DESIGN.md section 5).
    light=None: the "relative" light, i.e. the (detached) camera centres (renderer.py:168).
    after_cameras: a FlagSink (the flag travels to its pinned word behind the camera kernel, copy and event issued by the library
    call), or a callable invoked with the invalid-rotation flag tensor right after the camera kernel has been enqueued (the
    renderer records its event there, in front of the rasterizer)."""

    @staticmethod
    def forward(ctx, azim, elev, dist, geom: PackedMeshes, M, light, obj_rgb, bg_rgb, k00, k11, z_clip, H, W, K, flags,
                out_norm, out_dtype, after_cameras):
        sink = after_cameras if isinstance(after_cameras, FlagSink) else None
        a, e, d, R, T, Cc, bad = _look_at_launch(azim, elev, dist, sink)
        if after_cameras is not None and sink is None:
            after_cameras(bad)
        geom.finish()      # a deferred / worker-thread staging (PackedMeshes.begin) ends here, behind the camera launch
        cfg, saved, images, extras = _mesh_forward_launch(geom, M, R, T, Cc, Cc if light is None else light, obj_rgb, bg_rgb,
                                                          k00, k11, z_clip, H, W, K, flags, False, out_norm, out_dtype)
        ctx.set_materialize_grads(False)
        ctx.geom, ctx.M, ctx.cfg = geom, M, cfg
        ctx.shapes = (azim.shape, elev.shape, dist.shape)
        ctx.save_for_backward(a, e, d, *saved)
        ctx.mark_non_differentiable(bad, *extras)
        return (images, R, T, Cc, bad, *extras)

    @staticmethod
    def backward(ctx, g_images, gR_ext, gT_ext, gC_ext, *_unused):
        if g_images is None and gR_ext is None and gT_ext is None and gC_ext is None:
            return (None,) * 18
        a, e, d = ctx.saved_tensors[:3]
        if g_images is not None and gR_ext is None and gT_ext is None and gC_ext is None:
            # nothing arrives through the cameras object (the usual case): rasterizer backward, reduction and camera backward in
            # ONE call ending in (d azim, d elev, d dist) -- mvr_mesh_backward_angles
            ga, ge, gd, _ = _mesh_backward_launch(ctx.geom, ctx.M, ctx.cfg, ctx.saved_tensors[3:], g_images, False, (a, e, d))
            sa, se, sd = ctx.shapes
            return (ga.reshape(sa), ge.reshape(se), gd.reshape(sd)) + (None,) * 15
        gR = gT = gC = None
        if g_images is not None:
            gR, gT, gC, _ = _mesh_backward_launch(ctx.geom, ctx.M, ctx.cfg, ctx.saved_tensors[3:], g_images, False)
        # R, T, C are outputs too (the cameras object): gradients a caller sends through them join the renderer's
        if gR_ext is not None:
            gR = gR_ext if gR is None else gR + gR_ext
        if gT_ext is not None:
            gT = gT_ext if gT is None else gT + gT_ext
        if gC_ext is not None:
            gC = gC_ext if gC is None else gC + gC_ext
        ga, ge, gd = _look_at_backward_launch(a, e, d, gR, gT, gC)
        sa, se, sd = ctx.shapes
        return (ga.reshape(sa), ge.reshape(se), gd.reshape(sd)) + (None,) * 15


SOFT_SHADERS = {"soft_phong": 0, "soft_silhouette": 1}


class _MeshRenderSoft(torch.autograd.Function):
    """Blurred rasterizer (K fragments per pixel, signed edge distances, clipped barycentrics) + soft blend as one autograd
    node: (R, T, C) -> RGBA (n,4,H,W).  [upstream] MeshRasterizer(blur_radius, faces_per_pixel) + SoftPhongShader
    (softmax_rgb_blend) / SoftSilhouetteShader (sigmoid_alpha_blend); renderer.py:4-6, :91-92 (SURVEY 8f N3)."""

    @staticmethod
    def forward(ctx, R, T, Cc, geom: PackedMeshes, M, light, obj_rgb, bg_rgb, k00, k11, z_clip, H, W, K, flags, blur_radius,
                mode, sigma, gamma, znear, zfar):
        lib = L.load()
        cfg, saved, _hard, extras = _mesh_forward_launch(geom, M, R, T, Cc, light, obj_rgb, bg_rgb, k00, k11, z_clip, H, W, K, flags,
                                                         True, None, None, blur_radius=blur_radius)
        p2f, counters, zbuf, bary, dists = extras
        Rs, Ts, Cs, lt, col, _ = saved
        dev = geom.device
        N = geom.B * M
        rgba = torch.empty((N, 4, H, W), dtype=torch.float32, device=dev)
        light_stride = cfg[7]
        fl = cfg[5]
        bg = _f32c(bg_rgb)
        with _on(dev):
            L.check(lib.mvr_mesh_soft_blend_forward(_ptr(geom.geometry), _ptr(geom.vert_off), _ptr(geom.face_off), geom.B, M,
                                                    geom.total_verts, geom.total_faces, _ptr(Cs), _ptr(lt), light_stride,
                                                    _ptr(col), _ptr(bg), H, W, K, fl, mode, sigma, gamma, znear, zfar, _ptr(p2f),
                                                    _ptr(zbuf), _ptr(bary), _ptr(dists), _ptr(rgba), _stream(dev)),
                    "mvr_mesh_soft_blend_forward")
        ctx.set_materialize_grads(False)
        ctx.geom, ctx.M = geom, M
        ctx.cfg = (k00, k11, z_clip, blur_radius, H, W, K, fl, light_stride, mode, sigma, gamma, znear, zfar)
        ctx.save_for_backward(Rs, Ts, Cs, lt, col, bg, p2f)
        ctx.mark_non_differentiable(p2f, counters, zbuf, bary, dists)
        return rgba, p2f, counters, zbuf, bary, dists

    @staticmethod
    def backward(ctx, g_rgba, *_unused):
        if g_rgba is None:
            return (None,) * 21
        lib = L.load()
        geom, M = ctx.geom, ctx.M
        R, T, Cc, light, col, bg, p2f = ctx.saved_tensors
        k00, k11, z_clip, blur_radius, H, W, K, fl, light_stride, mode, sigma, gamma, znear, zfar = ctx.cfg
        dev = geom.device
        N = geom.B * M
        g_rgba = _f32c(g_rgba)
        g = torch.empty(15 * N, dtype=torch.float32, device=dev)
        gR, gT, gC = g[: 9 * N].view(N, 3, 3), g[9 * N: 12 * N].view(N, 3), g[12 * N:].view(N, 3)
        ws = workspace(dev, lib.mvr_mesh_workspace_bytes(geom.B, M, H, W, K, geom.total_verts, geom.total_faces))
        with _on(dev):
            L.check(lib.mvr_mesh_soft_backward(_ptr(geom.geometry), _ptr(geom.vert_off), _ptr(geom.face_off), geom.B, M,
                                               geom.total_verts, geom.total_faces, geom.max_verts, _ptr(R), _ptr(T), _ptr(Cc),
                                               _ptr(light), light_stride, _ptr(col), _ptr(bg), k00, k11, z_clip, blur_radius, H, W, K,
                                               fl, mode, sigma,
                                               gamma, znear, zfar, _ptr(p2f), _ptr(g_rgba), _ptr(gR), _ptr(gT), _ptr(gC), _ptr(ws),
                                               ws.numel(), _stream(dev)), "mvr_mesh_soft_backward")
        return (gR, gT, gC) + (None,) * 18


def render_meshes_from_angles(geom: PackedMeshes, M: int, azim, elev, dist, light, obj_rgb, bg_rgb, image_size,
                              faces_per_pixel=1, cull_backfaces=False, perspective_correct=True, fov=60.0, znear=1.0,
                              z_clip: Optional[float] = None, normalize=None, out_dtype=None, after_cameras=None):
    """look_at_view_transform + render_meshes in one autograd node (see _MeshRenderFromAngles).
    Returns images (B*M,3,H,W), (R, T, C, invalid flag), fragments dict."""
    k00, k11 = fov_projection_scale(fov, znear, aspect=1.0)
    if z_clip is None:
        z_clip = znear / 2 if perspective_correct else -1.0
    flags = (L.PERSPECTIVE_CORRECT if perspective_correct else 0) | (L.CULL_BACKFACES if cull_backfaces else 0)
    H, W = _hw(image_size)
    images, R, T, Cc, bad, p2f, counters = _MeshRenderFromAngles.apply(
        azim, elev, dist, geom, M, light, obj_rgb, bg_rgb, k00, k11, float(z_clip), H, W, int(faces_per_pixel), flags,
        _out_norm(normalize), out_dtype, after_cameras)
    return images, (R, T, Cc, bad), {"pix_to_face": p2f, "counters": counters}


def render_meshes(geom: PackedMeshes, M: int, R, T, Cc, light, obj_rgb, bg_rgb, image_size: int, faces_per_pixel=1,
                  cull_backfaces=False, perspective_correct=True, fov=60.0, znear=1.0, z_clip: Optional[float] = None,
                  fragments=False, verts: Optional[torch.Tensor] = None, _extra_flags=0, normalize=None, out_dtype=None,
                  shader="hard_phong", blur_radius=0.0, clip_barycentric_coords=None, sigma=1e-4, gamma=1e-4, zfar=100.0):
    """images (B*M,3,H,W) [+ dict of fragments].  HardPhong + hard blend, blur_radius 0 (MVTN's configuration), or --
    shader="soft_phong" / "soft_silhouette" (SURVEY 8f N3) -- RGBA (B*M,4,H,W) from the K = faces_per_pixel fragments of the
    BLURRED rasterizer ([upstream] blur_radius in squared NDC units, clip_barycentric_coords default True iff blur_radius > 0)
    blended by softmax_rgb_blend over per-fragment Phong colours / sigmoid_alpha_blend (sigma, gamma = BlendParams);
    differentiable w.r.t. R, T, C through colours, depths and the signed edge distances (grad_dists).
    `verts`: pass the packed (Vtot,3) vertex tensor the geometry was built from to get gradients w.r.t. it.
    `normalize=(mean, std)` / `out_dtype=torch.bfloat16`: consumer-side fusion (SURVEY 8f N2) -- the kernel writes
    (x - mean) / std (Trainer_mvt.py:41-49) in the dtype the CNN consumes; gradients flow through both."""
    H_, W_ = _hw(image_size)
    k00, k11 = fov_projection_scale(fov, znear, aspect=1.0)
    if z_clip is None:
        z_clip = znear / 2 if perspective_correct else -1.0   # [upstream] MeshRasterizer.forward
    flags = (L.PERSPECTIVE_CORRECT if perspective_correct else 0) | (L.CULL_BACKFACES if cull_backfaces else 0) | _extra_flags
    H, W = _hw(image_size)
    if clip_barycentric_coords is None:
        clip_barycentric_coords = blur_radius > 0
    if shader != "hard_phong":
        if shader not in SOFT_SHADERS:
            raise ValueError("shader must be 'hard_phong', 'soft_phong' or 'soft_silhouette'")
        if verts is not None or normalize is not None or out_dtype not in (None, torch.float32):
            raise ValueError("the soft shaders return fp32 RGBA and gradients w.r.t. the cameras only")
        flags |= L.CLIP_BARYCENTRIC if clip_barycentric_coords else 0
        out = _MeshRenderSoft.apply(R, T, Cc, geom, M, light, obj_rgb, bg_rgb, k00, k11, float(z_clip), H, W, int(faces_per_pixel),
                                    flags, float(blur_radius), SOFT_SHADERS[shader], float(sigma), float(gamma), float(znear), float(zfar))
        return out[0], {"pix_to_face": out[1], "counters": out[2], "zbuf": out[3], "bary_coords": out[4], "dists": out[5]}
    if blur_radius > 0 or clip_barycentric_coords:
        raise ValueError("blur_radius > 0 / clipped barycentrics need shader='soft_phong' or 'soft_silhouette'")
    out = _MeshRender.apply(R, T, Cc, verts, geom, M, light, obj_rgb, bg_rgb, k00, k11, float(z_clip), H, W,
                            int(faces_per_pixel), flags, bool(fragments), _out_norm(normalize), out_dtype)
    images, p2f, counters = out[0], out[1], out[2]
    frag = {"pix_to_face": p2f, "counters": counters}
    if fragments:
        frag.update(zbuf=out[3], bary_coords=out[4], dists=out[5])
    return images, frag


# --------------------------------------------------------------------------------------------------
# point rendering
# --------------------------------------------------------------------------------------------------
def _points_forward_launch(R, T, inv_dist, points, rgb, M, radius, bg_rgb, H, W, K, flags, want_fragments, out_norm, out_dtype):
    """Argument normalisation, output allocation and ONE mvr_points_forward call.
    Returns (cfg, saved, images, extras): cfg / saved are what the matching backward launch needs."""
    lib = L.load()
    _require_cuda(points, "points")
    dev = points.device
    pts = _f32c(points)
    if pts.dim() != 3 or pts.shape[2] != 3:
        raise ValueError("points must be (B,N,3)")
    B, Np, _ = pts.shape
    N = B * M
    R, T, inv_dist = _f32c(R), _f32c(T), _f32c(inv_dist).reshape(-1)
    if R.shape[0] != N or inv_dist.numel() != N:
        raise ValueError(f"expected {N} cameras (B*M)")
    rgb = _f32c(rgb.to(dev))
    if rgb.numel() != 3:
        if rgb.numel() != pts.numel():
            raise ValueError("rgb must be a 3-vector or one colour per point (B,N,3)")
        flags |= L.RGB_PER_ELEMENT
    bg_rgb = _f32c(bg_rgb)
    img_dtype, dt_flag = _image_dtype(out_dtype)
    flags |= dt_flag
    images = torch.empty((N, 3, H, W), dtype=img_dtype, device=dev)
    idx = torch.empty((N, H, W, K), dtype=torch.int32, device=dev)
    zbuf = d2 = None
    if want_fragments:
        zbuf = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
        d2 = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
    ws = workspace(dev, lib.mvr_points_workspace_bytes(B, Np, M, H, W, K, float(radius)))
    # one bit per pixel: the backward pass skips the (typically ~90 %) background without touching idx
    mask = torch.empty(max(lib.mvr_points_hit_mask_words(B, M, H, W), 1), dtype=torch.int32, device=dev)
    call_flags = flags if want_fragments else flags | L.IDX_SPARSE      # idx unwritten where the mask says "background" (_PointFragments)
    with _on(dev):
        L.check(lib.mvr_points_forward(_ptr(pts), _ptr(rgb), B, Np, M, _ptr(R), _ptr(T), _ptr(inv_dist), float(radius),
                                       _ptr(bg_rgb), H, W, K, call_flags, out_norm, _ptr(images), _ptr(idx), _ptr(zbuf), _ptr(d2),
                                       _ptr(mask), _ptr(ws), ws.numel(), _stream(dev)), "mvr_points_forward")
    cfg = (B, Np, M, float(radius), H, W, K, flags, out_norm, rgb.shape, points.shape)
    saved = (R, T, inv_dist, pts, rgb, idx, mask)
    extras = [idx] + ([zbuf, d2] if want_fragments else [mask])
    return cfg, saved, images, extras


def _points_backward_launch(cfg, saved, g_images, want_points, want_rgb):
    """ONE mvr_points_backward call -> (gR, gT, g_scale (flat), g_points | None, g_rgb | None)."""
    lib = L.load()
    R, T, inv_dist, pts, rgb, idx, mask = saved
    B, Np, M, radius, H, W, K, flags, out_norm, rgb_shape, points_shape = cfg
    dev = pts.device
    N = B * M
    g_images = _grad_like_images(g_images, flags)
    g = torch.empty(13 * N, dtype=torch.float32, device=dev)      # one allocation: gR | gT | g_scale
    gR, gT, gs = g[: 9 * N].view(N, 3, 3), g[9 * N: 12 * N].view(N, 3), g[12 * N:]
    gP = torch.zeros_like(pts) if want_points else None
    gF = torch.zeros_like(rgb) if want_rgb else None
    ws_bytes = lib.mvr_points_workspace_bytes(B, Np, M, H, W, K, float(radius))
    ws = workspace(dev, ws_bytes)
    with _on(dev):
        L.check(lib.mvr_points_backward(_ptr(pts), _ptr(rgb), B, Np, M, _ptr(R), _ptr(T), _ptr(inv_dist), radius, H,
                                        W, K, flags, out_norm, _ptr(idx), _ptr(mask), _ptr(g_images), _ptr(gR), _ptr(gT), _ptr(gs),
                                        _ptr(gP), _ptr(gF), _ptr(ws), ws.numel(), _stream(dev)),
                "mvr_points_backward")
    if gP is not None:
        gP = gP.reshape(points_shape)
    if gF is not None:
        gF = gF.reshape(rgb_shape)
    return gR, gT, gs, gP, gF


def _points_backward_angles_launch(cfg, saved, azim, elev, g_images, want_points, want_rgb):
    """ONE mvr_points_backward_angles call -> (g_azim, g_elev, g_dist (flat), g_points | None, g_rgb | None)."""
    lib = L.load()
    R, T, dist, pts, rgb, idx, mask = saved
    B, Np, M, radius, H, W, K, flags, out_norm, rgb_shape, points_shape = cfg
    dev = pts.device
    N = B * M
    g_images = _grad_like_images(g_images, flags)
    g = torch.empty(3 * N, dtype=torch.float32, device=dev)      # one allocation: g_azim | g_elev | g_dist
    ga, ge, gd = g[:N], g[N: 2 * N], g[2 * N:]
    gP = torch.zeros_like(pts) if want_points else None
    gF = torch.zeros_like(rgb) if want_rgb else None
    ws = workspace(dev, lib.mvr_points_workspace_bytes(B, Np, M, H, W, K, float(radius)))
    with _on(dev):
        L.check(lib.mvr_points_backward_angles(_ptr(pts), _ptr(rgb), B, Np, M, _ptr(R), _ptr(T), _ptr(azim), _ptr(elev), _ptr(dist), radius,
                                               H, W, K, flags, out_norm, _ptr(idx), _ptr(mask), _ptr(g_images), _ptr(ga), _ptr(ge), _ptr(gd),
                                               None, None, _ptr(gP), _ptr(gF), _ptr(ws), ws.numel(), _stream(dev)),
                "mvr_points_backward_angles")
    if gP is not None:
        gP = gP.reshape(points_shape)
    if gF is not None:
        gF = gF.reshape(rgb_shape)
    return ga, ge, gd, gP, gF


class _PointsRender(torch.autograd.Function):
    @staticmethod
    def forward(ctx, R, T, inv_dist, points, rgb, M, radius, bg_rgb, H, W, K, flags, want_fragments, out_norm=None,
                out_dtype=None):
        cfg, saved, images, extras = _points_forward_launch(R, T, inv_dist, points, rgb, M, radius, bg_rgb, H, W, K, flags,
                                                            want_fragments, out_norm, out_dtype)
        ctx.set_materialize_grads(False)
        ctx.cfg = cfg
        ctx.scale_shape = inv_dist.shape
        ctx.save_for_backward(*saved)
        ctx.mark_non_differentiable(*extras)
        return (images, *extras)

    @staticmethod
    def backward(ctx, g_images, *_unused):
        if g_images is None:
            return (None,) * 15
        gR, gT, gs, gP, gF = _points_backward_launch(ctx.cfg, ctx.saved_tensors, g_images, ctx.needs_input_grad[3],
                                                     ctx.needs_input_grad[4])
        return (gR, gT, gs.reshape(ctx.scale_shape), gP, gF) + (None,) * 10


class _PointsRenderFromAngles(torch.autograd.Function):
    """look_at + point render as ONE autograd node: (azim, elev, dist, points, rgb) -> images (+ R, T, C, flag, idx, mask).
    The clouds are scaled by 1 / dist inside the kernels (MVR_SCALE_IS_DIST), so `dist` reaches the images twice -- through
    the cameras and through the scale -- and its two gradients are summed here instead of by an AccumulateGrad node.
    The point path at MVTN's sizes is launch- and host-bound (DESIGN.md section 4): one Function.apply and one backward
    node less per step is measurable.  after_cameras: as in _MeshRenderFromAngles."""

    @staticmethod
    def forward(ctx, azim, elev, dist, points, rgb, M, radius, bg_rgb, H, W, K, flags, out_norm, out_dtype, after_cameras):
        sink = after_cameras if isinstance(after_cameras, FlagSink) else None
        a, e, d, R, T, Cc, bad = _look_at_launch(azim, elev, dist, sink)
        if after_cameras is not None and sink is None:
            after_cameras(bad)
        cfg, saved, images, extras = _points_forward_launch(R, T, d, points, rgb, M, radius, bg_rgb, H, W, K,
                                                            flags | L.SCALE_IS_DIST, False, out_norm, out_dtype)
        ctx.set_materialize_grads(False)
        ctx.cfg = cfg
        ctx.shapes = (azim.shape, elev.shape, dist.shape)
        ctx.save_for_backward(a, e, *saved)
        ctx.mark_non_differentiable(bad, *extras)
        return (images, R, T, Cc, bad, *extras)

    @staticmethod
    def backward(ctx, g_images, gR_ext, gT_ext, gC_ext, *_unused):
        if g_images is None and gR_ext is None and gT_ext is None and gC_ext is None:
            return (None,) * 15
        a, e = ctx.saved_tensors[:2]
        saved = ctx.saved_tensors[2:]
        d = saved[2]
        if g_images is not None and gR_ext is None and gT_ext is None and gC_ext is None:
            # nothing arrives through the cameras object (the usual case): rasterizer backward, reduction, camera backward and the
            # scale term in ONE call ending in (d azim, d elev, d dist) -- mvr_points_backward_angles
            ga, ge, gd, gP, gF = _points_backward_angles_launch(ctx.cfg, saved, a, e, g_images, ctx.needs_input_grad[3], ctx.needs_input_grad[4])
            sa, se, sd = ctx.shapes
            return (ga.reshape(sa), ge.reshape(se), gd.reshape(sd), gP, gF) + (None,) * 10
        gR = gT = gs = gP = gF = None
        if g_images is not None:
            gR, gT, gs, gP, gF = _points_backward_launch(ctx.cfg, saved, g_images, ctx.needs_input_grad[3], ctx.needs_input_grad[4])
        if gR_ext is not None:
            gR = gR_ext if gR is None else gR + gR_ext
        if gT_ext is not None:
            gT = gT_ext if gT is None else gT + gT_ext
        ga, ge, gd = _look_at_backward_launch(a, e, d, gR, gT, gC_ext)
        if gs is not None:
            gd = gd + gs
        sa, se, sd = ctx.shapes
        return (ga.reshape(sa), ge.reshape(se), gd.reshape(sd), gP, gF) + (None,) * 10


def render_points_from_angles(points, rgb, M: int, azim, elev, dist, radius: float, bg_rgb, image_size, points_per_pixel=1,
                              compositor="norm", normalize=None, out_dtype=None, after_cameras=None):
    """look_at_view_transform + render_points(dist=...) in one autograd node (see _PointsRenderFromAngles).
    Returns images (B*M,3,H,W), (R, T, C, invalid flag), fragments dict."""
    if compositor not in ("norm", "alpha"):
        raise ValueError("compositor must be 'norm' or 'alpha'")
    flags = L.COMPOSITE_ALPHA if compositor == "alpha" else 0
    H, W = _hw(image_size)
    images, R, T, Cc, bad, idx, mask = _PointsRenderFromAngles.apply(
        azim, elev, dist, points, rgb, M, radius, bg_rgb, H, W, int(points_per_pixel), flags, _out_norm(normalize), out_dtype,
        after_cameras)
    return images, (R, T, Cc, bad), _PointFragments(idx, mask, H, W)


def render_points(points, rgb, M: int, R, T, inv_dist, radius: float, bg_rgb, image_size: int, points_per_pixel=1,
                  compositor="norm", fragments=False, normalize=None, out_dtype=None, dist=None):
    """images (B*M,3,H,W) [+ fragments].  compositor: "norm" (NormWeightedCompositor) | "alpha".
    The clouds are scaled by inv_dist (renderer.py:142 scale_(1 / dist)); pass inv_dist=None and dist=(B*M,) or (B, M)
    to have the kernels take the reciprocal themselves (same IEEE division as torch's 1.0 / dist) and return the gradient
    w.r.t. dist directly -- no elementwise launches or autograd nodes around the renderer.
    normalize / out_dtype: as in render_meshes (consumer-side fusion)."""
    if compositor not in ("norm", "alpha"):
        raise ValueError("compositor must be 'norm' or 'alpha'")
    flags = L.COMPOSITE_ALPHA if compositor == "alpha" else 0
    if (inv_dist is None) == (dist is None):
        raise ValueError("pass exactly one of inv_dist and dist")
    if dist is not None:
        inv_dist = dist
        flags |= L.SCALE_IS_DIST
    H, W = _hw(image_size)
    out = _PointsRender.apply(R, T, inv_dist, points, rgb, M, radius, bg_rgb, H, W,
                              int(points_per_pixel), flags, bool(fragments), _out_norm(normalize), out_dtype)
    if fragments:
        frag = {"idx": out[1], "zbuf": out[2], "dists": out[3]}
    else:
        frag = _PointFragments(out[1], out[2], H, W)
    return out[0], frag


class _PointFragments(dict):
    """{"idx": (N,H,W,K) int32} of a render that did not ask for fragments.  The kernels then skip the `-1` stores of the
    background pixels (MVR_IDX_SPARSE: 277 of the 308 MB of idx at C3) -- the backward pass goes by the 1-bit hit mask --
    so the dense tensor the caller may still look at is completed here, on first access, outside the hot path."""

    def __init__(self, idx, mask, H, W):
        super().__init__(idx=None)
        self._raw = (idx, mask, H, W)

    def _dense(self):
        if self._raw is not None:
            idx, mask, H, W = self._raw
            N, mw = idx.shape[0], (W + 31) // 32
            words = mask[: N * H * mw].view(N, H, mw, 1)
            bits = (words >> torch.arange(32, device=idx.device, dtype=torch.int32)) & 1
            hit = bits.view(N, H, mw * 32)[:, :, :W].bool()
            dict.__setitem__(self, "idx", idx.masked_fill(~hit.unsqueeze(-1), -1))
            self._raw = None

    def __getitem__(self, k):
        self._dense()
        return dict.__getitem__(self, k)

    def get(self, k, default=None):
        self._dense()
        return dict.get(self, k, default)

    def items(self):
        self._dense()
        return dict.items(self)

    def values(self):
        self._dense()
        return dict.values(self)
