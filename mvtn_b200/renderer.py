"""MVRenderer -- drop-in for MVTN's models/renderer.py:MVRenderer on B200 (sm_100a).

Same constructor (renderer.py:52), same forward(meshes, points, azim, elev, dist, color=None) ->
(rendered_images (B,M,3,H,W), cameras) (renderer.py:173-198), same render_and_save (renderer.py:200-207),
same train()/eval() behaviour for colour and light randomisation, empty state_dict().  Everything PyTorch3D
did on this path (look_at, Meshes.extend, rasterizers, HardPhong shading, point compositing and their
autograd) is done by libmvr_b200.so through mvtn_b200.ops; nothing here falls back to CPU or eager torch.
"""
import sys

import numpy as np
import torch
from torch import nn

from . import ops
from ._lib import MVRError
from .cameras import FoVOrthographicCameras, FoVPerspectiveCameras
from .structures import unpack_mesh_list
from .util import is_cached_constant, torch_color

_small_cache = {}
_small_cache_by_id = {}


def _device_vec(values, device):
    """Small constant vectors (colours, fixed light) are uploaded once per (device, value) and reused: a
    pageable host->device copy synchronises the stream, and the reference pays one per call."""
    if isinstance(values, tuple):       # constant tuples (fixed light, default colours): hashable, no tensor round trip
        try:
            tkey = ("tuple", device.index, values)
            hit = _small_cache.get(tkey)
            if hit is None:
                if len(_small_cache) > 256:      # a fresh random light per training step lands here: bounded
                    _small_cache.clear()
                hit = torch.as_tensor(values, dtype=torch.float32).to(device)
                _small_cache[tkey] = hit
            return hit
        except TypeError:               # unhashable content (tensors inside): fall through to the generic path
            pass
    # identity fast path: the cached named colours (util.torch_color) and constant tuples come back as the same object
    ident = (id(values), device.index) if isinstance(values, torch.Tensor) and is_cached_constant(values) else None
    if ident is not None:
        hit = _small_cache_by_id.get(ident)
        if hit is not None and hit[0] is values:
            return hit[1]
    t = torch.as_tensor(values, dtype=torch.float32).detach()
    if t.is_cuda:
        return t.to(device)
    key = (str(device), tuple(t.reshape(-1).tolist()), tuple(t.shape))
    hit = _small_cache.get(key)
    if hit is None:
        if len(_small_cache) > 256:
            _small_cache.clear()
        hit = t.to(device)
        _small_cache[key] = hit
    if ident is not None and not values.requires_grad:
        if len(_small_cache_by_id) > 256:
            _small_cache_by_id.clear()
        _small_cache_by_id[ident] = (values, hit)      # keeps `values` alive, so the id cannot be reused
    return hit


_flag_bufs = {}


def _flag_reader(flag_dev):
    """Async D2H of a device int32 flag into a pinned word + an event; the returned callable waits for that event
    only (not for work enqueued afterwards) and returns the flag."""
    key = flag_dev.device.index
    pool = _flag_bufs.setdefault(key, [])
    host = pool.pop() if pool else torch.empty(1, dtype=torch.int32, pin_memory=True)
    host.copy_(flag_dev, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(flag_dev.device))
    state = {}

    def read():
        if "v" not in state:
            ev.synchronize()
            state["v"] = int(host[0])
            pool.append(host)
        return state["v"]

    return read


GRAPH_AUTO_MAX_VIEWS = 48     # cuda_graph=None: point steps up to this many views (B * M) are replayed from CUDA graphs
ORTHOGONAL_THRESHOLD = 1e-6   # renderer.py:29
EXAHSTION_LIMIT = 20          # renderer.py:30 (sic)


class MVRenderer(nn.Module):
    """The multi-view differentiable renderer (see models/renderer.py:33-50 for the argument docs).

    Extra keyword-only options (defaults reproduce the reference):
        compositor: "norm" (NormWeightedCompositor, renderer.py:138) or "alpha" (AlphaCompositor,
            imported at renderer.py:11; BASELINE config 3).
        perspective_correct: barycentric perspective correction (PyTorch3D >= 0.5 infers True for
            FoV perspective cameras).
        copy_stream: H2D of a collated host batch on a side stream (overlaps with the previous step's kernels when the
            loop does not synchronise every step; see ops.PackedMeshes.from_host_packed)
        stage_overlap (default True): a python list of host meshes (the reference's input, renderer.py:67-68) is gathered into pinned
            memory -- faces narrowed to uint16 ids when every mesh has at most 65536 vertices -- and copied by the library's staging
            thread and its private helper pool (mvr_host_stage_meshes_packed_begin) WHILE this thread builds the cameras and launches
            the camera kernel; joined right in front of mvr_mesh_prepare.  False: the same gather on the calling thread (OpenMP team).
            Per end-to-end step at 32 x 12 views: 1.37 -> 1.29 ms with OMP_WAIT_POLICY=passive (what bench.py runs under: the
            calling thread's OpenMP team would have to be woken for every batch), 1.27 vs 1.28 with the policy unset (the team is still
            spinning from the previous batch: no gain, no loss); with OMP_WAIT_POLICY=active every core is taken by a spinning OpenMP
            worker and the staging threads queue behind them (1.26 ... 1.45 ms vs 1.29) -- pass False there.
        cuda_graph (mesh path): only when True, and only for collated host batches (collate_meshes) rendered with the hard Phong
            shader: the device part of the forward and of the backward -- mvr_mesh_prepare, look_at, rasterizer, shader -- is captured
            once per batch SHAPE (the per-mesh vertex / face counts, views-require-grad) and replayed; a batch of another shape is
            captured too (the four most recent shapes are kept), so this is for loops over equal-sized batches -- small per-GPU
            batches of a strong-scaling run, evaluation over a fixed set -- where the step is launch- and host-bound (end to end from a
            collated batch: 0.57 -> 0.43 ms at 1 mesh x 12 views, 0.53 -> 0.46 at 4, even at 8, SLOWER from 16 on -- the copy of the
            images out of the captured buffer costs more than the launches saved; profiles/r3z_mesh_graph_mode.txt); ragged
            training batches should leave it off.  Same static-buffer rules as the point path below.
        cuda_graph: None (default) = automatic -- point steps of at most GRAPH_AUTO_MAX_VIEWS views (BASELINE configs[0]: one
            cloud x 12 views, a step that is pure launch latency) are replayed from CUDA graphs, larger ones run eagerly;
            True / False force it.  Point path only -- the device part of a step (look_at, binning, tile rasterizer + compositor, and their
            backward) is captured once per (B, N, views-require-grad) and replayed with ONE launch per direction: the
            point path at small batches is launch-bound (BASELINE configs[0], one cloud x 12 views: 0.470 -> 0.356 ms per
            end-to-end step, r2m); at 32 clouds the eager step is already GPU-bound and the copies into the captured buffers
            make this mode slower (0.516 -> 0.590 ms): leave it off there.  Needs one object colour and fixed shapes; anything else (per-point colours, invalid rotations, torch.no_grad()) takes the eager
            path.  In this mode `cameras` holds detached copies, `last_fragments` views the captured buffers (valid until the next
            replay) and the images are a copy of the
            captured buffer; the tensors the captured backward reads are static, so at most ONE forward may be outstanding
            per backward (two forwards of the same shapes before a backward would overwrite the first one's saved state).
        cache_geometry: keep the packed device geometry of the last mesh batch and reuse it when the
            same list object is rendered again (SURVEY 8f N1).
        shader / blur_radius / blend_sigma / blend_gamma / keep_alpha: mesh path -- "soft_phong" (SoftPhongShader) or
            "soft_silhouette" (SoftSilhouetteShader) blend the faces_per_pixel fragments of the blurred rasterizer (the
            shaders renderer.py:4-6 imports; SURVEY 8f N3); images keep 3 channels as renderer.py:112 unless keep_alpha.
            Gradients reach the cameras and, when the meshes' vertex tensors require grad, the vertices (through colours,
            depths and edge distances; tolerance-level: accumulated with float atomics), as with the hard shader.
        normalize: None or (mean, std) (3-vectors or scalars): the kernels write (image - mean) / std, the
            normalisation viewGCN/tools/Trainer_mvt.py:41-49 applies before the CNN (SURVEY 8f N2).
        out_dtype: torch.float32 (default) or torch.bfloat16 -- the dtype the images are written in (a bf16 backbone
            then reads them without a conversion pass); gradients flow through either.
    """

    def __init__(self, nb_views, image_size=224, pc_rendering=True, object_color="white", background_color="white",
                 faces_per_pixel=1, points_radius=0.006, points_per_pixel=1, light_direction="random",
                 cull_backfaces=False, *, compositor="norm", perspective_correct=True, cache_geometry=False,
                 normalize=None, out_dtype=None, copy_stream=False, cuda_graph=None, shader="hard_phong", blur_radius=0.0,
                 blend_sigma=1e-4, blend_gamma=1e-4, keep_alpha=False, stage_overlap=True):
        super().__init__()
        self.stage_overlap = bool(stage_overlap)
        self.shader, self.blur_radius, self.blend_sigma, self.blend_gamma, self.keep_alpha = shader, blur_radius, blend_sigma, blend_gamma, keep_alpha
        self.copy_stream = copy_stream
        self.cuda_graph = cuda_graph      # None = auto: replay small (launch-bound) point steps from CUDA graphs
        self._point_graphs = {}
        self._mesh_graphs = {}
        self.nb_views = nb_views
        self.image_size = image_size
        self.pc_rendering = pc_rendering
        self.object_color = object_color
        self.background_color = background_color
        self.faces_per_pixel = faces_per_pixel
        self.points_radius = points_radius
        self.points_per_pixel = points_per_pixel
        self.light_direction_type = light_direction
        self.cull_backfaces = cull_backfaces
        self.compositor = compositor
        self.perspective_correct = perspective_correct
        self.cache_geometry = cache_geometry
        self.normalize = normalize
        self.out_dtype = out_dtype
        self._geom_cache = (None, None)
        self.last_fragments = None

    # ---------------------------------------------------------------------------------------------
    def _device(self, azim):
        if isinstance(azim, torch.Tensor) and azim.is_cuda:
            return azim.device
        if not torch.cuda.is_available():
            raise MVRError("MVRenderer needs a CUDA device: mvtn_b200 has no CPU path")
        return torch.device("cuda", torch.cuda.current_device())

    def _views(self, azim, elev, dist, device):
        azim, elev, dist = (t.to(device) if t.device != device else t for t in (azim, elev, dist))
        if azim.shape != elev.shape or azim.shape != dist.shape or azim.dim() != 2:
            raise ValueError("azim, elev and dist must all be (B, M)")
        if azim.shape[1] != self.nb_views:
            raise ValueError(f"expected {self.nb_views} views, got {azim.shape[1]}")
        return azim, elev, dist

    def _cameras(self, azim, elev, dist, device):
        """look_at_view_transform + check_and_correct_rotation_matrix (renderer.py:79-82, ops.py:156-165).
        The validity test is fused into the look_at kernel; its flag is read AFTER the render has been
        enqueued (see forward), so the reference's host sync does not stall the pipeline."""
        azim, elev, dist = self._views(azim, elev, dist, device)
        R, T, C, bad = ops._LookAt.apply(azim, elev, dist)      # flattens (B, M) -> B*M itself, flat order b*M + m
        return azim, elev, dist, R, T, C, bad

    def _render_with_guard(self, azim, elev, dist, device, render, known_invalid=False):
        """The validity flag travels to pinned host memory right behind the look_at kernel and is awaited through an
        event recorded BEFORE the render is enqueued: the host check of util.py:403-420 (which the reference pays as a
        full device sync on every call) waits only for the camera kernel, never for the rasterizer.
        known_invalid: the caller's fast path has already seen the flag raised for these angles -- go straight to the
        redraw loop instead of rasterizing the rejected cameras once more.  `render` receives the camera centres of the
        ORIGINAL angles as its last argument: the reference evaluates the "relative" light once, before any redraw
        (renderer.py:168,190)."""
        azim, elev, dist, R, T, C, bad = self._cameras(azim, elev, dist, device)
        C_light = C.detach()
        render_ = render
        render = lambda R_, T_, C_, d_: render_(R_, T_, C_, d_, C_light)
        if known_invalid:
            invalid = lambda: 1
            out = None
        else:
            invalid = _flag_reader(bad)
            out = render(R, T, C, dist)
        exhastion = 0
        while invalid() != 0:
            exhastion += 1
            e2 = elev + 90.0 * torch.rand_like(elev)
            a2 = azim + 180.0 * torch.rand_like(azim)
            _, _, _, R, T, C, bad = self._cameras(a2, e2, dist, device)
            invalid = _flag_reader(bad)
            if invalid() != 0 and exhastion > EXAHSTION_LIMIT:
                sys.exit("Remedy did not work")   # ops.py:163-164
            if invalid() == 0:
                out = render(R, T, C, dist)
        return out, R, T, C

    def render_meshes(self, meshes, color, azim, elev, dist, lights, background_color=(1.0, 1.0, 1.0)):
        device = self._device(azim)
        # deferred: the meshes are staged (gather + H2D + mvr_mesh_prepare) inside render(), AFTER the camera kernel and
        # the constants below have been enqueued, so that the rasterizer launch follows the geometry with as little host
        # work in between as possible (the GPU would idle through it)
        if (self.cuda_graph is True and isinstance(meshes, ops.HostPackedMeshes) and self.shader == "hard_phong" and torch.is_grad_enabled()
                and meshes.vert_rgb is None and torch.as_tensor(color).numel() == 3 and len(meshes) == azim.shape[0] and len(meshes) > 0
                and not torch.cuda.is_current_stream_capturing()):
            out = self._render_meshes_graphed(meshes, color, azim, elev, dist, lights, background_color, device)
            if out is not None:
                return out
        geom = self._packed(meshes, color, device)
        if geom.B != azim.shape[0]:
            raise ValueError(f"{geom.B} meshes but azim has batch {azim.shape[0]}")
        bg = _device_vec(background_color, device)
        obj = None if geom.per_vertex_rgb else _device_vec(color, device)
        fixed_light = None if lights is None else _device_vec(lights, device)

        soft = self.shader != "hard_phong"

        def render(R, T, C, dist_, C_light):
            geom.finish()
            light = C_light if fixed_light is None else fixed_light
            if soft:
                return ops.render_meshes(geom, self.nb_views, R, T, C, light, obj, bg, self.image_size,
                                         faces_per_pixel=self.faces_per_pixel, cull_backfaces=self.cull_backfaces,
                                         perspective_correct=self.perspective_correct, verts=getattr(geom, "grad_verts", None),
                                         shader=self.shader, blur_radius=self.blur_radius, sigma=self.blend_sigma,
                                         gamma=self.blend_gamma)
            return ops.render_meshes(geom, self.nb_views, R, T, C, light, obj, bg, self.image_size,
                                     faces_per_pixel=self.faces_per_pixel, cull_backfaces=self.cull_backfaces,
                                     perspective_correct=self.perspective_correct, verts=getattr(geom, "grad_verts", None),
                                     normalize=self.normalize, out_dtype=self.out_dtype)

        try:
            out = None
            flag = None
            if getattr(geom, "grad_verts", None) is None and not soft:
                # fast path: cameras + rasterizer as ONE autograd node (ops.render_meshes_from_angles); the validity flag
                # is still awaited through an event recorded between the camera kernel and the rasterizer
                az, el, di = self._views(azim, elev, dist, device)
                # (the node finishes the geometry itself, after it has launched the camera kernel: a list of host meshes being
                # gathered on the library's worker thread -- stage_overlap -- is joined as late as possible)
                # the rotation flag travels to a pinned word behind the camera kernel: copy and event are issued by the library
                # call itself (ops.FlagSink), so nothing of it stands between the camera launch and the rasterizer launch
                flag = ops.FlagSink.get(device)
                images, (R, T, C, _bad), frag = ops.render_meshes_from_angles(
                    geom, self.nb_views, az, el, di, fixed_light, obj, bg, self.image_size,
                    faces_per_pixel=self.faces_per_pixel, cull_backfaces=self.cull_backfaces,
                    perspective_correct=self.perspective_correct, normalize=self.normalize, out_dtype=self.out_dtype,
                    after_cameras=flag)
                if flag.read() == 0:
                    out = (images, frag)
            if out is None:      # vertex gradients wanted, or invalid rotations: the general path with the redraw loop
                out, R, T, C = self._render_with_guard(azim, elev, dist, device, render, known_invalid=flag is not None)
            images, frag = out
        finally:
            geom.finish()      # never leave a deferred / in-flight staging behind (e.g. when the cameras were rejected)
        self.last_fragments = frag
        B = geom.B
        H, W = ops._hw(self.image_size)
        if soft:      # RGBA from the soft shaders; renderer.py:112 keeps [..., 0:3]
            rendered_images = images.view(B, self.nb_views, 4, H, W)
            if not self.keep_alpha:
                rendered_images = rendered_images[:, :, :3]
        else:
            rendered_images = images.view(B, self.nb_views, 3, H, W)
        return rendered_images, FoVPerspectiveCameras(R, T, C)

    def render_points(self, points, color, azim, elev, dist, background_color=(0.0, 0.0, 0.0)):
        device = self._device(azim)
        if points.shape[0] != azim.shape[0]:
            raise ValueError(f"{points.shape[0]} clouds but azim has batch {azim.shape[0]}")
        bg = _device_vec(background_color, device)
        rgb = torch.as_tensor(color, dtype=torch.float32)
        use_graph = self.cuda_graph
        if use_graph is None:      # auto: only where the step is launch-bound (DESIGN.md section 5)
            use_graph = (points.shape[0] * self.nb_views <= GRAPH_AUTO_MAX_VIEWS and not torch.cuda.is_current_stream_capturing())
        if use_graph and rgb.numel() == 3 and torch.is_grad_enabled():      # under no_grad the eager path runs
            az, el, di = self._views(azim, elev, dist, device)
            out = self._render_points_graphed(points, _device_vec(rgb, device), az, el, di, bg, device)
            if out is not None:
                return out
        pts = points.to(device=device, dtype=torch.float32, non_blocking=True)
        if rgb.numel() == 3:
            rgb = _device_vec(rgb, device)
        else:
            rgb = rgb.to(device) * torch.ones_like(pts)          # renderer.py:119-120 features = color * ones_like(points)

        def render(R, T, C, dist_, _C_light=None):
            # renderer.py:142 point_cloud.scale_(1/dist): the reciprocal is taken inside the kernels (dist=)
            return ops.render_points(pts, rgb, self.nb_views, R, T, None, self.points_radius, bg, self.image_size,
                                     points_per_pixel=self.points_per_pixel, compositor=self.compositor,
                                     normalize=self.normalize, out_dtype=self.out_dtype, dist=dist_)

        az, el, di = self._views(azim, elev, dist, device)
        # fast path: cameras + rasterizer + compositor as ONE autograd node (ops.render_points_from_angles); the validity
        # flag is awaited through an event recorded between the camera kernel and the rasterizer
        # the rotation flag travels to a pinned word behind the camera kernel, copy and event issued by the library call (ops.FlagSink):
        # the point step is bound by the HOST from end to end (~0.25 ms of python against ~0.23 ms of kernels at 32 x 12 views)
        flag = ops.FlagSink.get(device)
        images, (R, T, C, _bad), frag = ops.render_points_from_angles(
            pts, rgb, self.nb_views, az, el, di, self.points_radius, bg, self.image_size,
            points_per_pixel=self.points_per_pixel, compositor=self.compositor, normalize=self.normalize,
            out_dtype=self.out_dtype, after_cameras=flag)
        if flag.read() != 0:      # invalid rotations: the general path with the redraw loop
            (images, frag), R, T, C = self._render_with_guard(azim, elev, dist, device, render, known_invalid=True)
        self.last_fragments = frag
        rendered_images = images.view(pts.shape[0], self.nb_views, 3, self.image_size, self.image_size)
        return rendered_images, FoVOrthographicCameras(R, T, C, znear=0.01)

    def _render_meshes_graphed(self, hp, color, azim, elev, dist, lights, background_color, device):
        """CUDA-graph replay of the mesh step for a collated host batch whose shape has been seen before (see `cuda_graph` in the
        class docstring): vertices and faces are copied straight into the captured geometry buffers.  Returns None when the
        eager path must take over (invalid rotations, a replay still outstanding, a capture that failed)."""
        from . import graphs
        az, el, di = self._views(azim, elev, dist, device)
        grads = (az.requires_grad, el.requires_grad, di.requires_grad)
        key = (tuple(hp.num_verts), tuple(hp.num_faces), hp.faces.dtype, device.index, grads, lights is None)
        st = self._mesh_graphs.get(key)
        if st is not None and (st["busy"] or st.get("failed")):
            return None
        bg = _device_vec(background_color, device)
        obj = _device_vec(color, device)
        light = None if lights is None else _device_vec(lights, device)
        if st is None:
            import gc
            gc.collect()
            torch.cuda.synchronize(device)
            geom = ops.PackedMeshes.from_host_packed(hp, device)
            static_obj, static_bg = obj.clone(), bg.clone()
            static_light = None if light is None else light.clone().reshape(1, 3)
            sample = tuple(t.detach().clone().requires_grad_(g) for t, g in zip((az, el, di), grads))
            try:
                step = graphs.graphed_mesh_render(geom, self.nb_views, static_light, static_obj, static_bg, self.image_size, sample,
                                                  refresh_geometry=True, return_cameras=True, faces_per_pixel=self.faces_per_pixel,
                                                  cull_backfaces=self.cull_backfaces, perspective_correct=self.perspective_correct,
                                                  normalize=self.normalize, out_dtype=self.out_dtype)
            except RuntimeError as e:         # a capture invalidated from outside (another thread's CUDA call): stay eager
                import warnings
                warnings.warn(f"MVRenderer: CUDA-graph capture of the mesh step failed ({e}); this shape runs eagerly")
                self._mesh_graphs[key] = {"failed": True, "busy": False}
                return None
            if len(self._mesh_graphs) >= 4:   # a loop over ragged batches must not hoard captured buffers
                self._mesh_graphs.pop(next(iter(self._mesh_graphs)))
            st = self._mesh_graphs[key] = {"geom": geom, "obj": static_obj, "bg": static_bg, "light": static_light, "step": step,
                                           "obj_src": obj, "bg_src": bg, "light_src": light, "busy": False}
        else:
            geom = st["geom"]
            geom.verts.copy_(hp.verts, non_blocking=True)
            geom.faces.copy_(hp.faces, non_blocking=True)
            if st["obj_src"] is not obj:
                st["obj"].copy_(obj); st["obj_src"] = obj
            if st["bg_src"] is not bg:
                st["bg"].copy_(bg); st["bg_src"] = bg
            if light is not None and st["light_src"] is not light:      # (a fresh random light every training step lands here)
                st["light"].copy_(light.reshape(1, 3)); st["light_src"] = light
        images, cams, bad, p2f = st["step"](az, el, di)
        invalid = _flag_reader(bad)
        n = az.numel()
        cams = cams.detach().clone()
        if invalid() != 0:
            return None
        self.last_fragments = {"pix_to_face": p2f}      # (a view of the captured buffer: valid until the next replay of this shape)
        R, T, C = cams[: 9 * n].view(n, 3, 3), cams[9 * n: 12 * n].view(n, 3), cams[12 * n:].view(n, 3)
        out = images.clone()                             # the caller's images survive the next replay (see _render_points_graphed)
        if out.requires_grad:
            import weakref
            st["busy"] = True

            def release(*_a, _st=st):
                _st["busy"] = False

            out.register_hook(lambda g, _r=release: (_r(), g)[1])
            weakref.finalize(out, release)
        H, W = ops._hw(self.image_size)
        return out.view(len(hp), self.nb_views, 3, H, W), FoVPerspectiveCameras(R, T, C)

    def _render_points_graphed(self, points, rgb, az, el, di, bg, device):
        """CUDA-graph replay of the point step (see `cuda_graph` in the class docstring): `points` (host or device) is
        copied straight into the captured buffer.  Returns None when the eager path must take over (invalid rotations)."""
        from . import graphs
        grads = (az.requires_grad, el.requires_grad, di.requires_grad)
        key = (tuple(points.shape), device.index, grads, torch.is_grad_enabled())
        st = self._point_graphs.get(key)
        if st is not None and st["busy"]:
            # the previous replay's result is still alive and has not been back-propagated: its saved tensors live in the
            # captured buffers, which a second replay would overwrite -- this call takes the eager path instead
            return None
        if st is not None and st.get("failed"):
            return None
        if st is None:
            import gc
            gc.collect()                      # pending frees of other threads (autograd workers) must not land inside the capture
            torch.cuda.synchronize(device)
            static_pts = points.to(device=device, dtype=torch.float32).clone()
            static_rgb, static_bg = rgb.clone(), bg.clone()
            sample = tuple(t.detach().clone().requires_grad_(g) for t, g in zip((az, el, di), grads))
            try:
                step = graphs.graphed_points_render(static_pts, static_rgb, self.nb_views, self.points_radius, static_bg,
                                                    self.image_size, sample, points_per_pixel=self.points_per_pixel,
                                                    compositor=self.compositor, normalize=self.normalize,
                                                    out_dtype=self.out_dtype, return_cameras=True)
            except RuntimeError as e:         # a capture invalidated from outside (another thread's CUDA call): stay eager
                if self.cuda_graph:           # explicitly requested: say so
                    import warnings
                    warnings.warn(f"MVRenderer: CUDA-graph capture failed ({e}); this shape runs eagerly")
                self._point_graphs[key] = {"failed": True, "busy": False}
                return None
            st = self._point_graphs[key] = {"pts": static_pts, "rgb": static_rgb, "bg": static_bg, "step": step,
                                            "rgb_src": rgb, "bg_src": bg, "busy": False}
        else:
            st["pts"].copy_(points, non_blocking=True)
            if st["rgb_src"] is not rgb:          # named colours are cached constants: nothing to copy in the steady state
                st["rgb"].copy_(rgb); st["rgb_src"] = rgb
            if st["bg_src"] is not bg:
                st["bg"].copy_(bg); st["bg_src"] = bg
        images, cams, bad, idx, mask = st["step"](az, el, di)
        invalid = _flag_reader(bad)
        n = az.numel()
        cams = cams.detach().clone()              # the captured buffer is overwritten by the next replay
        if invalid() != 0:
            return None
        # (views of the captured buffers: valid until the next replay of this shape; completed lazily on first access)
        self.last_fragments = ops._PointFragments(idx, mask, *ops._hw(self.image_size))
        R, T, C = cams[: 9 * n].view(n, 3, 3), cams[9 * n: 12 * n].view(n, 3), cams[12 * n:].view(n, 3)
        # a copy, not a view of the captured output buffer: images kept by the caller (logging, two renders per loss)
        # survive the next replay.  What the captured BACKWARD reads (idx, hit mask, cameras) stays static, hence the
        # `busy` guard below: a forward issued while the previous result is alive and un-backpropagated runs eagerly.
        out = images.clone()
        if out.requires_grad:
            # one outstanding forward per captured backward: released when the gradient reaches the images (backward has
            # started; python is single-threaded, so it is enqueued before the next forward) or when the result dies
            import weakref
            st["busy"] = True

            def release(*_a, _st=st):
                _st["busy"] = False

            out.register_hook(lambda g, _r=release: (_r(), g)[1])
            weakref.finalize(out, release)
        rendered_images = out.view(points.shape[0], self.nb_views, 3, self.image_size, self.image_size)
        return rendered_images, FoVOrthographicCameras(R, T, C, znear=0.01)

    def _packed(self, meshes, color, device):
        if isinstance(meshes, ops.PackedMeshes):
            return meshes
        if isinstance(meshes, ops.HostPackedMeshes):     # collated by the data loader: two H2D copies, no gather
            color_t = torch.as_tensor(color, dtype=torch.float32)
            vert_rgb = None
            if color_t.numel() != 3:
                color_t = color_t.reshape(len(meshes), -1, 3)
                vert_rgb = torch.cat([color_t[b, :n] for b, n in enumerate(meshes.num_verts)], 0)
            return ops.PackedMeshes.from_host_packed(meshes, device, vert_rgb=vert_rgb, copy_stream=self.copy_stream)
        if meshes is None:
            raise ValueError("mesh rendering (pc_rendering=False) needs `meshes`")
        if self.cache_geometry and self._geom_cache[0] is meshes:
            return self._geom_cache[1]
        verts, faces = unpack_mesh_list(meshes)
        vert_rgb = None
        color_t = torch.as_tensor(color, dtype=torch.float32)
        if color_t.numel() != 3:
            # renderer.py:76-77 verts_rgb = color * ones((B, maxV, 3)): per-vertex colours (B, maxV, 3)
            color_t = color_t.reshape(len(verts), -1, 3)
            vert_rgb = torch.cat([color_t[b, : verts[b].shape[0]] for b in range(len(verts))], 0)
        # (a capturing stream must only see calls from the capturing thread: no worker-thread copies then)
        geom = ops.PackedMeshes.begin(verts, faces, device, vert_rgb=vert_rgb,
                                      overlap=self.stage_overlap and not torch.cuda.is_current_stream_capturing())
        if any(v.requires_grad for v in verts):      # vertex gradients: keep the autograd history of the packing
            geom.grad_verts = torch.cat([v.to(device=device, dtype=torch.float32) for v in verts], 0)
        if self.cache_geometry:
            self._geom_cache = (meshes, geom)
        return geom

    # ---------------------------------------------------------------------------------------------
    def rendering_color(self, custom_color=(1.0, 0, 0)):
        """renderer.py:153-160."""
        if self.object_color == "custom":
            color = custom_color
        elif self.object_color == "random" and not self.training:
            color = torch_color("white")
        else:
            color = torch_color(self.object_color, max_lightness=True)
        return color

    def light_direction(self, azim, elev, dist):
        """renderer.py:162-171.  Returns a (1,3) direction, or None for the "relative" light, in which case
        the (detached) camera centres computed by the look_at kernel are used (Variable(...) detaches)."""
        if self.light_direction_type == "fixed":
            return ((0, 1.0, 0),)
        elif self.light_direction_type == "random" and self.training:
            return (tuple(1.0 - 2 * np.random.rand(3)),)
        return None

    def forward(self, meshes, points, azim, elev, dist, color=None):
        """renderer.py:173-198: render meshes (pc_rendering False) or point clouds (True) from B x M views."""
        background_color = torch_color(self.background_color, max_lightness=True)
        color = self.rendering_color(color)
        if not self.pc_rendering:
            lights = self.light_direction(azim, elev, dist)
            rendered_images, cameras = self.render_meshes(meshes=meshes, color=color, azim=azim, elev=elev, dist=dist,
                                                          lights=lights, background_color=background_color)
        else:
            if points is None:
                raise ValueError("point rendering (pc_rendering=True) needs `points`")
            rendered_images, cameras = self.render_points(points=points, color=color, azim=azim, elev=elev, dist=dist,
                                                          background_color=background_color)
        return rendered_images, cameras

    def render_and_save(self, meshes, points, azim, elev, dist, images_path, cameras_path, color=None):
        """renderer.py:200-207."""
        from .viz import save_cameras, save_grid
        with torch.no_grad():
            rendered_images, cameras = self.forward(meshes, points, azim, elev, dist, color)
        save_grid(image_batch=rendered_images[0, ...], save_path=images_path, nrow=self.nb_views)
        save_cameras(cameras, save_path=cameras_path, scale=0.22, dpi=200)
