"""ctypes binding of libmvr_b200.so (include/mvr_b200.h).  Fails loudly: there is no CPU fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmvr_b200.so")

ABI_VERSION = 11
PERSPECTIVE_CORRECT = 1
CULL_BACKFACES = 2
COMPOSITE_ALPHA = 4
RGB_PER_ELEMENT = 8
FACES_I64 = 16
IMAGES_BF16 = 32
SCALE_IS_DIST = 64
WS_KEYS_ARMED = 128    # workspace reuse hints of the mesh path (include/mvr_b200.h)
WS_REARM_KEYS = 256
WS_PROJECTED = 512
IDX_SPARSE = 1024
CLIP_BARYCENTRIC = 4096   # [upstream] clip_barycentric_coords
FACES_U16 = 8192         # faces as uint16 (meshes of at most 65536 vertices): collate_meshes narrows when it can
TEST_TINY_QUEUES = 0x40000000   # tests only: shrink the scatter kernel's work queues to force their fallbacks
CNT_STRADDLE, CNT_BIG_FACES, NUM_COUNTERS = 0, 1, 4

_vp, _i, _f, _d, _i64, _sz = C.c_void_p, C.c_int, C.c_float, C.c_double, C.c_int64, C.c_size_t

# name -> (restype, argtypes): exactly the declarations of include/mvr_b200.h
SIGNATURES = {
    "mvr_abi_version": (_i, []),
    "mvr_last_error_string": (C.c_char_p, []),
    "mvr_launch_count": (C.c_longlong, []),
    "mvr_profile_enable": (_i, [C.c_char_p]),
    "mvr_profile_collect": (_i, [C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "mvr_host_set_threads": (_i, [_i]),
    "mvr_host_gather": (_i, [C.POINTER(C.c_void_p), C.POINTER(C.c_int64), _i, _vp, _i, _i]),
    "mvr_host_stage_meshes": (_i, [C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_int64), _i,
                                   _i, _vp, _vp, _vp, _vp, _vp]),
    "mvr_host_stage_meshes_packed": (_i, [C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_int64), _i,
                                          _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvr_host_stage_meshes_begin": (_i, [C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                         _i, _i, _vp, _vp, _vp, _vp, _i, _vp]),
    "mvr_host_stage_meshes_packed_begin": (_i, [C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                                _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "mvr_host_stage_meshes_end": (_i, [_i]),
    "mvr_look_at_forward": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "mvr_look_at_forward_flagged": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvr_look_at_backward": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvr_mesh_geometry_bytes": (_sz, [_i64, _i64]),
    "mvr_images_regularize_forward": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp]),
    "mvr_images_regularize_backward": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp]),
    "mvr_mesh_prepare": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _i64, _i, _vp, _i, _vp, _sz, _vp]),
    "mvr_mesh_get_normals": (_i, [_vp, _i64, _i64, _vp, _vp]),
    "mvr_mesh_normals_backward": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _i, _vp, _vp, _vp]),
    "mvr_mesh_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i64, _i64]),
    "mvr_mesh_forward": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i64, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _f, _f, _f, _f,
                              _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mvr_mesh_soft_blend_forward": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i64, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _f, _f, _f, _f,
                                         _vp, _vp, _vp, _vp, _vp, _vp]),
    "mvr_mesh_soft_backward": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i64, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _f, _f, _f, _f, _i, _i, _i, _i,
                                    _i, _f, _f, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mvr_mesh_backward": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i64, _i, _vp, _vp, _vp, _vp, _i, _vp, _f, _f, _f, _i, _i, _i, _i,
                               _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mvr_mesh_backward_angles": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i64, _i, _vp, _vp, _vp, _vp, _i, _vp, _f, _f, _f, _i, _i, _i, _i,
                                      _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mvr_points_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _d]),
    "mvr_points_hit_mask_words": (_sz, [_i, _i, _i, _i]),
    "mvr_points_forward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _d, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _sz, _vp]),
    "mvr_points_backward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _vp, _vp, _vp, _vp, _sz, _vp]),
    "mvr_points_backward_angles": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp, _vp, _vp,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
}

_lib = None


class MVRError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built: the product path never
    falls back to a CPU or eager-PyTorch implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MVRError(
            f"{LIB_PATH} is missing: build it with `python -m mvtn_b200.build` (or __graft_entry__.build()); "
            "mvtn_b200 has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.mvr_abi_version() != ABI_VERSION:
        raise MVRError(f"libmvr_b200.so ABI {lib.mvr_abi_version()} != expected {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc, who):
    if rc != 0:
        msg = load().mvr_last_error_string()
        raise MVRError(f"{who} failed with status {rc}: {msg.decode() if msg else ''}")
