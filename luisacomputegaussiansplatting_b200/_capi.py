"""ctypes binding of include/lcgs_b200.h (liblcgs_b200.so).

There is no fallback: if the CUDA library cannot be loaded this module raises, and every status
other than LCGS_B200_OK is turned into an exception.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

OK, ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_NO_DEVICE, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
NUM_STAGES = 7
STAGES = ("preprocess", "scan", "depth_sort", "duplicate_keys", "sort", "ranges", "blend")


class LcgsError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__("lcgs_b200 status %d: %s" % (status, msg))
        self.status = status


class CapacityError(LcgsError):
    pass


class Camera(C.Structure):
    """lcgs_b200_camera == lcgs::Camera (reference lcgs/include/lcgs/util/camera.h:15-25)."""

    _fields_ = [("position", C.c_float * 3), ("front", C.c_float * 3), ("up", C.c_float * 3),
                ("right", C.c_float * 3), ("fov", C.c_float), ("aspect_ratio", C.c_float), ("width", C.c_int),
                ("height", C.c_int)]


class ViewParams(C.Structure):
    _fields_ = [("view", C.c_float * 16), ("proj", C.c_float * 16), ("tanfovx", C.c_float), ("tanfovy", C.c_float),
                ("focalx", C.c_float), ("focaly", C.c_float), ("cam_pos", C.c_float * 3), ("width", C.c_int),
                ("height", C.c_int)]


class Scene(C.Structure):
    _fields_ = [("num_gaussians", C.c_int), ("sh_deg", C.c_int), ("pos", C.c_void_p), ("scale", C.c_void_p),
                ("rotq", C.c_void_p), ("sh", C.c_void_p), ("opacity", C.c_void_p), ("scale_modifier", C.c_float),
                ("alpha_consts", C.c_void_p)]


class Frame(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("bg_color", C.c_float * 3), ("means_2d", C.c_void_p),
                ("depth", C.c_void_p), ("conic", C.c_void_p), ("color", C.c_void_p), ("tiles_touched", C.c_void_p),
                ("point_offsets", C.c_void_p), ("point_list_keys_unsorted", C.c_void_p),
                ("point_list_unsorted", C.c_void_p), ("point_list_keys", C.c_void_p), ("point_list", C.c_void_p),
                ("ranges", C.c_void_p), ("list_capacity", C.c_size_t), ("target_img", C.c_void_p),
                ("radii", C.c_void_p), ("tile_row_begin", C.c_int), ("tile_row_end", C.c_int),
                ("target_rgb8", C.c_void_p), ("target_alpha", C.c_void_p), ("target_depth", C.c_void_p),
                ("target_n_contrib", C.c_void_p)]


class Grad(C.Structure):
    """lcgs_b200_grad: dL/dimg (and optionally dL/d of the alpha and depth planes) in, per-Gaussian gradients and the
    camera pose's gradient out (each output optional)."""

    _fields_ = [("dl_dimg", C.c_void_p), ("grad_pos", C.c_void_p), ("grad_scale", C.c_void_p), ("grad_rotq", C.c_void_p),
                ("grad_sh", C.c_void_p), ("grad_opacity", C.c_void_p), ("grad_means_2d", C.c_void_p),
                ("grad_conic", C.c_void_p), ("grad_color", C.c_void_p), ("dl_dalpha", C.c_void_p),
                ("dl_ddepth", C.c_void_p), ("grad_depth", C.c_void_p), ("grad_view", C.c_void_p),
                ("grad_cam_pos", C.c_void_p)]


PEER_HANDLE_BYTES = 64
_VP = C.c_void_p
_I = C.c_int
_F = C.c_float
_SZ = C.c_size_t
_PROTOS = {
    # name: (restype, argtypes)
    "lcgs_b200_version": (_I, []),
    "lcgs_b200_status_string": (C.c_char_p, [_I]),
    "lcgs_b200_ctx_create": (_I, [_I, C.POINTER(_VP)]),
    "lcgs_b200_ctx_destroy": (_I, [_VP]),
    "lcgs_b200_ctx_reserve": (_I, [_VP, _I, _SZ]),
    "lcgs_b200_last_error": (C.c_char_p, [_VP]),
    "lcgs_b200_get_lookat_cam": (_I, [C.POINTER(_F), C.POINTER(_F), C.POINTER(_F), C.POINTER(Camera)]),
    "lcgs_b200_local_to_world_matrix": (_I, [C.POINTER(Camera), C.POINTER(_F)]),
    "lcgs_b200_world_to_local_matrix": (_I, [C.POINTER(Camera), C.POINTER(_F)]),
    "lcgs_b200_projection_matrix": (_I, [_F, _F, _F, _F, C.POINTER(_F)]),
    "lcgs_b200_view_params_from_camera": (_I, [C.POINTER(Camera), C.POINTER(ViewParams)]),
    "lcgs_b200_sh_process": (_I, [_VP, _I, _I, C.POINTER(_F), _VP, _VP, _VP, _VP]),
    "lcgs_b200_project": (_I, [_VP, _I, _VP, _VP, _VP, _F, C.POINTER(ViewParams), _VP, _VP, _VP, _VP]),
    "lcgs_b200_allocate_tiles": (_I, [_VP, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP]),
    "lcgs_b200_fill_u32": (_I, [_VP, _VP, _SZ, C.c_uint32, _VP]),
    "lcgs_b200_fill_u64": (_I, [_VP, _VP, _SZ, C.c_uint64, _VP]),
    "lcgs_b200_fill_f32": (_I, [_VP, _VP, _SZ, _F, _VP]),
    "lcgs_b200_scan_temp_bytes": (_SZ, [_SZ]),
    "lcgs_b200_scan_inclusive_u32": (_I, [_VP, _VP, _VP, _SZ, _VP]),
    "lcgs_b200_duplicate_keys": (_I, [_VP, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _SZ, _I, _I, _VP]),
    "lcgs_b200_sort_temp_bytes": (_SZ, [_SZ]),
    "lcgs_b200_sort_pairs_u64_u32": (_I, [_VP, _VP, _VP, _VP, _VP, _SZ, _I, _I, _VP]),
    "lcgs_b200_tile_ranges": (_I, [_VP, _VP, _SZ, _VP, _I, _VP]),
    "lcgs_b200_blend": (_I, [_VP, _I, _I, _I, C.POINTER(_F), _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, _I, _VP]),
    "lcgs_b200_splat_forward": (_I, [_VP, _I, _VP, C.POINTER(Frame), _VP]),
    "lcgs_b200_render": (_I, [_VP, C.POINTER(Scene), C.POINTER(ViewParams), C.POINTER(Frame), _VP]),
    "lcgs_b200_render_backward": (_I, [_VP, C.POINTER(Scene), C.POINTER(ViewParams), C.POINTER(Frame), C.POINTER(Grad), _VP]),
    "lcgs_b200_ssim": (_I, [_VP, _I, _I, _VP, _VP, _VP, _VP, _VP]),
    "lcgs_b200_num_rendered": (_I, [_VP, _VP, C.POINTER(_I)]),
    "lcgs_b200_read_num_rendered_async": (_I, [_VP, _VP, _VP]),
    "lcgs_b200_read_image": (_I, [_VP, C.POINTER(Frame), _VP, _VP]),
    "lcgs_b200_read_image_rgb8": (_I, [_VP, C.POINTER(Frame), _VP, _VP]),
    "lcgs_b200_scene_prepare": (_I, [_VP, _I, _VP, _VP, _VP]),
    "lcgs_b200_transpose_rgba8": (_I, [_VP, _I, _I, _VP, _VP, _VP]),
    "lcgs_b200_set_profiling": (_I, [_VP, _I]),
    "lcgs_b200_stage_times": (_I, [_VP, C.POINTER(_F)]),
    "lcgs_b200_sort_breakdown": (_I, [_VP, C.POINTER(_F), C.POINTER(_F), C.POINTER(_I)]),
    "lcgs_b200_peer_alloc": (_I, [_VP, _SZ, C.POINTER(_VP), C.c_char_p]),
    "lcgs_b200_peer_open": (_I, [_VP, C.c_char_p, C.POINTER(_VP)]),
    "lcgs_b200_peer_read": (_I, [_VP, _VP, _VP, _SZ]),
    "lcgs_b200_peer_read_async": (_I, [_VP, _VP, _VP, _SZ, _VP]),
    "lcgs_b200_peer_close": (_I, [_VP, _VP]),
    "lcgs_b200_peer_free": (_I, [_VP, _VP]),
    "lcgs_b200_peer_signal": (_I, [_VP, _VP, C.c_uint32, _VP]),
    "lcgs_b200_peer_wait": (_I, [_VP, _VP, C.c_uint32, C.c_uint32, _VP]),
    "lcgs_b200_peer_error": (_I, [_VP, C.POINTER(C.c_uint32)]),
    "lcgs_b200_checksum_u32": (_I, [_VP, _VP, _SZ, _VP, _VP]),
}
EXPORTED_SYMBOLS = tuple(_PROTOS)

_lib = None


def library_path() -> str:
    return _build.LIB


def load() -> C.CDLL:
    """Load (building first if the in-tree .so is missing/stale and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    if os.environ.get("LCGS_TUNING") == "1":  # scripts/tune_*.py only: the -DLCGS_TUNING library, built explicitly
        path = _build.TUNING_LIB
        if not os.path.exists(path):
            raise RuntimeError("LCGS_TUNING=1 but %s is missing: run `python -m luisacomputegaussiansplatting_b200.build --tuning`" % path)
        lib = C.CDLL(path)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib
    path = _build.LIB
    if not os.path.exists(path) or _build.is_stale():
        try:
            _build.build_native()
        except Exception as e:  # no nvcc on this box
            if not os.path.exists(path):
                raise RuntimeError("liblcgs_b200.so is missing and could not be built (%s); the CUDA extension is "
                                   "required, there is no CPU fallback" % e)
    lib = C.CDLL(path)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, ctx=None):
    if status == OK:
        return
    lib = load()
    msg = lib.lcgs_b200_status_string(status).decode()
    if ctx:
        detail = lib.lcgs_b200_last_error(ctx).decode()
        if detail:
            msg += " (" + detail + ")"
    if status == ERR_CAPACITY:
        raise CapacityError(status, msg)
    raise LcgsError(status, msg)


def fvec(v) -> C.Array:
    return (C.c_float * len(v))(*[float(x) for x in v])
