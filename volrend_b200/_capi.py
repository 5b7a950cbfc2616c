"""ctypes binding of ``libvolrend_b200.so`` (C-ABI declared in ``include/volrend_b200.h``).

The library is built in-tree by ``make lib`` / ``__graft_entry__.build()``.  There is no
Python or CPU fallback: if the shared object is missing, importing anything that renders
raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# VR_LIB_SUFFIX selects a tuning build (e.g. "_b128m7", see Makefile); default is the product build
LIB_PATH = os.path.join(_HERE, "libvolrend_b200" + os.environ.get("VR_LIB_SUFFIX", "") + ".so")

VR_BASIS_MAX = 25
VR_OK, VR_EINVAL, VR_ENODEVICE, VR_ECUDA, VR_ENOMEM, VR_EUNSUPPORTED = 0, -1, -2, -3, -4, -5
VR_FMT_RGBA, VR_FMT_SH, VR_FMT_SG, VR_FMT_ASG = 0, 1, 2, 3


class vr_tree_desc(C.Structure):
    _fields_ = [("child", C.c_void_p), ("data", C.c_void_p), ("extra", C.c_void_p),
                ("capacity", C.c_int64), ("N", C.c_int32), ("data_dim", C.c_int32),
                ("format", C.c_int32), ("basis_dim", C.c_int32),
                ("offset", C.c_float * 3), ("scale", C.c_float * 3), ("use_ndc", C.c_int32),
                ("ndc_width", C.c_float), ("ndc_height", C.c_float), ("ndc_focal", C.c_float)]


class vr_tree_quant_desc(C.Structure):
    _fields_ = [("base", vr_tree_desc), ("quant_colors", C.c_void_p), ("quant_map", C.c_void_p),
                ("sigma", C.c_void_p), ("data_retained", C.c_void_p), ("n_quant", C.c_int32), ("n_retain", C.c_int32)]


class vr_camera(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("fx", C.c_float), ("fy", C.c_float),
                ("c2w", C.c_float * 12)]


class vr_options(C.Structure):
    _fields_ = [("step_size", C.c_float), ("sigma_thresh", C.c_float), ("stop_thresh", C.c_float),
                ("background_brightness", C.c_float), ("render_bbox", C.c_float * 6),
                ("basis_minmax", C.c_int32 * 2), ("rot_dirs", C.c_float * 3), ("render_depth", C.c_int32)]


class vr_rect(C.Structure):
    _fields_ = [("x0", C.c_int32), ("y0", C.c_int32), ("w", C.c_int32), ("h", C.c_int32)]


class vr_counters(C.Structure):
    _fields_ = [("samples", C.c_ulonglong), ("child_loads", C.c_ulonglong), ("shaded", C.c_ulonglong),
                ("rays_hit", C.c_ulonglong), ("node_fetches", C.c_ulonglong)]


class vr_tree_info(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("max_depth", C.c_int32), ("rec_bytes", C.c_int32),
                ("node_bytes", C.c_int64), ("rec_total_bytes", C.c_int64), ("top_bytes", C.c_int64),
                ("kernel_basis", C.c_int32), ("wide_parity", C.c_int32), ("n_tables", C.c_int64),
                ("wide_bytes", C.c_int64), ("wrecs_bytes", C.c_int64), ("kernel_bytes", C.c_int64),
                ("device_bytes", C.c_int64)]


# name -> (restype, argtypes); every symbol include/volrend_b200.h declares
SYMBOLS = {
    "vr_default_options": (None, [C.POINTER(vr_options)]),
    "vr_tree_create": (C.c_int, [C.POINTER(vr_tree_desc), C.POINTER(C.c_void_p)]),
    "vr_tree_create_quantized": (C.c_int, [C.POINTER(vr_tree_quant_desc), C.POINTER(C.c_void_p)]),
    "vr_tree_destroy": (None, [C.c_void_p]),
    "vr_tree_get_info": (C.c_int, [C.c_void_p, C.POINTER(vr_tree_info)]),
    "vr_render": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.POINTER(vr_options), C.POINTER(vr_rect),
                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vr_render_batch": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.c_int, C.POINTER(vr_options),
                                  C.POINTER(vr_rect), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vr_render_composite": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.POINTER(vr_options),
                                      C.POINTER(vr_rect), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vr_render_surface": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.POINTER(vr_options),
                                    C.c_ulonglong, C.c_ulonglong, C.c_void_p]),
    "vr_render_rays": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(vr_options),
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "vr_camera_rays": (C.c_int, [C.POINTER(vr_camera), C.POINTER(vr_rect), C.c_void_p, C.c_void_p, C.c_void_p]),
    "vr_render_frames_host": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.c_int, C.POINTER(vr_options),
                                        C.c_void_p]),
    "vr_write_png": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int, C.c_int]),
    "vr_render_frames_png": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.c_int, C.POINTER(vr_options),
                                       C.POINTER(C.c_char_p), C.c_int]),
    "vr_probe_lumisphere": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_void_p, C.c_void_p]),
    "vr_render_bands": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.POINTER(vr_options), C.c_int, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "vr_band_rows": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "vr_render_bands_batch": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.c_int, C.POINTER(vr_options), C.c_int, C.c_int,
                                        C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vr_debug_trace": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.POINTER(vr_options), C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "vr_set_variant": (C.c_int, [C.c_int]),
    "vr_get_variant": (C.c_int, []),
    "vr_tree_variant": (C.c_int, [C.c_void_p]),
    "vr_variant_supported": (C.c_int, [C.c_int, C.c_int]),
    "vr_set_max_ctas": (C.c_int, [C.c_int]),
    "vr_dev_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "vr_dev_free": (C.c_int, [C.c_void_p]),
    "vr_ipc_export": (C.c_int, [C.c_void_p, C.c_char_p]),
    "vr_ipc_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "vr_ipc_close": (C.c_int, [C.c_void_p]),
    "vr_copy_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vr_copy2d_async": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p]),
    "vr_mg_create": (C.c_int, [C.POINTER(vr_tree_desc), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "vr_mg_destroy": (None, [C.c_void_p]),
    "vr_mg_device_count": (C.c_int, [C.c_void_p]),
    "vr_mg_device": (C.c_int, [C.c_void_p, C.c_int]),
    "vr_mg_tree": (C.c_void_p, [C.c_void_p, C.c_int]),
    "vr_mg_render": (C.c_int, [C.c_void_p, C.POINTER(vr_camera), C.c_int, C.POINTER(vr_options), C.c_int, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]),
    "vr_mg_frames_dev0": (C.c_void_p, [C.c_void_p]),
    "vr_mg_last_error": (C.c_char_p, [C.c_void_p]),
    "vr_launch_count": (C.c_ulonglong, []),
    "vr_last_error": (C.c_char_p, []),
    "vr_version": (C.c_char_p, []),
}

_lib = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make lib` (or __graft_entry__.build()). "
                "volrend_b200 has no CPU/PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)      # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class VolrendError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"volrend_b200 error {code}: {msg}")
        self.code = code


def check(rc: int) -> None:
    if rc != VR_OK:
        raise VolrendError(rc, lib().vr_last_error().decode("utf-8", "replace"))
