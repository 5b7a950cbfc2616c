"""ctypes binding of oracle/libray_oracle.so (ray-batch entry points of the CPU restatement) and of the reference's
ray tap oracle/_ref/libvolrend_ref_rays.so -- TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import binding as ob

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libray_oracle.so")
REF_LIB_PATH = os.path.join(_HERE, "_ref", "libvolrend_ref_rays.so")

_lib = None
_ref = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        h = C.CDLL(LIB_PATH)
        h.orc_camera_rays.restype = None
        h.orc_camera_rays.argtypes = [C.POINTER(ob.orc_camera), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        h.orc_render_rays.restype = C.c_int
        h.orc_render_rays.argtypes = [C.POINTER(ob.orc_tree), C.POINTER(ob.orc_options), C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_void_p, C.POINTER(ob.orc_counters), C.c_int]
        _lib = h
    return _lib


def camera_rays(cam: ob.orc_camera, tile=None):
    """-> (origins [h*w,3], dirs [h*w,3]) float32, row-major over the tile (directions not normalised)."""
    x0, y0, w, h = tile if tile is not None else (0, 0, cam.width, cam.height)
    o = np.zeros((h * w, 3), np.float32)
    d = np.zeros((h * w, 3), np.float32)
    lib().orc_camera_rays(C.byref(cam), x0, y0, w, h, o.ctypes.data, d.ctypes.data)
    return o, d


def render_rays(tree: ob.OracleTree, opt: ob.orc_options, origins, dirs, t_max=None, nthreads=None):
    """-> (rgba_f32 [n,4], counters dict)"""
    o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
    d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
    t = None if t_max is None else np.ascontiguousarray(t_max, np.float32).reshape(-1)
    n = o.shape[0]
    out = np.zeros((n, 4), np.float32)
    cnt = ob.orc_counters()
    rc = lib().orc_render_rays(C.byref(tree.c), C.byref(opt), o.ctypes.data, d.ctypes.data,
                               t.ctypes.data if t is not None else None, n, out.ctypes.data, C.byref(cnt),
                               int(nthreads or os.cpu_count() or 1))
    if rc != 0:
        raise RuntimeError(f"orc_render_rays failed: {rc}")
    return out, dict(samples=cnt.samples, child_loads=cnt.child_loads, shaded=cnt.shaded, rays_hit=cnt.rays_hit)


def ref_available() -> bool:
    return os.path.exists(REF_LIB_PATH)


def ref_lib():
    global _ref
    if _ref is None:
        from . import ref_binding as rb
        h = C.CDLL(REF_LIB_PATH)
        h.ref_rays_tree_open.restype = C.c_void_p
        h.ref_rays_tree_open.argtypes = [C.c_char_p]
        h.ref_rays_tree_close.restype = None
        h.ref_rays_tree_close.argtypes = [C.c_void_p]
        h.ref_render_rays_f32.restype = C.c_int
        h.ref_render_rays_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                          C.POINTER(rb.ref_options), C.c_void_p]
        _ref = h
    return _ref


def ref_render_rays(npz_path: str, opt, origins, dirs, t_max=None) -> np.ndarray:
    """The reference's trace_ray on loaded rays (oracle/ref_rays.cu), tree read by the reference's own loader."""
    h = ref_lib().ref_rays_tree_open(npz_path.encode())
    if not h:
        raise RuntimeError(f"reference loader could not open {npz_path}")
    try:
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        t = None if t_max is None else np.ascontiguousarray(t_max, np.float32).reshape(-1)
        out = np.zeros((o.shape[0], 4), np.float32)
        rc = ref_lib().ref_render_rays_f32(h, o.ctypes.data, d.ctypes.data, t.ctypes.data if t is not None else None,
                                           o.shape[0], C.byref(opt), out.ctypes.data)
        if rc:
            raise RuntimeError(f"ref_render_rays_f32 failed {rc}")
        return out
    finally:
        ref_lib().ref_rays_tree_close(h)
