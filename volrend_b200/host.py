"""Host-side mirror of volrend's renderer surface, over the C-ABI.

Same names, argument meaning and error behaviour as the reference classes so tests read
like reference usage (paths relative to /root/reference):

* :class:`DataFormat`      ``include/volrend/data_format.hpp``, ``src/n3tree.cpp:55-101``
* :class:`N3Tree`          ``include/volrend/n3tree.hpp``, loader ``src/n3tree.cpp:111-362``;
  ``load_cuda``/``free_cuda`` (``src/cuda/n3tree.cu``) go through ``vr_tree_create``
* :class:`Camera`          ``include/volrend/camera.hpp``, ``src/camera.cpp:26-76``
* :class:`RenderOptions`   ``include/volrend/render_options.hpp:11-53``
* :func:`launch_renderer`  ``include/volrend/cuda/renderer_kernel.hpp:9-12``
* :class:`VolumeRenderer`  ``include/volrend/renderer.hpp:11-42`` with the GL-free offscreen
  Impl that replaces ``src/cuda_renderer.cpp``

PyTorch is used only to own device memory and streams.  The compiled C++ shim
(``volrend_b200/csrc/shim``) offers the same surface to the unchanged reference C++ callers.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

from . import _capi
from ._capi import check, lib

VOLREND_GLOBAL_BASIS_MAX = 25
CAMERA_DEFAULT_FOCAL_LENGTH = 1111.11


# ---------------------------------------------------------------------------- DataFormat
class DataFormat:
    RGBA, SH, SG, ASG = 0, 1, 2, 3
    _NAMES = {0: "RGBA", 1: "SH", 2: "SG", 3: "ASG"}

    def __init__(self, format: int = 0, basis_dim: int = -1):
        self.format = format
        self.basis_dim = basis_dim

    def parse(self, s: str) -> None:
        """'SH16', 'SG25', 'RGBA' ... (src/n3tree.cpp:55-78)."""
        idx = next((i for i, ch in enumerate(s) if not ch.isalpha()), -1)
        if idx >= 0:
            digits = ""
            for ch in s[idx:]:
                if ch.isdigit() or (not digits and ch in "+-"):
                    digits += ch
                else:
                    break
            try:
                self.basis_dim = int(digits)
            except ValueError:
                self.basis_dim = 0          # atoi semantics
            self.format = {"ASG": self.ASG, "SG": self.SG, "SH": self.SH}.get(s[:idx], self.RGBA)
        else:
            self.basis_dim = -1
            self.format = self.RGBA

    def to_string(self) -> str:
        out = self._NAMES.get(self.format, "UNKNOWN")
        if self.basis_dim != -1:
            out += str(self.basis_dim)
        return out


# ---------------------------------------------------------------------------- N3Tree
class N3Tree:
    """Read-only N3Tree: npz loader + device upload (re-layout happens in ``load_cuda``)."""

    def __init__(self, path: str | None = None, gpu_decode: bool = True):
        # gpu_decode: quantised files (quant_colors/quant_map/...) are decoded by the GPU at upload
        # (vr_tree_create_quantized) instead of the reference's CPU loop; ``data_`` then decodes
        # lazily on first access.
        self.gpu_decode = gpu_decode
        self.quant_ = None      # compressed arrays of a quantised file
        self.N = 0
        self.data_dim = 0
        self.data_format = DataFormat()
        self.capacity = 0
        self.scale = np.ones(3, np.float32)
        self.offset = np.zeros(3, np.float32)
        self.use_ndc = False
        self.ndc_width = self.ndc_height = self.ndc_focal = 0.0
        self._data = None       # fp16 [cap,N,N,N,data_dim]  (see the data_ property)
        self.child_ = None      # int32 [cap,N,N,N]
        self.extra_ = None      # f32
        self._handle = None     # vr_tree*
        self._data_loaded = False
        self._cuda_loaded = False
        if path is not None:
            self.open(path)

    @property
    def data_(self):
        """N3Tree::data_ (fp16 [capacity,N,N,N,data_dim]); decoded on demand for quantised files."""
        if self._data is None and self.quant_ is not None:
            self._data = self._decode_quantised()
        return self._data

    @data_.setter
    def data_(self, v):
        self._data = v

    # -- reference surface
    def is_data_loaded(self) -> bool:
        return self._data_loaded

    def is_cuda_loaded(self) -> bool:
        return self._cuda_loaded

    def clear_cpu_memory(self) -> None:
        self._data = None       # n3tree.cpp:441-447 keeps child_

    def open(self, path: str) -> None:
        """src/n3tree.cpp:111-154.  A missing file leaves the tree unloaded, like the reference."""
        self.free_cuda()
        self._data_loaded = False
        assert path.endswith(".npz")
        if not os.path.exists(path):
            print(f"Can't load because file does not exist: {path}")
            return
        with np.load(path) as npz:
            self.load_npz({k: npz[k] for k in npz.files})
        pb = path[:-4] + "_poses_bounds.npy"
        self.use_ndc = os.path.exists(pb)
        if self.use_ndc:
            self._unpack_llff_poses_bounds(np.load(pb))
        self.load_cuda()
        self._data_loaded = True

    def open_arrays(self, *, child, data, offset, invradius3, data_dim, data_format, extra=None) -> None:
        """In-memory equivalent of ``open_mem`` for already-decoded arrays."""
        self.free_cuda()
        npz = dict(child=child, data=data, offset=offset, invradius3=invradius3,
                   data_dim=np.int64(data_dim), data_format=np.array(data_format))
        if extra is not None:
            npz["extra_data"] = extra
        self.load_npz(npz)
        self.use_ndc = False
        self.load_cuda()
        self._data_loaded = True

    @classmethod
    def from_synth(cls, t) -> "N3Tree":
        tree = cls()
        tree.open_arrays(child=t.child, data=t.data, offset=t.offset, invradius3=t.invradius3,
                         data_dim=t.data_dim, data_format=t.data_format, extra=t.extra)
        return tree

    def load_npz(self, npz: dict) -> None:
        """src/n3tree.cpp:228-362 including the quantised-colour decode (:279-340)."""
        self.data_dim = int(np.asarray(npz["data_dim"]).reshape(-1)[0])
        self.data_format = DataFormat()
        if "data_format" in npz:
            self.data_format.parse(str(np.asarray(npz["data_format"]).reshape(-1)[0]))
        elif self.data_dim == 4:
            self.data_format.format = DataFormat.RGBA
        else:
            self.data_format.format = DataFormat.SH
            self.data_format.basis_dim = (self.data_dim - 1) // 3
        if "invradius3" in npz:
            self.scale = np.asarray(npz["invradius3"], np.float32).reshape(3).copy()
        else:
            self.scale = np.full(3, np.float32(np.asarray(npz["invradius"], np.float64).reshape(-1)[0]), np.float32)
        self.offset = np.asarray(npz["offset"], np.float32).reshape(3).copy()
        child = np.asarray(npz["child"])
        if child.dtype != np.int32:
            child = child.astype(np.int32)
        self.child_ = np.ascontiguousarray(child)
        self.N = int(self.child_.shape[1])
        if self.N != 2:
            print("WARNING: N != 2 probably doesn't work.")
        self.quant_ = None
        self._data = None
        if "quant_colors" in npz:
            qc = np.asarray(npz["quant_colors"])
            if qc.dtype.itemsize != 2:
                raise RuntimeError("codebook must be stored in half precision")
            qmap = np.asarray(npz["quant_map"])
            self.capacity = int(qmap.shape[1])
            n_basis = int(qmap.shape[0])
            if qc.shape[0] != n_basis:
                raise RuntimeError("codebook and map basis numbers does not match")
            retained = np.asarray(npz["data_retained"]) if "data_retained" in npz else None
            n_retain = 0 if retained is None else int(retained.shape[0])
            n_child = self.capacity * self.N ** 3
            self.quant_ = dict(
                colors=np.ascontiguousarray(qc.view(np.uint16).reshape(n_basis, 65536, 3)),
                map=np.ascontiguousarray(qmap.astype(np.uint16, copy=False).reshape(n_basis, n_child)),
                sigma=np.ascontiguousarray(np.asarray(npz["sigma"]).view(np.uint16).reshape(n_child)),
                retained=None if retained is None else np.ascontiguousarray(retained.view(np.uint16).reshape(n_retain, n_child, 3)),
                n_quant=n_basis, n_retain=n_retain)
            if not self.gpu_decode:
                self._data = self._decode_quantised()
        else:
            data = np.asarray(npz["data"])
            self.capacity = int(data.shape[0])
            if data.dtype.itemsize != 2:
                raise RuntimeError("data must be stored in half precision")
            self._data = np.ascontiguousarray(data.view(np.float16))
        self.extra_ = np.ascontiguousarray(np.asarray(npz["extra_data"], np.float32)) if "extra_data" in npz else None

    def _decode_quantised(self) -> np.ndarray:
        """Vectorised form of the scalar decode loops of src/n3tree.cpp:309-340."""
        q = self.quant_
        n_basis, n_retain = q["n_quant"], q["n_retain"]
        n_total = n_basis + n_retain
        n_child = self.capacity * self.N ** 3
        data = np.zeros((n_child, self.data_dim), np.uint16)
        for j in range(n_basis):
            cols = q["colors"][j][q["map"][j].astype(np.int64)]      # [n_child,3]
            for k in range(3):
                data[:, j + n_retain + k * n_total] = cols[:, k]
        data[:, self.data_dim - 1] = q["sigma"]
        for j in range(n_retain):
            for k in range(3):
                data[:, j + k * n_total] = q["retained"][j, :, k]
        return data.view(np.float16).reshape(self.capacity, self.N, self.N, self.N, self.data_dim)

    def _unpack_llff_poses_bounds(self, pb: np.ndarray) -> None:
        """src/n3tree.cpp:22-52 (only the fields the ray path uses)."""
        p = np.asarray(pb).reshape(-1)
        self.ndc_height, self.ndc_width, self.ndc_focal = float(p[4]), float(p[9]), float(p[14])

    # -- device side (replaces src/cuda/n3tree.cu)
    def load_cuda(self) -> None:
        self.free_cuda()
        use_quant = self.quant_ is not None and self.gpu_decode
        qd = _capi.vr_tree_quant_desc() if use_quant else None
        d = qd.base if use_quant else _capi.vr_tree_desc()
        d.child = self.child_.ctypes.data
        if not use_quant:
            data = np.ascontiguousarray(self.data_)
            d.data = data.ctypes.data
        d.extra = self.extra_.ctypes.data if self.extra_ is not None else None
        d.capacity, d.N, d.data_dim = self.capacity, self.N, self.data_dim
        d.format, d.basis_dim = self.data_format.format, self.data_format.basis_dim
        for i in range(3):
            d.offset[i] = float(self.offset[i])
            d.scale[i] = float(self.scale[i])
        d.use_ndc = int(self.use_ndc)
        d.ndc_width, d.ndc_height, d.ndc_focal = self.ndc_width, self.ndc_height, self.ndc_focal
        h = C.c_void_p()
        if use_quant:
            q = self.quant_
            qd.quant_colors, qd.quant_map, qd.sigma = q["colors"].ctypes.data, q["map"].ctypes.data, q["sigma"].ctypes.data
            qd.data_retained = q["retained"].ctypes.data if q["retained"] is not None else None
            qd.n_quant, qd.n_retain = q["n_quant"], q["n_retain"]
            check(lib().vr_tree_create_quantized(C.byref(qd), C.byref(h)))
        else:
            check(lib().vr_tree_create(C.byref(d), C.byref(h)))
        self._handle = h
        self._cuda_loaded = True
        import torch
        self._device = torch.cuda.current_device()    # the tree lives on the device current at creation

    def _plain_desc(self):
        """vr_tree_desc over the decoded host arrays (keeps them alive through the returned tuple)."""
        d = _capi.vr_tree_desc()
        data = np.ascontiguousarray(self.data_)
        d.child, d.data = self.child_.ctypes.data, data.ctypes.data
        d.extra = self.extra_.ctypes.data if self.extra_ is not None else None
        d.capacity, d.N, d.data_dim = self.capacity, self.N, self.data_dim
        d.format, d.basis_dim = self.data_format.format, self.data_format.basis_dim
        for i in range(3):
            d.offset[i] = float(self.offset[i])
            d.scale[i] = float(self.scale[i])
        d.use_ndc = int(self.use_ndc)
        d.ndc_width, d.ndc_height, d.ndc_focal = self.ndc_width, self.ndc_height, self.ndc_focal
        return d, data

    def free_cuda(self) -> None:
        if self._handle is not None:
            lib().vr_tree_destroy(self._handle)
            self._handle = None
        self._cuda_loaded = False

    def info(self) -> dict:
        inf = _capi.vr_tree_info()
        check(lib().vr_tree_get_info(self._handle, C.byref(inf)))
        return {k: getattr(inf, k) for k, _ in inf._fields_}

    def __del__(self):
        try:
            self.free_cuda()
        except Exception:
            pass


# ---------------------------------------------------------------------------- Camera
class Camera:
    def __init__(self, width: int = 256, height: int = 256, fx: float = CAMERA_DEFAULT_FOCAL_LENGTH, fy: float = -1.0):
        self.width, self.height = int(width), int(height)
        self.fx = CAMERA_DEFAULT_FOCAL_LENGTH if fx < 0 else float(fx)
        self.fy = self.fx if fy < 0 else float(fy)
        self.center = np.array([-3.55, 0.0, 3.55], np.float32)      # camera.cpp:32-35
        self.v_back = np.array([-0.7071068, 0.0, 0.7071068], np.float32)
        self.v_world_up = np.array([0.0, 0.0, 1.0], np.float32)
        self.origin = np.zeros(3, np.float32)
        self.transform = np.zeros((4, 3), np.float32)               # glm::mat4x3: 4 columns of vec3
        self._update()

    def _update(self, transform_from_vecs: bool = True, copy_cuda: bool = True) -> None:
        """camera.cpp:47-76 (the device copy is unnecessary: c2w travels by value)."""
        if transform_from_vecs:
            self.v_back = (self.v_back / np.linalg.norm(self.v_back)).astype(np.float32)
            r = np.cross(self.v_world_up, self.v_back)
            self.v_right = (r / np.linalg.norm(r)).astype(np.float32)
            self.v_up = np.cross(self.v_back, self.v_right).astype(np.float32)
            self.transform[0], self.transform[1] = self.v_right, self.v_up
            self.transform[2], self.transform[3] = self.v_back, self.center

    def set_c2w(self, c2w) -> None:
        """Row-major 3x4/4x4 camera-to-world, as read by main_headless.cpp:40-63."""
        m = np.asarray(c2w, np.float32)[:3, :4]
        self.transform = np.ascontiguousarray(m.T)

    def _as_c(self) -> _capi.vr_camera:
        c = _capi.vr_camera()
        c.width, c.height, c.fx, c.fy = self.width, self.height, self.fx, self.fy
        flat = np.ascontiguousarray(self.transform, np.float32).reshape(12)
        for i in range(12):
            c.c2w[i] = float(flat[i])
        return c


# ---------------------------------------------------------------------------- RenderOptions
@dataclass
class RenderOptions:
    step_size: float = 1e-4
    sigma_thresh: float = 1e-2
    stop_thresh: float = 1e-2
    background_brightness: float = 1.0
    render_bbox: list = field(default_factory=lambda: [0.0, 0.0, 0.0, 1.0, 1.0, 1.0])
    basis_minmax: list = field(default_factory=lambda: [0, VOLREND_GLOBAL_BASIS_MAX - 1])
    rot_dirs: list = field(default_factory=lambda: [0.0, 0.0, 0.0])
    show_grid: bool = False
    grid_max_depth: int = 4
    render_depth: bool = False
    enable_probe: bool = False
    probe: list = field(default_factory=lambda: [0.0, 0.0, 1.0])
    probe_disp_size: int = 100

    def _as_c(self) -> _capi.vr_options:
        o = _capi.vr_options()
        o.step_size, o.sigma_thresh, o.stop_thresh = self.step_size, self.sigma_thresh, self.stop_thresh
        o.background_brightness = self.background_brightness
        for i in range(6):
            o.render_bbox[i] = float(self.render_bbox[i])
        o.basis_minmax[0], o.basis_minmax[1] = int(self.basis_minmax[0]), int(self.basis_minmax[1])
        for i in range(3):
            o.rot_dirs[i] = float(self.rot_dirs[i])
        o.render_depth = int(self.render_depth)
        return o


def _cams_array(cams) -> "C.Array":
    arr = (_capi.vr_camera * len(cams))()
    for i, cam in enumerate(cams):
        arr[i] = cam._as_c()
    return arr


def _stream_ptr(stream) -> int:
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    return int(getattr(stream, "cuda_stream", stream))


def _rect(tile):
    if tile is None:
        return None
    r = _capi.vr_rect(*[int(v) for v in tile])
    return C.byref(r)


# ---------------------------------------------------------------------------- launch_renderer
def launch_renderer(tree: N3Tree, cam: Camera, options: RenderOptions, image_arr, depth_arr=None,
                    stream=None, offscreen: bool = False, *, float_out=None, counters=None, tile=None) -> None:
    """``launch_renderer`` (renderer_kernel.hpp:9-12).  ``image_arr``: CUDA uint8 tensor
    [H,W,4] written in full (row 0 = top row); ``depth_arr``: float32 [H,W] ray-distance limits,
    required unless ``offscreen``.  Asynchronous on ``stream``.  Extras (keyword-only):
    ``float_out`` float32 [H,W,4] tap of the un-quantised pixel, ``counters`` uint64[5] device
    tensor, ``tile`` (x0,y0,w,h)."""
    if not tree.is_cuda_loaded():
        raise RuntimeError("N3Tree is not loaded on the device")
    c, o = cam._as_c(), options._as_c()
    img = image_arr.data_ptr() if image_arr is not None else None
    fo = float_out.data_ptr() if float_out is not None else None
    s = _stream_ptr(stream)
    if offscreen:
        cn = counters.data_ptr() if counters is not None else None
        check(lib().vr_render(tree._handle, C.byref(c), C.byref(o), _rect(tile), img, fo, cn, s))
    else:
        if depth_arr is None or image_arr is None:
            raise ValueError("offscreen=False needs colour and depth inputs")
        check(lib().vr_render_composite(tree._handle, C.byref(c), C.byref(o), _rect(tile), img,
                                        depth_arr.data_ptr(), fo, s))


def render_bands(tree: N3Tree, cam: Camera, options: RenderOptions, band_h: int, n_parts: int, part: int,
                 image, *, float_out=None, stream=None) -> int:
    """Ray-tile sharding: render bands part, part+n_parts, ... (band_h rows each) of the frame into the
    compact ``image`` (uint8 [rows, W, 4]); returns the number of rows this part owns."""
    c, o = cam._as_c(), options._as_c()
    check(lib().vr_render_bands(tree._handle, C.byref(c), C.byref(o), int(band_h), int(n_parts), int(part),
                                image.data_ptr() if image is not None else None,
                                float_out.data_ptr() if float_out is not None else None, _stream_ptr(stream)))
    return lib().vr_band_rows(cam.height, int(band_h), int(n_parts), int(part))


def render_bands_batch(tree: N3Tree, cams, options: RenderOptions, band_h: int, n_parts: int, part: int, images, *,
                       float_out=None, stream=None) -> int:
    """render_bands for several views in ONE launch: ``images`` uint8 [V, rows, W, 4]; returns rows."""
    arr = _cams_array(cams)
    o = options._as_c()
    check(lib().vr_render_bands_batch(tree._handle, arr, len(cams), C.byref(o), int(band_h), int(n_parts), int(part),
                                      images.data_ptr() if images is not None else None,
                                      float_out.data_ptr() if float_out is not None else None, _stream_ptr(stream)))
    return lib().vr_band_rows(cams[0].height, int(band_h), int(n_parts), int(part)) if len(cams) else 0


VR_MG_VIEWS, VR_MG_TILES = 0, 1


class MultiGpuRenderer:
    """One process driving several GPUs (vr_mg_*, volrend_b200/csrc/vr_mg.cu): the tree replicated on
    ``devices``, views or ray tiles sharded over them, frames gathered on ``devices[0]`` by peer copies.
    ``tree`` is a host-loaded N3Tree (its own device copy is not used)."""

    def __init__(self, tree: N3Tree, devices):
        self.devices = [int(d) for d in devices]
        d, keep = tree._plain_desc()
        arr = (C.c_int * len(self.devices))(*self.devices)
        h = C.c_void_p()
        rc = lib().vr_mg_create(C.byref(d), arr, len(self.devices), C.byref(h))
        del keep
        if rc != 0:
            raise _capi.VolrendError(rc, lib().vr_mg_last_error(None).decode("utf-8", "replace"))
        self._h = h

    def render(self, cams, options: RenderOptions, *, mode=VR_MG_VIEWS, band_h=8, batch=0, out_dev0=None, out_host=None) -> float:
        """Renders every view; returns the device time in ms (max over devices).  ``out_dev0``: uint8 CUDA
        tensor [V,H,W,4] on devices[0] (or None: internal buffer); ``out_host``: optional CPU array/tensor."""
        arr = _cams_array(cams)
        o = options._as_c()
        ms = C.c_float(0)
        hp = None
        if out_host is not None:
            hp = out_host.data_ptr() if hasattr(out_host, "data_ptr") else out_host.ctypes.data
        rc = lib().vr_mg_render(self._h, arr, len(cams), C.byref(o), int(mode), int(band_h), int(batch),
                                out_dev0.data_ptr() if out_dev0 is not None else None, hp, C.byref(ms))
        if rc != 0:
            raise _capi.VolrendError(rc, lib().vr_mg_last_error(self._h).decode("utf-8", "replace"))
        return float(ms.value)

    def close(self):
        if self._h is not None:
            lib().vr_mg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def render_batch(tree: N3Tree, cams, options: RenderOptions, images, *, float_out=None, counters=None,
                 tile=None, stream=None) -> None:
    """The pose loop of main_headless.cpp:208-223 as one call; ``images``: uint8 [V,H,W,4]."""
    arr = _cams_array(cams)
    o = options._as_c()
    check(lib().vr_render_batch(tree._handle, arr, len(cams), C.byref(o), _rect(tile),
                                images.data_ptr() if images is not None else None,
                                float_out.data_ptr() if float_out is not None else None,
                                counters.data_ptr() if counters is not None else None, _stream_ptr(stream)))


def _check_rays(name, t, last, device=None, shape=None):
    """ValueError unless ``t`` is a contiguous float32 CUDA tensor [..., last] (on ``device``, of leading ``shape``)."""
    import torch
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    if last is not None and (t.dim() < 1 or t.shape[-1] != last):
        raise ValueError(f"{name} must have shape [..., {last}], got {tuple(t.shape)}")
    lead = tuple(t.shape[:-1]) if last is not None else tuple(t.shape)
    if shape is not None and lead != tuple(shape):
        raise ValueError(f"{name} has leading shape {lead}, expected {tuple(shape)}")
    if device is not None and t.device.index != device:
        raise ValueError(f"{name} is on cuda:{t.device.index}, expected cuda:{device}")
    return lead


def render_rays(tree: N3Tree, origins, dirs, options: RenderOptions, out, *, t_max=None, counters=None,
                stream=None) -> None:
    """Renders caller-supplied rays (``vr_render_rays``): ``origins`` and ``dirs`` float32 CUDA tensors [..., 3] in
    world space (directions of any non-zero length), ``out`` float32 [..., 4] receives premultiplied RGB + background
    and alpha per ray; ``t_max`` optional float32 [...] depth limits (world distance along the normalised direction
    for non-NDC trees).  Each ray is rendered exactly as ``launch_renderer`` renders a pixel, so the rays of
    :func:`camera_rays` reproduce its float output bit for bit.  Rays with non-finite values or a zero direction are
    misses (background, alpha 0).  Asynchronous on ``stream``."""
    if not tree.is_cuda_loaded():
        raise RuntimeError("N3Tree is not loaded on the device")
    dev = tree._device
    lead = _check_rays("origins", origins, 3, dev)
    _check_rays("dirs", dirs, 3, dev, lead)
    _check_rays("out", out, 4, dev, lead)
    if t_max is not None:
        _check_rays("t_max", t_max, None, dev, lead)
    n = 1
    for k in lead:
        n *= int(k)
    if n > 0x7fffffff:
        raise ValueError(f"{n} rays: at most 2^31 - 1 per call")
    if counters is not None and (not counters.is_cuda or counters.device.index != dev):
        raise ValueError(f"counters must be a CUDA tensor on cuda:{dev}")
    o = options._as_c()
    check(lib().vr_render_rays(tree._handle, origins.data_ptr(), dirs.data_ptr(),
                               t_max.data_ptr() if t_max is not None else None, n, C.byref(o), out.data_ptr(),
                               counters.data_ptr() if counters is not None else None, _stream_ptr(stream)))


def camera_rays(cam: Camera, origins, dirs, *, tile=None, stream=None) -> None:
    """The rays the march generates for ``cam`` (``vr_camera_rays``): one per pixel of ``tile`` (x0,y0,w,h; None =
    full frame), row-major, into float32 CUDA tensors [..., 3] with w*h rays (e.g. [h, w, 3]).  Origins are the
    camera centre, directions are not normalised.  Asynchronous on ``stream``."""
    w, h = (cam.width, cam.height) if tile is None else (int(tile[2]), int(tile[3]))
    lead = _check_rays("origins", origins, 3)
    _check_rays("dirs", dirs, 3, origins.device.index, lead)
    if origins.numel() != 3 * w * h:
        raise ValueError(f"origins/dirs hold {origins.numel() // 3} rays, the {w}x{h} tile has {w * h}")
    import torch
    c = cam._as_c()
    with torch.cuda.device(origins.device):
        check(lib().vr_camera_rays(C.byref(c), _rect(tile), origins.data_ptr(), dirs.data_ptr(), _stream_ptr(stream)))


def render_frames_host(tree: N3Tree, cams, options: RenderOptions, host_images) -> None:
    """main_headless.cpp:208-223 with ``-o``: every frame lands in host memory
    (``host_images``: uint8 CPU tensor / ndarray [V,H,W,4], ideally pinned)."""
    arr = _cams_array(cams)
    o = options._as_c()
    ptr = host_images.data_ptr() if hasattr(host_images, "data_ptr") else host_images.ctypes.data
    check(lib().vr_render_frames_host(tree._handle, arr, len(cams), C.byref(o), ptr))


def write_png_file(filename: str, rgba8, width: int | None = None, height: int | None = None) -> bool:
    """``internal::write_png_file`` (src/imwrite.cpp:14-79) without libpng; ``rgba8``: uint8 [H,W,4]
    host array / CPU tensor."""
    arr = rgba8.numpy() if hasattr(rgba8, "numpy") else np.asarray(rgba8)
    arr = np.ascontiguousarray(arr, np.uint8)
    h, w = (arr.shape[0], arr.shape[1]) if height is None else (height, width)
    return lib().vr_write_png(filename.encode(), arr.ctypes.data, int(w), int(h)) == 0


def render_frames_png(tree: N3Tree, cams, options: RenderOptions, paths, n_threads: int = 8) -> None:
    """main_headless.cpp:208-223 with ``-o``: render every pose and write one PNG per pose."""
    arr = _cams_array(cams)
    o = options._as_c()
    cp = (C.c_char_p * len(paths))(*[p.encode() for p in paths])
    check(lib().vr_render_frames_png(tree._handle, arr, len(cams), C.byref(o), cp, int(n_threads)))


# ---------------------------------------------------------------------------- VolumeRenderer
class VolumeRenderer:
    """GL-free offscreen ``VolumeRenderer`` (renderer.hpp:11-42)."""

    def __init__(self):
        self.camera = Camera()
        self.options = RenderOptions()
        self.meshes = []            # kept for API compatibility; GL meshes are out of scope
        self._tree = None
        self._image = None
        self._depth = None
        self.resize(self.camera.width, self.camera.height)

    def get_backend(self) -> str:
        return "CUDA"

    def set(self, tree: N3Tree) -> None:
        self._tree = tree           # cuda_renderer.cpp:171-180
        self.options.basis_minmax = [0, max(tree.data_format.basis_dim - 1, 0)]

    def clear(self) -> None:
        self._tree = None

    def resize(self, width: int, height: int) -> None:
        import torch
        self.camera.width, self.camera.height = int(width), int(height)
        if torch.cuda.is_available():
            self._image = torch.zeros((height, width, 4), dtype=torch.uint8, device="cuda")
        else:
            self._image = None

    def render(self):
        """cuda_renderer.cpp:83-126 without the GL mesh pass: offscreen march into the
        renderer-owned RGBA8 buffer, which is returned."""
        if self._image is None:
            raise RuntimeError("VolumeRenderer needs a CUDA device (no CPU fallback)")
        self.camera._update()
        if self._tree is None or not self._tree.is_cuda_loaded():
            bg = int(self.options.background_brightness * 255)
            self._image[..., :3] = bg
            self._image[..., 3] = 255
            return self._image
        launch_renderer(self._tree, self.camera, self.options, self._image, None, None, True)
        return self._image
