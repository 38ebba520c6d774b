"""ctypes binding of include/rf_b200.h.  Fails loudly when librf_b200.so is missing: there is no
Python / CPU implementation of the path behind it."""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

RF_PREC_FP32, RF_PREC_FP16, RF_PREC_INT8 = 0, 1, 2
RF_FLAG_NO_GRAPH, RF_FLAG_NO_TENSORCORE, RF_FLAG_SIMT_STEM, RF_FLAG_DW_1D, RF_FLAG_LEGACY_TC, RF_FLAG_NPP_RESIZE = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20
FACE_FLOATS = 15
PIPELINE_DEPTH = 6   # RF_PIPELINE_DEPTH

# every symbol include/rf_b200.h declares (checked by tests/test_capi_symbols.py)
EXPORTS = [
    "rf_abi_version", "rf_build_info", "rf_status_string", "rf_create", "rf_destroy", "rf_last_error",
    "rf_pinned_input", "rf_device_input", "rf_detect_batch", "rf_submit_batch", "rf_collect_batch", "rf_detect_batch_device", "rf_forward_heads",
    "rf_postprocess", "rf_preprocess", "rf_get_net_size", "rf_num_anchors", "rf_stream", "rf_synchronize", "rf_fence", "rf_last_stream",
    "rf_launches_per_batch", "rf_profile_layers", "rf_debug_get_tensor", "rf_debug_keep_all", "rf_model_inspect", "rf_calibrate_int8", "rf_kl_threshold_bins",
    "rf_detect_views", "rf_plan_describe",
    "rf_comm_export", "rf_comm_init", "rf_comm_nccl_unique_id", "rf_comm_init_nccl", "rf_comm_info", "rf_detect_batch_device_allgather",
    "rf_submit_batch_allgather", "rf_collect_batch_allgather", "rf_detect_batch_allgather",
    "rf_model_load", "rf_network_config", "rf_cache_status",
    "rf_detect_jpeg_batch", "rf_decode_jpeg", "rf_jpeg_backend",
    "rf_detect_align_batch", "rf_align_batch_device",
]
COMM_BLOB_BYTES = 128


class _View(C.Structure):       # rf_view
    _fields_ = [("shrink", C.c_float), ("flip", C.c_int32)]


RF_CROP_U8_BGR, RF_CROP_F16_RGB = 0, 1
# insightface's arcface_dst: the five-landmark template of a 112 x 112 recognizer crop (crop pixels, float32)
ARCFACE_112 = np.array([[38.2946, 51.6963], [73.5318, 51.5014], [56.0252, 71.7366], [41.5493, 92.3655], [70.7299, 92.2041]],
                       dtype=np.float32)


class _AlignSpec(C.Structure):  # rf_align_spec
    _fields_ = [("crop_w", C.c_int), ("crop_h", C.c_int), ("dst_x", C.c_float * 5), ("dst_y", C.c_float * 5),
                ("max_crops", C.c_int), ("layout", C.c_int), ("mean", C.c_float), ("scale", C.c_float)]


def align_spec(crop: Tuple[int, int] = (112, 112), template=None, max_crops: int = 16, layout: int = RF_CROP_U8_BGR,
               mean: float = 127.5, scale: float = float(np.float32(1 / 127.5))) -> _AlignSpec:
    """rf_align_spec: crop = (width, height); template = (5, 2) landmark positions in crop pixels, None -> the ArcFace template
    scaled by crop / 112 (sides must then be multiples of 112); mean / scale apply to RF_CROP_F16_RGB."""
    t = np.zeros((5, 2), dtype=np.float32) if template is None else np.asarray(template, dtype=np.float32).reshape(5, 2)
    return _AlignSpec(int(crop[0]), int(crop[1]), (C.c_float * 5)(*t[:, 0]), (C.c_float * 5)(*t[:, 1]), int(max_crops), int(layout),
                      float(mean), float(scale))


def crop_shape(spec: _AlignSpec) -> Tuple[Tuple[int, ...], type]:
    """(shape, dtype) of one crop in the spec's layout."""
    if spec.layout == RF_CROP_F16_RGB:
        return (3, spec.crop_h, spec.crop_w), np.float16
    return (spec.crop_h, spec.crop_w, 3), np.uint8


class RfError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"librf_b200 status {status}: {msg}")
        self.status = status


class _Config(C.Structure):
    _fields_ = [("caffemodel_path", C.c_char_p), ("int8_table_path", C.c_char_p), ("precision", C.c_int),
                ("net_w", C.c_int), ("net_h", C.c_int), ("max_batch", C.c_int), ("max_faces", C.c_int),
                ("device", C.c_int), ("max_image_w", C.c_int), ("max_image_h", C.c_int), ("flags", C.c_uint),
                ("streams", C.c_int), ("prototxt_path", C.c_char_p), ("cache_path", C.c_char_p), ("network", C.c_char_p)]


def lib_path() -> str:
    return os.environ.get("RF_B200_LIB", os.path.join(_HERE, "librf_b200.so"))


_lib = None


def load_library() -> C.CDLL:
    """dlopen librf_b200.so (built in-tree by retinaface_b200/build.py or __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise ImportError(f"{p} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(retinaface_b200 has no CPU fallback)")
    lib = C.CDLL(p)
    lib.rf_build_info.restype = C.c_char_p
    lib.rf_status_string.restype = C.c_char_p
    lib.rf_last_error.restype = C.c_char_p
    lib.rf_last_error.argtypes = [C.c_void_p]
    lib.rf_create.argtypes = [C.POINTER(_Config), C.POINTER(C.c_void_p)]
    lib.rf_destroy.argtypes = [C.c_void_p]
    lib.rf_destroy.restype = None
    lib.rf_pinned_input.restype = C.c_void_p
    lib.rf_pinned_input.argtypes = [C.c_void_p]
    lib.rf_device_input.restype = C.c_void_p
    lib.rf_device_input.argtypes = [C.c_void_p]
    lib.rf_stream.restype = C.c_void_p
    lib.rf_stream.argtypes = [C.c_void_p]
    lib.rf_last_stream.restype = C.c_void_p
    lib.rf_last_stream.argtypes = [C.c_void_p]
    for name in ("rf_synchronize", "rf_num_anchors", "rf_fence"):
        getattr(lib, name).argtypes = [C.c_void_p]
    lib.rf_launches_per_batch.argtypes = [C.c_void_p, C.c_int]
    lib.rf_get_net_size.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 4
    lib.rf_detect_batch.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                    C.POINTER(C.c_int), C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rf_detect_views.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(_View), C.c_int, C.c_float, C.c_float,
                                    C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p]
    lib.rf_submit_batch.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_float, C.c_float, C.POINTER(C.c_int)]
    lib.rf_collect_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rf_detect_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float,
                                           C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    lib.rf_forward_heads.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
    lib.rf_postprocess.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_float, C.c_float,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rf_preprocess.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.rf_profile_layers.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.rf_debug_get_tensor.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_void_p] + [C.POINTER(C.c_int)] * 3
    lib.rf_debug_keep_all.argtypes = [C.c_void_p]
    lib.rf_calibrate_int8.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_char_p]
    lib.rf_kl_threshold_bins.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.rf_kl_threshold_bins.restype = C.c_double
    lib.rf_cache_status.argtypes = [C.c_void_p]
    lib.rf_comm_export.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.rf_comm_init.argtypes = [C.c_void_p, C.c_void_p]
    lib.rf_comm_nccl_unique_id.argtypes = [C.c_void_p]
    lib.rf_comm_init_nccl.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.rf_comm_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.rf_detect_batch_device_allgather.argtypes = lib.rf_detect_batch_device.argtypes
    lib.rf_submit_batch_allgather.argtypes = lib.rf_submit_batch.argtypes
    lib.rf_collect_batch_allgather.argtypes = lib.rf_collect_batch.argtypes
    lib.rf_detect_batch_allgather.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rf_detect_jpeg_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]
    lib.rf_decode_jpeg.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.rf_jpeg_backend.restype = C.c_char_p
    lib.rf_detect_align_batch.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int,
                                          C.c_float, C.c_float, C.POINTER(_AlignSpec), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
    lib.rf_align_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(_AlignSpec), C.c_void_p,
                                          C.c_void_p]
    lib.rf_jpeg_backend.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def model_inspect(caffemodel: str, layer: str):
    """(w, b) folded parameters of one convolution, from the library's host-side model front end."""
    lib = load_library()
    dims = (C.c_int * 4)()
    rc = lib.rf_model_inspect(caffemodel.encode(), layer.encode(), None, 0, None, 0, dims)
    if rc != 0:
        raise RfError(rc, (lib.rf_last_error(None) or b"").decode())
    shape = tuple(dims)
    w = np.empty(shape, dtype=np.float32)
    b = np.empty(shape[0], dtype=np.float32)
    rc = lib.rf_model_inspect(caffemodel.encode(), layer.encode(), w.ctypes.data_as(C.c_void_p), w.size,
                              b.ctypes.data_as(C.c_void_p), b.size, dims)
    if rc != 0:
        raise RfError(rc, (lib.rf_last_error(None) or b"").decode())
    return w, b


def plan_describe(caffemodel: str, net_h: int, net_w: int, precision: int = RF_PREC_FP16, max_batch: int = 8, flags: int = 0,
                  int8_table: Optional[str] = None, streams: int = 0) -> str:
    """The layer plan rf_create would build (host-only entry point: no GPU needed)."""
    lib = load_library()
    cfg = _Config(caffemodel.encode(), int8_table.encode() if int8_table else None, precision, net_w, net_h, max_batch, 0, 0, 0, 0, flags, streams, None, None, None)
    buf = C.create_string_buffer(1 << 16)
    lib.rf_plan_describe.argtypes = [C.POINTER(_Config), C.c_char_p, C.c_int]
    rc = lib.rf_plan_describe(C.byref(cfg), buf, len(buf))
    if rc < 0:
        raise RfError(rc, (lib.rf_last_error(None) or b"").decode())
    return buf.value.decode()


def model_load(caffemodel: str, prototxt: Optional[str] = None, cache: Optional[str] = None, layer: Optional[str] = None):
    """rf_model_load (host-only): the load path of rf_create.  Returns (cache_status, input_dims, (w, b) of `layer` or None)."""
    lib = load_library()
    lib.rf_model_load.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                  C.POINTER(C.c_int)]
    cs = C.c_int(0)
    idims = (C.c_int * 4)()
    dims = (C.c_int * 4)()
    args = (caffemodel.encode(), prototxt.encode() if prototxt else None, cache.encode() if cache else None, C.byref(cs), idims, layer.encode() if layer else None)
    rc = lib.rf_model_load(*args, None, 0, None, 0, dims)
    if rc != 0:
        raise RfError(rc, (lib.rf_last_error(None) or b"").decode())
    wb = None
    if layer:
        w = np.empty(tuple(dims), dtype=np.float32)
        b = np.empty(dims[0], dtype=np.float32)
        rc = lib.rf_model_load(*args, w.ctypes.data_as(C.c_void_p), w.size, b.ctypes.data_as(C.c_void_p), b.size, dims)
        if rc != 0:
            raise RfError(rc, (lib.rf_last_error(None) or b"").decode())
        wb = (w, b)
    return cs.value, tuple(idims), wb


def network_config(network: str):
    """rf_network_config: (strides, scales per level, ratios) of the reference's network-name switch; RfError(-7) where unsupported."""
    lib = load_library()
    lib.rf_network_config.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_float), C.POINTER(C.c_int)]
    nl, nr = C.c_int(0), C.c_int(0)
    strides, scales, ratios = (C.c_int * 3)(), (C.c_int * 6)(), (C.c_float * 2)()
    rc = lib.rf_network_config(network.encode(), C.byref(nl), strides, scales, ratios, C.byref(nr))
    if rc != 0:
        raise RfError(rc, (lib.rf_last_error(None) or b"").decode())
    return list(strides)[:nl.value], [list(scales)[2 * i:2 * i + 2] for i in range(nl.value)], list(ratios)[:nr.value]


def nccl_unique_id() -> bytes:
    """A fresh ncclUniqueId (rank 0 creates it, the caller ships it to the other ranks) for Engine.comm_init_nccl."""
    lib = load_library()
    buf = C.create_string_buffer(128)
    rc = lib.rf_comm_nccl_unique_id(buf)
    if rc != 0:
        raise RfError(rc, (lib.rf_last_error(None) or b"").decode())
    return buf.raw


def kl_threshold_bins(hist: np.ndarray, levels: int = 128) -> float:
    """The calibrator's threshold search (host-only entry point of the library)."""
    lib = load_library()
    h = np.ascontiguousarray(hist, dtype=np.uint32)
    return float(lib.rf_kl_threshold_bins(h.ctypes.data_as(C.c_void_p), len(h), levels))


STRIDES = (32, 16, 8)


def head_shapes(net_h: int, net_w: int) -> List[Tuple[int, int, int]]:
    return [(c, net_h // s, net_w // s) for s in STRIDES for c in (4, 8, 20)]


class Engine:
    """One rf_handle: one GPU, one stream."""

    def __init__(self, caffemodel: str, net_h: int, net_w: int, precision: int = RF_PREC_FP16, max_batch: int = 8,
                 max_faces: int = 256, device: int = 0, int8_table: Optional[str] = None,
                 max_image: Optional[Tuple[int, int]] = None, flags: int = 0, streams: int = 0, prototxt: Optional[str] = None,
                 cache: Optional[str] = None, network: Optional[str] = None):
        self.lib = load_library()
        cfg = _Config(caffemodel.encode(), int8_table.encode() if int8_table else None, precision, net_w, net_h,
                      max_batch, max_faces, device, max_image[1] if max_image else 0, max_image[0] if max_image else 0, flags, streams,
                      prototxt.encode() if prototxt else None, cache.encode() if cache else None, network.encode() if network else None)
        h = C.c_void_p()
        rc = self.lib.rf_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise RfError(rc, (self.lib.rf_last_error(None) or b"").decode())
        self.h = h
        if net_h == 0 and net_w == 0:          # taken from the prototxt
            nw, nh = C.c_int(), C.c_int()
            self.lib.rf_get_net_size(h, C.byref(nw), C.byref(nh), None, None)
            net_h, net_w = nh.value, nw.value
        self.net_h, self.net_w = net_h, net_w
        self.max_batch, self.precision, self.device = max_batch, precision, device
        mf = C.c_int()
        self.lib.rf_get_net_size(self.h, None, None, None, C.byref(mf))
        self.max_faces = mf.value
        self.num_anchors = self.lib.rf_num_anchors(self.h)

    def close(self):
        if getattr(self, "h", None):
            self.lib.rf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc < 0:
            raise RfError(rc, (self.lib.rf_last_error(self.h) or b"").decode())
        return rc

    # -- buffers --------------------------------------------------------------------------
    def pinned_input(self) -> np.ndarray:
        """numpy view of the library's pinned staging: (max_batch, H, W, 3) u8."""
        p = self.lib.rf_pinned_input(self.h)
        n = self.max_batch * self.net_h * self.net_w * 3
        buf = (C.c_uint8 * n).from_address(p)
        return np.frombuffer(buf, dtype=np.uint8).reshape(self.max_batch, self.net_h, self.net_w, 3)

    def device_input_ptr(self) -> int:
        return int(self.lib.rf_device_input(self.h))

    def stream_ptr(self) -> int:
        return int(self.lib.rf_stream(self.h) or 0)

    def synchronize(self):
        self._check(self.lib.rf_synchronize(self.h))

    def fence(self):
        """Order stream_ptr() after everything queued so far on every execution context."""
        self._check(self.lib.rf_fence(self.h))

    def last_stream_ptr(self) -> int:
        return int(self.lib.rf_last_stream(self.h) or 0)

    # -- end to end ------------------------------------------------------------------------
    def detect_batch(self, images: Sequence[np.ndarray], thr: float, nms_thr: float, want_index: bool = False):
        """images: u8 BGR HWC arrays (any size <= max_image).  Returns list of (k,15) float32 arrays
        (FaceDetectInfo rows, score order) [+ list of anchor-index arrays]."""
        n = len(images)
        keep = [np.ascontiguousarray(im, dtype=np.uint8) if not (im.flags.c_contiguous and im.dtype == np.uint8) else im
                for im in images]
        for im in keep:
            if im.ndim != 3 or im.shape[2] != 3:
                raise ValueError(f"u8 BGR HWC images expected, got shape {im.shape}")
        ptrs = (C.c_void_p * n)(*[im.ctypes.data for im in keep])
        ws = (C.c_int * n)(*[im.shape[1] for im in keep])
        hs = (C.c_int * n)(*[im.shape[0] for im in keep])
        faces = np.empty((n, self.max_faces, FACE_FLOATS), dtype=np.float32)
        counts = np.zeros(n, dtype=np.int32)
        idx = np.empty((n, self.max_faces), dtype=np.int32) if want_index else None
        self._check(self.lib.rf_detect_batch(self.h, ptrs, ws, hs, None, n, thr, nms_thr, faces.ctypes.data,
                                             counts.ctypes.data, idx.ctypes.data if want_index else None))
        out = [faces[i, :counts[i]].copy() for i in range(n)]
        if want_index:
            return out, [idx[i, :counts[i]].copy() for i in range(n)]
        return out

    def detect_align(self, images: Sequence[np.ndarray], thr: float, nms_thr: float, crop: Tuple[int, int] = (112, 112), template=None,
                     max_crops: int = 16, layout: int = RF_CROP_U8_BGR, want_index: bool = False, spec: Optional[_AlignSpec] = None):
        """rf_detect_align_batch: detect_batch + the aligned crops of the top min(count, max_crops) faces of each image, sampled
        from the original image.  images: u8 BGR HWC arrays (rows may be padded: any view with pixel stride 3).  Returns
        (per image (faces (k, 15) in network-input pixels, crops (m, ...) in the layout of crop_shape, affine (m, 2, 3) image ->
        crop), map-back scales (n,)) [+ anchor-index arrays]."""
        spec = spec if spec is not None else align_spec(crop, template, max_crops, layout)
        n = len(images)
        keep = []
        for im in images:
            if im.ndim != 3 or im.shape[2] != 3:
                raise ValueError(f"u8 BGR HWC images expected, got shape {im.shape}")
            if im.dtype != np.uint8 or im.strides[1:] != (3, 1) or im.strides[0] < 3 * im.shape[1]:
                im = np.ascontiguousarray(im, dtype=np.uint8)
            keep.append(im)
        ptrs = (C.c_void_p * n)(*[im.ctypes.data for im in keep])
        ws = (C.c_int * n)(*[im.shape[1] for im in keep])
        hs = (C.c_int * n)(*[im.shape[0] for im in keep])
        rs = (C.c_int * n)(*[im.strides[0] for im in keep])
        shape, dt = crop_shape(spec)
        mc = spec.max_crops
        faces = np.empty((n, self.max_faces, FACE_FLOATS), dtype=np.float32)
        counts = np.zeros(n, dtype=np.int32)
        idx = np.empty((n, self.max_faces), dtype=np.int32)
        scales = np.empty(n, dtype=np.float32)
        crops = np.empty((n, mc) + shape, dtype=dt)
        affine = np.empty((n, mc, 2, 3), dtype=np.float64)
        self._check(self.lib.rf_detect_align_batch(self.h, ptrs, ws, hs, rs, n, thr, nms_thr, C.byref(spec), faces.ctypes.data,
                                                   counts.ctypes.data, idx.ctypes.data, scales.ctypes.data, crops.ctypes.data,
                                                   affine.ctypes.data))
        out = []
        for i in range(n):
            m = min(int(counts[i]), mc)
            out.append((faces[i, :counts[i]].copy(), crops[i, :m].copy(), affine[i, :m].copy()))
        if want_index:
            return out, scales, [idx[i, :counts[i]].copy() for i in range(n)]
        return out, scales

    def align_device(self, n: int, dev_images_ptr: int, dets_ptr: int, counts_ptr: int, out_ptr: int, spec: _AlignSpec,
                     affine_ptr: Optional[int] = None):
        """rf_align_batch_device: aligned crops of the records of a detect_device() call on the same network-sized device images,
        written to caller device memory out_ptr ([n][max_crops][crop], e.g. a torch CUDA tensor's data_ptr()) and, optionally,
        the image -> crop matrices to affine_ptr ([n][max_crops][6] doubles).  Asynchronous on last_stream_ptr()."""
        self._check(self.lib.rf_align_batch_device(self.h, dev_images_ptr, n, dets_ptr, counts_ptr, C.byref(spec), out_ptr, affine_ptr))

    def detect_jpeg(self, streams: Sequence[bytes], thr: float, nms_thr: float):
        """JPEG bitstreams (bytes) -> decoded on the GPU (nvJPEG), letter-boxed, detected.  Returns (list of (k,15) arrays in
        network-input pixels, list of (width, height) of the decoded images)."""
        n = len(streams)
        bufs = [np.frombuffer(b, dtype=np.uint8) for b in streams]
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in bufs])
        lens = (C.c_size_t * n)(*[b.size for b in bufs])
        faces = np.empty((n, self.max_faces, FACE_FLOATS), dtype=np.float32)
        counts = np.zeros(n, dtype=np.int32)
        ws, hs = (C.c_int * n)(), (C.c_int * n)()
        self._check(self.lib.rf_detect_jpeg_batch(self.h, ptrs, lens, n, thr, nms_thr, faces.ctypes.data, counts.ctypes.data, None, ws, hs))
        return [faces[i, :counts[i]].copy() for i in range(n)], [(ws[i], hs[i]) for i in range(n)]

    def decode_jpeg(self, stream: bytes) -> np.ndarray:
        """nvJPEG decode of one stream -> (h, w, 3) u8 BGR (what rf_detect_jpeg_batch letter-boxes)."""
        buf = np.frombuffer(stream, dtype=np.uint8)
        w, hh = C.c_int(), C.c_int()
        self._check(self.lib.rf_decode_jpeg(self.h, buf.ctypes.data, buf.size, None, 0, C.byref(w), C.byref(hh)))
        out = np.empty((hh.value, w.value, 3), dtype=np.uint8)
        self._check(self.lib.rf_decode_jpeg(self.h, buf.ctypes.data, buf.size, out.ctypes.data, out.nbytes, C.byref(w), C.byref(hh)))
        return out

    def jpeg_backend(self) -> str:
        return self.lib.rf_jpeg_backend(self.h).decode()

    def detect_pinned(self, n: int, thr: float, nms_thr: float, faces: np.ndarray, counts: np.ndarray):
        """Hot-loop variant for bench.py: the n images are already in pinned_input(); results go
        into caller-provided arrays.  Still the full H2D -> GPU -> D2H path."""
        base = self.lib.rf_pinned_input(self.h)
        sz = self.net_h * self.net_w * 3
        if not hasattr(self, "_pin_args") or self._pin_args[0] != n:
            self._pin_args = (n, (C.c_void_p * n)(*[base + i * sz for i in range(n)]),
                              (C.c_int * n)(*[self.net_w] * n), (C.c_int * n)(*[self.net_h] * n))
        _, ptrs, ws, hs = self._pin_args
        self._check(self.lib.rf_detect_batch(self.h, ptrs, ws, hs, None, n, thr, nms_thr, faces.ctypes.data,
                                             counts.ctypes.data, None))

    def _net_sized(self, images: Sequence[np.ndarray]):
        """rf_submit_batch reads net_h * net_w * 3 bytes from every pointer: refuse anything else."""
        for im in images:
            if im.shape != (self.net_h, self.net_w, 3) or im.dtype != np.uint8 or not im.flags.c_contiguous:
                raise ValueError(f"network-sized C-contiguous uint8 images of shape {(self.net_h, self.net_w, 3)} expected, got {im.shape} {im.dtype}")

    def submit(self, images: Sequence[np.ndarray], thr: float, nms_thr: float, allgather: bool = False) -> int:
        """Pipelined path: queue one batch of network-sized images (H2D on the copy stream + forward + D2H);
        returns a ticket for collect().  Up to PIPELINE_DEPTH batches in flight.  allgather: the multi-GPU exchange too."""
        n = len(images)
        self._net_sized(images)
        ptrs = (C.c_void_p * n)(*[im.ctypes.data for im in images])
        t = C.c_int()
        fn = self.lib.rf_submit_batch_allgather if allgather else self.lib.rf_submit_batch
        self._check(fn(self.h, ptrs, n, thr, nms_thr, C.byref(t)))
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[t.value] = (n, images, allgather)      # keep the sources alive until collected
        return t.value

    def collect(self, ticket: int, faces: Optional[np.ndarray] = None, counts: Optional[np.ndarray] = None):
        n, _, allgather = self._inflight.pop(ticket)
        rows = self.comm_world * self.max_batch if allgather else n
        if faces is None:
            faces = np.empty((rows, self.max_faces, FACE_FLOATS), dtype=np.float32)
        if counts is None:
            counts = np.zeros(rows, dtype=np.int32)
        fn = self.lib.rf_collect_batch_allgather if allgather else self.lib.rf_collect_batch
        self._check(fn(self.h, ticket, faces.ctypes.data, counts.ctypes.data, None))
        return faces, counts

    # -- multi-GPU ---------------------------------------------------------------------------
    comm_world = 1

    def comm_export(self, rank: int, world: int) -> bytes:
        blob = C.create_string_buffer(COMM_BLOB_BYTES)
        self._check(self.lib.rf_comm_export(self.h, rank, world, blob))
        return blob.raw

    def comm_init(self, blobs: Sequence[bytes]):
        raw = b"".join(blobs)
        self._check(self.lib.rf_comm_init(self.h, raw))
        self.comm_world = len(blobs)

    def comm_init_nccl(self, unique_id: bytes, rank: int, world: int):
        self._check(self.lib.rf_comm_init_nccl(self.h, unique_id, rank, world))
        self.comm_world = world

    def detect_device_allgather(self, n: int, thr: float, nms_thr: float, dev_ptr: int):
        d, c = C.c_void_p(), C.c_void_p()
        self._check(self.lib.rf_detect_batch_device_allgather(self.h, dev_ptr, n, thr, nms_thr, C.byref(d), C.byref(c)))
        return int(d.value), int(c.value)

    def detect_device(self, n: int, thr: float, nms_thr: float, dev_ptr: Optional[int] = None):
        """Asynchronous device-resident detect.  Returns (dets_ptr, counts_ptr) device addresses."""
        d, c = C.c_void_p(), C.c_void_p()
        self._check(self.lib.rf_detect_batch_device(self.h, dev_ptr if dev_ptr is not None else self.device_input_ptr(),
                                                    n, thr, nms_thr, C.byref(d), C.byref(c)))
        return int(d.value), int(c.value)

    # -- parity entry points -----------------------------------------------------------------
    def forward_heads(self, images: np.ndarray) -> List[np.ndarray]:
        images = np.ascontiguousarray(images, dtype=np.uint8)
        n = images.shape[0]
        assert images.shape[1:] == (self.net_h, self.net_w, 3), images.shape
        outs = [np.empty((n,) + s, dtype=np.float32) for s in head_shapes(self.net_h, self.net_w)]
        ptrs = (C.c_void_p * 9)(*[o.ctypes.data for o in outs])
        self._check(self.lib.rf_forward_heads(self.h, images.ctypes.data, n, ptrs))
        return outs

    def postprocess(self, heads: Sequence[np.ndarray], thr: float, nms_thr: float):
        """heads: 9 arrays (n,C,h,w).  Returns (faces list, index list, candidate counts)."""
        keep = [np.ascontiguousarray(h, dtype=np.float32) for h in heads]
        n = keep[0].shape[0]
        ptrs = (C.c_void_p * 9)(*[k.ctypes.data for k in keep])
        faces = np.empty((n, self.max_faces, FACE_FLOATS), dtype=np.float32)
        idx = np.empty((n, self.max_faces), dtype=np.int32)
        counts = np.zeros(n, dtype=np.int32)
        ncand = np.zeros(n, dtype=np.int32)
        self._check(self.lib.rf_postprocess(self.h, ptrs, n, thr, nms_thr, faces.ctypes.data, counts.ctypes.data,
                                            idx.ctypes.data, ncand.ctypes.data))
        return ([faces[i, :counts[i]].copy() for i in range(n)], [idx[i, :counts[i]].copy() for i in range(n)], ncand)

    def preprocess(self, img: np.ndarray) -> np.ndarray:
        img = np.ascontiguousarray(img, dtype=np.uint8)
        out = np.empty((self.net_h, self.net_w, 3), dtype=np.uint8)
        self._check(self.lib.rf_preprocess(self.h, img.ctypes.data, img.shape[1], img.shape[0], 0, out.ctypes.data))
        return out

    def detect_views(self, img: np.ndarray, views, thr: float, nms: float):
        """rf_detect_views: one image, views = [(shrink, flip), ...] run as one batch, merged on the GPU.  Returns
        (faces [k, 15] in ORIGINAL IMAGE pixels, view index of each face [k], map-back scale of each view)."""
        img = np.ascontiguousarray(img, dtype=np.uint8)
        nv = len(views)
        varr = (_View * max(nv, 1))(*[_View(float(s), int(bool(f))) for s, f in views])
        faces = np.empty((self.max_faces, 15), dtype=np.float32)
        view_of = np.empty(self.max_faces, dtype=np.int32)
        scales = np.empty(max(nv, 1), dtype=np.float32)
        count = C.c_int(0)
        self._check(self.lib.rf_detect_views(self.h, C.c_void_p(img.ctypes.data), img.shape[1], img.shape[0], 0, varr, nv, C.c_float(thr),
                                             C.c_float(nms), C.c_void_p(faces.ctypes.data), C.byref(count),
                                             C.c_void_p(view_of.ctypes.data), C.c_void_p(scales.ctypes.data)))
        return faces[:count.value].copy(), view_of[:count.value].copy(), scales[:nv].copy()

    def calibrate_int8(self, images: np.ndarray, out_table: str):
        """INT8 entropy calibration on an RF_PREC_FP32 engine; writes a TensorRT-format table."""
        images = np.ascontiguousarray(images, dtype=np.uint8)
        assert images.shape[1:] == (self.net_h, self.net_w, 3)
        self._check(self.lib.rf_calibrate_int8(self.h, images.ctypes.data, images.shape[0], out_table.encode()))

    def debug_keep_all(self):
        self._check(self.lib.rf_debug_keep_all(self.h))

    def debug_tensor(self, name: str, n: int) -> np.ndarray:
        c, hh, ww = C.c_int(), C.c_int(), C.c_int()
        self._check(self.lib.rf_debug_get_tensor(self.h, name.encode(), n, None, C.byref(c), C.byref(hh), C.byref(ww)))
        out = np.empty((n, c.value, hh.value, ww.value), dtype=np.float32)
        self._check(self.lib.rf_debug_get_tensor(self.h, name.encode(), n, out.ctypes.data, C.byref(c), C.byref(hh), C.byref(ww)))
        return out

    def launches_per_batch(self, n: int) -> int:
        return self._check(self.lib.rf_launches_per_batch(self.h, n))

    def profile_layers(self, n: int, iters: int = 20):
        cap = 128
        names = C.create_string_buffer(64 * cap)
        ms = (C.c_float * cap)()
        by = (C.c_double * cap)()
        fl = (C.c_double * cap)()
        k = self._check(self.lib.rf_profile_layers(self.h, n, iters, names, ms, by, fl, cap))
        out = []
        for i in range(k):
            nm = names.raw[64 * i:64 * (i + 1)].split(b"\0", 1)[0].decode()
            out.append(dict(name=nm, ms=float(ms[i]), bytes=float(by[i]), flops=float(fl[i])))
        return out
