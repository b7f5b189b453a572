"""ctypes binding of the C-ABI in include/yolo_b200.h (libyolo_b200.so).

This is the stub a reference-side maintainer would write (see INTEGRATION.md); the Python drop-in module and the
benchmarks go through it.  There is NO fallback: if the shared library is missing or no CUDA device is usable,
construction raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libyolo_b200.so")

MAX_LAYERS = 32
MAX_ANCHORS = 8
CONTRACT_F, CONTRACT_P = 0, 1
ROUND_RNE, ROUND_FLOOR, ROUND_HALF_UP = 0, 1, 2
WLAYOUT_OIHW, WLAYOUT_OHWI, WLAYOUT_WEIGHT_H = 0, 1, 2
HEAD_PYTHON, HEAD_C = 0, 1
YUV_NV12, YUV_I420, YUV_YUYV = 0, 1, 2      # cv2.COLOR_YUV2BGR_NV12 / _I420 / _YUYV frames (yolo_b200_forward_yuv)
# Bayer mosaics named by the sensor's top-left 2x2 (yolo_b200_forward_bayer): cv2.COLOR_BayerRGGB2BGR / _BGGR / _GRBG / _GBRG
BAYER_RGGB, BAYER_BGGR, BAYER_GRBG, BAYER_GBRG = 0, 1, 2, 3

EXPORTS = [
    "yolo_b200_abi_version", "yolo_b200_last_error", "yolo_b200_cstride", "yolo_b200_default_params",
    "yolo_b200_create", "yolo_b200_destroy", "yolo_b200_set_stream", "yolo_b200_load", "yolo_b200_set_thresholds",
    "yolo_b200_set_conv_backend", "yolo_b200_set_host_chunk", "yolo_b200_debug_requant",
    "yolo_b200_forward_rgb444", "yolo_b200_forward_int8", "yolo_b200_forward_f32", "yolo_b200_forward_u8bgr",
    "yolo_b200_forward_u8bgr_dev", "yolo_b200_quantize_u8bgr", "yolo_b200_u8bgr_lut",
    "yolo_b200_forward_rgb444_dev", "yolo_b200_forward_int8_dev", "yolo_b200_forward_f32_dev", "yolo_b200_sync",
    "yolo_b200_quantize_rgb444", "yolo_b200_quantize_f32", "yolo_b200_rgb444_lut", "yolo_b200_conv_layer",
    "yolo_b200_backbone", "yolo_b200_calibrate_f32", "yolo_b200_update_trackers_f32", "yolo_b200_measure_f32", "yolo_b200_get_layer_output", "yolo_b200_detect", "yolo_b200_overflow_count",
    "yolo_b200_launch_count", "yolo_b200_slow_path_count", "yolo_b200_enable_timing", "yolo_b200_layer_times_ms", "yolo_b200_draw_rectangles",
    "yolo_forward", "yolo_b200_set_default_context",
    "yolo_b200_pack_detections", "yolo_b200_ipc_alloc", "yolo_b200_ipc_open", "yolo_b200_ipc_close", "yolo_b200_copy_async",
    "yolo_b200_submit_rgb444", "yolo_b200_submit_u8bgr", "yolo_b200_wait",
    "yolo_b200_resize_taps", "yolo_b200_resize_u8bgr", "yolo_b200_forward_u8bgr_resize", "yolo_b200_forward_u8bgr_resize_dev",
    "yolo_b200_resize_u8bgr_ragged", "yolo_b200_forward_u8bgr_ragged", "yolo_b200_submit_u8bgr_ragged",
    "yolo_b200_forward_u8bgr_ragged_dev",
    "yolo_b200_yuv_frame_bytes", "yolo_b200_yuv_to_bgr_resize", "yolo_b200_forward_yuv", "yolo_b200_submit_yuv",
    "yolo_b200_forward_yuv_dev",
    "yolo_b200_bayer_to_bgr_resize", "yolo_b200_forward_bayer", "yolo_b200_submit_bayer", "yolo_b200_forward_bayer_dev",
]


class Layer(C.Structure):
    _fields_ = [("cin", C.c_int32), ("cout", C.c_int32), ("activ", C.c_int32), ("pool", C.c_int32),
                ("ksize", C.c_int32), ("in_from", C.c_int32), ("reorg", C.c_int32), ("concat_with", C.c_int32)]


class Params(C.Structure):
    _fields_ = [
        ("num_layers", C.c_int32), ("layers", Layer * MAX_LAYERS),
        ("scale_w", C.c_int32 * MAX_LAYERS), ("scale_b", C.c_int32 * MAX_LAYERS),
        ("scale_a", C.c_int32 * (MAX_LAYERS + 1)), ("retune", C.c_int32 * MAX_LAYERS),
        ("contract", C.c_int32), ("round_mode", C.c_int32), ("head_mode", C.c_int32),
        ("num_anchors", C.c_int32), ("num_classes", C.c_int32), ("stride", C.c_int32),
        ("anchors", (C.c_float * 2) * MAX_ANCHORS),
        ("conf_thresh", C.c_float), ("nms_thresh", C.c_float), ("max_det", C.c_int32),
    ]


class Det(C.Structure):
    _fields_ = [("x1", C.c_float), ("y1", C.c_float), ("x2", C.c_float), ("y2", C.c_float), ("score", C.c_float),
                ("cls", C.c_int32), ("anchor_index", C.c_int32), ("pad_", C.c_int32)]


DET_DTYPE = np.dtype([("x1", "<f4"), ("y1", "<f4"), ("x2", "<f4"), ("y2", "<f4"), ("score", "<f4"),
                      ("cls", "<i4"), ("anchor_index", "<i4"), ("pad_", "<i4")])
assert DET_DTYPE.itemsize == C.sizeof(Det) == 32

_lib = None


class YoloB200Error(RuntimeError):
    pass


def load_library(path: Optional[str] = None):
    """dlopen libyolo_b200.so and declare prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise YoloB200Error("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)" % p)
    L = C.CDLL(p)
    vp, i32, i8p = C.c_void_p, C.c_int, C.c_void_p
    L.yolo_b200_last_error.restype = C.c_char_p
    L.yolo_b200_default_params.argtypes = [C.POINTER(Params)]
    L.yolo_b200_create.argtypes = [C.POINTER(vp), i32]
    L.yolo_b200_destroy.argtypes = [vp]
    L.yolo_b200_destroy.restype = None
    L.yolo_b200_set_stream.argtypes = [vp, vp]
    L.yolo_b200_load.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(Params), i32]
    L.yolo_b200_set_thresholds.argtypes = [vp, C.c_float, C.c_float]
    L.yolo_b200_set_conv_backend.argtypes = [vp, i32]
    L.yolo_b200_set_host_chunk.argtypes = [vp, i32]
    L.yolo_b200_debug_requant.argtypes = [vp, i32, vp, C.c_size_t, vp, i32]
    L.yolo_b200_wait.argtypes = [vp, i32]
    for name in ("yolo_b200_forward_rgb444", "yolo_b200_forward_int8", "yolo_b200_forward_f32", "yolo_b200_forward_u8bgr",
                 "yolo_b200_submit_rgb444", "yolo_b200_submit_u8bgr",
                 "yolo_b200_forward_u8bgr_dev", "yolo_b200_forward_rgb444_dev", "yolo_b200_forward_int8_dev", "yolo_b200_forward_f32_dev"):
        getattr(L, name).argtypes = [vp, vp, i32, i32, i32, vp, vp]
    L.yolo_b200_sync.argtypes = [vp]
    L.yolo_b200_resize_u8bgr.argtypes = [vp, vp, i32, i32, i32, vp, i32, i32]
    L.yolo_b200_resize_taps.argtypes = [i32, i32, i32, vp]
    L.yolo_b200_forward_u8bgr_resize.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp]
    L.yolo_b200_forward_u8bgr_resize_dev.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp]
    L.yolo_b200_resize_u8bgr_ragged.argtypes = [vp, vp, i32, vp, vp, i32, i32]
    for name in ("yolo_b200_forward_u8bgr_ragged", "yolo_b200_submit_u8bgr_ragged", "yolo_b200_forward_u8bgr_ragged_dev"):
        getattr(L, name).argtypes = [vp, vp, i32, vp, i32, i32, vp, vp]
    L.yolo_b200_yuv_frame_bytes.argtypes = [i32, i32, i32]
    L.yolo_b200_yuv_to_bgr_resize.argtypes = [vp, vp, i32, i32, i32, i32, vp, i32, i32]
    for name in ("yolo_b200_forward_yuv", "yolo_b200_submit_yuv", "yolo_b200_forward_yuv_dev"):
        getattr(L, name).argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp]
    L.yolo_b200_bayer_to_bgr_resize.argtypes = [vp, vp, i32, i32, i32, i32, vp, i32, i32]
    for name in ("yolo_b200_forward_bayer", "yolo_b200_submit_bayer", "yolo_b200_forward_bayer_dev"):
        getattr(L, name).argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp]
    L.yolo_b200_quantize_rgb444.argtypes = [vp, vp, i32, i32, i32, vp]
    L.yolo_b200_quantize_f32.argtypes = [vp, vp, i32, i32, i32, vp]
    L.yolo_b200_rgb444_lut.argtypes = [vp, vp]
    L.yolo_b200_quantize_u8bgr.argtypes = [vp, vp, i32, i32, i32, vp]
    L.yolo_b200_calibrate_f32.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    L.yolo_b200_update_trackers_f32.argtypes = [vp, vp, i32, i32, i32, C.c_float, vp, vp, vp]
    L.yolo_b200_measure_f32.argtypes = [vp, vp, i32, i32, i32, vp]
    L.yolo_b200_pack_detections.argtypes = [vp, vp, vp, i32, vp, vp]
    L.yolo_b200_ipc_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp), C.c_char_p]
    L.yolo_b200_ipc_open.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    L.yolo_b200_ipc_close.argtypes = [vp, vp, i32]
    L.yolo_b200_copy_async.argtypes = [vp, vp, vp, C.c_size_t, vp]
    L.yolo_b200_u8bgr_lut.argtypes = [vp, vp]
    L.yolo_b200_conv_layer.argtypes = [vp, i32, i8p, i32, i32, i32, i8p]
    L.yolo_b200_backbone.argtypes = [vp, vp, i32, i32, i32, C.POINTER(vp), C.POINTER(i32), C.POINTER(i32)]
    L.yolo_b200_get_layer_output.argtypes = [vp, i32, vp, C.c_size_t]
    L.yolo_b200_detect.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp]
    L.yolo_b200_overflow_count.argtypes = [vp, C.POINTER(C.c_int64)]
    L.yolo_b200_launch_count.argtypes = [vp]
    L.yolo_b200_launch_count.restype = C.c_int64
    L.yolo_b200_slow_path_count.argtypes = [vp]
    L.yolo_b200_slow_path_count.restype = C.c_int64
    L.yolo_b200_enable_timing.argtypes = [vp, i32]
    L.yolo_b200_layer_times_ms.argtypes = [vp, C.POINTER(C.c_float), i32]
    L.yolo_b200_draw_rectangles.argtypes = [vp, i32, i32, vp, i32, i32]
    L.yolo_forward.argtypes = [C.c_char] * 6 + [vp, vp]
    L.yolo_forward.restype = None
    L.yolo_b200_set_default_context.argtypes = [vp]
    if path is None:
        _lib = L
    return L


def make_params(qnet, contract=CONTRACT_P, round_mode=ROUND_RNE, head_mode=HEAD_PYTHON, conf_thresh=0.1,
                nms_thresh=0.5, max_det=4096) -> Params:
    """Params from an export.QuantNet (tables are data, not compile-time constants)."""
    p = Params()
    p.num_layers = len(qnet.layers)
    # contract F is the 16-bit accumulator programme: it needs a retune[] that was derived from real activations
    retune = qnet.require_retune("contract F") if contract == CONTRACT_F else (qnet.retune or [0] * len(qnet.layers))
    for l, (cin, cout, activ, pool) in enumerate(qnet.layers):
        g = (getattr(qnet, "graph", None) or [{}] * len(qnet.layers))[l]
        p.layers[l] = Layer(cin, cout, activ, pool, g.get("ksize", 0), g.get("in_from", 0), g.get("reorg", 0), g.get("concat_with", 0))
        p.scale_w[l] = qnet.sw[l]; p.scale_b[l] = qnet.sb[l]; p.retune[l] = retune[l]
    for l, v in enumerate(qnet.sa):
        p.scale_a[l] = v
    p.contract = contract; p.round_mode = round_mode; p.head_mode = head_mode
    p.num_anchors = len(qnet.anchors); p.num_classes = qnet.num_classes; p.stride = qnet.stride
    for a, (w, h) in enumerate(qnet.anchors):
        p.anchors[a][0] = w; p.anchors[a][1] = h
    p.conf_thresh = conf_thresh; p.nms_thresh = nms_thresh; p.max_det = max_det
    return p


def _ptr(x):
    """Raw address of a numpy array / torch tensor (host or device) / int."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return x.data_ptr()        # torch.Tensor


def pack_images(images) -> "tuple[np.ndarray, np.ndarray]":
    """A list of uint8 BGR images [h][w][3] of any sizes (what cv2.imread returns) -> (flat uint8 buffer with the images
    back to back, int32 [n][2] of their (h, w)): the input of the *_ragged entry points."""
    shapes = np.zeros((len(images), 2), dtype=np.int32)
    for i, im in enumerate(images):
        if not isinstance(im, np.ndarray) or im.dtype != np.uint8 or im.ndim != 3 or im.shape[2] != 3:
            raise ValueError("image %d: need a uint8 array [h][w][3], got %s %s" % (i, getattr(im, "dtype", type(im)), getattr(im, "shape", "")))
        if not im.flags.c_contiguous:
            raise ValueError("image %d is not C-contiguous" % i)
        shapes[i] = im.shape[:2]
    flat = np.concatenate([im.reshape(-1) for im in images]) if len(images) else np.zeros(0, dtype=np.uint8)
    return flat, shapes


def yuv_frame_shape(fmt: int, sh: int, sw: int) -> "tuple[int, ...]":
    """The cv2 Mat shape of one YUV frame of source size sh x sw: (sh*3//2, sw) for YUV_NV12 / YUV_I420, (sh, sw, 2) for
    YUV_YUYV.  Raises ValueError for an unknown format or sizes the format cannot hold (4:2:0 needs even sh and sw, YUYV an
    even sw)."""
    if fmt not in (YUV_NV12, YUV_I420, YUV_YUYV):
        raise ValueError("unknown YUV format %r" % (fmt,))
    sh, sw = int(sh), int(sw)
    if sh < 1 or sw < 1 or sw % 2 or (fmt != YUV_YUYV and sh % 2):
        raise ValueError("YUV format %d cannot hold a %dx%d frame" % (fmt, sh, sw))
    return (sh * 3 // 2, sw) if fmt != YUV_YUYV else (sh, sw, 2)


def yuv_source_size(fmt: int, frame_shape) -> "tuple[int, int]":
    """(sh, sw) of a YUV frame from its cv2 Mat shape (the inverse of yuv_frame_shape)."""
    fs = tuple(int(x) for x in frame_shape)
    size = (fs[0] * 2 // 3, fs[1]) if fmt != YUV_YUYV and len(fs) == 2 else (fs[0], fs[1]) if len(fs) == 3 else None
    if size is None or yuv_frame_shape(fmt, *size) != fs:
        raise ValueError("%s is not the shape of a YUV format %r frame" % (fs, fmt))
    return size


def bayer_source_size(pattern: int, frame_shape) -> "tuple[int, int]":
    """(sh, sw) of Bayer frames [n][sh][sw] (frame_shape without n).  Raises ValueError for an unknown pattern or a frame
    smaller than 3x3 (cv2 itself returns zeros there; the library refuses such frames)."""
    if pattern not in (BAYER_RGGB, BAYER_BGGR, BAYER_GRBG, BAYER_GBRG):
        raise ValueError("unknown Bayer pattern %r" % (pattern,))
    fs = tuple(int(x) for x in frame_shape)
    if len(fs) != 2 or fs[0] < 3 or fs[1] < 3:
        raise ValueError("%s is not the shape of a Bayer frame [sh][sw] of at least 3x3" % (fs,))
    return fs


class Context:
    """One library context = one GPU (yolo_b200_create)."""

    def __init__(self, device: int = 0):
        self.L = load_library()
        h = C.c_void_p()
        self._h = None
        self._check(self.L.yolo_b200_create(C.byref(h), device))
        self._h = h
        self.device = device
        self.params: Optional[Params] = None
        self._keep = None

    def _check(self, rc):
        if rc != 0:
            raise YoloB200Error("yolo_b200 error %d: %s" % (rc, self.L.yolo_b200_last_error().decode()))

    def close(self):
        if self._h is not None:
            self.L.yolo_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- setup
    def load(self, weights: Sequence[np.ndarray], biases: Sequence[np.ndarray], params: Params, layout=WLAYOUT_OHWI):
        ws = [np.ascontiguousarray(w, dtype=np.int8) for w in weights]
        bs = [np.ascontiguousarray(b, dtype=np.int8) for b in biases]
        wp = (C.c_void_p * len(ws))(*[w.ctypes.data for w in ws])
        bp = (C.c_void_p * len(bs))(*[b.ctypes.data for b in bs])
        self._check(self.L.yolo_b200_load(self._h, wp, bp, C.byref(params), layout))
        self.params = params

    def load_quantnet(self, qnet, **kw):
        p = make_params(qnet, **kw)
        self.load(qnet.w, qnet.b, p, WLAYOUT_OHWI)
        return p

    def set_stream(self, stream_ptr: int):
        """stream_ptr: a cudaStream_t.  torch reports its default stream as 0, which the C-ABI reads as "use the
        context's own stream"; the legacy default stream is therefore passed as cudaStreamLegacy (0x1)."""
        self._check(self.L.yolo_b200_set_stream(self._h, stream_ptr or 1))

    def set_thresholds(self, conf, nms):
        self._check(self.L.yolo_b200_set_thresholds(self._h, conf, nms))
        self.params.conf_thresh = conf; self.params.nms_thresh = nms

    def set_conv_backend(self, backend: int):
        """0 auto, 1 integer dot-product kernels only, 2 tcgen05 only."""
        self._check(self.L.yolo_b200_set_conv_backend(self._h, backend))

    def set_host_chunk(self, frames: int):
        """Frames per chunk of the pipelined host-buffer entry points (0 = no chunking)."""
        self._check(self.L.yolo_b200_set_host_chunk(self._h, frames))

    def debug_requant(self, layer, d_acc, count, d_out, force_generic=False) -> int:
        rc = self.L.yolo_b200_debug_requant(self._h, layer, _ptr(d_acc), count, _ptr(d_out), int(force_generic))
        if rc < 0:
            self._check(rc)
        return rc

    def set_default(self):
        self._check(self.L.yolo_b200_set_default_context(self._h))

    # -- host-buffer forward (copies inside the call)
    def _forward_host(self, fn, n, *args):
        """A blocking host-buffer call fn(ctx, *args, dets, counts) over n frames -> (dets [n][max_det], counts [n])."""
        dets = np.zeros((n, self.params.max_det), dtype=DET_DTYPE)
        counts = np.zeros(n, dtype=np.int32)
        self._check(fn(self._h, *args, dets.ctypes.data, counts.ctypes.data))
        return dets, counts

    def _submit(self, fn, *args) -> int:
        """An asynchronous host-buffer call fn(ctx, *args) -> its ticket."""
        t = fn(self._h, *args)
        if t < 0:
            self._check(t)
        return t

    def forward_rgb444(self, frames: np.ndarray):
        f = np.ascontiguousarray(frames, dtype=np.uint16)
        n, h, w = f.shape
        return self._forward_host(self.L.yolo_b200_forward_rgb444, n, f.ctypes.data, n, h, w)

    def submit_rgb444(self, frames: np.ndarray, dets: np.ndarray, counts: np.ndarray) -> int:
        """Queue one batch (uint16 [n][h][w], C-contiguous; dets [n][max_det] DET_DTYPE, counts int32 [n]: the arrays must
        stay alive and untouched until wait(ticket)).  Returns the ticket."""
        assert frames.dtype == np.uint16 and frames.flags.c_contiguous and dets.flags.c_contiguous and counts.flags.c_contiguous
        n, h, w = frames.shape
        return self._submit(self.L.yolo_b200_submit_rgb444, frames.ctypes.data, n, h, w, dets.ctypes.data, counts.ctypes.data)

    def wait(self, ticket: int):
        self._check(self.L.yolo_b200_wait(self._h, ticket))

    def forward_u8bgr(self, images: np.ndarray):
        """uint8 BGR images [n][h][w][3] at network size (what cv2 delivers): BaseTransform arithmetic + tracker quantiser
        + forward pass, all on the GPU."""
        f = np.ascontiguousarray(images, dtype=np.uint8)
        n, h, w, c = f.shape
        assert c == 3
        return self._forward_host(self.L.yolo_b200_forward_u8bgr, n, f.ctypes.data, n, h, w)

    def forward_u8bgr_resize(self, images: np.ndarray, size):
        """uint8 BGR images [n][sh][sw][3] of any one size: the reference's whole BaseTransform (cv2.resize bilinear to
        size = (h, w), normalise, BGR -> RGB) + tracker quantiser + forward pass, all on the GPU."""
        f = np.ascontiguousarray(images, dtype=np.uint8)
        n, sh, sw, c = f.shape
        assert c == 3
        return self._forward_host(self.L.yolo_b200_forward_u8bgr_resize, n, f.ctypes.data, n, sh, sw, int(size[0]), int(size[1]))

    def forward_u8bgr_images(self, images, size):
        """A list of uint8 BGR images of any sizes (cv2.imread arrays) -> (dets [n][max_det], counts [n]) in one call: the
        whole BaseTransform (resize to size = (h, w) included) + forward pass on the GPU.  Boxes are normalised: image i
        scales them by its own [w, h, w, h]."""
        flat, shapes = pack_images(images)
        n = len(shapes)
        return self._forward_host(self.L.yolo_b200_forward_u8bgr_ragged, n, flat.ctypes.data, n, shapes.ctypes.data, int(size[0]), int(size[1]))

    def submit_u8bgr_images(self, packed, shapes: np.ndarray, size, dets: np.ndarray, counts: np.ndarray) -> int:
        """Queue one batch of packed images (pack_images; `packed` a numpy array or a pinned torch tensor) for size = (h, w);
        packed, dets [n][max_det] DET_DTYPE and counts int32 [n] must stay alive and untouched until wait(ticket)."""
        shapes = np.ascontiguousarray(shapes, dtype=np.int32)
        assert dets.flags.c_contiguous and counts.flags.c_contiguous and len(dets) >= len(shapes) and len(counts) >= len(shapes)
        return self._submit(self.L.yolo_b200_submit_u8bgr_ragged, _ptr(packed), len(shapes), shapes.ctypes.data, int(size[0]), int(size[1]),
                            dets.ctypes.data, counts.ctypes.data)

    def forward_yuv(self, frames: np.ndarray, fmt: int, size):
        """uint8 YUV frames [n, *yuv_frame_shape(fmt, sh, sw)] (cv2 Mat layout: decoder NV12 / I420, webcam YUYV) ->
        (dets [n][max_det], counts [n]): cv2.cvtColor to BGR, cv2.resize to size = (h, w) and the rest of
        forward_u8bgr_resize, all on the GPU; the frames cross the link as they are (1.5 or 2 bytes per pixel)."""
        f = np.ascontiguousarray(frames, dtype=np.uint8)
        sh, sw = yuv_source_size(fmt, f.shape[1:])
        n = f.shape[0]
        return self._forward_host(self.L.yolo_b200_forward_yuv, n, f.ctypes.data, fmt, n, sh, sw, int(size[0]), int(size[1]))

    def submit_yuv(self, frames, fmt: int, size, dets: np.ndarray, counts: np.ndarray) -> int:
        """Queue one batch of YUV frames [n, *yuv_frame_shape] (a C-contiguous numpy array or a pinned torch tensor) for
        size = (h, w); frames, dets [n][max_det] DET_DTYPE and counts int32 [n] must stay alive and untouched until
        wait(ticket).  Returns the ticket."""
        shape = tuple(frames.shape)
        sh, sw = yuv_source_size(fmt, shape[1:])
        n = shape[0]
        if isinstance(frames, np.ndarray):
            assert frames.dtype == np.uint8 and frames.flags.c_contiguous
        else:
            assert str(frames.dtype) == "torch.uint8" and frames.is_contiguous()
        assert dets.flags.c_contiguous and counts.flags.c_contiguous and len(dets) >= n and len(counts) >= n
        return self._submit(self.L.yolo_b200_submit_yuv, _ptr(frames), fmt, n, sh, sw, int(size[0]), int(size[1]),
                            dets.ctypes.data, counts.ctypes.data)

    def forward_bayer(self, frames: np.ndarray, pattern: int, size):
        """uint8 Bayer frames [n][sh][sw] (raw sensor mosaic, pattern BAYER_*) -> (dets [n][max_det], counts [n]):
        cv2.cvtColor to BGR, cv2.resize to size = (h, w) and the rest of forward_u8bgr_resize, all on the GPU; the frames
        cross the link as they are (1 byte per pixel)."""
        f = np.ascontiguousarray(frames, dtype=np.uint8)
        if f.ndim != 3:
            raise ValueError("Bayer frames are [n][sh][sw], got shape %s" % (f.shape,))
        sh, sw = bayer_source_size(pattern, f.shape[1:])
        n = f.shape[0]
        return self._forward_host(self.L.yolo_b200_forward_bayer, n, f.ctypes.data, pattern, n, sh, sw, int(size[0]), int(size[1]))

    def submit_bayer(self, frames, pattern: int, size, dets: np.ndarray, counts: np.ndarray) -> int:
        """Queue one batch of Bayer frames [n][sh][sw] (a C-contiguous numpy array or a pinned torch tensor) for
        size = (h, w); frames, dets [n][max_det] DET_DTYPE and counts int32 [n] must stay alive and untouched until
        wait(ticket).  Returns the ticket."""
        shape = tuple(frames.shape)
        if len(shape) != 3:
            raise ValueError("Bayer frames are [n][sh][sw], got shape %s" % (shape,))
        sh, sw = bayer_source_size(pattern, shape[1:])
        n = shape[0]
        if isinstance(frames, np.ndarray):
            assert frames.dtype == np.uint8 and frames.flags.c_contiguous
        else:
            assert str(frames.dtype) == "torch.uint8" and frames.is_contiguous()
        assert dets.flags.c_contiguous and counts.flags.c_contiguous and len(dets) >= n and len(counts) >= n
        return self._submit(self.L.yolo_b200_submit_bayer, _ptr(frames), pattern, n, sh, sw, int(size[0]), int(size[1]),
                            dets.ctypes.data, counts.ctypes.data)

    def forward_int8(self, nhwc4: np.ndarray):
        x = np.ascontiguousarray(nhwc4, dtype=np.int8)
        n, h, w, c = x.shape
        assert c == 4
        return self._forward_host(self.L.yolo_b200_forward_int8, n, x.ctypes.data, n, h, w)

    def forward_f32(self, nchw: np.ndarray):
        x = np.ascontiguousarray(nchw, dtype=np.float32)
        n, c, h, w = x.shape
        assert c == 3
        return self._forward_host(self.L.yolo_b200_forward_f32, n, x.ctypes.data, n, h, w)

    # -- device-buffer entry points (torch tensors or raw pointers), asynchronous
    def forward_int8_dev(self, d_in, n, h, w, d_dets, d_counts):
        self._check(self.L.yolo_b200_forward_int8_dev(self._h, _ptr(d_in), n, h, w, _ptr(d_dets), _ptr(d_counts)))

    def forward_rgb444_dev(self, d_in, n, h, w, d_dets, d_counts):
        self._check(self.L.yolo_b200_forward_rgb444_dev(self._h, _ptr(d_in), n, h, w, _ptr(d_dets), _ptr(d_counts)))

    def forward_f32_dev(self, d_in, n, h, w, d_dets, d_counts):
        self._check(self.L.yolo_b200_forward_f32_dev(self._h, _ptr(d_in), n, h, w, _ptr(d_dets), _ptr(d_counts)))

    def forward_u8bgr_dev(self, d_in, n, h, w, d_dets, d_counts):
        self._check(self.L.yolo_b200_forward_u8bgr_dev(self._h, _ptr(d_in), n, h, w, _ptr(d_dets), _ptr(d_counts)))

    def forward_u8bgr_resize_dev(self, d_in, n, sh, sw, h, w, d_dets, d_counts):
        self._check(self.L.yolo_b200_forward_u8bgr_resize_dev(self._h, _ptr(d_in), n, sh, sw, h, w, _ptr(d_dets), _ptr(d_counts)))

    def forward_u8bgr_ragged_dev(self, d_in, shapes, h, w, d_dets, d_counts):
        """Packed images of different sizes in device memory; shapes: host int32 [n][2] (pack_images)."""
        shapes = np.ascontiguousarray(shapes, dtype=np.int32).reshape(-1, 2)
        self._check(self.L.yolo_b200_forward_u8bgr_ragged_dev(self._h, _ptr(d_in), len(shapes), shapes.ctypes.data, h, w,
                                                              _ptr(d_dets), _ptr(d_counts)))

    def resize_u8bgr_ragged(self, d_src, shapes, d_dst, dh, dw):
        """cv2.resize (bilinear) of packed device images of different sizes (shapes: host int32 [n][2]) into d_dst [n][dh][dw][3]."""
        shapes = np.ascontiguousarray(shapes, dtype=np.int32).reshape(-1, 2)
        self._check(self.L.yolo_b200_resize_u8bgr_ragged(self._h, _ptr(d_src), len(shapes), shapes.ctypes.data, _ptr(d_dst), dh, dw))

    def forward_yuv_dev(self, d_in, fmt, n, sh, sw, h, w, d_dets, d_counts):
        """n YUV frames of source size sh x sw packed in device memory (layout of forward_yuv)."""
        self._check(self.L.yolo_b200_forward_yuv_dev(self._h, _ptr(d_in), fmt, n, sh, sw, h, w, _ptr(d_dets), _ptr(d_counts)))

    def yuv_to_bgr_resize(self, d_src, fmt, n, sh, sw, d_dst, dh, dw):
        """cv2.resize(cv2.cvtColor(frame, code), (dw, dh)) of n device YUV frames into d_dst uint8 [n][dh][dw][3]."""
        self._check(self.L.yolo_b200_yuv_to_bgr_resize(self._h, _ptr(d_src), fmt, n, sh, sw, _ptr(d_dst), dh, dw))

    def forward_bayer_dev(self, d_in, pattern, n, sh, sw, h, w, d_dets, d_counts):
        """n Bayer frames of source size sh x sw packed in device memory (layout of forward_bayer)."""
        self._check(self.L.yolo_b200_forward_bayer_dev(self._h, _ptr(d_in), pattern, n, sh, sw, h, w, _ptr(d_dets), _ptr(d_counts)))

    def bayer_to_bgr_resize(self, d_src, pattern, n, sh, sw, d_dst, dh, dw):
        """cv2.resize(cv2.cvtColor(frame, code), (dw, dh)) of n device Bayer frames into d_dst uint8 [n][dh][dw][3]."""
        self._check(self.L.yolo_b200_bayer_to_bgr_resize(self._h, _ptr(d_src), pattern, n, sh, sw, _ptr(d_dst), dh, dw))

    def resize_u8bgr(self, d_src, n, sh, sw, d_dst, dh, dw):
        """cv2.resize (bilinear) of n uint8 [sh][sw][3] device images into d_dst [n][dh][dw][3]."""
        self._check(self.L.yolo_b200_resize_u8bgr(self._h, _ptr(d_src), n, sh, sw, _ptr(d_dst), dh, dw))

    def calibrate_f32(self, d_nchw, n, h, w):
        """Derive scale_a / retune on the GPU from a float NCHW calibration batch (device tensor) by the reference's
        first-call tracker rule and overflow guard; the context is re-programmed in place.  Returns (scale_a, retune)."""
        nl = self.params.num_layers
        sa = np.zeros(nl + 1, dtype=np.int32)
        rt = np.zeros(nl, dtype=np.int32)
        self._check(self.L.yolo_b200_calibrate_f32(self._h, _ptr(d_nchw), n, h, w, sa.ctypes.data, rt.ctypes.data))
        for l in range(nl):
            self.params.scale_a[l] = int(sa[l]); self.params.retune[l] = int(rt[l])
        self.params.scale_a[nl] = int(sa[nl])
        return sa.tolist(), rt.tolist()

    def update_trackers_f32(self, d_nchw, n, h, w, momentum, tracker_scale):
        """One more calibration batch (slim_yolo_v2.py:25-31): tracker_scale = float32 [num_layers + 1], the `scale`
        buffers of a_tracker_in .. a_tracker_pred, updated in place (zeros = fresh trackers = first-call rule, otherwise the
        exponential average); the context is re-programmed with floor(log2(scale)).  Returns (scale_a, retune)."""
        nl = self.params.num_layers
        ts = np.ascontiguousarray(tracker_scale, dtype=np.float32)
        assert ts.shape == (nl + 1,)
        sa = np.zeros(nl + 1, dtype=np.int32)
        rt = np.zeros(nl, dtype=np.int32)
        self._check(self.L.yolo_b200_update_trackers_f32(self._h, _ptr(d_nchw), n, h, w, C.c_float(momentum), ts.ctypes.data,
                                                         sa.ctypes.data, rt.ctypes.data))
        tracker_scale[...] = ts
        for l in range(nl):
            self.params.scale_a[l] = int(sa[l]); self.params.retune[l] = int(rt[l])
        self.params.scale_a[nl] = int(sa[nl])
        return sa.tolist(), rt.tolist()

    def measure_f32(self, d_nchw, n, h, w):
        """max|a| at every tracker (input, then each layer after its leaky-ReLU) under the tables in force: the quantity the
        reference's find=True branch asserts on (slim_yolo_v2.py:222-226).  Nothing in the context changes."""
        mx = np.zeros(self.params.num_layers + 1, dtype=np.float64)
        self._check(self.L.yolo_b200_measure_f32(self._h, _ptr(d_nchw), n, h, w, mx.ctypes.data))
        return mx

    def quantize_u8bgr(self, d_bgr, n, h, w, d_out):
        self._check(self.L.yolo_b200_quantize_u8bgr(self._h, _ptr(d_bgr), n, h, w, _ptr(d_out)))

    def u8bgr_lut(self) -> np.ndarray:
        lut = np.zeros((3, 256), dtype=np.int8)
        self._check(self.L.yolo_b200_u8bgr_lut(self._h, lut.ctypes.data))
        return lut

    def quantize_rgb444(self, d_frames, n, h, w, d_out):
        self._check(self.L.yolo_b200_quantize_rgb444(self._h, _ptr(d_frames), n, h, w, _ptr(d_out)))

    def quantize_f32(self, d_nchw, n, h, w, d_out):
        self._check(self.L.yolo_b200_quantize_f32(self._h, _ptr(d_nchw), n, h, w, _ptr(d_out)))

    def conv_layer(self, layer, d_in, n, h, w, d_out):
        self._check(self.L.yolo_b200_conv_layer(self._h, layer, _ptr(d_in), n, h, w, _ptr(d_out)))

    def backbone(self, d_in, n, h, w):
        pred = C.c_void_p(); gh = C.c_int(); gw = C.c_int()
        self._check(self.L.yolo_b200_backbone(self._h, _ptr(d_in), n, h, w, C.byref(pred), C.byref(gh), C.byref(gw)))
        return pred.value, gh.value, gw.value

    def detect(self, d_pred, n, gh, gw, in_h, in_w, d_dets, d_counts):
        self._check(self.L.yolo_b200_detect(self._h, _ptr(d_pred), n, gh, gw, in_h, in_w, _ptr(d_dets), _ptr(d_counts)))

    def layer_output(self, layer: int, n: int, oh: int, ow: int) -> np.ndarray:
        cout = self.params.layers[layer].cout
        cs = self.L.yolo_b200_cstride(cout)
        out = np.zeros((n, oh, ow, cs), dtype=np.int8)
        self._check(self.L.yolo_b200_get_layer_output(self._h, layer, out.ctypes.data, out.nbytes))
        return out

    def rgb444_lut(self) -> np.ndarray:
        lut = np.zeros((4096, 4), dtype=np.int8)
        self._check(self.L.yolo_b200_rgb444_lut(self._h, lut.ctypes.data))
        return lut

    def sync(self):
        self._check(self.L.yolo_b200_sync(self._h))

    def overflow_count(self) -> int:
        v = C.c_int64()
        self._check(self.L.yolo_b200_overflow_count(self._h, C.byref(v)))
        return v.value

    def slow_path_count(self) -> int:
        return int(self.L.yolo_b200_slow_path_count(self._h))

    def launch_count(self) -> int:
        return int(self.L.yolo_b200_launch_count(self._h))

    def enable_timing(self, on=True):
        self._check(self.L.yolo_b200_enable_timing(self._h, int(on)))

    def layer_times_ms(self) -> List[float]:
        buf = (C.c_float * 64)()
        n = self.L.yolo_b200_layer_times_ms(self._h, buf, 64)
        if n < 0:
            self._check(n)
        return [buf[i] for i in range(n)]


def dets_to_arrays(dets: np.ndarray, count: int):
    """One frame's structured detections -> (bboxes [N,4] f32, scores [N] f32, cls [N] i64, anchor_index)."""
    d = dets[:count]
    b = np.stack([d["x1"], d["y1"], d["x2"], d["y2"]], axis=1).astype(np.float32) if count else np.zeros((0, 4), np.float32)
    return b, d["score"].astype(np.float32), d["cls"].astype(np.int64), d["anchor_index"].astype(np.int64)
