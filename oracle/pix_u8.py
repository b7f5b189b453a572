"""CPU oracle for the pixel-format front end (packed RGB, RGBA, BGRA, gray, planar RGB).  TEST INFRASTRUCTURE ONLY
(imported by tests/ and oracle/gen_golden_pix.py; the product never imports it).

Restates `cv2.cvtColor(frame, code)` (opencv-python 4.13.0) for the five layouts yolo_b200_forward_pix takes:

  RGB         uint8 [sh][sw][3] R,G,B     COLOR_RGB2BGR    B,G,R = bytes 2,1,0
  RGBA        uint8 [sh][sw][4] R,G,B,A   COLOR_RGBA2BGR   B,G,R = bytes 2,1,0 (alpha dropped, not composited)
  BGRA        uint8 [sh][sw][4] B,G,R,A   COLOR_BGRA2BGR   B,G,R = bytes 0,1,2
  GRAY        uint8 [sh][sw]              COLOR_GRAY2BGR   B = G = R = the byte
  RGB_PLANAR  uint8 [3][sh][sw] planes R,G,B (torch CHW): COLOR_RGB2BGR of the HWC transpose, B,G,R = planes 2,1,0

Every one selects or replicates channels per pixel, and cv2.resize treats the channels alike, so
resize(to_bgr(f)) == to_bgr'(resize(f)) where to_bgr' applies the same selection to the resized source channels.

Pinned: tests/golden/pix_cv2.npz holds cv2's own outputs (oracle/gen_golden_pix.py), including a few cv2.resize(cvtColor(f))
outputs; tests/test_gpu_pix_front_end.py checks this restatement against them bit for bit, and against the live cv2 when
it is importable.
"""
import numpy as np

RGB, RGBA, BGRA, GRAY, RGB_PLANAR = 0, 1, 2, 3, 4       # the library's format codes (YOLO_B200_PIX_*)
NAMES = {RGB: "rgb", RGBA: "rgba", BGRA: "bgra", GRAY: "gray", RGB_PLANAR: "rgb_planar"}


def cv2_code(fmt: int):
    """The cvtColor code of a format (RGB_PLANAR: of its HWC transpose)."""
    import cv2
    return {RGB: cv2.COLOR_RGB2BGR, RGBA: cv2.COLOR_RGBA2BGR, BGRA: cv2.COLOR_BGRA2BGR, GRAY: cv2.COLOR_GRAY2BGR,
            RGB_PLANAR: cv2.COLOR_RGB2BGR}[fmt]


def frame_shape(fmt: int, sh: int, sw: int):
    return {RGB: (sh, sw, 3), RGBA: (sh, sw, 4), BGRA: (sh, sw, 4), GRAY: (sh, sw), RGB_PLANAR: (3, sh, sw)}[fmt]


def to_bgr(frame: np.ndarray, fmt: int) -> np.ndarray:
    """One frame (frame_shape(fmt, sh, sw)) -> uint8 BGR [sh][sw][3]."""
    f = np.asarray(frame, dtype=np.uint8)
    if fmt == RGB or fmt == RGBA:
        out = f[:, :, 2::-1]
    elif fmt == BGRA:
        out = f[:, :, :3]
    elif fmt == GRAY:
        out = np.repeat(f[:, :, None], 3, axis=2)
    elif fmt == RGB_PLANAR:
        out = f[::-1].transpose(1, 2, 0)
    else:
        raise ValueError("unknown pixel format %r" % (fmt,))
    return np.ascontiguousarray(out)


def to_bgr_batch(frames: np.ndarray, fmt: int) -> np.ndarray:
    return np.stack([to_bgr(f, fmt) for f in frames])


def cv2_to_bgr(frame: np.ndarray, fmt: int) -> np.ndarray:
    """cv2.cvtColor's own output for one frame (RGB_PLANAR through the HWC transpose, as a CHW tensor is handed to cv2)."""
    import cv2
    f = np.ascontiguousarray(frame.transpose(1, 2, 0)) if fmt == RGB_PLANAR else frame
    return cv2.cvtColor(f, cv2_code(fmt))
