"""CPU oracle for the YUV camera / video front end.  TEST INFRASTRUCTURE ONLY (imported by tests/ and
oracle/gen_golden_yuv.py; the product never imports it).

Restates `cv2.cvtColor(frame, code)` for the three codes the library accepts (opencv-python 4.13.0; OpenCV's
modules/imgproc/src/color_yuv.simd.hpp, YUV420sp2RGB8Invoker / YUV420p2RGB8Invoker / YUV422toRGB8Invoker):

  COLOR_YUV2BGR_NV12  frame uint8 [sh*3/2][sw]:  Y plane, then sh/2 rows of interleaved U,V
  COLOR_YUV2BGR_I420  frame uint8 [sh*3/2][sw]:  Y plane, then the U plane (sh/2)x(sw/2), then the V plane
  COLOR_YUV2BGR_YUYV  frame uint8 [sh][sw][2]:   macropixel Y0 U Y1 V

BT.601 limited range in 20-bit fixed point, an arithmetic (floor) shift, nearest chroma (one U,V per 2x2 block for
4:2:0, per horizontal pixel pair for 4:2:2):

  y = max(Y - 16, 0) * 1220542;  u = U - 128;  v = V - 128
  R = sat8((y + 2^19 + 1673527 v) >> 20)
  G = sat8((y + 2^19 - 852492 v - 409993 u) >> 20)
  B = sat8((y + 2^19 + 2116026 u) >> 20)

Pinned: tests/golden/yuv_cv2.npz holds cv2's own outputs (oracle/gen_golden_yuv.py); tests/test_gpu_yuv_front_end.py checks
this restatement against them bit for bit, and against the live cv2 when it is importable.
"""
import numpy as np

NV12, I420, YUYV = 0, 1, 2
NAMES = {NV12: "nv12", I420: "i420", YUYV: "yuyv"}

CY, CUB, CUG, CVG, CVR = 1220542, 2116026, -409993, -852492, 1673527
SHIFT = 20
ROUND = 1 << (SHIFT - 1)


def frame_shape(fmt: int, sh: int, sw: int):
    """The cv2 Mat shape of one frame."""
    return (sh * 3 // 2, sw) if fmt in (NV12, I420) else (sh, sw, 2)


def cv2_code(fmt: int):
    import cv2
    return {NV12: cv2.COLOR_YUV2BGR_NV12, I420: cv2.COLOR_YUV2BGR_I420, YUYV: cv2.COLOR_YUV2BGR_YUYV}[fmt]


def planes(frame: np.ndarray, fmt: int):
    """(Y, U, V) at full resolution [sh][sw] int64, chroma repeated to the pixels that share it."""
    f = np.asarray(frame, dtype=np.uint8)
    if fmt == YUYV:
        y = f[:, :, 0]                               # [x][1] is U for even x, V for odd x
        u = np.repeat(f[:, 0::2, 1], 2, axis=1)
        v = np.repeat(f[:, 1::2, 1], 2, axis=1)
        return y.astype(np.int64), u.astype(np.int64), v.astype(np.int64)
    sh, sw = f.shape[0] * 2 // 3, f.shape[1]
    y = f[:sh]
    c = f[sh:]
    if fmt == NV12:
        u, v = c[:, 0::2], c[:, 1::2]
    else:
        flat = c.reshape(-1)
        q = (sh // 2) * (sw // 2)
        u, v = flat[:q].reshape(sh // 2, sw // 2), flat[q:2 * q].reshape(sh // 2, sw // 2)
    up = lambda a: np.repeat(np.repeat(a, 2, axis=0), 2, axis=1)
    return y.astype(np.int64), up(u).astype(np.int64), up(v).astype(np.int64)


def to_bgr(frame: np.ndarray, fmt: int) -> np.ndarray:
    """One frame -> uint8 BGR [sh][sw][3], equal to cv2.cvtColor(frame, cv2_code(fmt))."""
    Y, U, V = planes(frame, fmt)
    y = np.maximum(Y - 16, 0) * CY + ROUND
    u, v = U - 128, V - 128
    r = (y + CVR * v) >> SHIFT
    g = (y + CVG * v + CUG * u) >> SHIFT
    b = (y + CUB * u) >> SHIFT
    return np.clip(np.stack([b, g, r], axis=-1), 0, 255).astype(np.uint8)


def to_bgr_batch(frames: np.ndarray, fmt: int) -> np.ndarray:
    return np.stack([to_bgr(f, fmt) for f in frames])
