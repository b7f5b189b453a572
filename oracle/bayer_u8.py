"""CPU oracle for the Bayer raw-sensor front end.  TEST INFRASTRUCTURE ONLY (imported by tests/ and
oracle/gen_golden_bayer.py; the product never imports it).

Restates `cv2.cvtColor(raw, code)` for the four 8-bit Bayer-to-BGR codes with OpenCV's default bilinear demosaic
(opencv-python 4.13.0; OpenCV's modules/imgproc/src/demosaicing.cpp, Bayer2RGB_).  A pattern is named by the sensor's
top-left 2x2, as GenICam and ffmpeg name it; OpenCV's legacy names count from the second row and second column, so each
pattern has two cv2 names for one code:

  RGGB = COLOR_BayerRGGB2BGR = COLOR_BayerBG2BGR        GRBG = COLOR_BayerGRBG2BGR = COLOR_BayerGB2BGR
  BGGR = COLOR_BayerBGGR2BGR = COLOR_BayerRG2BGR        GBRG = COLOR_BayerGBRG2BGR = COLOR_BayerGR2BGR

At an interior site (1 <= y <= sh-2, 1 <= x <= sw-2), N/S/W/E its 4-neighbours and NW/NE/SW/SE its diagonals:
  own colour = the raw byte
  R or B site: G = (N+S+W+E+2) >> 2, the opposite colour = (NW+NE+SW+SE+2) >> 2
  G site:      the colour of its horizontal neighbours = (W+E+1) >> 1, that of its vertical neighbours = (N+S+1) >> 1
Borders: cv2 copies column 1 into column 0 and column sw-2 into sw-1, then row 1 into row 0 and row sh-2 into sh-1, so
BGR(y, x) = interior(clamp(y, 1, sh-2), clamp(x, 1, sw-2)).  A frame with a side below 3 comes back all zeros.

Pinned: tests/golden/bayer_cv2.npz holds cv2's own outputs (oracle/gen_golden_bayer.py); tests/test_gpu_bayer_front_end.py
checks this restatement against them bit for bit, and against the live cv2 when it is importable.
"""
import numpy as np

RGGB, BGGR, GRBG, GBRG = 0, 1, 2, 3            # the library's pattern codes (YOLO_B200_BAYER_*)
NAMES = {RGGB: "rggb", BGGR: "bggr", GRBG: "grbg", GBRG: "gbrg"}
CH = {"B": 0, "G": 1, "R": 2}


def cv2_code(pattern: int):
    import cv2
    return {RGGB: cv2.COLOR_BayerRGGB2BGR, BGGR: cv2.COLOR_BayerBGGR2BGR, GRBG: cv2.COLOR_BayerGRBG2BGR,
            GBRG: cv2.COLOR_BayerGBRG2BGR}[pattern]


def site_colours(sh: int, sw: int, pattern: int) -> np.ndarray:
    """int [sh][sw]: the colour channel (0 B, 1 G, 2 R) each sensor site samples."""
    m = np.empty((sh, sw), np.int64)
    name = NAMES[pattern].upper()
    for dy in range(2):
        for dx in range(2):
            m[dy::2, dx::2] = CH[name[2 * dy + dx]]
    return m


def to_bgr(raw: np.ndarray, pattern: int) -> np.ndarray:
    """One frame uint8 [sh][sw] -> uint8 BGR [sh][sw][3], equal to cv2.cvtColor(raw, cv2_code(pattern))."""
    r = np.asarray(raw, dtype=np.uint8).astype(np.int64)
    sh, sw = r.shape
    out = np.zeros((sh, sw, 3), np.int64)
    if sh < 3 or sw < 3:
        return out.astype(np.uint8)
    m = site_colours(sh, sw, pattern)
    c, C = m[1:-1, 1:-1], r[1:-1, 1:-1]
    N, S, W, E = r[:-2, 1:-1], r[2:, 1:-1], r[1:-1, :-2], r[1:-1, 2:]
    NW, NE, SW, SE = r[:-2, :-2], r[:-2, 2:], r[2:, :-2], r[2:, 2:]
    horiz = m[1:-1, :-2]                         # the colour of a site's horizontal neighbours
    cross, diag = (N + S + W + E + 2) >> 2, (NW + NE + SW + SE + 2) >> 2
    hv, vv = (W + E + 1) >> 1, (N + S + 1) >> 1
    g_site = c == 1
    for k in range(3):
        other = np.where(g_site, np.where(horiz == k, hv, vv), cross if k == 1 else diag)
        out[1:-1, 1:-1, k] = np.where(c == k, C, other)
    out[:, 0] = out[:, 1]
    out[:, -1] = out[:, -2]
    out[0] = out[1]
    out[-1] = out[-2]
    return out.astype(np.uint8)


def to_bgr_batch(frames: np.ndarray, pattern: int) -> np.ndarray:
    return np.stack([to_bgr(f, pattern) for f in frames])
