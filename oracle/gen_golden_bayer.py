"""Writes tests/golden/bayer_cv2.npz: cv2.cvtColor's own BGR output for seeded raw Bayer frames of the four patterns the
library accepts (oracle/bayer_u8.py), so the CPU tests can check the oracle where cv2 is not installed.

    python oracle/gen_golden_bayer.py

Frames per pattern: random bytes at 3x3, 3x64, 64x3, 5x6, 7x9 and 31x47 (seed = case index), and 33x41 extreme frames:
all 0, all 255, a checkerboard of 0 and 255, and one of 255 pixels on 0 next to each border and corner."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import bayer_u8 as bo  # noqa: E402

SIZES = [(3, 3), (3, 64), (64, 3), (5, 6), (7, 9), (31, 47)]
XH, XW = 33, 41


def random_frame(sh, sw, seed):
    return np.random.default_rng(seed).integers(0, 256, (sh, sw), dtype=np.uint8)


def extreme_frames():
    """name -> uint8 [XH][XW]"""
    hot = np.zeros((XH, XW), np.uint8)
    for y, x in [(0, 0), (0, 20), (0, XW - 1), (1, 1), (1, XW - 2), (16, 0), (16, 1), (16, XW - 2), (16, XW - 1),
                 (XH - 2, 10), (XH - 1, 30), (XH - 1, 0), (XH - 1, XW - 1), (XH - 2, XW - 2)]:
        hot[y, x] = 255
    return {"zero": np.zeros((XH, XW), np.uint8), "full": np.full((XH, XW), 255, np.uint8),
            "checker": ((np.indices((XH, XW)).sum(0) % 2) * 255).astype(np.uint8), "hot": hot}


def cases():
    """(name, pattern, frame) in a fixed order."""
    out = []
    for pat in (bo.RGGB, bo.BGGR, bo.GRBG, bo.GBRG):
        for i, (sh, sw) in enumerate(SIZES):
            out.append(("%s_%dx%d" % (bo.NAMES[pat], sh, sw), pat, random_frame(sh, sw, 100 * pat + i)))
        for kind, f in extreme_frames().items():
            out.append(("%s_%s" % (bo.NAMES[pat], kind), pat, f))
    return out


def main():
    import cv2
    arrays = {"cv2_version": np.array(cv2.__version__)}
    for name, pat, frame in cases():
        arrays["in_" + name] = frame
        arrays["out_" + name] = cv2.cvtColor(frame, bo.cv2_code(pat))
    path = os.path.join(HERE, "..", "tests", "golden", "bayer_cv2.npz")
    np.savez_compressed(path, **arrays)
    print("wrote %s (%d bytes, cv2 %s)" % (os.path.normpath(path), os.path.getsize(path), cv2.__version__))


if __name__ == "__main__":
    main()
