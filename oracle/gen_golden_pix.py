"""Writes tests/golden/pix_cv2.npz: cv2.cvtColor's own BGR output for seeded frames of the five pixel formats the library
accepts (oracle/pix_u8.py), so the CPU tests can check the oracle where cv2 is not installed.

    python oracle/gen_golden_pix.py

Frames per format at 1x1, 1x7, 7x1, 5x6, 31x47 and 417x333: random bytes (seed = 100 * format + size index), all 0, all
255, and per-channel-distinct (every channel its own constant, so a swapped or dropped channel cannot pass).  The
417x333 cases (large enough for cv2's vector loops and their tails) are stored as the SHA-256 of input and output (the
input is regenerated from its seed), which keeps the file small; the others as arrays.  Also cv2.resize(cvtColor(f)) of
random frames at 480x640 -> 416x416 (digests, seed 1000 + 10 * format) and 7x5 -> 16x16 (arrays), which pins that
conversion and resize commute."""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import pix_u8 as po  # noqa: E402

SIZES = [(1, 1), (1, 7), (7, 1), (5, 6), (31, 47), (417, 333)]
BIG = (417, 333)
RESIZES = [((480, 640), (416, 416)), ((7, 5), (16, 16))]
DISTINCT = (11, 97, 203, 251)            # channel k of a per-channel-distinct frame (gray: the first)


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def frame(fmt, sh, sw, kind, seed):
    shape = po.frame_shape(fmt, sh, sw)
    if kind == "random":
        return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)
    if kind == "zero":
        return np.zeros(shape, np.uint8)
    if kind == "full":
        return np.full(shape, 255, np.uint8)
    f = np.empty(shape, np.uint8)
    if fmt == po.GRAY:
        f[:] = DISTINCT[0]
    elif fmt == po.RGB_PLANAR:
        f[:] = np.array(DISTINCT[:3], np.uint8)[:, None, None]
    else:
        f[:] = np.array(DISTINCT[:shape[2]], np.uint8)
    return f


def cases():
    """(name, fmt, kind, seed, frame) in a fixed order."""
    out = []
    for fmt in po.NAMES:
        for i, (sh, sw) in enumerate(SIZES):
            for kind in ("random", "zero", "full", "distinct"):
                seed = 100 * fmt + i
                out.append(("%s_%dx%d_%s" % (po.NAMES[fmt], sh, sw, kind), fmt, kind, seed, frame(fmt, sh, sw, kind, seed)))
    return out


def resize_cases():
    """(name, fmt, frame, (dh, dw))"""
    out = []
    for fmt in po.NAMES:
        for j, ((sh, sw), dst) in enumerate(RESIZES):
            f = np.random.default_rng(1000 + 10 * fmt + j).integers(0, 256, po.frame_shape(fmt, sh, sw), dtype=np.uint8)
            out.append(("%s_%dx%d_to_%dx%d" % ((po.NAMES[fmt], sh, sw) + dst), fmt, f, dst))
    return out


def main():
    import cv2
    arrays = {"cv2_version": np.array(cv2.__version__)}
    for name, fmt, kind, seed, f in cases():
        out = po.cv2_to_bgr(f, fmt)
        if f.shape[-2:] == BIG or f.shape[:2] == BIG:
            arrays["sha_in_" + name] = np.array(sha(f))
            arrays["sha_out_" + name] = np.array(sha(out))
        else:
            arrays["in_" + name] = f
            arrays["out_" + name] = out
    for name, fmt, f, (dh, dw) in resize_cases():
        out = cv2.resize(po.cv2_to_bgr(f, fmt), (dw, dh))
        if f.size > 4096:
            arrays["sha_rin_" + name] = np.array(sha(f))
            arrays["sha_rout_" + name] = np.array(sha(out))
        else:
            arrays["rin_" + name] = f
            arrays["rout_" + name] = out
    path = os.path.join(HERE, "..", "tests", "golden", "pix_cv2.npz")
    np.savez_compressed(path, **arrays)
    print("wrote %s (%d bytes, cv2 %s)" % (os.path.normpath(path), os.path.getsize(path), cv2.__version__))


if __name__ == "__main__":
    main()
