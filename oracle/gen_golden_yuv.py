"""Writes tests/golden/yuv_cv2.npz: cv2.cvtColor's own BGR output for seeded YUV frames of the three formats the library
accepts (oracle/yuv_u8.py), so the CPU tests can check the oracle where cv2 is not installed.

    python oracle/gen_golden_yuv.py

Frames: random bytes at 2x2, 6x10, 34x66 and 64x96 (seed = case index), plus one 10x50 frame per format whose pixels run
over every combination of Y in {0, 15, 16, 235, 255} and U, V in {0, 1, 127, 128, 255}: both saturation sides and the
Y < 16 clamp."""
import itertools
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import yuv_u8 as yo  # noqa: E402

SIZES = [(2, 2), (6, 10), (34, 66), (64, 96)]
YS, CS = (0, 15, 16, 235, 255), (0, 1, 127, 128, 255)


def random_frame(fmt, sh, sw, seed):
    return np.random.default_rng(seed).integers(0, 256, yo.frame_shape(fmt, sh, sw), dtype=np.uint8)


def extreme_frame(fmt):
    """10 x 50: every (Y, U, V) of YS x CS x CS once; the chroma of a 2x2 (4:2:0) / 1x2 (4:2:2) block is shared, so each
    block carries one (U, V) and its pixels all take that block's Y."""
    combos = list(itertools.product(YS, CS, CS))               # 125
    sh, sw = 10, 50
    Y = np.zeros((sh, sw), np.uint8)
    if fmt == yo.YUYV:
        U = np.zeros((sh, sw // 2), np.uint8); V = np.zeros_like(U)
        for k, (y, u, v) in enumerate(combos):                 # 125 of the 250 pixel pairs, twice
            for r, c in ((k // 25, k % 25), (5 + k // 25, k % 25)):
                Y[r, 2 * c:2 * c + 2] = y; U[r, c] = u; V[r, c] = v
        f = np.zeros((sh, sw, 2), np.uint8)
        f[:, :, 0] = Y
        f[:, 0::2, 1] = U
        f[:, 1::2, 1] = V
        return f
    U = np.zeros((sh // 2, sw // 2), np.uint8); V = np.zeros_like(U)
    for k, (y, u, v) in enumerate(combos):                     # 125 blocks of 2x2
        r, c = k // 25, k % 25
        Y[2 * r:2 * r + 2, 2 * c:2 * c + 2] = y; U[r, c] = u; V[r, c] = v
    if fmt == yo.NV12:
        uv = np.zeros((sh // 2, sw), np.uint8)
        uv[:, 0::2] = U; uv[:, 1::2] = V
        return np.concatenate([Y, uv])
    return np.concatenate([Y, np.concatenate([U.reshape(-1), V.reshape(-1)]).reshape(sh // 2, sw)])


def cases():
    """(name, fmt, frame) in a fixed order."""
    out = []
    for fmt in (yo.NV12, yo.I420, yo.YUYV):
        for i, (sh, sw) in enumerate(SIZES):
            out.append(("%s_%dx%d" % (yo.NAMES[fmt], sh, sw), fmt, random_frame(fmt, sh, sw, 100 * fmt + i)))
        out.append(("%s_extreme" % yo.NAMES[fmt], fmt, extreme_frame(fmt)))
    return out


def main():
    import cv2
    arrays = {"cv2_version": np.array(cv2.__version__)}
    for name, fmt, frame in cases():
        arrays["in_" + name] = frame
        arrays["out_" + name] = cv2.cvtColor(frame, yo.cv2_code(fmt))
    path = os.path.join(HERE, "..", "tests", "golden", "yuv_cv2.npz")
    np.savez_compressed(path, **arrays)
    print("wrote %s (%d bytes, cv2 %s)" % (os.path.normpath(path), os.path.getsize(path), cv2.__version__))


if __name__ == "__main__":
    main()
