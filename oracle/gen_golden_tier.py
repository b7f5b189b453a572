"""Writes tests/golden/tier_ref.npz: what the reference's own C functions (c_embedding/yolo_forward.c, compiled into
oracle/_ref/libtierA.so / libtierB.so by oracle/Makefile) return on the seeded inputs of the tier-A / tier-B tests in
tests/test_oracle.py (tests/golden_util.py: tier_*), so that those tests keep their comparison where the reference is absent.

    python oracle/gen_golden_tier.py

Every value stored here is one the tests assert to be EXACTLY equal between the reference's compiled function and the
project's restatement on the same input (shift programme, shipped tables and anchors, RGB444 LUT, C head per anchor,
conf_sort + NMS permutation / flags / count, and the first layer on the interior tiles of the literal tier-B driver).
The values are written from the restatement: the file was recorded from the oracle as it stood when those tests last ran
against the reference's compiled C and passed (project history up to f332109), and neither the oracle nor the inputs have
changed since.  With the reference present, the tests compare its compiled functions with this file as well, so a
regenerated file is checked against the original whenever it is available."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import golden_util as gu  # noqa: E402
import oracle_lib as ol  # noqa: E402
import yolo_b200  # noqa: E402,F401
from yolo_b200 import export as ex  # noqa: E402


def main():
    L = ol.lib()
    out = {}
    shift = []
    for c in gu.tier_shift_cases():
        b = (C.c_int * 6)()
        L.oracle_shift_programme(*c, b)
        shift.append(list(b))
    out["shift"] = np.array(shift, np.int32)
    out["scale_w"], out["scale_b"] = np.array(ex.SHIPPED_SCALE_W, np.int32), np.array(ex.SHIPPED_SCALE_B, np.int32)
    out["scale_a"], out["retune"] = np.array(ex.SHIPPED_SCALE_A, np.int32), np.array(ex.SHIPPED_RETUNE, np.int32)
    out["anchors"] = np.array([round(v, 5) for p in ex.ANCHOR_SIZE_COCO for v in p], np.float64)
    out["rgb444_lut"] = np.stack([ol.rgb444_lut(sa)[:, :3] for sa in (0, 1)])

    anchors = np.asarray(ex.ANCHOR_SIZE_COCO, np.float32)
    hc, hs, hb = [], [], []
    for sa, pred in gu.tier_head_trials():
        (boxes, scores, cls, idx), cnt = ol.head_c(pred, 5, sa, anchors, 16, 0.0, 2.0)
        assert cnt == 5
        o = np.argsort(idx)
        hc.append(cls[o]); hs.append(scores[o]); hb.append(boxes[o].astype(np.int32))
    out["head_cls"], out["head_scores"], out["head_boxes"] = np.array(hc, np.int32), np.array(hs, np.float32), np.array(hb, np.int32)

    L.oracle_conf_sort_nms.restype = C.c_int
    L.oracle_conf_sort_nms.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_float), C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    tt, tn, to, tsup, tk = [], [], [], [], []
    for trial, boxes, conf in gu.tier_tie_trials():
        n = len(boxes)
        oo = (C.c_int * n)(); os_ = (C.c_int * n)()
        k = L.oracle_conf_sort_nms(n, boxes.ctypes.data_as(C.POINTER(C.c_int)), conf.ctypes.data_as(C.POINTER(C.c_float)),
                                   C.c_float(0.5), oo, os_)
        tt.append(trial); tn.append(n); to += list(oo); tsup += [int(v != 0) for v in os_]; tk.append(k)
    out["tie_trial"], out["tie_n"], out["tie_kept"] = np.array(tt, np.int32), np.array(tn, np.int32), np.array(tk, np.int32)
    out["tie_order"], out["tie_suppressed"] = np.array(to, np.int32), np.array(tsup, np.int8)

    frame, w, b = gu.tier_b_inputs()
    x8 = ol.quantize_rgb444(frame[:240 * 320].view(np.uint16).reshape(1, 240, 320), ex.SHIPPED_SCALE_A[0])
    ref, _ = ol.conv_layer(x8, w, b[:16], 3, 16, ex.SHIPPED_SCALE_A[0], ex.SHIPPED_SCALE_W[0], ex.SHIPPED_SCALE_B[0],
                           ex.SHIPPED_RETUNE[0], ex.SHIPPED_SCALE_A[1], 1, 1, 0, 0)
    out["tier_b_interior_sha256"] = np.array(gu.sha(ref[0][:112, :150]))     # 14 x 15 tiles of 8 x 10 pixels

    path = os.path.join(ROOT, "tests", "golden", "tier_ref.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
