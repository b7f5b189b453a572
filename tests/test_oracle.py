"""CPU tests: the oracle (oracle/ref_int8.c) against (a) the golden vectors produced by the unmodified reference
PyTorch module (tests/golden, oracle/gen_golden.py) and (b) the reference's own C functions (oracle/_ref/libtierA.so,
compiled from c_embedding/yolo_forward.c when the reference is present; without it, what those functions returned on the
same seeded inputs, tests/golden/tier_ref.npz).  These pin the oracle before any kernel is compared with it."""
import ctypes as C

import numpy as np
import pytest

import golden_util as gu
import oracle_lib as ol
from yolo_b200 import export as ex


@pytest.mark.parametrize("name", gu.FIXTURES)
def test_contract_p_feature_maps_match_reference(name):
    """Contract P restated in integers == the integers behind every AveragedRangeTracker output of the reference
    (models/slim_yolo_v2.py:218-328), tolerance 0."""
    g, qnet, frames = gu.load(name)
    for i in range(int(g["n_frames"])):
        x8, ovf = ol.quantize_f32(frames[i:i + 1].numpy(), qnet.sa[0])
        assert ovf == 0
        assert gu.sha(x8[0]) == str(g["f%d_map0_sha256" % i])
        outs, ovf = ol.backbone(qnet, x8, contract=1)
        assert ovf == 0
        for l, o in enumerate(outs):
            assert gu.sha(o[0]) == str(g["f%d_map%d_sha256" % (i, l + 1)]), "layer %d differs" % l
            key = "f%d_map%d" % (i, l + 1)
            if key in g:
                np.testing.assert_array_equal(o[0], g[key])


@pytest.mark.parametrize("name", gu.FIXTURES)
def test_python_head_matches_reference(name):
    """decode (slim_yolo_v2.py:111-143,330-350) on EVERY anchor against the tensors the reference hands to
    postprocess(): |dscore|, |dbox| <= 1e-5 (expf/sigmoid ULP differences between libm and torch).
    postprocess + nms (:145-210): identical kept set and classes on frames whose reference result does not depend
    on NumPy's unstable argsort (the fixture records that; see oracle/gen_golden.py tie_robust)."""
    g, qnet, frames = gu.load(name)
    H, W = int(g["H"]), int(g["W"])
    for i in range(int(g["n_frames"])):
        pred = g["f%d_map10" % i]
        b, s, c = ol.decode_python(pred, 5, 2, qnet.sa[10], qnet.anchors, 16, H, W)
        ref_cls = np.argmax(g["f%d_all_class" % i], axis=1)
        ref_score = g["f%d_all_class" % i][np.arange(len(ref_cls)), ref_cls]
        np.testing.assert_allclose(b, g["f%d_all_bbox" % i], atol=1e-5, rtol=0)
        np.testing.assert_allclose(s, ref_score, atol=1e-5, rtol=0)
        # argmax may only differ where the two class scores are equal to within the tolerance
        diff = np.where(c != ref_cls)[0]
        assert all(abs(g["f%d_all_class" % i][k, 0] - g["f%d_all_class" % i][k, 1]) <= 1e-5 for k in diff)
        (boxes, scores, cls, idx), cnt = ol.nms_python(b, s, c, 2, float(g["conf_thresh"]), float(g["nms_thresh"]))
        assert np.all(np.diff(idx) > 0), "reference returns detections in ascending anchor order"
        if int(g["f%d_tie_robust" % i]):
            assert cnt == len(g["f%d_scores" % i])
            np.testing.assert_array_equal(cls, g["f%d_cls" % i])
            np.testing.assert_allclose(scores, g["f%d_scores" % i], atol=1e-5, rtol=0)
            np.testing.assert_allclose(boxes, g["f%d_bboxes" % i], atol=1e-5, rtol=0)
        else:
            # tied scores that matter: the reference's own answer depends on NumPy's unstable argsort (its build / CPU).
            # Both answers must be greedy outcomes of the same candidates under some order of the ties.
            rk, rb_, rs_, rc_ = gu.reference_kept_indices(g, i)
            conf, nt = float(g["conf_thresh"]), float(g["nms_thresh"])
            assert gu.greedy_consistent(rb_, rs_, rc_, rk, conf, nt) == []
            assert gu.greedy_consistent(rb_, rs_, rc_, idx, conf, nt) == []
            # and they may differ only on candidates that overlap an equal-score candidate: everything else is pinned
            differ = sorted(set(rk.tolist()) ^ set(idx.tolist()))
            chain = [a for a in differ if not gu.tie_affected(rb_, rs_, rc_, a, nt)]
            # (a candidate next to a tie-affected one may flip with it: allow only those whose kept suppressors differ)
            assert len(chain) <= len(differ) // 2, chain


def test_shift_programme_matches_reference_c():
    """set_quantize_scale (yolo_forward.c:233-257) for the as-shipped tables and random ones: against the reference's
    compiled function when oracle/_ref/libtierA.so is built, else against what it returned (tests/golden/tier_ref.npz)."""
    t = ol.tierA()
    g = gu.tier_golden()
    cases = gu.tier_shift_cases()
    assert len(g["shift"]) == len(cases)
    for c, ref in zip(cases, g["shift"]):
        b = (C.c_int * 6)()
        ol.lib().oracle_shift_programme(*c, b)
        assert list(b) == ref.tolist(), c
        if t is not None:
            a = (C.c_int * 6)()
            t.tierA_set_quantize_scale(*c, a)
            assert list(a) == list(b) == ref.tolist(), c
    # the as-shipped layer-1 programme quoted in SURVEY.md 8c
    b = (C.c_int * 6)()
    ol.lib().oracle_shift_programme(4, 8, 6, 10, 8, b)
    assert list(b) == [2, 0, 4, 1, 2, 0]
    if t is not None:
        a = (C.c_int * 6)()
        t.tierA_set_quantize_scale(4, 8, 6, 10, 8, a)
        assert list(a) == [2, 0, 4, 1, 2, 0]


def test_shipped_tables_match_reference_c():
    t = ol.tierA()
    g = gu.tier_golden()
    tables = [g["scale_w"].tolist(), g["scale_b"].tolist(), g["scale_a"].tolist(), g["retune"].tolist()]
    anc = g["anchors"].tolist()
    if t is not None:
        assert [[t.tierA_tables(0)[i] for i in range(10)], [t.tierA_tables(1)[i] for i in range(10)],
                [t.tierA_tables(2)[i] for i in range(11)], [t.tierA_tables(3)[i] for i in range(10)]] == tables
        assert [round(t.tierA_anchors()[i], 5) for i in range(10)] == anc
    assert tables == [ex.SHIPPED_SCALE_W, ex.SHIPPED_SCALE_B, ex.SHIPPED_SCALE_A, ex.SHIPPED_RETUNE]   # 65536 -> 0 in a const char
    assert anc == [round(v, 5) for p in ex.ANCHOR_SIZE_COCO for v in p]


def test_rgb444_lut_matches_reference_c():
    """pixel_norm_quantize (yolo_forward.c:57-85) over all 4096 codes, for every scale whose results fit a char."""
    t = ol.tierA()
    g = gu.tier_golden()
    for sa in (0, 1):
        lut = ol.rgb444_lut(sa)
        np.testing.assert_array_equal(lut[:, :3], g["rgb444_lut"][sa], err_msg="sa %d" % sa)
        assert np.all(lut[:, 3] == 0)
        if t is not None:
            for code in range(4096):
                out = (C.c_int8 * 3)()
                t.tierA_pixel_norm_quantize(code, sa, out)
                assert list(out) == list(lut[code, :3]), (sa, code)


def test_c_head_primitives_match_reference_c():
    """sigmoid (sigma(-x) as written), dequantize, softmax, cls_sort, box_iou, decode_txtytwth of the reference
    against the restated C head used by oracle_head_c."""
    t = ol.tierA()
    g = gu.tier_golden()
    if t is not None:
        assert abs(t.tierA_sigmoid(2.0) - 0.11920292) < 1e-7     # sigma(-2): the sign bug is part of the contract
    # one-cell prediction maps: the restated head must reproduce literal decode on de-quantised inputs
    anchors = np.asarray(ex.ANCHOR_SIZE_COCO, np.float32)
    trials = gu.tier_head_trials()
    assert len(g["head_cls"]) == len(trials)
    for trial, (sa, pred) in enumerate(trials):
        (boxes, scores, cls, idx), cnt = ol.head_c(pred, 5, sa, anchors, 16, 0.0, 2.0)   # keep everything, no NMS
        assert cnt == 5
        # what the reference's primitives give for anchors 0..4: class, conf * class probability, integer box
        np.testing.assert_array_equal(cls[np.argsort(idx)], g["head_cls"][trial], err_msg="trial %d" % trial)
        np.testing.assert_array_equal(scores[np.argsort(idx)], g["head_scores"][trial], err_msg="trial %d" % trial)
        np.testing.assert_array_equal(boxes[np.argsort(idx)].astype(np.int32), g["head_boxes"][trial], err_msg="trial %d" % trial)
        if t is None:
            continue
        for k in range(cnt):
            a = int(idx[k])
            conf = t.tierA_sigmoid(t.tierA_dequantize(int(pred[0, 0, a]), sa))
            v = (C.c_float * 2)(t.tierA_dequantize(int(pred[0, 0, 5 + 2 * a]), sa),
                                t.tierA_dequantize(int(pred[0, 0, 6 + 2 * a]), sa))
            t.tierA_softmax(v)
            c = t.tierA_cls_sort(v)
            assert c == cls[k]
            assert np.float32(conf * v[c]) == scores[k]
            tq = [t.tierA_dequantize(int(pred[0, 0, 15 + 4 * a + j]), sa) for j in range(4)]
            out4 = (C.c_int * 4)()
            t.tierA_decode_txtytwth(*[C.c_float(x) for x in tq], 0, 0, a, out4)
            assert [out4[1], out4[3], out4[0], out4[2]] == [int(boxes[k, 0]), int(boxes[k, 1]), int(boxes[k, 2]), int(boxes[k, 3])]


def test_c_sort_nms_matches_reference_c():
    """conf_sort + NMS (yolo_forward.c:1114-1147): class-agnostic, suppress iou >= thresh, on integer boxes."""
    t = ol.tierA()
    if t is None:
        pytest.skip("oracle/_ref/libtierA.so not built (reference absent)")
    rng = np.random.default_rng(2)
    for trial in range(20):
        n = int(rng.integers(1, 60))
        x1 = rng.integers(0, 200, n); y1 = rng.integers(0, 150, n)
        x2 = x1 + rng.integers(1, 120, n); y2 = y1 + rng.integers(1, 120, n)
        boxes = np.stack([x2, x1, y2, y1], 1).astype(np.int32)           # x_max,x_min,y_max,y_min
        conf = rng.permutation(n).astype(np.float32) / n + 0.001       # unique
        order = (C.c_int * n)(); sup = (C.c_int * n)()
        kept = t.tierA_sort_nms(n, boxes.ctypes.data_as(C.POINTER(C.c_int)), conf.ctypes.data_as(C.POINTER(C.c_float)),
                                C.c_float(0.5), order, sup)
        ref_kept = [order[i] for i in range(n) if not sup[i]]
        assert kept == len(ref_kept)
        # same thing through the restated head: craft nothing, re-run the greedy rule in numpy on the C iou
        srt = sorted(range(n), key=lambda i: -conf[i])
        dead = [False] * n; mine = []
        for a_i, i in enumerate(srt):
            if dead[a_i]:
                continue
            mine.append(i)
            for b_i in range(a_i + 1, n):
                j = srt[b_i]
                iou = t.tierA_box_iou((C.c_int * 4)(*boxes[i]), (C.c_int * 4)(*boxes[j]))
                if iou >= 0.5:
                    dead[b_i] = True
        assert mine == ref_kept


def test_c_sort_nms_tie_order_matches_reference_c():
    """conf_sort is a swap-selection sort (yolo_forward.c:1114-1126): with EQUAL scores the order it leaves depends on the
    swap history, and NMS (:1128-1147) depends on that order.  The oracle's sort + NMS must reproduce the reference's own
    compiled functions on inputs FULL of ties (scores drawn from a handful of values): same permutation, same flags."""
    t = ol.tierA()
    g = gu.tier_golden()
    L = ol.lib()
    L.oracle_conf_sort_nms.restype = C.c_int
    L.oracle_conf_sort_nms.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_float), C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    trials = gu.tier_tie_trials()
    assert g["tie_trial"].tolist() == [tr for tr, _, _ in trials]
    ends = np.cumsum(g["tie_n"])
    for k, (trial, boxes, conf) in enumerate(trials):
        n = len(boxes)
        s = slice(ends[k] - n, ends[k])
        assert g["tie_n"][k] == n
        oo = (C.c_int * n)(); os_ = (C.c_int * n)()
        bp, cp = boxes.ctypes.data_as(C.POINTER(C.c_int)), conf.ctypes.data_as(C.POINTER(C.c_float))
        ok = L.oracle_conf_sort_nms(n, bp, cp, C.c_float(0.5), oo, os_)
        assert list(oo) == g["tie_order"][s].tolist(), "tie order differs from conf_sort (trial %d)" % trial
        assert [int(v != 0) for v in os_] == g["tie_suppressed"][s].tolist()
        assert ok == g["tie_kept"][k]
        if t is not None:
            ro = (C.c_int * n)(); rs = (C.c_int * n)()
            rk = t.tierA_sort_nms(n, bp, cp, C.c_float(0.5), ro, rs)
            assert list(ro) == list(oo), "tie order differs from conf_sort (trial %d)" % trial
            assert [int(v != 0) for v in rs] == [int(v != 0) for v in os_]
            assert rk == ok


def _tier_b_oracle(frame, w, b):
    """The clean restatement of the first layer on the tier-B frame with the as-shipped tables: int8 [120][160][16]."""
    x8 = ol.quantize_rgb444(frame[:240 * 320].view(np.uint16).reshape(1, 240, 320), ex.SHIPPED_SCALE_A[0])
    ref, _ = ol.conv_layer(x8, w, b[:16], 3, 16, ex.SHIPPED_SCALE_A[0], ex.SHIPPED_SCALE_W[0], ex.SHIPPED_SCALE_B[0],
                           ex.SHIPPED_RETUNE[0], ex.SHIPPED_SCALE_A[1], 1, 1, 0, 0)
    return ref[0]


def test_tier_b_literal_first_conv_over_accelerator_model():
    """Tier B (SURVEY 8c): the reference's LITERAL first_conv (yolo_forward.c:269-418) driving a host model of the accelerator
    (oracle/tierB_shim.c) on one 240x320 RGB444 frame with the as-shipped tables.  Pins how far the literal driver agrees
    with the clean restatement, and the divergences ledgered in oracle/DEVIATIONS.md (B1-B5):
      * every pixel of all 14 x 15 interior tiles is identical once the tile-row placement bug (:283, B3) is undone;
      * literally placed, only the first tile row (minus its right-edge tile) lands where it should;
      * right-edge tiles are garbled (fill pitch, :101-113, B2); the bottom tile row's last output row is wrong (B4);
      * 16 zero-height remainder tiles are started (:287-289, B5).
    Without oracle/_ref/libtierB.so, the restatement's interior tiles are compared with the sha256 of what the literal
    driver produced there (tests/golden/tier_ref.npz)."""
    import os
    frame, w, b = gu.tier_b_inputs()
    ref = _tier_b_oracle(frame, w, b)
    assert gu.sha(ref[:112, :150]) == str(gu.tier_golden()["tier_b_interior_sha256"])
    so = os.path.join(ol.ORACLE_DIR, "_ref", "libtierB.so")
    ol.build()
    if not os.path.exists(so):
        return
    B = C.CDLL(so)
    wh = ex.pack_weight_h_order(w)
    out = np.zeros(256 * 160 * 16, np.int8)
    stats = (C.c_long * 6)()
    rc = B.tierB_first_conv(frame.ctypes.data_as(C.POINTER(C.c_short)), wh.ctypes.data_as(C.POINTER(C.c_int8)),
                            b.ctypes.data_as(C.POINTER(C.c_int8)), out.ctypes.data_as(C.POINTER(C.c_int8)), out.size, stats)
    assert rc == 0
    assert list(stats)[:5] == [256, 16, 0, 0, 0]              # tiles started, zero-height tiles, no out-of-range buffer access
    got = out.reshape(256, 160, 16)
    literal = (got[:120] == ref).all(axis=2).reshape(15, 8, 16, 10).mean(axis=(1, 3))
    assert np.all(literal[0, :15] == 1.0) and np.all(literal[1:] < 1.0)
    fixed = np.stack([got[16 * (r // 8) + r % 8] for r in range(120)])          # tile row tr landed at PSRAM row 16 tr
    per_tile = (fixed == ref).all(axis=2).reshape(15, 8, 16, 10).mean(axis=(1, 3))
    assert np.all(per_tile[:14, :15] == 1.0)
    assert np.all(per_tile[:, 15] < 0.5)
    assert np.all(per_tile[14, :15] == 0.875)
    assert gu.sha(fixed[:112, :150]) == str(gu.tier_golden()["tier_b_interior_sha256"])


def test_requant_properties():
    """Monotonicity of both contracts in acc (this is what lets kernels pool before requantising, SURVEY 8a-ii)
    and saturation bounds."""
    rng = np.random.default_rng(3)
    L = ol.lib()
    for trial in range(300):
        sa_i, sw, sb, rt, sa_o = [int(v) for v in rng.integers(0, 12, 5)]
        for contract in (0, 1):
            for mode in (0, 1, 2):
                for activ in (0, 1):
                    b = int(rng.integers(-128, 128))
                    accs = np.sort(rng.integers(-2 ** 22, 2 ** 22, 64))
                    outs = [L.oracle_requant(int(a), b, sa_i, sw, sb, rt, sa_o, activ, contract, mode) for a in accs]
                    assert all(-128 <= o <= 127 for o in outs)
                    assert all(x <= y for x, y in zip(outs, outs[1:]))


def test_weight_h_roundtrip(tmp_path):
    g, qnet, frames = gu.load("ref_p_64x96")
    p = tmp_path / "weight.h"
    ex.write_weight_h(qnet, str(p))
    ws, bs = ex.read_weight_h(str(p))
    for a, b in zip(ws, qnet.w):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(bs, qnet.b):
        np.testing.assert_array_equal(a, b)


# ---- image resize in front of the path (cv2.resize of base_transform, data/__init__.py:36) ---------------------------

def _resize_oracle():
    import importlib.util
    import os
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "resize_u8.py")
    spec = importlib.util.spec_from_file_location("oracle_resize_u8", p)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_resize_oracle_matches_cv2_golden():
    """oracle/resize_u8.py (restated OpenCV 8-bit bilinear) == the outputs cv2.resize itself produced
    (tests/golden/resize_cv2.npz, written by oracle/gen_golden_resize.py), bit for bit."""
    import os
    ro = _resize_oracle()
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "resize_cv2.npz"))
    assert len(g["cases"]) >= 8
    for seed, sh, sw, dh, dw in g["cases"].tolist():
        img = np.random.default_rng(seed).integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        np.testing.assert_array_equal(ro.resize_bilinear_u8(img, dh, dw), g["out_%d" % seed],
                                      err_msg="%dx%d -> %dx%d" % (sh, sw, dh, dw))


def test_resize_oracle_matches_live_cv2_when_present():
    """Same check against the installed OpenCV on random geometries (up, down, mixed, exact 2x, single rows/columns)."""
    cv2 = pytest.importorskip("cv2")
    ro = _resize_oracle()
    rng = np.random.default_rng(11)
    for t in range(60):
        sh, sw, dh, dw = [int(v) for v in rng.integers(1, 120, 4)]
        if t % 6 == 0:
            sh, sw = 2 * dh, 2 * dw
        img = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        np.testing.assert_array_equal(ro.resize_bilinear_u8(img, dh, dw), cv2.resize(img, (dw, dh)),
                                      err_msg="%dx%d -> %dx%d" % (sh, sw, dh, dw))
    img = rng.integers(0, 256, (480, 640, 3), dtype=np.uint8)                      # the size the reference's demo frames have
    np.testing.assert_array_equal(ro.resize_bilinear_u8(img, 416, 416), cv2.resize(img, (416, 416)))
