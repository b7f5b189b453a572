"""Shared helpers for tests that use tests/golden/*.npz (made by oracle/gen_golden.py from the reference)."""
import hashlib
import os

import numpy as np

import yolo_b200  # noqa: F401
from yolo_b200 import export as ex

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIXTURES = ["ref_p_64x96", "ref_p_80x64_sparse", "ref_p_416x416", "ref_p_416x416_sparse", "ref_p_64x96_find"]
_cache = {}


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def basetransform_frame(img_seed, H, W, image_kind="noise"):
    """The frame of SURVEY 8(d) config 2 rebuilt WITHOUT the reference or cv2: BaseTransform([H, W]) of a seeded uint8
    480x640 image (data/__init__.py:30-56) = the resize oracle (bit-exact with cv2.resize, tests/test_oracle.py) followed
    by the float32 normalisation NumPy performs, then BGR -> RGB / CHW (test.py:79-80).  The fixture stores the sha256 of
    the frame the reference actually saw, so any drift fails loudly."""
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("resize_u8", os.path.join(os.path.dirname(GOLDEN), "..", "oracle", "resize_u8.py"))
    ro = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ro)
    img = ex.synthetic_image_u8(img_seed, kind=image_kind)
    x = ro.resize_bilinear_u8(img, H, W).astype(np.float32)
    x /= 255.
    x -= np.array((0.406, 0.456, 0.485), dtype=np.float32)
    x /= np.array((0.225, 0.224, 0.229), dtype=np.float32)
    x = x[:, :, (2, 1, 0)]
    return torch.from_numpy(np.ascontiguousarray(x.transpose(2, 0, 1)))[None]


def load(name):
    """Returns (npz dict, QuantNet rebuilt WITHOUT the reference, float frames [n,3,H,W])."""
    if name in _cache:
        return _cache[name]
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))
    H, W, seed = int(g["H"]), int(g["W"]), int(g["seed"])
    qnet = ex.random_quantnet(seed=seed, calib_hw=(H, W), calib_frames=2, head_bias_shift=float(g["head_bias_shift"]),
                              anchors=g["anchors"].tolist(), head_gain=float(g.get("head_gain", 1.0)), weight_gain=float(g.get("weight_gain", 1.0)))
    if int(g.get("find", 0)) or len(g.get("tracker_scales_ema", [])):
        # the reference's trackers were calibrated in the find branch / moved by un-frozen calls: their exponents are part of
        # the fixture, and the find branch's divisions by 2**k live in the weight / bias exponents (see model.py: _load)
        qnet.sa = g["sa"].tolist(); qnet.sw = g["sw"].tolist(); qnet.sb = g["sb"].tolist()
    assert qnet.sha256() == str(g["net_sha256"]), "rebuilt network differs from the one the reference ran"
    assert qnet.sa == g["sa"].tolist()
    import torch
    if str(g.get("frame_kind", "synthetic")) == "basetransform":
        frames = torch.cat([basetransform_frame(int(s), H, W, str(g.get("image_kind", "noise"))) for s in g["frame_seeds"]])
    else:
        frames = torch.cat([ex.synthetic_frames_f32(1, H, W, seed=int(s)) for s in g["frame_seeds"]])
    for i in range(int(g["n_frames"])):
        assert sha(frames[i:i + 1].numpy()) == str(g["f%d_frame_sha256" % i])
    _cache[name] = (g, qnet, frames)
    return _cache[name]


def tier_golden():
    """tests/golden/tier_ref.npz (oracle/gen_golden_tier.py): what the reference's compiled C functions return on the
    seeded inputs below, for the tier-A / tier-B tests to compare with when oracle/_ref/libtierA.so / libtierB.so are absent."""
    if "tier" not in _cache:
        _cache["tier"] = dict(np.load(os.path.join(GOLDEN, "tier_ref.npz"), allow_pickle=False))
    return _cache["tier"]


def tier_shift_cases():
    """(sa_in, sw, sb, retune, sa_out) of set_quantize_scale: the ten shipped layers, then 200 seeded random ones."""
    rng = np.random.default_rng(0)
    cases = [(ex.SHIPPED_SCALE_A[l], ex.SHIPPED_SCALE_W[l], ex.SHIPPED_SCALE_B[l], ex.SHIPPED_RETUNE[l],
              ex.SHIPPED_SCALE_A[l + 1]) for l in range(10)]
    return cases + [tuple(int(v) for v in rng.integers(0, 17, 5)) for _ in range(200)]


def tier_head_trials():
    """(sa, one-cell int8 prediction map [1][1][48]) for the C head primitives, 200 seeded trials."""
    rng = np.random.default_rng(1)
    out = []
    for _ in range(200):
        sa = int(rng.integers(2, 6))
        pred = np.zeros((1, 1, 48), np.int8)
        pred[0, 0, :35] = rng.integers(-40, 40, 35)
        out.append((sa, pred))
    return out


def tier_tie_trials():
    """(trial, boxes int32 [n][x_max, x_min, y_max, y_min], scores float32 [n]) with scores drawn from a handful of values
    (full of ties) and unique boxes, for conf_sort + NMS."""
    rng = np.random.default_rng(7)
    out = []
    for trial in range(60):
        n = int(rng.integers(2, 200))
        levels = int(rng.integers(1, 8))
        x1 = rng.integers(0, 200, n); y1 = rng.integers(0, 150, n)
        x2 = x1 + rng.integers(1, 120, n); y2 = y1 + rng.integers(1, 120, n)
        boxes = np.stack([x2, x1, y2, y1], 1).astype(np.int32)
        if len({tuple(b) for b in boxes}) != n:           # the shim maps sorted entries back by (score, box): keep boxes unique
            continue
        conf = (rng.integers(0, levels, n).astype(np.float32) + 1) / np.float32(levels + 1)
        out.append((trial, boxes, conf))
    return out


def tier_b_inputs():
    """One 240x320 RGB444 frame (with the slack rows the literal driver reads past its end), 16x3x3x3 int8 weights and
    the 32-entry bias buffer of the first layer."""
    rng = np.random.default_rng(0)
    frame = np.zeros(240 * 320 + 64 * 320, np.int16)
    frame[:240 * 320] = rng.integers(0, 4096, 240 * 320)
    w = rng.integers(-6, 6, (16, 3, 3, 3), dtype=np.int8)
    b = np.zeros(32, np.int8)
    b[:16] = rng.integers(-40, 40, 16)
    return frame, w, b


def reference_kept_indices(g, i):
    """Anchor indices of the detections the reference returned for frame i.  postprocess() returns them in ascending
    anchor order (np.where(keep > 0), slim_yolo_v2.py:205), so they are matched in one ascending pass against the
    per-anchor tensors the reference handed to postprocess()."""
    ab, ac = g["f%d_all_bbox" % i], g["f%d_all_class" % i]
    cls = np.argmax(ac, axis=1)
    sc = ac[np.arange(len(cls)), cls]
    rb, rs, rc = g["f%d_bboxes" % i], g["f%d_scores" % i], g["f%d_cls" % i]
    kept, p = [], 0
    for a in range(len(sc)):
        if p < len(rs) and sc[a] == rs[p] and cls[a] == rc[p] and np.array_equal(ab[a], rb[p]):
            kept.append(a)
            p += 1
    assert p == len(rs), "could not place every reference detection on an anchor"
    return np.asarray(kept, np.int64), ab, sc, cls


def _suppress_matrix(A, B, thresh):
    """slim_yolo_v2.py:159-169 in float32 for every pair (a in A, b in B): NOT (ovr <= thresh)."""
    f = np.float32
    A = np.asarray(A, f).reshape(-1, 4); B = np.asarray(B, f).reshape(-1, 4)
    w = np.maximum(f(1e-28), np.minimum(A[:, None, 2], B[None, :, 2]) - np.maximum(A[:, None, 0], B[None, :, 0]))
    h = np.maximum(f(1e-28), np.minimum(A[:, None, 3], B[None, :, 3]) - np.maximum(A[:, None, 1], B[None, :, 1]))
    inter = w * h
    aa = (A[:, 2] - A[:, 0]) * (A[:, 3] - A[:, 1]); ab = (B[:, 2] - B[:, 0]) * (B[:, 3] - B[:, 1])
    with np.errstate(divide="ignore", invalid="ignore"):
        ovr = inter / (aa[:, None] + ab[None, :] - inter)
    return ~(ovr <= f(thresh))


def greedy_consistent(boxes, scores, cls, kept, conf_thresh, nms_thresh):
    """Is `kept` a per-class greedy NMS outcome of these candidates under SOME order of the tied scores?
    (the reference sorts with NumPy's unstable argsort, slim_yolo_v2.py:154, so with ties its own answer depends on the
    NumPy build).  Checks: every kept box is a candidate; no two kept boxes of a class overlap beyond the threshold
    (whichever came first would have suppressed the other); every dropped candidate is overlapped beyond the threshold by
    a kept box of its class whose score is higher or tied.  Returns a list of violations (empty = consistent)."""
    bad = []
    kept = np.asarray(sorted(set(int(k) for k in kept)), np.int64)
    cand = np.where(scores >= np.float32(conf_thresh))[0]
    if not set(kept.tolist()) <= set(cand.tolist()):
        bad.append("kept box below the confidence threshold")
    for c in sorted(set(cls[cand].tolist())):
        ks = kept[cls[kept] == c]
        ds = np.asarray([a for a in cand if cls[a] == c and a not in set(ks.tolist())], np.int64)
        if len(ks):
            m = _suppress_matrix(boxes[ks], boxes[ks], nms_thresh)
            np.fill_diagonal(m, False)
            for x, y in zip(*np.where(np.triu(m))):
                bad.append("kept %d and %d overlap" % (ks[x], ks[y]))
        if len(ds):
            ok = np.zeros(len(ds), bool)
            if len(ks):
                m = _suppress_matrix(boxes[ks], boxes[ds], nms_thresh) & (scores[ks][:, None] >= scores[ds][None, :])
                ok = m.any(axis=0)
            for a in ds[~ok]:
                bad.append("dropped %d has no kept suppressor" % a)
    return bad


def tie_affected(boxes, scores, cls, a, nms_thresh):
    """Does candidate a overlap (beyond the threshold) another candidate of its class with exactly its score?"""
    bs = np.where((scores == scores[a]) & (cls == cls[a]))[0]
    bs = bs[bs != a]
    return bool(len(bs)) and bool(_suppress_matrix(boxes[bs], boxes[a], nms_thresh).any())
