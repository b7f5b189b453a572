"""Raw Bayer sensor frames: cv2.cvtColor (COLOR_Bayer{RGGB,BGGR,GRBG,GBRG}2BGR, bilinear demosaic) fused in front of the
resize front end (yolo_b200_bayer_to_bgr_resize, yolo_b200_forward_bayer / _submit_ / _dev, tools/detect.py --bayer).

The demosaic is checked against oracle/bayer_u8.py, which tests/golden/bayer_cv2.npz pins to cv2's own output; the resize
against oracle/resize_u8.py; the detections against yolo_b200_forward_u8bgr_resize run on the cvtColor'd frames."""
import importlib.util
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import golden_util as gu
import yolo_b200  # noqa: F401
from yolo_b200 import export as ex
from yolo_b200 import lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E_ARG, E_STATE, E_UNSUPPORTED = -1, -2, -3
PATTERNS = (lib.BAYER_RGGB, lib.BAYER_BGGR, lib.BAYER_GRBG, lib.BAYER_GBRG)
NAMES = {lib.BAYER_RGGB: "rggb", lib.BAYER_BGGR: "bggr", lib.BAYER_GRBG: "grbg", lib.BAYER_GBRG: "gbrg"}


def _oracle(name):
    spec = importlib.util.spec_from_file_location("oracle_" + name, os.path.join(ROOT, "oracle", name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


bo = _oracle("bayer_u8")


def _frames(rng, n, sh, sw):
    return rng.integers(0, 256, (n, sh, sw), dtype=np.uint8)


def _to_bgr(frames, pattern):
    """cv2.cvtColor where cv2 imports, the oracle otherwise (the two are equal: test_oracle_matches_live_cv2)."""
    try:
        import cv2
    except ImportError:
        return bo.to_bgr_batch(frames, pattern)
    return np.stack([cv2.cvtColor(f, bo.cv2_code(pattern)) for f in frames])


# ---- CPU ----------------------------------------------------------------------------------------------------------

def test_oracle_matches_stored_cv2_outputs():
    g = np.load(os.path.join(ROOT, "tests", "golden", "bayer_cv2.npz"))
    names = [k[3:] for k in g.files if k.startswith("in_")]
    assert len(names) == 40
    for n in NAMES.values():
        for case in ("3x3", "3x64", "64x3", "5x6", "7x9", "31x47", "zero", "full", "checker", "hot"):
            assert "%s_%s" % (n, case) in names
    for name in names:
        pat = {v: k for k, v in NAMES.items()}[name[:4]]
        np.testing.assert_array_equal(bo.to_bgr(g["in_" + name], pat), g["out_" + name], err_msg=name)
    assert (g["out_rggb_full"] == 255).all() and (g["out_rggb_zero"] == 0).all()
    assert (g["out_rggb_checker"] == 0).any() and (g["out_rggb_checker"] == 255).any()


def test_oracle_matches_live_cv2():
    cv2 = pytest.importorskip("cv2")
    # the pattern codes and cv2's legacy names (counted from the second row and column) are one code each
    assert cv2.COLOR_BayerRGGB2BGR == cv2.COLOR_BayerBG2BGR == bo.cv2_code(lib.BAYER_RGGB) == 46
    assert cv2.COLOR_BayerGRBG2BGR == cv2.COLOR_BayerGB2BGR == bo.cv2_code(lib.BAYER_GRBG) == 47
    assert cv2.COLOR_BayerBGGR2BGR == cv2.COLOR_BayerRG2BGR == bo.cv2_code(lib.BAYER_BGGR) == 48
    assert cv2.COLOR_BayerGBRG2BGR == cv2.COLOR_BayerGR2BGR == bo.cv2_code(lib.BAYER_GBRG) == 49
    rng = np.random.default_rng(7)
    sizes = [(3, 3), (3, 64), (64, 3), (5, 6), (7, 9), (31, 47), (417, 333), (480, 640), (1080, 1920), (2, 5), (5, 2), (1, 1)]
    for pat in PATTERNS:
        for sh, sw in sizes:
            frames = [rng.integers(0, 256, (sh, sw), dtype=np.uint8), np.zeros((sh, sw), np.uint8), np.full((sh, sw), 255, np.uint8),
                      ((np.indices((sh, sw)).sum(0) % 2) * 255).astype(np.uint8)]
            for k, f in enumerate(frames):
                np.testing.assert_array_equal(bo.to_bgr(f, pat), cv2.cvtColor(f, bo.cv2_code(pat)), err_msg="%s %dx%d #%d" % (NAMES[pat], sh, sw, k))


def test_bayer_source_size_and_validation():
    assert lib.bayer_source_size(lib.BAYER_RGGB, (480, 640)) == (480, 640)
    assert lib.bayer_source_size(lib.BAYER_GBRG, (3, 3)) == (3, 3)
    for pat, shape in [(4, (8, 8)), (-1, (8, 8)), (lib.BAYER_RGGB, (2, 8)), (lib.BAYER_BGGR, (8, 2)), (lib.BAYER_GRBG, (8, 8, 3)),
                       (lib.BAYER_GRBG, (8,))]:
        with pytest.raises(ValueError):
            lib.bayer_source_size(pat, shape)
    assert (lib.BAYER_RGGB, lib.BAYER_BGGR, lib.BAYER_GRBG, lib.BAYER_GBRG) == (0, 1, 2, 3)


def _header_defines():
    text = open(os.path.join(ROOT, "include", "yolo_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (YOLO_B200_BAYER_\w+)\s+(\d+)", text)}


def test_pattern_codes_match_the_header():
    assert _header_defines() == {"YOLO_B200_BAYER_RGGB": 0, "YOLO_B200_BAYER_BGGR": 1, "YOLO_B200_BAYER_GRBG": 2, "YOLO_B200_BAYER_GBRG": 3}


@pytest.fixture(scope="module")
def L():
    from yolo_b200 import build
    build.build()
    return lib.load_library()


def test_bayer_entry_points_fail_without_a_context(L):
    buf = np.zeros(4096, dtype=np.uint8)
    out = np.zeros(4096, dtype=np.int32)
    for pat in PATTERNS:
        assert L.yolo_b200_bayer_to_bgr_resize(None, buf.ctypes.data, pat, 2, 4, 4, buf.ctypes.data, 4, 4) < 0
        assert L.yolo_b200_forward_bayer(None, buf.ctypes.data, pat, 2, 4, 4, 4, 4, out.ctypes.data, out.ctypes.data) < 0
        assert L.yolo_b200_submit_bayer(None, buf.ctypes.data, pat, 2, 4, 4, 4, 4, out.ctypes.data, out.ctypes.data) < 0
        assert L.yolo_b200_forward_bayer_dev(None, buf.ctypes.data, pat, 2, 4, 4, 4, 4, out.ctypes.data, out.ctypes.data) < 0
    assert not buf.any() and not out.any()


def test_yuv_frame_bytes_refuses_the_bayer_formats(L):
    """The internal source formats of the Bayer patterns follow the YUV ones: a YUV entry point never takes them."""
    for fmt in range(3, 9):
        assert L.yolo_b200_yuv_frame_bytes(fmt, 8, 8) == E_ARG, fmt


# ---- GPU ----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    c = lib.Context(0)
    yield c
    c.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _torch_done():
    """The context runs on its own stream: buffers torch has just filled must be complete before a call reads them."""
    import torch
    torch.cuda.synchronize()


def _gpu_bayer_to_bgr(ctx, frames, pattern, dh, dw, src_mis=0, dst_mis=0):
    """The stage through the C-ABI, source at byte offset src_mis of an exact-size-plus-offset buffer, output at dst_mis into a
    canary-guarded buffer; returns [n][dh][dw][3]."""
    import torch
    n, sh, sw = frames.shape
    src = torch.zeros(src_mis + frames.size, dtype=torch.uint8, device="cuda")
    src[src_mis:] = _dev(frames.reshape(-1))
    size = n * dh * dw * 3
    buf = torch.full((dst_mis + size + 8,), 0xAB, dtype=torch.uint8, device="cuda")
    out = buf[dst_mis:dst_mis + size]
    _torch_done()
    before = ctx.launch_count()
    ctx.bayer_to_bgr_resize(src[src_mis:], pattern, n, sh, sw, out, dh, dw)
    ctx.sync()
    assert ctx.launch_count() == before + 1, "one launch per call"
    assert (buf[dst_mis + size:] == 0xAB).all() and (buf[:dst_mis] == 0xAB).all(), "written outside d_dst"
    return out.cpu().numpy().reshape(n, dh, dw, 3)


# (source, output, n): camera sizes, exact 2x decimation, identity, the smallest frame upscaled, odd sources and outputs
STAGE_GEOMS = [((480, 640), (416, 416), 2), ((1080, 1920), (416, 416), 2), ((832, 832), (416, 416), 2), ((416, 416), (416, 416), 2),
               ((3, 3), (416, 416), 2), ((37, 53), (33, 47), 3), ((3, 64), (17, 30), 4), ((64, 3), (31, 9), 4), ((31, 47), (64, 96), 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", PATTERNS, ids=[NAMES[p] for p in PATTERNS])
def test_bayer_stage_matches_the_oracle(ctx, pattern):
    ro = _oracle("resize_u8")
    rng = np.random.default_rng(61 + pattern)
    for (sh, sw), (dh, dw), n in STAGE_GEOMS:
        frames = _frames(rng, n, sh, sw)
        want = ro.resize_batch(bo.to_bgr_batch(frames, pattern), dh, dw)
        np.testing.assert_array_equal(_gpu_bayer_to_bgr(ctx, frames, pattern, dh, dw), want, err_msg="%dx%d -> %dx%d" % (sh, sw, dh, dw))
    # misaligned source and destination (word stores off, then on with a misaligned source), odd source sizes
    frames = _frames(rng, 3, 37, 53)
    want = ro.resize_batch(bo.to_bgr_batch(frames, pattern), 40, 44)
    for src_mis, dst_mis in ((1, 0), (2, 1), (3, 2), (0, 3), (3, 0)):
        np.testing.assert_array_equal(_gpu_bayer_to_bgr(ctx, frames, pattern, 40, 44, src_mis, dst_mis), want, err_msg="+%d/+%d" % (src_mis, dst_mis))
    # cv2's own outputs at identity geometry (cvtColor alone)
    g = np.load(os.path.join(ROOT, "tests", "golden", "bayer_cv2.npz"))
    for k in g.files:
        if k.startswith("in_" + NAMES[pattern]):
            f = g[k][None]
            np.testing.assert_array_equal(_gpu_bayer_to_bgr(ctx, f, pattern, *f.shape[1:])[0], g["out_" + k[3:]], err_msg=k)


def _same_dets(got, want, md):
    (dg, cg), (dw_, cw) = got, want
    np.testing.assert_array_equal(cg, cw)
    for i in range(len(cw)):
        k = int(min(cw[i], md))
        np.testing.assert_array_equal(dg[i][:k].view(np.int32), dw_[i][:k].view(np.int32), err_msg="frame %d" % i)


def _run_dev(ctx, fn, n, md):
    import torch
    d_dets = torch.zeros((n, md, 8), dtype=torch.int32, device="cuda")
    d_counts = torch.zeros(n, dtype=torch.int32, device="cuda")
    _torch_done()
    fn(d_dets, d_counts)
    ctx.sync()
    return d_dets.cpu().numpy().view(lib.DET_DTYPE).reshape(n, md), d_counts.cpu().numpy()


def _check_all_entry_points(ctx, frames, pattern, h, w, want, md):
    import torch
    n, sh, sw = frames.shape
    for chunk in (64, 3, 1):
        ctx.set_host_chunk(chunk)
        _same_dets(ctx.forward_bayer(frames, pattern, (h, w)), want, md)
    ctx.set_host_chunk(3)
    # two submissions in flight: the batch split in two, from pinned memory
    halves = [frames[:(n + 1) // 2], frames[(n + 1) // 2:]] if n > 1 else [frames]
    pinned = [torch.from_numpy(np.ascontiguousarray(p)).pin_memory() for p in halves]
    outs = [(np.zeros((len(p), md), lib.DET_DTYPE), np.zeros(len(p), np.int32)) for p in halves]
    tickets = [ctx.submit_bayer(pinned[k], pattern, (h, w), *outs[k]) for k in range(len(halves))]
    for t in tickets:
        ctx.wait(t)
    _same_dets((np.concatenate([o[0] for o in outs]), np.concatenate([o[1] for o in outs])), want, md)
    ctx.set_host_chunk(64)
    d_src = _dev(frames)
    _same_dets(_run_dev(ctx, lambda d, c: ctx.forward_bayer_dev(d_src, pattern, n, sh, sw, h, w, d, c), n, md), want, md)


@pytest.mark.gpu
@pytest.mark.parametrize("net", ["p_416", "f_416", "yolo_v2"])
def test_bayer_detections_equal_cvtcolor_then_forward(ctx, net):
    """slim_yolo_v2 416x416: the network of tests/golden/ref_p_416x416.npz, which answers thousands of detections per frame
    on random frames (every list is compared in full); yolo_v2 at 64x96."""
    if net == "yolo_v2":
        qnet = ex.random_quantnet_yolo_v2(seed=0, calib_hw=(64, 96), calib_frames=1)
        h, w, src, ns, conf, md = 64, 96, (96, 128), (7,), 0.02, 512
    else:
        _, qnet, _ = gu.load("ref_p_416x416")
        h, w, src, ns, conf, md = 416, 416, (480, 640), (1, 7, 64), 0.1, 4096
    contract = lib.CONTRACT_F if net.startswith("f_") else lib.CONTRACT_P
    ctx.load_quantnet(qnet, contract=contract, conf_thresh=conf, nms_thresh=0.5, max_det=md)
    rng = np.random.default_rng(71)
    try:
        for pattern in PATTERNS:
            for n in ns:
                frames = _frames(rng, n, *src)
                want = ctx.forward_u8bgr_resize(_to_bgr(frames, pattern), (h, w))
                assert (want[1] > 0).all() and (want[1] <= md).all(), "%s n=%d: every frame must have detections, all kept" % (NAMES[pattern], n)
                _check_all_entry_points(ctx, frames, pattern, h, w, want, md)
    finally:
        ctx.set_host_chunk(64)


@pytest.mark.gpu
def test_bayer_call_between_bgr_calls_of_another_geometry(ctx):
    """Table lifetime: a Bayer call (480x640 -> 416) queued between two BGR calls of another source size on the same
    context, through the device entry points without a synchronise and through two submissions in flight, returns what it
    returns alone, and so do the BGR calls around it."""
    import torch
    md = 4096
    _, qnet, _ = gu.load("ref_p_416x416")                                  # dense detections: the lists are compared in full
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=md)
    h = w = 416
    rng = np.random.default_rng(73)
    bgr_a = rng.integers(0, 256, (5, 300, 400, 3), dtype=np.uint8)
    bgr_b = rng.integers(0, 256, (4, 600, 500, 3), dtype=np.uint8)
    for pattern in PATTERNS:
        raw = _frames(rng, 6, 480, 640)
        want_a = ctx.forward_u8bgr_resize(bgr_a, (h, w))
        want_b = ctx.forward_u8bgr_resize(bgr_b, (h, w))
        want_r = ctx.forward_u8bgr_resize(_to_bgr(raw, pattern), (h, w))
        assert all((wnt[1] > 0).all() for wnt in (want_a, want_b, want_r))
        # device entry points, queued back to back
        d_a, d_b, d_r = _dev(bgr_a), _dev(bgr_b), _dev(raw)
        outs = [(torch.zeros((k, md, 8), dtype=torch.int32, device="cuda"), torch.zeros(k, dtype=torch.int32, device="cuda")) for k in (5, 6, 4)]
        _torch_done()
        ctx.forward_u8bgr_resize_dev(d_a, 5, 300, 400, h, w, *outs[0])
        ctx.forward_bayer_dev(d_r, pattern, 6, 480, 640, h, w, *outs[1])
        ctx.forward_u8bgr_resize_dev(d_b, 4, 600, 500, h, w, *outs[2])
        ctx.sync()
        for (dd, dc), want in zip(outs, (want_a, want_r, want_b)):
            n = dc.numel()
            _same_dets((dd.cpu().numpy().view(lib.DET_DTYPE).reshape(n, md), dc.cpu().numpy()), want, md)
        # host submissions: BGR a, Bayer, then BGR b once a's slot is free
        ctx.set_host_chunk(2)
        try:
            p_a, p_r, p_b = (torch.from_numpy(x).pin_memory() for x in (bgr_a, raw, bgr_b))
            res = [(np.zeros((k, md), lib.DET_DTYPE), np.zeros(k, np.int32)) for k in (5, 6, 4)]
            t_a = ctx.submit_u8bgr_images(p_a.numpy().reshape(-1), np.array([[300, 400]] * 5, np.int32), (h, w), *res[0])
            t_r = ctx.submit_bayer(p_r, pattern, (h, w), *res[1])
            ctx.wait(t_a)
            t_b = ctx.submit_u8bgr_images(p_b.numpy().reshape(-1), np.array([[600, 500]] * 4, np.int32), (h, w), *res[2])
            ctx.wait(t_r)
            ctx.wait(t_b)
        finally:
            ctx.set_host_chunk(64)
        for got, want in zip(res, (want_a, want_r, want_b)):
            _same_dets(got, want, md)


@pytest.mark.gpu
def test_bayer_errors_and_empty_batch(ctx):
    import torch
    g, qnet, _ = gu.load("ref_p_64x96")
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=512)
    L, hh = ctx.L, ctx._h
    d_src = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    d_dst = torch.full((1 << 16,), 7, dtype=torch.uint8, device="cuda")
    h_src = np.zeros(1 << 16, np.uint8)
    dets = np.full(512 * 8 * 2, 7, np.int32)
    counts = np.full(2, 7, np.int32)
    d_dets = torch.full((2, 512, 8), 7, dtype=torch.int32, device="cuda")
    d_counts = torch.full((2,), 7, dtype=torch.int32, device="cuda")
    _torch_done()

    def calls(pat, n, sh, sw, h=64, w=96, src=True):
        return [L.yolo_b200_bayer_to_bgr_resize(hh, d_src.data_ptr() if src else None, pat, n, sh, sw, d_dst.data_ptr(), h, w),
                L.yolo_b200_forward_bayer(hh, h_src.ctypes.data if src else None, pat, n, sh, sw, h, w, dets.ctypes.data, counts.ctypes.data),
                L.yolo_b200_submit_bayer(hh, h_src.ctypes.data if src else None, pat, n, sh, sw, h, w, dets.ctypes.data, counts.ctypes.data),
                L.yolo_b200_forward_bayer_dev(hh, d_src.data_ptr() if src else None, pat, n, sh, sw, h, w, d_dets.data_ptr(), d_counts.data_ptr())]

    for pat in PATTERNS:
        assert calls(pat, -1, 8, 8) == [E_ARG] * 4
        assert calls(pat, 2, 0, 8) == [E_ARG] * 4
        assert calls(pat, 2, 8, 0) == [E_ARG] * 4
        assert calls(pat, 2, 2, 8) == [E_ARG] * 4                         # a side below 3
        assert calls(pat, 2, 8, 2) == [E_ARG] * 4
        assert calls(pat, 2, 8, 8, h=0) == [E_ARG] * 4
        assert calls(pat, 2, 8, 8, w=0) == [E_ARG] * 4
        assert calls(pat, 2, 8, 8, src=False) == [E_ARG] * 4
        assert calls(pat, 2, 50000, 50000) == [E_UNSUPPORTED] * 4         # a frame over 2 GiB
        assert calls(pat, 0, 8, 8) == [0, 0, E_ARG, 0]                    # n == 0 writes nothing; submit needs n >= 1
    for pat in (4, -1, 7):
        assert calls(pat, 2, 8, 8) == [E_ARG] * 4
    assert L.yolo_b200_forward_bayer_dev(hh, d_src.data_ptr(), lib.BAYER_RGGB, 2, 8, 8, 64, 96, None, d_counts.data_ptr()) == E_ARG
    assert L.yolo_b200_forward_bayer(hh, h_src.ctypes.data, lib.BAYER_RGGB, 2, 8, 8, 64, 96, dets.ctypes.data, None) == E_ARG
    ctx.sync()
    assert (d_dst == 7).all() and (d_dets == 7).all() and (d_counts == 7).all()
    assert (dets == 7).all() and (counts == 7).all()
    # odd-sized frames and the 3x3 minimum are valid
    ro = _oracle("resize_u8")
    for sh, sw in ((7, 9), (3, 3), (5, 4)):
        for pat in PATTERNS:
            f = _frames(np.random.default_rng(79 + sh), 2, sh, sw)
            want = ro.resize_batch(bo.to_bgr_batch(f, pat), 16, 16)
            np.testing.assert_array_equal(_gpu_bayer_to_bgr(ctx, f, pat, 16, 16), want, err_msg="%s %dx%d" % (NAMES[pat], sh, sw))
    # a third submission while two are in flight
    frames = torch.from_numpy(_frames(np.random.default_rng(83), 3, 64, 96)).pin_memory()
    outs = [(np.zeros((3, 512), lib.DET_DTYPE), np.zeros(3, np.int32)) for _ in range(2)]
    tickets = [ctx.submit_bayer(frames, lib.BAYER_RGGB, (64, 96), *o) for o in outs]
    assert L.yolo_b200_submit_bayer(hh, frames.data_ptr(), lib.BAYER_RGGB, 3, 64, 96, 64, 96, dets.ctypes.data, counts.ctypes.data) == E_STATE
    for t in tickets:
        ctx.wait(t)
    _same_dets(outs[1], outs[0], 512)
    assert (dets == 7).all() and (counts == 7).all()
    d, c = ctx.forward_bayer(np.zeros((0, 96, 96), np.uint8), lib.BAYER_RGGB, (64, 96))
    assert d.shape == (0, 512) and c.shape == (0,)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rggb", "gbrg"])
def test_detect_cli_on_raw_bayer(tmp_path, name):
    """tools/detect.py --bayer: 7 raw frames in batches of 3 (two batches in flight, the last one short); the printed counts
    equal the library's counts for the cvtColor'd frames, and detections.avi holds 7 frames at the source size."""
    cv2 = pytest.importorskip("cv2")
    pattern = {v: k for k, v in NAMES.items()}[name]
    sh, sw, size = 72, 96, 96
    frames = _frames(np.random.default_rng(89), 7, sh, sw)
    raw = tmp_path / ("clip." + name)
    frames.tofile(str(raw))
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "detect.py"), "--trained_model", "random", "--bayer", str(raw),
                        "--bayer_pattern", name, "--bayer_size", "%dx%d" % (sw, sh), "-size", str(size), "--batch", "3", "--out", str(out)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    printed = {int(m.group(1)): int(m.group(2)) for m in re.finditer(r"^frame (\d+): (\d+) detections", r.stdout, re.M)}
    assert sorted(printed) == list(range(7))
    qnet = ex.random_quantnet(seed=0, calib_hw=(size, size), calib_frames=2, head_bias_shift=-3.0)      # detect.py's network
    c = lib.Context(0)
    try:
        c.load_quantnet(qnet, contract=lib.CONTRACT_P, head_mode=lib.HEAD_PYTHON, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
        _, counts = c.forward_u8bgr_resize(_to_bgr(frames, pattern), (size, size))
    finally:
        c.close()
    assert [printed[k] for k in range(7)] == [min(int(x), 1024) for x in counts]
    cap = cv2.VideoCapture(str(out / "detections.avi"))
    got = []
    while True:
        ok, im = cap.read()
        if not ok:
            break
        got.append(im.shape)
    cap.release()
    assert got == [(sh, sw, 3)] * 7
