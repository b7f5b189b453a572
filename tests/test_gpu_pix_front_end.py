"""Frames in packed RGB, RGBA, BGRA, gray and planar RGB: cv2.cvtColor (COLOR_RGB2BGR / _RGBA2BGR / _BGRA2BGR / _GRAY2BGR,
planar RGB through its HWC transpose) fused in front of the resize front end (yolo_b200_pix_to_bgr_resize,
yolo_b200_forward_pix / _submit_ / _dev, tools/detect.py --pix).

The conversion is checked against oracle/pix_u8.py, which tests/golden/pix_cv2.npz pins to cv2's own output; the resize
against oracle/resize_u8.py; the detections against yolo_b200_forward_u8bgr_resize run on the cvtColor'd frames."""
import hashlib
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
FORMATS = (lib.PIX_RGB, lib.PIX_RGBA, lib.PIX_BGRA, lib.PIX_GRAY, lib.PIX_RGB_PLANAR)
NAMES = {lib.PIX_RGB: "rgb", lib.PIX_RGBA: "rgba", lib.PIX_BGRA: "bgra", lib.PIX_GRAY: "gray", lib.PIX_RGB_PLANAR: "rgb_planar"}


def _oracle(name):
    spec = importlib.util.spec_from_file_location("oracle_" + name, os.path.join(ROOT, "oracle", name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


po = _oracle("pix_u8")
ro = _oracle("resize_u8")


def _frames(rng, fmt, n, sh, sw):
    return rng.integers(0, 256, (n,) + lib.pix_frame_shape(fmt, sh, sw), dtype=np.uint8)


def _to_bgr(frames, fmt):
    """cv2.cvtColor where cv2 imports, the oracle otherwise (the two are equal: test_oracle_matches_live_cv2)."""
    try:
        import cv2  # noqa: F401
    except ImportError:
        return po.to_bgr_batch(frames, fmt)
    return np.stack([po.cv2_to_bgr(f, fmt) for f in frames])


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---- CPU ----------------------------------------------------------------------------------------------------------

def test_oracle_matches_stored_cv2_outputs():
    g = np.load(os.path.join(ROOT, "tests", "golden", "pix_cv2.npz"))
    gen = _oracle("gen_golden_pix")
    cases = gen.cases()
    assert len(cases) == 5 * 6 * 4
    for name, fmt, kind, seed, f in cases:
        if "in_" + name in g.files:
            np.testing.assert_array_equal(g["in_" + name], f, err_msg=name)
            np.testing.assert_array_equal(po.to_bgr(f, fmt), g["out_" + name], err_msg=name)
        else:
            assert str(g["sha_in_" + name]) == _sha(f), name
            assert str(g["sha_out_" + name]) == _sha(po.to_bgr(f, fmt)), name
    # per-channel-distinct frames: each output channel is the constant of the channel cv2 takes it from
    want = {"rgb": (203, 97, 11), "rgba": (203, 97, 11), "bgra": (11, 97, 203), "gray": (11, 11, 11), "rgb_planar": (203, 97, 11)}
    for n, bgr in want.items():
        assert (g["out_%s_5x6_distinct" % n] == np.array(bgr, np.uint8)).all(), n
    # the commutation: resize(cvtColor(f)) = what the kernel computes from the source's own channels
    for name, fmt, f, (dh, dw) in gen.resize_cases():
        got = ro.resize_batch(po.to_bgr(f, fmt)[None], dh, dw)[0]
        if "rin_" + name in g.files:
            np.testing.assert_array_equal(g["rin_" + name], f, err_msg=name)
            np.testing.assert_array_equal(got, g["rout_" + name], err_msg=name)
        else:
            assert str(g["sha_rin_" + name]) == _sha(f) and str(g["sha_rout_" + name]) == _sha(got), name


def test_oracle_matches_live_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(7)
    for fmt in FORMATS:
        for sh, sw in [(1, 1), (1, 7), (7, 1), (3, 1), (5, 6), (31, 47), (417, 333), (480, 640), (1080, 1920)]:
            f = _frames(rng, fmt, 1, sh, sw)[0]
            np.testing.assert_array_equal(po.to_bgr(f, fmt), po.cv2_to_bgr(f, fmt), err_msg="%s %dx%d" % (NAMES[fmt], sh, sw))
        # the commutation claim: resize of the converted frame = the oracle resize (what the kernel computes)
        for (sh, sw), (dh, dw) in [((480, 640), (416, 416)), ((1080, 1920), (416, 416)), ((832, 832), (416, 416)),
                                   ((1, 1), (16, 16)), ((3, 1), (9, 5)), ((1, 7), (8, 8)), ((37, 53), (33, 47))]:
            f = _frames(rng, fmt, 1, sh, sw)[0]
            np.testing.assert_array_equal(ro.resize_batch(po.to_bgr(f, fmt)[None], dh, dw)[0],
                                          cv2.resize(po.cv2_to_bgr(f, fmt), (dw, dh)), err_msg="%s %dx%d" % (NAMES[fmt], sh, sw))
    assert cv2.COLOR_RGB2BGR == po.cv2_code(lib.PIX_RGB_PLANAR)


def test_pix_frame_shape_and_source_size():
    for fmt, shape in [(lib.PIX_RGB, (4, 5, 3)), (lib.PIX_RGBA, (4, 5, 4)), (lib.PIX_BGRA, (4, 5, 4)), (lib.PIX_GRAY, (4, 5)),
                       (lib.PIX_RGB_PLANAR, (3, 4, 5))]:
        assert lib.pix_frame_shape(fmt, 4, 5) == shape
        assert lib.pix_source_size(fmt, shape) == (4, 5)
    assert lib.pix_frame_shape(lib.PIX_GRAY, 1, 1) == (1, 1)
    for fmt, sh, sw in [(5, 4, 4), (-1, 4, 4), (lib.PIX_RGB, 0, 4), (lib.PIX_GRAY, 4, 0)]:
        with pytest.raises(ValueError):
            lib.pix_frame_shape(fmt, sh, sw)
    for fmt, shape in [(5, (4, 4, 3)), (lib.PIX_RGB, (4, 4, 4)), (lib.PIX_RGB, (4, 4)), (lib.PIX_RGBA, (4, 4, 3)),
                       (lib.PIX_GRAY, (4, 4, 1)), (lib.PIX_GRAY, (4,)), (lib.PIX_RGB_PLANAR, (4, 4, 3)), (lib.PIX_RGB_PLANAR, (3, 4)),
                       (lib.PIX_RGB, (0, 4, 3)), (lib.PIX_RGB_PLANAR, (3, 0, 4))]:
        with pytest.raises(ValueError):
            lib.pix_source_size(fmt, shape)


def test_format_codes_match_the_header():
    text = open(os.path.join(ROOT, "include", "yolo_b200.h")).read()
    got = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (YOLO_B200_PIX_\w+)\s+(\d+)", text)}
    assert got == {"YOLO_B200_PIX_RGB": lib.PIX_RGB, "YOLO_B200_PIX_RGBA": lib.PIX_RGBA, "YOLO_B200_PIX_BGRA": lib.PIX_BGRA,
                   "YOLO_B200_PIX_GRAY": lib.PIX_GRAY, "YOLO_B200_PIX_RGB_PLANAR": lib.PIX_RGB_PLANAR}
    assert FORMATS == (0, 1, 2, 3, 4) and (po.RGB, po.RGBA, po.BGRA, po.GRAY, po.RGB_PLANAR) == FORMATS


@pytest.fixture(scope="module")
def L():
    from yolo_b200 import build
    build.build()
    return lib.load_library()


def test_pix_entry_points_fail_without_a_context(L):
    buf = np.zeros(4096, dtype=np.uint8)
    out = np.zeros(4096, dtype=np.int32)
    for fmt in FORMATS:
        assert L.yolo_b200_pix_to_bgr_resize(None, buf.ctypes.data, fmt, 2, 4, 4, buf.ctypes.data, 4, 4) < 0
        assert L.yolo_b200_forward_pix(None, buf.ctypes.data, fmt, 2, 4, 4, 4, 4, out.ctypes.data, out.ctypes.data) < 0
        assert L.yolo_b200_submit_pix(None, buf.ctypes.data, fmt, 2, 4, 4, 4, 4, out.ctypes.data, out.ctypes.data) < 0
        assert L.yolo_b200_forward_pix_dev(None, buf.ctypes.data, fmt, 2, 4, 4, 4, 4, out.ctypes.data, out.ctypes.data) < 0
    assert not buf.any() and not out.any()


def test_pix_frame_bytes(L):
    for fmt in FORMATS:
        assert L.yolo_b200_pix_frame_bytes(fmt, 7, 5) == int(np.prod(lib.pix_frame_shape(fmt, 7, 5)))
        assert L.yolo_b200_pix_frame_bytes(fmt, 1, 1) == int(np.prod(lib.pix_frame_shape(fmt, 1, 1)))
        assert L.yolo_b200_pix_frame_bytes(fmt, 0, 5) == E_ARG and L.yolo_b200_pix_frame_bytes(fmt, 5, -1) == E_ARG
        assert L.yolo_b200_pix_frame_bytes(fmt, 50000, 50000) == E_UNSUPPORTED
    for fmt in (5, -1, 8, 12):
        assert L.yolo_b200_pix_frame_bytes(fmt, 8, 8) == E_ARG, fmt
    # the internal codes of the pixel formats follow the Bayer ones: the YUV entry points never take them
    for fmt in range(3, 13):
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


def _gpu_pix_to_bgr(ctx, frames, fmt, dh, dw, src_mis=0, dst_mis=0):
    """The stage through the C-ABI, source at byte offset src_mis of an exact-size-plus-offset buffer, output at dst_mis into a
    canary-guarded buffer; returns [n][dh][dw][3]."""
    import torch
    n = frames.shape[0]
    sh, sw = lib.pix_source_size(fmt, frames.shape[1:])
    src = torch.zeros(src_mis + frames.size, dtype=torch.uint8, device="cuda")
    src[src_mis:] = _dev(frames.reshape(-1))
    size = n * dh * dw * 3
    buf = torch.full((dst_mis + size + 8,), 0xAB, dtype=torch.uint8, device="cuda")
    out = buf[dst_mis:dst_mis + size]
    _torch_done()
    before = ctx.launch_count()
    ctx.pix_to_bgr_resize(src[src_mis:], fmt, n, sh, sw, out, dh, dw)
    ctx.sync()
    assert ctx.launch_count() == before + 1, "one launch per call"
    assert (buf[dst_mis + size:] == 0xAB).all() and (buf[:dst_mis] == 0xAB).all(), "written outside d_dst"
    return out.cpu().numpy().reshape(n, dh, dw, 3)


# (source, output, n): camera sizes, exact 2x decimation, identity, the smallest frames upscaled, odd sources and outputs
STAGE_GEOMS = [((480, 640), (416, 416), 2), ((1080, 1920), (416, 416), 2), ((832, 832), (416, 416), 2), ((416, 416), (416, 416), 2),
               ((1, 1), (416, 416), 2), ((1, 7), (20, 36), 3), ((7, 1), (30, 9), 3), ((37, 53), (33, 47), 3), ((31, 47), (64, 96), 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FORMATS, ids=[NAMES[f] for f in FORMATS])
def test_pix_stage_matches_the_oracle(ctx, fmt):
    rng = np.random.default_rng(61 + fmt)
    for (sh, sw), (dh, dw), n in STAGE_GEOMS:
        frames = _frames(rng, fmt, n, sh, sw)
        want = ro.resize_batch(po.to_bgr_batch(frames, fmt), dh, dw)
        np.testing.assert_array_equal(_gpu_pix_to_bgr(ctx, frames, fmt, dh, dw), want, err_msg="%dx%d -> %dx%d" % (sh, sw, dh, dw))
    # misaligned sources (the RGBA / BGRA byte loads) and destinations (word stores off), dw % 4 != 0
    frames = _frames(rng, fmt, 3, 37, 53)
    for dh, dw in ((40, 44), (40, 42)):
        want = ro.resize_batch(po.to_bgr_batch(frames, fmt), dh, dw)
        for src_mis, dst_mis in ((0, 0), (1, 0), (2, 1), (3, 2), (0, 3), (3, 0)):
            np.testing.assert_array_equal(_gpu_pix_to_bgr(ctx, frames, fmt, dh, dw, src_mis, dst_mis), want,
                                          err_msg="+%d/+%d -> %dx%d" % (src_mis, dst_mis, dh, dw))
    # cv2's own outputs at identity geometry (cvtColor alone)
    g = np.load(os.path.join(ROOT, "tests", "golden", "pix_cv2.npz"))
    for k in g.files:
        if k.startswith("in_%s_" % NAMES[fmt]) and (fmt != lib.PIX_RGB or not k.startswith("in_rgb_planar")):
            f = g[k][None]
            sh, sw = lib.pix_source_size(fmt, f.shape[1:])
            np.testing.assert_array_equal(_gpu_pix_to_bgr(ctx, f, fmt, sh, sw)[0], g["out_" + k[3:]], err_msg=k)


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


def _check_all_entry_points(ctx, frames, fmt, h, w, want, md):
    import torch
    n = frames.shape[0]
    sh, sw = lib.pix_source_size(fmt, frames.shape[1:])
    for chunk in (64, 3, 1):
        ctx.set_host_chunk(chunk)
        _same_dets(ctx.forward_pix(frames, fmt, (h, w)), want, md)
    ctx.set_host_chunk(3)
    # two submissions in flight: the batch split in two, from pinned memory
    halves = [frames[:(n + 1) // 2], frames[(n + 1) // 2:]] if n > 1 else [frames]
    pinned = [torch.from_numpy(np.ascontiguousarray(p)).pin_memory() for p in halves]
    outs = [(np.zeros((len(p), md), lib.DET_DTYPE), np.zeros(len(p), np.int32)) for p in halves]
    tickets = [ctx.submit_pix(pinned[k], fmt, (h, w), *outs[k]) for k in range(len(halves))]
    for t in tickets:
        ctx.wait(t)
    _same_dets((np.concatenate([o[0] for o in outs]), np.concatenate([o[1] for o in outs])), want, md)
    ctx.set_host_chunk(64)
    d_src = _dev(frames)
    _same_dets(_run_dev(ctx, lambda d, c: ctx.forward_pix_dev(d_src, fmt, n, sh, sw, h, w, d, c), n, md), want, md)


@pytest.mark.gpu
@pytest.mark.parametrize("net", ["p_416", "f_416", "yolo_v2"])
def test_pix_detections_equal_cvtcolor_then_forward(ctx, net):
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
        for fmt in FORMATS:
            for n in ns:
                frames = _frames(rng, fmt, n, *src)
                want = ctx.forward_u8bgr_resize(_to_bgr(frames, fmt), (h, w))
                assert (want[1] > 0).all() and (want[1] <= md).all(), "%s n=%d: every frame must have detections, all kept" % (NAMES[fmt], n)
                _check_all_entry_points(ctx, frames, fmt, h, w, want, md)
    finally:
        ctx.set_host_chunk(64)


@pytest.mark.gpu
def test_pix_call_between_bgr_calls_of_another_geometry(ctx):
    """Table lifetime: a pix call (480x640 -> 416) queued between two BGR calls of another source size on the same context,
    through the device entry points without a synchronise and through two submissions in flight, returns what it returns
    alone, and so do the BGR calls around it."""
    import torch
    md = 4096
    _, qnet, _ = gu.load("ref_p_416x416")                                  # dense detections: the lists are compared in full
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=md)
    h = w = 416
    rng = np.random.default_rng(73)
    bgr_a = rng.integers(0, 256, (5, 300, 400, 3), dtype=np.uint8)
    bgr_b = rng.integers(0, 256, (4, 600, 500, 3), dtype=np.uint8)
    for fmt in FORMATS:
        pix = _frames(rng, fmt, 6, 480, 640)
        want_a = ctx.forward_u8bgr_resize(bgr_a, (h, w))
        want_b = ctx.forward_u8bgr_resize(bgr_b, (h, w))
        want_r = ctx.forward_u8bgr_resize(_to_bgr(pix, fmt), (h, w))
        assert all((wnt[1] > 0).all() for wnt in (want_a, want_b, want_r))
        # device entry points, queued back to back
        d_a, d_b, d_r = _dev(bgr_a), _dev(bgr_b), _dev(pix)
        outs = [(torch.zeros((k, md, 8), dtype=torch.int32, device="cuda"), torch.zeros(k, dtype=torch.int32, device="cuda")) for k in (5, 6, 4)]
        _torch_done()
        ctx.forward_u8bgr_resize_dev(d_a, 5, 300, 400, h, w, *outs[0])
        ctx.forward_pix_dev(d_r, fmt, 6, 480, 640, h, w, *outs[1])
        ctx.forward_u8bgr_resize_dev(d_b, 4, 600, 500, h, w, *outs[2])
        ctx.sync()
        for (dd, dc), want in zip(outs, (want_a, want_r, want_b)):
            n = dc.numel()
            _same_dets((dd.cpu().numpy().view(lib.DET_DTYPE).reshape(n, md), dc.cpu().numpy()), want, md)
        # host submissions: BGR a, pix, then BGR b once a's slot is free
        ctx.set_host_chunk(2)
        try:
            p_a, p_r, p_b = (torch.from_numpy(x).pin_memory() for x in (bgr_a, pix, bgr_b))
            res = [(np.zeros((k, md), lib.DET_DTYPE), np.zeros(k, np.int32)) for k in (5, 6, 4)]
            t_a = ctx.submit_u8bgr_images(p_a.numpy().reshape(-1), np.array([[300, 400]] * 5, np.int32), (h, w), *res[0])
            t_r = ctx.submit_pix(p_r, fmt, (h, w), *res[1])
            ctx.wait(t_a)
            t_b = ctx.submit_u8bgr_images(p_b.numpy().reshape(-1), np.array([[600, 500]] * 4, np.int32), (h, w), *res[2])
            ctx.wait(t_r)
            ctx.wait(t_b)
        finally:
            ctx.set_host_chunk(64)
        for got, want in zip(res, (want_a, want_r, want_b)):
            _same_dets(got, want, md)


@pytest.mark.gpu
def test_pix_errors_and_empty_batch(ctx):
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

    def calls(fmt, n, sh, sw, h=64, w=96, src=True):
        return [L.yolo_b200_pix_to_bgr_resize(hh, d_src.data_ptr() if src else None, fmt, n, sh, sw, d_dst.data_ptr(), h, w),
                L.yolo_b200_forward_pix(hh, h_src.ctypes.data if src else None, fmt, n, sh, sw, h, w, dets.ctypes.data, counts.ctypes.data),
                L.yolo_b200_submit_pix(hh, h_src.ctypes.data if src else None, fmt, n, sh, sw, h, w, dets.ctypes.data, counts.ctypes.data),
                L.yolo_b200_forward_pix_dev(hh, d_src.data_ptr() if src else None, fmt, n, sh, sw, h, w, d_dets.data_ptr(), d_counts.data_ptr())]

    for fmt in FORMATS:
        assert calls(fmt, -1, 8, 8) == [E_ARG] * 4
        assert calls(fmt, 2, 0, 8) == [E_ARG] * 4
        assert calls(fmt, 2, 8, 0) == [E_ARG] * 4
        assert calls(fmt, 2, 8, 8, h=0) == [E_ARG] * 4
        assert calls(fmt, 2, 8, 8, w=0) == [E_ARG] * 4
        assert calls(fmt, 2, 8, 8, src=False) == [E_ARG] * 4
        assert calls(fmt, 2, 50000, 50000) == [E_UNSUPPORTED] * 4         # a frame over 2 GiB
        assert calls(fmt, 0, 8, 8) == [0, 0, E_ARG, 0]                    # n == 0 writes nothing; submit needs n >= 1
    for fmt in (5, -1, 8):
        assert calls(fmt, 2, 8, 8) == [E_ARG] * 4
    assert L.yolo_b200_forward_pix_dev(hh, d_src.data_ptr(), lib.PIX_RGB, 2, 8, 8, 64, 96, None, d_counts.data_ptr()) == E_ARG
    assert L.yolo_b200_forward_pix(hh, h_src.ctypes.data, lib.PIX_RGB, 2, 8, 8, 64, 96, dets.ctypes.data, None) == E_ARG
    ctx.sync()
    assert (d_dst == 7).all() and (d_dets == 7).all() and (d_counts == 7).all()
    assert (dets == 7).all() and (counts == 7).all()
    # a third submission while two are in flight
    for fmt in (lib.PIX_GRAY, lib.PIX_RGBA):
        frames = torch.from_numpy(_frames(np.random.default_rng(83), fmt, 3, 64, 96)).pin_memory()
        outs = [(np.zeros((3, 512), lib.DET_DTYPE), np.zeros(3, np.int32)) for _ in range(2)]
        tickets = [ctx.submit_pix(frames, fmt, (64, 96), *o) for o in outs]
        assert L.yolo_b200_submit_pix(hh, frames.data_ptr(), fmt, 3, 64, 96, 64, 96, dets.ctypes.data, counts.ctypes.data) == E_STATE
        for t in tickets:
            ctx.wait(t)
        _same_dets(outs[1], outs[0], 512)
        assert (dets == 7).all() and (counts == 7).all()
    d, c = ctx.forward_pix(np.zeros((0, 96, 96, 3), np.uint8), lib.PIX_RGB, (64, 96))
    assert d.shape == (0, 512) and c.shape == (0,)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rgb24", "gray"])
def test_detect_cli_on_raw_pix(tmp_path, name):
    """tools/detect.py --pix: 7 raw frames in batches of 3 (two batches in flight, the last one short); the printed counts
    equal the library's counts for the cvtColor'd frames, and detections.avi holds 7 frames at the source size."""
    cv2 = pytest.importorskip("cv2")
    fmt = {"rgb24": lib.PIX_RGB, "gray": lib.PIX_GRAY}[name]
    sh, sw, size = 72, 96, 96
    frames = _frames(np.random.default_rng(89), fmt, 7, sh, sw)
    raw = tmp_path / ("clip." + name)
    frames.tofile(str(raw))
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "detect.py"), "--trained_model", "random", "--pix", str(raw),
                        "--pix_format", name, "--pix_size", "%dx%d" % (sw, sh), "-size", str(size), "--batch", "3", "--out", str(out)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    printed = {int(m.group(1)): int(m.group(2)) for m in re.finditer(r"^frame (\d+): (\d+) detections", r.stdout, re.M)}
    assert sorted(printed) == list(range(7))
    qnet = ex.random_quantnet(seed=0, calib_hw=(size, size), calib_frames=2, head_bias_shift=-3.0)      # detect.py's network
    c = lib.Context(0)
    try:
        c.load_quantnet(qnet, contract=lib.CONTRACT_P, head_mode=lib.HEAD_PYTHON, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
        _, counts = c.forward_u8bgr_resize(_to_bgr(frames, fmt), (size, size))
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
