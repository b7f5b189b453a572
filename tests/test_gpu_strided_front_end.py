"""Frames at a pitched layout: row pitch, plane offsets and frame stride for every source format (yolo_b200_frames,
yolo_b200_frames_to_bgr_resize, yolo_b200_forward_frames / _submit_ / _dev, lib.frames_layout).

Every pitched result is checked against the family's packed call on the same frames compacted, byte for byte, and the
stage also against the oracles (oracle/resize_u8.py over yuv_u8 / bayer_u8 / pix_u8)."""
import importlib.util
import os
import re
import ctypes as C
import json
import shutil

import numpy as np
import pytest

import golden_util as gu
import yolo_b200  # noqa: F401
from yolo_b200 import lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
E_ARG, E_UNSUPPORTED = -1, -3


def _oracle(name):
    spec = importlib.util.spec_from_file_location("oracle_" + name, os.path.join(ROOT, "oracle", name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


yo, bo, po, ro = _oracle("yuv_u8"), _oracle("bayer_u8"), _oracle("pix_u8"), _oracle("resize_u8")

# (family, format, name) of every source format
FORMATS = [(lib.SRC_BGR, 0, "bgr"), (lib.SRC_PIX, lib.PIX_RGB, "rgb"), (lib.SRC_YUV, lib.YUV_NV12, "nv12"),
           (lib.SRC_YUV, lib.YUV_I420, "i420"), (lib.SRC_YUV, lib.YUV_YUYV, "yuyv"), (lib.SRC_BAYER, lib.BAYER_RGGB, "rggb"),
           (lib.SRC_BAYER, lib.BAYER_BGGR, "bggr"), (lib.SRC_BAYER, lib.BAYER_GRBG, "grbg"), (lib.SRC_BAYER, lib.BAYER_GBRG, "gbrg"),
           (lib.SRC_PIX, lib.PIX_RGBA, "rgba"), (lib.SRC_PIX, lib.PIX_BGRA, "bgra"), (lib.SRC_PIX, lib.PIX_GRAY, "gray"),
           (lib.SRC_PIX, lib.PIX_RGB_PLANAR, "rgb_planar")]
IDS = [f[2] for f in FORMATS]


def frame_shape(family, fmt, sh, sw):
    if family == lib.SRC_BGR:
        return (sh, sw, 3)
    if family == lib.SRC_YUV:
        return lib.yuv_frame_shape(fmt, sh, sw)
    if family == lib.SRC_BAYER:
        return (sh, sw)
    return lib.pix_frame_shape(fmt, sh, sw)


def planes(family, fmt, sh, sw):
    """[(rows, row bytes)] of each plane (the table of include/yolo_b200.h)."""
    if family == lib.SRC_YUV:
        return {lib.YUV_NV12: [(sh, sw), (sh // 2, sw)], lib.YUV_I420: [(sh, sw), (sh // 2, sw // 2), (sh // 2, sw // 2)],
                lib.YUV_YUYV: [(sh, 2 * sw)]}[fmt]
    if family == lib.SRC_BAYER:
        return [(sh, sw)]
    if family == lib.SRC_BGR:
        return [(sh, 3 * sw)]
    return {lib.PIX_RGB: [(sh, 3 * sw)], lib.PIX_RGBA: [(sh, 4 * sw)], lib.PIX_BGRA: [(sh, 4 * sw)], lib.PIX_GRAY: [(sh, sw)],
            lib.PIX_RGB_PLANAR: [(sh, sw)] * 3}[fmt]


def to_bgr(frames, family, fmt):
    if family == lib.SRC_BGR:
        return frames
    if family == lib.SRC_YUV:
        return yo.to_bgr_batch(frames, fmt)
    if family == lib.SRC_BAYER:
        return bo.to_bgr_batch(frames, fmt)
    return po.to_bgr_batch(frames, fmt)


def min_size(family, fmt):
    return (3, 3) if family == lib.SRC_BAYER else (2, 2) if family == lib.SRC_YUV else (1, 1)


def layout(family, fmt, sh, sw, pitch=lambda b: b, lead=0, plane_gap=0, frame_gap=0, chroma_rows=None):
    """A descriptor: planes back to back after `lead` bytes with plane_gap bytes between them, rows pitch(row bytes) apart,
    frame_gap bytes after a frame's last plane; chroma_rows: rows reserved for plane 0 before plane 1 (NVDEC aligns it)."""
    d = lib.Frames()
    d.family, d.format, d.sh, d.sw = family, fmt, sh, sw
    off = lead
    for p, (rows, rb) in enumerate(planes(family, fmt, sh, sw)):
        d.plane_offset[p], d.row_pitch[p] = off, pitch(rb)
        off += (chroma_rows if (p == 0 and chroma_rows) else rows) * pitch(rb) + plane_gap
    d.frame_stride = off + frame_gap
    return d


def lay_out(packed, family, fmt, d, fill, base=0):
    """The frames `packed` [n, *frame_shape] written at layout d into a buffer filled with `fill`, starting base bytes in;
    returns (buffer, span end)."""
    n = packed.shape[0]
    first, end = lib.frames_span(d, n)
    buf = np.full(base + end, fill, np.uint8)
    flat = packed.reshape(n, -1)
    src_off = 0
    for p, (rows, rb) in enumerate(planes(family, fmt, d.sh, d.sw)):
        view = np.lib.stride_tricks.as_strided(buf[base + d.plane_offset[p]:], shape=(n, rows, rb),
                                               strides=(d.frame_stride, d.row_pitch[p], 1), writeable=True)
        view[...] = flat[:, src_off:src_off + rows * rb].reshape(n, rows, rb)
        src_off += rows * rb
    assert src_off == flat.shape[1]
    return buf, end


def align(x, a):
    return (x + a - 1) // a * a


# the layouts of the stage test: (name, keyword arguments of layout(), base offset of the frames pointer)
LAYOUTS = [("packed", {}, 0), ("pitch+1", dict(pitch=lambda b: b + 1), 0), ("pitch+3", dict(pitch=lambda b: b + 3), 1),
           ("pitch+64", dict(pitch=lambda b: b + 64), 0), ("pitch512", dict(pitch=lambda b: align(b, 512)), 0),
           ("plane_gaps", dict(lead=5, plane_gap=7, pitch=lambda b: b + 2), 2), ("frame_gap", dict(frame_gap=131), 3),
           ("pitch4_base1", dict(pitch=lambda b: align(b + 1, 4), frame_gap=12), 1)]


# ---- CPU ----------------------------------------------------------------------------------------------------------

def test_header_codes_and_struct_match_lib():
    text = open(os.path.join(ROOT, "include", "yolo_b200.h")).read()
    got = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (YOLO_B200_SRC_\w+)\s+(\d+)", text)}
    assert got == {"YOLO_B200_SRC_BGR": lib.SRC_BGR, "YOLO_B200_SRC_YUV": lib.SRC_YUV, "YOLO_B200_SRC_BAYER": lib.SRC_BAYER,
                   "YOLO_B200_SRC_PIX": lib.SRC_PIX}
    body = re.search(r"typedef struct yolo_b200_frames \{(.*?)\} yolo_b200_frames;", text, re.S).group(1)
    fields = []
    for m in re.finditer(r"(int32_t|int64_t)\s+([^;]+);", body):
        for name in m.group(2).split(","):
            name = name.strip()
            k = re.match(r"(\w+)(?:\[(\d+)\])?", name)
            fields.append((k.group(1), m.group(1), int(k.group(2) or 1)))
    size, want = 0, []
    for name, ty, count in fields:                     # C layout: natural alignment
        b = 4 if ty == "int32_t" else 8
        size = align(size, b)
        want.append((name, size, b * count))
        size += b * count
    size = align(size, 8)
    assert [(n, getattr(lib.Frames, n).offset, getattr(lib.Frames, n).size) for n, _, _ in want] == want
    assert C.sizeof(lib.Frames) == size == 72


@pytest.fixture(scope="module")
def L():
    from yolo_b200 import build
    build.build()
    return lib.load_library()


def test_packed_layout_span_is_the_packed_frames(L):
    for family, fmt, name in FORMATS:
        for sh, sw in [min_size(family, fmt), (6, 8), (480, 640), (1080, 1920)]:
            d = lib.frames_packed(family, fmt, sh, sw)
            if family == lib.SRC_YUV:
                fb = L.yolo_b200_yuv_frame_bytes(fmt, sh, sw)
            elif family == lib.SRC_PIX:
                fb = L.yolo_b200_pix_frame_bytes(fmt, sh, sw)
            else:
                fb = sh * sw * (3 if family == lib.SRC_BGR else 1)
            assert fb == int(np.prod(frame_shape(family, fmt, sh, sw)))
            assert d.frame_stride == fb, name
            for n in (0, 1, 7):
                assert lib.frames_span(d, n) == (0, n * fb), (name, n)
            # the table of the header, plane by plane, back to back
            off = 0
            for p, (rows, rb) in enumerate(planes(family, fmt, sh, sw)):
                assert (d.plane_offset[p], d.row_pitch[p]) == (off, rb), (name, p)
                off += rows * rb


def _span_rc(L, d, n=2):
    a, b = C.c_int64(), C.c_int64()
    return L.yolo_b200_frames_span(C.byref(d), n, C.byref(a), C.byref(b))


def test_validation_errors(L):
    good = lib.frames_packed(lib.SRC_YUV, lib.YUV_NV12, 8, 8)
    assert _span_rc(L, good) == 0

    def bad(rc, **kw):
        d = lib.Frames.from_buffer_copy(good)
        for k, v in kw.items():
            if isinstance(v, tuple):
                getattr(d, k)[v[0]] = v[1]
            else:
                setattr(d, k, v)
        assert _span_rc(L, d) == rc, kw

    bad(E_ARG, family=4)
    bad(E_ARG, family=-1)
    bad(E_ARG, format=3)
    bad(E_ARG, sh=7)                                   # odd 4:2:0 height
    bad(E_ARG, sw=0)
    bad(E_ARG, frame_stride=-1)
    bad(E_ARG, plane_offset=(1, -8))
    bad(E_ARG, row_pitch=(0, 7))                       # below the 8 bytes of a row
    bad(E_ARG, row_pitch=(1, 7))
    bad(E_UNSUPPORTED, row_pitch=(0, 1 << 31))         # a frame spanning more than 2 GiB
    bad(E_UNSUPPORTED, plane_offset=(1, 1 << 31))
    bad(0, frame_stride=0)                             # overlapping frames are fine: the source is read only
    bad(0, plane_offset=(2, -5), row_pitch=(2, -1))    # NV12 has no plane 2: ignored
    assert L.yolo_b200_frames_span(C.byref(good), -1, C.byref(C.c_int64()), C.byref(C.c_int64())) == E_ARG
    assert L.yolo_b200_frames_span(None, 1, C.byref(C.c_int64()), C.byref(C.c_int64())) == E_ARG
    for family, fmt, sh, sw in [(lib.SRC_BAYER, lib.BAYER_RGGB, 2, 8), (lib.SRC_BAYER, 4, 8, 8), (lib.SRC_PIX, 5, 8, 8),
                                (lib.SRC_YUV, lib.YUV_YUYV, 4, 3), (lib.SRC_BGR, 0, 0, 4), (lib.SRC_PIX, lib.PIX_GRAY, 50000, 50000)]:
        with pytest.raises(lib.YoloB200Error):
            lib.frames_packed(family, fmt, sh, sw)
    # BGR ignores its format
    assert lib.frames_packed(lib.SRC_BGR, 7, 4, 5).frame_stride == 60
    # spans: the lowest plane start, the end of the last frame's farthest row
    d = layout(lib.SRC_YUV, lib.YUV_I420, 4, 8, pitch=lambda b: b + 3, lead=10, plane_gap=4, frame_gap=9)
    last = d.plane_offset[2] + 1 * d.row_pitch[2] + 4
    assert lib.frames_span(d, 3) == (10, 2 * d.frame_stride + last)


def test_entry_points_fail_without_a_context(L):
    buf = np.zeros(4096, dtype=np.uint8)
    out = np.zeros(4096, dtype=np.int32)
    d = lib.frames_packed(lib.SRC_PIX, lib.PIX_GRAY, 4, 4)
    assert L.yolo_b200_frames_to_bgr_resize(None, buf.ctypes.data, C.byref(d), 2, buf.ctypes.data, 4, 4) < 0
    for fn in (L.yolo_b200_forward_frames, L.yolo_b200_submit_frames, L.yolo_b200_forward_frames_dev):
        assert fn(None, buf.ctypes.data, C.byref(d), 2, 4, 4, out.ctypes.data, out.ctypes.data) < 0
    assert not buf.any() and not out.any()


def test_frames_layout_of_views():
    x = np.arange(5 * 20 * 30 * 3, dtype=np.int64).astype(np.uint8).reshape(5, 20, 30, 3)
    d = lib.frames_layout(x[:, 2:9, 4:15], lib.SRC_BGR, 0)             # NHWC crop
    assert (d.sh, d.sw, d.frame_stride, d.row_pitch[0]) == (7, 11, 1800, 90)
    d = lib.frames_layout(x[::2], lib.SRC_PIX, lib.PIX_RGB)           # every other frame
    assert (d.sh, d.sw, d.frame_stride, d.row_pitch[0], d.format) == (20, 30, 3600, 90, lib.PIX_RGB)
    chw = np.zeros((4, 3, 20, 30), np.uint8)
    d = lib.frames_layout(chw[1:3, :, 5:12, 3:20], lib.SRC_PIX, lib.PIX_RGB_PLANAR)   # CHW crop
    assert (d.sh, d.sw, d.frame_stride, list(d.plane_offset), list(d.row_pitch)) == (7, 17, 1800, [0, 600, 1200], [30, 30, 30])
    g = np.zeros((3, 10, 40), np.uint8)
    d = lib.frames_layout(g[:, 1:4, 8:24], lib.SRC_BAYER, lib.BAYER_GBRG)
    assert (d.sh, d.sw, d.frame_stride, d.row_pitch[0]) == (3, 16, 400, 40)
    rgba = np.zeros((2, 6, 9, 4), np.uint8)
    d = lib.frames_layout(rgba[:, :, 1:], lib.SRC_PIX, lib.PIX_BGRA)
    assert (d.sh, d.sw, d.frame_stride, d.row_pitch[0]) == (6, 8, 216, 36)
    yuyv = np.zeros((2, 4, 10, 2), np.uint8)
    assert lib.frames_layout(yuyv[:, :, 2:8], lib.SRC_YUV, lib.YUV_YUYV).row_pitch[0] == 20
    # a broadcast frame (stride 0) is a valid layout
    assert lib.frames_layout(np.broadcast_to(x[:1], (4,) + x.shape[1:]), lib.SRC_BGR, 0).frame_stride == 0
    # the descriptor reproduces the view: laid out from the compacted frames it equals the view's bytes
    v = x[1::2, 3:11, 5:19]
    d = lib.frames_layout(v, lib.SRC_BGR, 0)
    buf, _ = lay_out(np.ascontiguousarray(v), lib.SRC_BGR, 0, d, 0)
    got = np.lib.stride_tricks.as_strided(buf, shape=v.shape, strides=v.strides)
    np.testing.assert_array_equal(got, v)


def test_frames_layout_refusals():
    x = np.zeros((4, 10, 12, 3), np.uint8)
    for v, family, fmt in [(x[:, ::-1], lib.SRC_BGR, 0),                            # negative row stride
                           (x[::-1], lib.SRC_BGR, 0),                               # negative frame stride
                           (x[..., ::-1], lib.SRC_PIX, lib.PIX_RGB),                # channel stride -1
                           (x[:, :, ::2], lib.SRC_BGR, 0),                          # pixels not contiguous in a row
                           (np.zeros((4, 3, 10, 12), np.uint8).transpose(0, 2, 3, 1), lib.SRC_BGR, 0),   # HWC view of CHW
                           (np.zeros((4, 3, 10, 12), np.uint8)[..., ::2], lib.SRC_PIX, lib.PIX_RGB_PLANAR),
                           (np.zeros((4, 10, 12, 4), np.uint8), lib.SRC_BGR, 0),    # 4 channels for BGR
                           (np.zeros((4, 10, 12), np.uint8), lib.SRC_PIX, lib.PIX_RGB),
                           (np.zeros((4, 15, 12), np.uint8), lib.SRC_YUV, lib.YUV_NV12),   # several planes: explicit
                           (np.zeros((4, 10, 12, 3), np.float32), lib.SRC_BGR, 0),
                           (x, 9, 0)]:
        with pytest.raises(ValueError):
            lib.frames_layout(v, family, fmt)


def test_pitched_instantiations_do_not_spill():
    """-Xptxas -v of resize.cu: every pitched (LAYOUT) instantiation runs without spills.  (That the packed and ragged ones
    compile to the same SASS as before pitched layouts existed is checked against a git revision by tools/resize_sass.py.)"""
    if shutil.which("cuobjdump") is None and not os.path.exists("/usr/local/cuda/bin/cuobjdump"):
        pytest.skip("no cuobjdump")
    spec = importlib.util.spec_from_file_location("resize_sass", os.path.join(ROOT, "tools", "resize_sass.py"))
    rs = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rs)
    now = rs.compile_resize(ROOT)
    pitched = [n for n in now if "ELb1EEEv" in n]
    assert len(pitched) >= 30
    assert all(now[n][2] == 0 for n in pitched), [(n, now[n][1:]) for n in pitched if now[n][2]]


# ---- GPU ----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    c = lib.Context(0)
    yield c
    c.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _sync():
    import torch
    torch.cuda.synchronize()


def _packed_stage(ctx, frames, family, fmt, dh, dw):
    import torch
    n = frames.shape[0]
    if family == lib.SRC_YUV:
        sh, sw = lib.yuv_source_size(fmt, frames.shape[1:])
    elif family == lib.SRC_PIX:
        sh, sw = lib.pix_source_size(fmt, frames.shape[1:])
    else:
        sh, sw = frames.shape[1], frames.shape[2]
    src = _dev(frames)
    out = torch.zeros(n * dh * dw * 3, dtype=torch.uint8, device="cuda")
    _sync()
    if family == lib.SRC_BGR:
        ctx.resize_u8bgr(src, n, sh, sw, out, dh, dw)
    elif family == lib.SRC_YUV:
        ctx.yuv_to_bgr_resize(src, fmt, n, sh, sw, out, dh, dw)
    elif family == lib.SRC_BAYER:
        ctx.bayer_to_bgr_resize(src, fmt, n, sh, sw, out, dh, dw)
    else:
        ctx.pix_to_bgr_resize(src, fmt, n, sh, sw, out, dh, dw)
    ctx.sync()
    return out.cpu().numpy().reshape(n, dh, dw, 3)


def _pitched_stage(ctx, buf, base, d, n, dh, dw):
    import torch
    src = _dev(buf)
    out = torch.full((n * dh * dw * 3 + 8,), 0xAB, dtype=torch.uint8, device="cuda")
    _sync()
    before = ctx.launch_count()
    ctx.frames_to_bgr_resize(src.data_ptr() + base, d, n, out, dh, dw)
    ctx.sync()
    assert ctx.launch_count() == before + 1, "one launch per call"
    o = out.cpu().numpy()
    assert (o[n * dh * dw * 3:] == 0xAB).all(), "written past d_dst"
    return o[:n * dh * dw * 3].reshape(n, dh, dw, 3)


def _geoms(family, fmt):
    """(source, output, n): camera sizes, an upscale, exact 2x decimation, the smallest frame upscaled"""
    return [((480, 640), (416, 416), 2), ((1080, 1920), (416, 416), 2), ((38, 54), (64, 96), 3), ((832, 832), (416, 416), 2),
            (min_size(family, fmt), (16, 16), 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("family,fmt,name", FORMATS, ids=IDS)
def test_pitched_stage_equals_packed_stage_and_oracle(ctx, family, fmt, name):
    rng = np.random.default_rng(1000 + 17 * family + fmt)
    for (sh, sw), (dh, dw), n in _geoms(family, fmt):
        frames = rng.integers(0, 256, (n,) + tuple(frame_shape(family, fmt, sh, sw)), dtype=np.uint8)
        want = ro.resize_batch(to_bgr(frames, family, fmt), dh, dw)
        np.testing.assert_array_equal(_packed_stage(ctx, frames, family, fmt, dh, dw), want)
        lays = list(LAYOUTS)
        if family == lib.SRC_YUV and fmt == lib.YUV_NV12:       # NVDEC: pitch aligned to 256, UV at pitch * align16(sh)
            lays.append(("nvdec", dict(pitch=lambda b: align(b, 256), chroma_rows=align(sh, 16)), 0))
        for lname, kw, base in lays:
            d = layout(family, fmt, sh, sw, **kw)
            outs = []
            for fill in (0, 255):                               # padding is never read with weight
                buf, _ = lay_out(frames, family, fmt, d, fill, base)
                outs.append(_pitched_stage(ctx, buf, base, d, n, dh, dw))
            msg = "%s %dx%d -> %dx%d %s" % (name, sh, sw, dh, dw, lname)
            np.testing.assert_array_equal(outs[0], want, err_msg=msg)
            np.testing.assert_array_equal(outs[1], want, err_msg=msg + " (padding 255)")


@pytest.mark.gpu
@pytest.mark.parametrize("family,fmt,name", FORMATS, ids=IDS)
def test_span_ending_at_the_end_of_an_exact_allocation(ctx, family, fmt, name):
    """The frames' span ends exactly where a cudaMalloc of its size ends (yolo_b200_ipc_alloc is a plain cudaMalloc)."""
    import torch
    rng = np.random.default_rng(2000 + 17 * family + fmt)
    sh, sw = (30, 38) if family != lib.SRC_BAYER else (31, 37)
    n, dh, dw = 3, 41, 52
    frames = rng.integers(0, 256, (n,) + tuple(frame_shape(family, fmt, sh, sw)), dtype=np.uint8)
    want = ro.resize_batch(to_bgr(frames, family, fmt), dh, dw)
    for kw in ({}, dict(pitch=lambda b: b + 5, lead=3), dict(pitch=lambda b: align(b, 64), frame_gap=64)):
        d = layout(family, fmt, sh, sw, **kw)
        buf, end = lay_out(frames, family, fmt, d, 0)
        first, _ = lib.frames_span(d, n)
        size = end - first
        ptr, handle = C.c_void_p(), (C.c_char * 64)()
        ctx._check(ctx.L.yolo_b200_ipc_alloc(ctx._h, size, C.byref(ptr), handle))
        try:
            host = np.ascontiguousarray(buf[first:])
            ctx._check(ctx.L.yolo_b200_copy_async(ctx._h, ptr.value, host.ctypes.data, size, None))
            ctx.sync()
            out = torch.zeros(n * dh * dw * 3, dtype=torch.uint8, device="cuda")
            _sync()
            ctx.frames_to_bgr_resize(ptr.value - first, d, n, out, dh, dw)
            ctx.sync()
            np.testing.assert_array_equal(out.cpu().numpy().reshape(n, dh, dw, 3), want, err_msg="%s %s" % (name, kw))
        finally:
            ctx.L.yolo_b200_ipc_close(ctx._h, ptr.value, 0)


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
    _sync()
    fn(d_dets, d_counts)
    ctx.sync()
    return d_dets.cpu().numpy().view(lib.DET_DTYPE).reshape(n, md), d_counts.cpu().numpy()


@pytest.fixture(scope="module")
def net416(ctx):
    md = 4096
    _, qnet, _ = gu.load("ref_p_416x416")              # thousands of detections per random frame: lists compared in full
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=md)
    return md


@pytest.mark.gpu
def test_torch_views_through_frames_layout(ctx, net416):
    import torch
    md, h, w = net416, 416, 416
    g = torch.Generator().manual_seed(5)
    nhwc = torch.randint(0, 256, (6, 300, 420, 3), dtype=torch.uint8, generator=g).cuda()
    chw = torch.randint(0, 256, (6, 3, 300, 420), dtype=torch.uint8, generator=g).cuda()
    gray = torch.randint(0, 256, (6, 300, 420), dtype=torch.uint8, generator=g).cuda()
    cases = [(nhwc[:, 17:257, 33:353], lib.SRC_BGR, 0), (nhwc[::2], lib.SRC_PIX, lib.PIX_RGB),
             (chw[:, :, 10:250, 5:325], lib.SRC_PIX, lib.PIX_RGB_PLANAR), (chw[1::2], lib.SRC_PIX, lib.PIX_RGB_PLANAR),
             (gray[::2, 1:, 1:], lib.SRC_BAYER, lib.BAYER_GRBG)]
    for v, family, fmt in cases:
        d = lib.frames_layout(v, family, fmt)
        n = v.shape[0]
        got = _run_dev(ctx, lambda dd, dc: ctx.forward_frames_dev(v, d, n, h, w, dd, dc), n, md)
        c = v.contiguous()
        sh, sw = d.sh, d.sw
        if family == lib.SRC_BGR:
            want = _run_dev(ctx, lambda dd, dc: ctx.forward_u8bgr_resize_dev(c, n, sh, sw, h, w, dd, dc), n, md)
        elif family == lib.SRC_BAYER:
            want = _run_dev(ctx, lambda dd, dc: ctx.forward_bayer_dev(c, fmt, n, sh, sw, h, w, dd, dc), n, md)
        else:
            want = _run_dev(ctx, lambda dd, dc: ctx.forward_pix_dev(c, fmt, n, sh, sw, h, w, dd, dc), n, md)
        assert (want[1] > 0).all()
        _same_dets(got, want, md)


@pytest.mark.gpu
@pytest.mark.parametrize("family,fmt,name", [FORMATS[i] for i in (0, 2, 5, 9, 12)], ids=[IDS[i] for i in (0, 2, 5, 9, 12)])
def test_host_calls_equal_the_packed_host_call(ctx, net416, family, fmt, name):
    """70 frames in chunks of 64 (a short last chunk), frames with gaps between them and padded rows: the blocking call and
    two submissions in flight give the detections of the family's host call on the compacted frames."""
    import torch
    md, h, w = net416, 416, 416
    sh, sw, n = 240, 320, 70
    rng = np.random.default_rng(3000 + fmt)
    frames = rng.integers(0, 256, (n,) + tuple(frame_shape(family, fmt, sh, sw)), dtype=np.uint8)
    if family == lib.SRC_BGR:
        want = ctx.forward_u8bgr_resize(frames, (h, w))
    elif family == lib.SRC_YUV:
        want = ctx.forward_yuv(frames, fmt, (h, w))
    elif family == lib.SRC_BAYER:
        want = ctx.forward_bayer(frames, fmt, (h, w))
    else:
        want = ctx.forward_pix(frames, fmt, (h, w))
    assert (want[1] > 0).all()
    d = layout(family, fmt, sh, sw, pitch=lambda b: align(b, 512), lead=3, plane_gap=16, frame_gap=1000)
    buf, _ = lay_out(frames, family, fmt, d, 77)
    ctx.set_host_chunk(64)
    _same_dets(ctx.forward_frames(buf, d, n, (h, w)), want, md)
    # two submissions in flight from pinned memory: frames [0, 40) and [40, 70) of the same buffer
    pinned = torch.from_numpy(buf).pin_memory()
    outs = [(np.zeros((k, md), lib.DET_DTYPE), np.zeros(k, np.int32)) for k in (40, 30)]
    t0 = ctx.submit_frames(pinned, d, 40, (h, w), *outs[0])
    t1 = ctx.submit_frames(pinned.data_ptr() + 40 * d.frame_stride, d, 30, (h, w), *outs[1])
    ctx.wait(t0)
    ctx.wait(t1)
    _same_dets((np.concatenate([o[0] for o in outs]), np.concatenate([o[1] for o in outs])), want, md)
    # overlapping frames across chunks of 3: stride 0 (one frame 7 times) and a stride of half a frame's span
    ctx.set_host_chunk(3)
    try:
        one = frames[:1]
        d0 = layout(family, fmt, sh, sw, pitch=lambda b: b + 8)
        buf0, _ = lay_out(one, family, fmt, d0, 0)
        d0.frame_stride = 0
        want1 = ctx.forward_frames(np.ascontiguousarray(one), lib.frames_packed(family, fmt, sh, sw), 1, (h, w))
        assert want1[1][0] > 0
        _same_dets(ctx.forward_frames(buf0, d0, 7, (h, w)), (np.repeat(want1[0], 7, axis=0), np.repeat(want1[1], 7)), md)
        dh_ = layout(family, fmt, sh, sw)
        first, end = lib.frames_span(dh_, 1)
        dh_.frame_stride = (end - first) // 2
        big = np.random.default_rng(7).integers(0, 256, lib.frames_span(dh_, 7)[1], dtype=np.uint8)
        compact = np.stack([np.concatenate([np.lib.stride_tricks.as_strided(big[i * dh_.frame_stride + dh_.plane_offset[p]:],
                                                                             shape=(rows, rb), strides=(dh_.row_pitch[p], 1)).reshape(-1)
                                            for p, (rows, rb) in enumerate(planes(family, fmt, sh, sw))]) for i in range(7)])
        _same_dets(ctx.forward_frames(big, dh_, 7, (h, w)),
                   ctx.forward_frames(compact, lib.frames_packed(family, fmt, sh, sw), 7, (h, w)), md)
    finally:
        ctx.set_host_chunk(64)


@pytest.mark.gpu
def test_errors_write_nothing(ctx, net416):
    import torch
    L, hh = ctx.L, ctx._h
    d_src = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    d_dst = torch.full((1 << 16,), 7, dtype=torch.uint8, device="cuda")
    h_src = np.zeros(1 << 16, np.uint8)
    dets = np.full(4096 * 8 * 2, 7, np.int32)
    counts = np.full(2, 7, np.int32)
    d_dets = torch.full((2, 4096, 8), 7, dtype=torch.int32, device="cuda")
    d_counts = torch.full((2,), 7, dtype=torch.int32, device="cuda")
    _sync()

    def calls(d, n=2):
        p = C.byref(d) if d is not None else None
        return [L.yolo_b200_frames_to_bgr_resize(hh, d_src.data_ptr(), p, n, d_dst.data_ptr(), 64, 96),
                L.yolo_b200_forward_frames(hh, h_src.ctypes.data, p, n, 416, 416, dets.ctypes.data, counts.ctypes.data),
                L.yolo_b200_submit_frames(hh, h_src.ctypes.data, p, n, 416, 416, dets.ctypes.data, counts.ctypes.data),
                L.yolo_b200_forward_frames_dev(hh, d_src.data_ptr(), p, n, 416, 416, d_dets.data_ptr(), d_counts.data_ptr())]

    good = lib.frames_packed(lib.SRC_PIX, lib.PIX_RGBA, 8, 8)
    for kw, rc in [(dict(family=7), E_ARG), (dict(format=9), E_ARG), (dict(sh=0), E_ARG), (dict(frame_stride=-4), E_ARG),
                   (dict(row_pitch=31), E_ARG), (dict(plane_offset=-1), E_ARG), (dict(row_pitch=1 << 31), E_UNSUPPORTED)]:
        d = lib.Frames.from_buffer_copy(good)
        for k, v in kw.items():
            if k in ("row_pitch", "plane_offset"):
                getattr(d, k)[0] = v
            else:
                setattr(d, k, v)
        assert calls(d) == [rc] * 4, kw
    assert calls(None) == [E_ARG] * 4
    assert calls(good, -1) == [E_ARG] * 4
    assert calls(good, 0) == [0, 0, E_ARG, 0]
    ctx.sync()
    assert (d_dst == 7).all() and (d_dets == 7).all() and (d_counts == 7).all()
    assert (dets == 7).all() and (counts == 7).all()
