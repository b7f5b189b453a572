"""Images of different sizes in one call: the ragged form of the resize front end (yolo_b200_resize_u8bgr_ragged,
yolo_b200_forward_u8bgr_ragged / _submit_ / _dev, lib.pack_images, tools/detect.py image mode).

Every image is resized bit-exactly as cv2.resize does (oracle/resize_u8.py, tests/golden/resize_cv2.npz), and the
detections equal the reference's order of operations: resize each image on the host, then run it at network size."""
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


def _oracle(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location("oracle_" + name, os.path.join(ROOT, "oracle", name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _resize_oracle():
    return _oracle("resize_u8")


def _images(rng, shapes):
    return [rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8) for sh, sw in shapes]


# ---- CPU: packing and the no-context error path ------------------------------------------------------------------

@pytest.fixture(scope="module")
def L():
    from yolo_b200 import build
    build.build()
    return lib.load_library()


def test_ragged_entry_points_fail_without_a_context(L):
    buf = np.zeros(64, dtype=np.uint8)
    hw = np.array([[2, 3], [4, 1]], dtype=np.int32)
    out = np.zeros(64, dtype=np.int32)
    assert L.yolo_b200_resize_u8bgr_ragged(None, buf.ctypes.data, 2, hw.ctypes.data, buf.ctypes.data, 4, 4) < 0
    assert L.yolo_b200_forward_u8bgr_ragged(None, buf.ctypes.data, 2, hw.ctypes.data, 4, 4, out.ctypes.data, out.ctypes.data) < 0
    assert L.yolo_b200_submit_u8bgr_ragged(None, buf.ctypes.data, 2, hw.ctypes.data, 4, 4, out.ctypes.data, out.ctypes.data) < 0
    assert L.yolo_b200_forward_u8bgr_ragged_dev(None, buf.ctypes.data, 2, hw.ctypes.data, 4, 4, out.ctypes.data, out.ctypes.data) < 0
    assert not buf.any() and not out.any()


def test_pack_images_roundtrip_and_validation():
    rng = np.random.default_rng(0)
    shapes = [(3, 5), (1, 1), (7, 2), (4, 4)]
    imgs = _images(rng, shapes)
    flat, hw = lib.pack_images(imgs)
    assert flat.dtype == np.uint8 and hw.dtype == np.int32 and hw.tolist() == [list(s) for s in shapes]
    off = np.concatenate([[0], np.cumsum([3 * h * w for h, w in shapes])])
    assert flat.size == off[-1]
    for i, im in enumerate(imgs):
        np.testing.assert_array_equal(flat[off[i]:off[i + 1]].reshape(im.shape), im)
    flat0, hw0 = lib.pack_images([])
    assert flat0.size == 0 and hw0.shape == (0, 2)
    for bad in (np.zeros((4, 4, 3), np.float32), np.zeros((4, 4), np.uint8), np.zeros((4, 4, 4), np.uint8),
                np.zeros((4, 6, 3), np.uint8)[:, ::2], [[1, 2, 3]]):
        with pytest.raises(ValueError):
            lib.pack_images([imgs[0], bad])


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


def _gpu_resize_ragged(ctx, imgs, dh, dw, misalign=0):
    """Ragged resize through the C-ABI into a canary-guarded device buffer; returns [n][dh][dw][3]."""
    import torch
    flat, hw = lib.pack_images(imgs)
    n = len(imgs)
    size = n * dh * dw * 3
    buf = torch.full((size + 8,), 0xAB, dtype=torch.uint8, device="cuda")
    out = buf[misalign:misalign + size]
    d_flat = _dev(flat)
    _torch_done()
    before = ctx.launch_count()
    ctx.resize_u8bgr_ragged(d_flat, hw, out, dh, dw)
    ctx.sync()
    assert ctx.launch_count() == before + 1, "one launch per call whatever the number of sizes"
    assert int(buf[misalign + size]) == 0xAB, "written past the end of d_dst"
    return out.cpu().numpy().reshape(n, dh, dw, 3)


@pytest.mark.gpu
def test_ragged_resize_matches_the_oracle_frame_by_frame(ctx):
    ro = _resize_oracle()
    rng = np.random.default_rng(31)
    shapes = [(60, 80), (20, 30), (40, 44), (80, 88), (80, 37), (40, 88), (1, 1), (1, 23), (17, 1),
              (13, 7), (1, 3), (1, 2), (9, 5), (11, 3), (7, 9), (300, 401), (1, 1)]         # ... a 1x1 image last, after a large one
    off = np.cumsum([0] + [3 * h * w for h, w in shapes])[:-1]
    assert set((off % 4).tolist()) == {0, 1, 2, 3}, "images must start at every residue mod 4"
    imgs = _images(rng, shapes)
    for dh, dw, mis in ((40, 44, 0), (33, 47, 1), (40, 44, 2)):          # word stores; dw % 4 != 0; misaligned d_dst
        got = _gpu_resize_ragged(ctx, imgs, dh, dw, misalign=mis)
        for i, im in enumerate(imgs):
            np.testing.assert_array_equal(got[i], ro.resize_bilinear_u8(im, dh, dw), err_msg="image %d %s -> %dx%d (+%d)" % (i, im.shape, dh, dw, mis))
    one = _images(rng, [(37, 53)])
    np.testing.assert_array_equal(_gpu_resize_ragged(ctx, one, 40, 44)[0], ro.resize_bilinear_u8(one[0], 40, 44))
    # cv2's own outputs, one ragged batch per destination size
    g = np.load(os.path.join(ROOT, "tests", "golden", "resize_cv2.npz"))
    groups = {}
    for seed, sh, sw, dh, dw in g["cases"].tolist():
        groups.setdefault((dh, dw), []).append((seed, np.random.default_rng(seed).integers(0, 256, (1, sh, sw, 3), dtype=np.uint8)[0]))
    for (dh, dw), group in groups.items():
        got = _gpu_resize_ragged(ctx, [im for _, im in group], dh, dw)
        for k, (seed, _) in enumerate(group):
            np.testing.assert_array_equal(got[k], g["out_%d" % seed], err_msg="golden seed %d -> %dx%d" % (seed, dh, dw))
    # one source size: the ragged entry point equals the uniform one
    import torch
    same = _images(rng, [(48, 64)] * 5)
    got = _gpu_resize_ragged(ctx, same, 40, 44)
    uni = torch.zeros((5, 40, 44, 3), dtype=torch.uint8, device="cuda")
    d_same = _dev(np.stack(same))
    _torch_done()
    ctx.resize_u8bgr(d_same, 5, 48, 64, uni, 40, 44)
    ctx.sync()
    np.testing.assert_array_equal(got, uni.cpu().numpy())


@pytest.mark.gpu
def test_ragged_resize_with_images_past_4_gib(ctx):
    """Byte offsets are 64-bit: three 1.44 GB images (generated on the device) and a small one that starts past 4 GiB."""
    import torch
    ro = _resize_oracle()
    big, small = (20000, 24000), (37, 53)
    shapes = [big, big, big, small]
    off = np.cumsum([0] + [3 * h * w for h, w in shapes])
    assert off[3] > 2 ** 32 and 3 * big[0] * big[1] < 2 ** 31
    dh, dw = 64, 96
    gen = torch.Generator(device="cuda").manual_seed(5)
    src = torch.randint(0, 256, (int(off[-1]),), dtype=torch.uint8, device="cuda", generator=gen)
    out = torch.zeros((4, dh, dw, 3), dtype=torch.uint8, device="cuda")
    _torch_done()
    ctx.resize_u8bgr_ragged(src, np.array(shapes, dtype=np.int32), out, dh, dw)
    ctx.sync()
    got = out.cpu().numpy()
    last = src[int(off[3]):].cpu().numpy().reshape(small[0], small[1], 3)
    np.testing.assert_array_equal(got[3], ro.resize_bilinear_u8(last, dh, dw))
    # image 2 (rows on both sides of 4 GiB): the oracle's formula on the gathered rows and columns it reads
    img = src[int(off[2]):int(off[3])].view(big[0], big[1], 3)
    x0, x1, a0, a1 = ro.axis_table(big[1], dw, True)
    y0, y1, b0, b1 = ro.axis_table(big[0], dh, False)
    rows = img[torch.from_numpy(np.concatenate([y0, y1]).astype(np.int64)).cuda()]
    gath = rows[:, torch.from_numpy(np.concatenate([x0, x1]).astype(np.int64)).cuda()].cpu().numpy().astype(np.int64)
    hb = gath[:, :dw] * a0[None, :, None] + gath[:, dw:] * a1[None, :, None]
    want = (((b0[:, None, None] * (hb[:dh] >> 4)) >> 16) + ((b1[:, None, None] * (hb[dh:] >> 4)) >> 16) + 2) >> 2
    np.testing.assert_array_equal(got[2], want.astype(np.uint8))
    del src, img, rows
    torch.cuda.empty_cache()


def _same_dets(got, want, md):
    (dg, cg), (dw_, cw) = got, want
    np.testing.assert_array_equal(cg, cw)
    for i in range(len(cw)):
        k = int(min(cw[i], md))
        np.testing.assert_array_equal(dg[i][:k].view(np.int32), dw_[i][:k].view(np.int32), err_msg="frame %d" % i)


def _reference_dets(ctx, ro, imgs, h, w):
    """The reference's order of operations: cv2.resize of each image (oracle), then the network-size entry point."""
    return ctx.forward_u8bgr(np.stack([ro.resize_bilinear_u8(im, h, w) for im in imgs]))


MIX_SMALL = [(48, 64), (128, 192), (64, 96), (37, 53), (200, 150), (1, 1), (23, 301), (90, 31), (64, 97)]
MIX_416 = [(480, 640), (375, 500), (500, 375), (832, 832), (416, 416), (240, 320), (1080, 1920), (333, 500), (1, 1), (401, 263)]


@pytest.mark.gpu
@pytest.mark.parametrize("net", ["p_64x96", "f_64x96", "p_416", "f_416", "yolo_v2"])
def test_ragged_detections_equal_resize_then_forward(ctx, net):
    ro = _resize_oracle()
    rng = np.random.default_rng(41)
    if net in ("p_64x96", "f_64x96"):
        g, qnet, _ = gu.load("ref_p_64x96")
        h, w, mix, conf = 64, 96, MIX_SMALL, 0.1
    elif net in ("p_416", "f_416"):
        qnet = ex.random_quantnet(seed=0, calib_hw=(416, 416), calib_frames=2, head_bias_shift=-3.0)
        h, w, mix, conf = 416, 416, MIX_416, 0.1
    else:
        qnet = ex.random_quantnet_yolo_v2(seed=0, calib_hw=(64, 96), calib_frames=1)
        h, w, mix, conf = 64, 96, MIX_SMALL, 0.02
    contract = lib.CONTRACT_F if net.startswith("f_") else lib.CONTRACT_P
    ctx.load_quantnet(qnet, contract=contract, conf_thresh=conf, nms_thresh=0.5, max_det=512)
    imgs = _images(rng, mix)
    want = _reference_dets(ctx, ro, imgs, h, w)
    if net == "p_64x96":
        assert want[1].sum() > 0
    try:
        for chunk in (64, 3, 1):
            ctx.set_host_chunk(chunk)
            _same_dets(ctx.forward_u8bgr_images(imgs, (h, w)), want, 512)
    finally:
        ctx.set_host_chunk(64)


@pytest.mark.gpu
def test_ragged_device_and_staged_entry_points_agree(ctx):
    import torch
    g, qnet, _ = gu.load("ref_p_64x96")
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=512)
    h, w = 64, 96
    imgs = _images(np.random.default_rng(43), MIX_SMALL)
    n = len(imgs)
    want = ctx.forward_u8bgr_images(imgs, (h, w))
    flat, hw = lib.pack_images(imgs)
    d_src = _dev(flat)

    def run_dev(fn):
        d_dets = torch.zeros((n, 512, 8), dtype=torch.int32, device="cuda")
        d_counts = torch.zeros(n, dtype=torch.int32, device="cuda")
        _torch_done()
        fn(d_dets, d_counts)
        ctx.sync()
        return d_dets.cpu().numpy().view(lib.DET_DTYPE).reshape(n, 512), d_counts.cpu().numpy()

    _same_dets(run_dev(lambda d, c: ctx.forward_u8bgr_ragged_dev(d_src, hw, h, w, d, c)), want, 512)
    staged = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda")
    _torch_done()
    ctx.resize_u8bgr_ragged(d_src, hw, staged, h, w)
    _same_dets(run_dev(lambda d, c: ctx.forward_u8bgr_dev(staged, n, h, w, d, c)), want, 512)


@pytest.mark.gpu
def test_ragged_calls_in_flight_keep_their_own_tables(ctx):
    """No call overwrites tables that a still-queued resize reads: two submissions with different size mixes in flight, and
    device-entry-point calls queued back to back without a synchronise, each return what its blocking call returns."""
    import torch
    g, qnet, _ = gu.load("ref_p_64x96")
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=512)
    h, w = 64, 96
    rng = np.random.default_rng(47)
    mixes = [_images(rng, MIX_SMALL), _images(rng, [(300, 400), (31, 17), (64, 96), (129, 257), (2, 2)]),
             _images(rng, [(96, 64), (45, 45), (500, 20)] * 2)]
    want = [ctx.forward_u8bgr_images(m, (h, w)) for m in mixes]
    ctx.set_host_chunk(2)
    try:
        packs = [lib.pack_images(m) for m in mixes[:2]]
        pinned = [torch.from_numpy(p).pin_memory() for p, _ in packs]
        outs = [(np.zeros((len(hw), 512), lib.DET_DTYPE), np.zeros(len(hw), np.int32)) for _, hw in packs]
        tickets = [ctx.submit_u8bgr_images(pinned[k], packs[k][1], (h, w), *outs[k]) for k in range(2)]
        dummy = np.zeros(64, np.int32)
        rc = ctx.L.yolo_b200_submit_u8bgr_ragged(ctx._h, pinned[0].data_ptr(), len(packs[0][1]), packs[0][1].ctypes.data, h, w,
                                                 dummy.ctypes.data, dummy.ctypes.data)
        assert rc == E_STATE
        for t in tickets:
            ctx.wait(t)
        for k in range(2):
            _same_dets(outs[k], want[k], 512)
    finally:
        ctx.set_host_chunk(64)
    res = []
    for m in mixes + mixes[:1]:                                  # three calls: the staging buffers alternate and are reused
        flat, hw = lib.pack_images(m)
        res.append((_dev(flat), hw, torch.zeros((len(m), 512, 8), dtype=torch.int32, device="cuda"),
                    torch.zeros(len(m), dtype=torch.int32, device="cuda")))
    _torch_done()
    for src, hw, d_dets, d_counts in res:                        # queued back to back, no synchronise in between
        ctx.forward_u8bgr_ragged_dev(src, hw, h, w, d_dets, d_counts)
    ctx.sync()
    for (_, _, d_dets, d_counts), wnt in zip(res, want + want[:1]):
        n = d_counts.numel()
        _same_dets((d_dets.cpu().numpy().view(lib.DET_DTYPE).reshape(n, 512), d_counts.cpu().numpy()), wnt, 512)


@pytest.mark.gpu
def test_stage_calls_of_changing_geometry_queued_back_to_back(ctx):
    """Resize stages queued without a synchronise while the source geometry changes from call to call: the uniform tables
    are rewritten in stream order behind the resizes that still read them, and each of the two staging buffers is refilled
    while copies out of earlier ones are still queued.  Every output equals the oracle; every call is one launch."""
    import torch
    ro, yo = _resize_oracle(), _oracle("yuv_u8")
    rng = np.random.default_rng(59)
    dh, dw = 40, 44
    calls = []                                                   # (issue the call, device output, expected output)

    def uniform(sh, sw, n=3):
        imgs = rng.integers(0, 256, (n, sh, sw, 3), dtype=np.uint8)
        d, out = _dev(imgs), torch.zeros((n, dh, dw, 3), dtype=torch.uint8, device="cuda")
        calls.append((lambda: ctx.resize_u8bgr(d, n, sh, sw, out, dh, dw), out, ro.resize_batch(imgs, dh, dw)))

    def ragged(shapes):
        imgs = _images(rng, shapes)
        flat, hw = lib.pack_images(imgs)
        d, out = _dev(flat), torch.zeros((len(imgs), dh, dw, 3), dtype=torch.uint8, device="cuda")
        calls.append((lambda: ctx.resize_u8bgr_ragged(d, hw, out, dh, dw), out, np.stack([ro.resize_bilinear_u8(im, dh, dw) for im in imgs])))

    def yuv(fmt, sh, sw, n=2):
        frames = rng.integers(0, 256, (n,) + lib.yuv_frame_shape(fmt, sh, sw), dtype=np.uint8)
        d, out = _dev(frames), torch.zeros((n, dh, dw, 3), dtype=torch.uint8, device="cuda")
        calls.append((lambda: ctx.yuv_to_bgr_resize(d, fmt, n, sh, sw, out, dh, dw), out, ro.resize_batch(yo.to_bgr_batch(frames, fmt), dh, dw)))

    uniform(48, 64); uniform(37, 53); uniform(90, 31)           # three geometry changes in a row
    yuv(lib.YUV_NV12, 34, 66)
    ragged([(60, 80), (17, 9), (48, 64), (1, 1)])
    uniform(48, 64)
    ragged([(60, 80)] * 4)                                       # one size: the uniform kernel with the cached tables
    yuv(lib.YUV_YUYV, 7, 8)
    ragged(MIX_SMALL)
    uniform(200, 150); uniform(37, 53)
    _torch_done()
    before = ctx.launch_count()
    for k, (issue, _, _) in enumerate(calls):
        issue()
        assert ctx.launch_count() == before + k + 1, "call %d: one launch" % k
    ctx.sync()
    for k, (_, out, want) in enumerate(calls):
        np.testing.assert_array_equal(out.cpu().numpy(), want, err_msg="call %d" % k)


@pytest.mark.gpu
def test_ragged_errors_and_empty_batch(ctx):
    import torch
    g, qnet, _ = gu.load("ref_p_64x96")
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=512)
    L, hh = ctx.L, ctx._h
    d_src = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    d_dst = torch.full((4096,), 7, dtype=torch.uint8, device="cuda")
    h_src = np.zeros(4096, np.uint8)
    dets = np.full(512 * 8 * 2, 7, np.int32)
    counts = np.full(2, 7, np.int32)
    d_dets = torch.full((2, 512, 8), 7, dtype=torch.int32, device="cuda")
    d_counts = torch.full((2,), 7, dtype=torch.int32, device="cuda")
    ok = np.array([[8, 8], [5, 7]], np.int32)
    zero = np.array([[8, 8], [0, 7]], np.int32)
    huge = np.array([[8, 8], [30000, 30000]], np.int32)          # 2.7 GB > 2 GiB
    _torch_done()

    def calls(n, hw):
        p = hw.ctypes.data if hw is not None else None
        return [L.yolo_b200_resize_u8bgr_ragged(hh, d_src.data_ptr(), n, p, d_dst.data_ptr(), 16, 16),
                L.yolo_b200_forward_u8bgr_ragged(hh, h_src.ctypes.data, n, p, 64, 96, dets.ctypes.data, counts.ctypes.data),
                L.yolo_b200_forward_u8bgr_ragged_dev(hh, d_src.data_ptr(), n, p, 64, 96, d_dets.data_ptr(), d_counts.data_ptr())]

    assert calls(-1, ok) == [E_ARG] * 3
    assert calls(2, zero) == [E_ARG] * 3
    assert calls(2, None) == [E_ARG] * 3
    assert calls(2, huge) == [E_UNSUPPORTED] * 3
    assert L.yolo_b200_submit_u8bgr_ragged(hh, h_src.ctypes.data, 2, huge.ctypes.data, 64, 96, dets.ctypes.data, counts.ctypes.data) == E_UNSUPPORTED
    assert L.yolo_b200_submit_u8bgr_ragged(hh, h_src.ctypes.data, 2, None, 64, 96, dets.ctypes.data, counts.ctypes.data) == E_ARG
    assert L.yolo_b200_resize_u8bgr_ragged(hh, None, 2, ok.ctypes.data, d_dst.data_ptr(), 16, 16) == E_ARG
    assert calls(0, ok) == [0] * 3 and calls(0, None) == [0] * 3
    ctx.sync()
    assert (d_dst == 7).all() and (d_dets == 7).all() and (d_counts == 7).all()
    assert (dets == 7).all() and (counts == 7).all()
    d, c = ctx.forward_u8bgr_images([], (64, 96))
    assert d.shape == (0, 512) and c.shape == (0,)


@pytest.mark.gpu
def test_detect_cli_on_a_folder_of_mixed_sizes(tmp_path):
    """tools/detect.py image mode: one ragged call per batch, two batches in flight; one annotated file per input and, per
    image, the detection count of that image run alone through yolo_b200_forward_u8bgr_resize."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(53)
    shapes = [(72, 96), (50, 64), (96, 72), (33, 47), (128, 128), (72, 96), (1, 1), (200, 120)]
    src = tmp_path / "images"
    src.mkdir()
    for i, (h, w) in enumerate(shapes):
        assert cv2.imwrite(str(src / ("im%02d.png" % i)), rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    out = tmp_path / "out"
    size = 96
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "detect.py"), "--trained_model", "random", "--images", str(src),
                        "-size", str(size), "--batch", "3", "--out", str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert sorted(os.listdir(out)) == ["im%02d.jpg" % i for i in range(len(shapes))]
    printed = {m.group(1): int(m.group(2)) for m in re.finditer(r"^(im\d\d): (\d+) detections", r.stdout, re.M)}
    assert len(printed) == len(shapes)
    qnet = ex.random_quantnet(seed=0, calib_hw=(size, size), calib_frames=2, head_bias_shift=-3.0)      # detect.py's network
    c = lib.Context(0)
    try:
        c.load_quantnet(qnet, contract=lib.CONTRACT_P, head_mode=lib.HEAD_PYTHON, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
        for i in range(len(shapes)):
            img = cv2.imread(str(src / ("im%02d.png" % i)), cv2.IMREAD_COLOR)
            _, counts = c.forward_u8bgr_resize(img[None], (size, size))
            assert printed["im%02d" % i] == min(int(counts[0]), 1024), "image %d" % i
    finally:
        c.close()
