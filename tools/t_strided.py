#!/usr/bin/env python
"""Measures the pitched front end (yolo_b200_frames: row pitch, plane offsets, frame stride) on one GPU and writes a JSON
record.

    python tools/t_strided.py [--out profiles/strided_r3.json]

1. Stage time, 256 frames of 480x640 and of 1080x1920 -> 416x416, for BGR, NV12, RGGB, RGBA and planar RGB: the family's
   packed stage, the pitched stage on the same packed frames (the layout yolo_b200_frames_packed fills in) and the pitched
   stage on the frames with every row pitch rounded up to 512 bytes (what NVDEC and GpuMat allocators do).  The three
   alternate within every round (tools/t_ragged.py time_rounds); their outputs must be equal.  Every working set
   (source + 133 MB of output) exceeds the 126 MB L2.
2. End to end from pinned host memory (slim_yolo_v2 416x416, contract P), 256 NV12 frames of 480x640 per call: submit/wait
   with two calls in flight, packed (yolo_b200_submit_yuv) against pitched at 512 (yolo_b200_submit_frames, which copies
   the padding too); the detections must agree.
3. The three BGR instantiations on the same frames (tools/micro/resize_pitched_bgr.cu, compiled here): packed, pitched
   and ragged (one descriptor per frame, which a one-size call never reaches through the library), alternating rounds.
4. The card's name, power limit and max SM clock, read in the same run.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import yolo_b200  # noqa: E402,F401
from yolo_b200 import export as ex, lib  # noqa: E402
from t_ragged import card, stats, time_rounds  # noqa: E402

CASES = {"bgr": (lib.SRC_BGR, 0), "nv12": (lib.SRC_YUV, lib.YUV_NV12), "rggb": (lib.SRC_BAYER, lib.BAYER_RGGB),
         "rgba": (lib.SRC_PIX, lib.PIX_RGBA), "rgb_planar": (lib.SRC_PIX, lib.PIX_RGB_PLANAR)}
GEOMS = [(480, 640), (1080, 1920)]


def pitched(packed: lib.Frames, to=512) -> lib.Frames:
    """The layout of `packed` with every plane's pitch rounded up to a multiple of `to`, planes and frames back to back."""
    d = lib.Frames.from_buffer_copy(packed)
    rows = {lib.SRC_YUV: {lib.YUV_NV12: [d.sh, d.sh // 2]}}.get(d.family, {}).get(d.format)
    nplanes = 3 if (d.family == lib.SRC_PIX and d.format == lib.PIX_RGB_PLANAR) else len(rows or [0])
    rows = rows or [d.sh] * nplanes
    off = 0
    for p in range(nplanes):
        d.plane_offset[p] = off
        d.row_pitch[p] = (packed.row_pitch[p] + to - 1) // to * to
        off += rows[p] * d.row_pitch[p]
    d.frame_stride = off
    return d, rows


def relayout(src: torch.Tensor, packed: lib.Frames, d: lib.Frames, rows, n):
    """The packed frames src (device, flat) copied into a new device buffer at layout d (padding 0)."""
    _, end = lib.frames_span(d, n)
    out = torch.zeros(end, dtype=torch.uint8, device="cuda")
    for p, r in enumerate(rows):
        rb = packed.row_pitch[p]
        out.as_strided((n, r, rb), (d.frame_stride, d.row_pitch[p], 1), d.plane_offset[p]).copy_(
            src.as_strided((n, r, rb), (packed.frame_stride, rb, 1), packed.plane_offset[p]))
    return out


def seeded(nbytes, n, seed):
    """n frames of nbytes: a few distinct seeded frames repeated (host generation of 256 1080p frames would dominate)."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (8, nbytes), dtype=np.uint8)
    return np.ascontiguousarray(base[np.arange(n) % 8])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "strided_r3.json"))
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--e2e-reps", type=int, default=3)
    args = ap.parse_args()
    rec = {"card": card()}
    print(rec["card"])
    ctx = lib.Context(0)
    L = ctx.L
    s = torch.cuda.Stream()
    torch.cuda.set_stream(s)
    ctx.set_stream(s.cuda_stream)
    B, H, W = 256, 416, 416

    # 1. stages
    rec["stage"] = {}
    for sh, sw in GEOMS:
        entry = {}
        for name, (family, fmt) in CASES.items():
            packed = lib.frames_packed(family, fmt, sh, sw)
            src = torch.from_numpy(seeded(packed.frame_stride, B, 10 + fmt + 7 * family)).cuda().reshape(-1)
            d512, rows = pitched(packed)
            src512 = relayout(src, packed, d512, rows, B)
            outs = {k: torch.zeros((B, H, W, 3), dtype=torch.uint8, device="cuda") for k in ("packed", "pitched_packed", "pitched_512")}
            if family == lib.SRC_BGR:
                run_packed = lambda: ctx.resize_u8bgr(src, B, sh, sw, outs["packed"], H, W)  # noqa: E731
            elif family == lib.SRC_YUV:
                run_packed = lambda: ctx.yuv_to_bgr_resize(src, fmt, B, sh, sw, outs["packed"], H, W)  # noqa: E731
            elif family == lib.SRC_BAYER:
                run_packed = lambda: ctx.bayer_to_bgr_resize(src, fmt, B, sh, sw, outs["packed"], H, W)  # noqa: E731
            else:
                run_packed = lambda: ctx.pix_to_bgr_resize(src, fmt, B, sh, sw, outs["packed"], H, W)  # noqa: E731
            variants = {"packed": run_packed,
                        "pitched_packed": lambda: ctx.frames_to_bgr_resize(src, packed, B, outs["pitched_packed"], H, W),
                        "pitched_512": lambda: ctx.frames_to_bgr_resize(src512, d512, B, outs["pitched_512"], H, W)}
            res = time_rounds(variants, args.rounds, 20, s)
            torch.cuda.synchronize()
            assert torch.equal(outs["packed"], outs["pitched_packed"]) and torch.equal(outs["packed"], outs["pitched_512"]), \
                "%s %dx%d: pitched output differs" % (name, sh, sw)
            e = {k: dict(stats(v), source_bytes=B * (packed.frame_stride if k != "pitched_512" else d512.frame_stride))
                 for k, v in res.items()}
            e["pitched_packed_over_packed"] = e["pitched_packed"]["median_ms"] / e["packed"]["median_ms"]
            e["pitched_512_over_packed"] = e["pitched_512"]["median_ms"] / e["packed"]["median_ms"]
            e["pitch_512"] = list(d512.row_pitch)[:len(rows)]
            entry[name] = e
            print(name, "%dx%d" % (sh, sw), json.dumps({k: (v["median_ms"] if isinstance(v, dict) else v) for k, v in e.items()}))
            del src, src512, outs
        rec["stage"]["%d x %dx%d -> %dx%d" % (B, sh, sw, H, W)] = entry

    # 3. the BGR instantiations at the kernel level
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "resize_pitched_bgr")
        from yolo_b200 import build as b
        subprocess.run([b.nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
                        "-I", b.CSRC, "-o", exe,
                        os.path.join(ROOT, "tools", "micro", "resize_pitched_bgr.cu")], check=True)
        out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    print(out)
    rec["bgr_instantiations"] = {}
    for line in out.splitlines():
        m = re.match(r"256 x (\d+)x(\d+) -> 416x416: outputs equal 1 1, ms packed=([\d.]+) layout=([\d.]+) ragged=([\d.]+)", line)
        assert m, "unexpected output (outputs must agree): " + line
        rec["bgr_instantiations"]["%sx%s" % m.group(1, 2)] = {k: float(m.group(i)) for i, k in ((3, "packed"), (4, "pitched"), (5, "ragged"))}

    # 2. end to end from pinned host memory, submit/wait with two calls in flight
    qnet = ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2, head_bias_shift=-3.0)
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
    md = 1024
    mk = lambda: (torch.zeros((B, md, 8), dtype=torch.int32).pin_memory(), torch.zeros(B, dtype=torch.int32).pin_memory())  # noqa: E731
    pairs = [mk(), mk()]
    sh, sw = GEOMS[0]
    packed = lib.frames_packed(lib.SRC_YUV, lib.YUV_NV12, sh, sw)
    d512, rows = pitched(packed)
    host = torch.from_numpy(seeded(packed.frame_stride, B, 30)).reshape(-1)
    host512 = relayout(host.cuda(), packed, d512, rows, B).cpu().pin_memory()
    host = host.pin_memory()

    def submit(k, dd, cc):
        if k == "packed":
            t = L.yolo_b200_submit_yuv(ctx._h, host.data_ptr(), lib.YUV_NV12, B, sh, sw, H, W, dd.data_ptr(), cc.data_ptr())
        else:
            t = ctx.submit_frames(host512, d512, B, (H, W), dd.numpy().view(lib.DET_DTYPE).reshape(B, md), cc.numpy())
        assert t >= 0, L.yolo_b200_last_error()
        return t

    def pipelined(k, calls=8):
        tickets = []
        for i in range(calls):
            if len(tickets) == 2:
                ctx.wait(tickets.pop(0))
            tickets.append(submit(k, *pairs[i % 2]))
        while tickets:
            ctx.wait(tickets.pop(0))

    names = ["packed", "pitched_512"]
    for k in names:
        pipelined(k, 2)
    ctx.wait(submit("packed", *pairs[0]))
    ctx.wait(submit("pitched_512", *pairs[1]))
    assert np.array_equal(pairs[0][1].numpy(), pairs[1][1].numpy()), "pitched and packed detections disagree"
    t_sub = {k: [] for k in names}
    for r in range(args.e2e_reps):
        for k in (names if r % 2 == 0 else names[::-1]):
            t0 = time.perf_counter(); pipelined(k); t_sub[k].append((time.perf_counter() - t0) / 8)
    entry = {}
    for k in names:
        fb, ms = (packed if k == "packed" else d512).frame_stride, float(np.median(t_sub[k]))
        entry[k] = {"h2d_bytes_per_frame": fb, "submit_wait_ms_per_call": 1e3 * ms, "submit_wait_frames_per_s": B / ms,
                    "submit_wait_all_ms": [1e3 * x for x in t_sub[k]]}
    rec["end_to_end"] = {"network": "slim_yolo_v2 416x416, contract P, conf 0.1, max_det 1024", "frames_per_call": B,
                         "source": "NV12 %dx%d" % (sh, sw), "note": "pinned host frames; submit/wait = 8 calls with two in flight",
                         "calls": entry}
    print(json.dumps(entry, indent=1))
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
