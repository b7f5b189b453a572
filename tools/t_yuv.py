#!/usr/bin/env python
"""Measures the YUV front end (cvtColor NV12 / I420 / YUYV -> BGR fused into the resize) on one GPU and writes a JSON record.

    python tools/t_yuv.py [--out profiles/yuv_r3.json]

1. Kernel time, 256 frames of 480x640 and of 1080x1920 -> 416x416: the three YUV instantiations against the BGR resize
   kernel on the same geometry.  The variants alternate within every round (tools/t_ragged.py time_rounds); the YUV
   outputs must equal the BGR kernel's output on the cvtColor'd frames.  Working sets exceed the 126 MB L2.
2. End to end from pinned host memory (slim_yolo_v2 416x416, contract P), 256 frames per call: blocking calls and
   submit/wait with two calls in flight, YUV formats against the BGR path (yolo_b200_forward_u8bgr_resize, and its
   submit form through the one-size ragged call); the detections must agree.
3. Host-to-device bytes per frame of each input.
"""
import argparse
import json
import os
import sys
import time

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import yolo_b200  # noqa: E402,F401
from yolo_b200 import export as ex, lib  # noqa: E402
from t_ragged import card, stats, time_rounds  # noqa: E402

FORMATS = {"nv12": (lib.YUV_NV12, cv2.COLOR_YUV2BGR_NV12), "i420": (lib.YUV_I420, cv2.COLOR_YUV2BGR_I420),
           "yuyv": (lib.YUV_YUYV, cv2.COLOR_YUV2BGR_YUYV)}
GEOMS = [(480, 640), (1080, 1920)]


def seeded_frames(fmt, n, sh, sw, seed):
    """n YUV frames: a few distinct seeded frames repeated (host generation of 256 1080p frames would dominate the run)."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (8,) + lib.yuv_frame_shape(fmt, sh, sw), dtype=np.uint8)
    return np.ascontiguousarray(base[np.arange(n) % 8])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "yuv_r3.json"))
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

    # 1. kernels
    rec["kernel"] = {}
    for sh, sw in GEOMS:
        yuv = {k: torch.from_numpy(seeded_frames(f, B, sh, sw, 10 + f)).cuda() for k, (f, _) in FORMATS.items()}
        bgr_in = {k: torch.from_numpy(np.stack([cv2.cvtColor(x, code) for x in yuv[k][:8].cpu().numpy()])[np.arange(B) % 8]).cuda()
                  for k, (_, code) in FORMATS.items()}
        outs = {k: torch.zeros((B, H, W, 3), dtype=torch.uint8, device="cuda") for k in list(FORMATS) + ["bgr"]}
        variants = {"bgr": lambda: ctx.resize_u8bgr(bgr_in["nv12"], B, sh, sw, outs["bgr"], H, W)}
        for k, (f, _) in FORMATS.items():
            variants[k] = (lambda k=k, f=f: ctx.yuv_to_bgr_resize(yuv[k], f, B, sh, sw, outs[k], H, W))
        res = time_rounds(variants, args.rounds, 20, s)
        torch.cuda.synchronize()
        for k in FORMATS:                                     # each YUV output = the BGR kernel on its cvtColor'd frames
            ref = torch.zeros_like(outs[k])
            ctx.resize_u8bgr(bgr_in[k], B, sh, sw, ref, H, W)
            ctx.sync()
            assert torch.equal(outs[k], ref), "%s %dx%d differs from cvtColor + BGR resize" % (k, sh, sw)
        entry = {}
        for k, v in res.items():
            src_bytes = B * (sh * sw * 3 if k == "bgr" else int(np.prod(lib.yuv_frame_shape(FORMATS[k][0], sh, sw))))
            algo = src_bytes + B * H * W * 3
            entry[k] = dict(stats(v), source_bytes=src_bytes, gbs=algo / (np.median(v) / 1e3) / 1e9)
        rec["kernel"]["%d x %dx%d -> %dx%d" % (B, sh, sw, H, W)] = entry
        print(json.dumps(entry, indent=1))
        del yuv, bgr_in, outs

    # 2. end to end from pinned host memory
    qnet = ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2, head_bias_shift=-3.0)
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
    md = 1024
    mk = lambda: (torch.zeros((B, md, 8), dtype=torch.int32).pin_memory(), torch.zeros(B, dtype=torch.int32).pin_memory())  # noqa: E731
    pairs = [mk(), mk()]
    rec["end_to_end"] = {"network": "slim_yolo_v2 416x416, contract P, conf 0.1, max_det 1024", "frames_per_call": B,
                         "note": "pinned host frames; submit/wait = 8 calls with two in flight; blocking = one call at a time"}
    for sh, sw in GEOMS:
        host = {k: torch.from_numpy(seeded_frames(f, B, sh, sw, 20 + f)).pin_memory() for k, (f, _) in FORMATS.items()}
        host["bgr"] = torch.from_numpy(np.stack([cv2.cvtColor(x, cv2.COLOR_YUV2BGR_NV12) for x in host["nv12"][:8].numpy()])[np.arange(B) % 8]).pin_memory()
        hw = np.array([(sh, sw)] * B, np.int32)

        def blocking(k, d, c):
            if k == "bgr":
                r = L.yolo_b200_forward_u8bgr_resize(ctx._h, host[k].data_ptr(), B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
            else:
                r = L.yolo_b200_forward_yuv(ctx._h, host[k].data_ptr(), FORMATS[k][0], B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
            assert r == 0, L.yolo_b200_last_error()

        def submit(k, d, c):
            if k == "bgr":
                t = L.yolo_b200_submit_u8bgr_ragged(ctx._h, host[k].data_ptr(), B, hw.ctypes.data, H, W, d.data_ptr(), c.data_ptr())
            else:
                t = L.yolo_b200_submit_yuv(ctx._h, host[k].data_ptr(), FORMATS[k][0], B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
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

        names = ["bgr"] + list(FORMATS)
        for k in names:                                       # warm-up: allocations, tables, module loads
            blocking(k, *pairs[0]); pipelined(k, 2)
        # the BGR input is the cvtColor'd NV12 frames: their detections must agree
        blocking("bgr", *pairs[0]); c_bgr = pairs[0][1].numpy().copy()
        blocking("nv12", *pairs[1]); assert np.array_equal(pairs[1][1].numpy(), c_bgr), "NV12 and cvtColor + BGR disagree"
        t_blk = {k: [] for k in names}
        t_sub = {k: [] for k in names}
        for r in range(args.e2e_reps):
            order = names[r % len(names):] + names[:r % len(names)]
            for k in order:
                t0 = time.perf_counter(); blocking(k, *pairs[0]); t_blk[k].append(time.perf_counter() - t0)
                t0 = time.perf_counter(); pipelined(k); t_sub[k].append((time.perf_counter() - t0) / 8)
        entry = {}
        for k in names:
            fb = sh * sw * 3 if k == "bgr" else int(np.prod(lib.yuv_frame_shape(FORMATS[k][0], sh, sw)))
            mb, ms = float(np.median(t_blk[k])), float(np.median(t_sub[k]))
            entry[k] = {"h2d_bytes_per_frame": fb, "blocking_ms": 1e3 * mb, "blocking_frames_per_s": B / mb,
                        "submit_wait_ms_per_call": 1e3 * ms, "submit_wait_frames_per_s": B / ms,
                        "submit_wait_h2d_GBs": B * fb / ms / 1e9, "submit_wait_all_ms": [1e3 * x for x in t_sub[k]]}
        rec["end_to_end"]["%dx%d" % (sh, sw)] = entry
        print(json.dumps(entry, indent=1))
        del host
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
