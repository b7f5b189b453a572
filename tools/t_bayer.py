#!/usr/bin/env python
"""Measures the Bayer front end (cvtColor Bayer -> BGR demosaic fused into the resize) on one GPU and writes a JSON record.

    python tools/t_bayer.py [--out profiles/bayer_r3.json]

1. Stage time, 256 frames of 480x640 and of 1080x1920 -> 416x416: the four Bayer instantiations against the BGR resize
   kernel and the NV12 stage on the same geometry.  The variants alternate within every round (tools/t_ragged.py
   time_rounds); each Bayer output must equal the BGR kernel's output on the cvtColor'd frames.  Every working set
   (source + 133 MB of output) exceeds the 126 MB L2; the Bayer source alone is 79 MB at 480x640 and 531 MB at 1080x1920.
2. End to end from pinned host memory (slim_yolo_v2 416x416, contract P), 256 frames per call: blocking calls and
   submit/wait with two calls in flight, for Bayer RGGB, NV12 and BGR (yolo_b200_forward_u8bgr_resize, and its submit form
   through the one-size ragged call); the detections of Bayer and of BGR on the cvtColor'd frames must agree.
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

PATTERNS = {"rggb": (lib.BAYER_RGGB, cv2.COLOR_BayerRGGB2BGR), "bggr": (lib.BAYER_BGGR, cv2.COLOR_BayerBGGR2BGR),
            "grbg": (lib.BAYER_GRBG, cv2.COLOR_BayerGRBG2BGR), "gbrg": (lib.BAYER_GBRG, cv2.COLOR_BayerGBRG2BGR)}
GEOMS = [(480, 640), (1080, 1920)]


def seeded(shape, n, seed):
    """n frames of shape: a few distinct seeded frames repeated (host generation of 256 1080p frames would dominate the run)."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (8,) + tuple(shape), dtype=np.uint8)
    return np.ascontiguousarray(base[np.arange(n) % 8])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bayer_r3.json"))
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
        raw = torch.from_numpy(seeded((sh, sw), B, 10)).cuda()
        nv12 = torch.from_numpy(seeded(lib.yuv_frame_shape(lib.YUV_NV12, sh, sw), B, 11)).cuda()
        raw8 = raw[:8].cpu().numpy()
        bgr_of = {k: torch.from_numpy(np.stack([cv2.cvtColor(x, code) for x in raw8])[np.arange(B) % 8]).cuda() for k, (_, code) in PATTERNS.items()}
        outs = {k: torch.zeros((B, H, W, 3), dtype=torch.uint8, device="cuda") for k in list(PATTERNS) + ["bgr", "nv12"]}
        variants = {"bgr": lambda: ctx.resize_u8bgr(bgr_of["rggb"], B, sh, sw, outs["bgr"], H, W),
                    "nv12": lambda: ctx.yuv_to_bgr_resize(nv12, lib.YUV_NV12, B, sh, sw, outs["nv12"], H, W)}
        for k, (p, _) in PATTERNS.items():
            variants[k] = (lambda k=k, p=p: ctx.bayer_to_bgr_resize(raw, p, B, sh, sw, outs[k], H, W))
        res = time_rounds(variants, args.rounds, 20, s)
        torch.cuda.synchronize()
        for k in PATTERNS:                                    # each Bayer output = the BGR kernel on its cvtColor'd frames
            ref = torch.zeros_like(outs[k])
            ctx.resize_u8bgr(bgr_of[k], B, sh, sw, ref, H, W)
            ctx.sync()
            assert torch.equal(outs[k], ref), "%s %dx%d differs from cvtColor + BGR resize" % (k, sh, sw)
        entry = {}
        for k, v in res.items():
            per = {"bgr": sh * sw * 3, "nv12": sh * sw * 3 // 2}.get(k, sh * sw)
            algo = B * per + B * H * W * 3
            entry[k] = dict(stats(v), source_bytes=B * per, gbs=algo / (np.median(v) / 1e3) / 1e9)
        rec["stage"]["%d x %dx%d -> %dx%d" % (B, sh, sw, H, W)] = entry
        print(json.dumps(entry, indent=1))
        del raw, nv12, bgr_of, outs

    # 2. end to end from pinned host memory
    qnet = ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2, head_bias_shift=-3.0)
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
    md = 1024
    mk = lambda: (torch.zeros((B, md, 8), dtype=torch.int32).pin_memory(), torch.zeros(B, dtype=torch.int32).pin_memory())  # noqa: E731
    pairs = [mk(), mk()]
    rec["end_to_end"] = {"network": "slim_yolo_v2 416x416, contract P, conf 0.1, max_det 1024", "frames_per_call": B,
                         "note": "pinned host frames; submit/wait = 8 calls with two in flight; blocking = one call at a time"}
    for sh, sw in GEOMS:
        host = {"bayer": torch.from_numpy(seeded((sh, sw), B, 20)).pin_memory(),
                "nv12": torch.from_numpy(seeded(lib.yuv_frame_shape(lib.YUV_NV12, sh, sw), B, 21)).pin_memory()}
        host["bgr"] = torch.from_numpy(np.stack([cv2.cvtColor(x, cv2.COLOR_BayerRGGB2BGR) for x in host["bayer"][:8].numpy()])[np.arange(B) % 8]).pin_memory()
        hw = np.array([(sh, sw)] * B, np.int32)
        fbytes = {"bayer": sh * sw, "nv12": sh * sw * 3 // 2, "bgr": sh * sw * 3}

        def blocking(k, d, c):
            if k == "bgr":
                r = L.yolo_b200_forward_u8bgr_resize(ctx._h, host[k].data_ptr(), B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
            elif k == "nv12":
                r = L.yolo_b200_forward_yuv(ctx._h, host[k].data_ptr(), lib.YUV_NV12, B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
            else:
                r = L.yolo_b200_forward_bayer(ctx._h, host[k].data_ptr(), lib.BAYER_RGGB, B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
            assert r == 0, L.yolo_b200_last_error()

        def submit(k, d, c):
            if k == "bgr":
                t = L.yolo_b200_submit_u8bgr_ragged(ctx._h, host[k].data_ptr(), B, hw.ctypes.data, H, W, d.data_ptr(), c.data_ptr())
            elif k == "nv12":
                t = L.yolo_b200_submit_yuv(ctx._h, host[k].data_ptr(), lib.YUV_NV12, B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
            else:
                t = L.yolo_b200_submit_bayer(ctx._h, host[k].data_ptr(), lib.BAYER_RGGB, B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
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

        names = ["bgr", "nv12", "bayer"]
        for k in names:                                       # warm-up: allocations, tables, module loads
            blocking(k, *pairs[0]); pipelined(k, 2)
        # the BGR input is the cvtColor'd Bayer frames: their detections must agree
        blocking("bgr", *pairs[0]); c_bgr = pairs[0][1].numpy().copy()
        blocking("bayer", *pairs[1]); assert np.array_equal(pairs[1][1].numpy(), c_bgr), "Bayer and cvtColor + BGR disagree"
        t_blk = {k: [] for k in names}
        t_sub = {k: [] for k in names}
        for r in range(args.e2e_reps):
            order = names[r % len(names):] + names[:r % len(names)]
            for k in order:
                t0 = time.perf_counter(); blocking(k, *pairs[0]); t_blk[k].append(time.perf_counter() - t0)
                t0 = time.perf_counter(); pipelined(k); t_sub[k].append((time.perf_counter() - t0) / 8)
        entry = {}
        for k in names:
            fb = fbytes[k]
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
