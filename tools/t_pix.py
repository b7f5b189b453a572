#!/usr/bin/env python
"""Measures the pixel-format front end (cvtColor RGB / RGBA / BGRA / gray / planar RGB -> BGR fused into the resize) on one
GPU and writes a JSON record.

    python tools/t_pix.py [--out profiles/pix_r3.json]

1. Stage time, 256 frames of 480x640 and of 1080x1920 -> 416x416: the five pixel-format instantiations against the BGR
   resize kernel on the same geometry, the RGBA / BGRA word loads (aligned source) and byte loads (source at +1).  The
   variants alternate within every round (tools/t_ragged.py time_rounds); each output must equal the BGR kernel's output
   on the cvtColor'd frames.  Every working set (source + 133 MB of output) exceeds the 126 MB L2.
2. End to end from pinned host memory (slim_yolo_v2 416x416, contract P), 256 frames of 480x640 per call: submit/wait with
   two calls in flight, for each format and for BGR (through the one-size ragged call, the submit form of
   yolo_b200_forward_u8bgr_resize); the detections of each format and of BGR on its cvtColor'd frames must agree.
3. The card's name, power limit and max SM clock, read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import yolo_b200  # noqa: E402,F401
from yolo_b200 import export as ex, lib  # noqa: E402
from t_ragged import card, stats, time_rounds  # noqa: E402
import pix_u8 as po  # noqa: E402

FORMATS = {"rgb": lib.PIX_RGB, "rgba": lib.PIX_RGBA, "bgra": lib.PIX_BGRA, "gray": lib.PIX_GRAY, "rgb_planar": lib.PIX_RGB_PLANAR}
GEOMS = [(480, 640), (1080, 1920)]


def seeded(shape, n, seed):
    """n frames of shape: a few distinct seeded frames repeated (host generation of 256 1080p frames would dominate the run)."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (8,) + tuple(shape), dtype=np.uint8)
    return np.ascontiguousarray(base[np.arange(n) % 8])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pix_r3.json"))
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
        src = {k: torch.from_numpy(seeded(lib.pix_frame_shape(f, sh, sw), B, 10 + f)).cuda() for k, f in FORMATS.items()}
        bgr_of = {k: torch.from_numpy(po.to_bgr_batch(src[k][:8].cpu().numpy(), f)[np.arange(B) % 8]).cuda() for k, f in FORMATS.items()}
        shifted = {}
        for k in ("rgba", "bgra"):                          # the same frames at a source address that is not 4-byte aligned
            buf = torch.zeros(src[k].numel() + 1, dtype=torch.uint8, device="cuda")
            buf[1:] = src[k].reshape(-1)
            shifted[k] = buf[1:]
        names = ["bgr"] + list(FORMATS) + ["rgba_bytes", "bgra_bytes"]
        outs = {k: torch.zeros((B, H, W, 3), dtype=torch.uint8, device="cuda") for k in names}
        variants = {"bgr": lambda: ctx.resize_u8bgr(bgr_of["rgb"], B, sh, sw, outs["bgr"], H, W)}
        for k, f in FORMATS.items():
            variants[k] = (lambda k=k, f=f: ctx.pix_to_bgr_resize(src[k], f, B, sh, sw, outs[k], H, W))
        for k in ("rgba", "bgra"):
            variants[k + "_bytes"] = (lambda k=k: ctx.pix_to_bgr_resize(shifted[k], FORMATS[k], B, sh, sw, outs[k + "_bytes"], H, W))
        res = time_rounds(variants, args.rounds, 20, s)
        torch.cuda.synchronize()
        for k in names[1:]:                                 # each output = the BGR kernel on the cvtColor'd frames
            ref = torch.zeros_like(outs[k])
            ctx.resize_u8bgr(bgr_of[k.replace("_bytes", "")], B, sh, sw, ref, H, W)
            ctx.sync()
            assert torch.equal(outs[k], ref), "%s %dx%d differs from cvtColor + BGR resize" % (k, sh, sw)
        entry = {}
        for k, v in res.items():
            fmt = FORMATS.get(k.replace("_bytes", ""))
            per = sh * sw * 3 if fmt is None else int(np.prod(lib.pix_frame_shape(fmt, sh, sw)))
            algo = B * per + B * H * W * 3
            entry[k] = dict(stats(v), source_bytes=B * per, gbs=algo / (np.median(v) / 1e3) / 1e9)
        rec["stage"]["%d x %dx%d -> %dx%d" % (B, sh, sw, H, W)] = entry
        print(json.dumps(entry, indent=1))
        del src, bgr_of, shifted, outs

    # 2. end to end from pinned host memory, submit/wait with two calls in flight
    qnet = ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2, head_bias_shift=-3.0)
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
    md = 1024
    mk = lambda: (torch.zeros((B, md, 8), dtype=torch.int32).pin_memory(), torch.zeros(B, dtype=torch.int32).pin_memory())  # noqa: E731
    pairs = [mk(), mk()]
    rec["end_to_end"] = {"network": "slim_yolo_v2 416x416, contract P, conf 0.1, max_det 1024", "frames_per_call": B,
                         "note": "pinned host frames; submit/wait = 8 calls with two in flight"}
    sh, sw = GEOMS[0]
    host = {k: torch.from_numpy(seeded(lib.pix_frame_shape(f, sh, sw), B, 20 + f)).pin_memory() for k, f in FORMATS.items()}
    bgr_host = {k: torch.from_numpy(po.to_bgr_batch(host[k][:8].numpy(), f)[np.arange(B) % 8]).pin_memory() for k, f in FORMATS.items()}
    host["bgr"] = bgr_host["rgb"]
    hw = np.array([(sh, sw)] * B, np.int32)
    fbytes = {k: int(np.prod(lib.pix_frame_shape(f, sh, sw))) for k, f in FORMATS.items()}
    fbytes["bgr"] = sh * sw * 3

    def submit(k, d, c, frames=None):
        frames = host[k] if frames is None else frames
        if k == "bgr":
            t = L.yolo_b200_submit_u8bgr_ragged(ctx._h, frames.data_ptr(), B, hw.ctypes.data, H, W, d.data_ptr(), c.data_ptr())
        else:
            t = L.yolo_b200_submit_pix(ctx._h, frames.data_ptr(), FORMATS[k], B, sh, sw, H, W, d.data_ptr(), c.data_ptr())
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
        pipelined(k, 2)
    for k in FORMATS:                                     # each format's detections = BGR's on its cvtColor'd frames
        ctx.wait(submit("bgr", *pairs[0], frames=bgr_host[k])); c_bgr = pairs[0][1].numpy().copy()
        ctx.wait(submit(k, *pairs[1])); assert np.array_equal(pairs[1][1].numpy(), c_bgr), "%s and cvtColor + BGR disagree" % k
    t_sub = {k: [] for k in names}
    for r in range(args.e2e_reps):
        order = names[r % len(names):] + names[:r % len(names)]
        for k in order:
            t0 = time.perf_counter(); pipelined(k); t_sub[k].append((time.perf_counter() - t0) / 8)
    entry = {}
    for k in names:
        fb, ms = fbytes[k], float(np.median(t_sub[k]))
        entry[k] = {"h2d_bytes_per_frame": fb, "submit_wait_ms_per_call": 1e3 * ms, "submit_wait_frames_per_s": B / ms,
                    "submit_wait_h2d_GBs": B * fb / ms / 1e9, "submit_wait_all_ms": [1e3 * x for x in t_sub[k]]}
    rec["end_to_end"]["%dx%d" % (sh, sw)] = entry
    print(json.dumps(entry, indent=1))
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
