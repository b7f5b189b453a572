#!/usr/bin/env python
"""Measures the ragged resize front end (images of different sizes in one call) on one GPU and writes a JSON record.

    python tools/t_ragged.py [--parent-src DIR] [--out profiles/ragged_r3.json]

1. Resize kernel on the bench's resize workload (256 x 480x640 -> 416x416): the uniform instantiation and
   (--parent-src: a directory holding an earlier resize.cu + kernels.h + common.cuh, compiled here into a side library)
   the earlier kernel.  The variants alternate within every round; outputs must agree.  (A ragged call whose images all
   have one size runs the uniform kernel, so the ragged kernel is measured on the mix of 2.)
2. Ragged kernel on a seeded mix of 256 images (VOC-like sizes, camera sizes and random odd sizes) -> 416x416:
   algorithmic GB/s (source + destination bytes) and its fraction of the 7.7 TB/s HBM peak.
3. End to end on that mix (pinned host images -> detections, slim_yolo_v2 416x416): one ragged call, submit/wait with two
   calls in flight, and one call per distinct size (the grouping the image CLI used before).
4. Host cost of a ragged call's enqueue (descriptors + tables built and uploaded, one launch) against a uniform call's.
Kernel times are CUDA events over back-to-back launches; the working sets (369 MB / the mix) exceed the 126 MB L2.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import yolo_b200  # noqa: E402,F401
from yolo_b200 import build as yb_build, export as ex, lib  # noqa: E402

HBM_GBS = 7700.0
VOC_LIKE = [(375, 500), (500, 375), (333, 500), (480, 640), (240, 320), (416, 416), (832, 832), (720, 1280), (1080, 1920)]


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")]
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = "unknown (%s)" % e
    return info


def mix_shapes(n=256, seed=0):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        if rng.random() < 0.7:
            out.append(VOC_LIKE[int(rng.integers(len(VOC_LIKE)))])
        else:
            out.append((int(rng.integers(8, 650)) * 2 + 1, int(rng.integers(8, 950)) * 2 + 1))       # odd sizes
    return out


def parent_library(src_dir):
    """Compiles an earlier resize.cu into a side library exposing its uniform BGR launcher: resize_u8c3 where the source
    exports it, resize_u8bgr in sources from before it."""
    tmp = tempfile.mkdtemp(prefix="t_ragged_")
    wrap = os.path.join(tmp, "parent.cu")
    src = os.path.join(os.path.abspath(src_dir), "resize.cu")
    with open(src) as f:
        single = "cudaError_t resize_u8c3(" in f.read()
    head = ("yb::resize_u8c3((const uint8_t *)src, (size_t)n * sh * sw * 3, yb::RS_BGR, nullptr, n, sh, sw, " if single
            else "yb::resize_u8bgr((const uint8_t *)src, n, sh, sw, ")
    with open(wrap, "w") as f:
        f.write('#include "%s"\n' % src)
        f.write('extern "C" int parent_resize(const void *src, int n, int sh, int sw, void *dst, int dh, int dw, const void *xt, '
                'const void *yt, int sm, void *st) { return (int)%s(uint8_t *)dst, dh, dw, (const int2 *)xt, (const int4 *)yt, '
                'sm, (cudaStream_t)st); }\n' % head)
    so = os.path.join(tmp, "parent.so")
    subprocess.check_call([yb_build.nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
                           "-I" + os.path.join(ROOT, "include"), "-Xcompiler", "-fPIC", "-shared", "-cudart", "static", "-o", so, wrap])
    P = C.CDLL(so)
    P.parent_resize.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    return P


def tables(L, sh, sw, dh, dw):
    """The uniform kernel's tables (the layout ensure_resize_tables builds), from the exported tap programme."""
    ty = np.zeros((dh, 4), np.int32); tx = np.zeros((dw, 4), np.int32)
    L.yolo_b200_resize_taps(sh, dh, 0, ty.ctypes.data)
    L.yolo_b200_resize_taps(sw, dw, 1, tx.ctypes.data)
    y = np.stack([ty[:, 0], ty[:, 1], ty[:, 2] << 16, ty[:, 3] << 16], 1).astype(np.int32)
    x = np.stack([tx[:, 0] * 3, tx[:, 2] | (tx[:, 3] << 16)], 1).astype(np.int32)
    return torch.from_numpy(y).cuda(), torch.from_numpy(x).cuda()


def time_rounds(variants, rounds, reps, stream):
    """variants: name -> callable issuing one launch.  Alternates the variants (rotated order) every round; returns ms per
    launch of every round."""
    names = list(variants)
    res = {k: [] for k in names}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        order = names[r % len(names):] + names[:r % len(names)]
        for k in order:
            for _ in range(2):
                variants[k]()
            e0.record(stream)
            for _ in range(reps):
                variants[k]()
            e1.record(stream)
            e1.synchronize()
            res[k].append(e0.elapsed_time(e1) / reps)
    return res


def stats(v):
    v = np.asarray(v)
    return {"median_ms": float(np.median(v)), "min_ms": float(v.min()), "max_ms": float(v.max()), "rounds": len(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-src", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ragged_r3.json"))
    ap.add_argument("--rounds", type=int, default=15)
    args = ap.parse_args()
    rec = {"card": card()}
    print(rec["card"])
    ctx = lib.Context(0)
    L = ctx.L
    s = torch.cuda.Stream()
    torch.cuda.set_stream(s)
    ctx.set_stream(s.cuda_stream)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    B, SH, SW, H, W = 256, 480, 640, 416, 416

    # 1. uniform workload
    g = torch.Generator(device="cuda").manual_seed(0)
    src = torch.randint(0, 256, (B, SH, SW, 3), dtype=torch.uint8, device="cuda", generator=g)
    outs = {k: torch.zeros((B, H, W, 3), dtype=torch.uint8, device="cuda") for k in ("uniform", "parent")}
    variants = {"uniform": lambda: ctx.resize_u8bgr(src, B, SH, SW, outs["uniform"], H, W)}
    if args.parent_src:
        P = parent_library(args.parent_src)
        yt, xt = tables(L, SH, SW, H, W)
        variants["parent"] = lambda: P.parent_resize(src.data_ptr(), B, SH, SW, outs["parent"].data_ptr(), H, W, xt.data_ptr(),
                                                     yt.data_ptr(), sm, s.cuda_stream)
    res = time_rounds(variants, args.rounds, 20, s)
    torch.cuda.synchronize()
    for k in variants:
        assert torch.equal(outs[k], outs["uniform"]), "%s output differs from the uniform kernel's" % k
    ubytes = B * (SH * SW * 3 + H * W * 3)
    rec["uniform_workload"] = {"workload": "%d x %dx%d -> %dx%d" % (B, SH, SW, H, W), "algorithmic_bytes": ubytes,
                               "variants": {k: dict(stats(v), gbs=ubytes / (np.median(v) / 1e3) / 1e9) for k, v in res.items()}}
    print(json.dumps(rec["uniform_workload"], indent=1))
    del src, outs

    # 2. ragged kernel on the mix
    shapes = mix_shapes()
    rng = np.random.default_rng(1)
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]
    packed, hw = lib.pack_images(imgs)
    d_packed = torch.from_numpy(packed).cuda()
    d_out = torch.zeros((B, H, W, 3), dtype=torch.uint8, device="cuda")
    res = time_rounds({"ragged": lambda: ctx.resize_u8bgr_ragged(d_packed, hw, d_out, H, W)}, args.rounds, 10, s)
    mbytes = int(packed.size) + B * H * W * 3
    med = float(np.median(res["ragged"]))
    rec["ragged_mix"] = {"images": B, "distinct_sizes": len(set(shapes)), "source_bytes": int(packed.size), "algorithmic_bytes": mbytes,
                         **stats(res["ragged"]), "gbs": mbytes / (med / 1e3) / 1e9, "frac_of_hbm_peak": mbytes / (med / 1e3) / 1e9 / HBM_GBS}
    print(json.dumps(rec["ragged_mix"], indent=1))

    # 4. host cost of the enqueue (no synchronise inside the timed loop; the stream is drained between samples)
    def enqueue_us(fn, reps=50):
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        return float(np.median(ts) * 1e6)
    d_uni = torch.zeros((B, SH, SW, 3), dtype=torch.uint8, device="cuda")
    rec["host_enqueue_us"] = {"ragged_mix_256_images": enqueue_us(lambda: ctx.resize_u8bgr_ragged(d_packed, hw, d_out, H, W)),
                              "uniform_256_images": enqueue_us(lambda: ctx.resize_u8bgr(d_uni, B, SH, SW, d_out, H, W))}
    print(rec["host_enqueue_us"])
    del d_uni, d_packed, d_out

    # 3. end to end on the mix
    qnet = ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2, head_bias_shift=-3.0)
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.1, nms_thresh=0.5, max_det=1024)
    pin = torch.from_numpy(packed).pin_memory()
    md = 1024
    mk = lambda n: (torch.zeros((n, md, 8), dtype=torch.int32).pin_memory(), torch.zeros(n, dtype=torch.int32).pin_memory())   # noqa: E731

    def one_call(d, c):
        r = L.yolo_b200_forward_u8bgr_ragged(ctx._h, pin.data_ptr(), B, hw.ctypes.data, H, W, d.data_ptr(), c.data_ptr())
        assert r == 0, L.yolo_b200_last_error()

    groups = {}
    for i, sh in enumerate(shapes):
        groups.setdefault(sh, []).append(i)
    gin = {sh: torch.from_numpy(np.stack([imgs[i] for i in idx])).pin_memory() for sh, idx in groups.items()}
    gout = {sh: mk(len(idx)) for sh, idx in groups.items()}

    def grouped(counts_all):
        for sh, idx in groups.items():
            d, c = gout[sh]
            r = L.yolo_b200_forward_u8bgr_resize(ctx._h, gin[sh].data_ptr(), len(idx), sh[0], sh[1], H, W, d.data_ptr(), c.data_ptr())
            assert r == 0, L.yolo_b200_last_error()
            counts_all[idx] = c.numpy()

    d1, c1 = mk(B)
    cg = np.zeros(B, np.int32)
    for _ in range(2):                                    # warm-up (allocations, tables, module loads)
        one_call(d1, c1); grouped(cg)
    assert np.array_equal(c1.numpy(), cg), "one ragged call and the per-size calls disagree"
    reps = 5
    pairs = [mk(B) for _ in range(2)]
    t_one, t_grp, t_pair = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter(); one_call(d1, c1); t_one.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); grouped(cg); t_grp.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        tickets = []
        for k in range(8):                                # 8 batches, two in flight
            if len(tickets) == 2:
                ctx.wait(tickets.pop(0))
            d, c = pairs[k % 2]
            t = L.yolo_b200_submit_u8bgr_ragged(ctx._h, pin.data_ptr(), B, hw.ctypes.data, H, W, d.data_ptr(), c.data_ptr())
            assert t >= 0, L.yolo_b200_last_error()
            tickets.append(t)
        while tickets:
            ctx.wait(tickets.pop(0))
        t_pair.append((time.perf_counter() - t0) / 8)
    assert np.array_equal(pairs[0][1].numpy(), c1.numpy())
    rec["end_to_end"] = {"network": "slim_yolo_v2 416x416, contract P, conf 0.1, max_det 1024", "images_per_batch": B,
                         "one_ragged_call": {"median_ms": 1e3 * float(np.median(t_one)), "frames_per_s": B / float(np.median(t_one))},
                         "submit_wait_two_in_flight": {"median_ms_per_batch": 1e3 * float(np.median(t_pair)), "frames_per_s": B / float(np.median(t_pair))},
                         "one_call_per_size": {"calls": len(groups), "median_ms": 1e3 * float(np.median(t_grp)), "frames_per_s": B / float(np.median(t_grp))},
                         "note": "host images pinned; per-size batches pre-stacked in pinned memory outside the timed region; detections agree"}
    print(json.dumps(rec["end_to_end"], indent=1))
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
