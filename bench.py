#!/usr/bin/env python
"""bench.py — frames/sec of the fixed-point slim_yolo_v2 forward pass on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch of synthetic frames: 256 camera frames of 416x416 RGB444 (uint16,
the C path's input format, ov7670.h:203-230) per GPU (BASELINE.json configs[2]); random-init weights of the named
architecture quantised and calibrated by the reference's rules (yolo_b200.export.random_quantnet); contract F (the FPGA
shift programme), round-half-even.  The step is: RGB444 -> int8 LUT quantiser (fused into conv1), the ten conv layers,
decode, NMS.
Frames are independent, so ranks shard the batch with no data-path collective; only the detection lists are
gathered at the end of every step ("scaling": "weak").

Prints ONE JSON line (rank 0).  `value` = whole-job frames/s with inputs resident in HBM (CUDA events, max over
ranks); `e2e` = the same through the C-ABI host entry point with pinned HOST buffers (H2D of the frames and D2H of
the detections inside the timed region); `roofline` describes the dominant kernel; `cpu_baseline` is the CPU
oracle timed on this box's host cores on a bounded sample (rank 0, N=1 only).

--impl reference times the reference's own CPU implementation of the path: the C restatement under oracle/
(the C driver itself cannot run without the FPGA RTL, see DESIGN.md) with all host threads.

--scaling strong shards a FIXED global batch (--global-batch, default 2048 frames per step) over the GPUs instead of 256
frames per GPU (SURVEY.md 8d config 4).  At N = 1 the line also carries `other_configs`: the same step at the C path's
native geometry (240x320 RGB444), from fp32 NCHW input, and under contract P (the contract pinned on the reference module).

--dump-outputs DIR writes the detection lists of the last timed step (at N > 1, every rank's lists as collected on rank 0)
to DIR as .npy files (see dump_outputs).  Frames and weights are seeded, so two builds of the project run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

H = W = 416
BATCH = 256
METRIC = "frames/sec slim_yolo_v2 fixed-point"
WORKLOAD = "slim_yolo_v2 fixed-point batched inference, batch %d x 416x416 RGB444 camera frames per GPU (front-end quantiser + 10 conv layers + decode + NMS)"
CONF, NMS = 0.1, 0.5     # test.py:22-24 defaults
E2E_CHUNK = 128          # frames per copy / compute chunk of the streamed host path (tools/t_e2e_host.py: as fast as 64 on one GPU, 9 % faster with 4 GPUs copying at once)


def layer_work(qnet, h, w):
    """Algorithmic MACs and activation bytes per frame per layer (SURVEY.md 8d): in H*W*Cin + out H'*W'*Cout."""
    rows = []
    for (cin, cout, activ, pool) in qnet.layers:
        oh, ow = (h // 2, w // 2) if pool else (h, w)
        rows.append({"macs": h * w * 9 * cin * cout, "bytes": h * w * (4 if cin <= 4 else cin) + oh * ow * cout})
        h, w = oh, ow
    return rows


def peaks():
    """HBM GB/s and bf16 TFLOP/s from the driver-written MEASURED_PEAKS.json (else B200_PROFILING.md's fallback), and the
    INT8 tensor peak MEASURED on this pool's B200 with tools/micro/umma_peak.cu (148 persistent CTAs issuing
    tcgen05.mma.kind::i8 N=256 back to back; profiles/int8_peak_r2.json holds TOPS for a 4 ms burst and for 2 s sustained
    with the clock / power record).  The per-kernel fractions and the ~25 ms timed region use the BURST figure."""
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update({k: m[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in m})
        p["source"] = "measured"
    except Exception:
        pass
    p["int8_tops"], p["int8_source"] = 2.0 * p["bf16_tflops"], "2 x bf16 burst of MEASURED_PEAKS.json (%s)" % p["source"]
    try:
        with open(os.path.join(ROOT, "profiles", "int8_peak_r2.json")) as f:
            m = json.load(f)
        p["int8_tops"], p["int8_tops_sustained"] = float(m["int8_tops_burst"]), float(m["int8_tops_sustained"])
        p["int8_source"] = "measured_int8"
    except Exception:
        pass
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.t.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_qnet():
    import yolo_b200  # noqa: F401
    from yolo_b200 import export as ex
    # random-init weights of the named architecture, quantised by the reference's rule and calibrated (first-call rule,
    # slim_yolo_v2.py:22-27) on what the RGB444 front end delivers at scale_a[0] = 0 (the shipped table value)
    return ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2, calib_input="rgb444")


def oracle_frames(qnet, frames_u16):
    """The CPU restatement of the whole path on RGB444 frames (front-end LUT, backbone, head). Returns detections/frame."""
    import oracle_lib as ol
    x8 = ol.quantize_rgb444(frames_u16, qnet.sa[0])
    outs, _ = ol.backbone(qnet, x8, contract=0)
    cnt = []
    for i in range(frames_u16.shape[0]):
        _, c = ol.head_python(outs[-1][i], 5, 2, qnet.sa[10], qnet.anchors, 16, H, W, CONF, NMS)
        cnt.append(c)
    return cnt


def cpu_oracle_fps(qnet, seconds_budget):
    """Oracle on a bounded sample of the workload, all host threads (OpenMP over rows)."""
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    import yolo_b200  # noqa: F401
    from yolo_b200 import export as ex
    import oracle_lib as ol
    cores = ol.set_threads()
    done, t0 = 0, time.perf_counter()
    while True:
        oracle_frames(qnet, ex.synthetic_frames_rgb444(1, H, W, seed=9000 + done))
        done += 1
        el = time.perf_counter() - t0
        if el >= seconds_budget or done >= 64:
            break
    return done / el, cores, done


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU implementation of the path on this box's host cores.  The C driver itself
    cannot run (FPGA RTL and weight.h are not in the reference, DESIGN.md section 5), so this is the oracle port."""
    if rank != 0:
        return
    # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: the CPU arm must use every host thread whether it is
    # launched directly or under torchrun (set before the OpenMP runtime of liboracle.so starts)
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    import yolo_b200  # noqa: F401
    from yolo_b200 import export as ex
    import oracle_lib as ol
    qnet = make_qnet()
    ol.build()
    cores = ol.set_threads()
    frames_per_step = 4
    xs = ex.synthetic_frames_rgb444(frames_per_step, H, W, seed=123)
    for _ in range(max(1, min(args.warmup, 2))):
        oracle_frames(qnet, xs)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_frames(qnet, xs)
    dt = time.perf_counter() - t0
    fps = args.steps * frames_per_step / dt
    sample = "%d frames/step of the 416x416 RGB444 workload (front-end LUT + backbone + head), OpenMP over rows, %d host threads" % (frames_per_step, cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int8", "data": "synthetic",
        "config": {"workload": WORKLOAD % BATCH + " (bounded sample: %d frames per step)" % frames_per_step,
                   "frames_per_step": frames_per_step, "contract": "F/RNE"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def ol_quantize(x_nchw, sa):
    """float NCHW -> int8 NHWC4 by a_tracker_in's rule (numpy; input preparation for the yolo_v2 line, outside any timed region)."""
    q = np.clip(np.rint(x_nchw.astype(np.float32) * np.float32(2.0 ** sa)), -128, 127).astype(np.int8)
    out = np.zeros((q.shape[0], q.shape[2], q.shape[3], 4), np.int8)
    out[..., :3] = q.transpose(0, 2, 3, 1)
    return out


def yolo_v2_maps(qnet, h, w):
    """Input map size of every layer of a graph network (for the MAC count)."""
    pre, post, dims = {}, {}, []
    for l, ((cin, cout, activ, pool), g) in enumerate(zip(qnet.layers, qnet.graph)):
        if l == 0:
            d = (h, w)
        else:
            src = g.get("in_from", 0) - 1 if g.get("in_from", 0) else l - 1
            d = pre[src] if g.get("in_from", 0) else post[src]
        dims.append(d)
        pre[l] = d
        post[l] = (d[0] // 2, d[1] // 2) if pool else d
    return dims


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, counts, records, max_det):
    """Writes the detection lists of one step (counts [frames], records int32 [sum(counts), 8] in frame order, as the
    C-ABI's yolo_b200_det) to out_dir as float32 .npy files: frames (index of each dumped frame), counts, and per
    detection boxes (x1, y1, x2, y2), scores, classes, anchor_index.  The integer fields (frames, counts, classes,
    anchor_index) are float32 too, like every dumped array, and exact: they stay far below 2**24.  When max_det records per frame could exceed
    DUMP_BYTES, a fixed seeded sample of frames is written; it does not depend on the results, so two builds of the
    project dump the same frames and can be compared output for output."""
    n = len(counts)
    k = min(n, DUMP_BYTES // (max_det * 7 * 4 + 2 * 4))
    frames = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    start = np.concatenate([[0], np.cumsum(counts, dtype=np.int64)])
    assert start[-1] == len(records)
    rec = np.ascontiguousarray(records[np.concatenate([np.arange(start[f], start[f + 1]) for f in frames]).astype(np.int64)])
    os.makedirs(out_dir, exist_ok=True)
    out = {"frames": frames, "counts": np.asarray(counts)[frames], "boxes": rec.view(np.float32)[:, :4],
           "scores": rec.view(np.float32)[:, 4], "classes": rec[:, 5], "anchor_index": rec[:, 6]}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def time_steps(stream, fn, warm, steps):
    import torch
    for i in range(warm):
        fn(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        fn(i)
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="frames per GPU per step (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--global-batch", type=int, default=2048, help="frames per step over all GPUs (strong scaling)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip other_configs / sparse head / image front end")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the detections of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what --impl b200 computed")
    sys.dont_write_bytecode = True     # the tree may be read-only: nothing is cached next to the sources
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    import yolo_b200  # noqa: F401
    from yolo_b200 import export as ex
    from yolo_b200 import lib, runner

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    # stdout carries exactly ONE JSON line: anything a library prints there (NCCL's version banner, whatever NCCL_DEBUG says)
    # is sent to stderr; the line itself is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":   # keeps NCCL's banner out of stdout (one JSON line)
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    strong = args.scaling == "strong"
    if strong:
        lo, hi = runner.shard_range(args.global_batch, rank, world)
        B = hi - lo
    else:
        B = args.batch
    qnet = make_qnet()
    MAXDET = 4096
    ctx = lib.Context(local)
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=CONF, nms_thresh=NMS, max_det=MAXDET)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)

    # synthetic camera frames, RGB444 (the C path's input format), 3 alternating batches of 88.6 MB each; a step also
    # streams ~1.3 GB of feature maps, far more than the 126 MB L2
    n_sets = 3
    host_sets = [torch.from_numpy(ex.synthetic_frames_rgb444(B, H, W, seed=100 * rank + s).view(np.int16)).pin_memory() for s in range(n_sets)]
    dev_sets = [h.cuda(non_blocking=True) for h in host_sets]
    n_anchors = (H // 16) * (W // 16) * 5                       # bounds any per-frame detection count
    # N > 1: every rank's lists are collected on rank 0 by copy-engine peer writes of their filled part (runner.PeerCollector)
    coll = runner.PeerCollector(ctx, B, MAXDET, n_anchors, torch.device("cuda", local)) if world > 1 else None
    d_dets = torch.zeros((B, MAXDET, 8), dtype=torch.int32, device="cuda")
    d_counts = torch.zeros((B,), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()

    def step(i):
        if coll is None:
            ctx.forward_rgb444_dev(dev_sets[i % n_sets], B, H, W, d_dets, d_counts)
        else:
            buf = coll.buffers(i)
            ctx.forward_rgb444_dev(dev_sets[i % n_sets], B, H, W, buf.dets, buf.counts)
            coll.launch(i)          # packs step i; ships step i - 1 while step i computes

    def barrier():
        if coll is not None:
            coll.finish()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(args.steps):
        step(args.warmup + i)
    if coll is not None:
        coll.finish()                  # the last lists have landed on rank 0: the collection is inside the timed region
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count() - l0
    if args.dump_outputs and rank == 0:    # before the per-kernel timing passes below overwrite d_dets / d_counts
        if coll is None:
            filled = torch.arange(MAXDET, device="cuda")[None, :] < d_counts[:, None]
            counts, records = d_counts.cpu().numpy(), d_dets[filled].cpu().numpy()
        else:                              # every rank's lists as they arrived on rank 0
            parts = coll.collected(args.warmup + args.steps - 1)
            counts = np.concatenate([np.diff(off.cpu().numpy()) for off, _ in parts])
            records = np.concatenate([rec.cpu().numpy() for _, rec in parts])
        dump_outputs(args.dump_outputs, counts, records, MAXDET)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    total_frames = (args.global_batch if strong else world * B) * args.steps
    fps = total_frames / (ms / 1e3)
    collected = None
    if coll is not None:
        mean_dets = float(coll.bufs[(args.warmup + args.steps - 1) % coll.depth].counts.float().mean().item())
        if rank == 0:   # what arrived on rank 0 for the last step: records per rank
            collected = [int(off[-1].item()) for off, rec in coll.collected(args.warmup + args.steps - 1)]
            assert all(c >= 0 for c in collected)
        sent = torch.tensor([coll.sent_bytes / max(1, args.warmup + args.steps)], dtype=torch.float64, device="cuda")
        dist.all_reduce(sent, op=dist.ReduceOp.SUM)
        collect_bytes = float(sent.item())
    else:
        mean_dets = float(d_counts.float().mean().item())
        collect_bytes = 0.0

    # ---- per-kernel device times (CUDA events on the launching stream) -> dominant kernel and its roofline
    # (the RGB444 -> int8 quantiser is fused into conv1's tile load: conv1 reads the 2-byte camera pixels)
    names = ["conv1", "conv2", "conv3_1", "conv3_2", "conv4_1", "conv4_2", "conv5", "conv6", "conv7", "pred", "head"]
    reps = 5
    per = np.zeros(len(names))
    ctx.enable_timing(True)
    for i in range(reps):
        ctx.forward_rgb444_dev(dev_sets[i % n_sets], B, H, W, d_dets, d_counts)
        per += np.array(ctx.layer_times_ms())
    per /= reps
    ctx.enable_timing(False)
    # clocks / throttle reasons sampled from the start of the timed region to the end of the per-kernel timing passes (the
    # timed region alone lasts tens of milliseconds, too short for nvidia-smi's sampling period); stopped before the
    # end-to-end region because nvidia-smi polling perturbs host-side copies
    clocks = sampler.stop() if rank == 0 else None
    pk = peaks()
    work = layer_work(qnet, H, W)
    int8_peak_tops = pk["int8_tops"]                              # measured tcgen05 kind::i8 burst peak (profiles/int8_peak_r2.json)
    # algorithmic (MACs, bytes) per frame for every kernel of the step
    work[0]["bytes"] -= 2 * H * W      # conv1 reads RGB444 (2 B/pixel), not NHWC4
    rows = work + [{"macs": 0, "bytes": (H // 16) * (W // 16) * 48 + int(mean_dets) * 32}]
    top = int(np.argmax(per))
    t_top = per[top] / 1e3
    ops = 2.0 * rows[top]["macs"] * B
    byts = rows[top]["bytes"] * B
    tensor_bound = ops / (int8_peak_tops * 1e12) > byts / (pk["hbm_gbs"] * 1e9)
    if tensor_bound:
        roof = {"bound": "tensor", "achieved": ops / t_top / 1e12, "peak": int8_peak_tops, "unit": "TFLOP/s",
                "note": "int8 ops (2*MAC) counted as FLOPs; peak = %s" % pk["int8_source"]}
    else:
        roof = {"bound": "hbm", "achieved": byts / t_top / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "note": "algorithmic bytes (input map + output map, or prediction map + detection records for the head) / "
                        "CUDA-event time; peak = hbm_gbs of MEASURED_PEAKS.json (%s)" % pk["source"]}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["kernel"] = names[top]
    roof["kernel_ms"] = float(per[top])
    roof["peak_source"] = pk["int8_source"]
    roof["int8_peak_tops"] = {"burst_measured": pk.get("int8_tops"), "sustained_measured": pk.get("int8_tops_sustained"),
                              "two_x_bf16_burst": 2.0 * pk["bf16_tflops"], "two_x_bf16_sustained": 2.0 * pk["bf16_tflops_sustained"]}
    roof["traffic"] = None
    for tf in ("traffic_r2.json", "traffic_r1.json"):   # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
        try:
            with open(os.path.join(ROOT, "profiles", tf)) as f:
                tr = json.load(f)
            if names[top] in tr and tr.get("batch") == B:
                roof["traffic"] = tr[names[top]]
                roof["traffic_source"] = "profiles/" + tf
                break
        except Exception:
            pass
    bf2 = 2.0 * pk["bf16_tflops"]
    per_kernel = {}
    for n_, t_, r_ in zip(names, per, rows):
        tb = 2.0 * r_["macs"] * B / (int8_peak_tops * 1e12)
        hb = r_["bytes"] * B / (pk["hbm_gbs"] * 1e9)
        tb2 = 2.0 * r_["macs"] * B / (bf2 * 1e12)
        per_kernel[n_] = {"ms": round(float(t_), 4), "bound": "tensor" if tb > hb else "hbm",
                          "frac": round(max(tb, hb) / (float(t_) / 1e3), 4) if t_ > 0 else None,
                          "frac_vs_2x_bf16": round(max(tb2, hb) / (float(t_) / 1e3), 4) if t_ > 0 else None}
    roof["per_kernel"] = per_kernel
    t_roof = sum(max(2.0 * r["macs"] / (int8_peak_tops * 1e12), r["bytes"] / (pk["hbm_gbs"] * 1e9)) for r in rows)
    t_roof2 = sum(max(2.0 * r["macs"] / (bf2 * 1e12), r["bytes"] / (pk["hbm_gbs"] * 1e9)) for r in rows)
    per_frame_s = ms / 1e3 / (B * args.steps)
    roof["network_t_roof_us_per_frame"] = t_roof * 1e6
    roof["network_frac_of_roofline"] = t_roof / per_frame_s
    roof["network_frac_vs_2x_bf16"] = t_roof2 / per_frame_s

    # ---- e2e: the C-ABI host entry point, pinned host frames in, detections out (copies inside the timed region;
    #      the library pipelines them against the kernels chunk by chunk)
    h_dets = torch.zeros((B, MAXDET, 8), dtype=torch.int32).pin_memory()
    h_counts = torch.zeros((B,), dtype=torch.int32).pin_memory()
    L = ctx.L

    def e2e_step(i):
        rc = L.yolo_b200_forward_rgb444(ctx._h, host_sets[i % n_sets].data_ptr(), B, H, W, h_dets.data_ptr(), h_counts.data_ptr())
        if rc:
            raise RuntimeError(L.yolo_b200_last_error())
    e2e_steps = max(3, min(args.steps, 10))
    for i in range(2):
        e2e_step(i)
    barrier()
    l1 = ctx.launch_count()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    barrier()
    e2e_blocking_s = time.perf_counter() - t0
    e2e_launches = ctx.launch_count() - l1
    # the same K steps as a stream of batches: yolo_b200_submit_rgb444 / yolo_b200_wait with two calls in flight, each with its
    # own pinned output buffers (the tail of step i overlaps the host-to-device copy of step i + 1; every step's frames go
    # host -> device and every step's detections device -> host inside the timed region, the last wait included)
    out_bufs = [(h_dets, h_counts), (torch.zeros((B, MAXDET, 8), dtype=torch.int32).pin_memory(), torch.zeros((B,), dtype=torch.int32).pin_memory())]
    ctx.set_host_chunk(E2E_CHUNK)

    def e2e_stream(k0, k):
        tickets = []
        for i in range(k0, k0 + k):
            if len(tickets) == 2:
                ctx.wait(tickets.pop(0))
            d_, c_ = out_bufs[i % 2]
            t = L.yolo_b200_submit_rgb444(ctx._h, host_sets[i % n_sets].data_ptr(), B, H, W, d_.data_ptr(), c_.data_ptr())
            if t < 0:
                raise RuntimeError(L.yolo_b200_last_error())
            tickets.append(t)
        while tickets:
            ctx.wait(tickets.pop(0))
    e2e_stream(0, 3)
    barrier()
    t0 = time.perf_counter()
    e2e_stream(3, e2e_steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    ctx.set_host_chunk(64)
    if world > 1:
        t = torch.tensor([e2e_s, e2e_blocking_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s, e2e_blocking_s = float(t[0].item()), float(t[1].item())
    e2e_fps = (args.global_batch if strong else world * B) * e2e_steps / e2e_s
    e2e_blocking_fps = (args.global_batch if strong else world * B) * e2e_steps / e2e_blocking_s
    # what the end-to-end number is bounded by: the host -> device link, measured here with every rank copying its pinned batch at the
    # same time (GB/s per GPU; at N > 1 the ranks share the host's PCIe switches and memory controllers)
    barrier()
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record(stream)
    for i in range(4):
        dev_sets[i % n_sets].copy_(host_sets[i % n_sets], non_blocking=True)
    h1.record(stream)
    torch.cuda.synchronize()
    h2d_gbs = 4 * host_sets[0].numel() * 2 / (h0.elapsed_time(h1) / 1e3) / 1e9
    if world > 1:
        t = torch.tensor([h2d_gbs], dtype=torch.float64, device="cuda")
        allg = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allg, t)
        h2d_all = [round(float(x.item()), 1) for x in allg]
    else:
        h2d_all = [round(h2d_gbs, 1)]
    h2d_bound_fps = sum(g * 1e9 / (H * W * 2) for g in h2d_all)     # frames/s the measured links could carry (2 bytes per pixel)
    # bytes the library copies back per step: counts + one strided copy as wide as the batch's largest count
    hc = h_counts.numpy()
    d2h_bytes = int(4 * B + B * min(int(hc.max()), MAXDET) * 32)
    assert int(h_counts.sum()) > 0 or mean_dets == 0

    # ---- secondary: the same network with a trained-like sparse head (objectness bias - 5, SURVEY 8d)
    secondary = rank == 0 and world == 1 and not args.no_secondary and not strong
    # ---- other configurations of SURVEY 8d config 3 (N = 1): the C path's native geometry, fp32 input, contract P
    other = None
    if secondary:
        other = {}

        def run_cfg(name, fn, frames, note):
            ms_ = time_steps(stream, fn, 3, 10)
            other[name] = {"value": frames / (ms_ / 1e3), "unit": "frames/s", "ms_per_step": ms_, "frames_per_step": frames, "note": note}
        # 240 x 320 RGB444: what the camera delivers to yolo_forward (yolo_forward.c:1194-1197), shipped-style network calibrated at that size
        q240 = ex.random_quantnet(seed=0, calib_hw=(240, 320), calib_frames=2, calib_input="rgb444")
        ctx.load_quantnet(q240, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=CONF, nms_thresh=NMS, max_det=MAXDET)
        d240 = torch.from_numpy(ex.synthetic_frames_rgb444(B, 240, 320, seed=7).view(np.int16)).cuda()
        run_cfg("rgb444_240x320_contract_F", lambda i: ctx.forward_rgb444_dev(d240, B, 240, 320, d_dets, d_counts), B,
                "%d RGB444 frames of 240x320 (the C path's camera geometry), contract F/RNE, dense random-init head" % B)
        del d240
        # fp32 NCHW input at 416 x 416 (the Python path's input, test.py:79-80), contract P = the arithmetic pinned on the reference module
        qp = ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2)
        ctx.load_quantnet(qp, contract=lib.CONTRACT_P, conf_thresh=CONF, nms_thresh=NMS, max_det=MAXDET)
        xf = ex.synthetic_frames_f32(B, H, W, seed=11).cuda()
        run_cfg("f32_416x416_contract_P", lambda i: ctx.forward_f32_dev(xf, B, H, W, d_dets, d_counts), B,
                "%d float32 NCHW frames of 416x416 (531 MB read per step by the quantiser), contract P (PyTorch fake-quant, pinned on the reference module)" % B)
        ovf = ctx.overflow_count()
        other["f32_416x416_contract_P"]["int8_saturations"] = int(ovf)
        del xf
        # RGB444 416 x 416 under contract P (same workload as the headline, the pinned contract)
        qpr = make_qnet()
        ctx.load_quantnet(qpr, contract=lib.CONTRACT_P, conf_thresh=CONF, nms_thresh=NMS, max_det=MAXDET)
        run_cfg("rgb444_416x416_contract_P", lambda i: ctx.forward_rgb444_dev(dev_sets[i % n_sets], B, H, W, d_dets, d_counts), B,
                "the headline workload under contract P")

        # BASELINE configs[4]: yolo_v2 (darknet19 backbone, 20 classes) BN-folded fixed point at 416x416, batch 64 per GPU:
        # 14.68 GMAC per frame, 1x1 layers, 512 / 1024 / 1280 channels, route + reorg + concat (tests: test_yolo_v2_*)
        BV = 64
        qv = ex.random_quantnet_yolo_v2(seed=0, calib_hw=(H, W), calib_frames=1)
        ctx.load_quantnet(qv, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=CONF, nms_thresh=NMS, max_det=1024)
        xv = torch.from_numpy(ol_quantize(ex.synthetic_frames_f32(BV, H, W, seed=13).numpy(), qv.sa[0])).cuda()
        dv = torch.zeros((BV, 1024, 8), dtype=torch.int32, device="cuda")
        cv = torch.zeros((BV,), dtype=torch.int32, device="cuda")
        sp0 = ctx.slow_path_count()
        run_cfg("yolo_v2_416x416_contract_F", lambda i: ctx.forward_int8_dev(xv, BV, H, W, dv, cv), BV,
                "%d int8 NHWC4 frames of 416x416 through the 23-layer yolo_v2 graph (29.4 GOP per frame), contract F/RNE" % BV)
        gmac = sum(h_ * w_ * (g_.get("ksize", 3) ** 2) * ci * co for (ci, co, _, _), g_, (h_, w_) in zip(qv.layers, qv.graph, yolo_v2_maps(qv, H, W)))
        yv = other["yolo_v2_416x416_contract_F"]
        yv["gmac_per_frame"] = gmac / 1e9
        yv["tensor_tops"] = 2.0 * gmac * yv["value"] / 1e12
        yv["frac_of_int8_peak"] = yv["tensor_tops"] / int8_peak_tops
        yv["dot_product_fallback_launches_per_step"] = (ctx.slow_path_count() - sp0) / 13.0
        yv["mean_detections_per_frame"] = float(cv.float().mean().item())
        del xv, dv, cv

    sparse = None
    if secondary:
        qs = ex.random_quantnet(seed=0, calib_hw=(H, W), calib_frames=2, calib_input="rgb444", head_bias_shift=-5.0)
        ctx.load_quantnet(qs, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=CONF, nms_thresh=NMS, max_det=MAXDET)
        for i in range(3):
            ctx.forward_rgb444_dev(dev_sets[i % n_sets], B, H, W, d_dets, d_counts)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for i in range(10):
            ctx.forward_rgb444_dev(dev_sets[i % n_sets], B, H, W, d_dets, d_counts)
        s1.record(stream)
        torch.cuda.synchronize()
        sparse = {"value": B * 10 / (s0.elapsed_time(s1) / 1e3), "unit": "frames/s",
                  "mean_detections_per_frame": float(d_counts.float().mean().item()),
                  "note": "same step with pred objectness bias - 5 before quantisation (sparse detections of a trained network)"}
        for i in range(2):
            e2e_step(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            e2e_step(i)
        torch.cuda.synchronize()
        sparse["e2e"] = B * e2e_steps / (time.perf_counter() - t0)

    # ---- secondary: the reference's image front end on the GPU (cv2.resize of base_transform, data/__init__.py:36, on
    #      480x640 BGR frames -> 416x416, then the fused normalise/quantise first layer): the resize kernel alone against
    #      HBM, and the host entry point with the camera-size images in pinned memory
    front = None
    if secondary:
        SH, SW = 480, 640
        g = torch.Generator().manual_seed(5)
        h_imgs = torch.randint(0, 256, (B, SH, SW, 3), dtype=torch.uint8, generator=g).pin_memory()
        d_imgs = h_imgs.cuda()
        d_small = torch.empty((B, H, W, 3), dtype=torch.uint8, device="cuda")
        for i in range(3):
            ctx.resize_u8bgr(d_imgs, B, SH, SW, d_small, H, W)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for i in range(10):
            ctx.resize_u8bgr(d_imgs, B, SH, SW, d_small, H, W)
        s1.record(stream)
        torch.cuda.synchronize()
        r_ms = s0.elapsed_time(s1) / 10
        r_bytes = B * (SH * SW * 3 + H * W * 3)
        for i in range(3):
            ctx.forward_u8bgr_resize_dev(d_imgs, B, SH, SW, H, W, d_dets, d_counts)
        s0.record(stream)
        for i in range(10):
            ctx.forward_u8bgr_resize_dev(d_imgs, B, SH, SW, H, W, d_dets, d_counts)
        s1.record(stream)
        torch.cuda.synchronize()
        f_ms = s0.elapsed_time(s1) / 10

        def front_step():
            rc = L.yolo_b200_forward_u8bgr_resize(ctx._h, h_imgs.data_ptr(), B, SH, SW, H, W, h_dets.data_ptr(), h_counts.data_ptr())
            if rc:
                raise RuntimeError(L.yolo_b200_last_error())
        for i in range(2):
            front_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            front_step()
        torch.cuda.synchronize()
        front = {"workload": "%d BGR uint8 frames of %dx%d -> bilinear resize to %dx%d (cv2.resize semantics) + forward (sparse head)" % (B, SH, SW, H, W),
                 "resize_kernel_ms": r_ms, "resize_gbs": r_bytes / (r_ms / 1e3) / 1e9, "resize_frac_of_hbm": r_bytes / (r_ms / 1e3) / 1e9 / pk["hbm_gbs"],
                 "value": B / (f_ms / 1e3), "unit": "frames/s",
                 "e2e": B * e2e_steps / (time.perf_counter() - t0), "h2d_bytes_per_step": int(h_imgs.numel())}
        del d_imgs, d_small, h_imgs

    cpu_torch = None
    try:    # the reference's PyTorch CPU path cannot travel to the GPU box: timed in the build container (oracle/time_reference_pytorch.py)
        with open(os.path.join(ROOT, "profiles", "ref_pytorch_cpu_r2.json")) as f:
            rp = json.load(f)
        best = max((r for r in rp["runs"] if r["h"] == H and r["w"] == W), key=lambda r: r["frames_per_s"])
        cpu_torch = {"value": best["frames_per_s"], "unit": "frames/s", "cores": best["threads"], "kind": "reference",
                     "sample": "reference SlimYOLOv2_quantize_bnfuse.forward(quantization=True), batch 1 at %dx%d, 10 timed calls, measured in the "
                               "BUILD CONTAINER (%s, torch %s; /root/reference does not exist on the GPU box)" % (H, W, rp["cpu"], rp["torch"]),
                     "all_runs": rp["runs"]}
    except Exception:
        pass
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            v, cores, nfr = cpu_oracle_fps(qnet, args.cpu_seconds)
            cpu = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                   "sample": "%d frames of the same 416x416 RGB444 workload (front-end LUT + backbone + head), OpenMP over rows" % nfr}
        except Exception as e:  # the oracle is test infrastructure; its absence must not kill the GPU number
            cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "port", "sample": "oracle unavailable: %s" % e}

    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps({
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "int8", "data": "synthetic",
            "config": {"workload": WORKLOAD % B,
                       "frames_per_gpu_per_step": B, "global_frames_per_step": args.global_batch if strong else B * world, "contract": "F/RNE",
                       "weights": "random-init, reference quantisation + calibration rules (export.random_quantnet seed 0, calibrated on RGB444 input)",
                       "head": "conf %.2f nms %.2f, mean %.0f detections/frame (random-init dense worst case)" % (CONF, NMS, mean_dets),
                       "l2": "3 alternating input batches of 88.6 MB; each step also streams ~1.3 GB of feature maps (> 126 MB L2)",
                       "parallelism": "frames sharded over %d GPU(s); filled detection lists collected on rank 0 by copy-engine peer writes (no collective kernel)" % world,
                       "collection": None if coll is None else {"bytes_per_step_all_ranks": collect_bytes, "records_on_rank0_last_step": collected}},
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": int(host_sets[0].numel() * 2),
                    "d2h_bytes_per_step": d2h_bytes, "steps": e2e_steps,
                    "api": "yolo_b200_submit_rgb444 + yolo_b200_wait, two calls in flight (pinned host buffers; every step copies its 256 frames host -> device in %d-frame chunks overlapped with the convolution layers, runs decode + NMS on a second stream and copies the filled part of its lists back; the tail of step i overlaps the copy of step i + 1; timed to the last wait)" % E2E_CHUNK,
                    "h2d_gbs_per_gpu_concurrent": h2d_all, "h2d_bound_frames_per_s": h2d_bound_fps, "frac_of_h2d_bound": e2e_fps / h2d_bound_fps,
                    "blocking_call": {"value": e2e_blocking_fps, "unit": "frames/s", "api": "yolo_b200_forward_rgb444, one call at a time (64-frame chunks)"},
                    "gpu_launches": int(e2e_launches)},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "cpu_baseline_pytorch": cpu_torch,
            "other_configs": other, "sparse_head": sparse, "image_front_end": front,
        }) + "\n").encode())
    if coll is not None:
        dist.barrier()
        coll.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
