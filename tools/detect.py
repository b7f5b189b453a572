#!/usr/bin/env python
"""Image detection CLI for the fixed-point slim_yolo_v2 path on the GPU: the counterpart of the reference's test.py /
demo.py image mode for `-v slim_yolo_v2_q_bf` (test.py:13-99,165-181; demo.py:99-120), with the same flags where they
apply.  Every image goes through the whole hot path on the device: the uint8 BGR image (resized on the GPU with cv2.resize semantics, as
BaseTransform does, data/__init__.py:36) is normalised, quantised, convolved, decoded and NMS-ed by libyolo_b200.so.

    python tools/detect.py --trained_model slim_yolo_v2_retune_quantize1.pth --images dir/ -size 416 --out output/
    python tools/detect.py --trained_model random --images synthetic:4          (no checkpoint / no images at hand)
    python tools/detect.py --trained_model ckpt.pth --video clip.avi --batch 32  (demo.py's video / camera modes, batched)
    python tools/detect.py --yuv clip.nv12 --yuv_format nv12 --yuv_size 1920x1080   (raw decoder / webcam frames)
    python tools/detect.py --bayer clip.raw --bayer_pattern rggb --bayer_size 640x480  (raw sensor frames)
"""
import argparse
import glob
import os
import sys
import time

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import yolo_b200  # noqa: E402,F401
from yolo_b200 import export as ex, lib  # noqa: E402

MASK_CLASSES = ("face", "face_mask")                         # data/voc_mask.py:22-24
CLASS_COLORS = [(0, 0, 255), (0, 255, 0)]


def vis(img, bboxes, scores, cls_inds, thresh):
    """test.py:34-69 (dataset 'mask' branch)."""
    for i, box in enumerate(bboxes):
        if scores[i] > thresh:
            xmin, ymin, xmax, ymax = [int(v) for v in box]
            c = CLASS_COLORS[int(cls_inds[i]) % len(CLASS_COLORS)]
            cv2.rectangle(img, (xmin, ymin), (xmax, ymax), c, 1)
            cv2.rectangle(img, (xmin, abs(ymin) - 20), (xmax, ymin), c, -1)
            cv2.putText(img, MASK_CLASSES[int(cls_inds[i]) % len(MASK_CLASSES)], (xmin, ymin - 5), cv2.FONT_HERSHEY_SIMPLEX, 0.5, (0, 0, 0), 1)
    return img


def run_video(ctx, args, size):
    """demo.py video / camera modes (:60-96, :123-158) with the frames batched: `--batch` frames are read, go through
    yolo_b200_forward_u8bgr_resize in one call (resize, normalise, quantise, network, decode, NMS on the GPU), are annotated
    and appended to <out>/detections.avi (MJPG, the source's frame size and rate)."""
    cap = cv2.VideoCapture(int(args.video) if args.video.isdigit() else args.video)
    if not cap.isOpened():
        raise SystemExit("cannot open video source %s" % args.video)
    os.makedirs(args.out, exist_ok=True)
    fps = cap.get(cv2.CAP_PROP_FPS) or 25.0
    writer, frames, t_dev, done = None, 0, 0.0, False
    while not done:
        batch = []
        while len(batch) < args.batch:
            ok, frame = cap.read()
            if not ok or (args.max_frames and frames + len(batch) >= args.max_frames):
                done = True
                break
            batch.append(frame)
        if not batch:
            break
        t0 = time.time()
        dets, counts = ctx.forward_u8bgr_resize(np.stack(batch), size)
        t_dev += time.time() - t0
        for k, im in enumerate(batch):
            boxes, scores, cls, _ = lib.dets_to_arrays(dets[k], int(min(counts[k], 1024)))
            h, w = im.shape[:2]
            out = vis(im, boxes * np.array([[w, h, w, h]], dtype=np.float32), scores, cls, args.visual_threshold)   # demo.py:143-149
            if writer is None:
                writer = cv2.VideoWriter(os.path.join(args.out, "detections.avi"), cv2.VideoWriter_fourcc(*"MJPG"), fps, (w, h))
            writer.write(out)
        frames += len(batch)
    cap.release()
    if writer is not None:
        writer.release()
    print("%d frames, %.1f ms in yolo_b200_forward_u8bgr_resize (%.0f frames/s incl. copies)" % (frames, 1e3 * t_dev, frames / max(t_dev, 1e-9)))


YUV_FORMATS = {"nv12": lib.YUV_NV12, "i420": lib.YUV_I420, "yuyv": lib.YUV_YUYV}
YUV_CV2 = {"nv12": cv2.COLOR_YUV2BGR_NV12, "i420": cv2.COLOR_YUV2BGR_I420, "yuyv": cv2.COLOR_YUV2BGR_YUYV}
BAYER_PATTERNS = {"rggb": lib.BAYER_RGGB, "bggr": lib.BAYER_BGGR, "grbg": lib.BAYER_GRBG, "gbrg": lib.BAYER_GBRG}
BAYER_CV2 = {"rggb": cv2.COLOR_BayerRGGB2BGR, "bggr": cv2.COLOR_BayerBGGR2BGR, "grbg": cv2.COLOR_BayerGRBG2BGR, "gbrg": cv2.COLOR_BayerGBRG2BGR}


def run_raw(ctx, args, size, path, shape, sh, sw, submit, cv2_code, fps, api):
    """Raw video as `ffmpeg -f rawvideo` writes it (frames of `shape` back to back, no header): each batch of --batch frames
    goes to the GPU as it is (pinned) through submit(frames, size, dets, counts), which converts, resizes, normalises,
    quantises, convolves, decodes and NMS-es there, with two batches in flight.  The host converts with cvtColor (cv2_code)
    only to draw <out>/detections.avi (MJPG, the source size sh x sw, fps)."""
    fbytes = int(np.prod(shape))
    md = 1024
    os.makedirs(args.out, exist_ok=True)
    writer = cv2.VideoWriter(os.path.join(args.out, "detections.avi"), cv2.VideoWriter_fourcc(*"MJPG"), fps, (sw, sh))
    state = {"frames": 0}

    def finish(job):
        ticket, frames, dets, counts = job
        ctx.wait(ticket)
        for k in range(len(frames)):
            boxes, scores, cls, _ = lib.dets_to_arrays(dets[k], int(min(counts[k], md)))
            bgr = cv2.cvtColor(frames[k].numpy(), cv2_code)                                  # for drawing only
            writer.write(vis(bgr, boxes * np.array([[sw, sh, sw, sh]], dtype=np.float32), scores, cls, args.visual_threshold))
            print("frame %d: %d detections" % (state["frames"], len(scores)))
            state["frames"] += 1

    t0, inflight = time.time(), []
    with open(path, "rb") as f:
        while True:
            want = args.batch if not args.max_frames else min(args.batch, args.max_frames - state["frames"] - sum(len(j[1]) for j in inflight))
            if want <= 0:
                break
            raw = f.read(want * fbytes)
            n = len(raw) // fbytes
            if n == 0:
                break
            frames = torch.from_numpy(np.frombuffer(raw[:n * fbytes], dtype=np.uint8).reshape((n,) + shape).copy()).pin_memory()
            dets = np.zeros((n, md), dtype=lib.DET_DTYPE)
            counts = np.zeros(n, dtype=np.int32)
            if len(inflight) == 2:
                finish(inflight.pop(0))
            inflight.append((submit(frames, size, dets, counts), frames, dets, counts))
            if n < want:
                break
    while inflight:
        finish(inflight.pop(0))
    writer.release()
    print("%d frames, %.1f ms reading, detecting and writing (%s / yolo_b200_wait)" % (state["frames"], 1e3 * (time.time() - t0), api))


def frame_size(flag, value):
    """(sh, sw) of a WxH flag value."""
    try:
        sw, sh = (int(v) for v in value.lower().split("x"))
    except ValueError as e:
        raise SystemExit("%s %s: %s" % (flag, value, e))
    return sh, sw


def run_yuv(ctx, args, size):
    """Raw video as `ffmpeg -f rawvideo -pix_fmt {nv12,yuv420p,yuyv422}` writes it: 1.5 or 2 bytes per pixel cross the
    link and are converted to BGR on the GPU (yolo_b200_submit_yuv)."""
    fmt = YUV_FORMATS[args.yuv_format]
    sh, sw = frame_size("--yuv_size", args.yuv_size)
    try:
        shape = lib.yuv_frame_shape(fmt, sh, sw)
    except ValueError as e:
        raise SystemExit("--yuv_size %s: %s" % (args.yuv_size, e))
    run_raw(ctx, args, size, args.yuv, shape, sh, sw, lambda fr, sz, d, c: ctx.submit_yuv(fr, fmt, sz, d, c), YUV_CV2[args.yuv_format],
            args.yuv_fps, "yolo_b200_submit_yuv")


def run_bayer(ctx, args, size):
    """Raw sensor video as `ffmpeg -f rawvideo -pix_fmt bayer_{rggb,bggr,grbg,gbrg}8` writes it: 1 byte per pixel crosses
    the link and is demosaiced on the GPU (yolo_b200_submit_bayer)."""
    pattern = BAYER_PATTERNS[args.bayer_pattern]
    sh, sw = frame_size("--bayer_size", args.bayer_size)
    try:
        shape = lib.bayer_source_size(pattern, (sh, sw))
    except ValueError as e:
        raise SystemExit("--bayer_size %s: %s" % (args.bayer_size, e))
    run_raw(ctx, args, size, args.bayer, shape, sh, sw, lambda fr, sz, d, c: ctx.submit_bayer(fr, pattern, sz, d, c),
            BAYER_CV2[args.bayer_pattern], args.bayer_fps, "yolo_b200_submit_bayer")


def main():
    ap = argparse.ArgumentParser(description="slim_yolo_v2 fixed-point detection on B200")
    ap.add_argument("-v", "--version", default="slim_yolo_v2_q_bf", help="only slim_yolo_v2_q_bf runs on this path")
    ap.add_argument("-size", "--input_size", default=416, type=int)
    ap.add_argument("--trained_model", default="random", help="q_bf state_dict (.pth) or 'random'")
    ap.add_argument("--conf_thresh", default=0.1, type=float)
    ap.add_argument("--nms_thresh", default=0.50, type=float)
    ap.add_argument("--visual_threshold", default=0.3, type=float)
    ap.add_argument("--cuda", action="store_true", default=True, help="kept for compatibility: this path always runs on CUDA")
    ap.add_argument("--images", default="synthetic:2", help="directory / glob of images, or synthetic:N")
    ap.add_argument("--video", default=None, help="video file (demo.py --mode video, :123-158) or camera index (--mode camera, :60-96): frames are batched, detected on the GPU and written, annotated, to <out>/detections.avi")
    ap.add_argument("--yuv", default=None, help="raw YUV video file (ffmpeg -f rawvideo): frames are detected on the GPU straight from YUV and written, annotated, to <out>/detections.avi")
    ap.add_argument("--yuv_format", default="nv12", choices=sorted(YUV_FORMATS), help="pixel format of --yuv: nv12, i420 (ffmpeg yuv420p) or yuyv (yuyv422)")
    ap.add_argument("--yuv_size", default=None, help="frame size of --yuv as WxH, e.g. 640x480")
    ap.add_argument("--yuv_fps", default=25.0, type=float, help="frame rate written to detections.avi in --yuv mode")
    ap.add_argument("--bayer", default=None, help="raw Bayer sensor video file (ffmpeg -f rawvideo, 8 bits per pixel): frames are demosaiced and detected on the GPU and written, annotated, to <out>/detections.avi")
    ap.add_argument("--bayer_pattern", default="rggb", choices=sorted(BAYER_PATTERNS), help="mosaic of --bayer, named by the sensor's top-left 2x2 (ffmpeg bayer_rggb8 ..., GenICam BayerRG8 ...)")
    ap.add_argument("--bayer_size", default=None, help="frame size of --bayer as WxH, e.g. 640x480")
    ap.add_argument("--bayer_fps", default=25.0, type=float, help="frame rate written to detections.avi in --bayer mode")
    ap.add_argument("--max_frames", default=0, type=int, help="stop a --video / --yuv / --bayer run after this many frames (0 = to the end)")
    ap.add_argument("--out", default="output")
    ap.add_argument("--batch", default=64, type=int)
    args = ap.parse_args()
    if args.version != "slim_yolo_v2_q_bf":
        raise SystemExit("only -v slim_yolo_v2_q_bf is implemented (the fixed-point hot path)")
    size = (args.input_size, args.input_size)
    if args.trained_model == "random":
        qnet = ex.random_quantnet(seed=0, calib_hw=size, calib_frames=2, head_bias_shift=-3.0)
    else:
        sd = torch.load(args.trained_model, map_location="cpu")
        qnet = ex.quantnet_from_state_dict(sd, anchors=ex.ANCHOR_SIZE_MASK, num_classes=2)     # test.py:165-172
    ctx = lib.Context(0)
    ctx.load_quantnet(qnet, contract=lib.CONTRACT_P, head_mode=lib.HEAD_PYTHON, conf_thresh=args.conf_thresh,
                      nms_thresh=args.nms_thresh, max_det=1024)
    if args.yuv is not None:
        if not args.yuv_size:
            raise SystemExit("--yuv needs --yuv_size WxH")
        run_yuv(ctx, args, size)
        ctx.close()
        return
    if args.bayer is not None:
        if not args.bayer_size:
            raise SystemExit("--bayer needs --bayer_size WxH")
        run_bayer(ctx, args, size)
        ctx.close()
        return
    if args.video is not None:
        run_video(ctx, args, size)
        ctx.close()
        return
    md = 1024
    if args.images.startswith("synthetic:"):
        rng = np.random.default_rng(0)
        count = int(args.images.split(":")[1])
        sources = [("synthetic_%d" % i, lambda: rng.integers(0, 256, (480, 640, 3), dtype=np.uint8)) for i in range(count)]
    else:
        files = sorted(glob.glob(os.path.join(args.images, "*")) if os.path.isdir(args.images) else glob.glob(args.images))
        sources = [(os.path.splitext(os.path.basename(f))[0], lambda f=f: cv2.imread(f, cv2.IMREAD_COLOR)) for f in files]

    def batches():
        """Batches of --batch readable images, read only when the batch is formed (unreadable files are skipped)."""
        names, imgs = [], []
        for name, read in sources:
            im = read()
            if im is None:
                continue
            names.append(name); imgs.append(im)
            if len(imgs) == args.batch:
                yield names, imgs
                names, imgs = [], []
        if imgs:
            yield names, imgs

    def finish(job):
        ticket, names, imgs, dets, counts, _ = job
        ctx.wait(ticket)
        for k, im in enumerate(imgs):
            boxes, scores, cls, _ = lib.dets_to_arrays(dets[k], int(min(counts[k], md)))
            h, w = im.shape[:2]
            boxes = boxes * np.array([[w, h, w, h]], dtype=np.float32)          # test.py:88-90
            out = vis(im.copy(), boxes, scores, cls, args.visual_threshold)
            cv2.imwrite(os.path.join(args.out, names[k] + ".jpg"), out)
            print("%s: %d detections (%d above %.2f)" % (names[k], len(scores), int((scores > args.visual_threshold).sum()), args.visual_threshold))

    # data/__init__.py:36 (cv2.resize, bilinear) runs on the GPU too: each batch, whatever its mix of sizes, is one call.  Two
    # batches are in flight: reading batch k+1 and writing the annotated images of batch k-1 overlap the GPU work of batch k.
    os.makedirs(args.out, exist_ok=True)
    t0, total, inflight = time.time(), 0, []
    for names, imgs in batches():
        packed, shapes = lib.pack_images(imgs)
        packed = torch.from_numpy(packed).pin_memory()                     # asynchronous host-to-device copies
        dets = np.zeros((len(imgs), md), dtype=lib.DET_DTYPE)
        counts = np.zeros(len(imgs), dtype=np.int32)
        if len(inflight) == 2:
            finish(inflight.pop(0))
        inflight.append((ctx.submit_u8bgr_images(packed, shapes, size, dets, counts), names, imgs, dets, counts, packed))
        total += len(imgs)
    while inflight:
        finish(inflight.pop(0))
    print("%d images, %.1f ms reading, detecting and writing (yolo_b200_submit_u8bgr_ragged / yolo_b200_wait)" % (total, 1e3 * (time.time() - t0)))
    ctx.close()


if __name__ == "__main__":
    main()
