"""bench.py --dump-outputs: the detections of the last timed step, written as float32 .npy files that two builds of the
project can compare output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import oracle_lib as ol
from yolo_b200 import export as ex

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("frames", "counts", "boxes", "scores", "classes", "anchor_index")


def _records(counts, rng):
    rec = np.zeros((int(np.sum(counts)), 8), np.int32)
    rec.view(np.float32)[:, :5] = rng.random((len(rec), 5), dtype=np.float32)
    rec[:, 5] = rng.integers(0, 2, len(rec))
    rec[:, 6] = rng.integers(0, 3380, len(rec))
    return rec


def _load(d):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in NAMES}


def test_dump_outputs_splits_the_records_and_samples_frames_within_the_budget(tmp_path):
    rng = np.random.default_rng(0)
    counts = np.array([3, 0, 2], np.int32)
    rec = _records(counts, rng)
    bench.dump_outputs(str(tmp_path / "small"), counts, rec, 4096)
    d = _load(tmp_path / "small")
    assert all(a.dtype == np.float32 for a in d.values())
    np.testing.assert_array_equal(d["frames"], [0, 1, 2])
    np.testing.assert_array_equal(d["counts"], counts)
    np.testing.assert_array_equal(d["boxes"], rec.view(np.float32)[:, :4])
    np.testing.assert_array_equal(d["scores"], rec.view(np.float32)[:, 4])
    np.testing.assert_array_equal(d["classes"], rec[:, 5])
    np.testing.assert_array_equal(d["anchor_index"], rec[:, 6])

    # more frames than fit at the worst case of max_det records each: the same seeded sample whatever the results
    counts = rng.integers(0, 40, 2000).astype(np.int32)
    rec = _records(counts, rng)
    bench.dump_outputs(str(tmp_path / "a"), counts, rec, 4096)
    bench.dump_outputs(str(tmp_path / "b"), np.ones_like(counts), _records(np.ones_like(counts), rng), 4096)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    k = bench.DUMP_BYTES // (4096 * 7 * 4 + 2 * 4)
    assert len(a["frames"]) == k < len(counts) and np.all(np.diff(a["frames"]) > 0)
    np.testing.assert_array_equal(a["frames"], b["frames"])
    f = a["frames"].astype(np.int64)
    np.testing.assert_array_equal(a["counts"], counts[f])
    start = np.concatenate([[0], np.cumsum(counts)])
    rows = np.concatenate([np.arange(start[i], start[i + 1]) for i in f])
    np.testing.assert_array_equal(a["anchor_index"], rec[rows, 6])
    assert k * (4096 * 7 * 4 + 2 * 4) <= 64 << 20


@pytest.mark.gpu
def test_bench_dumps_the_detections_of_its_last_timed_step(tmp_path):
    """Two frames per step, one warm-up step and two timed steps: the last timed step (index 2) reads input set 2, and the
    dumped lists are what the CPU oracle finds on those frames."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", "2",
                        "--no-secondary", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["frames_per_gpu_per_step"] == 2
    d = _load(tmp_path)
    np.testing.assert_array_equal(d["frames"], [0, 1])
    qnet = bench.make_qnet()
    x8 = ol.quantize_rgb444(ex.synthetic_frames_rgb444(2, bench.H, bench.W, seed=2), qnet.sa[0])
    outs, _ = ol.backbone(qnet, x8, contract=0)
    start = 0
    for i in range(2):
        (ob, os_, oc, oidx), ocnt = ol.head_python(outs[-1][i], 5, 2, qnet.sa[10], qnet.anchors, 16, bench.H, bench.W,
                                                   bench.CONF, bench.NMS)
        assert d["counts"][i] == ocnt > 0
        s = slice(start, start + ocnt)
        np.testing.assert_array_equal(d["anchor_index"][s], oidx)
        np.testing.assert_array_equal(d["classes"][s], oc)
        np.testing.assert_allclose(d["scores"][s], os_, atol=1e-5, rtol=0)
        np.testing.assert_allclose(d["boxes"][s], ob, atol=1e-5, rtol=0)
        start += ocnt
    assert start == len(d["scores"])
