"""The network a context loads is on the device before the first call that reads it.

yolo_b200_load and the weights the tensor-core 1x1 / wide-layer kernel builds on its first use (yolo_v2) are uploaded on the
context stream, so the first forward after a load computes what every later one does."""
import numpy as np
import pytest

import yolo_b200  # noqa: F401
from yolo_b200 import export as ex
from yolo_b200 import lib


@pytest.mark.gpu
def test_first_forward_after_load_equals_the_next():
    qnet = ex.random_quantnet_yolo_v2(seed=0, calib_hw=(64, 96), calib_frames=1)
    bgr = np.random.default_rng(5).integers(0, 256, (7, 96, 128, 3), dtype=np.uint8)
    runs = []
    for _ in range(2):                                   # a fresh context each time: the first call builds the lazy weights
        c = lib.Context(0)
        try:
            c.load_quantnet(qnet, contract=lib.CONTRACT_P, conf_thresh=0.02, nms_thresh=0.5, max_det=512)
            runs.append([c.forward_u8bgr_resize(bgr, (64, 96)) for _ in range(2)])
        finally:
            c.close()
    ref_d, ref_c = runs[0][1]
    assert (ref_c > 0).all()
    for d, cnt in (runs[0][0], runs[1][0], runs[1][1]):
        np.testing.assert_array_equal(cnt, ref_c)
        for i in range(len(cnt)):
            np.testing.assert_array_equal(d[i][:cnt[i]].view(np.int32), ref_d[i][:cnt[i]].view(np.int32))
