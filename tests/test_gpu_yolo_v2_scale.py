"""yolo_v2 (darknet19, 20 classes, BASELINE configs[4]) at the batch and sizes the benchmark runs, against the CPU oracle.

The other yolo_v2 tests run batches of 2-3 frames, where every wide layer's CTA-pair kernel (conv_ws3.cu) gets at most one work
unit per CTA pair.  Here:
  A. the bench workload (64 frames of 416x416, the bench's network and frames): every layer of every frame, both contracts;
  B. conv_ws3.cu's schedule regimes (one, two, three or more units per CTA pair, a ragged last round, a dummy tile in a later
     unit) on every map width the kernel accepts, under all four epilogue instantiations, with a canary after the output;
  C. the wide 1x1 layers on conv_umma.cu past the wrap of its accumulator-buffer parity, and the whole graph at 320 / 512 / 608;
  D. the 20-class head on the bench's prediction maps, and detection lists longer than max_det through every entry point;
  E. every documented fallback switch, one fresh interpreter each."""
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

import bench
import golden_util as gu
import oracle_lib as ol
import yolo_b200  # noqa: F401
from yolo_b200 import export as ex
from yolo_b200 import lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BENCH_N, BENCH_HW, BENCH_MAXDET = 64, (416, 416), 1024
EPI_NAMES = {0: "EPI_GENERIC", 1: "EPI_F_RNE", 2: "EPI_P", 3: "EPI_F_RNE_NOHI"}
CANARY = 0x5A
TAIL = 64 * 1024                     # bytes of canary after every output map
DET_CANARY = -7                      # int32 words of an untouched detection record


@pytest.fixture(scope="module")
def ctx():
    c = lib.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def qv():
    """The bench's yolo_v2 network (bench.py: BASELINE configs[4])."""
    return ex.random_quantnet_yolo_v2(seed=0, calib_hw=BENCH_HW, calib_frames=1)


@pytest.fixture(scope="module")
def bench_x8(qv):
    """The bench's 64 yolo_v2 frames, quantised as the bench quantises them."""
    return bench.ol_quantize(ex.synthetic_frames_f32(BENCH_N, BENCH_HW[0], BENCH_HW[1], seed=13).numpy(), qv.sa[0])


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def random_tables(rng, qnet):
    """Random but valid exponent tables (bit-exactness must hold for ANY table, SURVEY.md 8a)."""
    L = len(qnet.layers)
    sa = [int(rng.integers(0, 9)) for _ in range(L + 1)]
    sw = [int(rng.integers(4, 12)) for _ in range(L)]
    sb = [int(rng.integers(2, 12)) for _ in range(L)]
    rt = [int(rng.integers(6, 14)) for _ in range(L)]
    return sa, sw, sb, rt


def det_arrays(ctx, pred_ptr, n, gh, gw, in_h, in_w):
    md = ctx.params.max_det
    d_dets = torch.zeros((n, md, 8), dtype=torch.int32, device="cuda")
    d_counts = torch.zeros((n,), dtype=torch.int32, device="cuda")
    ctx.detect(pred_ptr, n, gh, gw, in_h, in_w, d_dets, d_counts)
    ctx.sync()
    dets = d_dets.cpu().numpy().view(lib.DET_DTYPE).reshape(n, md)
    return dets, d_counts.cpu().numpy()


def output_shapes(qnet, h, w):
    """Consumer-visible output size (after the pool) of every layer of a graph network."""
    return [(d[0] // 2, d[1] // 2) if pool else d for d, (_, _, _, pool) in zip(bench.yolo_v2_maps(qnet, h, w), qnet.layers)]


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def oracle_layer(qnet, l, x, contract, round_mode=lib.ROUND_RNE):
    """One convolution of a graph network on the oracle, without its pool (a 1x1 kernel is the centre tap of a 3x3 one)."""
    cin, cout, activ, _ = qnet.layers[l]
    w = qnet.w[l]
    if w.shape[1] == 1:
        w3 = np.zeros((w.shape[0], 3, 3, w.shape[3]), np.int8)
        w3[:, 1, 1, :] = w[:, 0, 0, :]
        w = w3
    sa_i = ex.input_exponent(qnet.layers, qnet.graph, qnet.sa, l)
    return ol.conv_layer(x, w, qnet.b[l], cin, cout, sa_i, qnet.sw[l], qnet.sb[l], qnet.retune[l], qnet.sa[l + 1], activ, 0,
                         contract, round_mode)


def run_layer_with_canary(ctx, l, x, n, h, w, cs_out):
    """ctx.conv_layer into a map followed by TAIL bytes of canary; asserts the canary is untouched, returns the map."""
    size = n * h * w * cs_out
    buf = torch.full((size + TAIL,), CANARY, dtype=torch.int8, device="cuda")
    ctx.conv_layer(l, dev(x), n, h, w, buf[:size])
    ctx.sync()
    got = buf.cpu().numpy()
    bad = np.flatnonzero(got[size:] != CANARY)
    assert bad.size == 0, "layer %d (n=%d, %dx%d) wrote %d bytes past its output, the first %d bytes after the end" % (
        l, n, h, w, bad.size, bad[0])
    return got[:size].reshape(n, h, w, cs_out)


def assert_same_dets(dets_f, count, ref, where):
    (ob, os_, oc, oidx), ocnt = ref
    assert count == ocnt, "%s: %d detections, oracle %d" % (where, count, ocnt)
    k = min(int(count), len(dets_f))
    b, s_, c, idx = lib.dets_to_arrays(dets_f, k)
    np.testing.assert_array_equal(idx, oidx, err_msg=where)
    np.testing.assert_array_equal(c, oc, err_msg=where)
    np.testing.assert_allclose(s_, os_, atol=1e-5, rtol=0, err_msg=where)
    np.testing.assert_allclose(b, ob, atol=1e-5, rtol=0, err_msg=where)


def oracle_head_v2(qnet, pred, h, w, conf, nms, max_det):
    return ol.head_python(pred, len(qnet.anchors), qnet.num_classes, qnet.sa[-1], qnet.anchors, qnet.stride, h, w, conf, nms,
                          max_det=max_det)


# ---- A. the bench workload, every frame, every layer -----------------------------------------------------------------

_BENCH_PRED = {}                     # contract -> the 64 prediction maps of A's device run (reused by D)


def slow_layers(ctx, qnet, n, h, w):
    """Layers whose stand-alone launch at this batch goes to the dot-product kernel (to name them when the count moves)."""
    dims = bench.yolo_v2_maps(qnet, h, w)
    slow = []
    for l, ((cin, cout, _, pool), (ih, iw)) in enumerate(zip(qnet.layers, dims)):
        before = ctx.slow_path_count()
        oh, ow = (ih // 2, iw // 2) if pool else (ih, iw)
        ctx.conv_layer(l, torch.zeros((n, ih, iw, ex.cstride(cin)), dtype=torch.int8, device="cuda"), n, ih, iw,
                       torch.zeros((n, oh, ow, ex.cstride(cout)), dtype=torch.int8, device="cuda"))
        ctx.sync()
        if ctx.slow_path_count() != before:
            slow.append((l, qnet.layers[l], qnet.graph[l]))
    return slow


@pytest.mark.parametrize("contract", [lib.CONTRACT_F, lib.CONTRACT_P], ids=["F_RNE", "P"])
def test_yolo_v2_bench_workload_batch64_against_oracle(ctx, qv, bench_x8, contract):
    """The yolo_v2 line of bench.py: its network, its 64 frames of 416x416, its thresholds and capacity, through the device
    entry point: all 23 layer maps of all 64 frames equal the oracle's, the detections equal the oracle's and the host entry
    point's, no layer falls back to the dot-product kernel, and under contract P the saturation count equals the oracle's."""
    n, (H, W) = BENCH_N, BENCH_HW
    ctx.load_quantnet(qv, contract=contract, round_mode=lib.ROUND_RNE, conf_thresh=bench.CONF, nms_thresh=bench.NMS,
                      max_det=BENCH_MAXDET)
    ctx.overflow_count()                                       # reads reset the counter
    sp0 = ctx.slow_path_count()
    d_dets = torch.zeros((n, BENCH_MAXDET, 8), dtype=torch.int32, device="cuda")
    d_counts = torch.zeros((n,), dtype=torch.int32, device="cuda")
    ctx.forward_int8_dev(dev(bench_x8), n, H, W, d_dets, d_counts)
    ctx.sync()
    ovf = ctx.overflow_count()
    slow = ctx.slow_path_count() - sp0
    counts = d_counts.cpu().numpy()
    dets = d_dets.cpu().numpy().view(lib.DET_DTYPE).reshape(n, BENCH_MAXDET)
    shapes = output_shapes(qv, H, W)
    outs = [ctx.layer_output(l, n, oh, ow) for l, (oh, ow) in enumerate(shapes)]
    _BENCH_PRED[contract] = outs[-1]
    if slow:
        pytest.fail("%d dot-product launches in the 64-frame forward; layers that take that path alone: %s"
                    % (slow, slow_layers(ctx, qv, n, H, W)))
    ovf_ref = 0
    for f0 in range(0, n, 16):
        ref, o = ol.backbone_graph(qv, bench_x8[f0:f0 + 16], contract=contract)
        ovf_ref += o
        for l, r in enumerate(ref):
            got = outs[l][f0:f0 + 16]
            if not np.array_equal(got, r):
                f = f0 + int(np.flatnonzero([not np.array_equal(a, b) for a, b in zip(got, r)])[0])
                pytest.fail("layer %d %s %s, frame %d of the 64-frame batch differs from the oracle (%d bytes)"
                            % (l, qv.layers[l], qv.graph[l], f, int(np.count_nonzero(outs[l][f] != r[f - f0]))))
        for k in range(len(ref[-1])):
            f = f0 + k
            assert_same_dets(dets[f], int(counts[f]), oracle_head_v2(qv, ref[-1][k], H, W, bench.CONF, bench.NMS, BENCH_MAXDET),
                             "frame %d" % f)
        del ref
    if contract == lib.CONTRACT_P:
        assert ovf == ovf_ref, "contract P: %d saturations counted, oracle %d" % (ovf, ovf_ref)
    hdets, hcounts = ctx.forward_int8(bench_x8)
    np.testing.assert_array_equal(hcounts, counts)
    for f in range(n):
        k = min(int(counts[f]), BENCH_MAXDET)
        assert hdets[f][:k].tobytes() == dets[f][:k].tobytes(), "host and device entry points differ on frame %d" % f
    print("contract %d: detections per frame %s, saturations %d" % (contract, counts.tolist(), ovf))


# ---- B. conv_ws3.cu schedule matrix --------------------------------------------------------------------------------

def ws3_plan(cs_in, cs_out, n, H, W, sm):
    """Python mirror of conv_ws3.cu's ws3_plan: eligibility and unit arithmetic.  Returns (tiles, pairs, units, ncl) or None.
    A unit is (tile pair, 256-channel slice); CTA pair cid runs units cid, cid + ncl, ..."""
    if cs_in % 128 or cs_out % 256 or W % 8 == 0 or W + 1 > 64:
        return None
    period, rP = H + 1, W + 1
    tiles = -(-n * period * rP // 128)
    pairs = (tiles + 1) // 2
    units = pairs * (cs_out // 256)
    ncl = (min(2 * units, sm) & ~1) // 2
    return tiles, pairs, units, ncl


REGIMES = {
    # 1: one unit per pair at most (the control; what batches of 2-3 frames reach)
    1: ("one unit per pair", lambda t, p, u, c, s: u <= c, "max"),
    # 2: a second unit on most pairs: epilogue group 1, TMEM buffer 1, before any phase wrap
    2: ("two units on some pair", lambda t, p, u, c, s: c < u <= 2 * c, "max"),
    # 3: every pair runs three or more units: the tempty / tfull phase flips at it >= 2
    3: ("three or more units on every pair", lambda t, p, u, c, s: u >= 3 * c, "min"),
    # 4: units = k * ncl + r with k >= 2 and 0 < r <= slices: at most the units of one tile pair run a round later than all
    #    the others (r = 1 needs an odd ncl; units come in multiples of the slice count, so with 148 SMs r is 2 or 4)
    4: ("a few pairs run one unit more", lambda t, p, u, c, s: u > 2 * c and 0 < u % c <= s, "min"),
    # 5: an odd tile count and several units per pair: the last pair's dummy tile falls in a unit after a pair's first
    5: ("odd tile count, several units per pair", lambda t, p, u, c, s: t % 2 == 1 and u > c, "min"),
}


def batch_for_regime(cs_in, cs_out, H, W, regime, sm, n_max=20000):
    """The smallest (or, for the 'at most' regimes, the largest) batch that puts conv_ws3 in `regime` on this GPU."""
    name, pred, pick = REGIMES[regime]
    ok = [n for n in range(1, n_max + 1) if pred(*ws3_plan(cs_in, cs_out, n, H, W, sm), cs_out // 256)]
    assert ok, "no batch up to %d reaches regime %d (%s) for %d -> %d on %dx%d with %d SMs" % (n_max, regime, name, cs_in, cs_out, H, W, sm)
    return ok[-1] if pick == "max" else ok[0]


WS3_LAYERS = (8, 13, 18, 21)                    # 256->512, 512->1024, 1024->1024, 1280->1024 (10 planes)
WS3_MAPS = [(13, 13), (26, 26), (1, 1), (3, 3), (5, 63), (40, 7), (19, 19), (38, 38)]
EPI_VARIANTS = ["F_RNE", "F_FLOOR", "F_HALF_UP", "P", "F_RNE_random"]


def ws3_cases():
    """(layer, (H, W), regime, epilogue variant): every layer on the bench's 13x13 grid, the 2- and 4-slice layers 8 and 13 on
    26x26, the 2-slice layer 8 and the 10-plane layer 21 on the other maps; the variants rotate so that every variant meets
    every regime."""
    cases = []
    k = 0
    for hw in WS3_MAPS:
        for l in {(13, 13): WS3_LAYERS, (26, 26): (8, 13)}.get(hw, (8, 21)):
            for r in REGIMES:
                cases.append((l, hw, r, EPI_VARIANTS[(r + k) % len(EPI_VARIANTS)]))
            k += 1
    return cases


def variant_net(qv, variant):
    """(network, contract, round mode) of an epilogue variant."""
    if variant == "F_RNE_random":
        import copy
        q = copy.deepcopy(qv)
        q.sa, q.sw, q.sb, q.retune = random_tables(np.random.default_rng(zlib.crc32(b"ws3-random-32")), q)
        return q, lib.CONTRACT_F, lib.ROUND_RNE
    if variant == "P":
        return qv, lib.CONTRACT_P, lib.ROUND_RNE
    return qv, lib.CONTRACT_F, {"F_RNE": lib.ROUND_RNE, "F_FLOOR": lib.ROUND_FLOOR, "F_HALF_UP": lib.ROUND_HALF_UP}[variant]


def epi_mode(ctx, layer):
    """The epilogue instantiation layer `layer`'s tables select under the loaded network (the requant probe's return)."""
    acc = torch.zeros(16, dtype=torch.int32, device="cuda")
    out = torch.zeros(16, dtype=torch.int8, device="cuda")
    mode = ctx.debug_requant(layer, acc, 1, out)
    ctx.sync()
    return mode


@pytest.mark.parametrize("variant", EPI_VARIANTS)
def test_ws3_cta_pair_schedule_regimes_against_oracle(ctx, qv, variant):
    """conv_ws3.cu through the per-layer entry point at batches derived from the regime to reach (the unit arithmetic is
    mirrored above and asserted, so a GPU with another SM count still reaches every regime): bit-exact maps, an untouched
    canary after the output (gutter rows and the dummy tile are masked only by the epilogue's `inside`), and under contract P
    a non-zero saturation count equal to the oracle's.  The rotation of variants over the cases is in ws3_cases()."""
    sm = sm_count()
    q, contract, rmode = variant_net(qv, variant)
    ctx.load_quantnet(q, contract=contract, round_mode=rmode)
    cases = [c for c in ws3_cases() if c[3] == variant]
    seen_modes = set()
    for (l, (H, W), regime, _) in cases:
        cin, cout, activ, pool = q.layers[l]
        cs_in, cs_out = ex.cstride(cin), ex.cstride(cout)
        n = batch_for_regime(cs_in, cs_out, H, W, regime, sm)
        tiles, pairs, units, ncl = ws3_plan(cs_in, cs_out, n, H, W, sm)
        assert REGIMES[regime][1](tiles, pairs, units, ncl, cs_out // 256) and pool == 0
        mode = epi_mode(ctx, l)
        seen_modes.add(mode)
        print("ws3 layer %d %dx%d regime %d (%s) n=%d: tiles %d pairs %d units %d ncl %d, max %d units per pair, %s"
              % (l, H, W, regime, REGIMES[regime][0], n, tiles, pairs, units, ncl, -(-units // ncl), EPI_NAMES[mode]))
        rng = np.random.default_rng(zlib.crc32(("%d-%d-%d-%d-%s" % (l, H, W, regime, variant)).encode()))
        x = rng.integers(-128, 128, (n, H, W, cs_in), dtype=np.int8)
        x[..., cin:] = 0
        ctx.overflow_count()
        got = run_layer_with_canary(ctx, l, x, n, H, W, cs_out)
        ovf = ctx.overflow_count()
        ref, ovf_ref = oracle_layer(q, l, x, contract, rmode)
        if not np.array_equal(got, ref):
            bad = np.argwhere(got != ref)
            pytest.fail("ws3 layer %d %dx%d n=%d regime %d %s: %d bytes differ, first at (frame, y, x, channel) %s"
                        % (l, H, W, n, regime, variant, len(bad), tuple(bad[0])))
        if contract == lib.CONTRACT_P:
            assert ovf == ovf_ref and ovf > 0, "layer %d %dx%d n=%d: %d saturations counted, oracle %d" % (l, H, W, n, ovf, ovf_ref)
    _WS3_MODES.update(seen_modes)


_WS3_MODES = set()


def test_ws3_matrix_selected_every_epilogue(ctx, qv):
    """Across the regime matrix every epilogue instantiation of conv_ws3 (fp32 RNE with and without the upper 16-bit clamp,
    contract P, the generic integer path) was selected at least once."""
    if len(_WS3_MODES) == 0:
        for variant in EPI_VARIANTS:             # the matrix did not run in this session: ask the tables directly
            q, contract, rmode = variant_net(qv, variant)
            ctx.load_quantnet(q, contract=contract, round_mode=rmode)
            _WS3_MODES.update(epi_mode(ctx, l) for l in WS3_LAYERS)
    missing = [EPI_NAMES[m] for m in EPI_NAMES if m not in _WS3_MODES]
    assert not missing, "never selected: %s" % missing


# ---- C. conv_umma.cu at scale, and the graph at other input sizes ---------------------------------------------------------

@pytest.mark.parametrize("contract", [lib.CONTRACT_F, lib.CONTRACT_P], ids=["F_RNE", "P"])
def test_wide_1x1_layers_past_the_tmem_parity_wrap(ctx, qv, contract):
    """The 1x1 layers 14 / 16 (1024 -> 512), 20 (512 -> 64 on 26x26) and 22 (1024 -> 125, stored as 128 channels: the pad
    channels must be 0) at batches where tiles x slices is at least three grids, so every CTA's accumulator-buffer parity
    (tcount) wraps; canary after the output."""
    sm = sm_count()
    ctx.load_quantnet(qv, contract=contract)
    dims = bench.yolo_v2_maps(qv, *BENCH_HW)
    for l in (14, 16, 20, 22):
        cin, cout, activ, pool = qv.layers[l]
        assert qv.graph[l]["ksize"] == 1 and pool == 0
        cs_in, cs_out = ex.cstride(cin), ex.cstride(cout)
        H, W = dims[l]
        slices = max(cs_out // 256, 1)
        n = -(-3 * sm * 128 // (H * W * slices)) + 1            # >= 3 * grid work items whatever the tile shape (128 pixels)
        assert n * H * W * slices >= 3 * sm * 128
        rng = np.random.default_rng(100 + l)
        x = rng.integers(-128, 128, (n, H, W, cs_in), dtype=np.int8)
        ctx.overflow_count()
        got = run_layer_with_canary(ctx, l, x, n, H, W, cs_out)
        ovf = ctx.overflow_count()
        ref, ovf_ref = oracle_layer(qv, l, x, contract)
        if not np.array_equal(got, ref):
            bad = np.argwhere(got != ref)
            pytest.fail("1x1 layer %d n=%d %dx%d: %d bytes differ, first at %s" % (l, n, H, W, len(bad), tuple(bad[0])))
        assert not got[..., cout:].any(), "layer %d: pad channels %d..%d are not zero" % (l, cout, cs_out - 1)
        if contract == lib.CONTRACT_P:
            assert ovf == ovf_ref, "layer %d: %d saturations counted, oracle %d" % (l, ovf, ovf_ref)


@pytest.mark.parametrize("contract", [lib.CONTRACT_F, lib.CONTRACT_P], ids=["F_RNE", "P"])
@pytest.mark.parametrize("hw", [(320, 320), (512, 512), (608, 608)])
def test_yolo_v2_graph_at_other_input_sizes(ctx, qv, hw, contract):
    """The bench network at 320 (10 / 20 maps), 512 (16 / 32: W % 8 == 0 sends every wide 3x3 layer to conv_umma.cu instead of
    conv_ws3.cu) and 608 (19 / 38): batch 4, every layer and the 20-class detections at conf_thresh 0.02."""
    H, W = hw
    n = 4
    if hw == (512, 512):
        assert all(ws3_plan(1024, 1024, n, h, w, sm_count()) is None for (h, w) in ((16, 16), (32, 32)))
    ctx.load_quantnet(qv, contract=contract, round_mode=lib.ROUND_RNE, conf_thresh=0.02, nms_thresh=0.5, max_det=1024)
    x8 = bench.ol_quantize(ex.synthetic_frames_f32(n, H, W, seed=31 + H).numpy(), qv.sa[0])
    ctx.overflow_count()
    pred, gh, gw = ctx.backbone(dev(x8), n, H, W)
    ctx.sync()
    ovf = ctx.overflow_count()
    assert (gh, gw) == (H // 32, W // 32)
    ref, ovf_ref = ol.backbone_graph(qv, x8, contract=contract)
    for l, r in enumerate(ref):
        got = ctx.layer_output(l, n, r.shape[1], r.shape[2])
        assert np.array_equal(got, r), "%dx%d: layer %d %s %s differs from the oracle" % (H, W, l, qv.layers[l], qv.graph[l])
    if contract == lib.CONTRACT_P:
        assert ovf == ovf_ref
    dets, counts = det_arrays(ctx, pred, n, gh, gw, H, W)
    for f in range(n):
        assert_same_dets(dets[f], int(counts[f]), oracle_head_v2(qv, ref[-1][f], H, W, 0.02, 0.5, 1024), "%dx%d frame %d" % (H, W, f))
    assert counts.sum() > 0


# ---- D. 20-class head and list capacity --------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def bench_pred(ctx, qv, bench_x8):
    """The 64 prediction maps (13 x 13 x 128) of the bench workload under contract F: A's device run when it ran."""
    if lib.CONTRACT_F not in _BENCH_PRED:
        n, (H, W) = BENCH_N, BENCH_HW
        ctx.load_quantnet(qv, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=bench.CONF, nms_thresh=bench.NMS,
                          max_det=BENCH_MAXDET)
        pred, gh, gw = ctx.backbone(dev(bench_x8), n, H, W)
        ctx.sync()
        _BENCH_PRED[lib.CONTRACT_F] = ctx.layer_output(len(qv.layers) - 1, n, gh, gw)
    return _BENCH_PRED[lib.CONTRACT_F]


@pytest.mark.parametrize("nms_thresh", [0.5, 0.3, 0.7, 0.0])
def test_20_class_head_on_the_bench_prediction_maps(ctx, qv, bench_pred, nms_thresh):
    """Decode + per-class NMS of 5 anchors x 20 classes on the 13 x 13 grid of the bench's 64 frames at conf_thresh 0.02
    (hundreds of candidates per frame over most classes): same counts, anchors and classes as the oracle, scores and boxes
    to 1e-5.  nms_thresh 0.0 runs the sorted kernel (the grid kernel needs a positive threshold)."""
    n, (H, W) = BENCH_N, BENCH_HW
    ctx.load_quantnet(qv, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=bench.CONF, nms_thresh=bench.NMS,
                      max_det=BENCH_MAXDET)
    ctx.set_thresholds(0.02, nms_thresh)
    dets, counts = det_arrays(ctx, dev(bench_pred), n, 13, 13, H, W)
    classes = set()
    for f in range(n):
        ref = oracle_head_v2(qv, bench_pred[f], H, W, 0.02, nms_thresh, BENCH_MAXDET)
        assert_same_dets(dets[f], int(counts[f]), ref, "nms %.1f frame %d" % (nms_thresh, f))
        classes.update(ref[0][2].tolist())
    assert counts.min() > 0 and len(classes) >= 10, (counts.tolist(), sorted(classes))


def check_capped(dets, counts, preds, qnet, md, conf, nms, where):
    """counts[f] = the oracle's uncapped count, the first min(count, md) records = the oracle's."""
    over = 0
    for f in range(len(counts)):
        ref = oracle_head_v2(qnet, preds[f], 416, 416, conf, nms, md)
        assert_same_dets(dets[f][:md], int(counts[f]), ref, "%s max_det %d frame %d" % (where, md, f))
        over += ref[1] > md
    assert over > 0, "%s max_det %d: no frame has more detections than the capacity" % (where, md)


@pytest.mark.parametrize("md", [1, 16])
def test_detection_lists_longer_than_max_det(ctx, qv, bench_x8, bench_pred, md):
    """max_det below the kept count (fixed at load): counts report the uncapped total and the lists hold the oracle's first
    max_det records: the Python head (grid and sorted kernels), the device entry point, the pack kernel of the multi-GPU
    collection (offsets = prefix of min(count, max_det)) and the host entry point, which must not write past n x max_det
    records of the caller's buffer."""
    n, (H, W) = BENCH_N, BENCH_HW
    ctx.load_quantnet(qv, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=0.02, nms_thresh=0.5, max_det=md)
    for nms in (0.5, 0.0):
        ctx.set_thresholds(0.02, nms)
        dets, counts = det_arrays(ctx, dev(bench_pred), n, 13, 13, H, W)
        check_capped(dets, counts, bench_pred, qv, md, 0.02, nms, "head nms %.1f" % nms)
    ctx.set_thresholds(0.02, 0.5)
    nf = 8
    x8 = np.ascontiguousarray(bench_x8[:nf])
    # device entry point
    d_dets = torch.full((nf, md, 8), DET_CANARY, dtype=torch.int32, device="cuda")
    d_counts = torch.zeros((nf,), dtype=torch.int32, device="cuda")
    ctx.forward_int8_dev(dev(x8), nf, H, W, d_dets, d_counts)
    ctx.sync()
    counts = d_counts.cpu().numpy()
    check_capped(d_dets.cpu().numpy().view(lib.DET_DTYPE).reshape(nf, md), counts, bench_pred, qv, md, 0.02, 0.5, "device entry point")
    # pack kernel
    d_packed = torch.full((nf * md + 64, 8), DET_CANARY, dtype=torch.int32, device="cuda")
    d_off = torch.full((nf + 1,), -1, dtype=torch.int32, device="cuda")
    rc = ctx.L.yolo_b200_pack_detections(ctx._h, d_dets.data_ptr(), d_counts.data_ptr(), nf, d_packed.data_ptr(), d_off.data_ptr())
    assert rc == 0, ctx.L.yolo_b200_last_error()
    ctx.sync()
    off, packed, dd = d_off.cpu().numpy(), d_packed.cpu().numpy(), d_dets.cpu().numpy()
    np.testing.assert_array_equal(off, np.concatenate([[0], np.cumsum(np.minimum(counts, md))]))
    for f in range(nf):
        np.testing.assert_array_equal(packed[off[f]:off[f + 1]], dd[f, :min(int(counts[f]), md)], err_msg="packed frame %d" % f)
    assert (packed[off[nf]:] == DET_CANARY).all(), "the pack kernel wrote past the packed lists"
    # host entry point through the C-ABI: a buffer longer than n x max_det, canary after the last frame's slots
    buf = np.zeros(nf * md + 64, dtype=lib.DET_DTYPE)
    buf.view(np.int32)[:] = DET_CANARY
    hcounts = np.full(nf, -1, dtype=np.int32)
    rc = ctx.L.yolo_b200_forward_int8(ctx._h, x8.ctypes.data, nf, H, W, buf.ctypes.data, hcounts.ctypes.data)
    assert rc == 0, ctx.L.yolo_b200_last_error()
    np.testing.assert_array_equal(hcounts, counts)
    check_capped(buf[:nf * md].reshape(nf, md), hcounts, bench_pred, qv, md, 0.02, 0.5, "host entry point")
    assert (buf[nf * md:].view(np.int32) == DET_CANARY).all(), "the host entry point wrote past n x max_det records"


@pytest.mark.parametrize("md", [1, 16])
def test_c_head_lists_longer_than_max_det(ctx, md):
    """HEAD_C (2 classes, class-agnostic NMS) with max_det below the kept count: uncapped counts, the oracle's first records."""
    import copy
    g, qnet, frames = gu.load("ref_p_64x96")
    q = copy.deepcopy(qnet)
    q.anchors = [list(a) for a in ex.ANCHOR_SIZE_COCO]
    ctx.load_quantnet(q, contract=lib.CONTRACT_F, head_mode=lib.HEAD_C, conf_thresh=0.01, nms_thresh=0.5, max_det=md)
    rng = np.random.default_rng(40 + md)
    n, gh, gw = 3, 26, 26
    pred = np.zeros((n, gh, gw, 48), dtype=np.int8)
    pred[..., :35] = rng.integers(-60, 60, (n, gh, gw, 35), dtype=np.int8)
    dets, counts = det_arrays(ctx, dev(pred), n, gh, gw, gh * 16, gw * 16)
    over = 0
    for f in range(n):
        (ob, os_, oc, oidx), ocnt = ol.head_c(pred[f], 5, q.sa[10], q.anchors, 16, 0.01, 0.5, max_det=md)
        assert counts[f] == ocnt, "HEAD_C max_det %d frame %d: %d, oracle %d" % (md, f, counts[f], ocnt)
        b, s, c, idx = lib.dets_to_arrays(dets[f], min(int(counts[f]), md))
        np.testing.assert_array_equal(idx, oidx)
        np.testing.assert_array_equal(c, oc)
        np.testing.assert_allclose(s, os_, atol=1e-6, rtol=0)
        np.testing.assert_array_equal(b, ob)
        over += ocnt > md
    assert over > 0


# ---- E. fallback switches, one fresh interpreter each ---------------------------------------------------------------------

SWITCHES = [("YOLO_B200_FS", "0"), ("YOLO_B200_RP", "0"), ("YOLO_B200_WS_CTAPAIR", "0"), ("YOLO_B200_WS_PAIR", "0"),
            ("YOLO_B200_WS_WIDE", "0"), ("YOLO_B200_WS_RASTER", "0"), ("YOLO_B200_WS_RESIDENT", "0"), ("YOLO_B200_WS_STREAM", "0"),
            ("YOLO_B200_NMS_SORTED", "1"), ("YOLO_B200_FUSE_DECODE", "0"), ("YOLO_B200_PDL", "0")]


def fallback_switch_run():
    """Body of the switch test, run in a fresh interpreter (the library reads each switch once per process): the slim chain
    and yolo_v2, all maps and detections against the oracle.  Prints OK and the dot-product launch count."""
    c = lib.Context(0)
    g, qs, frames = gu.load("ref_p_64x96")
    conf, nms = float(g["conf_thresh"]), float(g["nms_thresh"])
    rng = np.random.default_rng(17)
    for (n, h, w) in ((3, 34, 38), (2, 416, 416)):
        x8 = rng.integers(-128, 128, (n, h, w, 4), dtype=np.int8)
        x8[..., 3] = 0
        for contract in (lib.CONTRACT_F, lib.CONTRACT_P):
            c.load_quantnet(qs, contract=contract, conf_thresh=conf, nms_thresh=nms, max_det=4096)
            pred, gh, gw = c.backbone(dev(x8), n, h, w)
            c.sync()
            ref, _ = ol.backbone(qs, x8, contract=contract)
            for l, r in enumerate(ref):
                assert np.array_equal(c.layer_output(l, n, r.shape[1], r.shape[2]), r), "slim %s contract %d layer %d" % ((n, h, w), contract, l)
            dets, counts = det_arrays(c, pred, n, gh, gw, h, w)
            for f in range(n):
                assert_same_dets(dets[f], int(counts[f]), ol.head_python(ref[-1][f], 5, 2, qs.sa[10], qs.anchors, 16, h, w, conf, nms),
                                 "slim %s contract %d frame %d" % ((n, h, w), contract, f))
    qv = ex.random_quantnet_yolo_v2(seed=0, calib_hw=BENCH_HW, calib_frames=1)
    c.load_quantnet(qv, contract=lib.CONTRACT_F, round_mode=lib.ROUND_RNE, conf_thresh=0.02, nms_thresh=0.5, max_det=1024)
    for (n, h, w) in ((3, 96, 64), (2, 416, 416)):
        x8 = bench.ol_quantize(ex.synthetic_frames_f32(n, h, w, seed=50 + h).numpy(), qv.sa[0])
        pred, gh, gw = c.backbone(dev(x8), n, h, w)
        c.sync()
        ref, _ = ol.backbone_graph(qv, x8, contract=lib.CONTRACT_F)
        for l, r in enumerate(ref):
            assert np.array_equal(c.layer_output(l, n, r.shape[1], r.shape[2]), r), "yolo_v2 %s layer %d" % ((n, h, w), l)
        dets, counts = det_arrays(c, pred, n, gh, gw, h, w)
        for f in range(n):
            assert_same_dets(dets[f], int(counts[f]), oracle_head_v2(qv, ref[-1][f], h, w, 0.02, 0.5, 1024), "yolo_v2 %s frame %d" % ((n, h, w), f))
    print("dot-product launches: %d" % c.slow_path_count())
    c.close()
    print("OK")


@pytest.mark.parametrize("switch", SWITCHES, ids=["%s=%s" % s for s in SWITCHES])
def test_fallback_switch_in_a_subprocess(switch):
    """Each documented switch selects a kernel path kept for comparison or as a fallback (DESIGN.md): the slim chain at
    (3, 34, 38) and (2, 416, 416) and yolo_v2 at (3, 96, 64) and (2, 416, 416) still equal the oracle on every map and list."""
    name, value = switch
    code = "import sys; sys.path[:0] = [%r, %r]; import test_gpu_yolo_v2_scale as t; t.fallback_switch_run()" % (
        ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **{name: value}), capture_output=True, text=True,
                       timeout=900)
    print("%s=%s: %s" % (name, value, r.stdout.strip().replace("\n", " | ")))
    assert r.returncode == 0 and r.stdout.rstrip().endswith("OK"), "%s=%s:\n%s%s" % (name, value, r.stdout, r.stderr[-4000:])
