"""GPU parity, stage (iii): whole networks through the reference's model API
against the CPU oracle on identical inputs and weights.
  * fp32 CUDA-core path ("reference precision"): head rows within 2e-4 * max|ref|
    (accumulation order), detections: class ids / keep indices exact and boxes
    within 1e-4 whenever the oracle's own decision margins allow it (reported);
  * fp16 tcgen05 path: head rows within 3e-2 * max|ref| (fp16 storage of 20-130
    layers; SURVEY.md "hard part" 1 -- graded stage-wise, never by loosening the
    tail tolerance: the tail is always exact on the rows the GPU produced)."""
import os

import numpy as np
import pytest

import margins as MG
from helpers import assert_boxes_close, model_cfg

pytestmark = pytest.mark.gpu


def _img(b, h, w, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (b, h, w, 3)).astype(np.float32)


def _oracle_rows(kind, weights, img, cfg):
    from oracle import nets as ON
    from oracle import tails as OT
    if kind in ("ssd300", "ssd512"):
        return OT.ssd_rows(ON.ssd_heads(weights, img, int(kind[3:])))
    if kind == "retinanet":
        return OT.retina_rows(ON.retinanet_heads(weights, img))
    if kind == "yolov3":
        return OT.yolo_rows(ON.yolov3_heads(weights, img))
    return OT.fcos_rows(ON.fcos_heads(weights, img))


def _model(kind, **over):
    import FCOS
    import RetinaNet
    import SSD300
    import SSD512
    import YOLOv3
    if kind == "ssd300":
        return SSD300.SSD300(model_cfg("ssd", **over), None)
    if kind == "ssd512":
        return SSD512.SSD512(model_cfg("ssd", **over), None)
    if kind == "retinanet":
        return RetinaNet.RetinaNet(model_cfg("retinanet", **over), None)
    if kind == "yolov3":
        return YOLOv3.YOLOv3(model_cfg("yolov3", **over), None)
    return FCOS.FCOS(model_cfg("fcos", **over), None)


def _tail_oracle_on_rows(kind, rows, cfg, image=0):
    """Oracle tail fed the GPU's own head rows (stage-wise parity)."""
    from oracle import tails as OT
    r = rows[image]
    thr, mb, iou = cfg["nms_score_threshold"], cfg["nms_max_boxes"], cfg["nms_iou_threshold"]
    if kind in ("ssd300", "ssd512"):
        size = int(kind[3:])
        shapes = ([(38, 38), (19, 19), (10, 10), (5, 5), (5, 5), (3, 3)] if size == 300 else
                  [(64, 64), (32, 32), (16, 16), (8, 8), (8, 8), (4, 4), (2, 2)])
        _, _, ayx, ahw = OT.ssd_anchors(size, shapes)
        return OT.softmax_tail(r[:, :21], r[:, 21:23], r[:, 23:], ayx, ahw, 20, thr, mb, iou)
    raise NotImplementedError


def _geom(kind, net, cfg):
    """Geometry dict of tests/margins.py from a built network."""
    shapes = [(h, w) for h, w, _ in net.levels]
    if kind in ("ssd300", "ssd512"):
        return {"size": int(kind[3:]), "shapes": shapes}
    if kind == "retinanet":
        return {"data_shape": cfg["data_shape"], "shapes": shapes}
    if kind == "yolov3":
        return {"levels": list(net.levels), "priors": cfg["priors"]}
    return {"levels": list(net.levels)}


MKIND = {"ssd300": "ssd", "ssd512": "ssd", "retinanet": "retina", "yolov3": "yolo", "fcos": "fcos"}


def _dense_threshold(kind, rows_ref, geom, frac):
    """Score threshold at which about `frac` * N candidates per class pass in the ORACLE (SURVEY 8d dense regime)."""
    tot, vals = 0, []
    for r in rows_ref:
        S, _, V, _ = MG.per_row(MKIND[kind], r, geom)
        vals.append(S[V].reshape(-1))
        tot += S.shape[0]
    v = np.concatenate(vals)
    k = int(min(max(frac * tot * 20, 40), v.size - 1))
    return float(np.partition(v, v.size - k)[v.size - k])


SHAPES = {"ssd300": (300, 300), "retinanet": (128, 128), "yolov3": (64, 64), "fcos": (128, 128)}


@pytest.mark.parametrize("kind", ["ssd300", "retinanet", "yolov3", "fcos"])
@pytest.mark.parametrize("precision,tol", [("fp32", 2e-4), ("fp16", 5e-3)])
def test_head_rows_vs_oracle(built, kind, precision, tol):
    if kind == "fcos" and precision == "fp16":
        tol = 1e-2   # measured 5.8e-3: every layer's GroupNorm re-normalises fp16-stored activations (a19)
    m = _model(kind, bn_init="trained", precision=precision)
    h, w = SHAPES[kind]
    img = _img(2, h, w, seed=4)
    m.detect_batch(img)
    rows = m.engine(2).head_buf.cpu().numpy()
    ref = _oracle_rows(kind, m.get_weights(), img, m.config)
    assert rows.shape == ref.shape
    scale = float(np.abs(ref).max())
    err = float(np.abs(rows - ref).max())
    print("%s %s: max|err| %.3g of max|ref| %.3g (%.2e rel)" % (kind, precision, err, scale, err / scale))
    assert np.isfinite(rows).all()
    assert err <= tol * scale, (kind, precision, err, scale)


def test_ssd300_reference_plumbing_config_fp32(built):
    """BASELINE config 0: random-init SSD300, ONE 300x300 image through
    test_one_image, reference-precision path, against the end-to-end oracle."""
    from oracle import nets as ON
    from oracle import tails as OT
    m = _model("ssd300", precision="fp32", nms_score_threshold=0.3)
    img = _img(1, 300, 300, seed=0)
    res = m.test_one_image(img)
    assert len(res) == 3 and res[0].dtype == np.float32 and res[2].dtype == np.int32
    assert res[1].shape == (len(res[0]), 4)
    net = m.engine(1)
    rows = net.head_buf.cpu().numpy()
    # (a) tail exact on the GPU's rows
    exp = _tail_oracle_on_rows("ssd300", rows, m.config)
    np.testing.assert_array_equal(res[2], exp[2])
    np.testing.assert_array_equal(net.tail.det_anchor.cpu().numpy()[0, :len(exp[3])], exp[3])
    assert_boxes_close(res[1], exp[1])
    # (b) end to end against the oracle's own forward: identical decisions wherever the oracle's margins
    #     exceed the measured row error, admissible ones elsewhere (tests/margins.py)
    preds = ON.ssd_heads(m.get_weights(), img, 300)
    rows_ref = OT.ssd_rows(preds)
    keep = net.tail.det_anchor.cpu().numpy()[0, :len(res[2])]
    rep = MG.compare_image("ssd", rows[0], rows_ref[0], _geom("ssd300", net, m.config), res[2], keep, res[1],
                           0.3, 20, 0.5)
    print("end-to-end fp32: %d/20 classes clean, %d identical, ds %.3g di %.3g, reasons %s, box err %.3g px"
          % (rep["clean"], rep["identical"], rep["ds"], rep["di"], rep["reasons"], rep["box_err"]))
    assert rep["ds"] <= 3e-5 and rep["clean"] >= 12 and rep["identical"] >= 18, rep
    # rows differ by ~1e-6 relative (accumulation order) and t_hw goes through exp(); random-weight boxes reach
    # 1e7 px, so the bar is relative to the box magnitude
    assert rep["box_err_rel"] <= 3e-4, rep


def test_ssd300_fp16_batch_and_api(built):
    m = _model("ssd300", precision="fp16", nms_score_threshold=0.3)
    img = _img(4, 300, 300, seed=9)
    res = m.test_one_image(img)
    assert isinstance(res, list) and len(res) == 4
    assert len(m.detect_batch(img)[1:3]) == 2  # the batched call returns a sequence over images
    one = m.test_one_image(img[2:3])
    # batch-invariance of the kernels: image 2 alone == image 2 inside the batch
    for a, b in zip(one, res[2]):
        np.testing.assert_array_equal(a, b)
    rows = m.engine(4).head_buf.cpu().numpy()
    for b in range(4):
        exp = _tail_oracle_on_rows("ssd300", rows, m.config, image=b)
        np.testing.assert_array_equal(res[b][2], exp[2])
        assert_boxes_close(res[b][1], exp[1])


def test_ssd512_builds_and_runs(built):
    m = _model("ssd512", precision="fp16", nms_score_threshold=0.3)
    res = m.test_one_image(_img(1, 512, 512))
    assert m.engine(1).N == 24912 and len(res) == 3


def test_tc_and_direct_paths_agree_on_network(built):
    m = _model("yolov3", precision="fp16", bn_init="trained")
    img = _img(2, 64, 64, seed=2)
    m.detect_batch(img)
    a = m.engine(2).head_buf.cpu().numpy().copy()
    net = m.engine(2, allow_tc=False, graph=False)
    net.image_buf.copy_(__import__("torch").from_numpy(img))
    net.run()
    __import__("torch").cuda.synchronize()
    b = net.head_buf.cpu().numpy()
    assert np.abs(a - b).max() <= 2e-2 * np.abs(b).max()


def test_retinanet_loss_forward_vs_oracle(built):
    from oracle import loss as OL
    from oracle import nets as ON
    from oracle import tails as OT
    m = _model("retinanet", precision="fp32", bn_init="trained")
    B, G = 2, 12
    img = _img(B, 128, 128, seed=6)
    rng = np.random.default_rng(3)
    gt = np.full((B, G, 5), -1.0, np.float32)
    for b in range(B):
        n = 3 + 4 * b
        gt[b, :n, 0:2] = rng.uniform(10, 118, (n, 2))
        gt[b, :n, 2:4] = rng.uniform(16, 64, (n, 2))
        gt[b, :n, 4] = rng.integers(0, 20, n)
    got = m.loss_forward(img, gt)
    rows = m.engine(B).head_buf.cpu().numpy()
    heads = ON.retinanet_heads(m.get_weights(), img)
    shapes = [(c.shape[1], c.shape[2]) for c, _ in heads]
    a1, a2, ayx, ahw = OT.retina_anchors([128, 128, 3], shapes)
    for b in range(B):
        ref, info = OL.retina_image_loss(rows[b, :, :21], rows[b, :, 21:23], rows[b, :, 23:], a1, a2, ayx,
                                         ahw, gt[b])
        print("image %d: loss gpu %.6f oracle %.6f (%d pos, %d neg)" % (b, got[b], ref, info["num_pos"],
                                                                       info["num_neg"]))
        assert abs(got[b] - ref) <= 2e-5 * max(abs(ref), 1.0)


@pytest.mark.parametrize("size", [300, 512])
def test_ssd_loss_forward_vs_oracle(built, size):
    """SSD training-loss forward (SURVEY 8f row 2) on the fp32 head rows: matching counts and the mined
    negative count exact, loss within 2e-5 relative (float summation order)."""
    from oracle import loss as OL
    from oracle import tails as OT
    name = "ssd300" if size == 300 else "ssd512"
    m = _model(name, precision="fp32", bn_init="trained")
    B, G = 2, 20
    img = _img(B, size, size, seed=16)
    rng = np.random.default_rng(8)
    gt = np.full((B, G, 5), -1.0, np.float32)
    for b in range(B):
        n = 2 + 5 * b
        gt[b, :n, 0:2] = rng.uniform(0.15 * size, 0.85 * size, (n, 2))
        gt[b, :n, 2:4] = rng.uniform(0.1 * size, 0.5 * size, (n, 2))
        gt[b, :n, 4] = rng.integers(0, 20, n)
    got, info = m.loss_forward(img, gt, return_info=True)
    net = m.engine(B)
    rows = net.head_buf.cpu().numpy()
    shapes = [(h, w) for h, w, _ in net.levels]
    a1, a2, ayx, ahw = OT.ssd_anchors(size, shapes)
    for b in range(B):
        ref, ri = OL.ssd_image_loss(rows[b, :, :21], rows[b, :, 21:23], rows[b, :, 23:], a1, a2, ayx, ahw, gt[b])
        print("image %d: loss gpu %.6f oracle %.6f (%d pos, %d neg, %d mined)" % (
            b, got[b], ref, ri["num_pos"], ri["num_neg"], ri["selected"]))
        assert tuple(info[b]) == (ri["num_pos"], ri["num_neg"], ri["selected"])
        assert abs(got[b] - ref) <= 2e-5 * max(abs(ref), 1.0)


def test_fcos_loss_forward_vs_oracle(built):
    """FCOS training-loss forward (SURVEY 8f row 2): GT sizes on several pyramid levels, one exactly on a
    level boundary (sqrt(h*w) = 64 belongs to P3 and P4), nested boxes (minimal-area rule)."""
    from oracle import loss as OL
    m = _model("fcos", precision="fp32", bn_init="trained", data_shape=[256, 256, 3])
    B, G = 2, 10
    img = _img(B, 256, 256, seed=31)
    gt = np.full((B, G, 5), -1.0, np.float32)
    gt[0, :4] = [[60, 70, 40, 50, 3], [128, 128, 64, 64, 7], [120, 130, 200, 180, 11], [125, 125, 100, 90, 7]]
    gt[1, :3] = [[200, 40, 30, 60, 0], [100, 160, 150, 120, 19], [90, 150, 300, 290, 5]]
    got = m.loss_forward(img, gt)
    net = m.engine(B)
    rows = net.head_buf.cpu().numpy()
    # the oracle loss runs on the GPU's own fp32 head rows (stage-wise parity): rebuild per-level tensors
    off, lv = 0, []
    for h, w, _ in net.levels:
        r = rows[:, off:off + h * w].reshape(B, h, w, 25)
        lv.append((r[..., :20], r[..., 20:21], r[..., 21:25]))
        off += h * w
    assert len(lv) == 5 and off == rows.shape[1]
    for b in range(B):
        ref = OL.fcos_image_loss(lv, gt[b], image=b)
        print("image %d: loss gpu %.6f oracle %.6f" % (b, got[b], ref))
        assert abs(got[b] - ref) <= 2e-5 * max(abs(ref), 1.0)


def test_yolov3_loss_forward_vs_oracle(built):
    """YOLOv3 training-loss forward (SURVEY 8f row 2) incl. the reference's quirks (unclamped
    intersections, mismatched GT / prior strides, the re-used no-object anchor form)."""
    from helpers import YOLO_PRIORS
    from oracle import loss as OL
    m = _model("yolov3", precision="fp32", bn_init="trained", data_shape=[416, 416, 3], obj_scale=5,
               coord_scale=2, noobj_scale=0.5, class_scale=1.5)
    B, G = 2, 12
    img = _img(B, 416, 416, seed=41)
    rng = np.random.default_rng(12)
    gt = np.full((B, G, 5), -1.0, np.float32)
    for b in range(B):
        n = 3 + 5 * b
        gt[b, :n, 0:2] = rng.uniform(30, 380, (n, 2))
        gt[b, :n, 2:4] = rng.uniform(12, 300, (n, 2))
        gt[b, :n, 4] = rng.integers(0, 20, n)
    got = m.loss_forward(img, gt)
    net = m.engine(B)
    rows = net.head_buf.cpu().numpy()
    off, preds = 0, []
    for h, w, a in net.levels:
        preds.append(rows[:, off:off + h * w * a].reshape(B, h, w, a * 25))
        off += h * w * a
    assert [p.shape[1] for p in preds] == [13, 26, 52]
    for b in range(B):
        ref = OL.yolo_image_loss(preds, YOLO_PRIORS, gt[b], coord_scale=2, noobj_scale=0.5, obj_scale=5,
                                 class_scale=1.5, image=b)
        print("image %d: loss gpu %.5f oracle %.5f" % (b, got[b], ref))
        assert abs(got[b] - ref) <= 2e-5 * max(abs(ref), 1.0)


def test_detect_stream_matches_detect_batch(built):
    """Pipelined public API (H2D of batch i+1 overlaps batch i) == synchronous API."""
    import torch
    m = _model("ssd300", precision="fp16", nms_score_threshold=0.3)
    batches = [_img(2, 300, 300, seed=s) for s in (21, 22, 23)]
    ref = [m.detect_batch(b) for b in batches]
    pinned = [torch.from_numpy(b).pin_memory() for b in batches]
    got = list(m.detect_stream(pinned))
    assert len(got) == 3
    for g, r in zip(got, ref):
        for gi, ri in zip(g, r):
            for a, b in zip(gi, ri):
                np.testing.assert_array_equal(a, b)


def test_detect_stream_results_survive_later_batches(built):
    """The read-back runs one step behind the launches: a yielded result must not alias a buffer that a later
    batch overwrites, and an un-pinned source / a single-batch stream work too."""
    m = _model("ssd300", precision="fp16", nms_score_threshold=0.3)
    batches = [_img(2, 300, 300, seed=s) for s in (31, 32, 33, 34, 35)]
    ref = [m.detect_batch(b) for b in batches]
    held = []
    for got in m.detect_stream(batches):        # numpy sources (pageable): still correct, just not overlapped
        held.append(got)
    assert len(held) == 5
    for g, r in zip(held, ref):
        for gi, ri in zip(g, r):
            for a, b in zip(gi, ri):
                np.testing.assert_array_equal(a, b)
    one = list(m.detect_stream(batches[:1]))
    assert len(one) == 1 and np.array_equal(one[0][1][0], ref[0][1][0])
    assert list(m.detect_stream([])) == []


@pytest.mark.parametrize("kind,hw", [("ssd300", 300), ("retinanet", 256)])
def test_pipelined_and_single_graph_streams_agree(built, monkeypatch, kind, hw):
    """The two-stage pipeline (tail of batch i on a second stream under the body of batch i+1, candidate rows / lists /
    records double-buffered by slot) against the one-graph-per-step stream and the synchronous call: identical
    detections for every batch of a 6-batch stream (each slot is reused three times), for two model families; then the
    engine-level run_pipelined() against run() on the packed records themselves."""
    import torch
    kw = {"nms_score_threshold": 0.3} if kind == "ssd300" else {"data_shape": [hw, hw, 3], "nms_score_threshold": 0.05}
    m = _model(kind, precision="fp16", **kw)
    batches = [_img(2, hw, hw, seed=s) for s in range(41, 47)]
    ref = [m.detect_batch(b) for b in batches]
    pinned = [torch.from_numpy(b).pin_memory() for b in batches]
    for mode in ("1", "0"):
        monkeypatch.setenv("ODT_PIPELINE", mode)
        got = list(m.detect_stream(pinned))
        assert len(got) == len(ref)
        for g, r in zip(got, ref):
            for gi, ri in zip(g, r):
                for a, b in zip(gi, ri):
                    np.testing.assert_array_equal(a, b)
    net = m.engine(2)
    net.capture_pipelined()
    recs = []
    for i, b in enumerate(batches[:4]):
        net.image_buf.copy_(torch.from_numpy(b))
        t = net.run_pipelined(i & 1)
        net.sync_pipelined()
        recs.append(t.rec.clone())
    for b, rec in zip(batches[:4], recs):
        net.image_buf.copy_(torch.from_numpy(b))
        net.run()
        torch.cuda.synchronize()
        want, got = net.tail.rec.cpu().numpy(), rec.cpu().numpy()
        np.testing.assert_array_equal(got[:, -2:], want[:, -2:])            # counts and overflow flags
        for img in range(want.shape[0]):                                     # rows past the count are stale by design
            n = int(want[img, -2]) * 6
            assert n > 0
            np.testing.assert_array_equal(got[img, :n], want[img, :n])


def test_overflow_is_reported_in_the_record(built):
    """cap < candidates: the status word AND the per-image flag of the packed record report it; the next launch
    with enough capacity is clean again (the status word describes one launch, ADVICE r1)."""
    from odt_b200 import lib as L
    from odt_b200 import nets
    from odt_b200.engine import RowsHarness
    from golden import make_golden as mg
    rows = mg.make_rows("tail_ssd", batch=2, seed=3)
    cfg = model_cfg("ssd", nms_score_threshold=0.05)
    t = nets.ssd_tail(300, cfg)
    t.cap = 8
    h = RowsHarness(t, mg.CASES["tail_ssd"]["levels"], rows)
    with pytest.raises(L.OdtError):
        h.run()
    assert int(h.tail.status.item()) == L.ERR_OVERFLOW
    rec = h.tail.rec.cpu().numpy()
    assert rec[:, -1].max() == 1.0
    t2 = nets.ssd_tail(300, cfg)    # enough capacity: clean status word and flags
    h2 = RowsHarness(t2, mg.CASES["tail_ssd"]["levels"], rows)
    res = h2.run()
    assert int(h2.tail.status.item()) == 0 and len(res) == 2
    rec2 = h2.tail.rec.cpu().numpy()
    assert rec2[:, -1].max() == 0.0 and np.array_equal(rec2[:, -2].astype(np.int32), h2.tail.det_count.cpu().numpy())


def test_halo_layout_does_not_change_results(built, monkeypatch):
    """ODT_HALO=0 (dense NHWC everywhere, im2col path only) vs the default halo-flat path."""
    img = _img(2, 300, 300, seed=5)
    m1 = _model("ssd300", precision="fp16", nms_score_threshold=0.3)
    m1.detect_batch(img)
    a = m1.engine(2).head_buf.cpu().numpy().copy()
    assert any(t.halo for t in m1.engine(2).acts), "halo layout expected on conv1_1/pool1/conv2_1 outputs"
    monkeypatch.setenv("ODT_HALO", "0")
    m2 = _model("ssd300", precision="fp16", nms_score_threshold=0.3)
    m2.detect_batch(img)
    b = m2.engine(2).head_buf.cpu().numpy()
    assert not any(t.halo for t in m2.engine(2).acts)
    assert np.abs(a - b).max() <= 2e-3 * np.abs(b).max()


# BASELINE.json configs at their OWN input sizes (VERDICT r1 weak item 1): the engine makes different choices here
# (halo layouts, CTA pairs, row-block pooling, 12 lanes) than at the 64-128 px shapes above.
FULL = {"ssd300": ({}, 300, 300, 2), "ssd512": ({}, 512, 512, 1),
        "retinanet": ({"data_shape": [800, 800, 3]}, 800, 800, 1),
        "yolov3": ({"data_shape": [416, 416, 3]}, 416, 416, 2),
        "fcos": ({"data_shape": [1024, 1024, 3]}, 1024, 1024, 1)}


@pytest.mark.parametrize("precision,row_tol,ds_tol", [("fp32", 2e-4, 1e-4), ("fp16", 5e-3, 3e-2)])
@pytest.mark.parametrize("kind", ["ssd300", "ssd512", "retinanet", "yolov3", "fcos"])
def test_full_size_end_to_end_decisions(built, kind, precision, row_tol, ds_tol):
    """Whole network at the BASELINE input size, dense score threshold (about 1 % of N candidates per class, taken
    from an oracle quantile), against the oracle's own forward: rows within tolerance, then margin-aware identity
    of class ids and keep indices (tests/margins.py), boxes of the common keeps reported."""
    over, h, w, B = FULL[kind]
    if kind == "fcos" and precision == "fp16":
        row_tol = 1.5e-2  # measured 1.04e-2: GroupNorm re-normalises fp16-stored activations in every layer (a19)
    img = _img(B, h, w, seed=11)
    probe = _model(kind, bn_init="trained", precision=precision, **over)
    ref = _oracle_rows(kind, probe.get_weights(), img, probe.config)
    spec = probe._build_spec()
    geom = _geom(kind, spec, probe.config)
    thr = _dense_threshold(kind, ref, geom, 0.01)
    m = _model(kind, bn_init="trained", precision=precision, nms_score_threshold=thr, **over)
    res = m.detect_batch(img)
    net = m.engine(B)
    rows = net.head_buf.cpu().numpy()
    assert rows.shape == ref.shape and np.isfinite(rows).all()
    scale, err = float(np.abs(ref).max()), float(np.abs(rows - ref).max())
    print("%s %s %dx%d: rows max|err| %.3g of max|ref| %.3g (%.2e rel), threshold %.4f"
          % (kind, precision, h, w, err, scale, err / scale, thr))
    assert err <= row_tol * scale, (kind, precision, err, scale)
    keep_all = net.tail.det_anchor.cpu().numpy()
    ncls = 19 if kind == "fcos" else 20
    mb, iou = m.config["nms_max_boxes"], m.config["nms_iou_threshold"]
    reps = []
    for b in range(B):
        k = len(res[b][2])
        reps.append(MG.compare_image(MKIND[kind], rows[b], ref[b], geom, res[b][2], keep_all[b, :k], res[b][1],
                                     thr, mb, iou, ncls))
    tot = MG.summarize(reps)
    cc = net.tail.cand_count.cpu().numpy()
    print("%s %s: candidates/class mean %.0f max %d; classes clean %d ambiguous %d (reasons %s) identical %d of %d; "
          "keeps oracle %d gpu %d common %d; ds %.3g di %.3g; common-keep box err %.3g px (%.2e rel)"
          % (kind, precision, cc.mean(), cc.max(), tot["clean"], tot["ambiguous"], tot["reasons"], tot["identical"],
             ncls * B, tot["kept_oracle"], tot["kept_gpu"], tot["same_keeps"], tot["ds"], tot["di"], tot["box_err"],
             tot["box_err_rel"]))
    assert cc.mean() >= 10, "dense regime expected (NMS must have work)"
    assert tot["ds"] <= ds_tol, tot
    assert tot["kept_gpu"] > 0 and tot["same_keeps"] >= 0.5 * tot["kept_oracle"], tot


def test_sharded_two_gpus_equals_single(built):
    """N > 1 on real GPUs: image shards on 2 ranks (torchrun, NCCL all-gather of the packed records) give the
    single-GPU detections image for image -- per-batch call, stream, consumer-rank stream (scripts/check_sharded.py)."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29547",
                        os.path.join(root, "scripts", "check_sharded.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "OK" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])


@pytest.mark.parametrize("kind,size", [("ssd300", 300), ("retinanet", 128), ("yolov3", 160), ("fcos", 256)])
def test_training_step_on_gpu(built, kind, size):
    """train_one_epoch's step on the GPU (odt_b200/train.py) for every family: training-mode forward of the engine's
    layer list, loss, backward, Momentum.  The autograd loss agrees with the hand-written CUDA loss-forward kernel of the
    family (csrc/loss.cu) on the same rows, the step changes the variables, and the updated weights flow into the
    inference engines."""
    import torch
    from odt_b200 import nets
    from odt_b200.engine import RowsHarness
    rng = np.random.default_rng(3)
    img = _img(2, size, size, seed=8)
    gt = np.full((2, 10, 5), -1.0, np.float32)
    for b in range(2):
        n = 3 + 2 * b
        gt[b, :n, 0:2] = rng.uniform(0.2 * size, 0.8 * size, (n, 2))
        gt[b, :n, 2:4] = rng.uniform(0.1 * size, 0.5 * size, (n, 2))
        gt[b, :n, 4] = rng.integers(0, 20, n)

    class It:
        def get_next(self):
            return img, gt
    provider = {"data_shape": [size, size, 3], "num_train": 2, "num_val": 0, "train_generator": ((lambda: None), It()),
                "val_generator": None}
    import FCOS
    import RetinaNet
    import SSD300
    import YOLOv3
    over = {} if kind == "ssd300" else {"data_shape": [size, size, 3]}
    cls, ckind, lkind = {"ssd300": (SSD300.SSD300, "ssd", "ssd"), "retinanet": (RetinaNet.RetinaNet, "retinanet", "retina"),
                         "yolov3": (YOLOv3.YOLOv3, "yolov3", "yolo"), "fcos": (FCOS.FCOS, "fcos", "fcos")}[kind]
    m = cls(model_cfg(ckind, mode="train", batch_size=2, bn_init="trained", **over), provider)
    tr = m.trainer()
    assert tr.device.type == "cuda"
    rows = tr.forward_rows(img)
    per = [float(tr.image_loss(rows[b], gt[b])) for b in range(2)]
    tail = {"ssd": lambda: nets.ssd_tail(300, m.config), "retina": lambda: nets.retina_tail(m.config),
            "yolo": lambda: nets.yolo_tail(m.config), "fcos": lambda: nets.fcos_tail(m.config)}[lkind]()
    hrn = RowsHarness(tail, list(tr.net.levels), rows.detach().cpu().numpy())
    kw = {}
    if lkind == "retina":
        kw = dict(alpha=m.config["alpha"], gamma=m.config["gamma"])
    if lkind == "yolo":
        kw = dict(coord_scale=m.config["coord_scale"], noobj_scale=m.config["noobj_scale"],
                  obj_scale=m.config["obj_scale"], class_scale=m.config["class_scale"])
    got = hrn.loss(lkind, gt, **kw)
    for b in range(2):
        print("%s image %d: autograd loss %.6f, CUDA loss-forward kernel %.6f" % (kind, b, per[b], got[b]))
        assert abs(per[b] - got[b]) <= 1e-4 * max(abs(per[b]), 1.0)
    w0 = {k: v.detach().clone() for k, v in tr.params.items()}
    loss = m.train_one_epoch(1e-3)
    assert np.isfinite(loss) and m.global_step == 1
    changed = sum(int(not torch.equal(w0[k], tr.params[k].detach())) for k in w0)
    assert changed >= 0.95 * len(w0), "(nearly) every trainable variable receives a gradient (data term or weight decay)"
    res = m.detect_batch(img[:1])          # inference engine rebuilt from the updated variables
    assert len(res) == 1
