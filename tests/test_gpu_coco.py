"""ops.COCODetectionEval / yb_coco_match / yb_coco_precision against the kernels' form of the oracle
(oracle/coco_ref.py evaluate, itself checked against the literal pycocotools transcription in test_coco_cpu.py).

Records, ground-truth counts and the precision / recall tables are compared bit for bit; the stats (means the host
takes) within 1e-12."""
import types

import numpy as np
import pytest
import torch

from yolo_from_scratch_b200 import ops
from oracle import coco_ref as C
from oracle import ref_path as R
from eval_data import _PresetHeads, _train_stand_in, host_images, packed, prior_heads
from eval_data import coco_synthetic_batch as synthetic_batch

pytestmark = pytest.mark.gpu
THR = np.asarray(ops.COCO_IOU_THRESHOLDS)
REC = np.asarray(ops.COCO_RECALL_THRESHOLDS)


def check_against_oracle(got, want):
    assert np.array_equal(got["precision"], want["precision"])
    assert np.array_equal(got["recall"], want["recall"])
    assert np.array_equal(got["n_gt"], want["n_gt"]) and np.array_equal(got["n_det"], want["n_det"])
    assert np.allclose(got["stats"], want["stats"], rtol=0, atol=1e-12)
    assert np.allclose(got["ap"], want["ap"], rtol=0, atol=1e-12)
    assert abs(got["map"] - want["map"]) <= 1e-12
    if want["map50"] is None:
        assert got["map50"] is None
    else:
        assert abs(got["map50"] - want["map50"]) <= 1e-12


@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("max_gt", [50, 200])
@pytest.mark.parametrize("max_det", [100, 300, "cap"])
def test_match_records_are_bit_exact(nc, max_gt, max_det):
    rng = np.random.default_rng(nc * 1000 + max_gt + (0 if max_det == "cap" else max_det))
    B, cap = 48, 360
    det, host, (labels, lb) = synthetic_batch(rng, B, nc, max_gt, cap)
    md = cap if max_det == "cap" else max_det
    metric = ops.COCODetectionEval(nc, max_det=md)
    metric.update(det, packed(labels, lb, max_gt=max_gt))
    got = torch.cat(metric._records).cpu().numpy()
    slots = min(md, cap)
    gt_count = np.zeros((4, nc), np.int64)
    areas = []
    for b, im in enumerate(host):
        rec, g, st = C.image_records(im, nc, THR, md)
        want = C.pack_records(rec)
        sl = slice(b * slots, (b + 1) * slots)
        assert np.array_equal(got[sl], want), (b, np.flatnonzero((got[sl] != want).any(1))[:5])
        gt_count += g
        assert st == 0
        gb, _, db, _, _, _ = C._image_inputs(im, nc, md)
        areas += [C.box_area(gb), C.box_area(db.astype(np.float64))]
    assert np.array_equal(metric._gt_count.cpu().numpy(), gt_count)
    assert int(metric._status.item()) == 0
    areas = np.concatenate(areas)
    assert np.any(areas == 32.0 ** 2) and np.any(areas == 96.0 ** 2)   # the range bounds themselves occur
    words = got.view(np.uint16).reshape(-1, 16)
    tp, ig = words[:, 6:10], words[:, 10:14]
    assert np.count_nonzero(tp[:, 0]) > 50 and np.count_nonzero(tp[:, 0] & 1) > np.count_nonzero(tp[:, 0] & (1 << 9))
    assert all(np.count_nonzero(ig[:, a]) > 0 and np.count_nonzero(tp[:, a]) > 0 for a in (1, 2, 3))
    if nc < 80:
        assert np.count_nonzero(words[:, 4] >= 10) > 0   # ranks past maxDets[1]


@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("max_dets", [(1, 10, 100), (1, 5, 20)])
def test_tables_are_bit_exact(nc, max_dets):
    rng = np.random.default_rng(nc + 7 * max_dets[1])
    metric = ops.COCODetectionEval(nc, max_dets=max_dets)
    det, host, (labels, lb) = synthetic_batch(rng, 48, nc, 50, 300)
    metric.update(det, packed(labels, lb))
    got = metric.compute()
    want = C.evaluate(host, nc, THR, REC, max_det=300, max_dets=max_dets)
    assert got["precision"].shape == (10, 101, nc, 4, 3) and got["recall"].shape == (10, nc, 4, 3)
    assert got["stats"].shape == (12,) and got["n_gt"].shape == (nc, 4)
    check_against_oracle(got, want)
    assert (got["stats"][0] == -1) == (100 not in max_dets)
    assert np.all(got["stats"][1:] > 0)


@pytest.mark.parametrize("nc", [1, 3, 80])
def test_accumulation_over_20_updates(nc):
    rng = np.random.default_rng(20 + nc)
    metric = ops.COCODetectionEval(nc)
    images = []
    for _ in range(20):
        det, host, (labels, lb) = synthetic_batch(rng, 8, nc, 30, 120)
        metric.update(det, packed(labels, lb))
        images += host
    got = metric.compute()
    check_against_oracle(got, C.evaluate(images, nc, THR, REC))
    assert 0 < got["stats"][0] < 1
    metric.reset()
    empty = metric.compute()
    assert np.all(empty["stats"] == -1) and np.all(empty["precision"] == -1) and np.all(empty["n_gt"] == 0)


def test_custom_thresholds():
    rng = np.random.default_rng(3)
    thr, rec = [0.3, 0.6, 0.75], np.linspace(0, 1, 11)
    metric = ops.COCODetectionEval(3, iou_thresholds=thr, recall_thresholds=rec, max_det=50, max_dets=(2, 4, 8))
    det, host, (labels, lb) = synthetic_batch(rng, 16, 3, 20, 80)
    metric.update(det, packed(labels, lb))
    got = metric.compute()
    check_against_oracle(got, C.evaluate(host, 3, thr, rec, max_det=50, max_dets=(2, 4, 8)))
    assert got["map50"] is None and got["stats"][0] == -1 and got["stats"][1] == -1 and got["stats"][2] > 0


def test_tables_equal_detection_map_where_the_protocols_agree():
    """Every area inside [0, 1e10] and at most 90 < maxDets[-1] detections of a class per image: the (all, 100)
    slice is DetectionMAP's table bit for bit."""
    rng = np.random.default_rng(17)
    coco, dmap = ops.COCODetectionEval(3), ops.DetectionMAP(3)
    for _ in range(4):
        det, host, (labels, lb) = synthetic_batch(rng, 16, 3, 40, 90)
        lab = packed(labels, lb)
        coco.update(det, lab)
        dmap.update(det, lab)
    got, want = coco.compute(), dmap.compute()
    assert np.array_equal(got["precision"][..., 0, 2], want["precision"])
    assert np.array_equal(got["recall"][..., 0, 2], want["recall"])
    assert np.array_equal(got["n_gt"][:, 0], want["n_gt"]) and np.array_equal(got["n_det"], want["n_det"])
    assert got["map"] == want["map"] and got["map50"] == want["map50"] and np.array_equal(got["ap"], want["ap"])


@pytest.mark.parametrize("nc", [1, 80])
def test_end_to_end_from_heads(nc):
    """prior heads + labels -> detect_batch(letterbox=...) -> update.  Half of the ground truths are jittered copies
    of kept detections, so there are TPs at every threshold and in every range."""
    rng = np.random.default_rng(nc)
    img, B = 320, 8
    metric = ops.COCODetectionEval(nc)
    images = []
    for step in range(3):
        heads = prior_heads(B, img, nc, 100 + step)
        lbx = [(float(rng.uniform(0.5, 1.5)), float(rng.integers(0, 20)), float(rng.integers(0, 20))) for _ in range(B)]
        det = ops.detect_batch(heads, R.default_anchors(), img, nc, conf_threshold=0.001, iou_threshold=0.4, letterbox=lbx)
        hb = host_images(det, [None] * B, [None] * B)
        labels, letterbox = [], []
        for b in range(B):
            ow, oh = (img - 2 * lbx[b][2]) / lbx[b][0], (img - 2 * lbx[b][1]) / lbx[b][0]
            k = hb[b]["keep"][:min(hb[b]["n_keep"], 25)]
            bx = hb[b]["boxes"][k].astype(np.float64) + rng.normal(0, 2, (len(k), 4))
            lab = np.column_stack([hb[b]["classes"][k], (bx[:, 0] + bx[:, 2]) / 2 / ow, (bx[:, 1] + bx[:, 3]) / 2 / oh,
                                   np.abs(bx[:, 2] - bx[:, 0]) / ow, np.abs(bx[:, 3] - bx[:, 1]) / oh])
            extra = np.column_stack([rng.integers(0, nc, 5), rng.uniform(0.1, 0.9, (5, 2)), rng.uniform(0.05, 0.3, (5, 2))])
            labels.append(np.concatenate([lab, extra]).reshape(-1, 5))
            letterbox.append((ow, oh) + lbx[b])
        metric.update(det, ops.pack_labels(labels, img, letterbox))
        images += host_images(det, labels, letterbox)
    got = metric.compute()
    check_against_oracle(got, C.evaluate(images, nc, THR, REC))
    assert got["map50"] > 0.1 and got["n_det"].sum() > 0


def test_empty_cases():
    rng = np.random.default_rng(9)
    metric = ops.COCODetectionEval(3)
    det, host, (labels, lb) = synthetic_batch(rng, 16, 3, 10, 40, n_keep_zero=0.5)
    for b in range(0, 16, 3):
        labels[b] = np.zeros((0, 5))
        host[b]["labels"] = labels[b]
    metric.update(det, packed(labels, lb))
    check_against_oracle(metric.compute(), C.evaluate(host, 3, THR, REC))
    metric = ops.COCODetectionEval(3)
    det["n_keep"].zero_()
    for im in host:
        im["n_keep"] = 0
    metric.update(det, packed(labels, lb))
    got = metric.compute()
    check_against_oracle(got, C.evaluate(host, 3, THR, REC))
    assert np.all(got["n_det"] == 0) and np.all(np.isin(got["stats"], (0.0, -1.0)))
    got = ops.COCODetectionEval(5).compute()
    assert np.all(got["stats"] == -1) and got["map"] == -1 and got["ap"].shape == (5, 10)
    assert np.all(got["recall"] == -1) and np.all(got["n_det"] == 0) and got["n_gt"].shape == (5, 4)
    # max_det 0: no records at all
    metric = ops.COCODetectionEval(3, max_det=0)
    metric.update(det, packed(labels, lb))
    got = metric.compute()
    assert np.all(got["n_det"] == 0) and np.all(got["recall"][:, got["n_gt"][:, 0] > 0, 0] == 0)


def test_errors():
    rng = np.random.default_rng(11)
    det, host, (labels, lb) = synthetic_batch(rng, 4, 3, 10, 20, n_keep_zero=0.0)
    bad = [l.copy() for l in labels]
    bad[1] = np.array([[5, 0.5, 0.5, 0.2, 0.2]])
    metric = ops.COCODetectionEval(3)
    metric.update(det, packed(bad, lb))
    with pytest.raises(IndexError):
        metric.compute()
    metric = ops.COCODetectionEval(3)
    det["n_keep"][2] = -1
    metric.update(det, packed(labels, lb))
    with pytest.raises(RuntimeError, match="NMS failed"):
        metric.compute()
    with pytest.raises(ValueError):
        ops.COCODetectionEval(3, iou_thresholds=np.linspace(0.1, 0.9, 17))
    with pytest.raises(ValueError):
        ops.COCODetectionEval(3, recall_thresholds=[0.0, 0.5, 0.25])
    for md in ((1, 10), (0, 10, 100), (1, 10, 65536), (1, 10, 100, 300)):
        with pytest.raises(ValueError):
            ops.COCODetectionEval(3, max_dets=md)


def test_update_does_not_synchronise():
    rng = np.random.default_rng(12)
    det, host, (labels, lb) = synthetic_batch(rng, 8, 3, 20, 60)
    lab = packed(labels, lb)
    metric = ops.COCODetectionEval(3)
    metric.update(det, lab)   # first call: library load and module initialisation
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            metric.update(det, lab)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    check_against_oracle(metric.compute(), C.evaluate(host * 4, 3, THR, REC))


def test_evaluate_coco_through_install(tmp_path):
    from PIL import Image
    from yolo_from_scratch_b200.install import install, uninstall
    nc, img, scale, pt, pl = 3, 160, 0.8, 16, 0
    wh = (200, 160)
    rng = np.random.default_rng(13)
    heads = prior_heads(3, img, nc, 7)
    model = _PresetHeads(heads, img, [a.cuda() for a in R.default_anchors()])
    imgs, lab_files, labels = [], [], []
    for i in range(7):
        p = tmp_path / f"im{i}.png"
        Image.fromarray(np.zeros((wh[1], wh[0], 3), dtype=np.uint8)).save(p)
        imgs.append(str(p))
        lf = tmp_path / f"im{i}.txt"
        lab = np.column_stack([rng.integers(0, nc, 4), rng.uniform(0.2, 0.8, (4, 2)), rng.uniform(0.05, 0.4, (4, 2))])
        if i != 4:   # image 4 has no label file: no objects
            with open(lf, "w") as f:
                for r in lab:
                    f.write(f"{int(r[0])} {r[1]} {r[2]} {r[3]} {r[4]}\n")
        else:
            lab = np.zeros((0, 5))
        lab_files.append(str(lf))
        labels.append(np.column_stack([lab[:, 0].astype(np.int64), lab[:, 1:]]).astype(np.float64).reshape(-1, 5))
    dataset = types.SimpleNamespace(imgs=imgs, labels=lab_files)
    train = install(_train_stand_in(scale, pt, pl))
    try:
        got = train.evaluate_coco(model, dataset, torch.device("cuda"), num_classes=nc, batch_size=3, max_dets=(1, 5, 50))
        assert hasattr(train, "evaluate_map")
    finally:
        uninstall(train)
    assert not hasattr(train, "evaluate_coco") and not hasattr(train, "evaluate_map")
    images = []
    for i0 in range(0, 7, 3):
        n = min(3, 7 - i0)
        lbx = [(scale, pt, pl)] * n
        det = ops.detect_batch([h[:n] for h in heads], R.default_anchors(), img, nc, 0.001, 0.4, letterbox=lbx)
        images += host_images(det, labels[i0:i0 + n], [wh + (scale, pt, pl)] * n)
    check_against_oracle(got, C.evaluate(images, nc, THR, REC, max_det=300, max_dets=(1, 5, 50)))
    assert got["n_gt"][:, 0].sum() == 24 and len(ops.format_coco_stats(got["stats"], THR, (1, 5, 50))) == 12
