"""ops.DetectionMAP / yb_map_match / yb_map_precision against the numpy oracle (oracle/map_ref.py).

Records, ground-truth counts and the precision / recall tables are compared bit for bit; ap, map and map50 (means
the host takes) within 1e-12."""
import types

import numpy as np
import pytest
import torch

import yolo_from_scratch_b200 as yb
from yolo_from_scratch_b200 import ops
from oracle import map_ref as M
from oracle import ref_path as R
from eval_data import _PresetHeads, _train_stand_in, host_images, packed, prior_heads, synthetic_batch

pytestmark = pytest.mark.gpu
THR = np.asarray(ops.COCO_IOU_THRESHOLDS)
REC = np.asarray(ops.COCO_RECALL_THRESHOLDS)


def device_records(metric):
    rec = torch.cat(metric._records).cpu().numpy()
    return rec[:, 0].view(np.float32), rec[:, 1], rec[:, 2]


@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("max_gt", [50, 200])
@pytest.mark.parametrize("max_det", [100, 300, "cap"])
def test_match_records_are_bit_exact(nc, max_gt, max_det):
    rng = np.random.default_rng(nc * 1000 + max_gt + (0 if max_det == "cap" else max_det))
    B, cap = 64, 360
    det, host, (labels, lb) = synthetic_batch(rng, B, nc, max_gt, cap)
    md = cap if max_det == "cap" else max_det
    metric = ops.DetectionMAP(nc, max_det=md)
    metric.update(det, packed(labels, lb, max_gt=max_gt))
    sc, cl, tp = device_records(metric)
    slots = min(md, cap)
    n_gt = np.zeros(nc, np.int64)
    for b, im in enumerate(host):
        s, c, m, g, st = M.image_records(im["boxes"], im["scores"], im["classes"], im["keep"], im["n_keep"], im["labels"],
                                         im["letterbox"], nc, THR, md, slots)
        sl = slice(b * slots, (b + 1) * slots)
        assert np.array_equal(sc[sl].view(np.int32), s.view(np.int32)), b
        assert np.array_equal(cl[sl], c), b
        assert np.array_equal(tp[sl], m.astype(np.int32)), (b, np.flatnonzero(tp[sl] != m)[:5])
        n_gt += g
        assert st == 0
    assert np.array_equal(metric._gt_count.cpu().numpy(), n_gt)
    assert int(metric._status.item()) == 0
    assert np.count_nonzero(tp) > 50 and np.count_nonzero(tp & 1) > np.count_nonzero(tp & (1 << 9))   # thresholds bite


def check_against_oracle(got, want):
    assert np.array_equal(got["precision"], want["precision"])
    assert np.array_equal(got["recall"], want["recall"])
    assert np.array_equal(got["n_gt"], want["n_gt"]) and np.array_equal(got["n_det"], want["n_det"])
    assert np.allclose(got["ap"], want["ap"], rtol=0, atol=1e-12)
    assert abs(got["map"] - want["map"]) <= 1e-12
    if want["map50"] is None:
        assert got["map50"] is None
    else:
        assert abs(got["map50"] - want["map50"]) <= 1e-12


@pytest.mark.parametrize("nc", [1, 3, 80])
def test_accumulation_over_20_updates(nc):
    rng = np.random.default_rng(20 + nc)
    metric = ops.DetectionMAP(nc)
    images = []
    for _ in range(20):
        det, host, (labels, lb) = synthetic_batch(rng, 8, nc, 30, 120)
        metric.update(det, packed(labels, lb))
        images += host
    got = metric.compute()
    want = M.evaluate(images, nc, THR, REC, max_det=300)
    assert got["precision"].shape == (10, 101, nc) and got["recall"].shape == (10, nc) and got["ap"].shape == (nc, 10)
    check_against_oracle(got, want)
    assert 0 < got["map"] < 1
    metric.reset()
    empty = metric.compute()
    assert empty["map"] == -1 and np.all(empty["precision"] == -1) and np.all(empty["n_gt"] == 0)


def test_custom_thresholds_without_050():
    rng = np.random.default_rng(3)
    thr, rec = [0.3, 0.6, 0.75], np.linspace(0, 1, 11)
    metric = ops.DetectionMAP(3, iou_thresholds=thr, recall_thresholds=rec, max_det=50)
    det, host, (labels, lb) = synthetic_batch(rng, 16, 3, 20, 80)
    metric.update(det, packed(labels, lb))
    got = metric.compute()
    check_against_oracle(got, M.evaluate(host, 3, thr, rec, max_det=50))
    assert got["map50"] is None


@pytest.mark.parametrize("nc", [1, 80])
def test_end_to_end_from_heads(nc):
    """prior heads + labels -> detect_batch(letterbox=...) -> update.  The oracle gets the device's own kept
    detections; half of the ground truths are jittered copies of them, so there are TPs at every threshold."""
    rng = np.random.default_rng(nc)
    img, B = 320, 8
    metric = ops.DetectionMAP(nc)
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
    check_against_oracle(got, M.evaluate(images, nc, THR, REC, max_det=300))
    assert got["map50"] > 0.1 and got["n_det"].sum() > 0


def test_empty_cases():
    rng = np.random.default_rng(9)
    # images without detections and images without ground truth, mixed
    metric = ops.DetectionMAP(3)
    det, host, (labels, lb) = synthetic_batch(rng, 16, 3, 10, 40, n_keep_zero=0.5)
    for b in range(0, 16, 3):
        labels[b] = np.zeros((0, 5))
        host[b]["labels"] = labels[b]
    metric.update(det, packed(labels, lb))
    check_against_oracle(metric.compute(), M.evaluate(host, 3, THR, REC))
    # n_keep == 0 everywhere: classes with ground truth read 0, the rest -1
    metric = ops.DetectionMAP(3)
    det["n_keep"].zero_()
    for im in host:
        im["n_keep"] = 0
    metric.update(det, packed(labels, lb))
    got = metric.compute()
    check_against_oracle(got, M.evaluate(host, 3, THR, REC))
    assert np.all(got["n_det"] == 0) and got["map"] in (0.0, -1.0)
    # an accumulator that never saw a batch
    got = ops.DetectionMAP(5).compute()
    assert got["map"] == -1 and got["map50"] == -1 and np.all(got["ap"] == -1) and got["ap"].shape == (5, 10)
    assert np.all(got["recall"] == -1) and np.all(got["n_det"] == 0)


def test_errors():
    rng = np.random.default_rng(11)
    det, host, (labels, lb) = synthetic_batch(rng, 4, 3, 10, 20, n_keep_zero=0.0)
    bad = [l.copy() for l in labels]
    bad[1] = np.array([[5, 0.5, 0.5, 0.2, 0.2]])
    metric = ops.DetectionMAP(3)
    metric.update(det, packed(bad, lb))
    with pytest.raises(IndexError):
        metric.compute()
    metric = ops.DetectionMAP(3)
    det["n_keep"][2] = -1
    metric.update(det, packed(labels, lb))
    with pytest.raises(RuntimeError, match="NMS failed"):
        metric.compute()
    with pytest.raises(ValueError):
        ops.DetectionMAP(3, iou_thresholds=np.linspace(0.1, 0.9, 17))


def test_update_does_not_synchronise():
    rng = np.random.default_rng(12)
    det, host, (labels, lb) = synthetic_batch(rng, 8, 3, 20, 60)
    lab = packed(labels, lb)
    metric = ops.DetectionMAP(3)
    metric.update(det, lab)   # first call: library load and module initialisation
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            metric.update(det, lab)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    check_against_oracle(metric.compute(), M.evaluate(host * 4, 3, THR, REC))


def test_evaluate_map_through_install(tmp_path):
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
                f.write("1 0.5 0.5 0.1\n")   # not five fields: skipped, as YOLODataset.__getitem__ skips it
        else:
            lab = np.zeros((0, 5))
        lab_files.append(str(lf))
        labels.append(np.column_stack([lab[:, 0].astype(np.int64), lab[:, 1:]]).astype(np.float64).reshape(-1, 5))
    dataset = types.SimpleNamespace(imgs=imgs, labels=lab_files)
    train = install(_train_stand_in(scale, pt, pl))
    try:
        got = train.evaluate_map(model, dataset, torch.device("cuda"), num_classes=nc, batch_size=3)
    finally:
        uninstall(train)
    assert not hasattr(train, "evaluate_map")
    # the oracle on the same detections: batches of 3, 3, 1 images, each fed the first n rows of the preset heads
    images = []
    for i0 in range(0, 7, 3):
        n = min(3, 7 - i0)
        lbx = [(scale, pt, pl)] * n
        det = ops.detect_batch([h[:n] for h in heads], R.default_anchors(), img, nc, 0.001, 0.4, letterbox=lbx)
        images += host_images(det, labels[i0:i0 + n], [wh + (scale, pt, pl)] * n)
    check_against_oracle(got, M.evaluate(images, nc, THR, REC, max_det=300))
    assert got["n_gt"].sum() == 24
