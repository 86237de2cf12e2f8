"""ops.DetectionReport / yb_report_match against the numpy oracle (oracle/report_ref.py).

The confusion matrix, the images per class and both histograms are integer counts and are compared exactly; the
curves, best_conf and p/r/f1 come from the same counts through the same fp64 expressions and are compared exactly too.
The AP columns must equal a plain DetectionMAP fed the same batches bit for bit."""
import pathlib
import types

import numpy as np
import pytest
import torch

from yolo_from_scratch_b200 import ops
from oracle import ref_path as R
from oracle import map_ref as M
from oracle import report_ref as P

pytestmark = pytest.mark.gpu
THR = np.asarray(ops.COCO_IOU_THRESHOLDS)
GRID = np.asarray(ops.DEFAULT_CONF_GRID)
# scores are multiples of 1/40 in fp32: this grid holds each of them exactly, plus random points
CUSTOM = dict(cm_conf=0.6, cm_iou=0.3, curve_iou=0.75,
              grid=np.unique(np.concatenate([np.float32(np.arange(41) / 40).astype(np.float64),
                                             np.random.default_rng(5).uniform(0, 1, 60)])))
DEFAULT = dict(cm_conf=0.25, cm_iou=0.45, curve_iou=0.5, grid=GRID)


def synthetic_batch(rng, B, nc, max_gt, cap, n_keep_zero=0.1):
    """Clustered ground truth with jittered detections: many IoUs near the thresholds, duplicated ground truths
    (equal IoU) and quantised scores (equal scores, scores on grid points).  Candidates are in a random order and keep
    lists them by descending score, as NMS does.  Returns (det dict on the GPU, per-image host dicts for the oracle,
    PackedLabels inputs)."""
    boxes = np.zeros((B, cap, 4), np.float32)
    scores = np.zeros((B, cap), np.float32)
    classes = np.zeros((B, cap), np.int64)
    keep = np.zeros((B, cap), np.int64)
    n_keep = np.zeros(B, np.int32)
    labels, letterbox, host = [], [], []
    for b in range(B):
        ow, oh = float(rng.integers(200, 800)), float(rng.integers(200, 800))
        n = int(rng.integers(0, max_gt + 1)) if rng.uniform() > 0.1 else 0
        centres = rng.uniform(0.2, 0.8, (max(1, n // 8 + 1), 2))
        lab = np.zeros((n, 5))
        lab[:, 0] = rng.integers(0, nc, n)
        lab[:, 1:3] = centres[rng.integers(0, len(centres), n)] + rng.normal(0, 0.02, (n, 2))
        lab[:, 3:5] = rng.uniform(0.05, 0.3, (n, 2))
        if n >= 4:
            lab[n // 2] = lab[n // 4]                                           # duplicate: equal IoU
        gb, _, _ = M.gt_boxes(lab, (ow, oh), max(nc, 2))
        m = int(rng.integers(0, cap + 1))
        src = rng.integers(0, max(n, 1), m)
        jit = rng.normal(0, 1, (m, 4)) * rng.choice([0.0, 2.0, 8.0], (m, 1))
        bx = (gb[src] + jit) if n else rng.uniform(0, 400, (m, 4))
        bx = np.concatenate([np.minimum(bx[:, :2], bx[:, 2:]), np.maximum(bx[:, :2], bx[:, 2:])], 1)
        if m:
            boxes[b, :m] = bx
            scores[b, :m] = np.round(rng.uniform(0.001, 1, m) * 40) / 40
            classes[b, :m] = np.where(rng.uniform(size=m) < 0.8, lab[src, 0] if n else 0, rng.integers(0, nc, m)) % nc
        order = np.argsort(-scores[b, :m], kind="stable")
        keep[b, :m] = order
        n_keep[b] = 0 if rng.uniform() < n_keep_zero else m
        labels.append(lab)
        letterbox.append((ow, oh, 1.0, 0.0, 0.0))
        host.append({"boxes": boxes[b], "scores": scores[b], "classes": classes[b], "keep": keep[b],
                     "n_keep": int(n_keep[b]), "labels": lab, "letterbox": letterbox[-1]})
    dev = torch.device("cuda")
    det = {"boxes": torch.from_numpy(boxes).to(dev), "scores": torch.from_numpy(scores).to(dev),
           "classes": torch.from_numpy(classes).to(dev), "keep": torch.from_numpy(keep).to(dev),
           "n_keep": torch.from_numpy(n_keep).to(dev)}
    return det, host, (labels, letterbox)


def packed(labels, letterbox, max_gt=None):
    lab, n_gt, lb = ops.pack_labels_host(labels, 640, letterbox, max_gt=max_gt)
    return ops.PackedLabels(lab.cuda(), n_gt.cuda(), lb.cuda(), 640)


def report(nc, params, max_det=300):
    return ops.DetectionReport(nc, max_det=max_det, conf_grid=params["grid"], curve_iou=params["curve_iou"],
                               cm_conf=params["cm_conf"], cm_iou=params["cm_iou"])


def oracle(images, nc, params, max_det=300):
    return P.evaluate(images, nc, THR, params["grid"], curve_iou=params["curve_iou"], cm_conf=params["cm_conf"],
                      cm_iou=params["cm_iou"], max_det=max_det)


def check_counts(rep, want):
    assert np.array_equal(rep._confusion.cpu().numpy(), want["confusion"])
    assert np.array_equal(rep._images.cpu().numpy(), want["images"])
    assert np.array_equal(rep._det_hist.cpu().numpy(), want["det_hist"])
    assert np.array_equal(rep._tp_hist.cpu().numpy(), want["tp_hist"])


def check_report(got, want):
    for k in ("confusion", "images", "px", "p_curve", "r_curve", "f1_curve", "p", "r", "f1", "n_gt", "n_det",
              "precision", "recall"):
        assert np.array_equal(got[k], want[k]), k
    assert got["best_conf"] == want["best_conf"] and got["images_total"] == want["images_total"]
    assert ops.format_detection_report(got) == ops.format_detection_report(want)


@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("max_gt,max_det,B,cap", [(50, 100, 64, 360), (200, 300, 32, 360), (30, "cap", 32, 700),
                                                  (4096, 300, 3, 320)])
@pytest.mark.parametrize("params", ["default", "custom"])
def test_counts_are_bit_exact(nc, max_gt, max_det, B, cap, params):
    """|D| up to 700 slots (more than the CTA's 256 threads) and max_gt 4096 (the largest staging)."""
    prm = DEFAULT if params == "default" else CUSTOM
    rng = np.random.default_rng(nc * 1000 + max_gt + cap + len(params))
    det, host, (labels, lb) = synthetic_batch(rng, B, nc, max_gt, cap)
    md = cap if max_det == "cap" else max_det
    rep = report(nc, prm, max_det=md)
    rep.update(det, packed(labels, lb, max_gt=max_gt))
    want = oracle(host, nc, prm, max_det=md)
    check_counts(rep, want)
    check_report(rep.compute(), want)
    assert want["confusion"][:nc, :nc].trace() > 0 and want["tp_hist"].sum() > 0   # matches and TPs do occur


@pytest.mark.parametrize("nc", [1, 3, 80])
def test_accumulation_over_20_updates_and_ap_columns(nc):
    rng = np.random.default_rng(20 + nc)
    rep = ops.DetectionReport(nc)
    plain = ops.DetectionMAP(nc)
    images = []
    for _ in range(20):
        det, host, (labels, lb) = synthetic_batch(rng, 8, nc, 30, 120)
        lab = packed(labels, lb)
        rep.update(det, lab)
        plain.update(det, lab)
        images += host
    got = rep.compute()
    want = oracle(images, nc, DEFAULT)
    check_counts(rep, want)
    check_report(got, want)
    ref = plain.compute()
    for k in ("precision", "recall", "ap", "n_gt", "n_det"):
        assert np.array_equal(got[k], ref[k]), k
    assert got["map"] == ref["map"] and got["map50"] == ref["map50"]
    assert got["best_conf"] is not None and got["images_total"] == 160
    rep.reset()
    empty = rep.compute()
    assert empty["confusion"].sum() == 0 and empty["best_conf"] is None and empty["images_total"] == 0


@pytest.mark.parametrize("nc", [1, 5])
def test_invariants(nc):
    grid = np.concatenate([[-1.0], GRID])   # every score is above grid[0]
    rng = np.random.default_rng(40 + nc)
    rep = ops.DetectionReport(nc, conf_grid=grid)
    images = []
    for _ in range(4):
        det, host, (labels, lb) = synthetic_batch(rng, 16, nc, 40, 200)
        rep.update(det, packed(labels, lb))
        images += host
    got = rep.compute()
    cmx = got["confusion"]
    assert np.array_equal(cmx[:, :nc].sum(axis=0), got["n_gt"]) and cmx[nc, nc] == 0
    above = np.zeros(nc, np.int64)
    for im in images:
        idx = im["keep"][:max(0, min(im["n_keep"], 300))]
        sel = im["scores"][idx].astype(np.float64) > 0.25
        above += np.bincount(im["classes"][idx][sel], minlength=nc)
    assert np.array_equal(cmx[:nc].sum(axis=1), above)
    assert np.array_equal(rep._det_hist.sum(dim=1).cpu().numpy(), got["n_det"])


def prior_heads(B, img, nc, seed):
    g = torch.Generator().manual_seed(seed)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (img // 8, img // 16, img // 32)]
    for h in heads:
        h[..., 4].mul_(2.0).sub_(4.6)   # SURVEY 8d "prior" heads
    return [h.cuda() for h in heads]


def host_images(det, labels, letterbox):
    d = {k: det[k].cpu().numpy() for k in ("boxes", "scores", "classes", "keep", "n_keep")}
    return [{"boxes": d["boxes"][b], "scores": d["scores"][b], "classes": d["classes"][b], "keep": d["keep"][b],
             "n_keep": int(d["n_keep"][b]), "labels": labels[b], "letterbox": letterbox[b]} for b in range(len(labels))]


@pytest.mark.parametrize("nc", [1, 80])
def test_end_to_end_from_heads(nc):
    """prior heads + labels -> detect_batch(letterbox=...) -> update.  The oracle gets the device's own kept
    detections; half of the ground truths are jittered copies of them, so the matrix has matches."""
    rng = np.random.default_rng(nc)
    img, B = 320, 8
    rep = ops.DetectionReport(nc, cm_conf=0.05)
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
        rep.update(det, ops.pack_labels(labels, img, letterbox))
        images += host_images(det, labels, letterbox)
    got = rep.compute()
    want = P.evaluate(images, nc, THR, GRID, cm_conf=0.05)
    check_counts(rep, want)
    check_report(got, want)
    assert got["confusion"][:nc, :nc].sum() > 0 and int(rep._tp_hist.sum()) > 0


def test_empty_cases():
    rng = np.random.default_rng(9)
    # images without detections and images without ground truth, mixed
    rep = ops.DetectionReport(3)
    det, host, (labels, lb) = synthetic_batch(rng, 16, 3, 10, 40, n_keep_zero=0.5)
    for b in range(0, 16, 3):
        labels[b] = np.zeros((0, 5))
        host[b]["labels"] = labels[b]
    rep.update(det, packed(labels, lb))
    want = oracle(host, 3, DEFAULT)
    check_counts(rep, want)
    check_report(rep.compute(), want)
    # no detections at all: every ground truth is in the background row, P = 1 and R = 0 everywhere
    rep = ops.DetectionReport(3)
    det["n_keep"].zero_()
    for im in host:
        im["n_keep"] = 0
    rep.update(det, packed(labels, lb))
    got = rep.compute()
    check_report(got, oracle(host, 3, DEFAULT))
    assert got["confusion"][:3].sum() == 0 and np.array_equal(got["confusion"][3, :3], got["n_gt"])
    # no ground truth at all: detections above cm_conf are in the background column, no best threshold
    rep = ops.DetectionReport(3)
    det, host, (labels, lb) = synthetic_batch(rng, 8, 3, 10, 40, n_keep_zero=0.0)
    empty = [np.zeros((0, 5))] * 8
    for im in host:
        im["labels"] = empty[0]
    rep.update(det, packed(empty, lb))
    got = rep.compute()
    check_report(got, oracle(host, 3, DEFAULT))
    assert got["best_conf"] is None and got["confusion"][:, :3].sum() == 0 and got["confusion"][:3, 3].sum() > 0
    # an empty batch and an accumulator that never saw a batch
    rep = ops.DetectionReport(2)
    det0 = {k: v[:0] for k, v in det.items()}
    rep.update(det0, packed([], []))
    got = rep.compute()
    assert got["images_total"] == 0 and got["confusion"].shape == (3, 3) and got["confusion"].sum() == 0
    assert np.all(got["p_curve"] == -1) and got["p_curve"].shape == (2, 1000)


def test_errors():
    rng = np.random.default_rng(11)
    det, host, (labels, lb) = synthetic_batch(rng, 4, 3, 10, 20, n_keep_zero=0.0)
    bad = [l.copy() for l in labels]
    bad[1] = np.array([[5, 0.5, 0.5, 0.2, 0.2]])
    rep = ops.DetectionReport(3)
    rep.update(det, packed(bad, lb))
    with pytest.raises(IndexError):
        rep.compute()
    rep = ops.DetectionReport(3)
    det["n_keep"][2] = -1
    rep.update(det, packed(labels, lb))
    with pytest.raises(RuntimeError, match="NMS failed"):
        rep.compute()
    for kw in (dict(curve_iou=0.52), dict(conf_grid=[0.0, 0.5, 0.5]), dict(conf_grid=[0.0, np.inf]), dict(conf_grid=[]),
               dict(cm_conf=np.nan), dict(cm_iou=np.inf), dict(iou_thresholds=np.linspace(0.1, 0.9, 17)),
               dict(max_det=-1)):
        with pytest.raises(ValueError):
            ops.DetectionReport(3, **kw)
    # more staging than one CTA's shared memory: an error, not a fault
    det, host, (labels, lb) = synthetic_batch(rng, 2, 3, 4, 4000, n_keep_zero=0.0)
    rep = ops.DetectionReport(3, max_det=4000)
    with pytest.raises(RuntimeError, match="shared memory"):
        rep.update(det, packed(labels, lb, max_gt=4096))


def test_update_does_not_synchronise():
    rng = np.random.default_rng(12)
    det, host, (labels, lb) = synthetic_batch(rng, 8, 3, 20, 60)
    lab = packed(labels, lb)
    rep = ops.DetectionReport(3)
    rep.update(det, lab)   # first call: library load and module initialisation
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            rep.update(det, lab)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    check_report(rep.compute(), oracle(host * 4, 3, DEFAULT))


class _PresetHeads:
    def __init__(self, heads, img_size, anchors):
        self.heads, self.img_size, self.anchors = heads, img_size, anchors

    def eval(self):
        return self

    def __call__(self, img):
        n = img.shape[0]
        return [h[:n] for h in self.heads]


def _train_stand_in(scale, pad_top, pad_left):
    """A module with the names install() rebinds in the reference's `train`, plus the Path and Image its dataset code
    uses.  Its letterbox_resize returns a fixed scale and padding."""
    from PIL import Image
    from yolo_from_scratch_b200.install import PATCHED_FUNCTIONS
    m = types.ModuleType("train")
    m.Image = Image
    m.Path = pathlib.Path
    m.letterbox_resize = lambda pil_img, img_size: (pil_img, scale, pad_top, pad_left)
    for n in PATCHED_FUNCTIONS + ("predict",):
        setattr(m, n, lambda *a, **k: "ref")
    return m


def test_evaluate_report_through_install(tmp_path):
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
        got = train.evaluate_report(model, dataset, torch.device("cuda"), num_classes=nc, batch_size=3)
    finally:
        uninstall(train)
    assert not hasattr(train, "evaluate_report")
    images = []
    for i0 in range(0, 7, 3):
        n = min(3, 7 - i0)
        lbx = [(scale, pt, pl)] * n
        det = ops.detect_batch([h[:n] for h in heads], R.default_anchors(), img, nc, 0.001, 0.4, letterbox=lbx)
        images += host_images(det, labels[i0:i0 + n], [wh + (scale, pt, pl)] * n)
    check_report(got, P.evaluate(images, nc, THR, GRID))
    assert got["n_gt"].sum() == 24 and got["images_total"] == 7 and len(ops.format_detection_report(got)) >= 2
