"""Known answers for the mAP oracle (oracle/map_ref.py), the checker of ops.DetectionMAP and the yb_map_* kernels.

Each case states its derivation.  A TP alone has precision tp / (fp + tp + 2^-52) = 1 / (1 + 2^-52) = 1 - 2^-52,
so "1" below is 1 - 2^-52 and the comparisons allow 1e-12."""
import numpy as np
import pytest

from oracle import map_ref as M
from oracle import ref_path as R

THR = np.linspace(0.5, 0.95, 10)
REC = np.linspace(0.0, 1.0, 101)
W = H = 100.0   # original image size: label (xc, yc, w, h) = pixel box / 100


def label(cls, x1, y1, x2, y2):
    return [cls, (x1 + x2) / 2 / W, (y1 + y2) / 2 / H, (x2 - x1) / W, (y2 - y1) / H]


def image(dets, labels):
    """dets: [(x1, y1, x2, y2, score, cls)] already in keep order (descending score)."""
    d = np.asarray(dets, dtype=np.float64).reshape(-1, 6)
    return {"boxes": d[:, :4].astype(np.float32), "scores": d[:, 4].astype(np.float32), "classes": d[:, 5].astype(np.int64),
            "keep": np.arange(len(d)), "n_keep": len(d), "labels": np.asarray(labels, dtype=np.float64).reshape(-1, 5),
            "letterbox": [W, H, 1.0, 0.0, 0.0]}


def run(images, nc=1, thr=THR):
    return M.evaluate(images, nc, thr, REC, max_det=300)


def test_one_exact_detection_gives_ap_1():
    # IoU 1 >= every threshold: TP everywhere, rc = 1, pr = 1 at every recall point
    out = run([image([(10, 10, 50, 50, 0.9, 0)], [label(0, 10, 10, 50, 50)])])
    assert out["ap"].shape == (1, 10)
    assert np.allclose(out["ap"], 1.0, atol=1e-12) and out["map"] == pytest.approx(1.0, abs=1e-12)
    assert out["map50"] == pytest.approx(1.0, abs=1e-12)
    assert np.array_equal(out["recall"], np.ones((10, 1)))


def test_two_gt_one_tp_gives_51_over_101():
    # rc = 1/2 after the only detection: recall points 0.00 .. 0.50 (51 of 101) read precision 1, the rest 0
    out = run([image([(10, 10, 50, 50, 0.9, 0)], [label(0, 10, 10, 50, 50), label(0, 60, 60, 90, 90)])])
    assert out["map"] == pytest.approx(51 / 101, abs=1e-12)
    assert np.array_equal(out["recall"], np.full((10, 1), 0.5))


def test_fp_above_the_only_tp_gives_ap_one_half():
    # order FP, TP: tp = [0,1], fp = [1,1], rc = [0,1], pr = [0, 1/2]; envelope [1/2, 1/2]; every r reads 1/2
    out = run([image([(60, 60, 90, 90, 0.9, 0), (10, 10, 50, 50, 0.8, 0)], [label(0, 10, 10, 50, 50)])])
    assert out["map"] == pytest.approx(0.5, abs=1e-12)
    assert np.allclose(out["precision"], 0.5, atol=1e-12)


def test_iou_exactly_one_half_is_tp_at_050_and_fp_at_055():
    # GT [0,0,2,1], detection [0,0,1,1]: inter 1, union 2 + 1 - 1 = 2, IoU 0.5 exactly
    gb = np.array([[0.0, 0.0, 2.0, 1.0]])
    assert M.iou_matrix(np.array([[0.0, 0.0, 1.0, 1.0]], np.float32), gb)[0, 0] == 0.5
    mask = M.match_image(np.array([[0, 0, 1, 1]], np.float32), np.array([0]), gb, np.array([0]), THR)
    assert mask.tolist() == [0b1]
    out = run([image([(0, 0, 1, 1, 0.9, 0)], [label(0, 0, 0, 2, 1)])])
    assert out["ap"][0, 0] == pytest.approx(1.0, abs=1e-12) and np.all(out["ap"][0, 1:] == 0)
    assert out["map50"] == pytest.approx(1.0, abs=1e-12) and out["map"] == pytest.approx(0.1, abs=1e-12)


def test_equal_iou_takes_the_later_gt():
    # A = [0,0,2,2], B = [1,0,3,2]; d1 = [1,0,2,2] has IoU 2/4 with both -> takes B (the later one);
    # d2 = A exactly then still finds A (IoU 1).  Had d1 taken A, d2 would be an FP (IoU with B = 2/6).
    gb = np.array([[0.0, 0.0, 2.0, 2.0], [1.0, 0.0, 3.0, 2.0]])
    db = np.array([[1, 0, 2, 2], [0, 0, 2, 2]], np.float32)
    assert M.iou_matrix(db, gb).tolist() == [[0.5, 0.5], [1.0, 2.0 / 6.0]]
    mask = M.match_image(db, np.array([0, 0]), gb, np.array([0, 0]), THR)
    assert mask.tolist() == [0b1, 0x3FF]


def test_equal_scores_across_images_follow_image_order():
    # one GT, in image b.  Image a's detection is an FP, image b's a TP, both scored 0.5.
    # a then b: FP, TP -> pr = [0, 1/2] -> AP 1/2.   b then a: TP, FP -> pr = [1, 1/2], rc = [1, 1] -> AP 1.
    a = image([(60, 60, 90, 90, 0.5, 0)], [])
    b = image([(10, 10, 50, 50, 0.5, 0)], [label(0, 10, 10, 50, 50)])
    assert run([a, b])["map"] == pytest.approx(0.5, abs=1e-12)
    assert run([b, a])["map"] == pytest.approx(1.0, abs=1e-12)


def test_class_without_gt_is_minus_one_and_class_without_detections_is_zero():
    # nc = 3: class 0 exact (AP 1), class 1 has a GT and no detection (AP 0), class 2 has a detection and no GT (-1)
    out = run([image([(10, 10, 50, 50, 0.9, 0), (60, 60, 90, 90, 0.8, 2)],
                     [label(0, 10, 10, 50, 50), label(1, 60, 10, 90, 40)])], nc=3)
    assert np.allclose(out["ap"][0], 1.0, atol=1e-12) and np.all(out["ap"][1] == 0) and np.all(out["ap"][2] == -1)
    assert np.all(out["precision"][:, :, 2] == -1) and np.all(out["recall"][:, 2] == -1) and np.all(out["recall"][:, 1] == 0)
    assert out["map"] == pytest.approx(0.5, abs=1e-12)
    assert out["n_gt"].tolist() == [1, 1, 0] and out["n_det"].tolist() == [1, 0, 1]


def test_nc1_counts_any_label_id_as_class_0():
    out = run([image([(10, 10, 50, 50, 0.9, 0)], [label(3, 10, 10, 50, 50)])], nc=1)
    assert out["n_gt"].tolist() == [1] and out["status"] == 0
    assert out["map"] == pytest.approx(1.0, abs=1e-12)
    # with nc > 1 the same id is out of range: status bit 1
    assert run([image([(10, 10, 50, 50, 0.9, 0)], [label(3, 10, 10, 50, 50)])], nc=3)["status"] & 1


def test_map50_is_none_without_threshold_050():
    out = run([image([(10, 10, 50, 50, 0.9, 0)], [label(0, 10, 10, 50, 50)])], thr=np.array([0.6, 0.7]))
    assert out["map50"] is None and out["ap"].shape == (1, 2)


def test_iou_matrix_equals_the_scalar_corner_iou():
    rng = np.random.default_rng(0)
    x, y = np.sort(rng.uniform(0, 100, (40, 2)), 1), np.sort(rng.uniform(0, 100, (40, 2)), 1)
    db = np.stack([x[:, 0], y[:, 0], x[:, 1], y[:, 1]], 1).astype(np.float32)
    gb = (db[:25] + rng.uniform(-5, 5, (25, 4))).astype(np.float64)
    gb[3] = [10.0, 10.0, 10.0, 20.0]   # zero area: union is the detection's area
    got = M.iou_matrix(db, gb)
    for i in range(len(db)):
        for j in range(len(gb)):
            want = R.corner_iou([float(v) for v in db[i]], gb[j].tolist())
            assert got[i, j] == want


def test_oracle_matches_pycocotools():
    pytest.importorskip("pycocotools")
    from pycocotools.coco import COCO
    from pycocotools.cocoeval import COCOeval
    rng = np.random.default_rng(4)
    nc, images, gts, dts = 3, [], [], []
    for i in range(12):
        labs, dets = [], []
        for _ in range(int(rng.integers(0, 6))):
            x1, y1 = rng.uniform(0, 70, 2)
            w, h = rng.uniform(8, 30, 2)
            c = int(rng.integers(0, nc))
            labs.append(label(c, x1, y1, x1 + w, y1 + h))
            gts.append({"id": len(gts) + 1, "image_id": i, "category_id": c, "bbox": [x1, y1, w, h], "area": w * h, "iscrowd": 0})
            for _ in range(int(rng.integers(0, 3))):
                j = rng.uniform(-4, 4, 4)
                dets.append((x1 + j[0], y1 + j[1], x1 + w + j[2], y1 + h + j[3], rng.uniform(0.01, 1), c))
        dets.sort(key=lambda d: -d[4])
        images.append(image(dets, labs))
        for d in dets:
            b = [float(np.float32(v)) for v in d[:4]]
            dts.append({"image_id": i, "category_id": d[5], "bbox": [b[0], b[1], b[2] - b[0], b[3] - b[1]],
                        "score": float(np.float32(d[4]))})
    coco = COCO()
    coco.dataset = {"images": [{"id": i} for i in range(12)], "annotations": gts,
                    "categories": [{"id": c} for c in range(nc)]}
    coco.createIndex()
    ev = COCOeval(coco, coco.loadRes(dts), "bbox")
    ev.params.maxDets = [300]
    ev.params.areaRng, ev.params.areaRngLbl = [[0, 1e10]], ["all"]
    ev.evaluate()
    ev.accumulate()
    want = ev.eval["precision"][:, :, :, 0, 0]
    got = run(images, nc=nc)["precision"]
    assert np.allclose(got, want, atol=1e-9)
