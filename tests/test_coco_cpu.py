"""Known answers for the COCO oracle (oracle/coco_ref.py), the checker of ops.COCODetectionEval and the yb_coco_*
kernels, and the literal transcription of pycocotools against the kernels' vectorised form.

The image is 128 x 128 pixels and every coordinate an integer, so label values are dyadic and the corners and areas
below are exact."""
import numpy as np
import pytest

from oracle import coco_ref as C
from yolo_from_scratch_b200 import ops

THR = np.linspace(0.5, 0.95, 10)
REC = np.linspace(0.0, 1.0, 101)
W = H = 128.0
ALL, SMALL, MEDIUM, LARGE = range(4)


def label(cls, x1, y1, x2, y2):
    return [cls, (x1 + x2) / 2 / W, (y1 + y2) / 2 / H, (x2 - x1) / W, (y2 - y1) / H]


def image(dets, labels):
    """dets: [(x1, y1, x2, y2, score, cls)] already in keep order (descending score)."""
    d = np.asarray(dets, dtype=np.float64).reshape(-1, 6)
    return {"boxes": d[:, :4].astype(np.float32), "scores": d[:, 4].astype(np.float32), "classes": d[:, 5].astype(np.int64),
            "keep": np.arange(len(d)), "n_keep": len(d), "labels": np.asarray(labels, dtype=np.float64).reshape(-1, 5),
            "letterbox": [W, H, 1.0, 0.0, 0.0]}


def records(im, nc=1, thr=THR):
    rec, gt_count, status = C.image_records(im, nc, thr, 300)
    assert status == 0
    return rec, gt_count


def both(images, nc=1, max_dets=C.MAX_DETS, max_det=300):
    """Both oracle forms; their tables must agree bit for bit."""
    got = C.evaluate(images, nc, THR, REC, max_det=max_det, max_dets=max_dets)
    lit = C.evaluate_literal(images, nc, THR, REC, max_det=max_det, max_dets=max_dets)
    assert np.array_equal(got["precision"], lit["precision"]) and np.array_equal(got["recall"], lit["recall"])
    assert np.array_equal(got["stats"], lit["stats"])
    return got


def test_area_exactly_on_a_bound_is_inside_both_ranges():
    # 32 x 32 = 1024 = 32^2: small and medium; 96 x 96 = 9216 = 96^2: medium and large
    im = image([(0, 0, 32, 32, 0.9, 0), (10, 10, 106, 106, 0.8, 0)], [label(0, 0, 0, 32, 32), label(0, 10, 10, 106, 106)])
    rec, gt_count = records(im)
    assert gt_count[:, 0].tolist() == [2, 1, 2, 1]
    # each detection matches its own ground truth exactly: a TP at every threshold in every range it lies in
    assert rec["tp"][0].tolist() == [0x3FF, 0x3FF, 0x3FF, 0] and rec["ig"][0].tolist() == [0, 0, 0, 0x3FF]
    assert rec["tp"][1].tolist() == [0x3FF, 0, 0x3FF, 0x3FF] and rec["ig"][1].tolist() == [0, 0x3FF, 0, 0]
    out = both([im])
    assert np.allclose(out["precision"][:, :, 0, :, 2], 1.0, atol=1e-12)
    assert out["n_gt"].tolist() == [[2, 1, 2, 1]]


def test_detection_matched_to_an_out_of_range_gt_is_ignored_not_fp():
    # GT 40 x 40 = 1600 (medium: ignored in small); detection 32 x 32 inside small, IoU 1024/1600 = 0.64.
    # small: thresholds 0.50, 0.55, 0.60 match the ignored GT -> ignored; 0.65.. unmatched inside small -> FP
    im = image([(0, 0, 32, 32, 0.9, 0)], [label(0, 0, 0, 40, 40)])
    rec, gt_count = records(im)
    assert rec["tp"][0, SMALL] == 0 and rec["ig"][0, SMALL] == 0b111
    assert rec["tp"][0, ALL] == 0b111 and rec["ig"][0, ALL] == 0
    assert gt_count[SMALL, 0] == 0
    out = both([im])
    assert np.all(out["precision"][:, :, 0, SMALL] == -1)   # no GT inside small


def test_non_ignored_gt_wins_over_an_ignored_one_with_higher_iou():
    # detection D = [0,0,30,30] (900, small).  A = [0,0,30,20] (600, small), IoU 600/900 = 0.667;
    # B = [0,0,32,33] (1056, medium), IoU 900/1056 = 0.852.
    # small: 0.50..0.65 take A (TP) although B is closer; 0.70..0.85 only B -> ignored; 0.90, 0.95 -> FP.
    # all: B is not ignored and closer: TP at 0.50..0.85, FP at 0.90, 0.95.
    im = image([(0, 0, 30, 30, 0.9, 0)], [label(0, 0, 0, 30, 20), label(0, 0, 0, 32, 33)])
    rec, _ = records(im)
    assert rec["tp"][0, SMALL] == 0b1111 and rec["ig"][0, SMALL] == 0b11110000
    assert rec["tp"][0, ALL] == 0xFF and rec["ig"][0, ALL] == 0
    both([im])


def test_unmatched_out_of_range_detection_is_ignored_matched_one_stays_tp():
    # medium: GT [0,0,33,34] (1122).  D1 = [0,0,32,31] (992, outside medium), IoU 992/1122 = 0.884: TP at 0.50..0.85,
    # ignored at 0.90 and 0.95 (unmatched, outside).  D2 = [100,100,110,110] (100, outside medium): ignored everywhere.
    im = image([(0, 0, 32, 31, 0.9, 0), (100, 100, 110, 110, 0.8, 0)], [label(0, 0, 0, 33, 34)])
    rec, _ = records(im)
    assert rec["tp"][0, MEDIUM] == 0xFF and rec["ig"][0, MEDIUM] == 0x300
    assert rec["tp"][1, MEDIUM] == 0 and rec["ig"][1, MEDIUM] == 0x3FF
    assert rec["tp"][1, ALL] == 0 and rec["ig"][1, ALL] == 0   # inside "all": an FP there
    out = both([im])
    # medium: the only counted detection is a TP at 0.50..0.85 -> precision 1 up to recall 1
    assert np.allclose(out["precision"][:8, :, 0, MEDIUM, 2], 1.0, atol=1e-12)
    assert np.all(out["precision"][8:, :, 0, MEDIUM, 2] == 0)


def test_equal_iou_goes_to_the_later_gt_in_each_group():
    # A = [0,0,40,40], B = [20,0,60,40] (1600 each).  d1 = [20,0,40,40] has IoU 800/1600 = 1/2 with both and takes B.
    # d2 = [0,0,32,32] has IoU 0.64 with A and 384/2240 with B, so it finds A only if d1 took B.
    # all: both TPs at 0.50..0.60.  small: A and B are ignored (1600): d1 and d2 match ignored GTs -> ignored there.
    im = image([(20, 0, 40, 40, 0.9, 0), (0, 0, 32, 32, 0.8, 0)], [label(0, 0, 0, 40, 40), label(0, 20, 0, 60, 40)])
    rec, _ = records(im)
    assert rec["tp"][:, ALL].tolist() == [0b1, 0b111]
    assert rec["ig"][:, SMALL].tolist() == [0b1, 0b111] and rec["tp"][:, SMALL].tolist() == [0, 0]
    both([im])


def test_rank_per_image_and_class():
    dets = [(i, i, i + 10, i + 10, 0.9 - i / 100, c) for i, c in enumerate([0, 1, 0, 2, 1, 0, 0])]
    a = image(dets, [])
    b = image(dets[:3], [])
    ra, _ = records(a, nc=3)
    rb, _ = records(b, nc=3)
    assert ra["rank"].tolist() == [0, 0, 1, 0, 1, 2, 3]
    assert rb["rank"].tolist() == [0, 0, 1]   # counted per image
    assert C.ranks([2, -1, 2, 2]).tolist() == [0, 0, 1, 2]


def test_max_dets_rank_filter():
    # three exact detections of class 0 in one image: maxDets 1 sees one TP of three GTs
    gts = [label(0, 0, 0, 20, 20), label(0, 40, 40, 60, 60), label(0, 80, 80, 100, 100)]
    im = image([(0, 0, 20, 20, 0.9, 0), (40, 40, 60, 60, 0.8, 0), (80, 80, 100, 100, 0.7, 0)], gts)
    out = both([im], max_dets=(1, 2, 10))
    assert np.all(out["recall"][:, 0, ALL, 0] == 1 / 3) and np.all(out["recall"][:, 0, ALL, 1] == 2 / 3)
    assert np.all(out["recall"][:, 0, ALL, 2] == 1.0)
    assert out["stats"][6] == pytest.approx(1 / 3) and out["stats"][7] == pytest.approx(2 / 3)


def test_stats0_is_minus_one_without_max_dets_100():
    im = image([(0, 0, 32, 32, 0.9, 0)], [label(0, 0, 0, 32, 32)])
    out = both([im], max_dets=(1, 5, 20))
    assert out["stats"][0] == -1
    assert out["stats"][1] == pytest.approx(1.0, abs=1e-12) and out["stats"][8] == 1.0
    out = both([im])
    assert out["stats"][0] == pytest.approx(1.0, abs=1e-12)
    # large has no GT: -1; small and medium both hold the 32^2 box
    assert out["stats"][5] == -1 and out["stats"][11] == -1 and out["stats"][3] > 0.99 and out["stats"][4] > 0.99


def test_format_coco_stats():
    stats = np.array([0.5, 0.75, 0.25, -1.0, 0.1234, 0.9996, 0.01, 0.2, 0.3, 0.4, 0.5, 0.6])
    assert ops.format_coco_stats(stats) == [
        " Average Precision  (AP) @[ IoU=0.50:0.95 | area=   all | maxDets=100 ] = 0.500",
        " Average Precision  (AP) @[ IoU=0.50      | area=   all | maxDets=100 ] = 0.750",
        " Average Precision  (AP) @[ IoU=0.75      | area=   all | maxDets=100 ] = 0.250",
        " Average Precision  (AP) @[ IoU=0.50:0.95 | area= small | maxDets=100 ] = -1.000",
        " Average Precision  (AP) @[ IoU=0.50:0.95 | area=medium | maxDets=100 ] = 0.123",
        " Average Precision  (AP) @[ IoU=0.50:0.95 | area= large | maxDets=100 ] = 1.000",
        " Average Recall     (AR) @[ IoU=0.50:0.95 | area=   all | maxDets=  1 ] = 0.010",
        " Average Recall     (AR) @[ IoU=0.50:0.95 | area=   all | maxDets= 10 ] = 0.200",
        " Average Recall     (AR) @[ IoU=0.50:0.95 | area=   all | maxDets=100 ] = 0.300",
        " Average Recall     (AR) @[ IoU=0.50:0.95 | area= small | maxDets=100 ] = 0.400",
        " Average Recall     (AR) @[ IoU=0.50:0.95 | area=medium | maxDets=100 ] = 0.500",
        " Average Recall     (AR) @[ IoU=0.50:0.95 | area= large | maxDets=100 ] = 0.600",
    ]
    lines = ops.format_coco_stats(stats, [0.3, 0.6], (1, 5, 20))
    assert lines[0] == " Average Precision  (AP) @[ IoU=0.30:0.60 | area=   all | maxDets=100 ] = 0.500"
    assert lines[2].endswith("maxDets= 20 ] = 0.250") and lines[7].endswith("maxDets=  5 ] = 0.200")


def test_summarize_coco_equals_the_oracle():
    rng = np.random.default_rng(5)
    precision = np.where(rng.uniform(size=(10, 101, 3, 4, 3)) < 0.1, -1.0, rng.uniform(size=(10, 101, 3, 4, 3)))
    recall = np.where(rng.uniform(size=(10, 3, 4, 3)) < 0.1, -1.0, rng.uniform(size=(10, 3, 4, 3)))
    for md in ((1, 10, 100), (1, 5, 20)):
        assert np.array_equal(ops.summarize_coco(precision, recall, THR, md), C.summarize(precision, recall, THR, md))


def random_images(rng, nc, n_img):
    """Small random images around the area bounds: boxes from 5 to 150 pixels on a 200-pixel image, jittered and
    duplicated detections, quantised scores, some images without detections or without ground truth."""
    images = []
    for _ in range(n_img):
        ow = oh = 200.0
        n = int(rng.integers(0, 6))
        wh = np.exp(rng.uniform(np.log(5), np.log(150), (n, 2)))
        xy = rng.uniform(0, 200 - wh)
        gt = np.column_stack([xy, xy + wh])
        lab = np.column_stack([rng.integers(0, nc, n), (gt[:, 0] + gt[:, 2]) / 2 / ow, (gt[:, 1] + gt[:, 3]) / 2 / oh,
                               wh[:, 0] / ow, wh[:, 1] / oh]) if n else np.zeros((0, 5))
        m = int(rng.integers(0, 9)) if rng.uniform() > 0.2 else 0
        src = rng.integers(0, max(n, 1), m)
        if n:
            bx = gt[src] + rng.normal(0, 1, (m, 4)) * rng.choice([0.0, 2.0, 6.0], (m, 1)) * np.sqrt(wh[src].mean(1))[:, None] / 4
            cls = np.where(rng.uniform(size=m) < 0.8, lab[src, 0], rng.integers(0, nc, m))
        else:
            bx = np.sort(rng.uniform(0, 200, (m, 4)).reshape(m, 2, 2), axis=1).transpose(0, 2, 1).reshape(m, 4)
            cls = rng.integers(0, nc, m)
        bx = np.concatenate([np.minimum(bx[:, :2], bx[:, 2:]), np.maximum(bx[:, :2], bx[:, 2:])], 1)
        scores = np.round(rng.uniform(0.01, 1, m) * 10) / 10
        order = np.argsort(-scores, kind="stable")
        images.append({"boxes": bx.astype(np.float32).reshape(-1, 4), "scores": scores.astype(np.float32),
                       "classes": cls.astype(np.int64), "keep": order, "n_keep": m, "labels": lab,
                       "letterbox": (ow, oh, 1.0, 0.0, 0.0)})
    return images


@pytest.mark.parametrize("block", range(8))
def test_literal_equals_vectorised_on_random_cases(block):
    """(a) pycocotools' loops and (b) the kernels' form agree bit for bit on the tables and the stats."""
    bites = {"ignored": 0, "ranked": 0}
    for seed in range(block * 40, block * 40 + 40):
        rng = np.random.default_rng(seed)
        nc = int(rng.integers(1, 4))
        max_dets = (1, 10, 100) if seed % 3 else (1, 2, 3)
        max_det = 300 if seed % 4 else 4
        images = random_images(rng, nc, int(rng.integers(1, 6)))
        got = C.evaluate(images, nc, THR, REC, max_det=max_det, max_dets=max_dets)
        lit = C.evaluate_literal(images, nc, THR, REC, max_det=max_det, max_dets=max_dets)
        assert np.array_equal(got["precision"], lit["precision"]), seed
        assert np.array_equal(got["recall"], lit["recall"]), seed
        assert np.array_equal(got["stats"], lit["stats"]), seed
        bites["ignored"] += int(np.count_nonzero(got["records"]["ig"]))
        bites["ranked"] += int(np.count_nonzero(got["records"]["rank"] >= max_dets[0]))
    assert bites["ignored"] > 0 and bites["ranked"] > 0
