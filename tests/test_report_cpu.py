"""Known answers for the validation-report oracle (oracle/report_ref.py), the checker of ops.DetectionReport and
yb_report_match, and the exact text of ops.format_detection_report.

Each case states its derivation.  Coordinates are small integers in a 100 x 100 image, so the IoUs below are exact."""
import numpy as np

from oracle import map_ref as M
from oracle import report_ref as P
from yolo_from_scratch_b200 import ops

THR = np.linspace(0.5, 0.95, 10)
GRID = np.linspace(0.0, 1.0, 1000)
W = H = 100.0


def label(cls, x1, y1, x2, y2):
    return [cls, (x1 + x2) / 2 / W, (y1 + y2) / 2 / H, (x2 - x1) / W, (y2 - y1) / H]


def image(dets, labels):
    """dets: [(x1, y1, x2, y2, score, cls)] already in keep order (descending score)."""
    d = np.asarray(dets, dtype=np.float64).reshape(-1, 6)
    return {"boxes": d[:, :4].astype(np.float32), "scores": d[:, 4].astype(np.float32), "classes": d[:, 5].astype(np.int64),
            "keep": np.arange(len(d)), "n_keep": len(d), "labels": np.asarray(labels, dtype=np.float64).reshape(-1, 5),
            "letterbox": [W, H, 1.0, 0.0, 0.0]}


def cm(dets, labels, nc, cm_conf=0.25, cm_iou=0.45):
    return P.evaluate([image(dets, labels)], nc, THR, GRID, cm_conf=cm_conf, cm_iou=cm_iou)["confusion"]


def test_one_detection_over_two_gt_takes_the_larger_iou():
    # A = [0,0,10,10] class 0, B = [5,0,15,10] class 1; d = A exactly (class 0): IoU 1 with A, 50/150 with B.
    # d keeps A (diagonal); B is unmatched (background row).
    got = cm([(0, 0, 10, 10, 0.9, 0)], [label(0, 0, 0, 10, 10), label(1, 5, 0, 15, 10)], nc=3)
    want = np.zeros((4, 4), np.int64)
    want[0, 0] = want[3, 1] = 1
    assert np.array_equal(got, want)


def test_two_detections_on_one_gt():
    # GT [0,0,10,10]; d1 [0,0,10,8] (IoU 0.8, score 0.9), d2 = GT (IoU 1, score 0.8).  Both pick the GT; it keeps
    # d2 (larger IoU), so d1 is a false positive (background column).
    got = cm([(0, 0, 10, 8, 0.9, 0), (0, 0, 10, 10, 0.8, 0)], [label(0, 0, 0, 10, 10)], nc=1)
    assert got.tolist() == [[1, 1], [0, 0]]


def test_equal_iou_in_step_1_takes_the_lower_gt():
    # A = [0,0,2,2] class 1, B = [1,0,3,2] class 2; d = [1,0,2,2] class 0 has IoU 1/2 with both -> A (lower index).
    gb = np.array([[0.0, 0.0, 2.0, 2.0], [1.0, 0.0, 3.0, 2.0]])
    assert M.iou_matrix(np.array([[1, 0, 2, 2]], np.float32), gb).tolist() == [[0.5, 0.5]]
    got = cm([(1, 0, 2, 2, 0.9, 0)], [label(1, 0, 0, 2, 2), label(2, 1, 0, 3, 2)], nc=3)
    want = np.zeros((4, 4), np.int64)
    want[0, 1] = want[3, 2] = 1
    assert np.array_equal(got, want)


def test_equal_iou_in_step_2_keeps_the_earlier_detection():
    # GT [0,0,10,10] class 0; d1 [0,0,10,8] class 1 and d2 [0,2,10,10] class 2 both have IoU 0.8 -> d1 (earlier).
    got = cm([(0, 0, 10, 8, 0.9, 1), (0, 2, 10, 10, 0.8, 2)], [label(0, 0, 0, 10, 10)], nc=3)
    want = np.zeros((4, 4), np.int64)
    want[1, 0] = want[2, 3] = 1
    assert np.array_equal(got, want)


def test_iou_equal_to_cm_iou_and_score_equal_to_cm_conf_do_not_count():
    # d [0,0,1,1] against GT [0,0,2,1]: IoU exactly 0.5.  With cm_iou 0.5 it is no match: FP and FN.
    assert M.iou_matrix(np.array([[0, 0, 1, 1]], np.float32), np.array([[0.0, 0.0, 2.0, 1.0]]))[0, 0] == 0.5
    assert cm([(0, 0, 1, 1, 0.9, 0)], [label(0, 0, 0, 2, 1)], nc=1, cm_iou=0.5).tolist() == [[0, 1], [1, 0]]
    assert cm([(0, 0, 1, 1, 0.9, 0)], [label(0, 0, 0, 2, 1)], nc=1, cm_iou=0.499).tolist() == [[1, 0], [0, 0]]
    # a score of exactly cm_conf = 0.25 leaves the detection out: only the GT's FN remains
    assert cm([(0, 0, 2, 1, 0.25, 0)], [label(0, 0, 0, 2, 1)], nc=1).tolist() == [[0, 0], [1, 0]]


def test_nan_score_is_left_out_of_matrix_and_histograms():
    out = P.evaluate([image([(0, 0, 10, 10, np.nan, 0)], [label(0, 0, 0, 10, 10)])], 1, THR, GRID)
    assert out["confusion"].tolist() == [[0, 0], [1, 0]]
    assert out["det_hist"].sum() == 0 and out["tp_hist"].sum() == 0


def test_cross_class_match_lands_off_the_diagonal():
    # a class-2 detection exactly on a class-0 GT: row 2, column 0
    got = cm([(10, 10, 50, 50, 0.9, 2)], [label(0, 10, 10, 50, 50)], nc=3)
    want = np.zeros((4, 4), np.int64)
    want[2, 0] = 1
    assert np.array_equal(got, want)


def test_nc1_is_a_2x2_matrix_and_any_label_id_is_class_0():
    # a TP, a duplicate FP on it, an FP elsewhere and a missed GT (label id 3 is class 0 with nc = 1)
    got = cm([(10, 10, 50, 50, 0.9, 0), (10, 10, 50, 46, 0.8, 0), (70, 70, 90, 90, 0.7, 0)],
             [label(3, 10, 10, 50, 50), label(0, 0, 60, 20, 90)], nc=1)
    assert got.shape == (2, 2) and got.tolist() == [[1, 2], [1, 0]]


def test_grid_point_d0_and_class_without_gt():
    # grid [0, .25, .5, .75]: a score of exactly 0.5 lands in bin 1 = (0.25, 0.5], so it counts at 0 and 0.25 but
    # not at 0.5.  It is a TP of class 0: P = R = F1 = 1 at k = 0, 1; at k = 2, 3 no detection is left: P = 1 (D = 0),
    # R = 0, F1 = 0.  Class 1 has a detection and no GT: its rows are -1.
    grid = [0.0, 0.25, 0.5, 0.75]
    out = P.evaluate([image([(10, 10, 50, 50, 0.5, 0), (60, 60, 90, 90, 0.4, 1)], [label(0, 10, 10, 50, 50)])], 2, THR,
                     grid)
    assert out["det_hist"].tolist() == [[0, 1, 0, 0], [0, 1, 0, 0]] and out["tp_hist"].tolist() == [[0, 1, 0, 0], [0] * 4]
    assert out["n_det_above"][0].tolist() == [1, 1, 0, 0]
    assert out["p_curve"][0].tolist() == [1.0, 1.0, 1.0, 1.0]
    assert out["r_curve"][0].tolist() == [1.0, 1.0, 0.0, 0.0]
    assert out["f1_curve"][0].tolist() == [1.0, 1.0, 0.0, 0.0]
    assert np.all(out["p_curve"][1] == -1) and np.all(out["r_curve"][1] == -1) and np.all(out["f1_curve"][1] == -1)
    assert out["images"].tolist() == [1, 0] and out["images_total"] == 1
    # best F1: mean over class 0 only, 1 at k = 0 and 1 -> the first
    assert out["best_conf"] == 0.0 and out["p"].tolist() == [1.0, -1.0] and out["f1"].tolist() == [1.0, -1.0]


def test_best_f1_tie_picks_the_first_threshold():
    # class 0: GT g1 and g2; a TP at 0.9 and an FP at 0.6.  k with grid <  0.6: P 1/2, R 1/2, F1 1/2;
    # 0.6 <= grid < 0.9: P 1, R 1/2, F1 2/3; grid >= 0.9: F1 0.  The maximum 2/3 first occurs at the first grid point
    # >= 0.6, which is 0.6 itself when it is on the grid (a score of exactly 0.6 does not count there).
    grid = [0.0, 0.3, float(np.float32(0.6)), 0.7, 0.8, 0.95]
    out = P.evaluate([image([(10, 10, 50, 50, 0.9, 0), (60, 60, 90, 90, 0.6, 0)],
                            [label(0, 10, 10, 50, 50), label(0, 0, 60, 20, 90)])], 1, THR, grid)
    assert out["f1_curve"][0].tolist() == [0.5, 0.5, 2 / 3, 2 / 3, 2 / 3, 0.0]
    assert out["best_conf"] == grid[2]
    assert out["p"].tolist() == [1.0] and out["r"].tolist() == [0.5]
    # no class with ground truth: no best threshold
    none = P.evaluate([image([(60, 60, 90, 90, 0.6, 0)], [])], 1, THR, grid)
    assert none["best_conf"] is None and none["p"].tolist() == [-1.0]


def test_report_curves_equal_the_oracle():
    # ops.report_curves (the host half of DetectionReport.compute) on the oracle's suffix sums
    rng = np.random.default_rng(0)
    det = rng.integers(0, 5, (4, 50))
    tp = np.minimum(det, rng.integers(0, 3, (4, 50)))
    n_gt = np.array([7, 0, 3, 1])
    want = P.curves(det, tp, n_gt, GRID[:50])
    got = ops.report_curves(want["n_det_above"], want["n_tp_above"], n_gt, GRID[:50])
    for k in ("px", "p_curve", "r_curve", "f1_curve", "p", "r", "f1"):
        assert np.array_equal(got[k], want[k]), k
    assert got["best_conf"] == want["best_conf"]


def test_format_detection_report_text():
    # image 1: a class-0 GT found exactly (score 0.9) and a class-1 GT missed; image 2: a class-1 FP (0.6), no GT.
    # Class 0: P = R = 1 for grid < 0.9; class 1: R = 0 everywhere.  Mean F1 1/2 from k = 0: best_conf 0, p = [1, 0].
    # AP: class 0 is 1 - 2^-52 at every threshold, class 1 is 0: map = map50 = (1 - 2^-52) / 2.
    out = P.evaluate([image([(10, 10, 50, 50, 0.9, 0)], [label(0, 10, 10, 50, 50), label(1, 60, 60, 90, 90)]),
                      image([(0, 0, 20, 20, 0.6, 1)], [])], 2, THR, GRID)
    assert out["best_conf"] == 0.0 and out["p"].tolist() == [1.0, 0.0]
    assert ops.format_detection_report(out, names=["person", "car"]) == [
        "                 Class     Images  Instances          P          R      mAP50   mAP50-95",
        "                   all          2          2        0.5        0.5        0.5        0.5",
        "                person          1          1          1          1          1          1",
        "                   car          1          1          0          0          0          0",
    ]
    # default names are the class indices; without a 0.5 threshold mAP50 is -1
    out = P.evaluate([image([(10, 10, 50, 50, 0.9, 0)], [label(0, 10, 10, 50, 50)])], 1, [0.6, 0.75], GRID,
                     curve_iou=0.75)
    assert ops.format_detection_report(out)[1:] == [
        "                   all          1          1          1          1         -1          1",
        "                     0          1          1          1          1         -1          1",
    ]
