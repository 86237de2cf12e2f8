"""Plain numpy restatement of the validation report (ops.DetectionReport, yb_report_match): the confusion matrix with
its two-step unique matching, the images per class, the confidence histograms and the P/R/F1 curves, best-F1
threshold and table values computed from them.  Per image with plain loops; it is the checker of the kernel and the
product never imports it.

The ground-truth corners and the fp64 IoUs are map_ref's (gt_boxes, iou_matrix), which are the kernels' operation for
operation, and the records are map_ref.image_records', so the integer outputs can be compared exactly."""
import numpy as np

from . import map_ref as M


def confusion_image(det_boxes, det_scores, det_classes, gt_box, gt_cls, nc, cm_conf, cm_iou):
    """The (nc+1, nc+1) confusion counts of one image (row predicted class, column true class, nc background).
    det_*: the image's first min(n_keep, max_det) kept detections in keep order; gt_cls -1 marks a bad class."""
    cm = np.zeros((nc + 1, nc + 1), dtype=np.int64)
    nd, ng = len(det_classes), len(gt_cls)
    D = [d for d in range(nd) if 0 <= int(det_classes[d]) < nc and float(np.float32(det_scores[d])) > cm_conf]
    G = [g for g in range(ng) if gt_cls[g] >= 0]
    iou = M.iou_matrix(np.asarray(det_boxes, np.float32).reshape(-1, 4), np.asarray(gt_box, np.float64).reshape(-1, 4))
    # step 1: each detection picks the ground truth with the largest IoU > cm_iou, the lower index on equal IoU
    pick = {}
    for d in D:
        best, bg = None, -1
        for g in G:
            v = iou[d, g]
            if v > cm_iou and (bg < 0 or v > best):
                best, bg = v, g
        pick[d] = bg
    # step 2: each picked ground truth keeps the detection with the largest IoU, the earlier one on equal IoU
    kept = {}
    for d in D:
        g = pick[d]
        if g >= 0 and (g not in kept or iou[d, g] > iou[kept[g], g]):
            kept[g] = d
    matched = {d: g for g, d in kept.items()}
    for d in D:
        cm[int(det_classes[d]), gt_cls[matched[d]] if d in matched else nc] += 1
    for g in G:
        if g not in kept:
            cm[nc, gt_cls[g]] += 1
    return cm


def histograms(scores, classes, tp, nc, grid, t_curve):
    """det_hist, tp_hist (nc, K): each record with class >= 0 and a non-NaN score s goes to bin
    j = #{k : grid[k] < s} - 1 when j >= 0; tp_hist only when its TP bit t_curve is set."""
    K = len(grid)
    det_hist = np.zeros((nc, K), dtype=np.int64)
    tp_hist = np.zeros((nc, K), dtype=np.int64)
    for s, c, m in zip(np.asarray(scores, np.float32).tolist(), np.asarray(classes).tolist(), np.asarray(tp).tolist()):
        if c < 0 or s != s:
            continue
        j = int(np.count_nonzero(np.asarray(grid) < s)) - 1
        if j >= 0:
            det_hist[c, j] += 1
            if (m >> t_curve) & 1:
                tp_hist[c, j] += 1
    return det_hist, tp_hist


def curves(det_hist, tp_hist, n_gt, grid):
    """The curves and the values at the best mean F1 from the histograms: n_det, n_tp (nc,K) = detections / TPs with
    score > grid[k] (suffix sums); P = TP/D (1 where D = 0), R = TP/n_gt, F1 = 2PR/(P+R) (0 where P+R = 0), rows of
    classes without ground truth -1; k* the first arg-max of the mean F1 over classes with ground truth."""
    nc, K = det_hist.shape
    n_det = np.zeros((nc, K), dtype=np.int64)
    n_tp = np.zeros((nc, K), dtype=np.int64)
    for c in range(nc):
        run_d = run_t = 0
        for k in range(K - 1, -1, -1):
            run_d += int(det_hist[c, k])
            run_t += int(tp_hist[c, k])
            n_det[c, k], n_tp[c, k] = run_d, run_t
    p = -np.ones((nc, K))
    r = -np.ones((nc, K))
    f1 = -np.ones((nc, K))
    for c in range(nc):
        if n_gt[c] == 0:
            continue
        for k in range(K):
            tp, d = float(n_tp[c, k]), float(n_det[c, k])
            p[c, k] = tp / d if d > 0 else 1.0
            r[c, k] = tp / float(n_gt[c])
            f1[c, k] = 2 * p[c, k] * r[c, k] / (p[c, k] + r[c, k]) if p[c, k] + r[c, k] != 0 else 0.0
    has_gt = np.asarray(n_gt) > 0
    if has_gt.any():
        k = int(np.argmax(f1[has_gt].mean(axis=0)))
        best_conf, at = float(grid[k]), (p[:, k].copy(), r[:, k].copy(), f1[:, k].copy())
    else:
        best_conf, at = None, (-np.ones(nc), -np.ones(nc), -np.ones(nc))
    return {"n_det_above": n_det, "n_tp_above": n_tp, "px": np.asarray(grid, np.float64), "p_curve": p, "r_curve": r,
            "f1_curve": f1, "best_conf": best_conf, "p": at[0], "r": at[1], "f1": at[2]}


def evaluate(images, nc, iou_thresholds, grid, curve_iou=0.5, cm_conf=0.25, cm_iou=0.45, max_det=300,
             recall_thresholds=np.linspace(0.0, 1.0, 101)):
    """images as map_ref.evaluate takes them (the device's own kept detections), in update order.  Returns
    map_ref.evaluate's fields plus confusion, images, images_total, det_hist, tp_hist and the fields of curves()."""
    iou_thresholds = np.asarray(iou_thresholds, dtype=np.float64)
    grid = np.asarray(grid, dtype=np.float64)
    t_curve = int(np.flatnonzero(iou_thresholds == curve_iou)[0])
    out = M.evaluate(images, nc, iou_thresholds, recall_thresholds, max_det=max_det)
    confusion = np.zeros((nc + 1, nc + 1), dtype=np.int64)
    per_class = np.zeros(nc, dtype=np.int64)
    det_hist = np.zeros((nc, len(grid)), dtype=np.int64)
    tp_hist = np.zeros((nc, len(grid)), dtype=np.int64)
    for im in images:
        slots = min(max_det, len(im["scores"]))
        gb, gc, _ = M.gt_boxes(im["labels"], im["letterbox"], nc)
        for c in set(int(c) for c in gc if c >= 0):
            per_class[c] += 1
        nd = max(0, min(int(im["n_keep"]), slots))
        idx = np.asarray(im["keep"][:nd], dtype=np.int64)
        confusion += confusion_image(np.asarray(im["boxes"])[idx], np.asarray(im["scores"])[idx],
                                     np.asarray(im["classes"])[idx], gb, gc, nc, cm_conf, cm_iou)
        sc, cl, tp, _, _ = M.image_records(im["boxes"], im["scores"], im["classes"], im["keep"], im["n_keep"],
                                           im["labels"], im["letterbox"], nc, iou_thresholds, max_det, slots)
        dh, th = histograms(sc, cl, tp, nc, grid, t_curve)
        det_hist += dh
        tp_hist += th
    out.update(curves(det_hist, tp_hist, out["n_gt"], grid), confusion=confusion, images=per_class,
               images_total=len(images), det_hist=det_hist, tp_hist=tp_hist, iou_thresholds=iou_thresholds)
    return out
