"""Plain numpy restatement of COCO's bbox evaluation (pycocotools COCOeval.evaluateImg + accumulate + summarize,
area range "all", no crowd annotations) with the project's restrictions: the detections of an image are its kept
detections in keep order, capped at `max_det` overall, and the ground truths come from label lines.  It is the
checker of ops.DetectionMAP and of the yb_map_* kernels; the product never imports it.

Every fp64 expression is written as the kernels evaluate it, so the records and the precision/recall tables can be
compared bit for bit."""
import numpy as np

EPS = np.spacing(1)   # COCOeval.accumulate: pr = tp / (fp + tp + np.spacing(1))


def gt_boxes(labels, letterbox, nc):
    """(n,5) label lines [cls, xc, yc, w, h] normalised to the original image -> (boxes (n,4) fp64 corners in
    original-image pixels, classes (n,) int, bad).  nc == 1: every ground truth is class 0 (train.py:201-202);
    otherwise an id outside [0, nc) is bad (class -1 here)."""
    labels = np.asarray(labels, dtype=np.float64).reshape(-1, 5)
    ow, oh = float(letterbox[0]), float(letterbox[1])
    boxes = np.empty((len(labels), 4), dtype=np.float64)
    classes = np.zeros(len(labels), dtype=np.int64)
    bad = False
    for g, (c, xc, yc, w, h) in enumerate(labels.tolist()):
        boxes[g] = ((xc - w / 2.0) * ow, (yc - h / 2.0) * oh, (xc + w / 2.0) * ow, (yc + h / 2.0) * oh)
        if nc > 1:
            c = int(c)
            if not 0 <= c < nc:
                bad, c = True, -1
            classes[g] = c
    return boxes, classes, bad


def iou_matrix(det_boxes, gt_box):
    """compute_iou_corners (train.py:1064-1084, oracle/ref_path.py: corner_iou) of every detection (fp32 corners
    widened to fp64) with every ground truth, elementwise in numpy: the scalar form's IEEE operations in its order."""
    d = np.asarray(det_boxes, dtype=np.float32).astype(np.float64)[:, None, :]
    g = np.asarray(gt_box, dtype=np.float64)[None, :, :]
    iw = np.maximum(0.0, np.minimum(d[..., 2], g[..., 2]) - np.maximum(d[..., 0], g[..., 0]))
    ih = np.maximum(0.0, np.minimum(d[..., 3], g[..., 3]) - np.maximum(d[..., 1], g[..., 1]))
    inter = iw * ih
    union = (d[..., 2] - d[..., 0]) * (d[..., 3] - d[..., 1]) + (g[..., 2] - g[..., 0]) * (g[..., 3] - g[..., 1]) - inter
    return np.where(union > 0, inter / np.where(union > 0, union, 1.0), 0.0)


def match_image(det_boxes, det_classes, gt_box, gt_cls, iou_thresholds):
    """COCOeval.evaluateImg's greedy matching for one image, all classes at once (a detection only ever meets
    ground truths of its own class): for each threshold, each detection in order takes the unmatched ground truth
    of its class with the highest IoU >= threshold, the later one on equal IoU (`if iou < best: continue`).
    Returns the TP mask (n_det,) uint16, bit t for threshold t."""
    det_classes = np.asarray(det_classes)
    nd, ng = len(det_classes), len(gt_cls)
    mask = np.zeros(nd, dtype=np.uint16)
    if nd == 0 or ng == 0:
        return mask
    iou = iou_matrix(det_boxes, gt_box)
    iou[det_classes[:, None] != np.asarray(gt_cls)[None, :]] = -np.inf
    iou[det_classes < 0] = -np.inf
    row_max = iou.max(axis=1)
    for t, thr in enumerate(iou_thresholds):
        taken = np.zeros(ng, dtype=bool)
        for d in np.flatnonzero(row_max >= thr):   # a detection without any IoU >= thr can never match
            row = np.where(taken, -np.inf, iou[d])
            best = row.max()
            if best >= thr:
                m = ng - 1 - int(np.argmax(row[::-1]))   # the last ground truth with the highest IoU
                taken[m] = True
                mask[d] |= np.uint16(1 << t)
    return mask


def image_records(boxes, scores, classes, keep, n_keep, labels, letterbox, nc, iou_thresholds, max_det, slots):
    """The records of one image as yb_map_match writes them: (score f32, class i32, tp u16) per slot, class -1 in
    unused slots; plus the ground-truth count per class and the status bits (1 bad class, 2 failed NMS)."""
    status = 0
    gb, gc, bad = gt_boxes(labels, letterbox, nc)
    status |= 1 if bad else 0
    n_gt = np.bincount(gc[gc >= 0], minlength=nc).astype(np.int64)
    if n_keep < 0:
        status |= 2
    nd = max(0, min(int(n_keep), slots))
    idx = np.asarray(keep[:nd], dtype=np.int64)
    dcls = np.asarray(classes, dtype=np.int64)[idx]
    if np.any((dcls < 0) | (dcls >= nc)):
        status |= 1
    dcls = np.where((dcls >= 0) & (dcls < nc), dcls, -1)
    sc = np.zeros(slots, dtype=np.float32)
    cl = np.full(slots, -1, dtype=np.int32)
    tp = np.zeros(slots, dtype=np.uint16)
    sc[:nd] = np.asarray(scores, dtype=np.float32)[idx]
    cl[:nd] = dcls
    tp[:nd] = match_image(np.asarray(boxes, dtype=np.float32)[idx], dcls, gb, gc, iou_thresholds)
    return sc, cl, tp, n_gt, status


def accumulate(scores, classes, tp, n_gt, iou_thresholds, recall_thresholds):
    """COCOeval.accumulate for records concatenated in image order (unused slots have class -1).
    Returns precision (T,R,nc) and recall (T,nc), -1 for classes without ground truth."""
    T, R, nc = len(iou_thresholds), len(recall_thresholds), len(n_gt)
    precision = -np.ones((T, R, nc))
    recall = -np.ones((T, nc))
    for c in range(nc):
        npig = int(n_gt[c])
        if npig == 0:
            continue
        sel = np.flatnonzero(classes == c)
        inds = np.argsort(-scores[sel], kind="mergesort")
        dtm = np.stack([(tp[sel][inds] >> t) & 1 for t in range(T)]).astype(bool) if len(sel) else np.zeros((T, 0), bool)
        tp_sum = np.cumsum(dtm, axis=1).astype(dtype=float)
        fp_sum = np.cumsum(np.logical_not(dtm), axis=1).astype(dtype=float)
        for t, (tps, fps) in enumerate(zip(tp_sum, fp_sum)):
            nd = len(tps)
            rc = tps / npig
            pr = tps / (fps + tps + EPS)
            recall[t, c] = rc[-1] if nd else 0
            q = np.zeros(R)
            pr = np.maximum.accumulate(pr[::-1])[::-1] if nd else pr   # `if pr[i] > pr[i-1]: pr[i-1] = pr[i]`
            pis = np.searchsorted(rc, recall_thresholds, side="left")
            for ri, pi in enumerate(pis):
                if pi >= nd:
                    break
                q[ri] = pr[pi]
            precision[t, :, c] = q
    return precision, recall


def summarize(precision, iou_thresholds):
    """COCOeval.summarize's means: map over every entry > -1, map50 at threshold 0.5 (None without it),
    ap (nc,T) the mean over recall points (-1 for a class without ground truth)."""
    def mean(s):
        s = s[s > -1]
        return float(np.mean(s)) if s.size else -1.0
    hit = np.flatnonzero(np.asarray(iou_thresholds) == 0.5)
    ap = np.full((precision.shape[2], precision.shape[0]), -1.0)
    for c in range(precision.shape[2]):
        for t in range(precision.shape[0]):
            if np.all(precision[t, :, c] > -1):
                ap[c, t] = np.mean(precision[t, :, c])
    return {"map": mean(precision), "map50": mean(precision[hit]) if hit.size else None, "ap": ap}


def evaluate(images, nc, iou_thresholds, recall_thresholds, max_det=300):
    """images: per image a dict with boxes (n,4) f32, scores (n,), classes (n,), keep, n_keep, labels (g,5),
    letterbox [orig_w, orig_h, ...], in update order.  Returns the fields of DetectionMAP.compute() plus status."""
    iou_thresholds = np.asarray(iou_thresholds, dtype=np.float64)
    recall_thresholds = np.asarray(recall_thresholds, dtype=np.float64)
    sc, cl, tp = [], [], []
    n_gt = np.zeros(nc, dtype=np.int64)
    status = 0
    for im in images:
        slots = min(max_det, len(im["scores"]))
        s, c, m, g, st = image_records(im["boxes"], im["scores"], im["classes"], im["keep"], im["n_keep"], im["labels"],
                                       im["letterbox"], nc, iou_thresholds, max_det, slots)
        sc.append(s); cl.append(c); tp.append(m)
        n_gt += g
        status |= st
    cat = lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dt)
    scores, classes, tps = cat(sc, np.float32), cat(cl, np.int32), cat(tp, np.uint16)
    precision, recall = accumulate(scores, classes, tps, n_gt, iou_thresholds, recall_thresholds)
    out = summarize(precision, iou_thresholds)
    out.update(precision=precision, recall=recall, n_gt=n_gt,
               n_det=np.array([np.count_nonzero(classes == c) for c in range(nc)], dtype=np.int64), status=status)
    return out
