"""COCO's bbox summary (pycocotools 2.0 COCOeval.evaluateImg + accumulate + summarize with area ranges and
per-(image, category) maxDets, no crowd) with the project's restrictions, in two forms.  It is the checker of
ops.COCODetectionEval and of the yb_coco_* kernels; the product never imports it.

  (a) evaluate_literal: a transcription of pycocotools' code with its per-(image, category, area) loops, kept as
      close to the original as the restrictions below allow.  Slow; it validates (b) on small cases.
  (b) evaluate: the kernels' form.  Per image it writes the records yb_coco_match writes (score, class, rank within
      (image, class), TP and ignored bits per threshold and area range), picking each match by the lexicographic
      key (not ignored, IoU, index) and applying maxDets as a rank filter; accumulate drops the ignored records.

Restrictions (include/yolo_b200.h states them): the detections of an image are its first min(n_keep, max_det) kept
detections in keep order, ground truths come from label lines in original-image pixels (map_ref.gt_boxes), the IoU
is the project's corner IoU (map_ref.iou_matrix), an area is (x2-x1)*(y2-y1) of fp64 corners (a detection's fp32
corners widened), and a NaN IoU never matches: the one deliberate departure from pycocotools, whose
`if ious[d, g] < iou: continue` lets a NaN through.  Every fp64 expression is the kernels', so (b) and the kernels
agree bit for bit, and (a) and (b) agree bit for bit on the tables."""
import numpy as np

from oracle import map_ref as MR

AREA_RNG = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]   # Params.areaRng
AREA_LBL = ["all", "small", "medium", "large"]
MAX_DETS = [1, 10, 100]
EPS = np.spacing(1)


def _image_inputs(im, nc, max_det):
    """(gt boxes (g,4) f64, gt classes (g,), det boxes (d,4) f32, det scores (d,) f32, det classes (d,), status)."""
    gb, gc, bad = MR.gt_boxes(im["labels"], im["letterbox"], nc)
    status = 1 if bad else 0
    if im["n_keep"] < 0:
        status |= 2
    slots = min(max_det, len(im["scores"]))
    nd = max(0, min(int(im["n_keep"]), slots))
    idx = np.asarray(im["keep"][:nd], dtype=np.int64)
    dcls = np.asarray(im["classes"], dtype=np.int64)[idx]
    if np.any((dcls < 0) | (dcls >= nc)):
        status |= 1
    dcls = np.where((dcls >= 0) & (dcls < nc), dcls, -1)
    return (gb, gc, np.asarray(im["boxes"], dtype=np.float32)[idx].reshape(-1, 4),
            np.asarray(im["scores"], dtype=np.float32)[idx], dcls, status)


def box_area(b):
    b = np.asarray(b, dtype=np.float64)
    return (b[..., 2] - b[..., 0]) * (b[..., 3] - b[..., 1])


# ------------------------------------------------------------------------------------------------------------
# (a) literal
# ------------------------------------------------------------------------------------------------------------
def evaluate_img(gt, dt, aRng, maxDet, iouThrs):
    """COCOeval.evaluateImg for one image, category and area range.  gt / dt: lists of dicts (id, box, area,
    score); dt is in keep order (pycocotools sorts by score here; the kept detections already are)."""
    if len(gt) == 0 and len(dt) == 0:
        return None
    for g in gt:
        if g["ignore"] or (g["area"] < aRng[0] or g["area"] > aRng[1]):
            g["_ignore"] = 1
        else:
            g["_ignore"] = 0
    # sort dt highest score first, sort gt ignore last
    gtind = np.argsort([g["_ignore"] for g in gt], kind="mergesort")
    gt = [gt[i] for i in gtind]
    dt = dt[0:maxDet]
    ious = MR.iou_matrix(np.array([d["box"] for d in dt], np.float32).reshape(-1, 4),
                         np.array([g["box"] for g in gt], np.float64).reshape(-1, 4))

    T = len(iouThrs)
    G = len(gt)
    D = len(dt)
    gtm = np.zeros((T, G))
    dtm = np.zeros((T, D))
    gtIg = np.array([g["_ignore"] for g in gt])
    dtIg = np.zeros((T, D))
    if not ious.size == 0:
        for tind, t in enumerate(iouThrs):
            for dind, d in enumerate(dt):
                # information about best match so far (m=-1 -> unmatched)
                iou = min([t, 1 - 1e-10])
                m = -1
                for gind, g in enumerate(gt):
                    # if this gt already matched, and not a crowd, continue
                    if gtm[tind, gind] > 0:
                        continue
                    # if dt matched to reg gt, and on ignore gt, stop
                    if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                        break
                    # continue to next gt unless better match made (a NaN IoU never matches: `not >=`)
                    if not ious[dind, gind] >= iou:
                        continue
                    # if match successful and best so far, store appropriately
                    iou = ious[dind, gind]
                    m = gind
                # if match made store id of match for both dt and gt
                if m == -1:
                    continue
                dtIg[tind, dind] = gtIg[m]
                dtm[tind, dind] = gt[m]["id"]
                gtm[tind, m] = d["id"]
    # set unmatched detections outside of area range to ignore
    a = np.array([d["area"] < aRng[0] or d["area"] > aRng[1] for d in dt]).reshape((1, len(dt)))
    dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
    return {"dtMatches": dtm, "gtMatches": gtm, "dtScores": [d["score"] for d in dt], "gtIgnore": gtIg,
            "dtIgnore": dtIg}


def accumulate_literal(evalImgs, K, A, I, iouThrs, recThrs, maxDets):
    """COCOeval.accumulate; evalImgs[k][a][i].  Returns precision (T,R,K,A,M) and recall (T,K,A,M)."""
    T = len(iouThrs)
    R = len(recThrs)
    M = len(maxDets)
    precision = -np.ones((T, R, K, A, M))
    recall = -np.ones((T, K, A, M))
    for k in range(K):
        for a in range(A):
            for m, maxDet in enumerate(maxDets):
                E = [evalImgs[k][a][i] for i in range(I)]
                E = [e for e in E if e is not None]
                if len(E) == 0:
                    continue
                dtScores = np.concatenate([np.asarray(e["dtScores"][0:maxDet], dtype=np.float64) for e in E])
                # different sorting method generates slightly different results.
                # mergesort is used to be consistent as Matlab implementation.
                inds = np.argsort(-dtScores, kind="mergesort")
                dtm = np.concatenate([e["dtMatches"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                dtIg = np.concatenate([e["dtIgnore"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                gtIg = np.concatenate([e["gtIgnore"] for e in E])
                npig = np.count_nonzero(gtIg == 0)
                if npig == 0:
                    continue
                tps = np.logical_and(dtm, np.logical_not(dtIg))
                fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
                tp_sum = np.cumsum(tps, axis=1).astype(dtype=float)
                fp_sum = np.cumsum(fps, axis=1).astype(dtype=float)
                for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
                    tp = np.array(tp)
                    fp = np.array(fp)
                    nd = len(tp)
                    rc = tp / npig
                    pr = tp / (fp + tp + np.spacing(1))
                    q = np.zeros((R,))
                    if nd:
                        recall[t, k, a, m] = rc[-1]
                    else:
                        recall[t, k, a, m] = 0
                    # numpy is slow without cython optimization for accessing elements
                    # use python array gets significant speed improvement
                    pr = pr.tolist()
                    q = q.tolist()
                    for i in range(nd - 1, 0, -1):
                        if pr[i] > pr[i - 1]:
                            pr[i - 1] = pr[i]
                    inds = np.searchsorted(rc, recThrs, side="left")
                    try:
                        for ri, pi in enumerate(inds):
                            q[ri] = pr[pi]
                    except IndexError:
                        pass
                    precision[t, :, k, a, m] = np.array(q)
    return precision, recall


def summarize(precision, recall, iouThrs, maxDets, areaRngLbl=AREA_LBL):
    """COCOeval.summarize / _summarizeDets: the 12 stats."""
    def _summarize(ap=1, iouThr=None, areaRng="all", maxDets_=100):
        aind = [i for i, aRng in enumerate(areaRngLbl) if aRng == areaRng]
        mind = [i for i, mDet in enumerate(maxDets) if mDet == maxDets_]
        if ap == 1:
            # dimension of precision: [TxRxKxAxM]
            s = precision
            # IoU
            if iouThr is not None:
                t = np.where(iouThr == np.asarray(iouThrs))[0]
                s = s[t]
            s = s[:, :, :, aind, mind]
        else:
            # dimension of recall: [TxKxAxM]
            s = recall
            if iouThr is not None:
                t = np.where(iouThr == np.asarray(iouThrs))[0]
                s = s[t]
            s = s[:, :, aind, mind]
        if len(s[s > -1]) == 0:
            mean_s = -1
        else:
            mean_s = np.mean(s[s > -1])
        return float(mean_s)

    stats = np.zeros((12,))
    stats[0] = _summarize(1)
    stats[1] = _summarize(1, iouThr=.5, maxDets_=maxDets[2])
    stats[2] = _summarize(1, iouThr=.75, maxDets_=maxDets[2])
    stats[3] = _summarize(1, areaRng="small", maxDets_=maxDets[2])
    stats[4] = _summarize(1, areaRng="medium", maxDets_=maxDets[2])
    stats[5] = _summarize(1, areaRng="large", maxDets_=maxDets[2])
    stats[6] = _summarize(0, maxDets_=maxDets[0])
    stats[7] = _summarize(0, maxDets_=maxDets[1])
    stats[8] = _summarize(0, maxDets_=maxDets[2])
    stats[9] = _summarize(0, areaRng="small", maxDets_=maxDets[2])
    stats[10] = _summarize(0, areaRng="medium", maxDets_=maxDets[2])
    stats[11] = _summarize(0, areaRng="large", maxDets_=maxDets[2])
    return stats


def evaluate_literal(images, nc, iou_thresholds, recall_thresholds, max_det=300, max_dets=MAX_DETS,
                     area_rng=AREA_RNG):
    """(a): COCOeval.evaluate + accumulate + summarize over `images` (map_ref.evaluate's input).
    Returns {precision, recall, stats}."""
    iou_thresholds = np.asarray(iou_thresholds, dtype=np.float64)
    recall_thresholds = np.asarray(recall_thresholds, dtype=np.float64)
    gts, dts = [], []   # per image: per category lists
    ann_id = 0
    for im in images:
        gb, gc, db, ds, dc, _ = _image_inputs(im, nc, max_det)
        g_by, d_by = [[] for _ in range(nc)], [[] for _ in range(nc)]
        for g in range(len(gc)):
            if gc[g] >= 0:
                ann_id += 1
                g_by[gc[g]].append({"id": ann_id, "box": gb[g], "area": float(box_area(gb[g])), "ignore": 0})
        for d in range(len(dc)):
            if dc[d] >= 0:
                ann_id += 1
                d_by[dc[d]].append({"id": ann_id, "box": db[d], "area": float(box_area(db[d].astype(np.float64))),
                                    "score": float(ds[d])})
        gts.append(g_by)
        dts.append(d_by)
    I = len(images)
    evalImgs = [[[evaluate_img([dict(g) for g in gts[i][k]], dts[i][k], aRng, max_dets[-1], iou_thresholds)
                  for i in range(I)] for aRng in area_rng] for k in range(nc)]
    precision, recall = accumulate_literal(evalImgs, nc, len(area_rng), I, iou_thresholds, recall_thresholds, max_dets)
    return {"precision": precision, "recall": recall,
            "stats": summarize(precision, recall, iou_thresholds, max_dets)}


# ------------------------------------------------------------------------------------------------------------
# (b) the kernels' form
# ------------------------------------------------------------------------------------------------------------
def match_image(det_boxes, det_classes, det_out, gt_box, gt_cls, gt_nig, iou_thresholds):
    """Greedy matching of one image and area range, all classes at once: for each threshold, each detection in
    order takes the untaken ground truth of its class that is best by (not ignored, IoU, index) among those with
    IoU >= min(t, 1-1e-10).  det_out: the detection is outside the range; gt_nig: the ground truth is inside it.
    Returns (tp, ig) (n_det,) uint16, bit t for threshold t."""
    det_classes = np.asarray(det_classes)
    nd, ng = len(det_classes), len(gt_cls)
    tp = np.zeros(nd, dtype=np.uint16)
    ig = np.zeros(nd, dtype=np.uint16)
    if nd and ng:
        iou = MR.iou_matrix(det_boxes, gt_box)
        same = (det_classes[:, None] == np.asarray(gt_cls)[None, :]) & (det_classes[:, None] >= 0)
        nig = np.asarray(gt_nig, dtype=bool)
        for t, t0 in enumerate(iou_thresholds):
            thr = min(t0, 1 - 1e-10)
            ok = same & (iou >= thr)   # a NaN IoU never matches
            taken = np.zeros(ng, dtype=bool)
            for d in np.flatnonzero(ok.any(axis=1)):
                c = ok[d] & ~taken
                if not c.any():
                    continue
                if (c & nig).any():
                    c = c & nig
                best = iou[d][c].max()
                m = int(np.flatnonzero(c & (iou[d] == best))[-1])   # the later one on equal IoU
                taken[m] = True
                if nig[m]:
                    tp[d] |= np.uint16(1 << t)
                else:
                    ig[d] |= np.uint16(1 << t)
    tmask = np.uint16((1 << len(iou_thresholds)) - 1)
    ig = np.where(np.asarray(det_out, dtype=bool), tmask & ~tp, ig).astype(np.uint16)
    return tp, ig


def ranks(det_classes):
    """Rank of every detection among the earlier detections of its class (saturating at 65535); 0 for class -1."""
    det_classes = np.asarray(det_classes, dtype=np.int64)
    rank = np.zeros(len(det_classes), dtype=np.int64)
    order = np.argsort(det_classes, kind="stable")
    sc = det_classes[order]
    start = np.searchsorted(sc, sc, side="left")
    rank[order] = np.arange(len(sc)) - start
    rank[det_classes < 0] = 0
    return np.minimum(rank, 65535).astype(np.uint16)


def image_records(im, nc, iou_thresholds, max_det, area_rng=AREA_RNG):
    """The records of one image as yb_coco_match writes them: dict of score f32, cls i32, rank u16, tp (slots,4)
    u16, ig (slots,4) u16 (unused slots class -1, zero elsewhere); plus gt_count (A,nc) and the status bits."""
    slots = min(max_det, len(im["scores"]))
    gb, gc, db, ds, dc, status = _image_inputs(im, nc, max_det)
    nd, A = len(dc), len(area_rng)
    rec = {"score": np.zeros(slots, np.float32), "cls": np.full(slots, -1, np.int32),
           "rank": np.zeros(slots, np.uint16), "tp": np.zeros((slots, 4), np.uint16),
           "ig": np.zeros((slots, 4), np.uint16)}
    rec["score"][:nd] = ds
    rec["cls"][:nd] = dc
    rec["rank"][:nd] = ranks(dc)
    ga, da = box_area(gb), box_area(db.astype(np.float64))
    gt_count = np.zeros((A, nc), np.int64)
    for a, (lo, hi) in enumerate(area_rng):
        g_nig = ~((ga < lo) | (ga > hi))
        gt_count[a] = np.bincount(gc[(gc >= 0) & g_nig], minlength=nc)
        tp, ig = match_image(db, dc, (da < lo) | (da > hi), gb, gc, g_nig, iou_thresholds)
        rec["tp"][:nd, a] = tp
        rec["ig"][:nd, a] = ig
    return rec, gt_count, status


def accumulate(rec, gt_count, iou_thresholds, recall_thresholds, max_dets):
    """COCOeval.accumulate on records concatenated in image order, the ignored ones dropped (they change neither
    table).  Returns precision (T,R,nc,A,M) and recall (T,nc,A,M)."""
    T, R, M = len(iou_thresholds), len(recall_thresholds), len(max_dets)
    A, nc = gt_count.shape
    precision = -np.ones((T, R, nc, A, M))
    recall = -np.ones((T, nc, A, M))
    for c in range(nc):
        sel = np.flatnonzero(rec["cls"] == c)
        sel = sel[np.argsort(-rec["score"][sel], kind="mergesort")]
        rank, tpb, igb = rec["rank"][sel], rec["tp"][sel], rec["ig"][sel]
        for a in range(A):
            npig = int(gt_count[a, c])
            if npig == 0:
                continue
            for m, md in enumerate(max_dets):
                counted = rank < md
                for t in range(T):
                    is_tp = ((tpb[:, a] >> t) & 1).astype(bool)
                    kept = counted & ~((igb[:, a] >> t) & 1).astype(bool)
                    tps = np.cumsum(is_tp[kept]).astype(float)
                    fps = np.cumsum(~is_tp[kept]).astype(float)
                    nd = len(tps)
                    rc = tps / npig
                    pr = tps / (fps + tps + EPS)
                    recall[t, c, a, m] = rc[-1] if nd else 0
                    q = np.zeros(R)
                    if nd:
                        pr = np.maximum.accumulate(pr[::-1])[::-1]
                        pis = np.searchsorted(rc, recall_thresholds, side="left")
                        hit = pis < nd
                        q[hit] = pr[pis[hit]]
                    precision[t, :, c, a, m] = q
    return precision, recall


def evaluate(images, nc, iou_thresholds, recall_thresholds, max_det=300, max_dets=MAX_DETS, area_rng=AREA_RNG):
    """(b): images as map_ref.evaluate takes them.  Returns the fields of COCODetectionEval.compute() plus the
    records (concatenated), gt_count (A,nc) and status."""
    iou_thresholds = np.asarray(iou_thresholds, dtype=np.float64)
    recall_thresholds = np.asarray(recall_thresholds, dtype=np.float64)
    parts, status = [], 0
    gt_count = np.zeros((len(area_rng), nc), np.int64)
    for im in images:
        r, g, st = image_records(im, nc, iou_thresholds, max_det, area_rng)
        parts.append(r)
        gt_count += g
        status |= st
    empty = {"score": np.zeros(0, np.float32), "cls": np.zeros(0, np.int32), "rank": np.zeros(0, np.uint16),
             "tp": np.zeros((0, 4), np.uint16), "ig": np.zeros((0, 4), np.uint16)}
    rec = {k: np.concatenate([p[k] for p in parts] + [v]) for k, v in empty.items()}
    precision, recall = accumulate(rec, gt_count, iou_thresholds, recall_thresholds, max_dets)
    out = MR.summarize(precision[..., 0, len(max_dets) - 1], iou_thresholds)
    out.update(stats=summarize(precision, recall, iou_thresholds, max_dets), precision=precision, recall=recall,
               n_gt=gt_count.T.copy(), n_det=np.array([np.count_nonzero(rec["cls"] == c) for c in range(nc)], np.int64),
               gt_count=gt_count, records=rec, status=status)
    return out


def pack_records(rec):
    """Records as the (N, 8) int32 words of yb_coco_record, for a bit-exact comparison with the device's."""
    n = len(rec["score"])
    out = np.zeros((n, 8), np.int32)
    out[:, 0] = rec["score"].view(np.int32)
    out[:, 1] = rec["cls"]
    u16 = out.view(np.uint16).reshape(n, 16)
    u16[:, 4] = rec["rank"]
    u16[:, 6:10] = rec["tp"]
    u16[:, 10:14] = rec["ig"]
    return out
