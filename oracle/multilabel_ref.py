"""ORACLE (test infrastructure): multi-label candidates with a per-image top-K cap.

The semantics are include/yolo_b200.h's (yb_filter_multilabel).  The decode and the sigmoid slicing are
`ref_path.candidates`' own, so every box equals that function's box of the same row; the candidate pairs come from
`(scores > conf).nonzero()` over the rows that pass the objectness test, which is (row, class) lexicographic order.
Functions are device agnostic: run on CUDA tensors they reproduce torch-CUDA's arithmetic, on CPU tensors torch-CPU's.
"""
import torch

from . import ref_path as R

__all__ = ["candidates_multilabel", "cap_indices"]


def cap_indices(scores, max_candidates):
    """Indices of the kept candidates in candidate order: all of them when N <= K, else argsort(-score, stable)[:K]
    (ties at the K-th score go to the earlier candidates) sorted back into candidate order."""
    n = scores.shape[0]
    if n <= max_candidates:
        return torch.arange(n, device=scores.device)
    order = torch.argsort(-scores, stable=True)[:max_candidates]
    return torch.sort(order).values


def candidates_multilabel(preds, anchors_list, img_size, nc=1, conf=0.001, max_candidates=30000, scale=1.0, pad_top=0,
                          pad_left=0):
    """preds: list of (1,H,W,A,5+nc).  Returns boxes (M,4), scores (M,), classes (M,) int64 of the kept candidates in
    candidate order, and N, the number of candidates before the cap."""
    boxes, scores, classes = [], [], []
    for p, anchors in zip(preds, anchors_list):
        d = R.decode(p, anchors, img_size)                                    # ref_path.candidates' decode and slicing
        d[..., 4] = torch.sigmoid(p[..., 4])
        d[..., 5:] = torch.sigmoid(p[..., 5:])
        rows = d[0][d[0][..., 4] > conf]                                      # objectness test, row-major order
        if rows.shape[0] == 0:
            continue
        sc = rows[:, 4:5] * rows[:, 5:5 + nc]                                 # (M, nc): sigmoid(obj) * sigmoid(cls_c)
        ri, ci = (sc > conf).nonzero(as_tuple=True)                           # (row, class) lexicographic
        cx, cy, w, h = (rows[:, k] * img_size for k in range(4))
        x1, y1, x2, y2 = cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2
        x1, y1, x2, y2 = x1 - pad_left, y1 - pad_top, x2 - pad_left, y2 - pad_top
        x1, y1, x2, y2 = x1 / scale, y1 / scale, x2 / scale, y2 / scale
        boxes.append(torch.stack([x1, y1, x2, y2], dim=1)[ri])
        scores.append(sc[ri, ci])
        classes.append(ci.to(torch.int64))
    dev = preds[0].device
    if not boxes:
        return (torch.zeros(0, 4, device=dev), torch.zeros(0, device=dev), torch.zeros(0, dtype=torch.long, device=dev),
                0)
    b, s, c = torch.cat(boxes), torch.cat(scores), torch.cat(classes)
    keep = cap_indices(s, max_candidates)
    return b[keep], s[keep], c[keep], int(s.shape[0])

