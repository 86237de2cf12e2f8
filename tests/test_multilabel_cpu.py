"""Multi-label candidates without a GPU: the oracle (oracle/multilabel_ref.py) against a literal YOLO-style
restatement, and the public signatures the multi-label options were added to."""
import inspect
import types

import pytest
import torch

from oracle import multilabel_ref as ML
from oracle import ref_path as R

ANCH = R.default_anchors()


def yolo_style(preds, img, nc, conf, K, scale=1.0, pt=0.0, pl=0.0):
    """The validation tools' pipeline, literally: one (rows, 5+nc) table of sigmoids, objectness filter,
    x[:, 5:] *= x[:, 4:5], (row, class) pairs from nonzero, the best K by a stable argsort, candidate order restored."""
    xs = []
    for p, a in zip(preds, ANCH):
        d = R.decode(p, a, img)
        d[..., 4] = torch.sigmoid(p[..., 4])
        d[..., 5:] = torch.sigmoid(p[..., 5:])
        xs.append(d[0].reshape(-1, 5 + nc))
    x = torch.cat(xs)
    x = x[x[:, 4] > conf]
    x[:, 5:] *= x[:, 4:5]
    xy, wh = x[:, :2] * img, x[:, 2:4] * img
    box = torch.cat([xy - wh / 2, xy + wh / 2], 1)
    box = (box - torch.tensor([pl, pt, pl, pt])) / scale
    i, j = (x[:, 5:] > conf).nonzero(as_tuple=False).T
    b, s, c = box[i], x[i, j + 5], j
    n = s.shape[0]
    if n > K:
        keep = torch.sort(s.argsort(descending=True, stable=True)[:K]).values
        b, s, c = b[keep], s[keep], c[keep]
    return b, s, c, n


def heads(nc, seed, img=96, kind="randn"):
    g = torch.Generator().manual_seed(seed)
    out = []
    for G in (img // 8, img // 16, img // 32):
        h = torch.randn(1, G, G, 3, 5 + nc, generator=g) * 2.0
        if kind == "ties":   # a handful of logits: large groups of equal scores
            vals = torch.tensor([-1.0, 0.0, 0.5, 2.0])
            h[..., 4:] = vals[torch.randint(0, 4, h[..., 4:].shape, generator=g)]
        elif kind == "special":
            flat = h.view(-1)
            idx = torch.randint(0, flat.numel(), (flat.numel() // 20,), generator=g)
            flat[idx] = torch.tensor([float("nan"), float("inf"), -float("inf")])[torch.randint(0, 3, idx.shape, generator=g)]
        out.append(h)
    return out


def check(preds, nc, conf, K, lb=(1.0, 0.0, 0.0)):
    b, s, c, n = ML.candidates_multilabel(preds, ANCH, 96, nc, conf, K, *lb)
    wb, ws, wc, wn = yolo_style(preds, 96, nc, conf, K, *lb)
    assert n == wn and s.shape[0] == min(n, K)
    assert torch.equal(c, wc)
    assert torch.equal(s.view(torch.int32), ws.view(torch.int32))
    assert torch.equal(b.view(torch.int32), wb.view(torch.int32))
    return n


@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("kind", ["randn", "ties", "special"])
@pytest.mark.parametrize("conf", [0.001, 0.25, 0.5])
def test_oracle_equals_yolo_style(nc, kind, conf):
    preds = heads(nc, nc * 7 + len(kind), kind=kind)
    n = check(preds, nc, conf, 10 ** 9)
    for K in sorted({1, max(1, n // 3), max(1, n - 1), max(1, n)}):
        check(preds, nc, conf, K, lb=(0.75, 6.0, 2.0))


def test_ties_straddle_the_cap():
    preds = heads(3, 5, kind="ties")
    _, s, _, n = ML.candidates_multilabel(preds, ANCH, 96, 3, 0.001, 10 ** 9)
    srt = torch.sort(s, descending=True).values
    straddling = [k for k in range(1, n) if srt[k - 1] == srt[k]]   # the K-th and the (K+1)-th score are equal
    assert len(straddling) > n // 2
    for K in straddling[:: max(1, len(straddling) // 20)]:
        check(preds, 3, 0.001, K)


def test_nan_logits_give_no_candidates():
    preds = heads(3, 1)
    preds[0][..., 4] = float("nan")                  # no row of P3 is considered
    preds[1][..., 5] = float("nan")                  # class 0 of P4 gives nothing
    _, s, c, n = ML.candidates_multilabel(preds, ANCH, 96, 3, 0.001, 10 ** 9)
    assert n == s.shape[0] and not bool(torch.isnan(s).any())
    assert n < ML.candidates_multilabel(heads(3, 1), ANCH, 96, 3, 0.001, 10 ** 9)[3]
    check(preds, 3, 0.001, 10 ** 9)


def _params(fn):
    return [(p.name, p.kind, p.default) for p in inspect.signature(fn).parameters.values()]


P, K = inspect.Parameter.POSITIONAL_OR_KEYWORD, inspect.Parameter.KEYWORD_ONLY
E = inspect.Parameter.empty


def test_detect_signatures_keep_their_positions():
    from yolo_from_scratch_b200 import ops
    old = [("predictions", P, E), ("anchors_list", P, E), ("img_size", P, E), ("num_classes", P, 1),
           ("conf_threshold", P, 0.5), ("iou_threshold", P, 0.4), ("letterbox", P, None),
           ("trick_max_numel", P, ops.TRICK_MAX_NUMEL_CUDA), ("algo", P, ops.NMS_GRAPH)]
    new = [("multi_label", K, False), ("max_candidates", K, None), ("agnostic", K, False), ("max_det", K, None)]
    assert _params(ops.detect_batch) == old + [("layout", P, ops.LAYOUT_BHWAC)] + new
    nchw = _params(ops.detect_batch_nchw)
    assert nchw == [("raw_heads", P, E)] + old[1:] + new
    assert _params(ops.nms_candidates) == [
        ("boxes", P, E), ("scores", P, E), ("classes", P, E), ("counts", P, E), ("iou_threshold", P, 0.4),
        ("trick_max_numel", P, ops.TRICK_MAX_NUMEL_CUDA), ("algo", P, ops.NMS_GRAPH), ("agnostic", K, False),
        ("max_det", K, None)]


def test_evaluate_signatures_keep_their_positions():
    from yolo_from_scratch_b200 import install, ops
    m = types.ModuleType("train")
    head = [("model", P, E), ("dataset", P, E), ("device", P, E), ("num_classes", P, 1), ("conf_threshold", P, 0.001),
            ("iou_threshold", P, 0.4), ("batch_size", P, 8), ("max_det", P, 300)]
    new = [("multi_label", K, False), ("agnostic", K, False), ("max_candidates", K, None)]
    assert _params(install._make_evaluate_map(m)) == head + [("group", P, None)] + new
    assert _params(install._make_evaluate_report(m)) == head + [("group", P, None)] + new
    assert _params(install._make_evaluate_coco(m)) == head + [("max_dets", P, ops.COCO_MAX_DETS), ("group", P, None)] + new


def test_single_label_rejects_max_candidates():
    from yolo_from_scratch_b200 import ops
    with pytest.raises(ValueError, match="multi_label"):
        ops.detect_batch([torch.zeros(1, 2, 2, 3, 6)], ANCH, 64, max_candidates=10)
