"""Pins the oracle (oracle/) against the reference: committed golden vectors produced by the
unmodified reference (oracle/make_golden.py, oracle/make_golden_pinned.py), the reference's own known-answer
tests and the installed torchvision operator."""
import numpy as np
import pytest
import torch

import oracle
from oracle import ref_path as R

ANCH = R.default_anchors()


def T(a):
    return torch.from_numpy(np.asarray(a))


def canon(dets):
    """Detections as an array ordered by descending score; rows with EQUAL scores are put in a
    canonical order, because torchvision's per-class path ends in an unstable sort
    (ops/boxes.py:120) and leaves their relative order unspecified."""
    a = np.array(dets, dtype=np.float64).reshape(-1, 6)
    order = np.lexsort((a[:, 3], a[:, 2], a[:, 1], a[:, 0], -a[:, 4]))
    return a[order]


# ---- decode -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["g13_nc1", "g20_nc3", "g7x5_nc0", "g12_nc80"])
def test_decode_matches_reference_bitwise(golden, name):
    g = golden("decode")
    x = T(g[f"{name}_in"]).requires_grad_(True)
    y = R.decode(x, T(g["anchors"]), int(g[f"{name}_img"]))
    assert torch.equal(y.detach(), T(g[f"{name}_out"]))
    (y * T(g[f"{name}_gout"])).sum().backward()
    torch.testing.assert_close(x.grad, T(g[f"{name}_gin"]), rtol=1e-6, atol=1e-7)


# ---- CIoU -------------------------------------------------------------------------------------
def test_ciou_matches_reference(golden):
    g = golden("ciou")
    p, t = T(g["pred"]).requires_grad_(True), T(g["tgt"]).requires_grad_(True)
    loss = R.ciou(p, t)
    assert float(loss.detach()) == float(g["loss"])
    loss.backward()
    torch.testing.assert_close(p.grad, T(g["gpred"]), rtol=1e-6, atol=1e-8)
    torch.testing.assert_close(t.grad, T(g["gtgt"]), rtol=1e-6, atol=1e-8)


def test_ciou_reference_inequalities():
    # reference tests/test_loss.py:12-54
    assert float(R.ciou(T([[0.5, 0.5, 0.2, 0.3]]).float(), T([[0.5, 0.5, 0.2, 0.3]]).float())) < 0.01
    assert float(R.ciou(T([[0.1, 0.1, 0.1, 0.1]]).float(), T([[0.9, 0.9, 0.1, 0.1]]).float())) > 1.0
    assert 0.0 < float(R.ciou(T([[0.5, 0.5, 0.3, 0.3]]).float(), T([[0.6, 0.6, 0.3, 0.3]]).float())) < 1.0
    assert float(R.ciou(T([[0.5, 0.5, 0.2, 0.4]]).float(), T([[0.5, 0.5, 0.4, 0.2]]).float())) > 0.5


# ---- losses -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["nc1", "nc3", "nc80"])
def test_multiscale_loss_matches_reference(golden, name):
    g = golden("loss")
    B, img, nc = (int(v) for v in g[f"{name}_cfg"])
    preds = [T(g[f"{name}_pred{s}"]).requires_grad_(True) for s in range(3)]
    tgts = [T(g[f"{name}_tgt{s}"]) for s in range(3)]
    res = R.multiscale_loss(preds, tgts, ANCH, nc)
    np.testing.assert_array_equal(np.array([float(r.detach()) for r in res], dtype=np.float32), g[f"{name}_losses"])
    res[0].backward()
    for s in range(3):
        torch.testing.assert_close(preds[s].grad, T(g[f"{name}_grad{s}"]), rtol=1e-6, atol=1e-9)
    p1 = T(g[f"{name}_pred1"]).requires_grad_(True)
    r1 = R.single_scale_loss(p1, tgts[1], ANCH[1], nc)
    np.testing.assert_array_equal(np.array([float(r.detach()) for r in r1], dtype=np.float32), g[f"{name}_single_losses"])


def test_loss_without_positives(golden):
    g = golden("loss")
    preds = [T(g[f"empty_pred{s}"]) for s in range(3)]
    res = R.multiscale_loss(preds, [torch.zeros_like(p) for p in preds], ANCH, 1)
    np.testing.assert_array_equal(np.array([float(r.detach()) for r in res], dtype=np.float32), g["empty_losses"])
    assert float(res[1]) == 0.0 and float(res[3]) == 0.0 and float(res[2]) > 0.0  # tests/test_loss.py:91-109


# ---- target assignment ------------------------------------------------------------------------
def _dense_from_sparse(g, name, s, G, nc):
    t = np.zeros((G, G, 3, 5 + nc), dtype=np.float32)
    idx = g[f"{name}_s{s}_idx"]
    if len(idx):
        t[idx[:, 0], idx[:, 1], idx[:, 2]] = g[f"{name}_s{s}_rows"]
    return t


@pytest.mark.parametrize("name", ["a", "b", "c", "d", "e", "f", "g"])
def test_assignment_matches_reference_bitwise(golden, name):
    g = golden("targets")
    img, nc = (int(v) for v in g[f"{name}_cfg"])
    grids = [img // 8, img // 16, img // 32]
    lb = tuple(g[f"{name}_letterbox"])
    lb = (int(lb[0]), int(lb[1]), float(lb[2]), int(lb[3]), int(lb[4]))
    anchors = [ANCH[0]] * 3 if name == "g" else ANCH
    out = R.assign_targets(g[f"{name}_labels"], anchors, grids, nc, img, lb)
    for s in range(3):
        np.testing.assert_array_equal(out[s], _dense_from_sparse(g, name, s, grids[s], nc))


def test_shape_iou_matches_reference(golden):
    g = golden("targets")
    for i, wh in enumerate(g["aiou_wh"]):
        for s in range(3):
            np.testing.assert_array_equal(R.shape_iou(wh, ANCH[s].numpy()), g["aiou"][i, s])


# ---- predict path: filter + NMS ---------------------------------------------------------------
@pytest.mark.parametrize("name", ["p_nc1", "p_nc3", "p_nc80", "p_nc1_dense"])
@pytest.mark.parametrize("arith", ["cpu", "cuda"])
def test_detect_matches_reference_predict(golden, name, arith):
    g = golden("predict")
    img, nc, conf, iou, scale, pt, pl = g[f"{name}_cfg"]
    heads = [T(g[f"{name}_head{s}"]) for s in range(3)]
    dets, _, _ = R.detect(heads, ANCH, int(img), int(nc), float(conf), float(iou), float(scale), int(pt), int(pl),
                          arith=arith, device_rule="cpu")
    ref = g[f"{name}_dets"]
    assert len(dets) == len(ref)
    np.testing.assert_array_equal(np.array(dets, dtype=np.float64)[:, 4], ref[:, 4])  # same score sequence
    np.testing.assert_array_equal(canon(dets), canon(ref))


def test_model_heads_fixture(golden):
    """configs[0]: heads of the real random-init nc=1 model at 640x640."""
    g = golden("model_heads")
    heads = [T(g[f"head{s}"]) for s in range(3)]
    tgts = []
    for s, h in enumerate(heads):
        t = torch.zeros_like(h)
        idx = g[f"tgt{s}_idx"]
        if len(idx):
            t[idx[:, 0], idx[:, 1], idx[:, 2], idx[:, 3]] = T(g[f"tgt{s}_rows"])
        tgts.append(t)
    preds = [h.clone().requires_grad_(True) for h in heads]
    res = R.multiscale_loss(preds, tgts, ANCH, 1)
    np.testing.assert_array_equal(np.array([float(r.detach()) for r in res], dtype=np.float32), g["losses"])
    res[0].backward()
    for s in range(3):
        torch.testing.assert_close(preds[s].grad[..., 4], T(g[f"grad{s}_obj"]), rtol=1e-6, atol=1e-12)
    for k, conf in enumerate(g["confs"]):
        dets, _, _ = R.detect(heads, ANCH, 640, 1, float(conf), 0.4, arith="cpu", device_rule="cpu")
        np.testing.assert_array_equal(canon(dets), canon(g[f"dets_{k}"]))


# ---- NMS restatement vs the installed torchvision operator ------------------------------------
@pytest.mark.parametrize("name", ["small", "cls", "big", "neg"])
@pytest.mark.parametrize("thr", [0.3, 0.4, 0.7])
def test_nms_matches_torchvision_golden(golden, name, thr):
    g = golden("nms")
    b, s, c = g[f"{name}_boxes"], g[f"{name}_scores"], g[f"{name}_idxs"]
    np.testing.assert_array_equal(R.nms_indices(b, s, thr, "cpu"), g[f"{name}_nms_{thr}"])
    got = R.batched_nms_indices(b, s, c, thr, "cpu", device_rule="cpu")
    ref = g[f"{name}_bnms_{thr}"]
    # the per-class path ends in an unstable sort: equal scores may be permuted
    assert sorted(got.tolist()) == sorted(ref.tolist())
    np.testing.assert_array_equal(s[got], s[ref])


def test_nms_matches_live_torchvision():
    tv = pytest.importorskip("torchvision")
    g = torch.Generator().manual_seed(5)
    for n in (1, 2, 63, 64, 65, 777):
        xy = torch.rand(n, 2, generator=g) * 100
        boxes = torch.cat([xy, xy + torch.rand(n, 2, generator=g) * 60 + 0.5], dim=1)
        scores = torch.rand(n, generator=g)
        ref = tv.ops.nms(boxes, scores, 0.45).numpy()
        np.testing.assert_array_equal(R.nms_indices(boxes.numpy(), scores.numpy(), 0.45, "cpu"), ref)
    assert len(R.nms_indices(np.zeros((0, 4), np.float32), np.zeros(0, np.float32), 0.5)) == 0


def test_reference_python_nms_known_answers():
    # reference tests/test_inference.py:16-76, restated through the tensor NMS oracle as well
    def tensor_nms(dets, thr):
        if not dets:
            return []
        a = np.array(dets, dtype=np.float32)
        return [dets[i] for i in R.nms_indices(a[:, :4], a[:, 4], thr)]

    for fn in (R.python_list_nms, tensor_nms):
        assert fn([], 0.5) == []
        one = [(10, 10, 50, 50, 0.9, 0)]
        assert fn(one, 0.5) == one
        d = [(10, 10, 50, 50, 0.9, 0), (12, 12, 52, 52, 0.8, 0), (100, 100, 150, 150, 0.85, 0)]
        assert fn(d, 0.5) == [d[0], d[2]]
        d = [(10, 10, 50, 50, 0.9, 0), (100, 100, 150, 150, 0.8, 0), (200, 200, 250, 250, 0.85, 0)]
        assert len(fn(d, 0.5)) == 3
        d = [(10, 10, 50, 50, 0.6, 0), (12, 12, 52, 52, 0.9, 0)]
        r = fn(d, 0.5)
        assert len(r) == 1 and r[0][4] == 0.9
        d = [(10, 10, 50, 50, 0.9, 0), (20, 20, 60, 60, 0.8, 0)]
        assert len(fn(d, 0.3)) == 1 and len(fn(d, 0.7)) == 2


def test_corner_iou_known_answers():
    # reference tests/test_inference.py:79-109, tests/test_utils.py:82-90
    assert abs(R.corner_iou((10, 10, 50, 50), (10, 10, 50, 50)) - 1.0) < 1e-6
    assert R.corner_iou((10, 10, 50, 50), (100, 100, 150, 150)) == 0.0
    assert abs(R.corner_iou((0, 0, 2, 2), (1, 0, 3, 2)) - 1.0 / 3.0) < 1e-6
    assert abs(R.corner_iou((10, 10, 50, 50), (20, 20, 60, 60)) - R.corner_iou((20, 20, 60, 60), (10, 10, 50, 50))) < 1e-6


def test_cuda_arith_differs_only_by_fma():
    """The two arithmetic modes agree except on razor-edge pairs; the fixture must contain none."""
    rng = np.random.default_rng(3)
    xy = rng.uniform(0, 300, size=(2000, 2)).astype(np.float32)
    b = np.concatenate([xy, xy + rng.uniform(1, 90, size=(2000, 2)).astype(np.float32)], axis=1)
    s = rng.uniform(size=2000).astype(np.float32)
    np.testing.assert_array_equal(R.nms_indices(b, s, 0.4, "cpu"), R.nms_indices(b, s, 0.4, "cuda"))


# ---- the original's decode_predictions / yolo_loss on one seeded input (oracle/make_golden_pinned.py) ----
def test_live_reference_agrees(golden):
    g = golden("live_reference")
    x, tg, img = T(g["x"]), T(g["tgt"]), int(g["img"])
    assert torch.equal(R.decode(x, ANCH[2], img), T(g["decode"]))
    b = R.single_scale_loss(x, tg, ANCH[2], 3)
    assert [float(v) for v in b] == g["yolo_loss"].tolist()


@pytest.mark.parametrize("name", ["e640", "e320"])
def test_eval_counts_match_reference_eval_epoch(golden, name):
    """Oracle restatement of eval_epoch's counting (train.py:993-1024) against the four values the
    unmodified reference returned on the same preset heads/targets (oracle/make_golden.py)."""
    g = golden("eval")
    img, nc, B, nb, conf, iou = g[f"{name}_cfg"]
    tp = fp = fn = 0
    loss = 0.0
    for k in range(int(nb)):
        heads = [torch.from_numpy(g[f"{name}_b{k}_head{s}"]) for s in range(3)]
        tg = [torch.from_numpy(g[f"{name}_b{k}_tgt{s}"]) for s in range(3)]
        a, b, c = R.eval_counts(heads, tg, R.default_anchors(), float(conf), float(iou))
        tp, fp, fn = tp + a, fp + b, fn + c
        loss += float(R.multiscale_loss(heads, tg, R.default_anchors(), int(nc))[0])
    want = g[f"{name}_result"]
    assert loss / int(nb) == want[0]
    assert R.eval_metrics(tp, fp, fn) == tuple(want[1:])
    assert tp > 0 and fp > 0 and fn > 0
