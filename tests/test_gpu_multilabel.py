"""Multi-label candidates on the device (yb_filter_multilabel, ops.filter_candidates_multilabel, detect_batch(
multi_label=True)) against the oracle (oracle/multilabel_ref.py, evaluated on CUDA tensors so that its sigmoids and
products are torch-CUDA's), against the single-label filter, and through NMS, graph capture and the evaluators.

Counts, classes and order are exact and scores bit for bit; boxes against the oracle keep the tolerance of the other
filter tests (the kernel multiplies by 1/W and 1/scale where the oracle divides), and are bit-identical to the
single-label filter's."""
import types

import numpy as np
import pytest
import torch

from yolo_from_scratch_b200 import ops
from oracle import coco_ref as C
from oracle import map_ref as M
from oracle import multilabel_ref as ML
from oracle import ref_path as R
from oracle import report_ref as P

pytestmark = pytest.mark.gpu

ANCH = R.default_anchors()
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
THR = np.asarray(ops.COCO_IOU_THRESHOLDS)
REC = np.asarray(ops.COCO_RECALL_THRESHOLDS)
GRID = np.asarray(ops.DEFAULT_CONF_GRID)


def bits(t):
    return t.contiguous().view(torch.int32)


def box_close(got, want):
    """Within the filter tests' tolerance; a NaN coordinate (a NaN box logit) must be NaN on both sides."""
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), "boxes: NaN coordinates differ"
    err = (got.double() - want.double()).abs()[~nan]
    tol = (1e-5 * want.double().abs() + 2e-4)[~nan]
    assert bool((err <= tol).all()), f"boxes: max err {float(err.max()):.3e}"


def to_nchw(h):
    B, H, W, A, Cc = h.shape
    return h.permute(0, 3, 4, 1, 2).reshape(B, A * Cc, H, W).contiguous()


def make_heads(B, img, nc, seed, dtype=torch.float32, kind="randn"):
    """Reference-layout heads on the GPU.  'randn': dense (every image far over a small cap at conf 0.001); 'prior':
    SURVEY 8d's prior objectness; 'ties': a handful of logits, so that equal scores straddle any cap; 'mixed': image 1
    is empty (objectness -30), image 2 has NaN and +-inf logits."""
    g = torch.Generator().manual_seed(seed)
    heads = []
    for G in (img // 8, img // 16, img // 32):
        h = torch.randn(B, G, G, 3, 5 + nc, generator=g) * 2.0
        if kind == "prior":
            h[..., 4].mul_(1.0).sub_(4.6)
        elif kind == "ties":
            vals = torch.tensor([-1.0, 0.0, 0.5, 2.0])
            h[..., 4:] = vals[torch.randint(0, 4, h[..., 4:].shape, generator=g)]
        elif kind == "mixed":
            if B > 1:
                h[1, ..., 4] = -30.0
            if B > 2:
                flat = h[2].reshape(-1)
                idx = torch.randint(0, flat.numel(), (flat.numel() // 20,), generator=g)
                flat[idx] = torch.tensor([float("nan"), float("inf"), -float("inf")])[
                    torch.randint(0, 3, idx.shape, generator=g)]
                h[2] = flat.view(h[2].shape)
        heads.append(h.to(dtype).cuda())
    return heads


def run(heads, img, nc, conf, K, layout="bhwac", lbx=None):
    hs = [to_nchw(h) for h in heads] if layout == "nchw" else heads
    lay = ops.LAYOUT_NCHW if layout == "nchw" else ops.LAYOUT_BHWAC
    return ops.filter_candidates_multilabel(hs, ANCH, img, nc, conf, letterbox=lbx, layout=lay, max_candidates=K)


def pairs(heads, img, nc):
    return sum(h.shape[1] * h.shape[2] * h.shape[3] for h in heads) * nc


@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("conf", [0.001, 0.25, 0.5])
@pytest.mark.parametrize("dt", list(DTYPES))
def test_uncapped_equals_oracle(nc, conf, dt):
    img, B = 96, 3
    heads = make_heads(B, img, nc, nc * 100 + int(conf * 1000), DTYPES[dt], kind="mixed")
    up = [h.float() for h in heads]                       # half heads: the fp32 oracle on the upcast heads
    lbx = [(0.75, 6.0, 2.0), (1.0, 0.0, 0.0), (1.25, 0.0, 8.0)]
    K = pairs(heads, img, nc)
    for layout in ("bhwac", "nchw"):
        for lb in (None, lbx):
            boxes, scores, classes, counts, totals = run(heads, img, nc, conf, K, layout, lb)
            assert boxes.shape[1] == K
            for b in range(B):
                sc, pt, pl = lb[b] if lb else (1.0, 0.0, 0.0)
                rb, rs, rc, n = ML.candidates_multilabel([h[b:b + 1] for h in up], ANCH, img, nc, conf, K, sc, pt, pl)
                what = f"{layout} lb={lb is not None} image {b}"
                assert int(counts[b]) == n == int(totals[b]) == rs.shape[0], what
                assert torch.equal(classes[b, :n], rc), what
                assert torch.equal(bits(scores[b, :n]), bits(rs)), what
                box_close(boxes[b, :n], rb)
            assert int(counts[1]) == 0   # the empty image
    assert int(counts[0]) > 0


def test_batch_of_zero_images():
    heads = [h[:0] for h in make_heads(1, 64, 3, 1)]
    boxes, scores, classes, counts, totals = ops.filter_candidates_multilabel(heads, ANCH, 64, 3, 0.001)
    assert boxes.shape == (0, min(ops.MAX_CANDIDATES, pairs(heads, 64, 3)), 4)
    assert counts.shape == (0,) and totals.shape == (0,)
    det = ops.detect_batch(heads, ANCH, 64, 3, 0.001, multi_label=True)
    assert det["n_keep"].shape == (0,)


@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
def test_against_single_label_filter(nc, layout):
    """Rows with candidates are the single-label candidates whose score > conf; their boxes are bit-identical and
    the largest multi-label score of a row is the single-label score."""
    img, conf = 160, 0.05
    heads = make_heads(2, img, nc, 40 + nc)
    hs = [to_nchw(h) for h in heads] if layout == "nchw" else heads
    lay = ops.LAYOUT_NCHW if layout == "nchw" else ops.LAYOUT_BHWAC
    lbx = [(0.8, 16.0, 0.0), (1.5, 0.0, 4.0)]
    sb, ss, sc, sn = ops.filter_candidates(hs, ANCH, img, nc, conf, letterbox=lbx, layout=lay)
    mb, ms, mc, mn, mt = ops.filter_candidates_multilabel(hs, ANCH, img, nc, conf, letterbox=lbx, layout=lay,
                                                          max_candidates=pairs(heads, img, nc))
    for b in range(2):
        n1, n = int(sn[b]), int(mn[b])
        sel = ss[b, :n1] > conf
        rb, rs = sb[b, :n1][sel], ss[b, :n1][sel]
        box, sco = bits(mb[b, :n]), ms[b, :n]
        new_row = torch.ones(n, dtype=torch.bool, device="cuda")
        new_row[1:] = (box[1:] != box[:-1]).any(1)          # candidates of a row are adjacent and share its box
        starts = new_row.nonzero().flatten()
        assert starts.numel() == rs.numel()
        assert torch.equal(box[starts], bits(rb))
        row_id = torch.cumsum(new_row.long(), 0) - 1
        best = torch.full((starts.numel(),), -1.0, device="cuda").scatter_reduce(0, row_id, sco, "amax")
        assert torch.equal(bits(best), bits(rs))
        if nc == 1:
            assert n == rs.numel() and torch.equal(bits(sco), bits(rs)) and bool((mc[b, :n] == 0).all())


def check_cap(full, capped, K):
    fb, fs, fc, fn, ft = full
    cb, cs, cc, cn, ct = capped
    for b in range(fb.shape[0]):
        n = int(fn[b])
        assert int(ft[b]) == n and int(ct[b]) == n, "totals = N"
        keep = ML.cap_indices(fs[b, :n], K)
        m = keep.numel()
        assert int(cn[b]) == min(n, K) == m
        assert torch.equal(bits(cs[b, :m]), bits(fs[b, :n][keep]))
        assert torch.equal(cc[b, :m], fc[b, :n][keep])
        assert torch.equal(bits(cb[b, :m]), bits(fb[b, :n][keep]))


@pytest.mark.parametrize("kind", ["randn", "ties"])
@pytest.mark.parametrize("layout,dt", [("bhwac", "f32"), ("nchw", "f32"), ("bhwac", "bf16"), ("nchw", "f16")])
def test_cap_equals_stable_topk_of_uncapped(kind, layout, dt):
    img, nc, conf = 128, 80 if kind == "randn" else 3, 0.001
    heads = make_heads(3, img, nc, 7, DTYPES[dt], kind=kind)
    full = run(heads, img, nc, conf, pairs(heads, img, nc), layout)
    N = int(full[3][0])
    assert N > 1000
    Ks = [1, N - 1, N, N + 1, N // 2, 30000]
    if kind == "ties":   # K inside a group of equal scores
        srt = torch.sort(full[1][0, :N], descending=True).values
        mid = ((srt[1:] == srt[:-1]).nonzero().flatten() + 1).tolist()
        Ks += mid[len(mid) // 3: len(mid) // 3 + 1] + mid[2 * len(mid) // 3: 2 * len(mid) // 3 + 1]
        assert len(mid) > N // 2
    for K in Ks:
        check_cap(full, run(heads, img, nc, conf, K, layout), K)


def check_keep(det, agnostic=False):
    keep, n_keep, counts = det["keep"].cpu(), det["n_keep"].cpu(), det["counts"].cpu()
    for b in range(keep.shape[0]):
        m = int(counts[b])
        bx, sc = det["boxes"][b, :m].cpu().numpy(), det["scores"][b, :m].cpu().numpy()
        cl = det["classes"][b, :m].cpu().numpy()
        want = R.nms_indices(bx, sc, det["iou_threshold"]) if agnostic else \
            R.batched_nms_indices(bx, sc, cl, det["iou_threshold"])
        got = keep[b, :int(n_keep[b])].numpy()
        assert np.array_equal(got, want), b


@pytest.mark.parametrize("K", [20000, 30000])
def test_nms_keep_sets(K):
    """K = 20000 at nc = 80 stays under batched_nms' 100,000-element dispatch (coordinate trick), 30000 takes the
    per-class loop."""
    heads = make_heads(2, 256, 80, 3, kind="prior")
    det = ops.detect_batch(heads, ANCH, 256, 80, 0.001, 0.4, multi_label=True, max_candidates=K)
    assert int(det["counts"].min()) == K and bool((det["totals"] > K).all())
    assert det["multi_label"] and det["max_candidates"] == K
    check_keep(det)


def test_agnostic_and_max_det():
    heads = make_heads(2, 256, 80, 4, kind="prior")
    lbx = [(0.5, 0.0, 64.0), (1.0, 0.0, 0.0)]
    det = ops.detect_batch(heads, ANCH, 256, 80, 0.001, 0.5, lbx, multi_label=True, max_candidates=6000, agnostic=True)
    assert det["agnostic"]
    check_keep(det, agnostic=True)
    cl = det["classes"]
    assert bool((cl[0, :int(det["counts"][0])] > 0).any())   # the detections keep their classes
    full = ops.detect_batch(heads, ANCH, 256, 80, 0.001, 0.5, lbx, multi_label=True, max_candidates=6000)
    for md in (0, 1, 100, 10 ** 6):
        cut = ops.detect_batch(heads, ANCH, 256, 80, 0.001, 0.5, lbx, multi_label=True, max_candidates=6000, max_det=md)
        assert torch.equal(cut["n_keep"], full["n_keep"].clamp(max=md)) and cut["max_det"] == md
        for b in range(2):
            k = int(cut["n_keep"][b])
            assert torch.equal(cut["keep"][b, :k], full["keep"][b, :k])
    lists = ops.detections_to_lists(ops.detect_batch(heads, ANCH, 256, 80, 0.001, 0.5, lbx, multi_label=True,
                                                     max_candidates=6000, max_det=7))
    assert [len(x) for x in lists] == [7, 7]


def test_max_det_keeps_a_failed_image_failed():
    """The bitmask NMS fails an image with a class id >= 65536 (n_keep = -1); max_det must leave that -1 and cut the
    other image's kept list."""
    g = torch.Generator().manual_seed(3)
    xy = torch.rand(2, 40, 2, generator=g) * 200
    boxes = torch.cat([xy, xy + 5 + torch.rand(2, 40, 2, generator=g) * 30], 2).cuda()
    scores = torch.rand(2, 40, generator=g).cuda()
    classes = torch.randint(0, 3, (2, 40), generator=g).cuda()
    classes[0, 7] = 70000
    counts = torch.tensor([40, 40], dtype=torch.int32, device="cuda")
    full = ops.nms_candidates(boxes, scores, classes, counts, 0.4, algo=ops.NMS_BITMASK)
    assert int(full["n_keep"][0]) == -1 and int(full["n_keep"][1]) > 3
    cut = ops.nms_candidates(boxes, scores, classes, counts, 0.4, algo=ops.NMS_BITMASK, max_det=3)
    assert cut["n_keep"].tolist() == [-1, 3]
    assert torch.equal(cut["keep"][1, :3], full["keep"][1, :3])
    with pytest.raises(RuntimeError):
        ops.detections_to_lists(cut)
    with pytest.raises(ValueError):
        ops.nms_candidates(boxes, scores, classes, counts, max_det=-1)


FLT_MIN = 1.1754943508222875e-38


@pytest.mark.parametrize("conf", [-0.5, 0.0, 1e-40, FLT_MIN, 2e-38, 1e-30])
def test_thresholds_near_and_below_flt_min(conf):
    """Thresholds at, below and above FLT_MIN, including 0 and a negative one, on logits around where 1/(1+expf(-x))
    leaves the normal range (-87.3, where the IEEE division takes its slow path) and reaches 0 (-103.3), -inf and NaN:
    candidates, classes and score bits (subnormal ones included) must equal the oracle's, capped and uncapped."""
    img, nc, B = 64, 3, 2
    g = torch.Generator().manual_seed(17)
    vals = torch.tensor([-120.0, -103.9, -103.3, -100.0, -95.0, -88.8, -88.7, -87.4, -87.3, -87.0, -60.0, -10.0, 0.0,
                         3.0, float("-inf"), float("nan")])
    heads = []
    for G in (img // 8, img // 16, img // 32):
        h = torch.randn(B, G, G, 3, 5 + nc, generator=g)
        h[..., 4:] = vals[torch.randint(0, len(vals), h[..., 4:].shape, generator=g)]
        heads.append(h.cuda())
    K = pairs(heads, img, nc)
    for layout in ("bhwac", "nchw"):
        full = run(heads, img, nc, conf, K, layout)
        for b in range(B):
            rb, rs, rc, n = ML.candidates_multilabel([h[b:b + 1] for h in heads], ANCH, img, nc, conf, K)
            assert int(full[3][b]) == n == rs.shape[0]
            assert torch.equal(full[2][b, :n], rc) and torch.equal(bits(full[1][b, :n]), bits(rs))
            box_close(full[0][b, :n], rb)
        n0 = int(full[3][0])
        assert n0 > 10
        for Kc in (1, n0 // 2, n0 - 1):
            check_cap(full, run(heads, img, nc, conf, Kc, layout), Kc)


@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
def test_defaults_are_unchanged(layout):
    heads = make_heads(3, 160, 3, 9, kind="prior")
    hs = [to_nchw(h) for h in heads] if layout == "nchw" else heads
    fn = ops.detect_batch_nchw if layout == "nchw" else ops.detect_batch
    lib = ops._lib.lib()
    n0 = lib.yb_launch_count()
    a = fn(hs, ANCH, 160, 3, 0.01, 0.4)
    n1 = lib.yb_launch_count()
    b = fn(hs, ANCH, 160, 3, 0.01, 0.4, multi_label=False, max_candidates=None, agnostic=False, max_det=None)
    n2 = lib.yb_launch_count()
    assert n1 - n0 == n2 - n1
    for k in ("boxes", "scores", "classes", "counts", "keep", "n_keep"):
        x, y = a[k], b[k]
        assert x.shape == y.shape and x.dtype == y.dtype, k
    for k in ("counts", "n_keep"):
        assert torch.equal(a[k], b[k])
    for bb in range(3):
        m, k = int(a["counts"][bb]), int(a["n_keep"][bb])
        assert torch.equal(bits(a["boxes"][bb, :m]), bits(b["boxes"][bb, :m]))
        assert torch.equal(bits(a["scores"][bb, :m]), bits(b["scores"][bb, :m]))
        assert torch.equal(a["classes"][bb, :m], b["classes"][bb, :m])
        assert torch.equal(a["keep"][bb, :k], b["keep"][bb, :k])
    assert "totals" not in a and not a["multi_label"] and not a["agnostic"] and a["max_det"] is None


@pytest.mark.parametrize("K", [500, 10 ** 7])
def test_graph_capture_replays_on_new_heads(K):
    img, nc = 128, 80
    static = make_heads(2, img, nc, 11)
    anch = [a.cuda() for a in ANCH]   # nothing to upload inside the capture
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.filter_candidates_multilabel(static, anch, img, nc, 0.001, max_candidates=K)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ops.filter_candidates_multilabel(static, anch, img, nc, 0.001, max_candidates=K)
    for seed, kind in ((12, "randn"), (13, "ties")):
        for st, h in zip(static, make_heads(2, img, nc, seed, kind=kind)):
            st.copy_(h)
        g.replay()
        torch.cuda.synchronize()
        want = ops.filter_candidates_multilabel(static, anch, img, nc, 0.001, max_candidates=K)
        n = int(want[3].max())
        for x, y in zip(out, want):
            if x.dim() == 1:
                assert torch.equal(x, y)
        for b in range(2):
            m = int(want[3][b])
            assert torch.equal(bits(out[0][b, :m]), bits(want[0][b, :m]))
            assert torch.equal(bits(out[1][b, :m]), bits(want[1][b, :m]))
            assert torch.equal(out[2][b, :m], want[2][b, :m])
        assert n > 0 and (K > 10 ** 6 or n == K)


# ---- evaluators ---------------------------------------------------------------------------------------------------
def host_images(det, labels, letterbox):
    d = {k: det[k].cpu().numpy() for k in ("boxes", "scores", "classes", "keep", "n_keep")}
    return [{"boxes": d["boxes"][b], "scores": d["scores"][b], "classes": d["classes"][b], "keep": d["keep"][b],
             "n_keep": int(d["n_keep"][b]), "labels": labels[b], "letterbox": letterbox[b]} for b in range(len(labels))]


def two_class_boxes(hb):
    """Kept detections of one image whose box is kept under two classes."""
    n = 0
    for im in hb:
        k = im["keep"][:min(im["n_keep"], 300)]
        seen = {}
        for i in k:
            key = im["boxes"][i].tobytes()
            seen.setdefault(key, set()).add(int(im["classes"][i]))
        n += sum(1 for v in seen.values() if len(v) > 1)
    return n


@pytest.mark.parametrize("nc", [3, 80])
@pytest.mark.parametrize("agnostic", [False, True])
def test_evaluators_on_multilabel_detections(nc, agnostic):
    rng = np.random.default_rng(nc + agnostic)
    img, B = 320, 6
    mp, co, rep = ops.DetectionMAP(nc), ops.COCODetectionEval(nc), ops.DetectionReport(nc, cm_conf=0.05)
    images, twice = [], 0
    for step in range(2):
        heads = make_heads(B, img, nc, 200 + step, kind="prior")
        lbx = [(float(rng.uniform(0.5, 1.5)), float(rng.integers(0, 20)), float(rng.integers(0, 20))) for _ in range(B)]
        det = ops.detect_batch(heads, ANCH, img, nc, 0.001, 0.4, lbx, multi_label=True, agnostic=agnostic)
        assert det["boxes"].shape[1] == min(ops.MAX_CANDIDATES, pairs(heads, img, nc))
        hb = host_images(det, [None] * B, [None] * B)
        twice += two_class_boxes(hb)
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
        pk = ops.pack_labels(labels, img, letterbox)
        for metric in (mp, co, rep):
            metric.update(det, pk)
        images += host_images(det, labels, letterbox)
    if not agnostic:
        assert twice > 0, "no box kept under two classes"
    got, want = mp.compute(), M.evaluate(images, nc, THR, REC, max_det=300)
    assert np.array_equal(got["precision"], want["precision"]) and np.array_equal(got["recall"], want["recall"])
    assert np.array_equal(got["n_gt"], want["n_gt"]) and np.array_equal(got["n_det"], want["n_det"])
    assert abs(got["map"] - want["map"]) <= 1e-12
    got, want = co.compute(), C.evaluate(images, nc, THR, REC)
    assert np.array_equal(got["precision"], want["precision"]) and np.array_equal(got["recall"], want["recall"])
    assert np.allclose(got["stats"], want["stats"], rtol=0, atol=1e-12)
    got, want = rep.compute(), P.evaluate(images, nc, THR, GRID, cm_conf=0.05)
    for k in ("confusion", "images", "p_curve", "r_curve", "f1_curve", "n_det", "precision", "recall"):
        assert np.array_equal(got[k], want[k]), k
    assert got["best_conf"] == want["best_conf"]


class _PresetHeads:
    def __init__(self, heads, img_size, anchors):
        self.heads, self.img_size, self.anchors = heads, img_size, anchors

    def eval(self):
        return self

    def __call__(self, img):
        return [h[:img.shape[0]] for h in self.heads]


def test_evaluate_map_multilabel_through_install(tmp_path):
    import pathlib

    from PIL import Image

    from yolo_from_scratch_b200.install import PATCHED_FUNCTIONS, install, uninstall
    nc, img, scale, pt, pl = 3, 160, 0.8, 16, 0
    wh = (200, 160)
    rng = np.random.default_rng(13)
    heads = make_heads(3, img, nc, 7, kind="prior")
    model = _PresetHeads(heads, img, [a.cuda() for a in ANCH])
    imgs, lab_files, labels = [], [], []
    for i in range(7):
        p = tmp_path / f"im{i}.png"
        Image.fromarray(np.zeros((wh[1], wh[0], 3), dtype=np.uint8)).save(p)
        imgs.append(str(p))
        lf = tmp_path / f"im{i}.txt"
        lab = np.column_stack([rng.integers(0, nc, 4), rng.uniform(0.2, 0.8, (4, 2)), rng.uniform(0.05, 0.4, (4, 2))])
        with open(lf, "w") as f:
            for r in lab:
                f.write(f"{int(r[0])} {r[1]} {r[2]} {r[3]} {r[4]}\n")
        lab_files.append(str(lf))
        labels.append(np.column_stack([lab[:, 0].astype(np.int64), lab[:, 1:]]).astype(np.float64).reshape(-1, 5))
    dataset = types.SimpleNamespace(imgs=imgs, labels=lab_files)
    m = types.ModuleType("train")
    m.Image, m.Path = Image, pathlib.Path
    m.letterbox_resize = lambda pil_img, img_size: (pil_img, scale, pt, pl)
    for n in PATCHED_FUNCTIONS + ("predict",):
        setattr(m, n, lambda *a, **k: "ref")
    train = install(m)
    try:
        dev = torch.device("cuda")
        got = train.evaluate_map(model, dataset, dev, nc, 0.001, 0.4, 3, 300, None, multi_label=True, max_candidates=900)
        plain = train.evaluate_map(model, dataset, dev, nc, 0.001, 0.4, 3)
        again = train.evaluate_map(model, dataset, dev, num_classes=nc, batch_size=3, multi_label=False)
    finally:
        uninstall(train)
    images, images1 = [], []
    for i0 in range(0, 7, 3):
        n = min(3, 7 - i0)
        lbx = [(scale, pt, pl)] * n
        det = ops.detect_batch([h[:n] for h in heads], ANCH, img, nc, 0.001, 0.4, letterbox=lbx, multi_label=True,
                               max_candidates=900)
        images += host_images(det, labels[i0:i0 + n], [wh + (scale, pt, pl)] * n)
        det1 = ops.detect_batch([h[:n] for h in heads], ANCH, img, nc, 0.001, 0.4, letterbox=lbx)
        images1 += host_images(det1, labels[i0:i0 + n], [wh + (scale, pt, pl)] * n)
    want = M.evaluate(images, nc, THR, REC, max_det=300)
    assert np.array_equal(got["precision"], want["precision"]) and abs(got["map"] - want["map"]) <= 1e-12
    want1 = M.evaluate(images1, nc, THR, REC, max_det=300)
    for r in (plain, again):
        assert np.array_equal(r["precision"], want1["precision"]) and r["map"] == plain["map"]
    assert not np.array_equal(got["n_det"], plain["n_det"])   # the multi-label run scored other detections
