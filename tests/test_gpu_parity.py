"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C-ABI,
against the oracle and the committed golden vectors of the reference.

Tolerances (BASELINE.json north_star): target assignment and NMS keep sets bit-exact; decoded
boxes, losses and gradients within 1e-5 relative fp32 (gradients: 1e-5 of the tensor's largest
magnitude plus 1e-4 elementwise, because single entries suffer cancellation in BOTH fp32
implementations — the reference's own CPU and CUDA runs differ by as much).
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ref_path as R  # noqa: E402  (checker only)

ANCH = R.default_anchors()
RTOL = 1e-5


def T(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture(scope="module")
def yb():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import yolo_from_scratch_b200 as m
    m._lib.lib()  # fail loudly if the extension is missing
    return m


def close(a, b, rtol=RTOL, atol=0.0):
    a, b = torch.as_tensor(a).detach().cpu().double(), torch.as_tensor(b).detach().cpu().double()
    err = (a - b).abs()
    tol = rtol * b.abs() + atol
    assert bool((err <= tol).all()), f"max err {float(err.max()):.3e}, max excess {float((err - tol).max()):.3e}"


def grad_close(a, b):
    b = torch.as_tensor(b)
    close(a, b, rtol=1e-4, atol=1e-5 * float(b.abs().max()) + 1e-12)


# ---- decode -----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["g13_nc1", "g20_nc3", "g7x5_nc0", "g12_nc80"])
def test_decode_golden(yb, golden, name):
    g = golden("decode")
    x = T(g[f"{name}_in"]).cuda().requires_grad_(True)
    y = yb.decode_predictions(x, T(g["anchors"]), int(g[f"{name}_img"]))
    ref = T(g[f"{name}_out"])
    assert y.shape == ref.shape and y.device.type == "cuda"
    close(y[..., :4], ref[..., :4], atol=1e-7)
    assert torch.equal(y[..., 4:].cpu(), ref[..., 4:])  # logits untouched, bit for bit
    (y * T(g[f"{name}_gout"]).cuda()).sum().backward()
    grad_close(x.grad, g[f"{name}_gin"])


def test_decode_cpu_tensor_staging(yb):
    # reference tests/test_loss.py:245-315 pass CPU tensors and expect CPU results / grads
    x = torch.randn(1, 20, 20, 3, 6, requires_grad=True)
    y = yb.decode_predictions(x, ANCH[0], img_size=640)
    assert y.device.type == "cpu" and y.shape == x.shape
    assert (y[..., 2] > 0).all() and (y[..., 3] > 0).all()
    assert torch.equal(y[..., 4:], x[..., 4:].detach())
    y[..., :4].mean().backward()
    assert x.grad is not None and x.grad.device.type == "cpu"
    z = yb.decode_predictions(torch.zeros(1, 20, 20, 3, 6), ANCH[0], img_size=640)
    assert (z[..., 0] >= 0).all() and (z[..., 0] <= 1).all()


@pytest.mark.parametrize("shape", [(64, 80, 80, 3, 6), (8, 40, 40, 3, 85), (1, 1, 1, 1, 5), (3, 5, 9, 2, 7)])
def test_decode_vs_oracle_sizes(yb, shape):
    g = torch.Generator().manual_seed(3)
    x = torch.randn(*shape, generator=g) * 3
    anc = torch.tensor([[10., 13.], [16., 30.], [33., 23.]])[: shape[3]]
    y = yb.decode_predictions(x.cuda(), anc, 640)
    ref = R.decode(x, anc, 640)
    close(y[..., :4], ref[..., :4], atol=1e-7)
    assert torch.equal(y[..., 4:].cpu(), ref[..., 4:])


# ---- CIoU -------------------------------------------------------------------------------------
def test_ciou_golden(yb, golden):
    g = golden("ciou")
    p, t = T(g["pred"]).cuda().requires_grad_(True), T(g["tgt"]).cuda().requires_grad_(True)
    loss = yb.ciou_loss(p, t)
    close(loss, float(g["loss"]))
    loss.backward()
    grad_close(p.grad, g["gpred"])
    grad_close(t.grad, g["gtgt"])


def test_ciou_reference_inequalities(yb):
    f = lambda a, b: float(yb.ciou_loss(torch.tensor([a]), torch.tensor([b])))
    assert f([0.5, 0.5, 0.2, 0.3], [0.5, 0.5, 0.2, 0.3]) < 0.01
    assert f([0.1, 0.1, 0.1, 0.1], [0.9, 0.9, 0.1, 0.1]) > 1.0
    assert 0.0 < f([0.5, 0.5, 0.3, 0.3], [0.6, 0.6, 0.3, 0.3]) < 1.0
    assert f([0.5, 0.5, 0.2, 0.4], [0.5, 0.5, 0.4, 0.2]) > 0.5
    assert torch.isnan(yb.ciou_loss(torch.zeros(0, 4), torch.zeros(0, 4)))


# ---- fused loss -------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["nc1", "nc3", "nc80"])
def test_multiscale_loss_golden(yb, golden, name):
    g = golden("loss")
    B, img, nc = (int(v) for v in g[f"{name}_cfg"])
    preds = [T(g[f"{name}_pred{s}"]).cuda().requires_grad_(True) for s in range(3)]
    tgts = [T(g[f"{name}_tgt{s}"]).cuda() for s in range(3)]
    res = yb.yolo_loss_multiscale(preds, tgts, ANCH, nc)
    for a, b in zip(res, g[f"{name}_losses"]):
        close(a, float(b), atol=1e-7)
    res[0].backward()
    for s in range(3):
        grad_close(preds[s].grad, g[f"{name}_grad{s}"])
    p1 = T(g[f"{name}_pred1"]).cuda().requires_grad_(True)
    r1 = yb.yolo_loss(p1, tgts[1], ANCH[1], nc)
    for a, b in zip(r1, g[f"{name}_single_losses"]):
        close(a, float(b), atol=1e-7)
    r1[0].backward()
    grad_close(p1.grad, g[f"{name}_single_grad"])


def test_loss_without_positives(yb, golden):
    g = golden("loss")
    preds = [T(g[f"empty_pred{s}"]).cuda() for s in range(3)]
    res = yb.yolo_loss_multiscale(preds, [torch.zeros_like(p) for p in preds], ANCH, 1)
    for a, b in zip(res, g["empty_losses"]):
        close(a, float(b), atol=1e-7)
    assert float(res[1]) == 0.0 and float(res[3]) == 0.0 and float(res[2]) > 0.0


def test_loss_cpu_tensors_and_grad_flow(yb):
    # reference tests/test_loss.py:208-242
    preds = [torch.randn(2, G, G, 3, 6, requires_grad=True) for G in (80, 40, 20)]
    tgts = [torch.zeros(2, G, G, 3, 6) for G in (80, 40, 20)]
    tgts[0][0, 40, 40, 0, :5] = torch.tensor([0.5, 0.5, 0.2, 0.3, 1.0])
    tgts[0][0, 40, 40, 0, 5] = 1.0
    total, bbox, obj, cls = yb.yolo_loss_multiscale(preds, tgts, ANCH, 1)
    assert total.device.type == "cpu" and not torch.isnan(total)
    total.backward()
    for p in preds:
        assert p.grad is not None and p.grad.device.type == "cpu"
    ref_p = [p.detach().clone().requires_grad_(True) for p in preds]
    ref = R.multiscale_loss(ref_p, tgts, ANCH, 1)
    ref[0].backward()
    for a, b in zip((total, bbox, obj, cls), ref):
        close(a, float(b.detach() if hasattr(b, "detach") else b), atol=1e-7)
    for p, q in zip(preds, ref_p):
        grad_close(p.grad, q.grad)


def test_loss_weight_identity_and_no_grad(yb):
    # reference tests/test_loss.py:111-129
    pred = torch.randn(2, 20, 20, 3, 6).cuda()
    tgt = torch.zeros(2, 20, 20, 3, 6)
    tgt[0, 10, 10, 0, :5] = torch.tensor([0.5, 0.5, 0.2, 0.3, 1.0])
    tgt[0, 10, 10, 0, 5] = 1.0
    with torch.no_grad():
        total, bbox, obj, cls = yb.yolo_loss(pred, tgt.cuda(), ANCH[0], 1)
    assert torch.allclose(total, 0.05 * bbox + 1.0 * obj + 0.5 * cls, atol=1e-5)
    assert not total.requires_grad


def test_loss_upstream_gradients(yb):
    """Non-unit upstream gradient on total, and gradients arriving on the other three outputs."""
    g = torch.Generator().manual_seed(9)
    heads = [torch.randn(2, G, G, 3, 7, generator=g) for G in (8, 4, 2)]
    tg = []
    for h in heads:
        t = torch.zeros_like(h)
        t[0, 1, 1, 1, :5] = torch.tensor([0.3, 0.3, 0.2, 0.25, 1.0])
        t[0, 1, 1, 1, 6] = 1.0
        tg.append(t)
    for combo in ((3.0, 0, 0, 0), (1.0, 0.5, 2.0, -1.0)):
        preds = [h.clone().cuda().requires_grad_(True) for h in heads]
        res = yb.yolo_loss_multiscale(preds, [t.cuda() for t in tg], ANCH, 2)
        sum(c * r for c, r in zip(combo, res) if c != 0).backward()
        ref_p = [h.clone().requires_grad_(True) for h in heads]
        ref = R.multiscale_loss(ref_p, tg, ANCH, 2)
        sum(c * r for c, r in zip(combo, ref) if c != 0).backward()
        for p, q in zip(preds, ref_p):
            grad_close(p.grad, q.grad)


def test_loss_full_size_vs_oracle(yb):
    """BASELINE configs[1] shape (nc=1, 640x640) at B=8; every scale dense with positives."""
    g = torch.Generator().manual_seed(1234)
    B, nc = 8, 1
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (80, 40, 20)]
    rng = np.random.default_rng(4321)
    labels = []
    for _ in range(B):
        n = int(rng.integers(0, 51))
        lab = np.zeros((n, 5))
        lab[:, 1:3] = rng.uniform(0.05, 0.95, (n, 2))
        lab[:, 3:5] = np.exp(rng.uniform(np.log(0.01), np.log(0.6), (n, 2)))
        labels.append(lab)
    tg = yb.build_targets(labels, ANCH, [80, 40, 20], nc, 640)
    preds = [h.cuda().requires_grad_(True) for h in heads]
    res = yb.yolo_loss_multiscale(preds, tg, ANCH, nc)
    res[0].backward()
    ref_p = [h.clone().requires_grad_(True) for h in heads]
    ref = R.multiscale_loss(ref_p, [t.cpu() for t in tg], ANCH, nc)
    ref[0].backward()
    for a, b in zip(res, ref):
        close(a, float(b.detach() if hasattr(b, "detach") else b), atol=1e-7)
    for p, q in zip(preds, ref_p):
        grad_close(p.grad, q.grad)


def test_loss_two_rank_emulation_on_one_gpu(yb):
    """SURVEY 8e on one GPU: two image shards, partial sums added as the all-reduce would, each
    shard finalised with the global sums -> same losses and the same gradient rows as the
    single-rank run over the whole batch."""
    from yolo_from_scratch_b200 import ops
    g = torch.Generator().manual_seed(21)
    B, nc = 6, 2
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g).cuda() for G in (16, 8, 4)]
    rng = np.random.default_rng(5)
    labels = []
    for _ in range(B):
        n = int(rng.integers(0, 9))
        lab = np.zeros((n, 5))
        lab[:, 0] = rng.integers(0, nc, n)
        lab[:, 1:3] = rng.uniform(0.1, 0.9, (n, 2))
        lab[:, 3:5] = rng.uniform(0.05, 0.6, (n, 2))
        labels.append(lab)
    tg = yb.build_targets(labels, ANCH, [16, 8, 4], nc, 128)
    anc = [a.cuda() for a in ANCH]
    w = ops.MULTISCALE_OBJ_WEIGHTS
    full4, _, full_g = ops.loss_forward_backward(heads, tg, anc, nc, w, [True] * 3)
    shards = [(0, 4), (4, 6)]  # unequal on purpose
    cut = lambda ts, lo, hi: [t[lo:hi].contiguous() for t in ts]
    parts = []
    for lo, hi in shards:  # pass 1: every rank's partial sums
        ops.loss_forward_backward(cut(heads, lo, hi), cut(tg, lo, hi), anc, nc, w, [True] * 3, b_global=B,
                                  reduce_fn=lambda p: (parts.append(p.clone()), p)[1])
    total = parts[0] + parts[1]
    for lo, hi in shards:  # pass 2: finalise with the reduced sums
        out4, _, grads = ops.loss_forward_backward(cut(heads, lo, hi), cut(tg, lo, hi), anc, nc, w, [True] * 3,
                                                   b_global=B, reduce_fn=lambda p: total.clone())
        close(out4, full4, rtol=2e-6, atol=1e-7)
        for s in range(3):
            close(grads[s], full_g[s][lo:hi], rtol=1e-5, atol=1e-9)


# ---- sparse-target loss (SURVEY 8f-4) ------------------------------------------------------------
def _random_labels(rng, B, nc, max_n, lo=0.05, hi=0.95):
    labels = []
    for _ in range(B):
        n = int(rng.integers(0, max_n + 1))
        lab = np.zeros((n, 5))
        lab[:, 0] = rng.integers(0, max(nc, 1), n)
        lab[:, 1:3] = rng.uniform(lo, hi, (n, 2))
        lab[:, 3:5] = np.exp(rng.uniform(np.log(0.01), np.log(0.6), (n, 2)))
        labels.append(lab)
    return labels


@pytest.mark.parametrize("B,nc,grids,img,max_n", [(8, 1, (80, 40, 20), 640, 50), (4, 3, (16, 8, 4), 128, 12),
                                                    (3, 80, (20, 10, 5), 160, 30), (2, 1, (13, 6, 3), 104, 0)])
def test_sparse_label_loss_equals_dense_and_oracle(yb, B, nc, grids, img, max_n):
    """yolo_loss_multiscale_labels (device-side assignment, sparse targets) == the dense call on
    yb.build_targets' tensors == the oracle on the oracle's own assignment, values and gradients.
    Duplicate cells (first ground truth wins) are forced by repeating labels."""
    g = torch.Generator().manual_seed(100 + B + nc)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in grids]
    rng = np.random.default_rng(B * 7 + nc)
    labels = _random_labels(rng, B, nc, max_n)
    if max_n:
        labels[0] = np.concatenate([labels[0], labels[0][:3] * np.array([1, 1, 1, 1.0001, 0.9999])])  # same cells
    sp = [h.cuda().requires_grad_(True) for h in heads]
    res_s = yb.yolo_loss_multiscale_labels(sp, labels, ANCH, nc, img)
    res_s[0].backward()
    tg = yb.build_targets(labels, ANCH, list(grids), nc, img)
    dp = [h.cuda().requires_grad_(True) for h in heads]
    res_d = yb.yolo_loss_multiscale(dp, tg, ANCH, nc)
    res_d[0].backward()
    for a, b in zip(res_s, res_d):
        close(a, b, rtol=1e-6, atol=1e-7)
    for p, q in zip(sp, dp):
        close(p.grad, q.grad, rtol=1e-6, atol=1e-10)
    ref_t = [R.assign_targets(l, ANCH, list(grids), nc, img) for l in labels]
    ref_tg = [torch.from_numpy(np.stack([t[s] for t in ref_t])) for s in range(3)]
    ref_p = [h.clone().requires_grad_(True) for h in heads]
    ref = R.multiscale_loss(ref_p, ref_tg, ANCH, nc)
    ref[0].backward()
    for a, b in zip(res_s, ref):
        close(a, float(b), atol=1e-7)
    for p, q in zip(sp, ref_p):
        grad_close(p.grad, q.grad)


def test_sparse_label_loss_packed_letterbox_and_errors(yb):
    """PackedLabels input with a real letterbox; a label outside the grid is reported like the
    reference's IndexError; no_grad and upstream-gradient paths work."""
    from yolo_from_scratch_b200 import ops
    nc, img, grids, B = 2, 256, (32, 16, 8), 3
    g = torch.Generator().manual_seed(9)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in grids]
    labels = _random_labels(np.random.default_rng(3), B, nc, 9, 0.2, 0.8)
    lb = [(500.0, 375.0, 0.512, 32.0, 0.0), (256.0, 256.0, 1.0, 0.0, 0.0), (300.0, 600.0, 256 / 600, 0.0, 64.0)]
    packed = ops.pack_labels(labels, img, lb)
    sp = [h.cuda().requires_grad_(True) for h in heads]
    res = yb.yolo_loss_multiscale_labels(sp, packed, ANCH, nc, img)
    (res[0] * 3.0).backward()
    packed.check()
    tg = yb.build_targets(labels, ANCH, list(grids), nc, img, letterbox=lb)
    dp = [h.cuda().requires_grad_(True) for h in heads]
    res_d = yb.yolo_loss_multiscale(dp, tg, ANCH, nc)
    (res_d[0] * 3.0).backward()
    for a, b in zip(res, res_d):
        close(a, b, rtol=1e-6, atol=1e-7)
    for p, q in zip(sp, dp):
        close(p.grad, q.grad, rtol=1e-6, atol=1e-10)
    with torch.no_grad():
        res_n = yb.yolo_loss_multiscale_labels([h.cuda() for h in heads], packed, ANCH, nc, img)
    close(res_n[0], res[0], rtol=1e-6, atol=1e-7)
    bad = [np.array([[0, -1.5, 0.5, 0.1, 0.1]])] + labels[1:]  # int(-1.5*G) < -G: IndexError in the reference
    pk = ops.pack_labels(bad, img)
    yb.yolo_loss_multiscale_labels([h.cuda() for h in heads], pk, ANCH, nc, img)
    with pytest.raises(IndexError):
        pk.check()


# ---- NCHW head layout (SURVEY 8f-2) -----------------------------------------------------------------
@pytest.mark.parametrize("B,nc,grids,img", [(4, 1, (80, 40, 20), 640), (2, 80, (20, 10, 5), 160), (3, 3, (13, 7, 5), 104)])
def test_nchw_heads_give_identical_results(yb, B, nc, grids, img):
    """The *_nchw entry points read the head convs' own output (B, A*(5+nc), H, W): loss values equal
    the reference-layout call, gradients equal its gradients permuted back, candidates / keep sets are
    identical, for dense targets and for label lists.  (13,7,5) exercises H*W not divisible by 4."""
    g = torch.Generator().manual_seed(31 + nc)
    raw = [torch.randn(B, 3 * (5 + nc), G, G, generator=g).cuda() for G in grids]
    heads = [yb.heads_from_nchw(r) for r in raw]
    labels = _random_labels(np.random.default_rng(nc + 2), B, nc, 30)
    tg = yb.build_targets(labels, ANCH, list(grids), nc, img)
    to_nchw = lambda t: t.permute(0, 3, 4, 1, 2).reshape(t.shape[0], -1, t.shape[1], t.shape[2])
    rp = [h.clone().requires_grad_(True) for h in heads]
    ref = yb.yolo_loss_multiscale(rp, tg, ANCH, nc)
    ref[0].backward()
    for targets in (tg, labels):
        xp = [r.clone().requires_grad_(True) for r in raw]
        out = yb.yolo_loss_multiscale_nchw(xp, targets, ANCH, nc, img)
        out[0].backward()
        for a, b in zip(out, ref):
            close(a, b, rtol=1e-6, atol=1e-7)
        for x, r in zip(xp, rp):
            close(x.grad, to_nchw(r.grad), rtol=1e-6, atol=1e-10)
    for conf in (0.5, 0.001):
        d0 = yb.detect_batch(heads, ANCH, img, nc, conf, 0.4)
        d1 = yb.detect_batch_nchw(raw, ANCH, img, nc, conf, 0.4)
        assert torch.equal(d0["counts"], d1["counts"]) and torch.equal(d0["n_keep"], d1["n_keep"])
        for b in range(B):
            m, k = int(d0["counts"][b]), int(d0["n_keep"][b])
            assert torch.equal(d0["boxes"][b, :m], d1["boxes"][b, :m])
            assert torch.equal(d0["scores"][b, :m], d1["scores"][b, :m])
            assert torch.equal(d0["classes"][b, :m], d1["classes"][b, :m])
            assert torch.equal(d0["keep"][b, :k], d1["keep"][b, :k])


@pytest.mark.parametrize("B,nc,grids,img", [(2, 1, (40, 20, 10), 320), (2, 80, (20, 10, 5), 160), (3, 3, (13, 7, 5), 104)])
def test_nchw_heads_against_the_oracle(yb, B, nc, grids, img):
    """f-2 against the oracle itself (not against the BHWAC CUDA path): losses, gradients (permuted to NCHW),
    candidates and keep sets of the *_nchw entry points equal the CPU restatement of the reference, for dense
    targets, label lists and PackedLabels."""
    from yolo_from_scratch_b200 import ops
    g = torch.Generator().manual_seed(41 + nc)
    raw = [torch.randn(B, 3 * (5 + nc), G, G, generator=g) for G in grids]
    heads = [r.view(B, 3, 5 + nc, G, G).permute(0, 3, 4, 1, 2).contiguous() for r, G in zip(raw, grids)]  # train.py:608-609
    labels = _random_labels(np.random.default_rng(nc + 5), B, nc, 20)
    tg = [torch.from_numpy(np.stack([R.assign_targets(l, ANCH, list(grids), nc, img)[s] for l in labels])) for s in range(3)]
    cp = [h.clone().requires_grad_(True) for h in heads]
    ref = R.multiscale_loss(cp, tg, ANCH, nc)
    ref[0].backward()
    to_nchw = lambda t: t.permute(0, 3, 4, 1, 2).reshape(t.shape[0], -1, t.shape[1], t.shape[2])
    for targets in ([t.cuda() for t in tg], labels, ops.pack_labels(labels, img)):
        xp = [r.clone().cuda().requires_grad_(True) for r in raw]
        out = yb.yolo_loss_multiscale_nchw(xp, targets, ANCH, nc, img)
        out[0].backward()
        for a, b in zip(out, ref):
            close(a, b, rtol=RTOL, atol=1e-7)
        for x, c in zip(xp, cp):
            grad_close(x.grad, to_nchw(c.grad))
    for conf in (0.5, 0.05):
        det = yb.detect_batch_nchw([r.cuda() for r in raw], ANCH, img, nc, conf, 0.4)
        counts, n_keep = det["counts"].cpu(), det["n_keep"].cpu()
        for b in range(B):
            rb, rs, rc = R.candidates([h[b:b + 1] for h in heads], ANCH, img, nc, conf)
            m = int(counts[b])
            bx, sc, cl = (det[k][b, :m].cpu().numpy() for k in ("boxes", "scores", "classes"))
            assert m == rb.shape[0] and np.array_equal(cl, rc.numpy())
            assert np.allclose(bx, rb.numpy(), rtol=1e-5, atol=1e-4) and np.allclose(sc, rs.numpy(), rtol=1e-5, atol=1e-7)
            want = R.batched_nms_indices(bx, sc, cl, 0.4, arith="cuda", device_rule="cuda")
            assert np.array_equal(det["keep"][b, :int(n_keep[b])].cpu().numpy(), want)


def test_loss_second_backward_with_retain_graph(yb):
    """ADVICE r1: backward twice through the same graph (retain_graph=True, which the reference loss supports)
    gives the reference's accumulated gradient, also with an upstream factor != 1."""
    B, nc, grids, img = 2, 2, (8, 4, 2), 64
    g = torch.Generator().manual_seed(9)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in grids]
    labels = _random_labels(np.random.default_rng(9), B, nc, 6)
    tg = yb.build_targets(labels, ANCH, list(grids), nc, img)
    xp = [h.clone().cuda().requires_grad_(True) for h in heads]
    out = yb.yolo_loss_multiscale(xp, tg, ANCH, nc)
    (out[0] * 3.0).backward(retain_graph=True)
    (out[0] * 3.0).backward()
    cp = [h.clone().requires_grad_(True) for h in heads]
    ref = R.multiscale_loss(cp, [t.cpu() for t in tg], ANCH, nc)
    (ref[0] * 6.0).backward()
    for x, c in zip(xp, cp):
        grad_close(x.grad, c.grad)


def test_label_list_check_flag(yb):
    """ADVICE r1: the label-list wrappers raise like the reference (IndexError) when asked to check."""
    nc, img, grids = 1, 64, (8, 4, 2)
    heads = [torch.randn(1, G, G, 3, 6).cuda() for G in grids]
    bad = [np.array([[0, -1.5, 0.5, 0.1, 0.1]])]
    with pytest.raises(IndexError):
        yb.yolo_loss_multiscale_labels(heads, bad, ANCH, nc, img, check=True)
    raw = [h.permute(0, 3, 4, 1, 2).reshape(1, -1, h.shape[1], h.shape[2]).contiguous() for h in heads]
    with pytest.raises(IndexError):
        yb.yolo_loss_multiscale_nchw(raw, bad, ANCH, nc, img, check=True)
    yb.yolo_loss_multiscale_labels(heads, [np.array([[0, .5, .5, .1, .1]])], ANCH, nc, img, check=True)


# ---- CUDA-graph step ------------------------------------------------------------------------------------
@pytest.mark.parametrize("targets,layout", [("labels", 0), ("dense", 0), ("labels", 1)])
def test_hot_path_graph_replays_equal_eager(yb, targets, layout):
    """The captured step (loss fwd+bwd + detect + pack) gives the eager results, replay after replay,
    for new inputs copied into its static buffers."""
    from yolo_from_scratch_b200 import ops
    B, nc, img, grids = 3, 2, 160, (20, 10, 5)
    hp = yb.HotPathGraph(B, img, nc, ANCH, conf_threshold=0.4, iou_threshold=0.4, max_gt=12, targets=targets,
                         layout=layout)
    for seed in (1, 2, 3):
        g = torch.Generator().manual_seed(seed)
        raw = [torch.randn(B, 3 * (5 + nc), G, G, generator=g).cuda() for G in grids]
        heads = [yb.heads_from_nchw(r) for r in raw]
        labels = _random_labels(np.random.default_rng(seed), B, nc, 12)
        lab, n_gt, lb = ops.pack_labels_host(labels, img, max_gt=12)
        for dst, src in zip(hp.heads, raw if layout else heads):
            dst.copy_(src)
        tg = yb.build_targets(labels, ANCH, list(grids), nc, img)
        if targets == "labels":
            hp.labels.labels.copy_(lab); hp.labels.n_gt.copy_(n_gt); hp.labels.letterbox.copy_(lb)
        else:
            for dst, src in zip(hp.targets, tg):
                dst.copy_(src)
        losses, grads, det = hp.replay()
        ep = [h.clone().requires_grad_(True) for h in heads]
        ref = yb.yolo_loss_multiscale(ep, tg, ANCH, nc)
        ref[0].backward()
        close(losses, torch.stack([r.detach() for r in ref]), rtol=1e-6, atol=1e-7)
        back = (lambda t: yb.heads_from_nchw(t)) if layout else (lambda t: t)
        for gph, e in zip(grads, ep):
            close(back(gph), e.grad, rtol=1e-6, atol=1e-10)
        d0 = yb.detect_batch(heads, ANCH, img, nc, 0.4, 0.4)
        assert torch.equal(det["n_keep"], d0["n_keep"]) and torch.equal(det["counts"], d0["counts"])
        for b in range(B):
            k = int(d0["n_keep"][b])
            assert torch.equal(det["keep"][b, :k], d0["keep"][b, :k])
        rows0, off0 = yb.pack_detections(d0)
        assert torch.equal(hp.offsets, off0) and torch.equal(hp.rows[:int(off0[-1])], rows0[:int(off0[-1])])


def test_nchw_filter_sparse_empty_and_letterbox(yb):
    """NCHW filter edge cases: letterbox reverse, a threshold nothing passes, a threshold a few rows pass
    (sparse tiles), images with no candidate at all; all equal to the reference-layout kernels."""
    nc, img, grids, B = 3, 256, (32, 16, 8), 4
    g = torch.Generator().manual_seed(77)
    raw = [torch.randn(B, 3 * (5 + nc), G, G, generator=g).cuda() for G in grids]
    for r in raw:
        r[1, 4::(5 + nc)] = -20.0          # image 1: objectness off everywhere
    heads = [yb.heads_from_nchw(r) for r in raw]
    lb = [(0.5, 10.0, 0.0), (1.0, 0.0, 0.0), (0.8, 0.0, 25.6), (0.3, 3.0, 4.0)]
    for conf in (0.9999999, 0.98, 0.5):
        d0 = yb.detect_batch(heads, ANCH, img, nc, conf, 0.4, letterbox=lb)
        d1 = yb.detect_batch_nchw(raw, ANCH, img, nc, conf, 0.4, letterbox=lb)
        assert torch.equal(d0["counts"], d1["counts"]) and int(d0["counts"][1]) == 0
        assert torch.equal(d0["n_keep"], d1["n_keep"])
        for b in range(B):
            m, k = int(d0["counts"][b]), int(d0["n_keep"][b])
            assert torch.equal(d0["boxes"][b, :m], d1["boxes"][b, :m])
            assert torch.equal(d0["scores"][b, :m], d1["scores"][b, :m])
            assert torch.equal(d0["classes"][b, :m], d1["classes"][b, :m])
            assert torch.equal(d0["keep"][b, :k], d1["keep"][b, :k])
    assert int(yb.detect_batch_nchw(raw, ANCH, img, nc, 0.9999999, 0.4)["counts"].sum()) == 0


# ---- eval_epoch counting (SURVEY 8f-1) -------------------------------------------------------------
@pytest.mark.parametrize("name", ["e640", "e320"])
def test_eval_epoch_matches_reference_golden(yb, golden, name):
    """yb.eval_epoch on the preset heads/targets the UNMODIFIED reference's eval_epoch was run on
    (oracle/make_golden.py): precision/recall/F1 exact (they are ratios of integer counts), loss 1e-5."""
    g = golden("eval")
    img, nc, B, nb, conf, iou = g[f"{name}_cfg"]
    nc, nb = int(nc), int(nb)

    class Model:
        anchors = ANCH
        k = 0

        def eval(self):
            return self

        def __call__(self, imgs):
            heads = [torch.from_numpy(g[f"{name}_b{self.k}_head{s}"]) for s in range(3)]
            self.k += 1
            return heads
    loader = []
    for k in range(nb):
        tg = [torch.from_numpy(g[f"{name}_b{k}_tgt{s}"]) for s in range(3)]
        loader.append((torch.zeros(int(B), 3, 8, 8), [[tg[s][b] for s in range(3)] for b in range(int(B))]))
    res = yb.eval_epoch(Model(), loader, torch.device("cpu"), num_classes=nc, iou_threshold=float(iou),
                        conf_threshold=float(conf))
    want = g[f"{name}_result"]
    close(res[0], want[0])
    assert tuple(res[1:]) == tuple(want[1:])


@pytest.mark.parametrize("nc,B,grids,conf,iou", [(1, 4, (80, 40, 20), 0.5, 0.5), (80, 2, (20, 10, 5), 0.25, 0.3),
                                                  (3, 3, (13, 7, 5), 0.5, 0.0)])
def test_eval_counts_vs_oracle(yb, nc, B, grids, conf, iou):
    """Counts are integers: exact against the oracle, on heads steered towards their targets so that
    all three counters and both sides of the IoU threshold are populated."""
    g = torch.Generator().manual_seed(5 + nc)
    rng = np.random.default_rng(nc)
    img = grids[0] * 8
    labels = _random_labels(rng, B, nc, 40)
    tg = [t.cpu() for t in yb.build_targets(labels, ANCH, list(grids), nc, img)]
    heads = [torch.randn(t.shape, generator=g) for t in tg]
    for s, t in enumerate(tg):  # copy decoded-target-ish logits into half of the positive rows
        pos = (t[..., 4] > 0.5).nonzero()
        for b, gy, gx, a in pos.tolist()[::2]:
            G = t.shape[1]
            xc, yc, w, h = [float(v) for v in t[b, gy, gx, a, 0:4]]
            sx = min(max((xc * G - gx + 0.5) / 2, 0.02), 0.98)
            sy = min(max((yc * G - gy + 0.5) / 2, 0.02), 0.98)
            sw = min(max(np.sqrt(w * rng.uniform(0.6, 1.6) * 640.0 / float(ANCH[s][a, 0])) / 2, 0.02), 0.98)
            sh = min(max(np.sqrt(h * rng.uniform(0.6, 1.6) * 640.0 / float(ANCH[s][a, 1])) / 2, 0.02), 0.98)
            lg = lambda p: float(np.log(p / (1 - p)))
            heads[s][b, gy, gx, a, 0:4] = torch.tensor([lg(sx), lg(sy), lg(sw), lg(sh)])
            heads[s][b, gy, gx, a, 4] = 2.0
    want = R.eval_counts(heads, tg, ANCH, conf, iou)
    got = yb.eval_counts([h.cuda() for h in heads], [t.cuda() for t in tg], ANCH, conf, iou)
    assert tuple(int(v) for v in got.cpu()) == tuple(want)
    assert min(want) > 0 or iou == 0.0
    again = yb.eval_counts(heads, tg, ANCH, conf, iou, out=got)          # CPU tensors staged; accumulates
    assert tuple(int(v) for v in again.cpu()) == tuple(2 * w for w in want)


# ---- target assignment ------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["a", "b", "c", "d", "e", "f", "g"])
def test_build_targets_golden_bitexact(yb, golden, name):
    g = golden("targets")
    img, nc = (int(v) for v in g[f"{name}_cfg"])
    grids = [img // 8, img // 16, img // 32]
    anchors = [ANCH[0]] * 3 if name == "g" else ANCH
    # batch of 3: the golden image, an empty image, the golden image again
    out = yb.build_targets([g[f"{name}_labels"], np.zeros((0, 5)), g[f"{name}_labels"]], anchors, grids, nc, img,
                           letterbox=[g[f"{name}_letterbox"], [img, img, 1.0, 0, 0], g[f"{name}_letterbox"]])
    for s in range(3):
        ref = np.zeros((grids[s], grids[s], 3, 5 + nc), dtype=np.float32)
        idx = g[f"{name}_s{s}_idx"]
        if len(idx):
            ref[idx[:, 0], idx[:, 1], idx[:, 2]] = g[f"{name}_s{s}_rows"]
        got = out[s].cpu().numpy()
        assert np.array_equal(got[0], ref) and np.array_equal(got[2], ref)
        assert not got[1].any()


def test_anchor_iou_golden(yb, golden):
    g = golden("targets")
    for s in range(3):
        got = yb.compute_anchor_iou(T(g["aiou_wh"]), ANCH[s])
        assert np.array_equal(got.numpy(), g["aiou"][:, s])
    one = yb.compute_anchor_iou(torch.tensor([50.0, 60.0]), ANCH[0])  # reference tests/test_dataset.py:85-96
    assert one.shape == (3,) and (one >= 0).all() and (one <= 1).all() and one[2] > one[0]


def test_build_targets_random_vs_oracle(yb):
    rng = np.random.default_rng(12)
    for img, nc in ((640, 1), (416, 5), (1280, 80)):
        grids = [img // 8, img // 16, img // 32]
        labels, lbs = [], []
        for _ in range(6):
            n = int(rng.integers(0, 60))
            lab = np.zeros((n, 5))
            lab[:, 0] = rng.integers(0, nc, n)
            lab[:, 1:3] = rng.uniform(0.0, 1.0, (n, 2))
            lab[:, 3:5] = np.exp(rng.uniform(np.log(0.005), np.log(0.9), (n, 2)))
            labels.append(lab)
            ow, oh = int(rng.integers(200, 2000)), int(rng.integers(200, 2000))
            sc = min(img / ow, img / oh)
            nw, nh = int(ow * sc), int(oh * sc)
            lbs.append((ow, oh, sc, (img - nh) // 2, (img - nw) // 2))
        out = yb.build_targets(labels, ANCH, grids, nc, img, letterbox=lbs)
        for b in range(6):
            ref = R.assign_targets(labels[b], ANCH, grids, nc, img, lbs[b])
            for s in range(3):
                assert np.array_equal(out[s][b].cpu().numpy(), ref[s])


# ---- candidate filter -------------------------------------------------------------------------
@pytest.mark.parametrize("nc,conf", [(1, 0.5), (1, 0.001), (3, 0.25), (80, 0.25), (80, 0.001)])
def test_filter_vs_oracle(yb, nc, conf):
    g = torch.Generator().manual_seed(100 + nc)
    B, img = 3, 256
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (32, 16, 8)]
    lb = [(0.8, 10, 0), (1.0, 0, 0), (0.5, 0, 33)]
    boxes, scores, classes, counts = yb.filter_candidates([h.cuda() for h in heads], ANCH, img, nc, conf, letterbox=lb)
    for b in range(B):
        rb, rs, rc = R.candidates([h[b:b + 1] for h in heads], ANCH, img, nc, conf, lb[b][0], lb[b][1], lb[b][2])
        m = int(counts[b])
        assert m == rb.shape[0]
        assert np.array_equal(classes[b, :m].cpu().numpy(), rc.numpy())
        close(boxes[b, :m], rb, atol=2e-4)   # pixel coordinates: 1e-5 relative of ~100 px
        close(scores[b, :m], rs, atol=1e-8)


# ---- NMS --------------------------------------------------------------------------------------
def rand_boxes(n, seed, span=300.0, neg=0.0, wmax=80.0):
    g = torch.Generator().manual_seed(seed)
    xy = torch.rand(n, 2, generator=g) * span - neg
    wh = torch.rand(n, 2, generator=g) * wmax + 1.0
    return torch.cat([xy, xy + wh], dim=1), torch.rand(n, generator=g)


ALGOS = [0, 1]  # YB_NMS_GRAPH (sparse graph, default), YB_NMS_BITMASK (dense bitmask)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000, 5000])
@pytest.mark.parametrize("thr", [0.4, 0.0, 0.7, 1.0, -0.5])
def test_nms_vs_oracle_and_torchvision(yb, n, thr, algo):
    import torchvision
    boxes, scores = rand_boxes(n, n)
    got = yb.nms(boxes.cuda(), scores.cuda(), thr, algo=algo).cpu().numpy()
    assert np.array_equal(got, R.nms_indices(boxes.numpy(), scores.numpy(), thr, "cuda"))
    assert np.array_equal(got, torchvision.ops.nms(boxes.cuda(), scores.cuda(), thr).cpu().numpy())


@pytest.mark.parametrize("algo", ALGOS)
def test_nms_ties_degenerate_and_nan(yb, algo):
    import torchvision
    boxes, scores = rand_boxes(700, 5)
    scores[::5] = 0.5          # ties: lower index wins
    scores[3] = float("nan")   # NaN sorts first
    boxes[10] = torch.tensor([5.0, 5.0, 5.0, 5.0])      # zero area
    boxes[11] = torch.tensor([5.0, 5.0, 5.0, 5.0])      # identical zero-area pair: 0/0
    boxes[12] = torch.tensor([50.0, 50.0, 20.0, 90.0])  # negative width
    boxes[13] = torch.tensor([float("nan"), 0.0, 10.0, 10.0])
    got = yb.nms(boxes.cuda(), scores.cuda(), 0.4, algo=algo).cpu().numpy()
    assert np.array_equal(got, torchvision.ops.nms(boxes.cuda(), scores.cuda(), 0.4).cpu().numpy())
    assert np.array_equal(got, R.nms_indices(boxes.numpy(), scores.numpy(), 0.4, "cuda"))
    assert yb.nms(torch.zeros(0, 4).cuda(), torch.zeros(0).cuda(), 0.5, algo=algo).numel() == 0


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("n,nc,neg", [(800, 4, 0.0), (800, 4, 200.0), (24000, 80, 100.0), (26000, 80, 100.0), (26000, 1, 0.0),
                                      (30000, 3, 50.0)])  # 30000 > 26,880: the graph NMS sorts with the ballot kernel
def test_batched_nms_both_regimes(yb, n, nc, neg, algo):
    """n <= 25000 uses torchvision's coordinate trick (incl. its negative-coordinate cross-class
    quirk), larger n its per-class loop (boxes.py:80)."""
    import torchvision
    boxes, scores = rand_boxes(n, n + nc, span=600.0, neg=neg, wmax=120.0)
    idxs = torch.randint(0, nc, (n,), generator=torch.Generator().manual_seed(1))
    got = yb.batched_nms(boxes.cuda(), scores.cuda(), idxs.cuda(), 0.4, algo=algo).cpu().numpy()
    ref = torchvision.ops.batched_nms(boxes.cuda(), scores.cuda(), idxs.cuda(), 0.4).cpu().numpy()
    assert np.array_equal(np.sort(got), np.sort(ref))
    assert np.array_equal(scores.numpy()[got], scores.numpy()[ref])
    want = R.batched_nms_indices(boxes.numpy(), scores.numpy(), idxs.numpy(), 0.4, "cuda", "cuda")
    assert np.array_equal(got, want)


def test_batched_nms_cpu_caller_uses_cpu_dispatch_rule(yb):
    boxes, scores = rand_boxes(1500, 77, neg=150.0)
    idxs = torch.randint(0, 3, (1500,), generator=torch.Generator().manual_seed(2))
    got = yb.batched_nms(boxes, scores, idxs, 0.4)
    assert got.device.type == "cpu" and got.dtype == torch.int64
    want = R.batched_nms_indices(boxes.numpy(), scores.numpy(), idxs.numpy(), 0.4, "cuda", "cpu")
    assert np.array_equal(got.numpy(), want)


def test_nms_reference_known_answers(yb):
    # reference tests/test_inference.py:16-76 through the tensor API
    def run(dets, thr):
        if not dets:
            return []
        a = torch.tensor(dets, dtype=torch.float32)
        return [dets[i] for i in yb.nms(a[:, :4], a[:, 4], thr).tolist()]
    d = [(10, 10, 50, 50, 0.9, 0), (12, 12, 52, 52, 0.8, 0), (100, 100, 150, 150, 0.85, 0)]
    assert run(d, 0.5) == [d[0], d[2]]
    d = [(10, 10, 50, 50, 0.6, 0), (12, 12, 52, 52, 0.9, 0)]
    assert run(d, 0.5) == [d[1]]
    d = [(10, 10, 50, 50, 0.9, 0), (20, 20, 60, 60, 0.8, 0)]
    assert len(run(d, 0.3)) == 1 and len(run(d, 0.7)) == 2


@pytest.mark.parametrize("algo", ALGOS)
def test_batched_nms_padded_varied_counts(yb, algo):
    B, cap = 5, 3000
    boxes = torch.zeros(B, cap, 4)
    scores = torch.zeros(B, cap)
    classes = torch.zeros(B, cap, dtype=torch.int64)
    counts = [0, 1, 64, 1999, 3000]
    for b, m in enumerate(counts):
        bx, sc = rand_boxes(max(m, 1), 40 + b)
        boxes[b, :m], scores[b, :m] = bx[:m], sc[:m]
        classes[b, :m] = torch.randint(0, 3, (m,), generator=torch.Generator().manual_seed(b))
    keep, n_keep = yb.batched_nms_padded(boxes.cuda(), scores.cuda(), classes.cuda(),
                                         torch.tensor(counts, dtype=torch.int32).cuda(), 0.4, algo=algo)
    for b, m in enumerate(counts):
        want = R.batched_nms_indices(boxes[b, :m].numpy(), scores[b, :m].numpy(), classes[b, :m].numpy(), 0.4)
        assert int(n_keep[b]) == len(want)
        assert np.array_equal(keep[b, :len(want)].cpu().numpy(), want)


def clustered_boxes(n, seed, n_clusters=40):
    """Detector-like input: tight clusters of heavily overlapping boxes (long suppression chains)."""
    g = torch.Generator().manual_seed(seed)
    centres = torch.rand(n_clusters, 2, generator=g) * 500 + 50
    sizes = torch.rand(n_clusters, 2, generator=g) * 120 + 20
    which = torch.randint(0, n_clusters, (n,), generator=g)
    c = centres[which] + torch.randn(n, 2, generator=g) * 6
    wh = sizes[which] * (1 + torch.randn(n, 2, generator=g) * 0.08).clamp(0.5, 1.5)
    return torch.cat([c - wh / 2, c + wh / 2], dim=1), torch.rand(n, generator=g)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("n", [500, 6000])
def test_nms_clustered_detections(yb, n, algo):
    import torchvision
    boxes, scores = clustered_boxes(n, n)
    got = yb.nms(boxes.cuda(), scores.cuda(), 0.45, algo=algo).cpu().numpy()
    assert np.array_equal(got, torchvision.ops.nms(boxes.cuda(), scores.cuda(), 0.45).cpu().numpy())
    assert np.array_equal(got, R.nms_indices(boxes.numpy(), scores.numpy(), 0.45, "cuda"))


def test_nms_graph_overflow_resolved_on_device(yb):
    """3000 identical boxes: 4.5M edges do not fit the default edge list.  The graph algorithm resolves
    the image inside the same launch (blocked greedy pass): no n_keep = -1, no host round trip."""
    n = 3000
    boxes = torch.tensor([[10.0, 10.0, 50.0, 60.0]]).repeat(n, 1)
    scores = torch.rand(n, generator=torch.Generator().manual_seed(3))
    keep, n_keep = yb.batched_nms_padded(boxes.cuda().unsqueeze(0), scores.cuda().unsqueeze(0), None, None, 0.5)
    want = R.nms_indices(boxes.numpy(), scores.numpy(), 0.5, "cuda")
    assert int(n_keep[0]) == 1 == len(want)
    assert np.array_equal(keep[0, :1].cpu().numpy(), want)
    assert np.array_equal(yb.nms(boxes.cuda(), scores.cuda(), 0.5).cpu().numpy(), want)


def _clusters(n_clusters, per, n_cls, seed, span=600.0, neg=False):
    """A trained detector at a low confidence threshold: tight clusters of jittered boxes around objects."""
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(n_clusters, 2, generator=g) * span - (200.0 if neg else 0.0)
    wh = torch.rand(n_clusters, 2, generator=g) * 120.0 + 20.0
    cc = c[:, None, :] + torch.randn(n_clusters, per, 2, generator=g) * 4.0
    ww = wh[:, None, :] * (1.0 + 0.15 * torch.randn(n_clusters, per, 2, generator=g)).clamp(0.3, 2.0)
    boxes = torch.cat([cc - ww / 2, cc + ww / 2], dim=2).reshape(-1, 4)
    cls = torch.randint(0, n_cls, (n_clusters, 1), generator=g).repeat(1, per)
    flip = torch.rand(n_clusters, per, generator=g) < 0.2
    cls = torch.where(flip, torch.randint(0, n_cls, (n_clusters, per), generator=g), cls).reshape(-1)
    scores = torch.rand(boxes.shape[0], generator=g)
    scores[::11] = scores[0]
    return boxes, scores, cls


@pytest.mark.parametrize("mode,n_cls", [("plain", 1), ("trick", 7), ("class", 7), ("trick_neg", 5), ("bigcls", 3000)])
def test_nms_greedy_fallback_is_exact(yb, monkeypatch, mode, n_cls):
    """Force the on-device fallback (edge list of 1 edge per box on clustered boxes; class ids >= 512) and
    compare with torchvision's CUDA kernels and the C oracle, in every batched_nms regime."""
    import torchvision
    from yolo_from_scratch_b200 import ops
    if mode != "bigcls":
        monkeypatch.setattr(ops, "GRAPH_EDGES_PER_BOX", 1)
    B = 3
    cases = [_clusters(50, 90 + 10 * b, n_cls, 100 + b, neg=(mode == "trick_neg")) for b in range(B)]
    cap = max(c[0].shape[0] for c in cases)
    boxes = torch.zeros(B, cap, 4); scores = torch.zeros(B, cap); classes = torch.zeros(B, cap, dtype=torch.int64)
    counts = torch.zeros(B, dtype=torch.int32)
    for b, (bx, sc, cl) in enumerate(cases):
        m = bx.shape[0]
        boxes[b, :m], scores[b, :m], classes[b, :m], counts[b] = bx, sc, cl, m
    trick = -1 if mode == "class" else (1 << 40)
    cls_arg = None if mode == "plain" else classes.cuda()
    keep, n_keep, ws = yb.batched_nms_padded(boxes.cuda(), scores.cuda(), cls_arg, counts.cuda(), 0.4, trick,
                                             return_workspace=True)
    for b, (bx, sc, cl) in enumerate(cases):
        got = keep[b, :int(n_keep[b])].cpu().numpy()
        if mode == "plain":
            want_tv = torchvision.ops.nms(bx.cuda(), sc.cuda(), 0.4).cpu().numpy()
            want = R.nms_indices(bx.numpy(), sc.numpy(), 0.4, "cuda")
        elif mode == "class":
            want_tv = torchvision.ops.boxes._batched_nms_vanilla(bx.cuda(), sc.cuda(), cl.cuda(), 0.4).cpu().numpy()
            want = None
        else:
            want_tv = torchvision.ops.boxes._batched_nms_coordinate_trick(bx.cuda(), sc.cuda(), cl.cuda(), 0.4).cpu().numpy()
            want = None
        assert int(n_keep[b]) >= 0
        assert np.array_equal(got, want_tv), (mode, b, len(got), len(want_tv))
        if want is not None:
            assert np.array_equal(got, want)
    if mode != "bigcls":   # the edge list really overflowed: more edges than its capacity of 1 per box
        ev, ed = ctypes_stats(yb, ws, B, cap)
        assert ed > B * cap


def ctypes_stats(yb, ws, B, cap):
    import ctypes
    ev, ed, ca = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
    yb._lib.check(yb._lib.lib().yb_nms_graph_stats(ws.data_ptr(), ws.numel(), B, cap, ctypes.byref(ev), ctypes.byref(ed),
                                                   ctypes.byref(ca), torch.cuda.current_stream().cuda_stream), "stats")
    return int(ev.value), int(ed.value)


def test_hot_path_graph_with_overflowing_images(yb):
    """VERDICT r1 item 8: on the CUDA-graph path an image whose suppression graph overflows the edge list must
    come back with the oracle's keep set, not with zero detections.  Heads with huge, heavily overlapping boxes
    (tw = th = +6: 4x the anchor) and every row above the confidence threshold."""
    from yolo_from_scratch_b200 import ops
    B, nc, img, grids = 3, 1, 160, (20, 10, 5)
    hp = yb.HotPathGraph(B, img, nc, ANCH, conf_threshold=0.3, iou_threshold=0.4, max_gt=4, targets="labels")
    g = torch.Generator().manual_seed(5)
    heads = [torch.randn(B, G, G, 3, 6, generator=g) for G in grids]
    for h in heads:
        h[0, ..., 2:4] = 6.0      # image 0: every box 4x its anchor -> dense graph
        h[0, ..., 4] = 3.0
        h[2, ..., 2:4] = 5.0
        h[2, ..., 4] = 2.0
    for dst, src in zip(hp.heads, heads):
        dst.copy_(src.cuda())
    for _ in range(2):
        _, _, det = hp.replay()
    torch.cuda.synchronize()
    counts, n_keep = det["counts"].cpu(), det["n_keep"].cpu()
    ev, ed = ctypes_stats(yb, det["nms_ws"], B, det["boxes"].shape[1])
    assert ed > ops.GRAPH_EDGES_PER_BOX * int(counts[0])        # image 0 alone overflows its edge list
    off = hp.offsets.cpu()
    assert int(off[-1]) == int(n_keep.sum()) and (n_keep > 0).all()
    for b in range(B):
        m = int(counts[b])
        bx, sc, cl = (det[k][b, :m].cpu().numpy() for k in ("boxes", "scores", "classes"))
        want = R.batched_nms_indices(bx, sc, cl, 0.4, arith="cuda", device_rule="cuda")
        assert np.array_equal(det["keep"][b, :int(n_keep[b])].cpu().numpy(), want), b


def test_pack_reports_a_failed_image(yb):
    """pack_detections never turns n_keep = -1 into "no detections": the total becomes -1 and
    detections_to_lists raises.  (Only the bitmask algorithm with an undersized workspace can produce -1.)"""
    det = yb.detect_batch([torch.randn(2, G, G, 3, 6).cuda() for G in (8, 4, 2)], ANCH, 64, 1, 0.3, 0.4)
    det["n_keep"][1] = -1
    rows, offsets = yb.pack_detections(det)
    assert int(offsets[-1]) == -1
    with pytest.raises(RuntimeError):
        yb.detections_to_lists(det)


# ---- end to end: the reference's predict() goldens ----------------------------------------------
def canon(dets):
    a = np.array(dets, dtype=np.float64).reshape(-1, 6)
    return a[np.lexsort((a[:, 3], a[:, 2], a[:, 1], a[:, 0], -a[:, 4]))]


@pytest.mark.parametrize("name", ["p_nc1", "p_nc3", "p_nc80", "p_nc1_dense"])
def test_detect_matches_reference_predict(yb, golden, name):
    g = golden("predict")
    img, nc, conf, iou, scale, pt, pl = g[f"{name}_cfg"]
    heads = [T(g[f"{name}_head{s}"]).cuda() for s in range(3)]
    det = yb.detect_batch(heads, ANCH, int(img), int(nc), float(conf), float(iou), letterbox=[(scale, pt, pl)],
                          trick_max_numel=4000)  # the golden ran on CPU tensors (boxes.py:80)
    dets = yb.detections_to_lists(det)[0]
    ref = g[f"{name}_dets"]
    assert len(dets) == len(ref)
    a, b = canon(dets), canon(ref)
    assert np.array_equal(a[:, 5], b[:, 5])
    np.testing.assert_allclose(a[:, :4], b[:, :4], rtol=1e-5, atol=2e-4)
    np.testing.assert_allclose(a[:, 4], b[:, 4], rtol=1e-5, atol=1e-8)


def test_model_heads_fixture(yb, golden):
    g = golden("model_heads")
    heads = [T(g[f"head{s}"]) for s in range(3)]
    tgts = []
    for s, h in enumerate(heads):
        t = torch.zeros_like(h)
        idx = g[f"tgt{s}_idx"]
        if len(idx):
            t[idx[:, 0], idx[:, 1], idx[:, 2], idx[:, 3]] = T(g[f"tgt{s}_rows"])
        tgts.append(t.cuda())
    preds = [h.cuda().requires_grad_(True) for h in heads]
    res = yb.yolo_loss_multiscale(preds, tgts, ANCH, 1)
    for a, b in zip(res, g["losses"]):
        close(a, float(b), atol=1e-7)
    res[0].backward()
    for s in range(3):
        grad_close(preds[s].grad[..., 4], g[f"grad{s}_obj"])
        idx = g[f"tgt{s}_idx"]
        if len(idx):
            grad_close(preds[s].grad.cpu()[idx[:, 0], idx[:, 1], idx[:, 2], idx[:, 3]], g[f"grad{s}_rows"])
    # detection on these heads: every sigmoid(obj) lies within 50 ulp of 0.01 and the scores are
    # heavily tied, so the END-TO-END keep set is decided by the last bit of the sigmoid
    # implementation (torch's CPU and CUDA kernels disagree with each other here).  Parity is
    # therefore graded in two steps: candidates within 1e-5, NMS bit-exact on identical inputs.
    conf = float(g["confs"][0])
    det = yb.detect_batch([h.cuda() for h in heads], ANCH, 640, 1, conf, 0.4)
    m = int(det["counts"][0])
    rb, rs, rc = R.candidates(heads, ANCH, 640, 1, conf)
    assert m == rb.shape[0] == 25200 and len(g["dets_0"]) > 0
    close(det["boxes"][0, :m], rb, atol=2e-4)
    close(det["scores"][0, :m], rs, atol=1e-9)
    want = R.batched_nms_indices(det["boxes"][0, :m].cpu().numpy(), det["scores"][0, :m].cpu().numpy(),
                                 det["classes"][0, :m].cpu().numpy(), 0.4, "cuda", "cuda")
    assert np.array_equal(det["keep"][0, :int(det["n_keep"][0])].cpu().numpy(), want)


# ---- full-size properties (BASELINE configs[1..3]) -----------------------------------------------
@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("nc,B,conf", [(1, 64, 0.25), (80, 8, 0.001)])
def test_full_size_properties(yb, nc, B, conf, algo):
    g = torch.Generator().manual_seed(1234)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g).cuda() for G in (80, 40, 20)]
    det = yb.detect_batch(heads, ANCH, 640, nc, conf, 0.4, algo=algo)
    counts, n_keep = det["counts"].cpu(), det["n_keep"].cpu()
    assert (n_keep > 0).all() and (n_keep <= counts).all()
    for b in (0, B - 1):
        m, k = int(counts[b]), int(n_keep[b])
        keep = det["keep"][b, :k]
        sc = det["scores"][b].index_select(0, keep)
        assert bool((sc[:-1] >= sc[1:]).all())                      # descending score order
        assert len(torch.unique(keep)) == k                         # no duplicates
        # idempotence: NMS of the kept set keeps everything, in the same order
        bx = det["boxes"][b].index_select(0, keep)
        cl = det["classes"][b].index_select(0, keep)
        again = yb.batched_nms(bx, sc, cl, 0.4)
        assert torch.equal(again.cpu(), torch.arange(k))
        # image b against the oracle, bit-exact, on identical NMS inputs
        want = R.batched_nms_indices(det["boxes"][b, :m].cpu().numpy(), det["scores"][b, :m].cpu().numpy(),
                                     det["classes"][b, :m].cpu().numpy(), 0.4, "cuda", "cuda")
        assert np.array_equal(keep.cpu().numpy(), want)


def _check_image_against_oracle_and_torchvision(yb, det, heads_cpu, b, img, nc, conf, iou):
    """One image of a detect_batch result: candidates vs the oracle's filter, keep set bit-exact vs
    torchvision.ops.batched_nms on CUDA tensors (the reference's GPU path, train.py:1232-1233) and the C oracle."""
    import torchvision
    m, k = int(det["counts"][b]), int(det["n_keep"][b])
    bx, sc, cl = det["boxes"][b, :m], det["scores"][b, :m], det["classes"][b, :m]
    rb, rs, rc = R.candidates([h[b:b + 1] for h in heads_cpu], ANCH, img, nc, conf)
    assert m == rb.shape[0] and torch.equal(cl.cpu(), rc)
    close(bx, rb, atol=1e-5 * img)
    close(sc, rs, atol=1e-8)
    want_tv = torchvision.ops.batched_nms(bx, sc, cl, iou)          # picks the per-class loop above 25,000 boxes
    got = det["keep"][b, :k]
    assert torch.equal(got, want_tv), (k, int(want_tv.numel()))
    want = R.batched_nms_indices(bx.cpu().numpy(), sc.cpu().numpy(), cl.cpu().numpy(), iou, "cuda", "cuda")
    assert np.array_equal(got.cpu().numpy(), want)


def test_config3_full_size_1280_nc80_dense(yb):
    """BASELINE configs[3] at its real per-image size: nc=80 heads at 1280x1280, conf 0.001 -> 100,800 candidates per
    image (4 spatial chunks, the ballot score sort, torchvision's per-class regime).  B=2 keeps the oracle fast."""
    nc, img, B, conf, iou = 80, 1280, 2, 0.001, 0.4
    g = torch.Generator().manual_seed(1234)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (160, 80, 40)]
    det = yb.detect_batch([h.cuda() for h in heads], ANCH, img, nc, conf, iou)
    assert det["counts"].cpu().tolist() == [100800, 100800]
    for b in range(B):
        _check_image_against_oracle_and_torchvision(yb, det, heads, b, img, nc, conf, iou)
    # the dense bitmask algorithm agrees
    d1 = yb.detect_batch([h[:1].cuda() for h in heads], ANCH, img, nc, conf, iou, algo=yb.NMS_BITMASK)
    k = int(det["n_keep"][0])
    assert int(d1["n_keep"][0]) == k and torch.equal(d1["keep"][0, :k], det["keep"][0, :k])


def test_config2_full_batch_640_nc80_dense(yb):
    """BASELINE configs[2] at its real batch: nc=80, 640x640, B=64, conf 0.001 (25,200 candidates per image: just above
    torchvision's 25,000-box switch to the per-class loop); first, middle and last image against the oracle."""
    nc, img, B, conf, iou = 80, 640, 64, 0.001, 0.4
    g = torch.Generator().manual_seed(1234)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (80, 40, 20)]
    det = yb.detect_batch([h.cuda() for h in heads], ANCH, img, nc, conf, iou)
    assert bool((det["counts"] == 25200).all()) and bool((det["n_keep"] > 0).all())
    for b in (0, 31, 63):
        _check_image_against_oracle_and_torchvision(yb, det, heads, b, img, nc, conf, iou)


def test_config1_conf_sweep_keep_sets(yb):
    """configs[1] heads (nc=1, 640x640) at the three thresholds of SURVEY 8d: 0.5 (coordinate-trick regime, 12.6 K
    candidates), 0.25 and 0.001 (25,200 > 25,000: per-class regime) for two images each."""
    nc, img, B, iou = 1, 640, 4, 0.4
    g = torch.Generator().manual_seed(1234)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (80, 40, 20)]
    for conf in (0.5, 0.25, 0.001):
        det = yb.detect_batch([h.cuda() for h in heads], ANCH, img, nc, conf, iou)
        for b in (0, 3):
            _check_image_against_oracle_and_torchvision(yb, det, heads, b, img, nc, conf, iou)


@pytest.mark.parametrize("nc,conf", [(1, 0.25), (80, 0.25), (80, 0.05)])
def test_prior_heads_keep_sets(yb, nc, conf):
    """SURVEY 8d's "prior" variant: objectness logit 2*randn - 4.6 (a detector's prior: a few per cent of the rows
    pass), i.e. the sparse side of the one-pass filter (most tiles of a group hold no candidate) and small, ragged
    per-image candidate counts for the NMS; candidates vs the oracle, keep sets vs torchvision's CUDA kernel."""
    img, B, iou = 640, 6, 0.4
    g = torch.Generator().manual_seed(77)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (80, 40, 20)]
    for h in heads:
        h[..., 4].mul_(2.0).sub_(4.6)
    heads[1][2, ..., 4] = -30.0          # an image whose P4 head has no candidate at all
    det = yb.detect_batch([h.cuda() for h in heads], ANCH, img, nc, conf, iou)
    counts = det["counts"].cpu()
    assert 0 < int(counts.min()) and int(counts.max()) < 25200 // 4
    for b in range(B):
        _check_image_against_oracle_and_torchvision(yb, det, heads, b, img, nc, conf, iou)


def _fuzz_boxes(rng, n, kind):
    """Box sets that stress the half-precision filter's frames and rounding: sizes spanning 6 decades inside one
    image, extreme aspect ratios, sub-pixel boxes next to image-sized ones, duplicates, jittered clusters, huge
    coordinate offsets, integer grids."""
    if kind == "decades":
        c = rng.uniform(0, 1000, (n, 2)); wh = 10.0 ** rng.uniform(-3, 3, (n, 2))
    elif kind == "aspect":
        c = rng.uniform(0, 640, (n, 2)); w = 10.0 ** rng.uniform(-1, 2.5, n); ar = 10.0 ** rng.uniform(-2.5, 2.5, n)
        wh = np.stack([w, w * ar], 1)
    elif kind == "clusters":
        k = max(1, n // 40); cc = rng.uniform(0, 800, (k, 2)); ww = 10.0 ** rng.uniform(0, 2.3, (k, 2))
        idx = rng.integers(0, k, n)
        c = cc[idx] + rng.normal(0, 0.08, (n, 2)) * ww[idx]; wh = ww[idx] * np.exp(rng.normal(0, 0.12, (n, 2)))
    elif kind == "offset":
        c = rng.uniform(0, 300, (n, 2)) + 3.0e5; wh = rng.uniform(1, 120, (n, 2))
    elif kind == "grid":
        c = rng.integers(0, 64, (n, 2)).astype(np.float64) * 8.0; wh = rng.integers(1, 6, (n, 2)).astype(np.float64) * 8.0
    else:  # "tiny": sub-pixel boxes spread over a large image, plus a few big ones
        c = rng.uniform(0, 2000, (n, 2)); wh = 10.0 ** rng.uniform(-4, -1, (n, 2))
        big = rng.random(n) < 0.05
        wh[big] = rng.uniform(100, 900, (int(big.sum()), 2))
    boxes = np.concatenate([c - wh / 2, c + wh / 2], 1).astype(np.float32)
    dup = rng.random(n) < 0.05                      # exact duplicates
    boxes[dup] = boxes[rng.integers(0, n, int(dup.sum()))]
    scores = rng.random(n).astype(np.float32)
    scores[rng.random(n) < 0.1] = scores[0]         # score ties
    return torch.from_numpy(boxes), torch.from_numpy(scores)


@pytest.mark.parametrize("kind", ["decades", "aspect", "clusters", "offset", "grid", "tiny"])
def test_nms_fuzz_against_torchvision(yb, kind):
    """The graph algorithm's half-precision filter may only ADD work, never lose an edge: keep sets equal
    torchvision's CUDA kernels bit for bit on adversarial box distributions, thresholds from 0.03 to 0.9, with and
    without classes, batched with ragged counts."""
    import torchvision
    rng = np.random.default_rng({"decades": 11, "aspect": 12, "clusters": 13, "offset": 14, "grid": 15, "tiny": 16}[kind])
    for trial, thr in enumerate((0.03, 0.1, 0.3, 0.4, 0.5, 0.7, 0.9)):
        B = 3
        ns = [int(rng.integers(1, 9000)) for _ in range(B)]
        cap = max(ns)
        boxes = torch.zeros(B, cap, 4); scores = torch.zeros(B, cap); classes = torch.zeros(B, cap, dtype=torch.int64)
        sets = []
        for b, n in enumerate(ns):
            bx, sc = _fuzz_boxes(rng, n, kind)
            cl = torch.from_numpy(rng.integers(0, 1 if trial % 2 else 12, n))
            boxes[b, :n], scores[b, :n], classes[b, :n] = bx, sc, cl
            sets.append((bx, sc, cl))
        counts = torch.tensor(ns, dtype=torch.int32)
        keep, n_keep = yb.batched_nms_padded(boxes.cuda(), scores.cuda(), classes.cuda(), counts.cuda(), thr)
        for b, (bx, sc, cl) in enumerate(sets):
            want = torchvision.ops.batched_nms(bx.cuda(), sc.cuda(), cl.cuda(), thr)
            got = keep[b, :int(n_keep[b])]
            assert torch.equal(got, want), (kind, thr, b, int(n_keep[b]), int(want.numel()))


def test_launch_counter_and_library(yb):
    lib = yb._lib.lib()
    before = lib.yb_launch_count()
    yb.decode_predictions(torch.zeros(1, 4, 4, 3, 6).cuda(), ANCH[0])
    assert lib.yb_launch_count() == before + 1


def test_batched_sigmoid_is_bit_identical_exhaustively(yb):
    """rcp_normal / sigmoid_ref_batch (the filter's emit and the long-row decode) against the compiler's IEEE
    division and sigmoidf_ref over EVERY float of their domains, on the device (yb_selftest_sigmoid)."""
    import ctypes
    out = (ctypes.c_ulonglong * 2)(7, 7)
    yb._lib.check(yb._lib.lib().yb_selftest_sigmoid(out, torch.cuda.current_stream().cuda_stream), "yb_selftest_sigmoid")
    assert (int(out[0]), int(out[1])) == (0, 0)


def test_bench_dump_outputs_are_the_last_timed_step(yb, tmp_path):
    """bench.py --dump-outputs: graph replay and eager launches dump the same files, and they are what the step
    computes on the input set of the last timed step ((steps - 1) % n_sets), not on another set."""
    import importlib.util
    import os
    import subprocess
    import sys
    from yolo_from_scratch_b200 import ops
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    bench_py = os.path.join(root, "bench.py")
    B, img, nc, steps = 4, 160, 3, 3
    base = [sys.executable, bench_py, "--batch", str(B), "--img", str(img), "--nc", str(nc), "--steps", str(steps),
            "--warmup", "1", "--reps", "1", "--no-other-configs", "--no-variants", "--no-e2e", "--no-cpu-baseline",
            "--no-torch-gpu-baseline", "--full-out", ""]
    for launch in ("graph", "eager"):
        p = subprocess.run(base + ["--launch", launch, "--dump-outputs", str(tmp_path / launch)], capture_output=True,
                           text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-3000:]
    names = sorted(os.listdir(tmp_path / "graph"))
    assert names == sorted(os.listdir(tmp_path / "eager")) and "grad_s0.npy" in names and "detections.npy" in names
    load = lambda d, n: np.load(str(tmp_path / d / n))
    for n in names:
        assert np.array_equal(load("graph", n), load("eager", n)), n

    spec = importlib.util.spec_from_file_location("bench_mod", bench_py)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    dev = torch.device("cuda")
    anchors, grids = ops.default_anchors(dev), [img // 8, img // 16, img // 32]

    def step_of_set(k):   # run_workload's input set k on rank 0
        heads = [h.to(dev) for h in bench.make_heads(B, img, nc, 1234 + 1000 * k)]
        tg = ops.build_targets(bench.make_labels(np.random.default_rng(4321 + k), B, nc), anchors, grids, nc, img)
        out4, _, grads = ops.loss_forward_backward(heads, tg, anchors, nc, ops.MULTISCALE_OBJ_WEIGHTS, [True] * 3)
        rows, offsets = ops.pack_detections(ops.detect_batch(heads, anchors, img, nc, bench.CONF, bench.IOU))
        return out4.cpu().numpy(), [g.cpu().numpy() for g in grads], rows[:int(offsets[-1])].cpu().numpy()

    last = (steps - 1) % 4
    losses, grads, dets = step_of_set(last)
    np.testing.assert_array_equal(load("graph", "losses.npy"), losses)
    for s in range(3):
        np.testing.assert_array_equal(load("graph", f"grad_s{s}.npy"), grads[s])
    np.testing.assert_array_equal(load("graph", "detections.npy"), dets)
    assert not np.array_equal(step_of_set(last - 1)[0], losses)
