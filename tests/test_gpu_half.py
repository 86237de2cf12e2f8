"""Native bf16 / fp16 heads: loss forward and backward, decode, candidate filter, detect_batch and HotPathGraph.

The contract: a half tensor converts exactly to fp32, so every result must equal, bit for bit, what the fp32 path
gives on `heads.float()` (NaNs compare equal whatever their payload).  Half outputs are the fp32 values rounded to
the head dtype; a loss gradient for upstream gradient s is round_D(round_f32(G * s)), with s applied before the
rounding to half.
"""
import os
import socket
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ref_path as R  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ANCH = R.default_anchors()
HALF = [torch.bfloat16, torch.float16]
IDS = ["bf16", "fp16"]


@pytest.fixture(scope="module")
def yb():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import yolo_from_scratch_b200 as m
    m._lib.lib()
    return m


def bits_equal(a, b):
    """Bitwise equality with NaN == NaN (any payload)."""
    a, b = a.detach(), b.detach()
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    iv = {2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    same = (a.view(iv) == b.view(iv))
    if a.is_floating_point():
        same |= torch.isnan(a) & torch.isnan(b)
    bad = int((~same).sum())
    assert bad == 0, f"{bad} of {a.numel()} entries differ"


def to_nchw(h):
    B, H, W, A, row = h.shape
    return h.permute(0, 3, 4, 1, 2).reshape(B, A * row, H, W).contiguous()


def random_labels(rng, B, nc, max_n=8):
    out = []
    for _ in range(B):
        n = int(rng.integers(0, max_n + 1))
        lab = np.zeros((n, 5))
        lab[:, 0] = rng.integers(0, nc, n)
        lab[:, 1:3] = rng.uniform(0.05, 0.95, (n, 2))
        lab[:, 3:5] = np.exp(rng.uniform(np.log(0.02), np.log(0.6), (n, 2)))
        out.append(lab)
    return out


def make_case(yb, B, grids, nc, img, seed, dtype, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    heads = [(torch.randn(B, G, G, 3, 5 + nc, generator=g) * scale).to(dtype).cuda() for G in grids]
    labels = random_labels(np.random.default_rng(seed), B, nc)
    tg = yb.build_targets(labels, ANCH, list(grids), nc, img)
    return heads, labels, tg


def loss_call(yb, preds, tg, labels, nc, img, layout, targets):
    from yolo_from_scratch_b200 import ops
    if layout == "nchw":
        preds = [to_nchw(p) if p.dim() == 5 else p for p in preds]
        return ops.yolo_loss_multiscale_nchw(preds, tg if targets == "dense" else labels, ANCH, nc, img)
    if targets == "dense":
        return yb.yolo_loss_multiscale(preds, tg, ANCH, nc)
    return yb.yolo_loss_multiscale_labels(preds, labels, ANCH, nc, img)


def leaf(h, layout, dtype=None):
    t = h if dtype is None else h.to(dtype)
    t = to_nchw(t) if layout == "nchw" else t.clone()
    return t.requires_grad_(True)


def check_loss(yb, heads, tg, labels, nc, img, layout, targets, dtype, scales=(1.0,), components=False):
    for s in scales:
        p = [leaf(h, layout) for h in heads]
        q = [leaf(h, layout, torch.float32) for h in heads]
        oh = loss_call(yb, p, tg, labels, nc, img, layout, targets)
        of = loss_call(yb, q, tg, labels, nc, img, layout, targets)
        bits_equal(torch.stack(oh), torch.stack(of))
        lh, lf = oh[0] * s, of[0] * s
        if components:
            lh, lf = lh + oh[1] * 0.25 + oh[2] * 3.0, lf + of[1] * 0.25 + of[2] * 3.0
        lh.backward()
        lf.backward()
        for a, b in zip(p, q):
            bits_equal(a.grad, b.grad.to(dtype))


# ---- 1. loss ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("nc", [1, 3, 80])
@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
@pytest.mark.parametrize("targets", ["dense", "labels"])
def test_loss_bit_exact(yb, dtype, nc, layout, targets):
    heads, labels, tg = make_case(yb, 3, (16, 8, 5), nc, 128, 7 + nc, dtype)
    check_loss(yb, heads, tg, labels, nc, 128, layout, targets, dtype, scales=(1.0, 65536.0, 0.3, 2.0 ** 24))
    check_loss(yb, heads, tg, labels, nc, 128, layout, targets, dtype, components=True)


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
def test_loss_retain_graph_second_backward(yb, dtype, layout):
    nc = 3
    heads, labels, tg = make_case(yb, 2, (16, 8, 4), nc, 128, 3, dtype)
    p = [leaf(h, layout) for h in heads]
    q = [leaf(h, layout, torch.float32) for h in heads]
    oh = loss_call(yb, p, tg, labels, nc, 128, layout, "dense")
    of = loss_call(yb, q, tg, labels, nc, 128, layout, "dense")
    for k, s in enumerate((65536.0, 0.3)):
        (oh[0] * s).backward(retain_graph=True)
        (of[0] * s).backward(retain_graph=True)
        for a, b in zip(p, q):
            bits_equal(a.grad, b.grad.to(dtype))
            a.grad = None
            b.grad = None


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("cfg", ["configs1", "configs2"])
def test_loss_full_scale_set(yb, dtype, cfg):
    nc = 1 if cfg == "configs1" else 80
    heads, labels, tg = make_case(yb, 64 if nc == 1 else 16, (80, 40, 20), nc, 640, 11, dtype)
    check_loss(yb, heads, tg, labels, nc, 640, "bhwac", "dense", dtype, scales=(65536.0,))
    check_loss(yb, heads, tg, labels, nc, 640, "nchw", "labels", dtype, scales=(1.0,))


def test_fp16_objectness_below_normal_range_scaled_before_rounding(yb):
    """B*H*W*A large: coef/(B*H*W*A) puts the objectness gradients below 2^-14, where fp16 is subnormal.  At
    s = 65536 they are normal numbers; rounding to fp16 first and scaling afterwards would lose them."""
    nc, dtype = 1, torch.float16
    heads, labels, tg = make_case(yb, 8, (80, 40, 20), nc, 640, 5, dtype)
    p = [h.clone().requires_grad_(True) for h in heads]
    q = [h.float().requires_grad_(True) for h in heads]
    (yb.yolo_loss_multiscale(p, tg, ANCH, nc)[0] * 65536.0).backward()
    (yb.yolo_loss_multiscale(q, tg, ANCH, nc)[0] * 65536.0).backward()
    g_obj = q[0].grad[..., 4] / 65536.0
    assert float(g_obj.abs().max()) < 2.0 ** -14 and float(g_obj.abs().min()) > 0.0
    for a, b in zip(p, q):
        bits_equal(a.grad, b.grad.to(dtype))
    rounded_first = (g_obj.to(dtype).float() * 65536.0).to(dtype)
    assert not torch.equal(rounded_first, p[0].grad[..., 4])


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("targets", ["dense", "labels"])
def test_loss_two_rank_emulation_half(yb, dtype, targets):
    from yolo_from_scratch_b200 import ops
    B, nc = 6, 2
    heads, labels, tg = make_case(yb, B, (16, 8, 4), nc, 128, 21, dtype)
    anc = [a.cuda() for a in ANCH]
    w = ops.MULTISCALE_OBJ_WEIGHTS
    cut = lambda ts, lo, hi: [t[lo:hi].contiguous() for t in ts]
    shards = [(0, 4), (4, 6)]

    def run(hs, scale):
        parts = []
        for lo, hi in shards:
            kw = dict(sparse=yb.pack_labels(labels[lo:hi], 128)) if targets == "labels" else {}
            ops.loss_forward_backward(cut(hs, lo, hi), None if kw else cut(tg, lo, hi), anc, nc, w, [True] * 3,
                                      b_global=B, reduce_fn=lambda p: (parts.append(p.clone()), p)[1], **kw)
        total = parts[0] + parts[1]
        res = []
        for lo, hi in shards:
            kw = dict(sparse=yb.pack_labels(labels[lo:hi], 128)) if targets == "labels" else {}
            gs = torch.full((1,), scale, device="cuda") if hs[0].dtype != torch.float32 else None
            out4, _, grads = ops.loss_forward_backward(cut(hs, lo, hi), None if kw else cut(tg, lo, hi), anc, nc, w,
                                                       [True] * 3, b_global=B, reduce_fn=lambda p: total.clone(),
                                                       grad_scale=gs, **kw)
            res.append((out4, grads))
        return res

    for scale in (1.0, 65536.0):
        rh, rf = run(heads, scale), run([h.float() for h in heads], scale)
        for (oh, gh), (of, gf) in zip(rh, rf):
            bits_equal(oh, of)
            for a, b in zip(gh, gf):
                bits_equal(a, (b * scale if scale != 1.0 else b).to(dtype))


# ---- 2. decode --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("nc", [1, 2, 3, 6, 80])
def test_decode_forward_backward(yb, dtype, nc):
    g = torch.Generator().manual_seed(nc)
    h = (torch.randn(3, 7, 9, 3, 5 + nc, generator=g) * 3).to(dtype).cuda()
    go = torch.randn(h.shape, generator=g).to(dtype).cuda()
    p = h.clone().requires_grad_(True)
    q = h.float().requires_grad_(True)
    oh = yb.decode_predictions(p, ANCH[0], 640)
    of = yb.decode_predictions(q, ANCH[0], 640)
    assert oh.dtype == dtype
    bits_equal(oh, of.to(dtype))
    oh.backward(go)
    of.backward(go.float())
    bits_equal(p.grad, q.grad.to(dtype))


# ---- 3. filter --------------------------------------------------------------------------------------------------
ANCH4 = torch.tensor([[10., 13.], [33., 23.], [62., 45.], [116., 90.]])


def filter_equal(yb, heads, anchors, img, nc, conf, layout):
    from yolo_from_scratch_b200 import ops
    lay = ops.LAYOUT_NCHW if layout == "nchw" else ops.LAYOUT_BHWAC
    hh = [to_nchw(h) if layout == "nchw" else h for h in heads]
    a = yb.filter_candidates(hh, anchors, img, nc, conf, layout=lay)
    b = yb.filter_candidates([h.float() for h in hh], anchors, img, nc, conf, layout=lay)
    bits_equal(a[3], b[3])
    for i, n in enumerate(a[3].tolist()):
        for x, y in zip(a[:3], b[:3]):
            bits_equal(x[i, :n], y[i, :n])
    return int(a[3].sum())


def all_patterns(dtype):
    return torch.arange(-32768, 32768, dtype=torch.int32).to(torch.int16).view(dtype)


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
@pytest.mark.parametrize("nc", [1, 80])
def test_filter_every_objectness_pattern(yb, dtype, layout, nc):
    g = torch.Generator().manual_seed(1)
    h = (torch.randn(1, 128, 128, 4, 5 + nc, generator=g) * 4).to(dtype)
    h[..., 4] = all_patterns(dtype).reshape(1, 128, 128, 4)
    h = h.cuda()
    for conf in (0.001, 0.25, 0.5, 0.9999):
        assert filter_equal(yb, [h], [ANCH4], 1024, nc, conf, layout) > 0


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
def test_filter_every_class_pattern_and_near_ties(yb, dtype, layout):
    pat = all_patterns(dtype).reshape(1, 128, 128, 4)
    nxt = torch.roll(pat.view(torch.int16), -1).view(dtype)   # the neighbouring bit pattern: a near-tie
    h = torch.zeros(1, 128, 128, 4, 8, dtype=dtype)
    h[..., 4] = 12.0   # every row passes
    h[..., 5], h[..., 6], h[..., 7] = pat, nxt, -pat
    h[..., :4] = (torch.randn(1, 128, 128, 4, 4, generator=torch.Generator().manual_seed(2))).to(dtype)
    assert filter_equal(yb, [h.cuda()], [ANCH4], 1024, 3, 0.5, layout) == 65536


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
def test_filter_ragged_tails_and_offset_views(yb, dtype, layout):
    nc = 2
    g = torch.Generator().manual_seed(9)
    heads = [(torch.randn(3, G, G, 3, 5 + nc, generator=g) * 3).to(dtype).cuda() for G in (7, 5, 3)]
    for conf in (0.001, 0.25, 0.5):
        filter_equal(yb, heads, ANCH, 56, nc, conf, layout)
    # a view at a 2-byte offset: not 16-byte aligned
    flat = torch.randn(heads[0].numel() + 1, generator=g).to(dtype).cuda()
    view = flat[1:].view(heads[0].shape)
    assert view.data_ptr() % 16 != 0
    filter_equal(yb, [view] + heads[1:], ANCH, 56, nc, 0.25, layout)


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
@pytest.mark.parametrize("layout", ["bhwac", "nchw"])
@pytest.mark.parametrize("nc", [1, 80])
def test_detect_batch_keep_sets(yb, dtype, layout, nc):
    from yolo_from_scratch_b200 import ops
    lay = ops.LAYOUT_NCHW if layout == "nchw" else ops.LAYOUT_BHWAC
    g = torch.Generator().manual_seed(nc)
    heads = [(torch.randn(2, G, G, 3, 5 + nc, generator=g) * 2).to(dtype).cuda() for G in (16, 8, 4)]
    hh = [to_nchw(h) if layout == "nchw" else h for h in heads]
    for conf in (0.5, 0.25, 0.001):
        a = yb.detect_batch(hh, ANCH, 128, nc, conf, 0.4, layout=lay)
        b = yb.detect_batch([h.float() for h in hh], ANCH, 128, nc, conf, 0.4, layout=lay)
        bits_equal(a["counts"], b["counts"])
        bits_equal(a["n_keep"], b["n_keep"])
        for i, k in enumerate(a["n_keep"].tolist()):
            bits_equal(a["keep"][i, :k], b["keep"][i, :k])
            bits_equal(a["scores"][i, a["keep"][i, :k]], b["scores"][i, b["keep"][i, :k]])


# ---- 4. memory --------------------------------------------------------------------------------------------------
def test_no_hidden_fp32_copy(yb):
    """Each call's own rise of the peak stays below the fp32 size of the heads: a conversion to fp32 alone would be
    that large.  (Together the loss gradients and detect_batch's candidates and NMS workspace at conf 0.001 exceed
    it, so each call is measured from its own starting point.)"""
    nc, B = 80, 64
    heads, labels, tg = make_case(yb, B, (80, 40, 20), nc, 640, 4, torch.bfloat16)
    p = [h.requires_grad_(True) for h in heads]
    fp32_bytes = sum(h.numel() * 4 for h in heads)

    def rise(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base, out

    grown, _ = rise(lambda: yb.yolo_loss_multiscale(p, tg, ANCH, nc)[0].backward())
    assert grown < fp32_bytes, (grown, fp32_bytes)
    assert p[0].grad.dtype == torch.bfloat16
    grown, det = rise(lambda: yb.detect_batch([h.detach() for h in p], ANCH, 640, nc, 0.001, 0.4))
    assert grown < fp32_bytes, (grown, fp32_bytes)
    assert det["counts"].numel() == B


# ---- 5. autocast end to end -------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", HALF, ids=IDS)
def test_autocast_step_equals_upcast_path(yb, dtype):
    from yolo_from_scratch_b200 import ops
    nc, B, img = 3, 2, 128
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
    torch.manual_seed(0)
    convs = torch.nn.ModuleList([torch.nn.Conv2d(16, 3 * (5 + nc), 1) for _ in range(3)]).cuda()
    xs = [torch.randn(B, 16, G, G, device="cuda") for G in (16, 8, 4)]
    labels = random_labels(np.random.default_rng(0), B, nc)
    tg = yb.build_targets(labels, ANCH, [16, 8, 4], nc, img)
    grads = []
    for upcast in (False, True):
        convs.zero_grad(set_to_none=True)
        scaler = torch.amp.GradScaler("cuda", enabled=dtype == torch.float16)
        with torch.autocast("cuda", dtype=dtype):
            heads = [c(x) for c, x in zip(convs, xs)]
            assert heads[0].dtype == dtype
            if upcast:
                heads = [h.float() for h in heads]
            loss = ops.yolo_loss_multiscale_nchw(heads, tg, ANCH, nc, img)[0]
        scaler.scale(loss).backward()
        grads.append([p.grad.clone() for p in convs.parameters()])
    for a, b in zip(*grads):
        bits_equal(a, b)


# ---- 6. HotPathGraph --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", HALF, ids=IDS)
def test_hot_path_graph_half(yb, dtype):
    nc, B, img = 3, 2, 128
    heads, labels, tg = make_case(yb, B, (16, 8, 4), nc, img, 8, dtype)
    hp = yb.HotPathGraph(B, img, nc, ANCH, conf_threshold=0.25, targets="dense", dtype=dtype)
    for s in range(3):
        hp.heads[s].copy_(heads[s])
        hp.targets[s].copy_(tg[s])
    for scale in (1.0, 65536.0, 0.3):
        hp.grad_scale.fill_(scale)
        losses, grads, det = hp.replay()
        p = [h.clone().requires_grad_(True) for h in heads]
        out = yb.yolo_loss_multiscale(p, tg, ANCH, nc)
        (out[0] * scale).backward()
        bits_equal(losses, torch.stack(out).detach())
        for a, b in zip(grads, p):
            bits_equal(a, b.grad)
        ref = yb.detect_batch(heads, ANCH, img, nc, 0.25, 0.4)
        bits_equal(det["n_keep"], ref["n_keep"])


def test_hot_path_graph_adopt_heads_dtype_checked(yb):
    heads = [torch.zeros(2, G, G, 3, 8, dtype=torch.float64, device="cuda") for G in (16, 8, 4)]
    before = yb._lib.lib().yb_launch_count()
    with pytest.raises(ValueError):
        yb.HotPathGraph(2, 128, 3, ANCH, adopt_heads=heads, dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        yb.HotPathGraph(2, 128, 3, ANCH, adopt_heads=heads)
    assert yb._lib.lib().yb_launch_count() == before


# ---- 7. two GPUs (NCCL) -----------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, dtype, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import yolo_from_scratch_b200 as yb
        from yolo_from_scratch_b200 import dist as ybd
        B, nc, grids, img = 6, 3, (20, 10, 5), 160
        heads, labels, tg = make_case(yb, B, grids, nc, img, 17, dtype)
        lo, hi = ybd.shard_range(B, rank, world)
        ok = True
        for sparse in (False, True):
            p = [h[lo:hi].clone().requires_grad_(True) for h in heads]
            f = [h[lo:hi].float().requires_grad_(True) for h in heads]
            outs = []
            for x in (p, f):
                if sparse:
                    o = yb.yolo_loss_multiscale_labels(x, labels[lo:hi], ANCH, nc, img, group=dist.group.WORLD)
                else:
                    o = ybd.yolo_loss_multiscale_sharded(x, [t[lo:hi] for t in tg], ANCH, nc, group=dist.group.WORLD)
                (o[0] * 65536.0).backward()
                outs.append(torch.stack(o).detach())
            ok &= torch.equal(outs[0], outs[1])
            for a, b in zip(p, f):
                ref = b.grad.to(dtype)
                ok &= bool(((a.grad.view(torch.int16) == ref.view(torch.int16)) |
                            (torch.isnan(a.grad) & torch.isnan(ref))).all())
        q.put((rank, ok))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("dtype", HALF, ids=IDS)
def test_nccl_sharded_half_loss(dtype):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, dtype, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok in results), results
