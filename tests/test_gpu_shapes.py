"""The per-row kernels off the square three-anchor three-scale shape (run with -m gpu on the B200 box).

Every per-row kernel splits a flat row index into (b, gy, gx, an) with FastDivs built per scale, decodes with 1/W and
1/H and scales the objectness gradient by coef / (B*H*W*A).  The other files use square grids, A = 3 and S = 3 almost
everywhere, where H and W, or one scale's offsets and another's, cannot be told apart.  Here every grid has H != W
(one dimension 1, odd H*W, B*H*W*A not a multiple of the loss kernel's 256-row tile, scales of fewer rows than one
tile), A in {1, 2, 5, 8} with anchors that differ per scale, S in {1, 2, 4} and nc in {0, 1, 2, 7, 80}.

The loss runs in two value regimes: unit-scale logits, and saturated ones as a trained detector produces them.
Saturated logits give gradient entries many decades below the tensor's largest, which the relative-to-max gradient
tolerance of DESIGN §4 cannot see; the objectness and class columns are therefore also checked element by element
against the oracle run in float64 (`check_columns_fp64`).

References: losses and gradients against the oracle on CPU fp32 (DESIGN §4 tolerances), filter / multi-label filter /
eval counts bit-exact against the oracle evaluated on CUDA tensors (torch-CUDA's own sigmoid and compare), targets
bit-exact against the oracle's assignment, bf16 / fp16 heads bit-identical to the fp32 path on `heads.float()`.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import multilabel_ref as ML  # noqa: E402
from oracle import ref_path as R  # noqa: E402

HALF = [torch.bfloat16, torch.float16]
U32 = 2.0 ** -24          # unit roundoff of fp32
TINY = 2.0 ** -126        # smallest normal fp32
LOSS_IMG = 640            # the loss and eval_counts decode with the reference's default img_size


@pytest.fixture(scope="module")
def yb():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import yolo_from_scratch_b200 as m
    m._lib.lib()  # fail loudly if the extension is missing
    return m


# ---- comparisons ------------------------------------------------------------------------------------------------
def close(a, b, rtol=1e-5, atol=0.0, what=""):
    a, b = torch.as_tensor(a).detach().cpu().double(), torch.as_tensor(b).detach().cpu().double()
    err = (a - b).abs()
    tol = rtol * b.abs() + atol
    assert bool((err <= tol).all()), f"{what}: max err {float(err.max()):.3e}, max excess {float((err - tol).max()):.3e}"


def grad_close(a, b, what=""):
    b = torch.as_tensor(b)
    close(a, b, rtol=1e-4, atol=1e-5 * float(b.abs().max()) + 1e-12, what=what)


def bits_equal(a, b, what=""):
    """Bitwise equality with NaN == NaN (any payload)."""
    a, b = a.detach(), b.detach()
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    iv = {2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    same = a.contiguous().view(iv) == b.contiguous().view(iv)
    if a.is_floating_point():
        same |= torch.isnan(a) & torch.isnan(b)
    bad = int((~same).sum())
    assert bad == 0, f"{what}: {bad} of {a.numel()} entries differ"


def box_close(got, want, what=""):
    err = (got.double() - want.double()).abs()
    tol = 1e-5 * want.double().abs() + 2e-4
    assert bool((err <= tol).all()), f"{what} boxes: max err {float(err.max()):.3e}"


# ---- shapes -----------------------------------------------------------------------------------------------------
def to_nchw(h):
    B, H, W, A, C = h.shape
    return h.permute(0, 3, 4, 1, 2).reshape(B, A * C, H, W).contiguous()


def from_nchw(g, A):
    B, AC, H, W = g.shape
    return g.view(B, A, AC // A, H, W).permute(0, 3, 4, 1, 2).contiguous()


def make_anchors(S, A, seed):
    """(A, 2) pixel anchors per scale, growing by ~2.2x a scale, with per-anchor aspect ratios that differ per scale."""
    rng = np.random.default_rng(seed)
    out = []
    for s in range(S):
        base = 12.0 * 2.2 ** s * np.exp(np.linspace(-0.6, 0.6, A))
        wh = np.stack([base * np.exp(rng.uniform(-0.5, 0.5, A)), base * np.exp(rng.uniform(-0.5, 0.5, A))], 1)
        out.append(torch.tensor(wh, dtype=torch.float32))
    return out


def assert_non_square(grids):
    assert all(h != w for h, w in grids), grids


# ---- 1. fused loss, dense targets -------------------------------------------------------------------------------
# (B, per-scale (H, W), A, nc).  Rows per scale, B*H*W*A (the loss kernel's tile is 256 rows):
#   s1_a1_nc0:  819 (H*W = 273 odd, last tile ragged)
#   s1_a2_nc1:  36 (a 1x9 grid: one tile, smaller than a tile)
#   s2_a8_nc2:  1120, 144 (scale 1 starts at tile 5 and is smaller than a tile; 1x9 grid)
#   s4_a5_nc7:  2040, 540, 150, 20 (odd H*W 15 and a 2x1 grid; every scale starts after a ragged tile)
#   s4_a2_nc80: 252, 70, 24, 4 (every scale smaller than one tile; H*W = 35 odd)
LOSS_CASES = {
    "s1_a1_nc0": (3, [(13, 21)], 1, 0),
    "s1_a2_nc1": (2, [(1, 9)], 2, 1),
    "s2_a8_nc2": (2, [(10, 7), (1, 9)], 8, 2),
    "s4_a5_nc7": (2, [(12, 17), (6, 9), (3, 5), (2, 1)], 5, 7),
    "s4_a2_nc80": (1, [(9, 14), (5, 7), (3, 4), (1, 2)], 2, 80),
}
OBJ_WEIGHTS = (4.0, 1.0, 0.4, 0.1)   # the reference's three and a fourth for S = 4


def dense_targets(B, grids, A, nc, rng):
    """Reference-layout targets with soft values.  Objectness: positives of 1.0 and of nextafter(0.5, 1) (the smallest
    value the reference's `> 0.5` counts), exactly 0.5 (not positive), 0.25 and 0.  Positive rows get a box and a
    one-hot class vector, hard (1/0) or smoothed (0.9/0.1); other rows carry junk that the loss must ignore."""
    above = float(np.nextafter(np.float32(0.5), np.float32(1.0)))
    tg = []
    for H, W in grids:
        n = B * H * W * A
        t = torch.zeros(n, 5 + nc)
        t[:, :4] = torch.from_numpy(rng.uniform(0.0, 1.0, (n, 4)).astype(np.float32))
        if nc:
            t[:, 5:] = torch.from_numpy(rng.uniform(0.0, 1.0, (n, nc)).astype(np.float32))
        perm = rng.permutation(n)
        n_pos, n_half, n_soft = max(2, n // 12), max(1, n // 24), n // 12
        pos, half, soft = perm[:n_pos], perm[n_pos:n_pos + n_half], perm[n_pos + n_half:n_pos + n_half + n_soft]
        t[pos, 4] = torch.tensor([above if k % 3 == 0 else 1.0 for k in range(n_pos)])
        t[half, 4] = 0.5
        t[soft, 4] = 0.25
        rest = perm[n_pos + n_half + n_soft:]
        t[rest, 4] = 0.0
        xy = rng.uniform(0.05, 0.95, (n_pos, 2))
        wh = np.exp(rng.uniform(np.log(0.02), np.log(0.6), (n_pos, 2)))
        t[pos, :4] = torch.from_numpy(np.concatenate([xy, wh], 1).astype(np.float32))
        if nc:
            cls = rng.integers(0, nc, n_pos)
            smooth = rng.random(n_pos) < 0.5
            t[pos, 5:] = torch.from_numpy(np.where(smooth[:, None], 0.1, 0.0).astype(np.float32))
            t[pos, 5 + cls] = torch.from_numpy(np.where(smooth, 0.9, 1.0).astype(np.float32))
        tg.append(t.reshape(B, H, W, A, 5 + nc))
    return tg


def loss_heads(B, grids, A, nc, regime, tgts, gen):
    """'unit': randn logits.  'saturated': background objectness in [-100, -8], positive rows' objectness and target
    class logit in [5, 25], every other class logit in [-25, -5], box logits in [-20, 20]."""
    heads = []
    for (H, W), t in zip(grids, tgts):
        shape = (B, H, W, A, 5 + nc)
        if regime == "unit":
            heads.append(torch.randn(*shape, generator=gen))
            continue
        uni = lambda lo, hi, *s: lo + (hi - lo) * torch.rand(*s, generator=gen)
        h = torch.empty(shape)
        pos = t[..., 4] > 0.5
        h[..., :4] = uni(-20.0, 20.0, *shape[:4], 4)
        h[..., 4] = torch.where(pos, uni(5.0, 25.0, *shape[:4]), uni(-100.0, -8.0, *shape[:4]))
        if nc:
            h[..., 5:] = uni(-25.0, -5.0, *shape[:4], nc)
            top = t[..., 5:].argmax(-1)
            idx = pos.nonzero(as_tuple=True)
            h[idx + (5 + top[idx],)] = uni(5.0, 25.0, int(pos.sum()))
        heads.append(h)
    return heads


def oracle_loss(preds, tgts, anchors, nc, weights):
    """yolo_loss_multiscale (train.py:840-886) with explicit objectness weights, any number of scales:
    (total, sum bbox, sum obj, sum cls) and the per-scale (bbox, obj, cls)."""
    total = box = obj = cls = 0.0
    per = []
    for p, t, a, w in zip(preds, tgts, anchors, weights):
        _, b_, o_, c_ = R.single_scale_loss(p, t, a, nc)
        total = total + (0.05 * b_ + w * o_ + 0.5 * c_)
        box, obj, cls = box + b_, obj + o_, cls + c_
        per.append((b_, o_, c_))
    return (total, box, obj, cls), per


def run_loss(heads, tgts, ancs, nc, weights, layout, sparse=None):
    """ops.loss_forward_backward on device heads (reference layout); gradients returned in the reference layout."""
    from yolo_from_scratch_b200 import ops
    A = ancs[0].shape[0]
    lay = ops.LAYOUT_NCHW if layout == "nchw" else ops.LAYOUT_BHWAC
    preds = [to_nchw(h) if layout == "nchw" else h.contiguous() for h in heads]
    out4, per_scale, grads = ops.loss_forward_backward(preds, tgts, ancs, nc, weights, [True] * len(heads),
                                                       layout=lay, sparse=sparse)
    if layout == "nchw":
        grads = [from_nchw(g, A) for g in grads]
    return out4, per_scale, grads


def check_columns_fp64(grads, heads, tgts, anchors, nc, weights, what):
    """The objectness and class columns of the gradient are elementwise:
        d total / d x_obj = (sigma(x) - t) * c_obj,  c_obj = w_s / (B*H*W*A)
        d total / d x_cls = (sigma(x) - t) * c_cls,  c_cls = 0.5 / (P_s*nc) on the P_s positive rows, 0 elsewhere
    The kernels evaluate them in fp32 as fl(fl(sigma32(x) - t) * fl32(c)), with t exact (an fp32 input), so against
    the exact value (the oracle run in float64, whose own error is ~1e-16 relative):
      - sigma32(x) = 1/(1+expf(-x)): expf within 2 ulp, the sum and the division each rounded once, so within 4u of
        sigma(x) while the result is a normal number (u = 2^-24); where sigma(x) < 2^-126 (x < -87.3) the result is
        subnormal or 0, off by less than 2^-126;
      - the difference with t: one rounding, u * (|sigma| + |t|);
      - the coefficient: w_s as fp32 (u) and the fp64 quotient rounded to fp32 (u);
      - the product: one rounding (u), or an absolute 2^-150 when it is subnormal.
    To first order |err| <= c * (8u * (|sigma| + |t|) + 2^-126) + 2^-150.  The bound used is
        c * (10u * (|sigma| + |t|) + 2^-126) + 2^-126,
    leaving 2u for the second-order terms.  It scales with the entry, not with the tensor's largest entry: an objectness
    gradient of 1e-35 must be right to ~1e-41."""
    ref_p = [h.detach().cpu().double().requires_grad_(True) for h in heads]
    ref_t = [t.detach().cpu().double() for t in tgts]
    (total, *_), _ = oracle_loss(ref_p, ref_t, [a.cpu().double() for a in anchors], nc, weights)
    total.backward()
    for s, (g, p, t, w) in enumerate(zip(grads, ref_p, ref_t, weights)):
        x = p.detach()
        B, H, W, A, _ = x.shape
        pos = t[..., 4] > 0.5
        P = int(pos.sum())
        coef = torch.zeros(B, H, W, A, 1 + nc, dtype=torch.float64)
        coef[..., 0] = w / (B * H * W * A)
        if nc and P:
            coef[..., 1:] = torch.where(pos, 0.5 / (P * nc), 0.0).unsqueeze(-1)
        mag = torch.sigmoid(x[..., 4:]).abs() + t[..., 4:].abs()
        tol = coef * (10 * U32 * mag + TINY) + TINY
        got, want = g[..., 4:].detach().cpu().double(), p.grad[..., 4:]
        err = (got - want).abs()
        bad = err > tol
        if bool(bad.any()):
            i = tuple(int(v) for v in bad.nonzero()[0])
            raise AssertionError(f"{what} scale {s}: {int(bad.sum())} obj/cls gradient entries off, first at {i}: "
                                 f"got {float(got[i])!r}, want {float(want[i])!r}, tol {float(tol[i]):.3e}")


def check_loss_vs_oracle(out4, per_scale, grads, heads, tgts, anchors, nc, weights, what):
    """Loss values and gradients against the oracle on CPU fp32 (DESIGN §4)."""
    ref_p = [h.detach().cpu().clone().requires_grad_(True) for h in heads]
    ref4, per = oracle_loss(ref_p, [t.cpu() for t in tgts], [a.cpu() for a in anchors], nc, weights)
    ref4[0].backward()
    for k, (a, b) in enumerate(zip(out4, ref4)):
        close(a, float(b.detach()), atol=1e-7, what=f"{what} loss[{k}]")
    for s, trip in enumerate(per):
        for k, b in enumerate(trip):
            close(per_scale[s, k], float(b.detach()), atol=1e-7, what=f"{what} scale {s} term {k}")
    for s, (g, q) in enumerate(zip(grads, ref_p)):
        grad_close(g, q.grad, what=f"{what} scale {s} gradient")


@pytest.mark.parametrize("regime", ["unit", "saturated"])
@pytest.mark.parametrize("case", list(LOSS_CASES))
def test_loss_dense_shapes(yb, case, regime):
    """Fused loss with dense soft targets, both layouts: fp32 against the oracle (values, per-scale terms, gradients,
    and the objectness / class columns element by element in float64), bf16 and fp16 bit-identical to fp32."""
    B, grids, A, nc = LOSS_CASES[case]
    S = len(grids)
    assert_non_square(grids)
    seed = sum(map(ord, case)) + (0 if regime == "unit" else 1000)
    rng = np.random.default_rng(seed)
    gen = torch.Generator().manual_seed(seed)
    anchors = make_anchors(S, A, seed)
    tgts = dense_targets(B, grids, A, nc, rng)
    for s, t in enumerate(tgts):   # positives on every scale, and the soft objectness values are there
        assert int((t[..., 4] > 0.5).sum()) >= 2, f"scale {s} has no positives"
        assert bool((t[..., 4] == 0.5).any()) and bool((t[..., 4] == np.nextafter(np.float32(0.5), 1)).any())
    heads = loss_heads(B, grids, A, nc, regime, tgts, gen)
    weights = OBJ_WEIGHTS[:S]
    ancs = [a.cuda() for a in anchors]
    tg_d = [t.cuda() for t in tgts]
    hd = [h.cuda() for h in heads]
    for layout in ("bhwac", "nchw"):
        what = f"{case} {regime} {layout}"
        out4, per_scale, grads = run_loss(hd, tg_d, ancs, nc, weights, layout)
        check_loss_vs_oracle(out4, per_scale, grads, heads, tgts, anchors, nc, weights, what)
        check_columns_fp64(grads, heads, tgts, anchors, nc, weights, what)
        if regime == "saturated":   # entries the relative-to-max tolerance cannot see are really there
            g = torch.cat([x[..., 4:].reshape(-1) for x in grads])
            assert bool(((g != 0) & (g.abs() < 1e-5 * g.abs().max())).any())
        for dtype in HALF:
            hh = [h.to(dtype) for h in hd]
            o_h, p_h, g_h = run_loss(hh, tg_d, ancs, nc, weights, layout)
            o_f, p_f, g_f = run_loss([h.float() for h in hh], tg_d, ancs, nc, weights, layout)
            bits_equal(o_h, o_f, f"{what} {dtype} losses")
            bits_equal(p_h, p_f, f"{what} {dtype} per-scale")
            for s, (a, b) in enumerate(zip(g_h, g_f)):
                bits_equal(a, b.to(dtype), f"{what} {dtype} scale {s} gradient")


# ---- 2. label lists, device-side assignment, build_targets (square grids: the reference assigns on G x G) ---------
# (B, grids, A, nc, img_size)
SPARSE_CASES = {
    "s1_a1_nc1": (3, (13,), 1, 1, 104),
    "s2_a5_nc7": (2, (12, 5), 5, 7, 96),
    "s4_a8_nc2": (2, (15, 7, 3, 1), 8, 2, 120),
}


def matched_labels(anchors, img, nc, B, per_scale, rng):
    """Per image, `per_scale` labels whose size is one of scale s's anchors (so that the assignment's best anchor is on
    that scale) for every scale, plus a few random ones and a repeat of the first (same cell: first one wins)."""
    out = []
    for _ in range(B):
        rows = []
        for a in anchors:
            for _ in range(per_scale):
                aw, ah = (float(v) for v in a[rng.integers(0, a.shape[0])])
                rows.append([rng.integers(0, nc), *rng.uniform(0.05, 0.95, 2),
                             aw / img * np.exp(rng.uniform(-0.1, 0.1)), ah / img * np.exp(rng.uniform(-0.1, 0.1))])
        for _ in range(3):
            rows.append([rng.integers(0, nc), *rng.uniform(0.05, 0.95, 2), *np.exp(rng.uniform(np.log(0.01), 0.0, 2))])
        rows.append(list(rows[0]))
        out.append(np.asarray(rows, np.float64))
    return out


@pytest.mark.parametrize("regime", ["unit", "saturated"])
@pytest.mark.parametrize("case", list(SPARSE_CASES))
def test_label_lists_and_build_targets_shapes(yb, case, regime):
    """build_targets bit-exact against the oracle's assignment; the loss on label lists (device-side assignment,
    sparse targets: a bit map for objectness, an entry's class id for the class targets) equal to the loss on
    build_targets' dense targets and to the oracle, with the objectness and class columns also element by element
    in float64, both layouts, bf16 / fp16 bit-identical to fp32."""
    from yolo_from_scratch_b200 import ops
    B, grids, A, nc, img = SPARSE_CASES[case]
    S = len(grids)
    seed = sum(map(ord, case))
    rng = np.random.default_rng(seed)
    anchors = make_anchors(S, A, seed)
    labels = matched_labels(anchors, img, nc, B, 3, rng)
    ref = [R.assign_targets(l, anchors, list(grids), nc, img) for l in labels]
    tg = yb.build_targets(labels, anchors, list(grids), nc, img)
    for s in range(S):
        want = np.stack([r[s] for r in ref])
        assert np.array_equal(tg[s].cpu().numpy(), want), f"build_targets scale {s}"
        assert int((want[..., 4] > 0.5).sum()) > 0, f"scale {s} has no positives"
    ref_tg = [torch.from_numpy(np.stack([r[s] for r in ref])) for s in range(S)]
    gen = torch.Generator().manual_seed(seed)
    if regime == "unit":
        heads = [torch.randn(B, G, G, A, 5 + nc, generator=gen) * 2.0 for G in grids]
    else:
        heads = loss_heads(B, [(G, G) for G in grids], A, nc, regime, ref_tg, gen)
    weights = OBJ_WEIGHTS[:S]
    ancs = [a.cuda() for a in anchors]
    hd = [h.cuda() for h in heads]
    for layout in ("bhwac", "nchw"):
        what = f"{case} {regime} {layout}"
        packed = ops.pack_labels(labels, img)
        o_s, p_s, g_s = run_loss(hd, None, ancs, nc, weights, layout, sparse=packed)
        packed.check()
        o_d, p_d, g_d = run_loss(hd, tg, ancs, nc, weights, layout)
        close(o_s, o_d, rtol=1e-6, atol=1e-7, what=what + " sparse vs dense")
        close(p_s, p_d, rtol=1e-6, atol=1e-7, what=what + " sparse vs dense per-scale")
        for a, b in zip(g_s, g_d):
            close(a, b, rtol=1e-6, atol=1e-10, what=what + " sparse vs dense gradient")
        check_loss_vs_oracle(o_s, p_s, g_s, heads, ref_tg, anchors, nc, weights, what)
        check_columns_fp64(g_s, heads, ref_tg, anchors, nc, weights, what)
        if regime == "saturated":   # entries the relative-to-max tolerance cannot see are really there
            g = torch.cat([x[..., 4:].reshape(-1) for x in g_s])
            assert bool(((g != 0) & (g.abs() < 1e-5 * g.abs().max())).any())
        for dtype in HALF:
            hh = [h.to(dtype) for h in hd]
            o_h, _, g_h = run_loss(hh, None, ancs, nc, weights, layout, sparse=ops.pack_labels(labels, img))
            o_f, _, g_f = run_loss([h.float() for h in hh], None, ancs, nc, weights, layout,
                                   sparse=ops.pack_labels(labels, img))
            bits_equal(o_h, o_f, f"{what} {dtype} losses")
            for a, b in zip(g_h, g_f):
                bits_equal(a, b.to(dtype), f"{what} {dtype} gradient")


# ---- 3. decode --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 5, 11, 1, 6), (1, 1, 9, 8, 12), (3, 13, 4, 8, 5), (2, 7, 3, 1, 85)],
                         ids=lambda s: "x".join(map(str, s)))
def test_decode_shapes(yb, shape):
    """decode_predictions forward and backward at A in {1, 8} on H != W grids against the oracle's decode; bf16 and
    fp16 bit-identical to fp32."""
    B, H, W, A, row = shape
    assert H != W
    gen = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(*shape, generator=gen) * 3
    gout = torch.randn(*shape, generator=gen)
    anc = make_anchors(1, A, sum(shape))[0]
    img = 8 * max(H, W)
    xd = x.cuda().requires_grad_(True)
    y = yb.decode_predictions(xd, anc, img)
    xr = x.clone().requires_grad_(True)
    ref = R.decode(xr, anc, img)
    close(y[..., :4], ref[..., :4], atol=1e-7, what="decode")
    assert torch.equal(y[..., 4:].detach().cpu(), ref[..., 4:].detach())
    y.backward(gout.cuda())
    ref.backward(gout)
    grad_close(xd.grad, xr.grad, what="decode backward")
    for dtype in HALF:
        h = x.to(dtype).cuda()
        p, q = h.clone().requires_grad_(True), h.float().requires_grad_(True)
        oh, of = yb.decode_predictions(p, anc, img), yb.decode_predictions(q, anc, img)
        bits_equal(oh, of.to(dtype), f"{dtype} decode")
        go = gout.to(dtype).cuda()
        oh.backward(go)
        of.backward(go.float())
        bits_equal(p.grad, q.grad.to(dtype), f"{dtype} decode backward")


# ---- 4. single-label and multi-label candidate filters ------------------------------------------------------------
# (B, grids, A, nc); the filters need nc >= 1
FILTER_CASES = {
    "s4_a8_nc1": (2, [(12, 17), (6, 9), (3, 5), (1, 2)], 8, 1),
    "s2_a5_nc7": (3, [(1, 9), (10, 7)], 5, 7),
    "s1_a2_nc80": (2, [(13, 21)], 2, 80),
    "s4_a1_nc2": (2, [(9, 14), (5, 7), (3, 4), (2, 1)], 1, 2),
}


def filter_case(case):
    B, grids, A, nc = FILTER_CASES[case]
    assert_non_square(grids)
    seed = sum(map(ord, case))
    gen = torch.Generator().manual_seed(seed)
    heads = [(torch.randn(B, H, W, A, 5 + nc, generator=gen) * 2.0).cuda() for H, W in grids]
    img = 8 * max(grids[0])
    return heads, make_anchors(len(grids), A, seed), img, nc


def filter_layouts(heads):
    from yolo_from_scratch_b200 import ops
    return (("bhwac", heads, ops.LAYOUT_BHWAC), ("nchw", [to_nchw(h) for h in heads], ops.LAYOUT_NCHW))


@pytest.mark.parametrize("case", list(FILTER_CASES))
def test_filter_shapes(yb, case):
    """filter_candidates against the oracle on CUDA tensors: counts, row order, classes and score bits exact, boxes
    within the filter tests' tolerance; candidates from every scale of every image; bf16 / fp16 bit-identical to fp32."""
    heads, anchors, img, nc = filter_case(case)
    ancs = [a.cuda() for a in anchors]
    conf = 0.25
    B = heads[0].shape[0]
    refs = [R.candidates([h[b:b + 1] for h in heads], ancs, img, nc, conf) for b in range(B)]
    for b in range(B):
        for s, h in enumerate(heads):
            assert R.candidates([h[b:b + 1]], [ancs[s]], img, nc, conf)[1].shape[0] > 0, \
                f"image {b}: no candidates on scale {s}"
    for lay, hs, code in filter_layouts(heads):
        boxes, scores, classes, counts = yb.filter_candidates(hs, ancs, img, nc, conf, layout=code)
        for b, (rb, rs, rc) in enumerate(refs):
            m = int(counts[b])
            what = f"{case} {lay} image {b}"
            assert m == rs.shape[0], f"{what}: {m} candidates, reference {rs.shape[0]}"
            assert torch.equal(classes[b, :m], rc), what + " classes"
            bits_equal(scores[b, :m], rs, what + " scores")
            box_close(boxes[b, :m], rb, what)
        for dtype in HALF:
            a = yb.filter_candidates([h.to(dtype) for h in hs], ancs, img, nc, conf, layout=code)
            f = yb.filter_candidates([h.to(dtype).float() for h in hs], ancs, img, nc, conf, layout=code)
            bits_equal(a[3], f[3], f"{case} {lay} {dtype} counts")
            for b, n in enumerate(a[3].tolist()):
                for x, y in zip(a[:3], f[:3]):
                    bits_equal(x[b, :n], y[b, :n], f"{case} {lay} {dtype} image {b}")


@pytest.mark.parametrize("case", list(FILTER_CASES))
def test_multilabel_filter_shapes(yb, case):
    """filter_candidates_multilabel against the oracle on CUDA tensors, uncapped and with max_candidates inside every
    image's candidate count (the radix select and refine passes run); candidates from every scale of every image;
    bf16 / fp16
    bit-identical to fp32."""
    from yolo_from_scratch_b200 import ops
    heads, anchors, img, nc = filter_case(case)
    ancs = [a.cuda() for a in anchors]
    conf = 0.05
    B = heads[0].shape[0]
    pairs = sum(h.shape[1] * h.shape[2] * h.shape[3] for h in heads) * nc
    full = [ML.candidates_multilabel([h[b:b + 1] for h in heads], ancs, img, nc, conf, pairs) for b in range(B)]
    n_min = min(r[3] for r in full)
    for b in range(B):
        for s, h in enumerate(heads):
            assert ML.candidates_multilabel([h[b:b + 1]], [ancs[s]], img, nc, conf, pairs)[3] > 0, \
                f"image {b}: no candidates on scale {s}"
    K_cap = n_min // 2
    assert 1 <= K_cap < n_min
    for K in (pairs, K_cap):
        refs = full if K == pairs else \
            [ML.candidates_multilabel([h[b:b + 1] for h in heads], ancs, img, nc, conf, K) for b in range(B)]
        for lay, hs, code in filter_layouts(heads):
            boxes, scores, classes, counts, totals = ops.filter_candidates_multilabel(hs, ancs, img, nc, conf,
                                                                                      layout=code, max_candidates=K)
            for b, (rb, rs, rc, n) in enumerate(refs):
                m = int(counts[b])
                what = f"{case} {lay} K={K} image {b}"
                assert int(totals[b]) == n and m == rs.shape[0] == min(n, K), what
                assert torch.equal(classes[b, :m], rc), what + " classes"
                bits_equal(scores[b, :m], rs, what + " scores")
                box_close(boxes[b, :m], rb, what)
            for dtype in HALF:
                a = ops.filter_candidates_multilabel([h.to(dtype) for h in hs], ancs, img, nc, conf, layout=code,
                                                     max_candidates=K)
                f = ops.filter_candidates_multilabel([h.to(dtype).float() for h in hs], ancs, img, nc, conf,
                                                     layout=code, max_candidates=K)
                bits_equal(a[3], f[3], f"{case} {lay} K={K} {dtype} counts")
                bits_equal(a[4], f[4], f"{case} {lay} K={K} {dtype} totals")
                for b, n in enumerate(a[3].tolist()):
                    for x, y in zip(a[:3], f[:3]):
                        bits_equal(x[b, :n], y[b, :n], f"{case} {lay} K={K} {dtype} image {b}")


# ---- 5. eval_epoch's counting -------------------------------------------------------------------------------------
# (B, grids, A, nc)
EVAL_CASES = {
    "s4_a5_nc7": (2, [(12, 17), (6, 9), (3, 5), (2, 1)], 5, 7),
    "s2_a8_nc0": (3, [(1, 9), (10, 7)], 8, 0),
    "s1_a1_nc2": (2, [(13, 21)], 1, 2),
}


@pytest.mark.parametrize("case", list(EVAL_CASES))
def test_eval_counts_shapes(yb, case):
    """eval_counts against the oracle on CUDA tensors.  Rows per scale: predicted and true with the target box equal
    to the decoded prediction up to 1% (a hit), predicted and true with a random box, predicted only, true only; so
    TP, FP and FN are non-zero on every scale, and a box decoded with the wrong grid scale misses."""
    B, grids, A, nc = EVAL_CASES[case]
    assert_non_square(grids)
    seed = sum(map(ord, case))
    rng = np.random.default_rng(seed)
    gen = torch.Generator().manual_seed(seed)
    anchors = [a.cuda() for a in make_anchors(len(grids), A, seed)]
    heads, tgts = [], []
    for (H, W), anc in zip(grids, anchors):
        h = torch.randn(B, H, W, A, 5 + nc, generator=gen).cuda()
        n = B * H * W * A
        kind = torch.from_numpy(rng.integers(0, 5, n)).cuda().reshape(B, H, W, A)   # 0 hit, 1 miss, 2 pred, 3 true, 4 none
        kind.view(-1)[:4] = torch.arange(4, device="cuda")                          # every kind on every scale
        h[..., 4] = torch.where(kind <= 2, 4.0, -4.0)
        dec = R.decode(h, anc, LOSS_IMG)[..., :4]
        t = torch.zeros_like(h)
        t[..., 4] = torch.where((kind == 0) | (kind == 1) | (kind == 3), 1.0, 0.0)
        jitter = 1.0 + 0.01 * (torch.rand(B, H, W, A, 4, generator=gen).cuda() * 2 - 1)
        rand_box = torch.rand(B, H, W, A, 4, generator=gen).cuda() * 0.5 + 0.25
        t[..., :4] = torch.where((kind == 0).unsqueeze(-1), dec * jitter, rand_box)
        heads.append(h)
        tgts.append(t)
    for s in range(len(grids)):
        tp, fp, fn = R.eval_counts([heads[s]], [tgts[s]], [anchors[s]], 0.5, 0.5)
        assert tp > 0 and fp > 0 and fn > 0, f"scale {s}: {(tp, fp, fn)}"
    want = R.eval_counts(heads, tgts, anchors, 0.5, 0.5)
    got = yb.eval_counts(heads, tgts, anchors, 0.5, 0.5)
    assert tuple(int(v) for v in got.cpu()) == tuple(want)
