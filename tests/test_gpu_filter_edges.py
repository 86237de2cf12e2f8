"""The candidate filter's exact decisions at their boundaries (run with -m gpu on the B200 box).

The filter (yb_filter.cu) decides `sigmoid(obj) > conf` from the logit alone outside a band around
logit(conf), and takes the class arg-max in logit space with a re-evaluation window for near-ties.  Both
shortcuts rest on hand-derived bounds.  These tests put logits on and around every boundary and require the
result to equal torch's own arithmetic on the same device: the oracle's `candidates` (and `eval_counts`)
evaluated on CUDA tensors, so that objectness decisions are torch-CUDA's `torch.sigmoid(x) > conf` (an fp32
compare: torch casts the Python threshold to the tensor's dtype) and class ids are torch's `max(dim=1)` (first
index of the maximum, NaN propagated).  Counts, row order, class ids and scores must be exact, scores bit for
bit; boxes keep the tolerance of the other filter tests (the kernel multiplies by 1/W where the reference
divides by W).
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ref_path as R  # noqa: E402  (checker only)

ANCH = R.default_anchors()
IMG = 1024
W_GRID = 128          # grid width of the synthetic single-scale heads; H follows from the number of rows
INF, NAN = float("inf"), float("nan")


@pytest.fixture(scope="module")
def yb():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import yolo_from_scratch_b200 as m
    m._lib.lib()  # fail loudly if the extension is missing
    return m


# ---- fp32 helpers ---------------------------------------------------------------------------------------
def f32(x):
    return np.float32(x)


def ordered_keys(x):
    """fp32 values -> int64 keys that are monotone in the float order (-0 and +0 both map to 0)."""
    b = np.asarray(x, np.float32).reshape(-1).view(np.int32).astype(np.int64)
    return np.where(b >= 0, b, -(b & 0x7fffffff))


def from_keys(k):
    k = np.asarray(k, np.int64)
    return np.where(k >= 0, k, -k - (1 << 31)).astype(np.int32).view(np.float32)


def neighbours(x, span):
    """Every fp32 value within +-span ulps of fp32(x), x itself included."""
    k = int(ordered_keys(f32(x))[0])
    return from_keys(np.arange(k - span, k + span + 1))


def ulps_from(x, n):
    """fp32(x) moved by n ulps (n < 0: towards -inf)."""
    return float(from_keys(ordered_keys(f32(x)) + n)[0])


def obj_band(conf):
    """(logit(conf), margin) of the filter's objectness shortcut (yb_filter.cu, yb_filter_compact: the block that
    sets obj_lo / obj_hi), or None where the shortcut is off and every row evaluates the sigmoid.  The threshold
    reaches the kernel as fp32."""
    c = float(f32(conf))
    if not (1e-4 < c < 1.0 - 1e-4):
        return None
    lg = math.log(c / (1.0 - c))
    m = 64.0 * 4.8e-7 / (c if c < 0.5 else 1.0 - c) + 1e-5 * abs(lg) + 1e-6
    return lg, m


def sigmoid_dev(x):
    """torch's CUDA sigmoid, checked bit for bit against the unfused 1/(1+exp(-x)) that the kernels evaluate
    (sigmoidf_ref, yb_common.cuh)."""
    y = torch.sigmoid(x)
    d = 1.0 + torch.exp(-x)
    plain = torch.ones_like(d) / d
    assert torch.equal(y.view(torch.int32), plain.view(torch.int32)), "torch.sigmoid is not 1/(1+exp(-x)) here"
    return y


def max_ulp_error(x):
    """Largest |sigmoid_fp32(x) - sigmoid(x)| over x (device tensor), in ulps of the fp32 result."""
    y = sigmoid_dev(x)
    ref = 1.0 / (1.0 + torch.exp(-x.double()))
    ulp = torch.nextafter(y, torch.full_like(y, INF)).double() - y.double()
    return float(((y.double() - ref).abs() / ulp).max())


def same_bits(got, want, what):
    """Bit-exact fp32 equality, NaN equal to NaN."""
    got, want = got.contiguous(), want.contiguous()
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    ng, nw = torch.isnan(got), torch.isnan(want)
    bad = (ng != nw) | (~ng & (got.view(torch.int32) != want.view(torch.int32)))
    if bool(bad.any()):
        i = int(bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} mismatches, first at {i}: got {float(got[i])!r}, "
                             f"want {float(want[i])!r}")


def box_close(got, want):
    err = (got.double() - want.double()).abs()
    tol = 1e-5 * want.double().abs() + 2e-4
    assert bool((err <= tol).all()), f"boxes: max err {float(err.max()):.3e}"


# ---- heads ------------------------------------------------------------------------------------------------
def make_head(obj, nc, seed, cls=None, B=1):
    """(B, H, 128, 3, 5+nc) reference-layout head whose objectness channel holds `obj` (B*rows values, image by
    image, padded with NaN, which never passes), class logits `cls` (rows, nc) or random, box logits random."""
    obj = torch.as_tensor(np.asarray(obj, np.float32)).reshape(B, -1)
    n = obj.shape[1]
    H = -(-n // (3 * W_GRID))
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(B, H * W_GRID * 3, 5 + nc, generator=g)
    if nc > 1:
        h[..., 5:] *= 2.0
    h[..., 4] = NAN
    h[:, :n, 4] = obj
    if cls is not None:
        h[:, :n, 5:] = torch.as_tensor(np.asarray(cls, np.float32)).reshape(B, n, nc)
    return h.reshape(B, H, W_GRID, 3, 5 + nc).cuda()


def to_nchw(h):
    B, H, W, A, C = h.shape
    return h.permute(0, 3, 4, 1, 2).reshape(B, A * C, H, W).contiguous()


def reference(h, nc, conf, b=0):
    """The oracle's filter on the CUDA tensor: torch-CUDA's own decisions."""
    rb, rs, rc = R.candidates([h[b:b + 1]], [ANCH[0]], IMG, nc, conf)
    return rb.cuda(), rs.cuda(), rc.cuda()


def check_layouts(yb, h, nc, conf, layouts=("bhwac", "nchw")):
    """Every layout's candidates equal the reference for every image; returns the reference of image 0."""
    from yolo_from_scratch_b200 import ops
    refs = [reference(h, nc, conf, b) for b in range(h.shape[0])]
    for lay in layouts:
        if lay == "nchw":
            out = yb.filter_candidates([to_nchw(h)], [ANCH[0]], IMG, nc, conf, layout=ops.LAYOUT_NCHW)
        else:
            out = yb.filter_candidates([h], [ANCH[0]], IMG, nc, conf)
        boxes, scores, classes, counts = out
        for b, (rb, rs, rc) in enumerate(refs):
            m = int(counts[b])
            what = f"{lay} nc={nc} conf={conf!r} image {b}"
            assert m == rs.shape[0], f"{what}: {m} candidates, reference {rs.shape[0]}"
            cl = classes[b, :m]
            if not torch.equal(cl, rc):
                i = int((cl != rc).nonzero()[0])
                raise AssertionError(f"{what}: class ids differ first at candidate {i}: {int(cl[i])} vs {int(rc[i])}")
            same_bits(scores[b, :m], rs, what + " scores")
            box_close(boxes[b, :m], rb)
    return refs[0]


# ---- thresholds and objectness sweep data -------------------------------------------------------------
SIG_X = 0.3   # a threshold equal to sigmoid(fp32(0.3)) on the device: equality must fail


def thresholds():
    t = [0.001, 0.005, 0.05, 0.1, 0.25, 0.3, 0.4, 0.5, 0.6, 0.7, 0.9, 0.99, 0.9999]
    for edge in (1e-4, 1.0 - 1e-4):   # the shortcut turns on / off between these fp32 neighbours
        t += [ulps_from(edge, -1), float(f32(edge)), ulps_from(edge, 1)]
    t += [0.0, -0.5, 1.0, "sigmoid(0.3)"]
    return t


def conf_value(c):
    if c == "sigmoid(0.3)":
        return float(sigmoid_dev(torch.tensor([SIG_X], device="cuda"))[0])
    return c


def sweep_logits(conf, span=1 << 16, n_rand=1 << 18, seed=0):
    """Every fp32 value within +-span ulps of lg, lg-m and lg+m (the band of obj_band), n_rand uniform floats in
    [lg-8m, lg+8m], and +-0, +-inf, NaN.  Without a band (thresholds <= 1e-4, >= 1-1e-4, 0, negative, 1) the
    centres are where the fp32 sigmoid leaves 0 (expf(-x) overflows; subnormal results) and reaches 1."""
    band = obj_band(conf)
    if band is None:
        centres, lo, hi = [-88.7228, -87.3365, 16.6355], -110.0, 30.0
        if 0.0 < conf < 1.0:
            lg = math.log(conf / (1.0 - conf))
            centres[2], lo, hi = lg, lg - 2.0, lg + 2.0
    else:
        lg, m = band
        centres, lo, hi = [lg, lg - m, lg + m], lg - 8 * m, lg + 8 * m
    rng = np.random.default_rng(seed)
    parts = [neighbours(c, span) for c in centres]
    parts.append(rng.uniform(lo, hi, n_rand).astype(np.float32))
    parts.append(np.array([0.0, -0.0, INF, -INF, NAN], np.float32))
    return np.concatenate(parts)


_BASE = {}


def sweep_head(obj, nc):
    """Random head of the sweep's size, made once per nc; the objectness channel is overwritten per threshold."""
    n = obj.shape[0]
    if (nc, n) not in _BASE:
        _BASE[(nc, n)] = make_head(np.zeros(n, np.float32), nc, seed=11 + nc)
    h = _BASE[(nc, n)]
    flat = h.view(-1, 5 + nc)
    flat[:n, 4] = torch.from_numpy(obj).cuda()
    return h


# ---- (a) the premise of the objectness margin and the tie window ------------------------------------------
def window_floats(lo, hi, chunk=1 << 26):
    """Every fp32 value in [lo, hi], in chunks, on the device."""
    k0, k1 = int(ordered_keys(f32(lo))[0]), int(ordered_keys(f32(hi))[0])
    for s in range(k0, k1 + 1, chunk):
        k = torch.arange(s, min(s + chunk, k1 + 1), device="cuda", dtype=torch.int64)
        yield torch.where(k >= 0, k, -k - (1 << 31)).to(torch.int32).view(torch.float32)


def test_sigmoid_premise_every_float_in_the_bands(yb):
    """DESIGN §3.4: the fp32 sigmoid 1/(1+expf(-x)) is within 4 ulp of the real one.  Checked against fp64 over
    every float of [lg-m, lg+m] for each threshold with a band (for 0.5 that is the ~1.9e9 floats around 0)."""
    worst = {}
    for c in thresholds():
        conf = conf_value(c)
        band = obj_band(conf)
        if band is None:
            continue
        lg, m = band
        e = max(max_ulp_error(x) for x in window_floats(lg - m, lg + m))
        worst[str(c)] = e
        assert e <= 4.0, f"conf {c}: sigmoid error {e:.3f} ulp in the band"
    print("max sigmoid error in ulp per band:", {k: round(v, 3) for k, v in worst.items()})
    print("max over all bands: %.3f ulp" % max(worst.values()))


# ---- (b) objectness boundary sweep ----------------------------------------------------------------------
@pytest.mark.parametrize("c", thresholds(), ids=str)
def test_objectness_boundary_sweep(yb, c):
    """Logits on and around logit(conf) and the band edges in the objectness channel: the reference layout with
    nc=1 (short rows staged in shared memory), nc=8 and nc=80 (long rows, objectness read with __ldg), and NCHW
    (no shortcut), each equal to torch's decisions and scores."""
    conf = conf_value(c)
    obj = sweep_logits(conf)
    x = torch.from_numpy(obj).cuda()
    s = sigmoid_dev(x)
    if c == "sigmoid(0.3)":   # the equality case is really there
        assert bool((s == f32(conf)).any())
    for nc, layouts in ((1, ("bhwac", "nchw")), (8, ("bhwac", "nchw")), (80, ("bhwac",))):
        h = sweep_head(obj, nc)
        rb, rs, rc = check_layouts(yb, h, nc, conf, layouts)
        assert rs.shape[0] == int((s > conf).sum())


# ---- (c) class near-ties --------------------------------------------------------------------------------
TOPS = [-100.0, -89.0, -88.0, -30.0, -1.0, 0.0, 4.99, 5.0, 5.01, 8.0, 13.0, 13.0001, 14.0, 14.0001, 17.0, 20.0,
        88.0, 89.0, INF]


def runner_ups(m):
    """Values below (or equal to) the top logit m that may round to the same probability: 1..64 ulps below m,
    and a few ulps either side of the window edges m-3.1e-4, m-2e-6(1+e^m) and 13 (evaluated in fp32 like the
    kernel)."""
    out = [m] + [ulps_from(m, -k) for k in range(1, 65)]
    mf = f32(m)
    edges = [mf - f32(3.1e-4), f32(13.0)]
    if m <= 14.0:
        edges.append(mf - f32(2e-6) * (f32(1.0) + np.exp(mf)))
    for e in edges:
        if np.isfinite(e):
            out += [ulps_from(e, k) for k in range(-3, 4)]
    return [v for v in out if v <= m]


def placements(nc):
    """(runner-up index, top index) pairs: before and after the top, at index 0, across the 8-wide unrolled
    loop (indices 1..8k) and its tail."""
    p = {(0, nc - 1), (nc - 1, 0), (1, nc - 1), (nc - 1, 1), (nc // 2, nc - 1), (nc - 1, nc // 2)}
    if nc == 80:   # unrolled part 1..72, tail 73..79
        p |= {(10, 40), (40, 10), (74, 78), (78, 74), (5, 75), (75, 5), (0, 30), (0, 77)}
    return sorted(q for q in p if q[0] != q[1])


def tie_rows(nc, seed):
    rng = np.random.default_rng(seed)
    rows = []

    def filler(m):
        if m == -INF:
            return np.full(nc, -INF, np.float32)
        top = min(m, 80.0)
        return (top - rng.uniform(40.0, 60.0, nc)).astype(np.float32)

    for m in TOPS:
        for r in runner_ups(m):
            for ri, mi in placements(nc):
                row = filler(m)
                row[ri], row[mi] = r, m
                rows.append(row)
        if nc >= 3:   # three-way near-ties, in both orders
            a, b = ulps_from(m, -1), ulps_from(m, -2)
            for order in ((b, a, m), (m, a, b), (a, m, b)):
                row = filler(m)
                row[[0, nc // 2, nc - 1]] = order
                rows.append(row)
        row = filler(m)   # an exact tie
        row[[1, nc - 1]] = m
        rows.append(row)
    rows.append(np.full(nc, -INF, np.float32))   # all -inf
    row = np.full(nc, -INF, np.float32)
    row[nc - 1] = -100.0                          # every probability 0
    rows.append(row)
    return np.stack(rows)


@pytest.mark.parametrize("nc", [2, 8, 9, 80])
def test_class_near_ties(yb, nc):
    """Rows that all pass, whose class logits put a runner-up at or just below the top logit m and around each
    re-evaluation window edge: class ids must be torch.max(dim=1)'s first index of the maximal probability."""
    cls = tie_rows(nc, seed=nc)
    n = cls.shape[0]
    x = torch.from_numpy(cls).cuda()
    fin = x[torch.isfinite(x)]
    sample = fin[torch.randperm(fin.numel(), device="cuda")[:1 << 20]]
    sample = sample[sample > -88.7]   # below, expf(-x) overflows and the fp32 result is 0 by construction
    e = max_ulp_error(sample)
    print(f"nc={nc}: {n} tie rows, max sigmoid error on their logits {e:.3f} ulp")
    assert e <= 4.0
    h = make_head(np.full(n, 10.0, np.float32), nc, seed=20 + nc, cls=cls)
    rb, rs, rc = check_layouts(yb, h, nc, 0.5)
    assert rs.shape[0] == n


# ---- (d) staging paths ----------------------------------------------------------------------------------
PASS_COUNTS = (0, 1, 31, 32, 33, 127, 128)


def tile_objectness(scale_rows, B, seed, first_tiles=None):
    """Objectness of B images whose scales have scale_rows rows each.  The kernels tile every scale separately
    (128 rows a tile); tile t of image b (counted over all scales) gets PASS_COUNTS[(t + b) % 7] passing rows,
    capped at the tile's rows, at random positions.  first_tiles[b], where given, replaces the pattern of image b
    by a per-tile count list whose last entry repeats (None: every row passes)."""
    rng = np.random.default_rng(seed)
    obj = np.full((B, sum(scale_rows)), -10.0, np.float32)
    for b in range(B):
        t, base = 0, 0
        for rows in scale_rows:
            for lo in range(0, rows, 128):
                hi = min(rows, lo + 128)
                if first_tiles is not None and b < len(first_tiles):
                    spec = first_tiles[b]
                    k = hi - lo if spec is None else spec[min(t, len(spec) - 1)]
                else:
                    k = PASS_COUNTS[(t + b) % len(PASS_COUNTS)]
                k = min(k, hi - lo)
                obj[b, base + lo + rng.choice(hi - lo, k, replace=False)] = 10.0
                t += 1
            base += rows
    return obj


def multi_scale(obj_rows, grids, nc, seed):
    """Split per-image objectness (B, rows) into reference-layout heads of the given grids (3 anchors)."""
    B = obj_rows.shape[0]
    g = torch.Generator().manual_seed(seed)
    heads, off = [], 0
    for G in grids:
        gh, gw = G if isinstance(G, tuple) else (G, G)
        n = gh * gw * 3
        h = torch.randn(B, n, 5 + nc, generator=g)
        h[..., 4] = torch.from_numpy(obj_rows[:, off:off + n])
        heads.append(h.reshape(B, gh, gw, 3, 5 + nc).cuda())
        off += n
    return heads


def check_multi(yb, heads, nc, conf=0.5):
    from yolo_from_scratch_b200 import ops
    anc = ANCH[:len(heads)]
    img = 8 * heads[0].shape[2]
    for lay in ("bhwac", "nchw"):
        if lay == "nchw":
            boxes, scores, classes, counts = yb.filter_candidates([to_nchw(h) for h in heads], anc, img, nc, conf,
                                                                  layout=ops.LAYOUT_NCHW)
        else:
            boxes, scores, classes, counts = yb.filter_candidates(heads, anc, img, nc, conf)
        for b in range(heads[0].shape[0]):
            rb, rs, rc = R.candidates([h[b:b + 1] for h in heads], anc, img, nc, conf)
            m = int(counts[b])
            what = f"{lay} nc={nc} image {b}"
            assert m == rs.shape[0], f"{what}: {m} candidates, reference {rs.shape[0]}"
            assert torch.equal(classes[b, :m], rc.cuda()), what + ": class ids"
            same_bits(scores[b, :m], rs.cuda(), what + " scores")
            box_close(boxes[b, :m], rb.cuda())


@pytest.mark.parametrize("nc", [1, 2, 7, 8, 80, 395, 396, 1000])
def test_staging_ragged_grids(yb, nc):
    """Tiles with 0, 1, 31, 32, 33, 127 and 128 passing rows (the long-row kernel stages a tile from 32 of 128
    on).  nc=7 stages exactly 48 KB per group, nc=8 is the first long-row case, nc=395 the last whose tile fits
    the staging buffer, nc>=396 reads global memory only.  Grids (13,7,5) x 3 anchors leave last tiles of 123,
    19 and 75 rows and odd images misaligned, so the bulk copy's 16-byte test fails for some tiles."""
    grids, B = (13, 7, 5), 3
    obj = tile_objectness([3 * G * G for G in grids], B, seed=nc)
    check_multi(yb, multi_scale(obj, grids, nc, seed=nc), nc)


@pytest.mark.parametrize("nc", [1, 80])
def test_staging_many_groups_look_back(yb, nc):
    """106x106x3 = 33,708 rows per image: 264 tiles, 33 groups of 8 tiles, so the decoupled look-back of the
    last groups walks more than one window of 32 predecessors."""
    obj = tile_objectness([106 * 106 * 3], 2, seed=7)
    check_multi(yb, multi_scale(obj, (106,), nc, seed=70 + nc), nc)


@pytest.mark.parametrize("nc", [80, 395, 396])
def test_staging_speculative_copy(yb, nc):
    """Images 0-2 have every row passing; image 3 has an empty first tile and dense later tiles, image 4 a first
    tile with one passing row and nothing dense, image 5 nothing at all.  Long-row CTAs that start after dense
    groups have finished issue a speculative bulk copy of their first tile; with the later images that copy lands
    in an empty tile (and must complete before the next copy), turns out useful for a sparse tile, or is not
    needed at all.  Which CTAs see a dense history depends on scheduling and cannot be forced, so these paths
    are made likely rather than certain."""
    G, B = 32, 6
    first = [None, None, None, [0, 128, 33, 32], [1, 0], [0]]
    obj = tile_objectness([3 * G * G], B, seed=nc, first_tiles=first)   # 24 tiles, 3 groups
    check_multi(yb, multi_scale(obj, (G,), nc, seed=90 + nc), nc)


# ---- (e) eval threshold ---------------------------------------------------------------------------------
@pytest.mark.parametrize("conf", [0.5, 0.25, 0.1, "below sigmoid(0.3)"], ids=str)
def test_eval_counts_objectness_sweep(yb, conf):
    """eval_epoch's counting compares sigmoid(obj) with the threshold in double (`.item()` gives a Python float),
    the filter in fp32.  The objectness sweeps across logit(conf); counts must equal the oracle's on CUDA
    tensors.  The last case is a threshold just below an fp32 sigmoid value s: eval counts that row (s > conf in
    double) while the filter does not (fp32(conf) == s)."""
    if conf == "below sigmoid(0.3)":
        s = conf_value("sigmoid(0.3)")
        conf = float(np.nextafter(s, -INF))
        x0 = f32(SIG_X)
    else:
        x0 = None
    lg = math.log(conf / (1.0 - conf))
    rng = np.random.default_rng(3)
    obj = np.concatenate([neighbours(lg, 1 << 12), rng.uniform(lg - 0.01, lg + 0.01, 1 << 14).astype(np.float32),
                          np.array([0.0, INF, -INF, NAN, SIG_X], np.float32)])
    n = obj.shape[0]
    h = make_head(obj, 1, seed=5)
    t = torch.zeros_like(h)
    flat = t.view(-1, 6)
    flat[0::2, 4] = 1.0                     # every other row is a target: both FP and FN are populated
    flat[:, 0:4] = torch.rand(flat.shape[0], 4, device="cuda") * 0.5 + 0.25
    want = R.eval_counts([h], [t], [ANCH[0]], conf, 0.5)
    got = yb.eval_counts([h], [t], [ANCH[0]], conf, 0.5)
    assert tuple(int(v) for v in got.cpu()) == tuple(want)
    if x0 is not None:
        one = make_head(np.array([x0], np.float32), 1, seed=6)
        t1 = torch.zeros_like(one)
        e1 = yb.eval_counts([one], [t1], [ANCH[0]], conf, 0.5)
        assert tuple(int(v) for v in e1.cpu()) == (0, 1, 0) == R.eval_counts([one], [t1], [ANCH[0]], conf, 0.5)
        assert int(yb.filter_candidates([one], [ANCH[0]], IMG, 1, conf)[3][0]) == 0
        assert R.candidates([one], [ANCH[0]], IMG, 1, conf)[1].shape[0] == 0
    assert n > 0


# ---- (f) NaN and +-inf class logits ----------------------------------------------------------------------
def nan_rows(nc, seed):
    rng = np.random.default_rng(seed)
    specs = [{0: NAN}, {nc // 2: NAN}, {nc - 1: NAN}, {1: NAN, nc - 2: NAN}, {1: INF, nc - 1: NAN},
             {nc - 1: INF, 1: NAN}, {nc // 2: INF}, {0: -INF, nc - 1: INF}, {0: INF, 1: INF}]
    rows = []
    for spec in specs:
        for rep in range(4):
            row = (rng.standard_normal(nc) * 2).astype(np.float32)
            if rep == 1:
                row[:] = -INF
            elif rep == 2:
                row[:] = 20.0
            for i, v in spec.items():
                row[min(i, nc - 1)] = v
            rows.append(row)
    return np.stack(rows)


@pytest.mark.parametrize("nc", [2, 9, 80])
def test_nan_and_inf_class_logits(yb, nc):
    """torch.max(dim=1) propagates NaN and returns the first NaN's index, so the candidate's score is NaN; +inf
    ties with +inf and with logits whose probability rounds to 1.  Both layouts."""
    cls = nan_rows(nc, seed=nc)
    h = make_head(np.full(cls.shape[0], 3.0, np.float32), nc, seed=30 + nc, cls=cls)
    check_layouts(yb, h, nc, 0.5)


# ---- (g) end to end -------------------------------------------------------------------------------------
def tv_keep(rb, rs, rc, iou):
    import torchvision
    if rs.numel() == 0:
        return torch.zeros(0, dtype=torch.int64, device="cuda")
    return torchvision.ops.batched_nms(rb, rs, rc, iou)


@pytest.mark.parametrize("case", ["sweep", "nan"])
def test_detect_batch_keep_sets_on_edge_data(yb, case):
    """detect_batch keep sets equal torchvision.ops.batched_nms on the CUDA reference's candidates: the sweep data
    of the boundary test (with +-2^9 ulps and 2^12 random logits per threshold, so that torchvision's dense
    NMS stays small) at nc=8, and the NaN/inf class rows at nc=9."""
    runs = []
    if case == "sweep":
        for c in thresholds():
            conf = conf_value(c)
            obj = sweep_logits(conf, span=1 << 9, n_rand=1 << 12, seed=1)
            runs.append((make_head(obj, 8, seed=40), 8, conf))
    else:
        cls = nan_rows(9, seed=2)
        runs.append((make_head(np.full(cls.shape[0], 3.0, np.float32), 9, seed=41, cls=cls), 9, 0.5))
    for h, nc, conf in runs:
        det = yb.detect_batch([h], [ANCH[0]], IMG, nc, conf, 0.4)
        rb, rs, rc = reference(h, nc, conf)
        m, k = int(det["counts"][0]), int(det["n_keep"][0])
        assert m == rs.shape[0]
        want = tv_keep(rb, rs, rc, 0.4)
        got = det["keep"][0, :k]
        assert torch.equal(got, want), f"conf {conf!r}: keep sets differ ({k} vs {want.numel()})"
