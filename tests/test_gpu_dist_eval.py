"""compute(group) of DetectionMAP, COCODetectionEval and DetectionReport, and train.evaluate_* with a group, against
one process that sees every image.

Every rank runs in its own spawned process (tests/test_dist_eval_cpu.py's run_ranks: process-group timeout, joined
with a deadline, no child left behind).  With gloo every rank shares cuda:0 and the collectives carry CUDA tensors,
so the merge is tested on one GPU; the NCCL case needs two.  The data are the synthetic batches of the single-process
GPU tests, taken image by image so that the ranks and the single process can use different batch sizes.  With
contiguous shards (dist.shard_range) every field must equal the single process's bit for bit."""
import types

import numpy as np
import pytest
import torch

from yolo_from_scratch_b200 import ops
from oracle import ref_path as R
import eval_data as E
from test_dist_eval_cpu import run_ranks

pytestmark = pytest.mark.gpu
KINDS = ("map", "coco", "report")
GENERATORS = {"map": E.synthetic_batch, "coco": E.coco_synthetic_batch, "report": E.synthetic_batch}
CUSTOM_THR = (0.3, 0.6, 0.75)
CUSTOM_REC = tuple(np.linspace(0.0, 1.0, 11).tolist())
COUNT_KEYS = {"map": ("n_gt", "n_det", "recall"), "coco": ("n_gt", "n_det", "recall"),
              "report": ("n_gt", "n_det", "recall", "confusion", "images", "images_total", "px", "p_curve", "r_curve",
                         "f1_curve", "best_conf", "p", "r", "f1")}


def make_metric(kind, nc, params="default", **over):
    """The metric of `kind` with default or custom thresholds, max_det, maxDets and confidence grid; `over` replaces
    single arguments (a rank that disagrees with the others)."""
    custom = params == "custom"
    if kind == "map":
        kw = dict(iou_thresholds=CUSTOM_THR, recall_thresholds=CUSTOM_REC, max_det=50) if custom else {}
        return ops.DetectionMAP(nc, **{**kw, **over})
    if kind == "coco":
        kw = (dict(iou_thresholds=CUSTOM_THR, recall_thresholds=CUSTOM_REC, max_det=50, max_dets=(1, 5, 20))
              if custom else {})
        return ops.COCODetectionEval(nc, **{**kw, **over})
    kw = dict(iou_thresholds=CUSTOM_THR, max_det=50, conf_grid=E.CUSTOM_GRID, curve_iou=0.75, cm_conf=0.6,
              cm_iou=0.3) if custom else {}
    return ops.DetectionReport(nc, **{**kw, **over})


def make_images(kind, nc, n, seed):
    rng = np.random.default_rng(seed)
    det, _, (labels, lb) = GENERATORS[kind](rng, n, nc, 30, 120)
    return det, list(labels), list(lb)


def batches(data, idx, batch):
    """(det, PackedLabels) of the images `idx` in batches of `batch`, built before any update."""
    det, labels, lb = data
    out = []
    for i0 in range(0, len(idx), batch):
        sel = idx[i0:i0 + batch]
        t = torch.tensor(sel, dtype=torch.int64, device=det["boxes"].device)
        out.append(({k: v.index_select(0, t) for k, v in det.items()},
                    E.packed([labels[i] for i in sel], [lb[i] for i in sel])))
    return out


def feed(metric, data, idx, batch, no_sync=False):
    """update() over the images `idx`; with no_sync, under torch's sync debug mode "error" (test_gpu_map's check)."""
    work = batches(data, idx, batch)
    torch.cuda.synchronize()
    if no_sync:
        torch.cuda.set_sync_debug_mode("error")
    try:
        for d, lab in work:
            metric.update(d, lab)
    finally:
        torch.cuda.set_sync_debug_mode(0)


def shard(n, rank, world, interleave):
    from yolo_from_scratch_b200.dist import shard_range
    return list(range(rank, n, world)) if interleave else list(range(*shard_range(n, rank, world)))


def single(c):
    """One process over every image, in batches of c["single_batch"]."""
    metric = make_metric(c["kind"], c["nc"], c["params"])
    feed(metric, make_images(c["kind"], c["nc"], c["n"], c["seed"]), list(range(c["n"])), c["single_batch"])
    return metric.compute()


def assert_same(got, want, keys=None):
    assert set(got) == set(want)
    for k in keys or want:
        a, b = got[k], want[k]
        if isinstance(b, np.ndarray):
            assert isinstance(a, np.ndarray) and a.dtype == b.dtype and np.array_equal(a, b), k
        else:
            assert type(a) is type(b) and a == b, (k, a, b)


def _warm_up():
    """First launches load the library and its modules; the sync check starts after them."""
    data = make_images("report", 3, 2, 0)
    for kind in KINDS:
        m = make_metric(kind, 3)
        feed(m, data, [0, 1], 2)
        m.compute()


def eval_worker(rank, world, group, cases):
    """Per case: this rank's shard, update() never synchronising, then compute(group) twice and compute() before and
    after: compute(group) must not change the local state."""
    _warm_up()
    out = []
    for c in cases:
        metric = make_metric(c["kind"], c["nc"], c["params"])
        idx = shard(c["n"], rank, world, c["interleave"])
        feed(metric, make_images(c["kind"], c["nc"], c["n"], c["seed"]), idx, c["batch"], no_sync=True)
        local = metric.compute()
        got = metric.compute(group)
        assert_same(metric.compute(group), got)
        assert_same(metric.compute(), local)
        out.append((len(idx), got, local))
    return out


def cases_for(world, n, nc_list=(1, 3, 80), params_list=("default", "custom"), interleave=False):
    return [dict(kind=k, nc=nc, params=p, n=n, seed=1000 * nc + 10 * KINDS.index(k) + len(p), batch=4, single_batch=5,
                 interleave=interleave) for k in KINDS for nc in nc_list for p in params_list]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_compute_is_bit_exact(world):
    """Uneven contiguous shards (13 images over 2 ranks, 17 over 3) in batches of 4 against one process in batches of
    5, for the three metrics at nc 1, 3 and 80 with default and custom arguments; at world 3 also 2 images, so that
    rank 2 has none.  Every rank's update() runs under the sync check."""
    cases = cases_for(world, {2: 13, 3: 17}[world])
    if world == 3:
        cases += [dict(kind=k, nc=3, params=p, n=2, seed=7, batch=4, single_batch=1, interleave=False)
                  for k in KINDS for p in ("default", "custom")]
    res = run_ranks(eval_worker, world, (cases,))
    for i, c in enumerate(cases):
        want = single(c)
        sizes = [res[r][i][0] for r in range(world)]
        assert sum(sizes) == c["n"] and (c["n"] > 2 or sizes[-1] == 0)
        for r in range(world):
            assert_same(res[r][i][1], want)
        if c["kind"] == "report":
            assert want["images_total"] == c["n"] and res[0][i][2]["images_total"] == sizes[0]
        if c["n"] > 2:
            assert want["n_det"].sum() > 0 and want["n_gt"].sum() > 0


def test_world_size_one_equals_compute():
    cases = cases_for(1, 9, nc_list=(3,))
    res = run_ranks(eval_worker, 1, (cases,))
    for i, c in enumerate(cases):
        n, got, local = res[0][i]
        assert n == 9
        assert_same(got, local)
        assert_same(got, single(c))


def test_interleaved_shards_keep_every_count():
    """DistributedSampler's assignment (image i on rank i % world): the counts and everything taken from them are
    identical; only the precision table may differ, through the order of equal scores of different images."""
    cases = cases_for(3, 17, nc_list=(3, 80), params_list=("default",), interleave=True)
    res = run_ranks(eval_worker, 3, (cases,))
    for i, c in enumerate(cases):
        want = single(c)
        for r in range(3):
            assert_same(res[r][i][1], want, keys=COUNT_KEYS[c["kind"]])


MISMATCHES = [("map", dict(nc=4)), ("map", dict(max_det=100)), ("map", dict(iou_thresholds=(0.5, 0.75))),
              ("map", dict(recall_thresholds=CUSTOM_REC)), ("coco", dict(max_dets=(1, 10, 50))),
              ("coco", dict(max_det=299)), ("report", dict(cm_conf=0.3)), ("report", dict(curve_iou=0.75)),
              ("report", dict(conf_grid=np.linspace(0.0, 1.0, 100))), ("report", dict(nc=5))]


def mismatch_worker(rank, world, group):
    """Rank 1 builds each metric with one argument changed.  Every rank must raise ValueError from compute(group);
    a matching compute(group) afterwards shows that no rank was left inside a collective."""
    _warm_up()
    data = make_images("report", 3, 9, 11)
    idx = shard(9, rank, world, False)
    out = []
    for kind, over in MISMATCHES:
        kw = dict(over) if rank == 1 else {}
        metric = make_metric(kind, kw.pop("nc", 3), **kw)
        feed(metric, data, idx, 4)
        try:
            metric.compute(group)
            out.append(None)
        except Exception as e:   # the type is what the test checks
            out.append((type(e).__name__, str(e)))
    metric = make_metric("report", 3)
    feed(metric, data, idx, 4)
    return out, metric.compute(group)["images_total"]


def test_configuration_mismatch_raises_on_every_rank():
    res = run_ranks(mismatch_worker, 2, timeout_s=300)
    for errors, images_total in res:
        for (kind, over), err in zip(MISMATCHES, errors):
            assert err is not None and err[0] == "ValueError", (kind, over, err)
            assert "configurations differ" in err[1]
        assert images_total == 9


def bad_class_worker(rank, world, group):
    """Rank 1's first image has a ground truth of class 5 with nc = 3: every rank must raise IndexError."""
    _warm_up()
    out = []
    for kind in KINDS:
        det, labels, lb = make_images(kind, 3, 9, 12)
        idx = shard(9, rank, world, False)
        if rank == 1:
            labels[idx[0]] = np.array([[5, 0.5, 0.5, 0.2, 0.2]])
        metric = make_metric(kind, 3)
        feed(metric, (det, labels, lb), idx, 4)
        try:
            metric.compute(group)
            out.append(None)
        except Exception as e:
            out.append(type(e).__name__)
    return out


def test_bad_class_on_one_rank_raises_on_every_rank():
    for errors in run_ranks(bad_class_worker, 2, timeout_s=300):
        assert errors == ["IndexError"] * len(KINDS)


class _ImageHeads(E._PresetHeads):
    """Preset heads selected by image: image i is filled with the pixel value i, so each image gets the same heads
    whichever rank and batch it is in."""

    def __call__(self, img):
        idx = (img[:, 0, 0, 0] * 255).round().long()
        return [h[idx] for h in self.heads]


NC, IMG, N_FILES = 3, 160, 7
LETTERBOX = (0.8, 16, 0)


def write_dataset(path):
    """N_FILES images of 200x160 with their label files; image 4 has no label file."""
    from PIL import Image
    rng = np.random.default_rng(13)
    imgs, lab_files = [], []
    for i in range(N_FILES):
        p = path / f"im{i}.png"
        Image.fromarray(np.full((160, 200, 3), i, dtype=np.uint8)).save(p)
        imgs.append(str(p))
        lf = path / f"im{i}.txt"
        lab = np.column_stack([rng.integers(0, NC, 4), rng.uniform(0.2, 0.8, (4, 2)), rng.uniform(0.05, 0.4, (4, 2))])
        if i != 4:
            with open(lf, "w") as f:
                for r in lab:
                    f.write(f"{int(r[0])} {r[1]} {r[2]} {r[3]} {r[4]}\n")
        lab_files.append(str(lf))
    return types.SimpleNamespace(imgs=imgs, labels=lab_files)


def evaluate_all(dataset, batch_size, group=None):
    from yolo_from_scratch_b200.install import install, uninstall
    model = _ImageHeads(E.prior_heads(N_FILES, IMG, NC, 7), IMG, [a.cuda() for a in R.default_anchors()])
    train = install(E._train_stand_in(*LETTERBOX))
    try:
        dev = torch.device("cuda")
        return [train.evaluate_map(model, dataset, dev, num_classes=NC, batch_size=batch_size, group=group),
                train.evaluate_coco(model, dataset, dev, num_classes=NC, batch_size=batch_size, max_dets=(1, 5, 50),
                                    group=group),
                train.evaluate_report(model, dataset, dev, num_classes=NC, batch_size=batch_size, group=group)]
    finally:
        uninstall(train)


def evaluate_worker(rank, world, group, imgs, labels):
    return evaluate_all(types.SimpleNamespace(imgs=imgs, labels=labels), 2, group)


def test_evaluate_through_install_with_group(tmp_path):
    dataset = write_dataset(tmp_path)
    want = evaluate_all(dataset, 3)
    assert want[2]["images_total"] == N_FILES and want[0]["n_gt"].sum() == 24 and want[0]["n_det"].sum() > 0
    for got in run_ranks(evaluate_worker, 2, (dataset.imgs, dataset.labels)):
        for g, w in zip(got, want):
            assert_same(g, w)


def test_nccl_sharded_compute_is_bit_exact():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cases = cases_for(2, 13, nc_list=(3, 80), params_list=("default",))
    res = run_ranks(eval_worker, 2, (cases,), backend="nccl")
    for i, c in enumerate(cases):
        want = single(c)
        for r in range(2):
            assert_same(res[r][i][1], want)
