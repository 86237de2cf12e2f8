"""Generates tests/golden/*.npz by running the UNMODIFIED reference (/root/reference/train.py) and
the installed torchvision on seeded inputs.  Run in the build container only:

    python oracle/make_golden.py

The reference cannot travel to the GPU box, so the vectors are committed.  Inputs are stored next
to the reference's outputs; nothing here is product code.
"""
import os
import sys
import tempfile

import numpy as np
import torch

REF = "/root/reference"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)
import train as ref  # noqa: E402  the reference itself
import torchvision  # noqa: E402
from PIL import Image  # noqa: E402
from oracle.golden_store import pack_seeded_randn  # noqa: E402  seeded randn inputs stored compactly


def gen(seed):
    g = torch.Generator()
    g.manual_seed(seed)
    return g


def anchors3():
    return [torch.tensor(a, dtype=torch.float32) for a in (
        [[10, 13], [16, 30], [33, 23]], [[30, 61], [62, 45], [59, 119]], [[116, 90], [156, 198], [373, 326]])]


def golden_decode():
    out = {}
    cases = [("g13_nc1", 2, 13, 13, 1, 416), ("g20_nc3", 1, 20, 20, 3, 640), ("g7x5_nc0", 3, 7, 5, 0, 640),
             ("g12_nc80", 1, 12, 12, 80, 1280)]
    for name, B, H, W, nc, img in cases:
        x = (torch.randn(B, H, W, 3, 5 + nc, generator=gen(11)) * 2.0).requires_grad_(True)
        anc = anchors3()[1]
        y = ref.decode_predictions(x, anc, img)
        w = torch.randn(y.shape, generator=gen(12))
        (y * w).sum().backward()
        out[f"{name}_in"] = x.detach().numpy()
        out[f"{name}_img"] = np.array(img)
        out[f"{name}_out"] = y.detach().numpy()
        out[f"{name}_gout"] = w.numpy()
        out[f"{name}_gin"] = x.grad.numpy()
    out["anchors"] = anchors3()[1].numpy()
    np.savez_compressed(os.path.join(OUT, "decode.npz"), **out)


def golden_ciou():
    g = gen(21)
    n = 96
    p = torch.rand(n, 4, generator=g) * torch.tensor([1.0, 1.0, 0.5, 0.5]) + torch.tensor([0, 0, 0.01, 0.01])
    t = torch.rand(n, 4, generator=g) * torch.tensor([1.0, 1.0, 0.5, 0.5]) + torch.tensor([0, 0, 0.01, 0.01])
    # hand-made edge cases: identical, disjoint, contained, touching edges, shared corner
    p[0], t[0] = torch.tensor([0.5, 0.5, 0.2, 0.3]), torch.tensor([0.5, 0.5, 0.2, 0.3])
    p[1], t[1] = torch.tensor([0.1, 0.1, 0.1, 0.1]), torch.tensor([0.9, 0.9, 0.1, 0.1])
    p[2], t[2] = torch.tensor([0.5, 0.5, 0.1, 0.1]), torch.tensor([0.5, 0.5, 0.4, 0.4])
    p[3], t[3] = torch.tensor([0.25, 0.5, 0.5, 0.5]), torch.tensor([0.75, 0.5, 0.5, 0.5])
    p[4], t[4] = torch.tensor([0.5, 0.5, 0.2, 0.4]), torch.tensor([0.5, 0.5, 0.4, 0.2])
    p = p.clone().requires_grad_(True)
    t = t.clone().requires_grad_(True)
    loss = ref.ciou_loss(p, t)
    loss.backward()
    np.savez_compressed(os.path.join(OUT, "ciou.npz"), pred=p.detach().numpy(), tgt=t.detach().numpy(),
                        loss=loss.detach().numpy(), gpred=p.grad.numpy(), gtgt=t.grad.numpy())


def random_labels(rng, n, nc):
    lab = np.zeros((n, 5), dtype=np.float64)
    lab[:, 0] = rng.integers(0, max(nc, 1), size=n)
    lab[:, 1:3] = rng.uniform(0.05, 0.95, size=(n, 2))
    lab[:, 3:5] = np.exp(rng.uniform(np.log(0.01), np.log(0.6), size=(n, 2)))
    return lab


def reference_targets(labels, orig_wh, img_size, nc, anchors=None):
    """Runs the reference's YOLODataset.__getitem__ on a real image file + label file."""
    with tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "images"))
        os.makedirs(os.path.join(tmp, "labels"))
        Image.fromarray(np.zeros((orig_wh[1], orig_wh[0], 3), dtype=np.uint8)).save(os.path.join(tmp, "images", "a.png"))
        with open(os.path.join(tmp, "labels", "a.txt"), "w") as f:
            for r in labels:
                f.write(f"{int(r[0])} {float(r[1])!r} {float(r[2])!r} {float(r[3])!r} {float(r[4])!r}\n")
        ds = ref.YOLODataset(os.path.join(tmp, "images"), num_classes=nc, anchors=anchors, img_size=img_size)
        _, targets = ds[0]
        pil = Image.open(os.path.join(tmp, "images", "a.png")).convert("RGB")
        _, scale, pad_top, pad_left = ref.letterbox_resize(pil, img_size)
    return [t.numpy() for t in targets], (orig_wh[0], orig_wh[1], scale, pad_top, pad_left)


def golden_targets():
    rng = np.random.default_rng(31)
    out = {}
    cases = [("a", (640, 640), 640, 1, 50), ("b", (500, 375), 640, 3, 37), ("c", (300, 480), 416, 1, 12),
             ("d", (1280, 720), 640, 80, 50), ("e", (640, 640), 640, 1, 0), ("f", (640, 480), 320, 2, 200)]
    for name, wh, img, nc, n in cases:
        lab = random_labels(rng, n, nc)
        if name == "f":  # force slot collisions: many boxes in few cells
            lab[:, 1:3] = rng.uniform(0.4, 0.6, size=(n, 2))
        tg, lb = reference_targets(lab, wh, img, nc)
        out[f"{name}_labels"] = lab
        out[f"{name}_letterbox"] = np.array(lb, dtype=np.float64)
        out[f"{name}_cfg"] = np.array([img, nc])
        for s, t in enumerate(tg):
            nz = np.argwhere(t[..., 4] > 0)
            out[f"{name}_s{s}_idx"] = nz.astype(np.int32)
            out[f"{name}_s{s}_rows"] = t[nz[:, 0], nz[:, 1], nz[:, 2]] if len(nz) else np.zeros((0, 5 + nc), np.float32)
            assert np.count_nonzero(t) == np.count_nonzero(out[f"{name}_s{s}_rows"])
    # single-anchor-set back-compat (identical anchors on all scales -> first scale wins ties)
    lab = random_labels(rng, 20, 1)
    tg, lb = reference_targets(lab, (640, 640), 640, 1, anchors=[[10, 13], [16, 30], [33, 23]])
    out["g_labels"], out["g_letterbox"], out["g_cfg"] = lab, np.array(lb, dtype=np.float64), np.array([640, 1])
    for s, t in enumerate(tg):
        nz = np.argwhere(t[..., 4] > 0)
        out[f"g_s{s}_idx"] = nz.astype(np.int32)
        out[f"g_s{s}_rows"] = t[nz[:, 0], nz[:, 1], nz[:, 2]] if len(nz) else np.zeros((0, 6), np.float32)
    # compute_anchor_iou known values
    ds_anch = anchors3()
    wh = torch.tensor([[50.0, 60.0], [10.0, 13.0], [400.0, 20.0], [0.0, 0.0], [33.5, 22.75]])
    dummy = ref.YOLODataset.__new__(ref.YOLODataset)
    out["aiou_wh"] = wh.numpy()
    out["aiou"] = np.stack([np.stack([dummy.compute_anchor_iou(w, a).numpy() for a in ds_anch]) for w in wh])
    np.savez_compressed(os.path.join(OUT, "targets.npz"), **out)


def dense_targets_from_labels(B, img, nc, rng, max_n):
    ts = None
    for b in range(B):
        lab = random_labels(rng, int(rng.integers(0, max_n + 1)), nc)
        tg, _ = reference_targets(lab, (img, img), img, nc)
        if ts is None:
            ts = [[] for _ in tg]
        for s, t in enumerate(tg):
            ts[s].append(torch.from_numpy(t))
    return [torch.stack(x) for x in ts]


def golden_loss():
    out = {}
    rng = np.random.default_rng(41)
    for name, B, img, nc in [("nc1", 3, 160, 1), ("nc3", 2, 224, 3), ("nc80", 2, 128, 80)]:
        grids = [img // 8, img // 16, img // 32]
        tgts = dense_targets_from_labels(B, img, nc, rng, 12)
        preds = [torch.randn(B, g, g, 3, 5 + nc, generator=gen(50 + s)).requires_grad_(True) for s, g in enumerate(grids)]
        res = ref.yolo_loss_multiscale(preds, tgts, anchors3(), nc)
        res[0].backward()
        out[f"{name}_cfg"] = np.array([B, img, nc])
        out[f"{name}_losses"] = np.array([float(r) for r in res], dtype=np.float32)
        for s in range(3):
            out.update(pack_seeded_randn(f"{name}_pred{s}", preds[s].detach().numpy(), 50 + s))
            out[f"{name}_tgt{s}"] = tgts[s].numpy()
            out[f"{name}_grad{s}"] = preds[s].grad.numpy()
        # single-scale yolo_loss on scale 1 (weights 0.05/1.0/0.5)
        p1 = preds[1].detach().clone().requires_grad_(True)
        r1 = ref.yolo_loss(p1, tgts[1], anchors3()[1], nc)
        r1[0].backward()
        out[f"{name}_single_losses"] = np.array([float(r) for r in r1], dtype=np.float32)
        out[f"{name}_single_grad"] = p1.grad.numpy()
    # a scale with no positives at all (bbox = cls = 0.0, train.py:820,:832)
    preds = [torch.randn(1, g, g, 3, 6, generator=gen(60 + s)) for s, g in enumerate([8, 4, 2])]
    tgts = [torch.zeros_like(p) for p in preds]
    res = ref.yolo_loss_multiscale(preds, tgts, anchors3(), 1)
    out["empty_losses"] = np.array([float(r) for r in res], dtype=np.float32)
    for s in range(3):
        out.update(pack_seeded_randn(f"empty_pred{s}", preds[s].numpy(), 60 + s))
    np.savez_compressed(os.path.join(OUT, "loss.npz"), **out)


class FakeModel:
    """Stands in for YOLO inside the reference's predict(): returns preset heads."""

    def __init__(self, heads, img_size, anchors):
        self.heads, self.img_size, self.anchors = heads, img_size, anchors

    def eval(self):
        return self

    def __call__(self, img):
        return self.heads


def golden_predict():
    """The reference's own predict() (train.py:1114-1250) on preset heads: filter + letterbox
    reverse + torchvision batched_nms end to end."""
    out = {}
    cases = [("p_nc1", 160, 1, 0.5, (200, 160), 71), ("p_nc3", 224, 3, 0.3, (224, 224), 72),
             ("p_nc80", 128, 80, 0.25, (100, 128), 73), ("p_nc1_dense", 160, 1, 0.001, (160, 160), 74)]
    with tempfile.TemporaryDirectory() as tmp:
        for name, img, nc, conf, wh, seed in cases:
            path = os.path.join(tmp, f"{name}.png")
            Image.fromarray(np.zeros((wh[1], wh[0], 3), dtype=np.uint8)).save(path)
            grids = [img // 8, img // 16, img // 32]
            heads = [torch.randn(1, g, g, 3, 5 + nc, generator=gen(seed * 10 + s)) for s, g in enumerate(grids)]
            model = FakeModel(heads, img, anchors3())
            dets = ref.predict(model, path, torch.device("cpu"), num_classes=nc, conf_threshold=conf, iou_threshold=0.4)
            pil = Image.open(path).convert("RGB")
            _, scale, pad_top, pad_left = ref.letterbox_resize(pil, img)
            out[f"{name}_cfg"] = np.array([img, nc, conf, 0.4, scale, pad_top, pad_left], dtype=np.float64)
            for s in range(3):
                out[f"{name}_head{s}"] = heads[s].numpy()
            out[f"{name}_dets"] = np.array(dets, dtype=np.float64).reshape(-1, 6)
            print(name, "detections", len(dets))
    np.savez_compressed(os.path.join(OUT, "predict.npz"), **out)


def golden_nms():
    """torchvision.ops.nms / batched_nms (CPU kernels of the installed 0.26.0) on seeded boxes."""
    out = {}
    g = gen(81)
    for name, n, nc, span in [("small", 300, 1, 200.0), ("cls", 900, 7, 300.0), ("big", 1500, 3, 400.0),
                              ("neg", 600, 4, 300.0)]:
        xy = torch.rand(n, 2, generator=g) * span - (150.0 if name == "neg" else 0.0)
        wh = torch.rand(n, 2, generator=g) * 80.0 + 1.0
        boxes = torch.cat([xy, xy + wh], dim=1)
        scores = torch.rand(n, generator=g)
        scores[::7] = scores[0]  # ties
        idxs = torch.randint(0, nc, (n,), generator=g)
        out[f"{name}_boxes"], out[f"{name}_scores"], out[f"{name}_idxs"] = boxes.numpy(), scores.numpy(), idxs.numpy()
        for thr in (0.3, 0.4, 0.7):
            out[f"{name}_nms_{thr}"] = torchvision.ops.nms(boxes, scores, thr).numpy()
            out[f"{name}_bnms_{thr}"] = torchvision.ops.batched_nms(boxes, scores, idxs, thr).numpy()
    out["torchvision_version"] = np.array(torchvision.__version__)
    np.savez_compressed(os.path.join(OUT, "nms.npz"), **out)


def golden_model_heads():
    """configs[0]: real random-init 'cone' (nc=1) model heads at 640x640 -> loss + predict."""
    torch.manual_seed(91)
    model = ref.YOLO(num_classes=1, img_size=640)
    model.eval()
    img = torch.rand(1, 3, 640, 640, generator=gen(92))
    with torch.no_grad():
        heads = model(img)
    rng = np.random.default_rng(93)
    tgts = dense_targets_from_labels(1, 640, 1, rng, 20)
    preds = [h.detach().clone().requires_grad_(True) for h in heads]
    res = ref.yolo_loss_multiscale(preds, tgts, [a.cpu() for a in model.anchors], 1)
    res[0].backward()
    out = {"losses": np.array([float(r) for r in res], dtype=np.float32)}
    for s in range(3):
        out[f"head{s}"] = heads[s].numpy()
        nz = np.argwhere(tgts[s].numpy()[..., 4] > 0)
        out[f"tgt{s}_idx"] = nz.astype(np.int32)
        out[f"tgt{s}_rows"] = tgts[s].numpy()[nz[:, 0], nz[:, 1], nz[:, 2], nz[:, 3]]
        g = preds[s].grad.numpy()
        out[f"grad{s}_obj"] = g[..., 4].copy()                     # dense objectness column
        out[f"grad{s}_rows"] = g[nz[:, 0], nz[:, 1], nz[:, 2], nz[:, 3]]  # full rows at the positives
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "x.png")
        Image.fromarray(np.zeros((640, 640, 3), dtype=np.uint8)).save(path)
        fake = FakeModel(heads, 640, model.anchors)
        # the bias init puts every sigmoid(obj) within 50 ulp of 0.01 (105 distinct values), so a
        # threshold inside that cluster is decided by the last bit of the sigmoid implementation;
        # 0.009 passes every row: a dense, heavily tied NMS input
        confs = [0.009]
        out["confs"] = np.array(confs, dtype=np.float64)
        for k, conf in enumerate(confs):
            dets = ref.predict(fake, path, torch.device("cpu"), num_classes=1, conf_threshold=conf, iou_threshold=0.4)
            out[f"dets_{k}"] = np.array(dets, dtype=np.float64).reshape(-1, 6)
            print("model heads conf", conf, "detections", len(dets))
    np.savez_compressed(os.path.join(OUT, "model_heads.npz"), **out)


class FakeEvalModel:
    """Stands in for YOLO inside the reference's eval_epoch(): preset heads per batch."""

    def __init__(self, batches, img, anchors):
        self.batches, self.k = batches, 0
        self.anchors = anchors
        self.grid_size_p3, self.grid_size_p4, self.grid_size_p5 = img // 8, img // 16, img // 32

    def eval(self):
        return self

    def __call__(self, imgs):
        heads = self.batches[self.k]
        self.k += 1
        return heads


def heads_near_targets(tgts, anchors, nc, seed, hit=0.7, jitter=0.35):
    """randn heads; on a share of the positive cells the logits are set so that the decoded box
    lands near the target (objectness high): gives eval_epoch true positives, misses and misfits."""
    heads = []
    rng = np.random.default_rng(seed)
    for s, t in enumerate(tgts):
        B, G = t.shape[0], t.shape[1]
        h = torch.randn(t.shape, generator=gen(seed * 10 + s))
        pos = (t[..., 4] > 0.5).nonzero()
        for b, gy, gx, a in pos.tolist():
            if rng.uniform() > hit:
                continue
            xc, yc, w, hh = [float(v) for v in t[b, gy, gx, a, 0:4]]
            j = lambda: float(np.exp(rng.normal(0, jitter)))
            sx = min(max((xc * G - gx + 0.5) / 2 + rng.normal(0, 0.05), 0.02), 0.98)
            sy = min(max((yc * G - gy + 0.5) / 2 + rng.normal(0, 0.05), 0.02), 0.98)
            sw = min(max(np.sqrt(w * j() * 640.0 / float(anchors[s][a, 0])) / 2, 0.02), 0.98)
            sh = min(max(np.sqrt(hh * j() * 640.0 / float(anchors[s][a, 1])) / 2, 0.02), 0.98)
            logit = lambda p: float(np.log(p / (1 - p)))
            h[b, gy, gx, a, 0:4] = torch.tensor([logit(sx), logit(sy), logit(sw), logit(sh)])
            h[b, gy, gx, a, 4] = float(rng.normal(1.5, 1.5))
        heads.append(h)
    return heads


def golden_eval():
    """The reference's own eval_epoch() (train.py:960-1032) on preset heads and reference-assigned
    targets: loss + the python TP/FP/FN loop -> (avg_loss, precision, recall, f1)."""
    out = {}
    rng = np.random.default_rng(91)
    for name, img, nc, B, nb, conf, iou in [("e640", 640, 1, 2, 1, 0.5, 0.5), ("e320", 320, 3, 2, 2, 0.3, 0.4)]:
        batches, loader = [], []
        for k in range(nb):
            tgts = dense_targets_from_labels(B, img, nc, rng, 14)
            heads = heads_near_targets(tgts, anchors3(), nc, 900 + k + img)
            batches.append(heads)
            imgs = torch.zeros(B, 3, 8, 8)
            loader.append((imgs, [[tgts[s][b] for s in range(3)] for b in range(B)]))
            for s in range(3):
                out.update(pack_seeded_randn(f"{name}_b{k}_head{s}", heads[s].numpy(), (900 + k + img) * 10 + s))
                out[f"{name}_b{k}_tgt{s}"] = tgts[s].numpy()
        model = FakeEvalModel(batches, img, anchors3())
        res = ref.eval_epoch(model, loader, torch.device("cpu"), num_classes=nc, iou_threshold=iou, conf_threshold=conf)
        out[f"{name}_cfg"] = np.array([img, nc, B, nb, conf, iou], dtype=np.float64)
        out[f"{name}_result"] = np.array([float(r) for r in res], dtype=np.float64)
        print(name, "eval_epoch ->", res)
    np.savez_compressed(os.path.join(OUT, "eval.npz"), **out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    golden_decode()
    golden_ciou()
    golden_targets()
    golden_loss()
    golden_predict()
    golden_nms()
    golden_model_heads()
    golden_eval()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
