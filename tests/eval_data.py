"""Data and stand-ins the evaluation GPU tests share (test_gpu_map, test_gpu_coco, test_gpu_report and
test_gpu_dist_eval): synthetic batches with their host copies for the oracles, packed labels, "prior" heads and a
stand-in for the reference's train module."""
import pathlib
import types

import numpy as np
import torch

from yolo_from_scratch_b200 import ops
from oracle import map_ref as M

SIZES = np.array([8, 16, 31, 32, 33, 48, 95, 96, 97, 128, 200])   # pixels: around the 32 and 96 bounds
# scores are multiples of 1/40 in fp32: this confidence grid holds each of them exactly, plus random points
CUSTOM_GRID = np.unique(np.concatenate([np.float32(np.arange(41) / 40).astype(np.float64),
                                        np.random.default_rng(5).uniform(0, 1, 60)]))


def synthetic_batch(rng, B, nc, max_gt, cap, n_keep_zero=0.1):
    """Clustered ground truth with jittered detections: many IoUs near the thresholds, duplicated ground truths
    (equal IoU) and quantised scores (equal scores).  Candidates are in a random order and keep lists them by
    descending score, as NMS does.  Returns (det dict on the GPU, per-image host dicts for the oracle, PackedLabels
    inputs)."""
    boxes = np.zeros((B, cap, 4), np.float32)
    scores = np.zeros((B, cap), np.float32)
    classes = np.zeros((B, cap), np.int64)
    keep = np.zeros((B, cap), np.int64)
    n_keep = np.zeros(B, np.int32)
    labels, letterbox, host = [], [], []
    for b in range(B):
        ow, oh = float(rng.integers(200, 800)), float(rng.integers(200, 800))
        n = int(rng.integers(0, max_gt + 1)) if rng.uniform() > 0.1 else 0
        centres = rng.uniform(0.2, 0.8, (max(1, n // 8 + 1), 2))
        lab = np.zeros((n, 5))
        lab[:, 0] = rng.integers(0, nc, n)
        lab[:, 1:3] = centres[rng.integers(0, len(centres), n)] + rng.normal(0, 0.02, (n, 2))
        lab[:, 3:5] = rng.uniform(0.05, 0.3, (n, 2))
        if n >= 4:
            lab[n // 2] = lab[n // 4]                                           # duplicate: equal IoU
        gb, _, _ = M.gt_boxes(lab, (ow, oh), max(nc, 2))
        m = int(rng.integers(0, cap + 1))
        src = rng.integers(0, max(n, 1), m)
        jit = rng.normal(0, 1, (m, 4)) * rng.choice([0.0, 2.0, 8.0], (m, 1))
        bx = (gb[src] + jit) if n else rng.uniform(0, 400, (m, 4))
        bx = np.concatenate([np.minimum(bx[:, :2], bx[:, 2:]), np.maximum(bx[:, :2], bx[:, 2:])], 1)
        if m:
            boxes[b, :m] = bx
            scores[b, :m] = np.round(rng.uniform(0.001, 1, m) * 40) / 40
            classes[b, :m] = np.where(rng.uniform(size=m) < 0.8, lab[src, 0] if n else 0, rng.integers(0, nc, m)) % nc
        order = np.argsort(-scores[b, :m], kind="stable")
        keep[b, :m] = order
        n_keep[b] = 0 if rng.uniform() < n_keep_zero else m
        labels.append(lab)
        letterbox.append((ow, oh, 1.0, 0.0, 0.0))
        host.append({"boxes": boxes[b], "scores": scores[b], "classes": classes[b], "keep": keep[b],
                     "n_keep": int(n_keep[b]), "labels": lab, "letterbox": letterbox[-1]})
    dev = torch.device("cuda")
    det = {"boxes": torch.from_numpy(boxes).to(dev), "scores": torch.from_numpy(scores).to(dev),
           "classes": torch.from_numpy(classes).to(dev), "keep": torch.from_numpy(keep).to(dev),
           "n_keep": torch.from_numpy(n_keep).to(dev)}
    return det, host, (labels, letterbox)


def coco_synthetic_batch(rng, B, nc, max_gt, cap, n_keep_zero=0.1):
    """Clustered ground truths with jittered detections, on images of 256, 512 or 1024 pixels.  Every label value is a
    multiple of 2^-10, so corners are exact; sides are drawn from SIZES, so some areas are exactly 32^2 and 96^2.
    Detections are copies of ground truths (exact ones too) jittered by multiples of 1/2 pixel, with duplicated
    ground truths (equal IoU) and quantised scores (equal scores); keep lists them by descending score."""
    boxes = np.zeros((B, cap, 4), np.float32)
    scores = np.zeros((B, cap), np.float32)
    classes = np.zeros((B, cap), np.int64)
    keep = np.zeros((B, cap), np.int64)
    n_keep = np.zeros(B, np.int32)
    labels, letterbox, host = [], [], []
    for b in range(B):
        ow, oh = float(rng.choice([256, 512, 1024])), float(rng.choice([256, 512, 1024]))
        n = int(rng.integers(0, max_gt + 1)) if rng.uniform() > 0.1 else 0
        wh = rng.choice(SIZES, (n, 2)).astype(np.float64)
        centres = np.round(rng.uniform(0.2, 0.8, (max(1, n // 8 + 1), 2)) * 64) * 4
        c = centres[rng.integers(0, len(centres), n)] / 256 * np.array([ow, oh]) + rng.integers(-8, 9, (n, 2)) * 2
        x1 = np.round(c - wh / 2)
        lab = np.zeros((n, 5))
        lab[:, 0] = rng.integers(0, nc, n)
        if n >= 4:                                                              # duplicate: equal IoU
            x1[n // 2], wh[n // 2], lab[n // 2, 0] = x1[n // 4], wh[n // 4], lab[n // 4, 0]
        lab[:, 1] = (x1[:, 0] + wh[:, 0] / 2) / ow
        lab[:, 2] = (x1[:, 1] + wh[:, 1] / 2) / oh
        lab[:, 3], lab[:, 4] = wh[:, 0] / ow, wh[:, 1] / oh
        gb = np.column_stack([x1, x1 + wh]) if n else np.zeros((0, 4))
        m = int(rng.integers(0, cap + 1))
        src = rng.integers(0, max(n, 1), m)
        jit = rng.integers(-4, 5, (m, 4)) * 0.5 * rng.choice([0.0, 1.0, 4.0], (m, 1))
        bx = (gb[src] + jit) if n else rng.integers(0, 400, (m, 4)).astype(np.float64)
        bx = np.concatenate([np.minimum(bx[:, :2], bx[:, 2:]), np.maximum(bx[:, :2], bx[:, 2:])], 1)
        if m:
            boxes[b, :m] = bx
            scores[b, :m] = np.round(rng.uniform(0.001, 1, m) * 40) / 40
            classes[b, :m] = np.where(rng.uniform(size=m) < 0.8, lab[src, 0] if n else 0, rng.integers(0, nc, m)) % nc
        keep[b, :m] = np.argsort(-scores[b, :m], kind="stable")
        n_keep[b] = 0 if rng.uniform() < n_keep_zero else m
        labels.append(lab)
        letterbox.append((ow, oh, 1.0, 0.0, 0.0))
        host.append({"boxes": boxes[b], "scores": scores[b], "classes": classes[b], "keep": keep[b],
                     "n_keep": int(n_keep[b]), "labels": lab, "letterbox": letterbox[-1]})
    dev = torch.device("cuda")
    det = {"boxes": torch.from_numpy(boxes).to(dev), "scores": torch.from_numpy(scores).to(dev),
           "classes": torch.from_numpy(classes).to(dev), "keep": torch.from_numpy(keep).to(dev),
           "n_keep": torch.from_numpy(n_keep).to(dev)}
    return det, host, (labels, letterbox)


def packed(labels, letterbox, max_gt=None):
    lab, n_gt, lb = ops.pack_labels_host(labels, 640, letterbox, max_gt=max_gt)
    return ops.PackedLabels(lab.cuda(), n_gt.cuda(), lb.cuda(), 640)


def prior_heads(B, img, nc, seed):
    g = torch.Generator().manual_seed(seed)
    heads = [torch.randn(B, G, G, 3, 5 + nc, generator=g) for G in (img // 8, img // 16, img // 32)]
    for h in heads:
        h[..., 4].mul_(2.0).sub_(4.6)   # SURVEY 8d "prior" heads
    return [h.cuda() for h in heads]


def host_images(det, labels, letterbox):
    d = {k: det[k].cpu().numpy() for k in ("boxes", "scores", "classes", "keep", "n_keep")}
    return [{"boxes": d["boxes"][b], "scores": d["scores"][b], "classes": d["classes"][b], "keep": d["keep"][b],
             "n_keep": int(d["n_keep"][b]), "labels": labels[b], "letterbox": letterbox[b]} for b in range(len(labels))]


class _PresetHeads:
    def __init__(self, heads, img_size, anchors):
        self.heads, self.img_size, self.anchors = heads, img_size, anchors

    def eval(self):
        return self

    def __call__(self, img):
        n = img.shape[0]
        return [h[:n] for h in self.heads]


def _train_stand_in(scale, pad_top, pad_left):
    """A module with the names install() rebinds in the reference's `train`, plus the Path and Image its dataset code
    uses.  Its letterbox_resize returns a fixed scale and padding."""
    from PIL import Image
    from yolo_from_scratch_b200.install import PATCHED_FUNCTIONS
    m = types.ModuleType("train")
    m.Image = Image
    m.Path = pathlib.Path
    m.letterbox_resize = lambda pil_img, img_size: (pil_img, scale, pad_top, pad_left)
    for n in PATCHED_FUNCTIONS + ("predict",):
        setattr(m, n, lambda *a, **k: "ref")
    return m
