"""COCO-val-sized COCO bbox summary on the device against the oracle's kernel form on the host.

Workload of tools/bench_map.py: 5,000 images of 640x640 in batches of 64, nc = 80, SURVEY 8d "prior" heads
(objectness logit 2*randn - 4.6), 0..50 ground truths per image from bench.py's label generator; conf 0.001, NMS IoU
0.4, max_det 300.  Each batch runs detect_batch, then DetectionMAP.update and COCODetectionEval.update on the same
detections; the library's per-launch events give each kernel's own device time (coco_match_kernel against
map_match_kernel and detect_batch's kernels).  compute() is timed with CUDA events, then oracle/coco_ref.py
(evaluate, the kernels' form) runs on the same kept detections and the tables are compared bit for bit.
Prints one JSON line (with the device name and power limit).

  python tools/bench_coco.py [--images 5000] [--batch 64]
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import make_labels   # noqa: E402  (the 8d label generator)
from bench_map import power_limit   # noqa: E402
from oracle import coco_ref as C   # noqa: E402
from oracle import ref_path as R   # noqa: E402
import yolo_from_scratch_b200 as yb   # noqa: E402
from yolo_from_scratch_b200 import ops   # noqa: E402

DETECT_KERNELS = ("filter_", "graph_", "nms_")   # detect_batch's kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--nc", type=int, default=80)
    ap.add_argument("--img", type=int, default=640)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_coco.py needs a CUDA device")
    dev = torch.device("cuda")
    img, nc, B = args.img, args.nc, args.batch
    anchors = [a.to(dev) for a in R.default_anchors()]
    rng = np.random.default_rng(0)
    g = torch.Generator(device=dev).manual_seed(0)
    metric = ops.COCODetectionEval(nc)
    dmap = ops.DetectionMAP(nc)
    lib = yb._lib.lib()
    lib.yb_timing_enable(1)   # per-launch events of the library's own kernels: device time without host gaps
    ev, host = [], []
    for i0 in range(0, args.images, B):
        n = min(B, args.images - i0)
        heads = [torch.randn(n, G, G, 3, 5 + nc, generator=g, device=dev) for G in (img // 8, img // 16, img // 32)]
        for h in heads:
            h[..., 4].mul_(2.0).sub_(4.6)
        labels = make_labels(rng, n, nc)
        letterbox = [(img, img, 1.0, 0.0, 0.0)] * n
        packed = ops.pack_labels(labels, img, letterbox)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        det = ops.detect_batch(heads, anchors, img, nc, conf_threshold=0.001, iou_threshold=0.4, letterbox=[(1.0, 0.0, 0.0)] * n)
        e[1].record()
        dmap.update(det, packed)
        metric.update(det, packed)
        ev.append(e)
        d = {k: det[k].cpu().numpy() for k in ("boxes", "scores", "classes", "keep", "n_keep")}
        host += [{"boxes": d["boxes"][b], "scores": d["scores"][b], "classes": d["classes"][b], "keep": d["keep"][b],
                  "n_keep": int(d["n_keep"][b]), "labels": labels[b], "letterbox": letterbox[b]} for b in range(n)]
    torch.cuda.synchronize()
    detect_ms = [a.elapsed_time(b) for a, b in ev][1:]   # the first batch loads the modules
    buf = ctypes.create_string_buffer(1 << 16)
    lib.yb_timing_collect(buf, len(buf))
    kernels = {}
    for line in buf.value.decode().splitlines():
        name, count, total = line.split()
        kernels[name] = {"count": int(count), "ms_per_launch": float(total) / int(count)}
    compute_ms = []
    for _ in range(4):   # the first call includes first-launch costs of the sort and the precision kernel
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        got = metric.compute()
        c1.record()
        torch.cuda.synchronize()
        compute_ms.append(c0.elapsed_time(c1))
    buf = ctypes.create_string_buffer(1 << 16)
    lib.yb_timing_collect(buf, len(buf))
    lib.yb_timing_enable(0)
    for line in buf.value.decode().splitlines():
        name, count, total = line.split()
        if name == "coco_precision_kernel":
            kernels[name] = {"count": int(count), "ms_per_launch": float(total) / int(count)}
    t0 = time.perf_counter()
    want = C.evaluate(host, nc, metric.iou_thresholds, metric.recall_thresholds, max_det=300, max_dets=metric.max_dets)
    oracle_s = time.perf_counter() - t0
    equal = bool(np.array_equal(got["precision"], want["precision"]) and np.array_equal(got["recall"], want["recall"])
                 and np.array_equal(got["n_gt"], want["n_gt"]) and np.array_equal(got["n_det"], want["n_det"])
                 and np.allclose(got["stats"], want["stats"], rtol=0, atol=1e-12))
    ms = lambda k: kernels.get(k, {}).get("ms_per_launch")
    print(json.dumps({
        "device": torch.cuda.get_device_name(), "power_limit": power_limit(), "images": args.images, "batch": B,
        "nc": nc, "img": img, "records": int(got["n_det"].sum()), "gt_per_image": float(got["n_gt"][:, 0].sum()) / args.images,
        "coco_match_kernel_ms": ms("coco_match_kernel"), "map_match_kernel_ms": ms("map_match_kernel"),
        "detect_batch_ms_median": float(np.median(detect_ms)),
        "detect_batch_kernels_ms": sum(v["ms_per_launch"] * v["count"] for k, v in kernels.items()
                                       if any(s in k for s in DETECT_KERNELS)) / len(ev),
        "compute_ms_first": compute_ms[0], "compute_ms": min(compute_ms[1:]),
        "coco_precision_kernel_ms": ms("coco_precision_kernel"), "kernels": kernels, "oracle_host_s": oracle_s,
        "stats": got["stats"].tolist(), "lines": ops.format_coco_stats(got["stats"]), "equal": equal}))


if __name__ == "__main__":
    main()
