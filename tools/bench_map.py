"""COCO-val-sized mAP evaluation on the device against the numpy oracle on the host.

Workload: 5,000 images of 640x640 in batches of 64, nc = 80, SURVEY 8d "prior" heads (objectness logit 2*randn - 4.6),
0..50 ground truths per image from bench.py's label generator; conf 0.001, NMS IoU 0.4, max_det 300.
Times detect_batch and DetectionMAP.update per batch and compute() with CUDA events (the per-batch figures include
any host enqueue gap; the library's per-launch events give each kernel's own device time), then the oracle
(oracle/map_ref.py) on the same kept detections, and checks that the precision and recall tables are equal.
Prints one JSON line (with the device name and power limit).

  python tools/bench_map.py [--images 5000] [--batch 64]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import make_labels   # noqa: E402  (the 8d label generator)
from oracle import map_ref as M   # noqa: E402
from oracle import ref_path as R   # noqa: E402
import yolo_from_scratch_b200 as yb   # noqa: E402
from yolo_from_scratch_b200 import ops   # noqa: E402


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--nc", type=int, default=80)
    ap.add_argument("--img", type=int, default=640)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_map.py needs a CUDA device")
    dev = torch.device("cuda")
    img, nc, B = args.img, args.nc, args.batch
    anchors = [a.to(dev) for a in R.default_anchors()]
    rng = np.random.default_rng(0)
    g = torch.Generator(device=dev).manual_seed(0)
    metric = ops.DetectionMAP(nc)
    lib = yb._lib.lib()
    lib.yb_timing_enable(1)   # per-launch events of the library's own kernels: device time without host gaps
    ev = []
    host = []
    for i0 in range(0, args.images, B):
        n = min(B, args.images - i0)
        heads = [torch.randn(n, G, G, 3, 5 + nc, generator=g, device=dev) for G in (img // 8, img // 16, img // 32)]
        for h in heads:
            h[..., 4].mul_(2.0).sub_(4.6)
        labels = make_labels(rng, n, nc)
        letterbox = [(img, img, 1.0, 0.0, 0.0)] * n
        packed = ops.pack_labels(labels, img, letterbox)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        det = ops.detect_batch(heads, anchors, img, nc, conf_threshold=0.001, iou_threshold=0.4, letterbox=[(1.0, 0.0, 0.0)] * n)
        e[1].record()
        metric.update(det, packed)
        e[2].record()
        ev.append(e)
        d = {k: det[k].cpu().numpy() for k in ("boxes", "scores", "classes", "keep", "n_keep")}
        host += [{"boxes": d["boxes"][b], "scores": d["scores"][b], "classes": d["classes"][b], "keep": d["keep"][b],
                  "n_keep": int(d["n_keep"][b]), "labels": labels[b], "letterbox": letterbox[b]} for b in range(n)]
    torch.cuda.synchronize()
    detect_ms = [a.elapsed_time(b) for a, b, _ in ev][1:]   # the first batch loads the modules
    update_ms = [b.elapsed_time(c) for _, b, c in ev][1:]
    buf = ctypes.create_string_buffer(1 << 16)
    lib.yb_timing_collect(buf, len(buf))
    lib.yb_timing_enable(0)
    kernels = {}
    for line in buf.value.decode().splitlines():
        name, count, total = line.split()
        kernels[name] = {"count": int(count), "ms_per_launch": float(total) / int(count)}
    compute_ms = []
    for _ in range(3):   # the first call includes first-launch costs of the sort and the precision kernel
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        got = metric.compute()
        c1.record()
        torch.cuda.synchronize()
        compute_ms.append(c0.elapsed_time(c1))
    t0 = time.perf_counter()
    want = M.evaluate(host, nc, metric.iou_thresholds, metric.recall_thresholds, max_det=300)
    oracle_s = time.perf_counter() - t0
    equal = bool(np.array_equal(got["precision"], want["precision"]) and np.array_equal(got["recall"], want["recall"])
                 and np.array_equal(got["n_gt"], want["n_gt"]) and np.array_equal(got["n_det"], want["n_det"]))
    print(json.dumps({
        "device": torch.cuda.get_device_name(), "power_limit": power_limit(), "images": args.images, "batch": B,
        "nc": nc, "img": img, "detections_per_image": float(got["n_det"].sum()) / args.images,
        "gt_per_image": float(got["n_gt"].sum()) / args.images,
        "detect_batch_ms_median": float(np.median(detect_ms)), "update_ms_median": float(np.median(update_ms)),
        "compute_ms_first": compute_ms[0], "compute_ms": min(compute_ms[1:]),
        "map_match_kernel_ms": kernels.get("map_match_kernel", {}).get("ms_per_launch"), "kernels": kernels,
        "oracle_host_s": oracle_s, "map": got["map"], "map50": got["map50"], "map_oracle": want["map"], "equal": equal}))


if __name__ == "__main__":
    main()
