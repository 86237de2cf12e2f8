"""The validation report on the device against the numpy oracle on the host, on tools/bench_map.py's workload.

Workload: 5,000 images of 640x640 in batches of 64, nc = 80 (or --nc 1, the reference's model and the case where
every count of a batch lands on four matrix cells and a few histogram bins), SURVEY 8d "prior" heads, 0..50 ground
truths per image from bench.py's label generator; conf 0.001, NMS IoU 0.4, max_det 300.  Times DetectionReport.update
per batch with CUDA events, report_match_kernel beside map_match_kernel with the library's per-launch events, and warm
compute() beside DetectionMAP.compute() on the same records; then runs the oracle (oracle/report_ref.py) on the same
kept detections and checks that the counts, curves and tables are equal.  Prints one JSON line (with the device name
and power limit).

  python tools/bench_report.py [--images 5000] [--batch 64] [--nc 80]
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
from bench import make_labels   # noqa: E402  (the 8d label generator)
from oracle import ref_path as R   # noqa: E402
from oracle import report_ref as P   # noqa: E402
from tools.bench_map import power_limit   # noqa: E402
import yolo_from_scratch_b200 as yb   # noqa: E402
from yolo_from_scratch_b200 import ops   # noqa: E402


def timed(fn):
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    out = fn()
    c1.record()
    torch.cuda.synchronize()
    return c0.elapsed_time(c1), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--nc", type=int, default=80)
    ap.add_argument("--img", type=int, default=640)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_report.py needs a CUDA device")
    dev = torch.device("cuda")
    img, nc, B = args.img, args.nc, args.batch
    anchors = [a.to(dev) for a in R.default_anchors()]
    rng = np.random.default_rng(0)
    g = torch.Generator(device=dev).manual_seed(0)
    rep = ops.DetectionReport(nc)
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
        det = ops.detect_batch(heads, anchors, img, nc, conf_threshold=0.001, iou_threshold=0.4, letterbox=[(1.0, 0.0, 0.0)] * n)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        rep.update(det, packed)
        e[1].record()
        ev.append(e)
        d = {k: det[k].cpu().numpy() for k in ("boxes", "scores", "classes", "keep", "n_keep")}
        host += [{"boxes": d["boxes"][b], "scores": d["scores"][b], "classes": d["classes"][b], "keep": d["keep"][b],
                  "n_keep": int(d["n_keep"][b]), "labels": labels[b], "letterbox": letterbox[b]} for b in range(n)]
    torch.cuda.synchronize()
    update_ms = [a.elapsed_time(b) for a, b in ev][1:]   # the first batch loads the modules
    buf = ctypes.create_string_buffer(1 << 16)
    lib.yb_timing_collect(buf, len(buf))
    lib.yb_timing_enable(0)
    kernels = {}
    for line in buf.value.decode().splitlines():
        name, count, total = line.split()
        kernels[name] = {"count": int(count), "ms_per_launch": float(total) / int(count)}
    # alternate the two computes over the same records; the first call of each includes first-launch costs
    report_ms, map_ms = [], []
    for _ in range(6):
        ms, got = timed(rep.compute)
        report_ms.append(ms)
        map_ms.append(timed(rep.map.compute)[0])
    # the host half of compute(): the curves from the suffix sums
    above = [np.cumsum(h.cpu().numpy()[:, ::-1], axis=1)[:, ::-1] for h in (rep._det_hist, rep._tp_hist)]
    t0 = time.perf_counter()
    ops.report_curves(above[0], above[1], got["n_gt"], rep.conf_grid)
    curves_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    want = P.evaluate(host, nc, rep.map.iou_thresholds, rep.conf_grid, max_det=300)
    oracle_s = time.perf_counter() - t0
    equal = bool(all(np.array_equal(got[k], want[k]) for k in
                     ("confusion", "images", "p_curve", "r_curve", "f1_curve", "p", "r", "f1", "precision", "recall",
                      "n_gt", "n_det"))
                 and got["best_conf"] == want["best_conf"]
                 and ops.format_detection_report(got) == ops.format_detection_report(want))
    k_rep = kernels.get("report_match_kernel", {}).get("ms_per_launch")
    k_map = kernels.get("map_match_kernel", {}).get("ms_per_launch")
    print(json.dumps({
        "device": torch.cuda.get_device_name(), "power_limit": power_limit(), "images": args.images, "batch": B,
        "nc": nc, "img": img, "detections_per_image": float(got["n_det"].sum()) / args.images,
        "gt_per_image": float(got["n_gt"].sum()) / args.images,
        "matrix_detections_per_image": float(got["confusion"][:nc].sum()) / args.images,
        "report_match_kernel_ms": k_rep, "map_match_kernel_ms": k_map,
        "report_over_map_kernel": (k_rep / k_map) if k_rep and k_map else None,
        "update_ms_median": float(np.median(update_ms)),
        "compute_ms_first": report_ms[0], "compute_ms": min(report_ms[1:]),
        "map_compute_ms_first": map_ms[0], "map_compute_ms": min(map_ms[1:]),
        "compute_over_map_compute": min(report_ms[1:]) / min(map_ms[1:]), "host_curves_ms": curves_ms,
        "kernels": kernels,
        "oracle_host_s": oracle_s, "best_conf": got["best_conf"], "map": got["map"], "map50": got["map50"],
        "table": ops.format_detection_report(got)[:2], "equal": equal}))


if __name__ == "__main__":
    main()
