"""Multi-label candidates with the top-K cap (yb_filter_multilabel) and multi-label detect_batch on the device.

Workload: nc = 80, 640x640, B = 64, conf 0.001, NMS IoU 0.4, K = max_candidates = 30000, max_det 300, on two head sets
of SURVEY 8d: dense `randn` heads (every image far over the cap) and its "prior" heads (objectness logits 2*randn-4.6).
For each set it times, with the library's per-launch events, the four kernels of the filter (count, select, refine,
emit); with CUDA events the filter call, the NMS on its candidates, the whole multi-label detect_batch and the
single-label detect_batch on the same heads (alternated, medians); reports totals / counts statistics, the algorithmic
bytes of every pass over the heads and their fraction of the 6,546.6 GB/s copy peak (DESIGN §8); and checks two images
against the oracle (oracle/multilabel_ref.py on the same CUDA heads: counts, classes, score bits, boxes, NMS keep set).
Prints one JSON line with the device name and power limit.

  python tools/bench_multilabel.py [--iters 10] [--batch 64] [--nc 80] [--img 640]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import multilabel_ref as ML   # noqa: E402
from oracle import ref_path as R   # noqa: E402
from tools.bench_map import power_limit   # noqa: E402
import yolo_from_scratch_b200 as yb   # noqa: E402
from yolo_from_scratch_b200 import ops   # noqa: E402

COPY_PEAK_GBS = 6546.6   # measured HBM copy peak of DESIGN §8


def events(fn, iters):
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), out


def kernel_times(lib, fn, iters):
    """Median-free per-launch device time: the library's own events around every launch, summed by name."""
    torch.cuda.synchronize()
    lib.yb_timing_collect(None, 0)
    lib.yb_timing_enable(1)
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.yb_timing_collect(buf, len(buf))
    lib.yb_timing_enable(0)
    out = {}
    for line in buf.value.decode().splitlines():
        name, count, total = line.split()
        out[name] = {"launches_per_call": int(count) / iters, "ms_per_call": float(total) / iters}
    return out


def stats(t):
    v = t.double().cpu()
    return {"min": int(v.min()), "median": float(v.median()), "max": int(v.max()), "mean": float(v.mean())}


def check_oracle(heads, det, img, nc, conf, K, images=(0, 1)):
    """Counts, classes, score bits and boxes of `images` against the oracle on the same CUDA heads, and the NMS keep
    set against the torchvision restatement on the device's own candidates."""
    ok = True
    for b in images:
        rb, rs, rc, n = ML.candidates_multilabel([h[b:b + 1].float() for h in heads], [a.cuda() for a in R.default_anchors()],
                                                 img, nc, conf, K)
        m = int(det["counts"][b])
        ok &= m == rs.shape[0] and int(det["totals"][b]) == n
        ok &= bool(torch.equal(det["classes"][b, :m], rc))
        ok &= bool(torch.equal(det["scores"][b, :m].view(torch.int32), rs.view(torch.int32)))
        err = (det["boxes"][b, :m].double() - rb.double()).abs()
        ok &= bool((err <= 1e-5 * rb.double().abs() + 2e-4).all())
        bx, sc, cl = (det[k][b, :m].cpu().numpy() for k in ("boxes", "scores", "classes"))
        want = R.batched_nms_indices(bx, sc, cl, 0.4)
        ok &= np.array_equal(det["keep"][b, :int(det["n_keep"][b])].cpu().numpy(), want[:300])
    return bool(ok)


def run_set(name, heads, anchors, args, lib):
    img, nc, K, conf = args.img, args.nc, args.max_candidates, 0.001
    B = heads[0].shape[0]
    filt = lambda: ops.filter_candidates_multilabel(heads, anchors, img, nc, conf, max_candidates=K)   # noqa: E731
    ml = lambda: ops.detect_batch(heads, anchors, img, nc, conf, 0.4, multi_label=True, max_candidates=K,   # noqa: E731
                                  max_det=args.max_det)
    sl = lambda: ops.detect_batch(heads, anchors, img, nc, conf, 0.4)   # noqa: E731
    for fn in (filt, ml, sl):   # warm up every shape
        fn()
    torch.cuda.synchronize()
    kernels = kernel_times(lib, filt, args.iters)
    f_ms, ml_ms, sl_ms, nms_ms = [], [], [], []
    cand = filt()
    nms = lambda: ops.nms_candidates(*cand[:4], 0.4, max_det=args.max_det)   # noqa: E731
    for _ in range(args.iters):   # alternated, so that drift hits all four alike
        f_ms.append(events(filt, 1)[0])
        nms_ms.append(events(nms, 1)[0])
        ml_ms.append(events(ml, 1)[0])
        sl_ms.append(events(sl, 1)[0])
    det = ml()
    sdet = sl()
    torch.cuda.synchronize()
    # algorithmic bytes of one pass over the heads: one 32-byte sector per row for the objectness (a row is longer
    # than a sector), the class logits of the rows that pass it; the emit adds the box logits of those rows and the
    # 28 bytes of every kept candidate.  Refinement passes read only the capped images.
    es = heads[0].element_size()
    rows = sum(h.shape[1] * h.shape[2] * h.shape[3] for h in heads)
    passing = sum(int((torch.sigmoid(h[..., 4].float()) > conf).sum()) for h in heads)
    capped = det["totals"] > K
    cap_frac = float(capped.float().mean())
    obj_bytes = B * rows * min(32, (5 + nc) * es)
    cls_bytes = passing * nc * es
    count_bytes = obj_bytes + cls_bytes
    refine_bytes = cap_frac * count_bytes
    emit_bytes = count_bytes + passing * 4 * es + int(det["counts"].sum()) * 28
    passes = {"count": count_bytes, "refine": 3 * refine_bytes, "emit": emit_bytes}
    frac = {}
    for k, nbytes in passes.items():
        t = kernels.get(f"filter_ml_{k}_kernel", {}).get("ms_per_call")
        frac[k] = {"bytes": nbytes, "ms": t, "GBs": nbytes / t / 1e6 if t else None,
                   "frac_copy_peak": nbytes / t / 1e6 / COPY_PEAK_GBS if t else None}
    return {
        "heads": name, "filter_ms": float(np.median(f_ms)), "nms_ms": float(np.median(nms_ms)),
        "detect_multilabel_ms": float(np.median(ml_ms)), "detect_single_label_ms": float(np.median(sl_ms)),
        "kernels": kernels, "passes": frac, "rows_passing_obj_per_image": passing / B,
        "totals": stats(det["totals"]), "counts": stats(det["counts"]), "capped_images": int(capped.sum()),
        "n_keep": stats(det["n_keep"]), "single_label_counts": stats(sdet["counts"]),
        "single_label_n_keep": stats(sdet["n_keep"]),
        "oracle_equal": check_oracle(heads, det, img, nc, conf, K),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--nc", type=int, default=80)
    ap.add_argument("--img", type=int, default=640)
    ap.add_argument("--max-candidates", type=int, default=30000)
    ap.add_argument("--max-det", type=int, default=300)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_multilabel.py needs a CUDA device")
    dev = torch.device("cuda")
    lib = yb._lib.lib()
    anchors = [a.to(dev) for a in R.default_anchors()]
    g = torch.Generator(device=dev).manual_seed(0)
    out = {"device": torch.cuda.get_device_name(), "power_limit": power_limit(), "batch": args.batch, "nc": args.nc,
           "img": args.img, "conf": 0.001, "iou": 0.4, "max_candidates": args.max_candidates, "max_det": args.max_det,
           "iters": args.iters, "copy_peak_GBs": COPY_PEAK_GBS, "sets": []}
    for name in ("randn", "prior"):
        heads = [torch.randn(args.batch, G, G, 3, 5 + args.nc, generator=g, device=dev)
                 for G in (args.img // 8, args.img // 16, args.img // 32)]
        if name == "prior":
            for h in heads:
                h[..., 4].mul_(2.0).sub_(4.6)
        out["sets"].append(run_set(name, heads, anchors, args, lib))
        del heads
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
