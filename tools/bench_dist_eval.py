"""Image-sharded evaluation: compute(group) of DetectionMAP, COCODetectionEval and DetectionReport against one process.

Workload: tools/bench_map.py's, 5,000 images of 640x640, nc = 80, SURVEY 8d "prior" heads (objectness logit
2*randn - 4.6), 0..50 ground truths per image from bench.py's label generator; conf 0.001, NMS IoU 0.4, max_det 300.
Image i's heads and labels come from seed i, so every split of the images gives each image the same inputs.

One process first evaluates every image in batches of 64 and times compute() of each metric.  Then W ranks
(--backend gloo | nccl) each take their contiguous block (dist.shard_range), update in batches of 64 and time
compute(group) with a host clock after a barrier (compute returns after its last device synchronisation).  Every
rank's result must equal the single process's bit for bit (`equal`).  The bytes are computed from shapes: what each
rank contributes to the collectives (header, counts, records padded to the largest shard) and the records of all
ranks without padding.  With gloo the collectives stage CUDA tensors through the host, so its times say nothing about
NCCL.  Prints one JSON line with the device name and power limit.

  python tools/bench_dist_eval.py [--world 2] [--backend gloo] [--images 5000]
"""
import argparse
import datetime
import json
import os
import socket
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import make_labels   # noqa: E402  (the 8d label generator)
from bench_map import power_limit   # noqa: E402
from oracle import ref_path as R   # noqa: E402
from yolo_from_scratch_b200 import ops   # noqa: E402
from yolo_from_scratch_b200.dist import FINGERPRINT_FIELDS, shard_range   # noqa: E402

NC, IMG, BATCH, REPEATS = 80, 640, 64, 5
HEADER_BYTES = (len(FINGERPRINT_FIELDS) + 6) * 8   # dist.gather_eval_state's header


def metrics():
    return {"map": ops.DetectionMAP(NC), "coco": ops.COCODetectionEval(NC), "report": ops.DetectionReport(NC)}


def evaluate(lo, hi, dev):
    """Every metric updated with the images [lo, hi) in batches of BATCH."""
    ms = metrics()
    anchors = [a.to(dev) for a in R.default_anchors()]
    g = torch.Generator(device=dev)
    for i0 in range(lo, hi, BATCH):
        n = min(BATCH, hi - i0)
        heads = [torch.empty(n, G, G, 3, 5 + NC, device=dev) for G in (IMG // 8, IMG // 16, IMG // 32)]
        labels = []
        for j in range(n):
            g.manual_seed(i0 + j)
            for h in heads:
                h[j].normal_(generator=g)
            labels += make_labels(np.random.default_rng(i0 + j), 1, NC)
        for h in heads:
            h[..., 4].mul_(2.0).sub_(4.6)
        det = ops.detect_batch(heads, anchors, IMG, NC, conf_threshold=0.001, iou_threshold=0.4,
                               letterbox=[(1.0, 0.0, 0.0)] * n)
        packed = ops.pack_labels(labels, IMG, [(IMG, IMG, 1.0, 0.0, 0.0)] * n)
        for m in ms.values():
            m.update(det, packed)
    return ms


def shapes(ms):
    """(record rows, record bytes per row, count bytes) of each metric's state on this process."""
    rows = sum(r.shape[0] for r in ms["map"]._records)
    report_counts = ms["report"].map._gt_count.numel() + ms["report"]._counts.numel()
    return {"map": (rows, 12, ms["map"]._gt_count.numel() * 8),
            "coco": (sum(r.shape[0] for r in ms["coco"]._records), 32, ms["coco"]._gt_count.numel() * 8),
            "report": (rows, 12, report_counts * 8)}


def time_compute(m, group, barrier):
    out, ms = None, []
    for _ in range(REPEATS):   # the first call includes first launches of the sort and the precision kernels
        barrier()
        t0 = time.perf_counter()
        out = m.compute(group) if group is not None else m.compute()
        ms.append((time.perf_counter() - t0) * 1e3)
    return out, ms


def rank_main(rank, world, port, backend, images, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank if backend == "nccl" or torch.cuda.device_count() >= world else 0)
    torch.cuda.set_device(dev)
    kw = {"device_id": dev} if backend == "nccl" else {}
    dist.init_process_group(backend, rank=rank, world_size=world, timeout=datetime.timedelta(seconds=600), **kw)
    try:
        lo, hi = shard_range(images, rank, world)
        ms = evaluate(lo, hi, dev)
        torch.cuda.synchronize()
        res = {name: time_compute(m, dist.group.WORLD, dist.barrier) for name, m in ms.items()}
        q.put((rank, hi - lo, shapes(ms), res))
    finally:
        dist.destroy_process_group()


def same(a, b):
    for k in b:
        if isinstance(b[k], np.ndarray):
            if not (isinstance(a[k], np.ndarray) and a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k])):
                return False
        elif type(a[k]) is not type(b[k]) or a[k] != b[k]:
            return False
    return set(a) == set(b)


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--world", type=int, default=2)
    ap.add_argument("--backend", choices=("gloo", "nccl"), default="gloo")
    ap.add_argument("--images", type=int, default=5000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dist_eval.py needs a CUDA device")
    if args.backend == "nccl" and torch.cuda.device_count() < args.world:
        raise SystemExit(f"nccl with {args.world} ranks needs {args.world} GPUs, found {torch.cuda.device_count()}")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ms = evaluate(0, args.images, dev)
    torch.cuda.synchronize()
    single = {name: time_compute(m, None, lambda: None) for name, m in ms.items()}
    del ms
    torch.cuda.empty_cache()

    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=rank_main, args=(r, args.world, port, args.backend, args.images, q))
             for r in range(args.world)]
    try:
        for p in procs:
            p.start()
        ranks = sorted((q.get(timeout=1800) for _ in procs), key=lambda x: x[0])
        for p in procs:
            p.join(timeout=120)
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
            p.join(timeout=30)
    if any(p.exitcode != 0 for p in procs):
        raise SystemExit(f"a rank failed: exit codes {[p.exitcode for p in procs]}")

    out = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "backend": args.backend,
           "world": args.world, "gpus_used": len({r if args.backend == "nccl" or torch.cuda.device_count() >= args.world
                                                  else 0 for r in range(args.world)}),
           "images": args.images, "images_per_rank": [r[1] for r in ranks]}
    equal = True
    for name in ("map", "coco", "report"):
        rows = [r[2][name][0] for r in ranks]
        width, count_bytes = ranks[0][2][name][1], ranks[0][2][name][2]
        sent = HEADER_BYTES + count_bytes + max(rows) * width
        want, single_ms = single[name]
        group_ms = [r[3][name][1] for r in ranks]
        ok = all(same(r[3][name][0], want) for r in ranks)
        equal = equal and ok
        out[name] = {"records": sum(rows), "record_bytes_total": sum(rows) * width,
                     "bytes_contributed_per_rank": sent, "compute_ms": float(np.median(single_ms[1:])),
                     "compute_group_ms": float(np.median([np.median(m[1:]) for m in group_ms])),
                     "compute_group_ms_per_rank": [float(np.median(m[1:])) for m in group_ms],
                     "compute_ms_first": single_ms[0], "compute_group_ms_first": max(m[0] for m in group_ms),
                     "equal": ok}
    out["equal"] = equal
    print(json.dumps(out))


if __name__ == "__main__":
    main()
