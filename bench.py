#!/usr/bin/env python
"""bench.py — decode+global-NMS images/s and CIoU-loss fwd+bwd ms @640^2 bs64 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the per-box hot path over one batch of synthetic heads/labels:
fused multi-scale loss forward+backward, then decode + confidence filter + global NMS.
Workload = BASELINE.json configs[1]: nc=1, 640x640, 64 images per GPU, <=50 GT boxes per image,
randn heads (seed 1234+scale), predict()'s default thresholds (conf 0.5, IoU 0.4; train.py:1114).
N GPUs = 64 images on each (weak scaling, sharded by image); the loss partial sums are all-reduced
once per step over NCCL, NMS needs no collective.

`value` is timed with the inputs resident in HBM; `e2e` goes through the public Python API with
pinned HOST buffers (H2D of heads+targets and D2H of losses + detections inside the timed region).
`--impl reference` times the reference's CPU implementation of the path on the host cores: the
UNMODIFIED reference (baseline/_ref/train.py: yolo_loss_multiscale + predict) when it has been staged,
else the oracle port of the same code path.

Rank 0 prints ONE compact JSON line (< 4 KB: the contract keys + roofline + hbm_kernels + cpu_baseline +
e2e).  The per-kernel tables, the other BASELINE configs and every variant go to
a new <tempdir>/yolo_b200_bench_full_*.json (--full-out).  `--dump-outputs DIR` writes the losses, gradients and
detections of the last timed step as .npy files; the inputs are seeded, so two builds run with the same arguments
can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

IMG, NC, B_PER_GPU, MAX_GT = 640, 1, 64, 50
CONF, IOU = 0.5, 0.4
METRIC = "decode+global-NMS + CIoU-loss fwd+bwd throughput @640^2 bs64 nc1"
UNIT = "images/s"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
MAX_LINE_BYTES = 4096


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nc", type=int, default=NC)
    ap.add_argument("--img", type=int, default=IMG)
    ap.add_argument("--batch", type=int, default=B_PER_GPU, help="images per GPU")
    ap.add_argument("--conf", type=float, default=CONF)
    ap.add_argument("--iou", type=float, default=IOU)
    ap.add_argument("--reps", type=int, default=7,
                    help="the K-step timed region is repeated this many times, each bracketed by barrier + sync; "
                         "ms_per_step is the median over the repetitions and the spread is reported")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--launch", default="graph", choices=["graph", "eager"],
                    help="what `value` times: the step replayed as a CUDA graph (yb.HotPathGraph; at N>1 the NCCL "
                         "all-reduce is captured inside the graph), or eager launches.  Per-kernel times always come "
                         "from an eager pass of the same K steps; both throughputs are reported.")
    ap.add_argument("--layout", default="bhwac", choices=["bhwac", "nchw"],
                    help="head layout of the device-resident step: the reference's (B,H,W,A,5+nc) or the head conv's own "
                         "NCHW output (SURVEY 8f-2)")
    ap.add_argument("--targets", default="dense", choices=["dense", "labels"],
                    help="dense reference targets, or label lists assigned on the device (SURVEY 8f-4)")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true")
    ap.add_argument("--numa", default="auto", choices=["auto", "off"],
                    help="auto: bind the rank to its GPU's local CPUs (nvml) before the pinned host buffers are allocated")
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="images per step of the reference arm / cpu_baseline leg: N > 0 = exactly N, -1 = every image of the "
                         "batch, 0 = auto: as many (same seeds, first images of the batch) as keep the whole K+W-step run "
                         "within --cpu-budget-s, measured on a 2-image calibration pass")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0)
    ap.add_argument("--full-out", default=None,
                    help="file that receives the full, uncompacted result ('' = none); default: a new file in the "
                         "temporary directory (the source tree may be read-only), named in the printed line's `full`")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last timed step of the main workload computed (losses, "
                         "gradients, detections) as DIR/<name>.npy, for comparing two builds output for output")
    args = ap.parse_args(argv)
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# ------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY 8d)
# ------------------------------------------------------------------------------------------------
def make_labels(rng, B, nc):
    labels = []
    for _ in range(B):
        n = int(rng.integers(0, MAX_GT + 1))
        lab = np.zeros((n, 5), dtype=np.float64)
        lab[:, 0] = rng.integers(0, nc, size=n)
        lab[:, 1:3] = rng.uniform(0.05, 0.95, size=(n, 2))
        lab[:, 3:5] = np.exp(rng.uniform(np.log(0.01), np.log(0.6), size=(n, 2)))
        labels.append(lab)
    return labels


def make_heads(B, img, nc, seed):
    grids = [img // 8, img // 16, img // 32]
    heads = []
    for s, G in enumerate(grids):
        g = torch.Generator().manual_seed(seed + s)
        heads.append(torch.randn(B, G, G, 3, 5 + nc, generator=g))
    return heads


def tensor_bytes(ts):
    return int(sum(t.numel() * t.element_size() for t in ts))


DUMP_BUDGET_BYTES = 64 << 20
# the detections' share of the budget: their number depends on the data, the gradients' size only on the arguments
DUMP_DETECTIONS_BYTES = 16 << 20
DUMP_SMALL_BYTES = 1 << 20      # losses, offsets, candidate counts: always whole


def _sample_rows(a, nbytes):
    """Rows of `a` (first axis) at fixed seeded positions, sorted, chosen from len(a) and nbytes alone; each kept
    row also costs 8 bytes of stored position."""
    k = int(nbytes // (a[0].nbytes + 8))
    return np.unique(np.random.default_rng(1234).integers(0, len(a), k))


def dump_outputs(out_dir, losses, grads, det, rows, offsets):
    """--dump-outputs: what a caller of the step receives, as out_dir/<name>.npy (float32, or float64 for integers):
      losses (4,) [total, bbox, obj, cls];  grad_s<k>: d total / d heads[k], shaped like the heads;
      detections (n, 6) [x1, y1, x2, y2, conf, class], the kept boxes of every image in order, best first;
      detection_offsets (B+1,): image b's detections are rows offsets[b]:offsets[b+1];
      candidates (B,): boxes per image that passed the confidence threshold.
    The files stay within DUMP_BUDGET_BYTES.  Gradients larger together than their share are written as a sample of
    their flattened elements, and detections larger than DUMP_DETECTIONS_BYTES as a sample of their rows.  The sampled
    positions are drawn from a fixed seed and depend only on the array's own shape (the gradients' shapes, for their
    share), so two builds that compute the same arrays write the same files.  A sampled array <name> comes with
    <name>_index.npy (the positions, float64) and <name>_shape.npy (its full shape)."""
    torch.cuda.synchronize()
    n = max(int(offsets[-1]), 0)
    arrays = {"losses": losses}
    arrays.update({f"grad_s{k}": g for k, g in enumerate(grads)})
    arrays.update({"detections": rows[:n], "detection_offsets": offsets, "candidates": det["counts"]})
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v.astype(np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    grad_budget = DUMP_BUDGET_BYTES - DUMP_DETECTIONS_BYTES - DUMP_SMALL_BYTES
    grad_bytes = sum(arrays[f"grad_s{k}"].nbytes for k in range(len(grads)))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        pick = None
        if k.startswith("grad_s") and grad_bytes > grad_budget:
            pick = _sample_rows(a.reshape(-1), grad_budget * a.nbytes / grad_bytes)
        elif k == "detections" and a.nbytes > DUMP_DETECTIONS_BYTES:
            pick = _sample_rows(a, DUMP_DETECTIONS_BYTES)
        if pick is not None:
            np.save(os.path.join(out_dir, k + "_index.npy"), pick.astype(np.float64))
            np.save(os.path.join(out_dir, k + "_shape.npy"), np.array(a.shape, dtype=np.float64))
            a = a.reshape(-1)[pick] if k.startswith("grad_s") else a[pick]
        np.save(os.path.join(out_dir, k + ".npy"), a)


def r3(x):
    """3 significant digits for the compact line."""
    if x is None:
        return None
    x = float(x)
    if x == 0.0 or x != x:
        return x
    from math import floor, log10
    return round(x, max(0, 2 - int(floor(log10(abs(x))))))


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvml)
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.stop_flag, self.max_mhz, self.ok = [], set(), False, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.003)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs nvml reports as local to GPU `index`, so that the pinned host buffers
    allocated afterwards are first-touched on that NUMA node (the H2D path then does not cross the
    socket interconnect).  Returns a short description for the result line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [w * 64 + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1 and w * 64 + b < n_cpu]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return "off (nvml reports no local CPUs)"
        os.sched_setaffinity(0, allowed)
        return f"gpu-local cpus ({len(allowed)} of {n_cpu})"
    except Exception as e:  # pragma: no cover
        return f"off ({type(e).__name__})"


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's CPU implementation of the path on the host cores
# ------------------------------------------------------------------------------------------------
class _PresetHeadsModel:
    """Stands in for the YOLO model inside the reference's predict(): the conv backbone is out of scope
    (SURVEY 8), so the model call returns the synthetic heads of the image being predicted."""

    def __init__(self, img_size, anchors):
        self.img_size, self.anchors, self.heads = img_size, anchors, None

    def eval(self):
        return self

    def __call__(self, img):
        return self.heads


def load_unmodified_reference():
    """The reference's train.py as staged (byte-identical copy) in baseline/_ref by __graft_entry__.build();
    None when it is not there (then the oracle port of the same code path is used)."""
    path = os.path.join(REF_DIR, "train.py")
    if not os.path.exists(path):
        return None
    import importlib.util
    spec = importlib.util.spec_from_file_location("yolo_reference_train_unmodified", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_cpu_reference(args, sample_images, steps, warmup):
    """loss fwd+bwd (torch CPU, all threads) + per-image decode/filter/NMS (train.py:1152-1238), images spread
    over the host threads.  Returns (images/s, ms per step, cores, kind, sample description)."""
    from concurrent.futures import ThreadPoolExecutor
    import tempfile
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    ref = load_unmodified_reference()
    heads = [h[:sample_images].contiguous() for h in make_heads(args.batch, args.img, args.nc, 1234)]
    labels = make_labels(np.random.default_rng(4321), args.batch, args.nc)[:sample_images]
    grids = [args.img // 8, args.img // 16, args.img // 32]
    from oracle import ref_path as R   # the CPU arm is the one place bench.py may execute oracle/
    anchors = R.default_anchors()
    tg = [R.assign_targets(l, anchors, grids, args.nc, args.img) for l in labels]
    tgts = [torch.from_numpy(np.stack([t[s] for t in tg])) for s in range(3)]
    workers = max(1, min(cores, sample_images))
    pool = ThreadPoolExecutor(max_workers=workers)
    tmp = tempfile.TemporaryDirectory()
    if ref is not None:
        from PIL import Image
        img_path = os.path.join(tmp.name, "blank.png")  # letterbox identity: predict() reads it, the preset heads ignore it
        Image.fromarray(np.zeros((args.img, args.img, 3), dtype=np.uint8)).save(img_path)
        cpu = torch.device("cpu")

        def one(b):
            m = _PresetHeadsModel(args.img, anchors)
            m.heads = [h[b:b + 1] for h in heads]
            return len(ref.predict(m, img_path, cpu, num_classes=args.nc, conf_threshold=args.conf, iou_threshold=args.iou))

        def loss():
            preds = [h.clone().requires_grad_(True) for h in heads]
            total = ref.yolo_loss_multiscale(preds, tgts, anchors, args.nc)[0]
            total.backward()
            return float(total.detach())
        kind = "reference"
        what = "UNMODIFIED reference (baseline/_ref/train.py): yolo_loss_multiscale(...).backward() on torch CPU + predict() per image on preset heads (torchvision CPU batched_nms)"
    else:
        import torchvision

        def one(b):
            bx, sc, cl = R.candidates([h[b:b + 1] for h in heads], anchors, args.img, args.nc, args.conf)
            return int(torchvision.ops.batched_nms(bx, sc, cl, args.iou).numel()) if bx.shape[0] else 0

        def loss():
            preds = [h.clone().requires_grad_(True) for h in heads]
            total = R.multiscale_loss(preds, tgts, anchors, args.nc)[0]
            total.backward()
            return float(total.detach())
        kind = "port"
        what = "oracle port of the reference's CPU path: loss fwd+bwd on torch CPU + per-image decode/filter/torchvision CPU batched_nms"

    def step():
        loss()
        return list(pool.map(one, range(sample_images)))

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    pool.shutdown()
    tmp.cleanup()
    sample = f"{sample_images} of {args.batch} images/step, {steps} steps; {what}; {workers} threads"
    return sample_images / dt, dt * 1e3, cores, kind, sample


def reference_main(args, rank):
    if rank != 0:
        return
    if hasattr(os, "sched_setaffinity"):
        try:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
        except OSError:
            pass
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    if args.cpu_sample > 0:
        sample_images = max(1, min(args.batch, args.cpu_sample))
    elif args.cpu_sample < 0:
        sample_images = args.batch
    else:  # bounded sample: a calibration pass on 2 images sizes the step so that K+W steps fit the budget
        n_cal = min(2, args.batch)
        _, ms_cal, _, _, _ = run_cpu_reference(args, n_cal, 1, 0)
        per_image_s = ms_cal * 1e-3 / n_cal
        sample_images = int(max(1, min(args.batch, args.cpu_budget_s / ((steps + warmup) * per_image_s))))
    v, ms, cores, kind, sample = run_cpu_reference(args, sample_images, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(args):
    """cpu_baseline of the product line: the reference arm in a fresh process (no CUDA context, full CPU
    affinity), bounded: 2 steps + 1 warm-up over the batch (about 10-20 s)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
           "--nc", str(args.nc), "--img", str(args.img), "--batch", str(args.batch), "--conf", str(args.conf),
           "--iou", str(args.iou), "--cpu-sample", str(args.cpu_sample), "--cpu-budget-s", "25"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
        lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
        d = json.loads(lines[-1])
        cb = d["cpu_baseline"]
        cb["ms_per_step"] = d["ms_per_step"]
        return cb
    except Exception as e:  # pragma: no cover
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e!r}"[:200]}


def workload_config(args, world, n_sets=4):
    base = (args.nc, args.img, args.batch) == (1, 640, 64)
    return {
        "workload": f"BASELINE {'configs[1]' if base else 'variant'}: nc={args.nc} heads {args.img}x{args.img}, "
                    f"{args.batch} images/GPU, <={MAX_GT} GT/image, randn heads, conf {args.conf}, iou {args.iou}",
        "global_batch": args.batch * world, "images_per_gpu": args.batch, "img_size": args.img, "nc": args.nc,
        "conf_thres": args.conf, "iou_thres": args.iou, "parallelism": f"image-sharded x{world}",
        "head_layout": args.layout, "targets": args.targets,
        "l2": f"inputs rotate over {n_sets} sets/rank (> 126 MB L2)",
    }


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
OTHER_CONFIGS = {  # BASELINE.json configs[2], configs[3]: (nc, img, images/GPU, conf, head layout, targets)
    "cfg2_nc80_640_B64_conf.001": (80, 640, 64, 0.001, "bhwac", "dense"),
    "cfg3_nc80_1280_B32_conf.001": (80, 1280, 32, 0.001, "bhwac", "dense"),
    # the same work on the 'next' rows of SURVEY 8f: NCHW conv output read directly + label-list targets
    "cfg1_nchw_labels": (1, 640, 64, 0.5, "nchw", "labels"),
    "cfg2_nchw_labels": (80, 640, 64, 0.001, "nchw", "labels"),
}
SHARDED_CONFIGS = {  # BASELINE.json configs[4]: nc=80, 640^2, global batch 64 x N sharded by image (N=8: 512)
    "cfg4_nc80_640_B64perGPU_conf.001": (80, 640, 64, 0.001, "bhwac", "dense"),
}


def b200_main(args, rank, local_rank, world):
    import yolo_from_scratch_b200 as yb
    lib = yb._lib.lib()  # raises if the CUDA extension is missing: no fallback
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl b200) needs a GPU; the CUDA path has no fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if args.numa == "auto" else "off"
    group = None
    if world > 1:
        import torch.distributed as dist
        import datetime
        # a short collective timeout: a rank-asymmetric bug must fail in minutes, not hold N GPUs for the default 10
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
        group = dist.group.WORLD
    full = run_workload(args, rank, local_rank, world, dev, group, lib, full=True)
    others = {}
    if not args.no_other_configs:
        import copy
        for name, (nc, img, batch, conf, layout, targets) in (OTHER_CONFIGS if world == 1 else SHARDED_CONFIGS).items():
            a2 = copy.copy(args)
            a2.nc, a2.img, a2.batch, a2.conf, a2.layout, a2.targets = nc, img, batch, conf, layout, targets
            a2.steps, a2.warmup, a2.reps = max(3, min(args.steps, 6)), 3, 3
            o = run_workload(a2, rank, local_rank, world, dev, group, lib, full=False)   # every rank takes part
            if rank == 0:
                others[name] = o
            torch.cuda.empty_cache()
    dist_parity = None
    if world > 1:
        dist_parity = check_dist_parity(yb, dev, rank, world, group)
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
        if not dist_parity["ok"]:
            raise SystemExit(f"sharded loss differs from the single-rank loss: {dist_parity}")
    if rank != 0:
        return
    full["numa"] = numa
    full_out = args.full_out
    if full_out is None:   # a new file of this run's own: the temporary directory may be shared by several users
        fd, full_out = tempfile.mkstemp(prefix="yolo_b200_bench_full_", suffix=".json")
        os.close(fd)
    full["full_out"] = full_out or None
    full["other_configs"] = others
    full["dist_parity"] = dist_parity
    if not args.no_cpu_baseline:
        full["cpu_baseline"] = cpu_baseline_subprocess(args)
    line = compact_line(full)
    if full_out:
        try:
            os.makedirs(os.path.dirname(full_out) or ".", exist_ok=True)
            with open(full_out, "w") as f:
                json.dump(full, f, indent=1)
        except OSError as e:  # pragma: no cover
            print(f"bench.py: could not write {full_out}: {e}", file=sys.stderr)
    print(json.dumps(line, separators=(",", ":")), flush=True)


def compact_line(full):
    """The ONE line the driver parses: the contract keys plus roofline, hbm_kernels (name -> [us, frac of the
    measured HBM peak]), cpu_baseline and e2e; everything else stays in the full result file."""
    def pick(d, keys):
        return None if d is None else {k: (r3(d[k]) if isinstance(d.get(k), float) else d.get(k)) for k in keys if k in d}
    roof = full.get("roofline") or {}
    line = {k: full[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                                 "scaling", "vs_baseline", "dtype", "data", "config")}
    line["value"], line["ms_per_step"] = r3(full["value"]) if full["value"] < 1e3 else round(full["value"], 1), round(full["ms_per_step"], 5)
    line["timing"] = {"launch": full["launch"], "reps": full["reps"], "ms_per_step_min_max": [round(x, 5) for x in full["ms_per_step_min_max"]],
                      "timed_ms_total": r3(full["timed_ms_total"]), "eager_ms_per_step": r3(full["eager"]["ms_per_step"]),
                      "loss_fwd_bwd_ms": r3(full["loss_fwd_bwd_ms"]), "decode_nms_ms": r3(full["decode_nms_ms"]),
                      "pipelined_2_streams_ms_per_step": r3((full.get("pipelined_2_streams") or {}).get("ms_per_step")),
                      "kernel_times": "cuda events around every launch of the eager pass (same K steps)"}
    line["roofline"] = pick(roof, ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic", "share", "us",
                                   "algorithmic_speedup", "what", "peak_source"))
    line["hbm_kernels"] = {k: [r3(v["us"]), r3(v["frac"])] for k, v in (full.get("hbm_kernels") or {}).items()}
    line["kernels_us"] = {k: r3(v["avg_ms"] * 1e3) for k, v in (full.get("kernels") or {}).items()}
    cb = full.get("cpu_baseline")
    line["cpu_baseline"] = None if cb is None else {"value": r3(cb.get("value")), "unit": cb.get("unit"), "cores": cb.get("cores"),
                                                    "kind": cb.get("kind"), "sample": str(cb.get("sample"))[:160]}
    tg = full.get("torch_gpu_baseline")
    if tg:
        line["torch_gpu_baseline"] = pick(tg, ("value", "unit", "loss_fwd_bwd_ms", "decode_nms_ms_per_image", "error"))
    e2e_keys = ("value", "unit", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step", "copy_ceiling", "frac_of_copy_ceiling", "api")
    line["e2e"] = pick(full.get("e2e"), e2e_keys)
    if full.get("e2e_labels"):
        line["e2e_labels"] = pick(full["e2e_labels"], e2e_keys)
    if full.get("e2e_graph"):
        line["e2e_graph"] = pick(full["e2e_graph"], e2e_keys[:-1] + ("error",))
    line["gpu_launches"] = full["gpu_launches"]
    line["clocks"] = full["clocks"]
    oc = full.get("other_configs") or {}
    if oc:
        line["configs"] = {k: (round(v["value"], 1) if v and "value" in v else None) for k, v in oc.items()}
    if full.get("variants"):
        line["variants"] = {k: round(v["decode_nms_images_per_s"], 1) for k, v in full["variants"].items()}
    if full.get("dist_parity") is not None:
        line["dist_parity"] = full["dist_parity"]
    line["numa"] = full.get("numa")
    line["full"] = full.get("full_out")
    n = len(json.dumps(line, separators=(",", ":")))
    for drop in ("kernels_us", "variants", "e2e_graph", "torch_gpu_baseline", "numa"):  # never exceed the driver's parse window
        if n <= MAX_LINE_BYTES:
            break
        line.pop(drop, None)
        n = len(json.dumps(line, separators=(",", ":")))
    return line


def check_dist_parity(yb, dev, rank, world, group):
    """Outside every timed region: the sharded loss (one NCCL all-reduce of S*4 doubles) on a small fixed case
    must equal the single-rank loss over the whole batch, values and gradient rows, on THIS hardware."""
    import torch.distributed as dist
    from yolo_from_scratch_b200 import dist as ybd
    from yolo_from_scratch_b200 import ops
    per, nc, img = 3, 3, 160
    B = per * world
    grids = [img // 8, img // 16, img // 32]
    heads = make_heads(B, img, nc, 777)
    labels = make_labels(np.random.default_rng(778), B, nc)
    anchors = ops.default_anchors(dev)
    lo, hi = ybd.shard_range(B, rank, world)
    whole = [h.to(dev).requires_grad_(True) for h in heads]
    tg = ops.build_targets(labels, anchors, grids, nc, img)
    ref = ops.yolo_loss_multiscale(whole, tg, anchors, nc)
    ref[0].backward()
    mine = [h[lo:hi].to(dev).requires_grad_(True) for h in heads]
    out = ybd.yolo_loss_multiscale_sharded(mine, [t[lo:hi].contiguous() for t in tg], anchors, nc, group=group)
    out[0].backward()
    rel = max(abs(float(a) - float(b)) / max(abs(float(b)), 1e-12) for a, b in zip(out, ref))
    gerr = 0.0
    for s in range(3):
        want = whole[s].grad[lo:hi]
        gerr = max(gerr, float((mine[s].grad - want).abs().max()) / max(float(want.abs().max()), 1e-30))
    # and the label-list form (device-side assignment) on the same shard
    mine2 = [h[lo:hi].to(dev).requires_grad_(True) for h in heads]
    out2 = ops.yolo_loss_multiscale_labels(mine2, labels[lo:hi], anchors, nc, img, group=group)
    rel = max(rel, max(abs(float(a) - float(b)) / max(abs(float(b)), 1e-12) for a, b in zip(out2, ref)))
    t = torch.tensor([rel, gerr], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    rel, gerr = float(t[0]), float(t[1])
    return {"max_rel_err": r3(rel), "grad_max_rel_err": r3(gerr), "ok": bool(rel <= 1e-5 and gerr <= 1e-5),
            "case": f"{B} images sharded {per}/rank, nc={nc}, {img}^2, dense + label-list targets vs single-rank"}


def timed_reps(run_steps, steps, reps, barrier, max_over_ranks):
    """`reps` repetitions of: barrier+sync, event, K steps, event, barrier+sync.  Returns ms per step of every
    repetition (max over ranks)."""
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        run_steps(steps)
        e1.record()
        barrier()
        out.append(max_over_ranks(e0.elapsed_time(e1)) / steps)
    return out


def run_workload(args, rank, local_rank, world, dev, group, lib, full):
    import yolo_from_scratch_b200 as yb
    from yolo_from_scratch_b200 import ops
    B, img, nc = args.batch, args.img, args.nc
    # rotate over enough input sets that the working set exceeds the 126 MB L2
    T_est = sum(B * G * G * 3 for G in (img // 8, img // 16, img // 32)) * (5 + nc) * 4
    n_sets = 4 if T_est * 3 * 4 <= (8 << 30) else 2
    grids = [img // 8, img // 16, img // 32]
    anchors = ops.default_anchors(dev)  # train.py:372-374
    weights = ops.MULTISCALE_OBJ_WEIGHTS

    # n_sets input sets per rank, on the device and (full run) mirrored in pinned host memory
    layout = ops.LAYOUT_NCHW if args.layout == "nchw" else ops.LAYOUT_BHWAC
    use_labels = args.targets == "labels"
    dev_sets, host_sets, label_sets = [], [], []
    for k in range(n_sets):
        seed = 1234 + 1000 * k + 100000 * rank
        heads = make_heads(B, img, nc, seed)
        labels = make_labels(np.random.default_rng(4321 + k + 1000 * rank), B, nc)
        tg = ops.build_targets(labels, anchors, grids, nc, img)
        d_heads = [h.to(dev) for h in heads]
        if layout == ops.LAYOUT_NCHW:  # the same values as the head conv would have produced them
            d_heads = [h.permute(0, 3, 4, 1, 2).reshape(h.shape[0], -1, h.shape[1], h.shape[2]).contiguous()
                       for h in d_heads]
        packed = ops.pack_labels_host(labels, img, max_gt=MAX_GT)
        packed = ops.PackedLabels(packed[0].to(dev), packed[1].to(dev), packed[2].to(dev), img)
        dev_sets.append((d_heads, tg, packed))
        if full and not args.no_e2e:
            host_sets.append(([h.pin_memory() for h in heads], [t.cpu().pin_memory() for t in tg]))
            label_sets.append(ops.pack_labels_host(labels, img, pin=True, max_gt=MAX_GT))
        del heads
    torch.cuda.synchronize()
    T_bytes = tensor_bytes(dev_sets[0][0])
    rows = sum(B * G * G * 3 for G in grids)
    row_bytes = (5 + nc) * 4

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident step, eager launches ----------------------------------------------------
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    last_eager = {}   # outputs of the most recent eager step, for --dump-outputs with --launch eager

    def step(i, conf=None, record=None):
        heads, tg, packed = dev_sets[i % n_sets]
        if record:
            record[0].record()
        out4, per_scale, grads = ops.loss_forward_backward(heads, None if use_labels else tg, anchors, nc, weights,
                                                           [True] * 3, group=group, sparse=packed if use_labels else None,
                                                           layout=layout)
        if record:
            record[1].record()
        det = ops.detect_batch(heads, anchors, img, nc, args.conf if conf is None else conf, args.iou, layout=layout)
        if record:
            record[2].record()
        if args.dump_outputs:
            last_eager["out"] = (out4, grads, det)
        return out4, det

    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()
    # candidate statistics per input set (outside the timed region)
    pair_counts, cand_counts, keep_counts, eval_counts, edge_counts = [], [], [], [], []
    for k in range(n_sets):
        _, det = step(k)
        m = det["counts"].cpu().double()
        cand_counts.append(float(m.sum()))
        if nc > 1 and float(m.max()) * 4 > ops.TRICK_MAX_NUMEL_CUDA:
            # per-class regime: only same-class pairs are algorithmic work
            cl = det["classes"]
            valid = torch.arange(cl.shape[1], device=dev)[None, :] < det["counts"][:, None]
            oh = torch.zeros(B, nc, dtype=torch.float64, device=dev)
            oh.scatter_add_(1, cl.clamp(0, nc - 1), valid.double())
            pair_counts.append(float((oh * (oh - 1) / 2).sum()))
        else:
            pair_counts.append(float((m * (m - 1) / 2).sum()))
        keep_counts.append(float(det["n_keep"].cpu().double().sum()))
        assert int(det["n_keep"].min()) >= 0
        st = ops.nms_graph_stats(det)
        if st is not None:
            eval_counts.append(st[0])
            edge_counts.append(st[1])
        del det
    barrier()

    # eager pass: K steps with a CUDA-event pair around every launch of the library (per-kernel times)
    lib.yb_timing_enable(1)
    launches0 = lib.yb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(i, record=ev[i])
    e1.record()
    barrier()
    eager_launches = lib.yb_launch_count() - launches0
    lib.yb_timing_enable(0)
    buf = ctypes.create_string_buffer(1 << 16)
    lib.yb_timing_collect(buf, len(buf))
    loss_ms = float(np.mean([r[0].elapsed_time(r[1]) for r in ev]))
    det_ms = float(np.mean([r[1].elapsed_time(r[2]) for r in ev]))
    kernels = {}
    for ln in buf.value.decode().strip().splitlines():
        name, cnt, tot = ln.split()
        kernels[name] = {"launches_per_step": int(cnt) / args.steps, "avg_ms": float(tot) / int(cnt),
                         "ms_per_step": float(tot) / args.steps}
    ksum = sum(k["ms_per_step"] for k in kernels.values())
    for k in kernels.values():
        k["share"] = k["ms_per_step"] / ksum if ksum else 0.0
    # eager throughput without the event pairs
    def eager_steps(n):
        for i in range(n):
            step(i)

    eager_reps = timed_reps(eager_steps, args.steps, max(1, min(args.reps, 3)), barrier, max_over_ranks)
    eager_ms = float(np.median(eager_reps))

    # ---- `value`: the same step replayed as CUDA graphs (one graph per rotating input set) -----------
    sampler = ClockSampler(local_rank)
    sampler.start()
    use_graph = args.launch == "graph"
    graph_launches = None
    pipelined_ms = None
    if use_graph:
        c0 = lib.yb_launch_count()
        graphs = [yb.HotPathGraph(B, img, nc, anchors, args.conf, args.iou, max_gt=MAX_GT, layout=layout,
                                  adopt_heads=ds[0], adopt_targets=ds[2] if use_labels else ds[1], group=group)
                  for ds in dev_sets]
        graph_launches = (lib.yb_launch_count() - c0) // (3 * n_sets)   # 2 warm-up passes + 1 capture per graph
        for i in range(max(3, args.warmup)):
            graphs[i % n_sets].replay()
        sampler.samples.clear()
        def graph_steps(n):
            for i in range(n):
                graphs[i % n_sets].replay()

        reps_ms = timed_reps(graph_steps, args.steps, args.reps, barrier, max_over_ranks)
        assert int(graphs[0].det["n_keep"].min()) >= 0
        if full and rank == 0 and args.dump_outputs:
            g = graphs[(args.steps - 1) % n_sets]   # the graph the last timed step replayed
            dump_outputs(args.dump_outputs, g.losses, g.grads, g.det, g.rows, g.offsets)
        # extra (N=1 only; `value` stays the strictly sequential replay): the same K steps with the graphs of
        # consecutive input sets alternating between two streams, as a double-buffered consumer would run them — the
        # narrow tail of step i (resolve, pack: 64 CTAs) overlaps the head of step i+1.  Not used at N>1: two graphs
        # with a collective on the same communicator must not run concurrently.
        if world == 1 and full:
            two = [torch.cuda.Stream(), torch.cuda.Stream()]

            def graph_steps_2(n):
                cur = torch.cuda.current_stream()
                for st2 in two:
                    st2.wait_stream(cur)
                for i in range(n):
                    with torch.cuda.stream(two[i % 2]):
                        graphs[i % n_sets].replay()
                for st2 in two:
                    cur.wait_stream(st2)
            graph_steps_2(4)
            pipelined_ms = float(np.median(timed_reps(graph_steps_2, args.steps, max(3, args.reps // 2), barrier, max_over_ranks)))
        del graphs
        torch.cuda.empty_cache()
    else:
        sampler.samples.clear()
        reps_ms = timed_reps(eager_steps, args.steps, args.reps, barrier, max_over_ranks)
        if full and rank == 0 and args.dump_outputs:
            out4, grads, det = last_eager.pop("out")
            dump_outputs(args.dump_outputs, out4, grads, det, *ops.pack_detections(det))
    sampler.stop_flag = True
    sampler.join()
    step_ms = float(np.median(reps_ms))

    # ---- a-1: decode_predictions forward / backward on the same heads (2T / 3T bytes) ---------------
    decode = None
    if layout == ops.LAYOUT_BHWAC and (full or rank == 0):
        decode = time_decode(lib, dev_sets, anchors, img, nc, n_sets, args.steps)

    # ---- e2e through the public API with host buffers ---------------------------------------------
    e2e = e2e_labels = e2e_graph = None
    if full and not args.no_e2e:
        ceil_dense = run_copy_ceiling(args, dev, world, host_sets, None, n_sets, barrier, max_over_ranks)
        ceil_labels = run_copy_ceiling(args, dev, world, host_sets, label_sets, n_sets, barrier, max_over_ranks)
        e2e = run_e2e(args, yb, ops, dev, group, world, host_sets, anchors, weights, grids, n_sets, barrier,
                      max_over_ranks)
        e2e_labels = run_e2e(args, yb, ops, dev, group, world, host_sets, anchors, weights, grids, n_sets, barrier,
                             max_over_ranks, label_sets=label_sets)
        for e, c in ((e2e, ceil_dense), (e2e_labels, ceil_labels)):
            e["copy_ceiling"] = c["value"]
            e["copy_ceiling_gbs_per_rank"] = c["h2d_gbs_per_rank"]
            e["frac_of_copy_ceiling"] = e["value"] / c["value"]
        if world == 1:
            try:
                e2e_graph = run_e2e_graph(args, yb, ops, dev, world, host_sets, label_sets, anchors, grids, n_sets,
                                          barrier, max_over_ranks)
                e2e_graph["copy_ceiling"] = ceil_labels["value"]
                e2e_graph["frac_of_copy_ceiling"] = e2e_graph["value"] / ceil_labels["value"]
            except Exception as e:  # pragma: no cover
                e2e_graph = {"error": repr(e)[:200]}

    # ---- variants: other confidence thresholds (device-resident, detect only) ---------------------
    variants = {}
    if full and not args.no_variants and rank == 0:
        import gc
        gc.collect()              # the e2e legs' CUDA graphs and pools are released here, not inside a timed loop
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
        for conf in (0.25, 0.001):
            for i in range(4):  # detect only: rank 0 runs this alone, so no collective may be enqueued here
                ops.detect_batch(dev_sets[i % n_sets][0], anchors, img, nc, conf, args.iou, layout=layout)
            torch.cuda.synchronize()
            n_it = max(5, args.steps // 3)
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_it + 1)]
            evs[0].record()
            for i in range(n_it):
                heads = dev_sets[i % n_sets][0]
                det = ops.detect_batch(heads, anchors, img, nc, conf, args.iou, layout=layout)
                evs[i + 1].record()
            torch.cuda.synchronize()
            ms = float(np.median([evs[i].elapsed_time(evs[i + 1]) for i in range(n_it)]))
            variants[f"conf_{conf}"] = {"decode_nms_ms": ms, "decode_nms_images_per_s": B / (ms * 1e-3),
                                        "candidates_per_image": float(det["counts"].double().mean()),
                                        "kept_per_image": float(det["n_keep"].double().mean())}
            del det
        # SURVEY 8d's "prior" heads: objectness logit 2*randn - 4.6 (a detector's prior: ~4 % of the rows pass conf 0.25)
        prior_sets = []
        for k in range(n_sets):
            hs = [h.clone() for h in dev_sets[k][0]]
            for h in hs:
                if layout == 1:   # NCHW: the objectness planes are channels a*row + 4
                    h[:, 4::5 + nc].mul_(2.0).sub_(4.6)
                else:
                    h[..., 4].mul_(2.0).sub_(4.6)
            prior_sets.append(hs)
        for i in range(4):
            ops.detect_batch(prior_sets[i % n_sets], anchors, img, nc, 0.25, args.iou, layout=layout)
        torch.cuda.synchronize()
        n_it = max(5, args.steps // 3)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_it + 1)]
        evs[0].record()
        for i in range(n_it):
            det = ops.detect_batch(prior_sets[i % n_sets], anchors, img, nc, 0.25, args.iou, layout=layout)
            evs[i + 1].record()
        torch.cuda.synchronize()
        ms = float(np.median([evs[i].elapsed_time(evs[i + 1]) for i in range(n_it)]))
        variants["prior_conf_0.25"] = {"decode_nms_ms": ms, "decode_nms_images_per_s": B / (ms * 1e-3),
                                       "candidates_per_image": float(det["counts"].double().mean()),
                                       "kept_per_image": float(det["n_keep"].double().mean())}
        del det, prior_sets
    barrier()

    torch_gpu = None
    if full and world == 1 and rank == 0 and not args.no_torch_gpu_baseline:
        try:
            torch_gpu = run_torch_gpu_reference(args, dev, min(B, 8))
        except Exception as e:  # pragma: no cover
            torch_gpu = {"error": repr(e)[:200]}

    if rank != 0:
        return None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json"))).get(
            f"nc{nc}_img{img}_B{B}", {})
    except Exception:
        pass
    clocks = sampler.summary()
    sm_mhz = clocks.get("sm_mhz") or 1965.0

    # ---- HBM-bound kernels: algorithmic bytes (SURVEY 8d) / measured launch time --------------------
    pos = float(np.mean([sum(float((t[..., 4] > 0.5).sum()) for t in ds[1]) for ds in dev_sets]))
    M_tot = float(np.mean(cand_counts))
    sector = min(row_bytes, 32)
    obj_read = rows * (4 if args.layout == "nchw" else sector)
    alg_bytes = {
        # T (dense grad write) + obj sectors of pred and target + positive rows of pred and target
        "loss_main_kernel": T_bytes + (1 if use_labels else 2) * rows * sector + 2 * pos * row_bytes,
        # NCHW: the objectness logits are contiguous planes (4 B per row); dense targets keep their sectors
        "loss_main_nchw_kernel": T_bytes + rows * 4 + (rows / 8 if use_labels else rows * sector),
        # two-pass filter: objectness sector of every row, then again + the candidate rows + 28 B of output per candidate
        "filter_count_kernel": obj_read,
        "filter_emit_kernel": obj_read + M_tot * row_bytes + 28 * M_tot,
        # one-pass filter: every objectness sector once + candidate rows + outputs
        "filter_onepass_kernel": obj_read + M_tot * max(row_bytes - sector, 0) + 28 * M_tot,
    }
    hbm_kernels = {}
    for name, a_bytes in alg_bytes.items():
        if name in kernels:
            ach = a_bytes / (kernels[name]["avg_ms"] * 1e-3) / 1e9
            hbm_kernels[name] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                                 "us": kernels[name]["avg_ms"] * 1e3, "algorithmic_bytes": a_bytes,
                                 "share": kernels[name]["share"], "traffic": traffic.get(name), "peak_source": peak_src}
    if decode:
        for name, (ms, nbytes) in decode.items():
            ach = nbytes / (ms * 1e-3) / 1e9
            hbm_kernels[name] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                                 "us": ms * 1e3, "algorithmic_bytes": nbytes, "share": None, "traffic": traffic.get(name),
                                 "peak_source": peak_src}
    # ---- NMS: executed IoU pair tests against the fp32 issue rate --------------------------------------
    pairs = float(np.mean(pair_counts))
    issue_peak = 148 * 4 * 32 * sm_mhz * 1e6 / 17.0 / 1e9  # Gpair/s at 17 warp-instructions per 32 pairs
    nms_ms = sum(kernels[k]["ms_per_step"] for k in kernels if k.startswith(("graph_", "nms_")))
    nms_roof = {}
    if "graph_edge_kernel" in kernels:
        ek = kernels["graph_edge_kernel"]
        evald = float(np.mean(eval_counts)) if eval_counts else None  # pair tests executed (yb_nms_graph_stats)
        ach = (evald / (ek["avg_ms"] * 1e-3) / 1e9) if evald else None
        nms_roof = {
            "kernel": "graph_edge_kernel", "bound": "fp32-issue", "unit": "Gpair/s", "peak": issue_peak,
            "peak_source": "148 SM x 4 schedulers x 32 lanes x sampled SM clock / 17 warp-instr per 32 exact IoU>thr tests "
                           "(SASS of the dense bitmask kernel)",
            "what": "IoU pair tests EXECUTED per launch / launch time; the pairs the graph algorithm culls are in algorithmic_speedup",
            "achieved": ach, "frac": (ach / issue_peak) if ach else None,
            "evaluated_pairs_per_launch": evald,
            "algorithmic_pairs_per_launch": pairs,          # what torchvision's kernel evaluates: M(M-1)/2 per image
            "algorithmic_speedup": (pairs / evald) if evald else None,
            "algorithmic_gpairs": pairs / (ek["avg_ms"] * 1e-3) / 1e9,
            "edges_per_launch": float(np.mean(edge_counts)) if edge_counts else None,
            "whole_nms_algorithmic_gpairs": pairs / (nms_ms * 1e-3) / 1e9 if nms_ms else None,
            "us": ek["avg_ms"] * 1e3, "share": ek["share"], "traffic": traffic.get("graph_edge_kernel"),
        }
    dominant = max(kernels, key=lambda k: kernels[k]["share"]) if kernels else None
    if dominant in hbm_kernels:
        roofline = dict(hbm_kernels[dominant], kernel=dominant)
    elif dominant == "graph_edge_kernel":
        roofline = dict(nms_roof)
    else:
        roofline = {"kernel": dominant, "bound": "latency", "achieved": None, "peak": None, "frac": None,
                    "share": kernels[dominant]["share"] if dominant else None,
                    "us": kernels[dominant]["avg_ms"] * 1e3 if dominant else None}

    result = {
        "metric": METRIC, "value": B * world / (step_ms * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world, n_sets),
        "launch": ("cuda-graph replay (HotPathGraph per input set" + (", NCCL all-reduce captured inside)" if world > 1 else ")"))
                  if use_graph else "eager",
        "reps": args.reps, "ms_per_step_reps": reps_ms, "ms_per_step_min_max": [min(reps_ms), max(reps_ms)],
        "timed_ms_total": float(sum(reps_ms)) * args.steps,
        "pipelined_2_streams": None if pipelined_ms is None else {
            "ms_per_step": pipelined_ms, "value": B * world / (pipelined_ms * 1e-3), "unit": UNIT,
            "what": "the same graphs replayed on two alternating streams (consecutive steps overlap); not `value`"},
        "eager": {"value": B * world / (eager_ms * 1e-3), "ms_per_step": eager_ms, "unit": UNIT, "reps_ms": eager_reps,
                  "what": "the same K steps with eager launches (one launch per kernel from Python/ctypes)"},
        "loss_fwd_bwd_ms": loss_ms, "decode_nms_ms": det_ms, "decode_nms_images_per_s": B * world / (det_ms * 1e-3),
        "candidates_per_image": float(np.mean(cand_counts)) / B, "kept_per_image": float(np.mean(keep_counts)) / B,
        "e2e": e2e, "e2e_labels": e2e_labels, "e2e_graph": e2e_graph,
        # kernels of libyolo_b200.so that execute inside ONE K-step timed region
        "gpu_launches": int((graph_launches if use_graph else eager_launches / args.steps) * args.steps),
        "gpu_launches_note": "kernels of libyolo_b200.so per K-step timed region: counted at graph capture (replays re-run them) "
                             "or, eager, by the library's launch counter",
        "kernels": kernels, "roofline": roofline, "hbm_kernels": hbm_kernels, "roofline_nms": nms_roof,
        "cpu_baseline": None, "torch_gpu_baseline": torch_gpu, "clocks": clocks, "variants": variants,
    }
    del dev_sets, host_sets
    return result


def time_decode(lib, dev_sets, anchors, img, nc, n_sets, steps):
    """decode_predictions forward and backward (a-1) over the three heads, CUDA events on the launching stream,
    rotating input sets.  Returns {name: (ms per pass over all scales, algorithmic bytes)}."""
    st = torch.cuda.current_stream().cuda_stream
    outs = [[torch.empty_like(h) for h in ds[0]] for ds in dev_sets[:2]]
    T = tensor_bytes(dev_sets[0][0])

    def fwd(i):
        for s, h in enumerate(dev_sets[i % n_sets][0]):
            B, H, W, A, row = h.shape
            lib.yb_decode_fwd(h.data_ptr(), anchors[s].data_ptr(), outs[i % 2][s].data_ptr(), B, H, W, A, row - 5, float(img), st)

    def bwd(i):
        for s, h in enumerate(dev_sets[i % n_sets][0]):
            B, H, W, A, row = h.shape
            lib.yb_decode_bwd(h.data_ptr(), anchors[s].data_ptr(), dev_sets[(i + 1) % n_sets][0][s].data_ptr(),
                              outs[i % 2][s].data_ptr(), B, H, W, A, row - 5, float(img), st)
    T3 = tensor_bytes(dev_sets[0][0][:1])

    def box_sectors(heads):   # the backward reads only the four box logits of pred: one 32-byte sector per row (SURVEY 8d's granularity)
        return sum(h.numel() // h.shape[-1] * min(h.shape[-1] * 4, 32) for h in heads)
    Tb, Tb3 = box_sectors(dev_sets[0][0]), box_sectors(dev_sets[0][0][:1])

    def fwd_p3(i):   # the reference's call is per scale (train.py:796): the P3 head alone is the launch that carries the bytes
        h = dev_sets[i % n_sets][0][0]
        B, H, W, A, row = h.shape
        lib.yb_decode_fwd(h.data_ptr(), anchors[0].data_ptr(), outs[i % 2][0].data_ptr(), B, H, W, A, row - 5, float(img), st)

    def bwd_p3(i):
        h = dev_sets[i % n_sets][0][0]
        B, H, W, A, row = h.shape
        lib.yb_decode_bwd(h.data_ptr(), anchors[0].data_ptr(), dev_sets[(i + 1) % n_sets][0][0].data_ptr(),
                          outs[i % 2][0].data_ptr(), B, H, W, A, row - 5, float(img), st)
    res = {}
    for name, fn, nbytes in (("decode_fwd(3 scales)", fwd, 2 * T), ("decode_bwd(3 scales)", bwd, 2 * T + Tb),
                             ("decode_fwd(P3)", fwd_p3, 2 * T3), ("decode_bwd(P3)", bwd_p3, 2 * T3 + Tb3)):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        res[name] = (a.elapsed_time(b) / steps, nbytes)
    return res


def run_copy_ceiling(args, dev, world, host_sets, label_sets, n_sets, barrier, max_over_ranks):
    """The host->device ceiling of the e2e legs: the same pinned buffers copied into device buffers, no kernels,
    every rank at once, K steps."""
    slots = []
    for k in range(2):
        heads_d = [torch.empty_like(h, device=dev) for h in host_sets[0][0]]
        if label_sets is None:
            extra = [torch.empty_like(t, device=dev) for t in host_sets[0][1]]
        else:
            extra = [torch.empty_like(t, device=dev) for t in label_sets[0]]
        slots.append((heads_d, extra))
    nbytes = tensor_bytes(slots[0][0]) + tensor_bytes(slots[0][1])

    def run(n):
        for i in range(n):
            hd, ex = slots[i % 2]
            for d, h in zip(hd, host_sets[i % n_sets][0]):
                d.copy_(h, non_blocking=True)
            for d, h in zip(ex, host_sets[i % n_sets][1] if label_sets is None else label_sets[i % n_sets]):
                d.copy_(h, non_blocking=True)
    run(3)
    barrier()
    t0 = time.perf_counter()
    run(args.steps)
    torch.cuda.synchronize()
    ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    barrier()
    return {"value": args.batch * world / (ms * 1e-3), "ms_per_step": ms, "h2d_bytes_per_step": nbytes,
            "h2d_gbs_per_rank": nbytes / (ms * 1e-3) / 1e9}


def run_e2e(args, yb, ops, dev, group, world, host_sets, anchors, weights, grids, n_sets, barrier, max_over_ranks,
            label_sets=None):
    """The same step through the public API with pinned HOST buffers.  Every step copies its inputs
    host->device (heads + dense targets for the reference-signature call; heads + packed label lists
    for the sparse-target call when `label_sets` is given), runs loss fwd+bwd, detect and pack, and
    copies the 4 losses and the detection rows device->host — all inside the timed region.  Copies and
    kernels are pipelined over three input slots (copy stream / compute stream / result stream): step
    i+1's inputs travel while step i computes, as a training loop's prefetching loader does."""
    B, img, nc = args.batch, args.img, args.nc
    comp = torch.cuda.current_stream()
    h2d_stream, d2h_stream = torch.cuda.Stream(), torch.cuda.Stream()
    n_slots = 3
    slots = []
    for k in range(n_slots):
        heads_d = [torch.empty_like(h, device=dev) for h in host_sets[0][0]]
        if label_sets is None:
            tg_d = [torch.empty_like(t, device=dev) for t in host_sets[0][1]]
        else:
            lab, n_gt, lb = label_sets[0]
            tg_d = ops.PackedLabels(torch.empty_like(lab, device=dev), torch.empty_like(n_gt, device=dev),
                                    torch.empty_like(lb, device=dev), img)
        slots.append({"heads": heads_d, "tg": tg_d, "ready": torch.cuda.Event(), "free": torch.cuda.Event(),
                      "loss_host": torch.empty(4, dtype=torch.float32).pin_memory(),
                      "off_host": torch.empty(B + 1, dtype=torch.int32).pin_memory(),
                      "off_ready": torch.cuda.Event(), "rows_done": torch.cuda.Event(),
                      "det_host": torch.empty(B * sum(G * G * 3 for G in grids), 6, dtype=torch.float32).pin_memory()})
    if label_sets is None:
        h2d = tensor_bytes(host_sets[0][0]) + tensor_bytes(host_sets[0][1])
    else:
        h2d = tensor_bytes(host_sets[0][0]) + tensor_bytes(list(label_sets[0]))
    d2h_acc = []

    def enqueue_h2d(i):
        sl = slots[i % n_slots]
        with torch.cuda.stream(h2d_stream):
            h2d_stream.wait_event(sl["free"])          # the slot's previous user has finished computing
            for d, h in zip(sl["heads"], host_sets[i % n_sets][0]):
                d.copy_(h, non_blocking=True)
            if label_sets is None:
                for d, h in zip(sl["tg"], host_sets[i % n_sets][1]):
                    d.copy_(h, non_blocking=True)
            else:
                lab, n_gt, lb = label_sets[i % n_sets]
                sl["tg"].labels.copy_(lab, non_blocking=True)
                sl["tg"].n_gt.copy_(n_gt, non_blocking=True)
                sl["tg"].letterbox.copy_(lb, non_blocking=True)
            sl["ready"].record(h2d_stream)

    def compute(i):
        sl = slots[i % n_slots]
        comp.wait_event(sl["ready"])
        comp.wait_event(sl["rows_done"])               # the slot's host result buffers are free again
        preds = [h.detach().requires_grad_(True) for h in sl["heads"]]
        if label_sets is not None:
            total, bbox, obj, cls = ops.yolo_loss_multiscale_labels(preds, sl["tg"], anchors, nc, img, group=group)
        elif group is None:
            total, bbox, obj, cls = yb.yolo_loss_multiscale(preds, sl["tg"], anchors, nc)
        else:
            total, bbox, obj, cls = ops._loss_common(preds, sl["tg"], anchors, nc, weights, group=group)
        total.backward()
        sl["loss_host"].copy_(torch.stack([total.detach(), bbox.detach(), obj.detach(), cls.detach()]),
                              non_blocking=True)
        det = yb.detect_batch(sl["heads"], anchors, img, nc, args.conf, args.iou)
        rows_d, offsets = yb.pack_detections(det)
        sl["off_host"].copy_(offsets, non_blocking=True)
        sl["free"].record(comp)
        sl["off_ready"].record(comp)
        sl["rows_d"], sl["grads"] = rows_d, [p.grad for p in preds]

    def collect(i):
        sl = slots[i % n_slots]
        sl["off_ready"].synchronize()                  # host needs the row count; step i+1's H2D is in flight
        n = int(sl["off_host"][-1])
        if n < 0:
            raise RuntimeError("NMS reported a failed image")
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(sl["off_ready"])
            sl["det_host"][:n].copy_(sl["rows_d"][:n], non_blocking=True)
            sl["rows_d"].record_stream(d2h_stream)
            sl["rows_done"].record(d2h_stream)
        d2h_acc.append(16 + sl["off_host"].numel() * 4 + n * 24)

    def run(n_steps):
        # software pipeline: inputs of step i+2 travel and step i+1 is already enqueued while the host
        # waits for the row count of step i
        enqueue_h2d(0)
        if n_steps > 1:
            enqueue_h2d(1)
        compute(0)
        for i in range(n_steps):
            if i + 2 < n_steps:
                enqueue_h2d(i + 2)
            if i + 1 < n_steps:
                compute(i + 1)
            collect(i)
        d2h_stream.synchronize()
        comp.synchronize()

    run(max(3, args.warmup))
    d2h_acc.clear()
    barrier()
    t0 = time.perf_counter()
    run(args.steps)
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    e2e_ms = max_over_ranks(wall_ms) / args.steps
    api = ("yolo_loss_multiscale_labels(heads, label lists)" if label_sets is not None
           else "yolo_loss_multiscale(heads, dense targets)")
    return {"value": B * world / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(np.mean(d2h_acc)),
            "api": api + ".backward()+detect_batch+pack_detections; pinned host in/out, 3-slot pipeline, host wall clock"}


def run_e2e_graph(args, yb, ops, dev, world, host_sets, label_sets, anchors, grids, n_sets, barrier, max_over_ranks):
    """e2e with the step captured as a CUDA graph (yb.HotPathGraph, label-list targets): per step the
    pinned host heads + packed labels are copied into a graph's static inputs, the graph is replayed,
    and the 4 losses + detection rows are copied back.  Three graphs = three pipeline slots."""
    B, img, nc = args.batch, args.img, args.nc
    comp = torch.cuda.current_stream()
    h2d_stream, d2h_stream = torch.cuda.Stream(), torch.cuda.Stream()
    n_slots = 3
    slots = []
    for k in range(n_slots):
        hp = yb.HotPathGraph(B, img, nc, anchors, args.conf, args.iou, max_gt=MAX_GT, targets="labels")
        slots.append({"hp": hp, "ready": torch.cuda.Event(), "free": torch.cuda.Event(),
                      "loss_host": torch.empty(4, dtype=torch.float32).pin_memory(),
                      "off_host": torch.empty(B + 1, dtype=torch.int32).pin_memory(),
                      "off_ready": torch.cuda.Event(), "rows_done": torch.cuda.Event(),
                      "det_host": torch.empty(B * sum(G * G * 3 for G in grids), 6, dtype=torch.float32).pin_memory()})
    h2d = tensor_bytes(host_sets[0][0]) + tensor_bytes(list(label_sets[0]))
    d2h_acc = []

    def enqueue_h2d(i):
        sl = slots[i % n_slots]
        hp = sl["hp"]
        with torch.cuda.stream(h2d_stream):
            h2d_stream.wait_event(sl["free"])
            for d, h in zip(hp.heads, host_sets[i % n_sets][0]):
                d.copy_(h, non_blocking=True)
            lab, n_gt, lb = label_sets[i % n_sets]
            hp.labels.labels.copy_(lab, non_blocking=True)
            hp.labels.n_gt.copy_(n_gt, non_blocking=True)
            hp.labels.letterbox.copy_(lb, non_blocking=True)
            sl["ready"].record(h2d_stream)

    def compute(i):
        sl = slots[i % n_slots]
        hp = sl["hp"]
        comp.wait_event(sl["ready"])
        comp.wait_event(sl["rows_done"])
        hp.replay()
        sl["loss_host"].copy_(hp.losses, non_blocking=True)
        sl["off_host"].copy_(hp.offsets, non_blocking=True)
        sl["free"].record(comp)
        sl["off_ready"].record(comp)

    def collect(i):
        sl = slots[i % n_slots]
        sl["off_ready"].synchronize()
        n = int(sl["off_host"][-1])
        if n < 0:
            raise RuntimeError("NMS reported a failed image")
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(sl["off_ready"])
            sl["det_host"][:n].copy_(sl["hp"].rows[:n], non_blocking=True)
            sl["rows_done"].record(d2h_stream)
        d2h_acc.append(16 + sl["off_host"].numel() * 4 + n * 24)

    def run(n_steps):
        enqueue_h2d(0)
        if n_steps > 1:
            enqueue_h2d(1)
        compute(0)
        for i in range(n_steps):
            if i + 2 < n_steps:
                enqueue_h2d(i + 2)
            if i + 1 < n_steps:
                compute(i + 1)
            collect(i)
        d2h_stream.synchronize()
        comp.synchronize()

    run(max(3, args.warmup))
    d2h_acc.clear()
    barrier()
    t0 = time.perf_counter()
    run(args.steps)
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    e2e_ms = max_over_ranks(wall_ms) / args.steps
    return {"value": B * world / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(np.mean(d2h_acc)),
            "api": "HotPathGraph(targets='labels').replay(): loss fwd+bwd + detect + pack as one CUDA graph; pinned host "
                   "heads + packed labels copied in, losses + detection rows copied out, 3 pipeline slots, host wall clock"}


def run_torch_gpu_reference(args, dev, sample_images):
    """The reference's GPU-PyTorch path (north_star's comparison point): train.py's loss (:840-886, autograd
    backward) and predict()'s per-image decode/filter + torchvision's CUDA batched_nms (:1152-1238) on CUDA
    tensors — the unmodified reference functions when baseline/_ref is staged, else the oracle port.
    Reported only; not on the product path."""
    from oracle import ref_path as R
    import torchvision
    B, img, nc = args.batch, args.img, args.nc
    anchors = [a.to(dev) for a in R.default_anchors()]
    heads = [h.to(dev) for h in make_heads(B, img, nc, 1234)]
    labels = make_labels(np.random.default_rng(4321), B, nc)
    grids = [img // 8, img // 16, img // 32]
    tg = [R.assign_targets(l, R.default_anchors(), grids, nc, img) for l in labels]
    tgts = [torch.from_numpy(np.stack([t[s] for t in tg])).to(dev) for s in range(3)]
    ref = load_unmodified_reference()
    loss_fn = ref.yolo_loss_multiscale if ref is not None else R.multiscale_loss

    def loss_step():
        preds = [h.clone().requires_grad_(True) for h in heads]
        loss_fn(preds, tgts, anchors, nc)[0].backward()

    def det_step(n_img):
        kept = 0
        for b in range(n_img):  # predict() is single-image: a batch is a python loop (SURVEY 3c)
            bx, sc, cl = R.candidates([h[b:b + 1] for h in heads], anchors, img, nc, args.conf)
            if bx.shape[0]:
                kept += int(torchvision.ops.batched_nms(bx, sc, cl.to(dev), args.iou).numel())
        return kept

    def timed(fn, n):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return max(a.elapsed_time(b), (time.perf_counter() - t0) * 1e3) / n

    loss_ms = timed(loss_step, 5)                       # whole batch of B images
    det_ms = timed(lambda: det_step(sample_images), 3)  # sample_images images
    per_image_ms = loss_ms / B + det_ms / sample_images
    return {"value": 1e3 / per_image_ms, "unit": UNIT, "loss_fwd_bwd_ms": loss_ms,
            "decode_nms_ms_per_image": det_ms / sample_images,
            "kind": ("unmodified reference loss" if ref is not None else "port loss") + " + port of predict()'s body on CUDA tensors "
                    "(torch eager + torchvision CUDA nms)",
            "sample": f"loss on all {B} images, decode+NMS on {sample_images} of {B} images"}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_main(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    b200_main(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
