"""Native bf16 / fp16 heads against fp32 heads and against today's conversion path (heads.float() passed in).

Workload: configs[1] (nc=1, conf 0.5) and configs[2] (nc=80, conf 0.001) shapes, B=64, 640x640, three scales,
reference layout and NCHW, dense targets from bench.py's label generator; the heads are randn with the objectness
logit at 2*randn - 4.6 (SURVEY 8d "prior" heads).  The heads are 70 MB (nc=1, fp32) and 548 MB (nc=80, fp32): the
nc=80 working set is larger than the 126 MB L2, the nc=1 one is not, and every timed pass reads it again.

Reports, per (config, layout, dtype):
  - per-kernel device times from the library's own launch events (yb_timing_enable), with a byte model per kernel
    at the element size and its fraction of the copy peak bench.py uses;
  - user-visible calls timed with CUDA events (median): loss forward+backward at s = 1 and s = 65536, decode
    forward+backward, detect_batch — native against the conversion path;
  - peak memory of the loss forward+backward, native against the conversion path;
  - HotPathGraph replay, fp32 against bf16 (reference layout);
  - `equal`: outputs of the native and the conversion path compared bit for bit at the timed sizes.
Prints one JSON line with the device name and power limit.

  python tools/bench_half.py [--iters 20]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import make_labels   # noqa: E402
from oracle import ref_path as R   # noqa: E402
import yolo_from_scratch_b200 as yb   # noqa: E402
from yolo_from_scratch_b200 import ops   # noqa: E402

DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
CONFIGS = {"configs1": (1, 0.5), "configs2": (80, 0.001)}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def copy_peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback 6650 GB/s (as bench.py)"


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def kernel_times(fn, iters):
    lib = yb._lib.lib()
    fn()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.yb_timing_collect(buf, len(buf))   # drop the warm-up
    lib.yb_timing_enable(1)
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    lib.yb_timing_collect(buf, len(buf))
    lib.yb_timing_enable(0)
    out = {}
    for line in buf.value.decode().splitlines():
        name, count, total = line.split()
        out[name] = float(total) / iters * 1e3   # us per call of fn
    return out


def byte_model(nc, layout, es, rows, cand):
    """Bytes each kernel must move (one call): T = heads at element size es, fp32 dense targets read one 32-byte
    sector per row for their objectness, positive rows are few and left out."""
    row_b = (5 + nc) * es
    T = rows * row_b
    obj_read = rows * es if layout == "nchw" else rows * min(row_b, 32)
    m = {"decode_fwd_kernel": 2 * T, "decode_bwd_kernel": 3 * T,
         "filter": T + 28 * cand}
    if es == 4:
        m["loss_main"] = obj_read + 32 * rows + T        # + the dense gradient write
    else:
        m["loss_main"] = obj_read + 32 * rows + 4 * rows  # + the compact objectness gradient
        m["loss_grad_emit_kernel"] = T + 4 * rows
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--img", type=int, default=640)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_half.py needs a CUDA device")
    dev = torch.device("cuda")
    B, img, it = args.batch, args.img, args.iters
    anchors = [a.to(dev) for a in R.default_anchors()]
    grids = [img // 8, img // 16, img // 32]
    peak, peak_src = copy_peak_gbs()
    result = {"device": torch.cuda.get_device_name(), "power_limit": power_limit(), "batch": B, "img": img,
              "iters": it, "copy_peak_gbs": peak, "copy_peak_source": peak_src, "runs": {}}
    all_equal = True
    for cname, (nc, conf) in CONFIGS.items():
        g = torch.Generator(device=dev).manual_seed(0)
        base = [torch.randn(B, G, G, 3, 5 + nc, generator=g, device=dev) for G in grids]
        for h in base:
            h[..., 4].mul_(2.0).sub_(4.6)
        labels = make_labels(np.random.default_rng(0), B, nc)
        tg = yb.build_targets(labels, anchors, grids, nc, img)
        rows = sum(h.numel() // (5 + nc) for h in base)
        for layout in ("bhwac", "nchw"):
            lay = ops.LAYOUT_NCHW if layout == "nchw" else ops.LAYOUT_BHWAC
            for dname, dt in DT.items():
                heads = [h.to(dt) for h in base]
                if layout == "nchw":
                    heads = [h.permute(0, 3, 4, 1, 2).reshape(h.shape[0], -1, h.shape[1], h.shape[2]).contiguous()
                             for h in heads]
                lossf = ops.yolo_loss_multiscale_nchw if layout == "nchw" else ops.yolo_loss_multiscale
                leaves = [h.clone().requires_grad_(True) for h in heads]

                def loss_step(s, upcast=False):
                    for p in leaves:
                        p.grad = None
                    x = [p.float() for p in leaves] if upcast else leaves
                    out = lossf(x, tg, anchors, nc)
                    (out[0] * s).backward()
                    return out

                def detect(upcast=False):
                    return ops.detect_batch([h.float() for h in heads] if upcast else heads, anchors, img, nc, conf,
                                            0.4, layout=lay)

                def decode(upcast=False):
                    x = (heads[0].float() if upcast else heads[0].detach()).requires_grad_(True)
                    out = ops.decode_predictions(x, anchors[0], img)
                    out.backward(out.detach())

                r = {}
                r["kernels_loss_us"] = kernel_times(lambda: loss_step(65536.0), it)
                r["kernels_filter_us"] = kernel_times(lambda: ops.filter_candidates(heads, anchors, img, nc, conf,
                                                                                    layout=lay), it)
                if layout == "bhwac":
                    r["kernels_decode_p3_us"] = kernel_times(decode, it)
                cand = int(ops.filter_candidates(heads, anchors, img, nc, conf, layout=lay)[3].sum())
                model = byte_model(nc, layout, heads[0].element_size(), rows, cand)
                model["decode_fwd_kernel"] = model["decode_fwd_kernel"] * grids[0] ** 2 * 3 * B // rows
                model["decode_bwd_kernel"] = model["decode_bwd_kernel"] * grids[0] ** 2 * 3 * B // rows
                times = dict(r["kernels_loss_us"])
                times["loss_main"] = times.get("loss_main_kernel", 0.0) + times.get("loss_main_nchw_kernel", 0.0)
                times["filter"] = sum(r["kernels_filter_us"].values())
                times.update(r.get("kernels_decode_p3_us", {}))
                r["byte_model"] = {k: {"bytes": b, "us": times.get(k), "frac_of_copy_peak":
                                       (b / (times[k] * 1e-6) / 1e9 / peak) if times.get(k) else None}
                                   for k, b in model.items()}
                r["loss_fwd_bwd_ms"] = {f"s={s:g}": timed(lambda: loss_step(s), it) for s in (1.0, 65536.0)}
                r["detect_batch_ms"] = timed(detect, it)
                if layout == "bhwac":
                    r["decode_p3_fwd_bwd_ms"] = timed(decode, it)
                if dt != torch.float32:
                    r["conversion_path"] = {
                        "loss_fwd_bwd_ms": {f"s={s:g}": timed(lambda: loss_step(s, True), it) for s in (1.0, 65536.0)},
                        "detect_batch_ms": timed(lambda: detect(True), it)}
                    if layout == "bhwac":
                        r["conversion_path"]["decode_p3_fwd_bwd_ms"] = timed(lambda: decode(True), it)
                    peaks = []
                    for upcast in (False, True):
                        torch.cuda.synchronize()
                        torch.cuda.reset_peak_memory_stats()
                        m0 = torch.cuda.memory_allocated()
                        loss_step(65536.0, upcast)
                        torch.cuda.synchronize()
                        peaks.append((torch.cuda.max_memory_allocated() - m0) / 2 ** 20)
                    r["loss_peak_extra_mib"] = {"native": peaks[0], "conversion": peaks[1]}
                    # equality at the timed sizes
                    eq = True
                    for s in (1.0, 65536.0):
                        o1 = loss_step(s)
                        g1 = [p.grad.clone() for p in leaves]
                        o2 = loss_step(s, True)
                        g2 = [p.grad for p in leaves]
                        eq &= torch.equal(torch.stack(o1), torch.stack(o2))
                        for a, b in zip(g1, g2):
                            same = (a.view(torch.int16) == b.view(torch.int16)) | (torch.isnan(a) & torch.isnan(b))
                            eq &= bool(same.all())
                    d1, d2 = detect(), detect(True)
                    eq &= torch.equal(d1["counts"], d2["counts"]) and torch.equal(d1["n_keep"], d2["n_keep"])
                    for i, k in enumerate(d1["n_keep"].tolist()):
                        eq &= torch.equal(d1["keep"][i, :k], d2["keep"][i, :k])
                    r["equal"] = bool(eq)
                    all_equal &= bool(eq)
                result["runs"][f"{cname}/{layout}/{dname}"] = r
                del leaves, heads
                torch.cuda.empty_cache()
        # HotPathGraph replay, fp32 against bf16 (reference layout, dense targets)
        for dname in ("f32", "bf16"):
            hp = ops.HotPathGraph(B, img, nc, anchors, conf_threshold=conf, targets="dense", dtype=DT[dname])
            for s in range(3):
                hp.heads[s].copy_(base[s])
                hp.targets[s].copy_(tg[s])
            result["runs"].setdefault(f"{cname}/graph", {})[f"replay_ms_{dname}"] = timed(hp.replay, it)
            del hp
            torch.cuda.empty_cache()
        del base, tg
        torch.cuda.empty_cache()
    result["equal"] = all_equal
    print(json.dumps(result))


if __name__ == "__main__":
    main()
