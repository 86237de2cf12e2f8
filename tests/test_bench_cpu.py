"""bench.py's driver contract, as far as it can be checked without a GPU: the reference arm prints one JSON
line with the agreed keys, rank != 0 stays silent, and the B200 arm refuses to run without CUDA."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, env=e, timeout=600)


def test_reference_arm_json_contract():
    p = run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--batch", "2", "--img", "160"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_reference_arm_other_ranks_print_nothing():
    p = run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_b200_arm_fails_loudly_without_cuda():
    p = run(["--steps", "1", "--warmup", "1"])
    assert p.returncode != 0 and "no fallback" in p.stderr


def _fake_full(n_gpus=1):
    """A full result with every optional block present and realistically long strings/tables."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    args = bench.parse([])
    kern = {n: {"launches_per_step": 1.0, "avg_ms": 0.123456789, "ms_per_step": 0.123456789, "share": 0.123456789}
            for n in ("graph_edge_kernel", "graph_sort_kernel", "filter_emit_kernel", "graph_resolve_kernel", "loss_main_kernel",
                      "graph_gather_kernel", "loss_positive_kernel", "filter_count_kernel", "loss_finalize_kernel",
                      "filter_onepass_kernel", "nms_overflow_kernel", "pack_kernel")}
    hbm = {n: {"bound": "hbm", "achieved": 4559.123456, "peak": 6546.6, "unit": "GB/s", "frac": 0.696412345, "us": 25.4567,
               "algorithmic_bytes": 116121600.0, "share": 0.048, "traffic": 87200000, "peak_source": "MEASURED_PEAKS.json hbm_gbs"}
           for n in ("loss_main_kernel", "filter_count_kernel", "filter_emit_kernel", "filter_onepass_kernel",
                     "decode_fwd(3 scales)", "decode_bwd(3 scales)")}
    e2e = {"value": 43552.123456, "unit": "images/s", "ms_per_step": 1.4695123, "h2d_bytes_per_step": 77414400,
           "d2h_bytes_per_step": 14100000, "copy_ceiling": 45000.123, "copy_ceiling_gbs_per_rank": 52.7,
           "frac_of_copy_ceiling": 0.967, "api": "x" * 160}
    full = {
        "metric": bench.METRIC, "value": 126553.123456, "unit": "images/s", "n_gpus": n_gpus, "steps": 20, "warmup": 5,
        "ms_per_step": 0.50571234, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": bench.workload_config(args, n_gpus), "launch": "cuda-graph replay (HotPathGraph per input set, NCCL all-reduce captured inside)",
        "reps": 7, "ms_per_step_reps": [0.5] * 7, "ms_per_step_min_max": [0.501234, 0.512345], "timed_ms_total": 70.8,
        "eager": {"value": 110118.0, "ms_per_step": 0.581, "unit": "images/s"},
        "loss_fwd_bwd_ms": 0.0641234, "decode_nms_ms": 0.5141234, "e2e": e2e, "e2e_labels": dict(e2e), "e2e_graph": dict(e2e),
        "gpu_launches": 220, "kernels": kern, "hbm_kernels": hbm,
        "roofline": {"kernel": "graph_edge_kernel", "bound": "fp32-issue", "unit": "Gpair/s", "peak": 2189.70352, "peak_source": "y" * 150,
                     "what": "z" * 140, "achieved": 254.123, "frac": 0.116123, "algorithmic_speedup": 60.4123, "us": 331.0123,
                     "share": 0.62, "traffic": 23500000, "evaluated_pairs_per_launch": 84.1e6},
        "cpu_baseline": {"value": 19.8332, "unit": "images/s", "cores": 16, "kind": "reference", "sample": "s" * 400, "ms_per_step": 3200.0},
        "torch_gpu_baseline": {"value": 99.0123, "unit": "images/s", "loss_fwd_bwd_ms": 8.4123, "decode_nms_ms_per_image": 10.0123, "kind": "k" * 100},
        "clocks": {"sm_mhz": 1965.0, "sm_max_mhz": 1965, "reasons": ["sw_power_cap"], "samples": 40},
        "variants": {"conf_0.25": {"decode_nms_images_per_s": 66838.1}, "conf_0.001": {"decode_nms_images_per_s": 51909.2}},
        "other_configs": {k: {"value": 82559.123} for k in list(bench.OTHER_CONFIGS) + list(bench.SHARDED_CONFIGS)},
        "dist_parity": {"max_rel_err": 1.2e-7, "grad_max_rel_err": 0.0, "ok": True, "case": "c" * 90}, "numa": "gpu-local cpus (56 of 224)",
    }
    return bench, full


@pytest.mark.parametrize("n_gpus", [1, 8])
def test_compact_line_fits_the_drivers_parse_window(n_gpus):
    """BENCH_r01: the driver could not parse a 21 KB line.  The one printed line must stay under 4 KB with
    every optional block present, keep the contract keys, and carry roofline (frac <= ~1), cpu_baseline, e2e."""
    bench, full = _fake_full(n_gpus)
    line = bench.compact_line(full)
    text = json.dumps(line, separators=(",", ":"))
    assert len(text) < bench.MAX_LINE_BYTES, len(text)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks",
              "hbm_kernels"):
        assert k in line, k
    assert line["value"] > 0 and line["n_gpus"] == n_gpus
    r = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] <= 1.4
    assert "algorithmic_speedup" in r          # the culling factor is NOT folded into frac
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"]) and line["e2e"]["h2d_bytes_per_step"] > 0
    assert "workload" in line["config"] and "model" not in line["config"]
    for name, (us, frac) in line["hbm_kernels"].items():
        assert us > 0 and 0 < frac < 1.4
    json.loads(text)


def test_reference_arm_honours_steps_and_warmup():
    p = run(["--impl", "reference", "--steps", "3", "--warmup", "2", "--batch", "2", "--img", "160", "--cpu-sample", "-1"])
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])
    assert d["steps"] == 3 and d["warmup"] == 2
    assert "2 of 2 images" in d["cpu_baseline"]["sample"]     # every image of the batch, not a subset
    ref_staged = os.path.exists(os.path.join(ROOT, "baseline", "_ref", "train.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_staged else "port")


def test_dump_outputs_are_float_arrays_within_the_budget(tmp_path, monkeypatch):
    """--dump-outputs: one float32/float64 .npy per output; small arrays whole, the detections cut at offsets[B]; over
    the budget, gradients and detections are sampled at seeded positions that depend on their own shapes only, so
    a different detection count leaves the gradient files unchanged, and the positions and shapes are stored."""
    import numpy as np
    bench, _ = _fake_full()
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 1 << 20)
    monkeypatch.setattr(bench, "DUMP_DETECTIONS_BYTES", 1 << 12)
    monkeypatch.setattr(bench, "DUMP_SMALL_BYTES", 1 << 14)
    g = torch.Generator().manual_seed(0)
    grads = [torch.randn(2, G, G, 3, 85, generator=g) for G in (32, 16, 8)]
    rows = torch.randn(2 * 500, 6, generator=g)
    det = {"counts": torch.tensor([600, 700], dtype=torch.int32)}
    for out, last in (("a", 900), ("b", 900), ("c", 901)):
        offsets = torch.tensor([0, 400, last], dtype=torch.int32)
        bench.dump_outputs(str(tmp_path / out), torch.arange(4.0), grads, det, rows, offsets)
    load = lambda d, n: np.load(str(tmp_path / d / n))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(["candidates.npy", "detection_offsets.npy", "losses.npy"] +
                           [f"{k}{x}.npy" for k in ("detections", "grad_s0", "grad_s1", "grad_s2")
                            for x in ("", "_index", "_shape")])
    assert sum(load("a", n).nbytes for n in names) <= 1 << 20
    for n in names:
        assert load("a", n).dtype in (np.float32, np.float64) and np.array_equal(load("a", n), load("b", n)), n
        if n.startswith("grad_s"):
            assert np.array_equal(load("a", n), load("c", n)), n     # independent of the detection count
    for s, gr in enumerate(grads):
        idx, v = load("a", f"grad_s{s}_index.npy").astype(np.int64), load("a", f"grad_s{s}.npy")
        assert 0 < v.size < gr.numel() and load("a", f"grad_s{s}_shape.npy").tolist() == list(gr.shape)
        assert np.array_equal(v, gr.numpy().reshape(-1)[idx])
    idx = load("a", "detections_index.npy").astype(np.int64)
    assert load("a", "detections_shape.npy").tolist() == [900, 6] and idx.max() < 900
    assert np.array_equal(load("a", "detections.npy"), rows[:900].numpy()[idx])
    assert np.array_equal(load("a", "detection_offsets.npy"), [0, 400, 900]) and load("a", "losses.npy").shape == (4,)
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 64 << 20)
    monkeypatch.setattr(bench, "DUMP_DETECTIONS_BYTES", 16 << 20)
    bench.dump_outputs(str(tmp_path / "whole"), torch.arange(4.0), grads, det, rows, offsets)
    assert np.array_equal(load("whole", "grad_s0.npy"), grads[0].numpy()) and not os.path.exists(tmp_path / "whole" / "grad_s0_index.npy")
    assert np.array_equal(load("whole", "detections.npy"), rows[:901].numpy())
