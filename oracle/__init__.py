"""ORACLE — test infrastructure only.

A CPU restatement of the reference's per-box hot path (reference `train.py`, cited per function
in `ref_path.py`) plus a C restatement of torchvision's NMS arithmetic (`nms_ref.c`).
Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s baseline legs (cpu_baseline, the
torch_gpu_baseline comparison point, `--impl reference`) may import this package; the product
(`yolo-from-scratch_b200/`) and bench.py's own arm never do.

Pinning: `oracle/make_golden.py` imported the real reference from /root/reference and the
installed torchvision 0.26.0 in the build container and wrote `tests/golden/*.npz` (decode, CIoU,
losses + gradients, target assignment, predict() detections, eval_epoch() metrics, NMS keep sets);
`tests/test_oracle_cpu.py` checks this restatement against those vectors, against the reference's
own known-answer tests (tests/test_inference.py:16-76, tests/test_utils.py:82-90), and against the
original's outputs and signatures stored by `oracle/make_golden_pinned.py`.
"""
from .ref_path import *  # noqa: F401,F403
