"""Writes tests/golden/live_reference.npz and tests/golden/reference_signatures.json: what three tests used to read
from a live import of the original yolo-from-scratch (train.py), stored so that they run from a clean checkout.

    python oracle/make_golden_pinned.py

Provenance.  The original is not part of this repository.  At commit 636ac80 (VERDICT.md of commit 265a9a6:
"The 69 CPU tests pass here, including `test_live_reference_agrees`") the three tests
(test_oracle_cpu.py::test_live_reference_agrees, test_host_cpu.py::test_install_on_live_reference and
::test_eval_epoch_signature_matches_reference) passed against the live original.  They asserted bit-for-bit
equality of the original's decode_predictions / yolo_loss with this oracle on the seeded input below, equal
parameter names and defaults of the four rebound functions, and equal signature strings of predict and eval_epoch.
oracle/ and yolo-from-scratch_b200/ are unchanged since then.  So the values written here, computed by the oracle
and read from the product, are the original's values on those inputs.
"""
import inspect
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)
from oracle import ref_path as R  # noqa: E402


def live_reference_vectors():
    """The input of test_live_reference_agrees, and the original's decode_predictions and yolo_loss on it."""
    anchors = R.default_anchors()[2]
    g = torch.Generator().manual_seed(77)
    x = torch.randn(2, 10, 10, 3, 8, generator=g)
    tg = torch.zeros_like(x)
    tg[0, 3, 4, 1, :5] = torch.tensor([0.4, 0.35, 0.2, 0.3, 1.0])
    tg[0, 3, 4, 1, 6] = 1.0
    tg[1, 9, 0, 2, :5] = torch.tensor([0.05, 0.95, 0.1, 0.1, 1.0])
    tg[1, 9, 0, 2, 5] = 1.0
    np.savez_compressed(os.path.join(OUT, "live_reference.npz"), x=x.numpy(), tgt=tg.numpy(), img=np.array(320),
                        decode=R.decode(x, anchors, 320).numpy(),
                        yolo_loss=np.array([float(v) for v in R.single_scale_loss(x, tg, anchors, 3)], dtype=np.float64))


def reference_signatures():
    """Parameter names and defaults (repr) of the functions install() rebinds, and the signature strings of
    predict and eval_epoch, as the original declares them."""
    import yolo_from_scratch_b200  # noqa: F401
    from yolo_from_scratch_b200 import install, ops
    out = {n: [[p.name, None if p.default is p.empty else repr(p.default)]
               for p in inspect.signature(getattr(ops, n)).parameters.values()] for n in install.PATCHED_FUNCTIONS}
    predict, _ = install._make_predict(None)
    out["predict"] = str(inspect.signature(predict))
    out["eval_epoch"] = str(inspect.signature(ops.eval_epoch))
    with open(os.path.join(OUT, "reference_signatures.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    live_reference_vectors()
    reference_signatures()
