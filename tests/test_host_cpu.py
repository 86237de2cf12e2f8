"""CPU-only tests of the host side: the C-ABI library loads and exports every symbol the header
declares, the ctypes structs match the C layout, the installer rebinds the reference's names,
the launcher extracts the CLI block, and the product fails loudly without CUDA (no fallback)."""
import ctypes
import os
import re
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def yb():
    import __graft_entry__ as g
    g.build()
    import yolo_from_scratch_b200 as m
    return m


def header_functions():
    text = open(os.path.join(ROOT, "include", "yolo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(yb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_header_symbol(yb):
    names = header_functions()
    assert len(names) >= 20
    lib = ctypes.CDLL(yb._lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/yolo_b200.h but not exported"
    # and the binding table covers the header one to one
    assert sorted(yb._lib.SIGNATURES) == names
    assert yb._lib.lib().yb_version() >= 100


def test_struct_layout_matches_c(yb, tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "yolo_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
                   'sizeof(yb_loss_desc), offsetof(yb_loss_desc, pred), offsetof(yb_loss_desc, grad),'
                   'sizeof(yb_heads_desc), offsetof(yb_heads_desc, pred));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    L, H = yb._lib.LossDesc, yb._lib.HeadsDesc
    assert out == [ctypes.sizeof(L), L.pred.offset, L.grad.offset, ctypes.sizeof(H), H.pred.offset]


def test_workspace_queries_do_not_need_a_gpu(yb):
    lib = yb._lib.lib()
    assert lib.yb_nms_workspace_bytes(64, 25200) >= lib.yb_nms_graph_workspace_bytes(64, 25200, 16)
    assert lib.yb_nms_graph_workspace_bytes(64, 25200, 16) > lib.yb_nms_min_workspace_bytes(64, 25200)
    d = yb._lib.LossDesc()
    d.S, d.B, d.A, d.nc = 3, 64, 3, 1
    for s, g in enumerate((80, 40, 20)):
        d.H[s] = d.W[s] = g
    assert lib.yb_loss_workspace_bytes(ctypes.byref(d)) >= 64 * 25200 * 4
    assert lib.yb_ciou_scratch_bytes(10) >= 8


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback(yb):
    x = torch.zeros(1, 4, 4, 3, 6)
    a = torch.tensor([[10., 13.], [16., 30.], [33., 23.]])
    for call in (lambda: yb.decode_predictions(x, a), lambda: yb.yolo_loss(x, x, a, 1),
                 lambda: yb.batched_nms(torch.zeros(2, 4), torch.zeros(2), torch.zeros(2, dtype=torch.long), 0.5),
                 lambda: yb.build_targets([[[0, .5, .5, .1, .1]]], [a, a, a], [8, 4, 2], 1, 64)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()


def test_bad_arguments_are_reported(yb):
    lib = yb._lib.lib()
    rc = lib.yb_decode_fwd(None, None, None, 1, 4, 4, 3, 1, 640.0, None)
    assert rc != 0 and b"null" in lib.yb_last_error()
    rc = lib.yb_batched_nms(None, None, None, None, 1, 8, 0.5, 100000, 7, None, None, None, 0, None)
    assert rc != 0


def test_new_entry_points_validate_arguments(yb):
    """yb_loss_partials_sparse / yb_eval_counts / layout field: bad arguments come back as error codes
    with a message, before anything touches the GPU."""
    lib = yb._lib.lib()
    d = yb._lib.LossDesc()
    d.S, d.B, d.B_global, d.A, d.nc = 3, 2, 2, 3, 1
    for s, g in enumerate((8, 4, 2)):
        d.H[s] = d.W[s] = g
    assert lib.yb_loss_sparse_workspace_bytes(ctypes.byref(d), 10) > lib.yb_loss_workspace_bytes(ctypes.byref(d))
    assert lib.yb_loss_partials_sparse(ctypes.byref(d), None, None, None, None, 10, 64, None, None, None, 0, None) != 0
    d.layout = 7
    assert lib.yb_loss_partials(ctypes.byref(d), None, None, 0, None) != 0 and b"layout" in lib.yb_last_error()
    h = yb._lib.HeadsDesc()
    h.S, h.B, h.A, h.nc, h.layout = 3, 1, 3, 1, 1
    assert lib.yb_eval_counts(ctypes.byref(h), None, 0.5, 0.5, None, None) != 0


HEAD_CHECK_SCRIPT = r'''
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
import torch
import yolo_from_scratch_b200 as yb
assert torch.cuda.device_count() == 0, "the calls below pass stand-in device addresses"
L = yb._lib
lib = L.lib()
P = 1 << 20                                   # a 16-byte aligned stand-in address; no device is visible
CASES = {
    "valid": {}, "S=0": {"S": 0}, "S=5": {"S": 5}, "A=0": {"A": 0}, "A=9": {"A": 9}, "H=0": {"H": 0},
    "layout=7": {"layout": 7}, "dtype=7": {"dtype": 7}, "layout=7,B=0": {"layout": 7, "B": 0},
    "dtype=7,B=0": {"dtype": 7, "B": 0}, "2^32 elements": {"H": 1 << 14, "W": 1 << 14},
    "null pred": {"pred": 0}, "misaligned pred": {"pred": P + 4},
}
DECODE_ONLY_S1 = ("S=0", "S=5", "layout=7", "layout=7,B=0")   # decode takes one scale and no layout

def desc(cls, case, dtype):
    d = cls()
    d.S, d.B, d.A, d.nc, d.img_size, d.layout, d.dtype = 3, 2, 3, 2, 64.0, 0, dtype
    for s, g in enumerate((8, 4, 2)):
        d.H[s] = d.W[s] = g
        d.pred[s], d.anchors[s] = P * (s + 1), P * (s + 5)
    if cls is L.LossDesc:
        d.B_global = 2
        for s in range(3):
            d.tgt[s], d.grad[s] = P * (s + 9), P * (s + 13)
    for k, v in CASES[case].items():
        if k in ("H", "W"):
            getattr(d, k)[0] = v
        elif k == "pred":
            d.pred[0] = v
        else:
            setattr(d, k, v)
    return d

def decode(bwd):
    def call(case):
        d = desc(L.HeadsDesc, case, 0)
        args = (d.pred[0], d.anchors[0]) + ((P,) if bwd else ()) + (P, d.B, d.H[0], d.W[0], d.A, d.nc, 64.0, d.dtype, None)
        return (lib.yb_decode_bwd_t if bwd else lib.yb_decode_fwd_t)(*args)
    return call

big = 1 << 40
ENTRIES = {
    "decode_fwd": ("decode", decode(False)),
    "decode_bwd": ("decode", decode(True)),
    "loss_partials": ("loss", lambda c: lib.yb_loss_partials(ctypes.byref(desc(L.LossDesc, c, 0)), P, P, big, None)),
    "loss_partials_sparse": ("loss(sparse)", lambda c: lib.yb_loss_partials_sparse(
        ctypes.byref(desc(L.LossDesc, c, 0)), P, P, P, P, 4, 64, P, P, P, big, None)),
    "loss_grad_emit": ("loss_grad_emit", lambda c: lib.yb_loss_grad_emit(
        ctypes.byref(desc(L.LossDesc, c, 1)), P, P, -1, P, big, None)),
    "filter_compact": ("filter", lambda c: lib.yb_filter_compact(
        ctypes.byref(desc(L.HeadsDesc, c, 0)), 0.5, None, P, P, P, P, 100, P, big, None)),
    "filter_multilabel": ("filter_multilabel", lambda c: lib.yb_filter_multilabel(
        ctypes.byref(desc(L.HeadsDesc, c, 0)), 0.5, None, 100, P, P, P, P, None, 1 << 20, P, big, None)),
    "eval_counts": ("eval_counts", lambda c: lib.yb_eval_counts(
        ctypes.byref(desc(L.HeadsDesc, c, 0)), (ctypes.c_void_p * 4)(P, P, P, P), 0.5, 0.5, P, None)),
}
out = []
for name, (who, call) in ENTRIES.items():
    for case in CASES:
        if name.startswith("decode") and case in DECODE_ONLY_S1:
            continue
        rc = call(case)
        out.append([name, who, case, rc, lib.yb_last_error().decode() if rc else ""])
print(json.dumps(out))
'''


def test_every_head_entry_point_rejects_the_same_malformed_descriptors(yb):
    """Every entry point that reads head tensors checks its descriptor the same way: a table of malformed
    descriptors comes back as YB_EINVAL with a message that names the entry point, at B = 0 too.  The calls run
    in a process that sees no GPU, so that a missing check fails at the first CUDA call instead of launching; the
    well-formed descriptor gets past the checks and fails there with a CUDA error."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", HEAD_CHECK_SCRIPT, ROOT], env=env, capture_output=True, text=True,
                         timeout=300)
    assert res.returncode == 0, res.stderr
    rows = __import__("json").loads(res.stdout.strip().splitlines()[-1])
    assert len({r[0] for r in rows}) == 8 and len(rows) == 8 * 13 - 2 * 4
    for name, who, case, rc, msg in rows:
        if case == "valid":
            assert rc > 0, (name, rc, msg)   # past the argument checks: a CUDA error, not YB_EINVAL
        else:
            assert rc == -1 and msg.startswith(who + ":"), (name, case, rc, msg)


def fake_train_module():
    """A stand-in with the reference's hot-path names; internal callers resolve them through the
    module globals exactly like train.py does."""
    m = types.ModuleType("train")
    src = '''
class YOLODataset:
    def compute_anchor_iou(self, box_wh, anchors): return "ref"
    def __getitem__(self, idx): return "ref"
def decode_predictions(raw_preds, anchors, img_size=640): return "ref"
def ciou_loss(p, t, eps=1e-7): return "ref"
def yolo_loss(predictions, targets, anchors, num_classes=1): return decode_predictions(predictions, anchors)
def yolo_loss_multiscale(predictions, targets, anchors_list, num_classes=1): return "ref"
def train_epoch(): return yolo_loss_multiscale
def predict():
    from torchvision.ops import batched_nms
    return batched_nms
if __name__ == "__main__":
    RESULT = ("cli ran", decode_predictions.__module__)
'''
    exec(compile(src, "train.py", "exec"), m.__dict__)
    return m, src


def test_install_rebinds_reference_names(yb):
    from yolo_from_scratch_b200 import install as inst, ops
    import torchvision
    tv_nms = torchvision.ops.batched_nms
    m, _ = fake_train_module()
    orig_getitem, orig_predict = m.YOLODataset.__getitem__, m.predict
    inst.install(m)
    try:
        assert m.decode_predictions is ops.decode_predictions and m.ciou_loss is ops.ciou_loss
        assert m.yolo_loss is ops.yolo_loss and m.train_epoch() is ops.yolo_loss_multiscale
        # predict is rebound as a whole (f-3) with the reference's signature, plus a batched variant;
        # torchvision is NOT patched process-wide any more
        import inspect
        assert m.predict is not orig_predict and callable(m.predict_batch)
        assert list(inspect.signature(m.predict).parameters) == ["model", "image_path", "device", "num_classes",
                                                                 "conf_threshold", "iou_threshold"]
        assert torchvision.ops.batched_nms is tv_nms
        assert m.YOLODataset.__getitem__ is not orig_getitem
        inst.install(m)  # idempotent
    finally:
        inst.uninstall(m)
    assert m.predict is orig_predict and not hasattr(m, "predict_batch")
    assert m.decode_predictions(None, None) == "ref" and m.YOLODataset.__getitem__ is orig_getitem
    # the round-1 behaviour is still available: the reference's own predict with torchvision's name rebound
    m2, _ = fake_train_module()
    inst.install(m2, patch_torchvision=True, patch_predict=False)
    try:
        assert m2.predict() is ops.batched_nms
    finally:
        inst.uninstall(m2)
    assert m2.predict() is tv_nms and torchvision.ops.batched_nms is tv_nms


def test_import_hook_and_launcher(yb, tmp_path):
    from yolo_from_scratch_b200 import install as inst, ops, run
    _, src = fake_train_module()
    (tmp_path / "train.py").write_text(src)
    sys.modules.pop("train", None)
    old_path = list(sys.path)
    try:
        run.main([str(tmp_path / "train.py"), "data.yaml"])
        mod = sys.modules["train"]
        assert mod.decode_predictions is ops.decode_predictions      # patched at import
        assert mod.RESULT == ("cli ran", ops.__name__)                # __main__ block ran in the patched namespace
        assert sys.argv[1:] == ["data.yaml"]
    finally:
        inst.uninstall(sys.modules.get("train"))
        inst.disable_import_hook()
        sys.modules.pop("train", None)
        sys.path[:] = old_path


def reference_signatures():
    """The original's signatures of the rebound functions (tests/golden/reference_signatures.json,
    oracle/make_golden_pinned.py)."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_signatures.json")) as f:
        return json.load(f)


def signature_stand_in():
    """A module with the original's hot-path names, each declared with the original's parameters and defaults."""
    sigs = reference_signatures()
    src = ["class YOLODataset:\n    def compute_anchor_iou(self, box_wh, anchors): return 'ref'\n"
           "    def __getitem__(self, idx): return 'ref'"]
    for name, params in sigs.items():
        if isinstance(params, list):
            args = ", ".join(n if d is None else f"{n}={d}" for n, d in params)
            src.append(f"def {name}({args}): return 'ref'")
        else:
            src.append(f"def {name}{params}: return 'ref'")
    m = types.ModuleType("train")
    exec(compile("\n".join(src) + "\n", "train.py", "exec"), m.__dict__)
    return m


def test_install_on_live_reference(yb):
    """A module declared like the original gets every hot-path name rebound, with the original's parameter names,
    defaults and predict signature."""
    from yolo_from_scratch_b200 import install as inst, ops
    ref = signature_stand_in()
    assert inst.looks_like_reference(ref)
    inst.install(ref)
    try:
        for n in inst.PATCHED_FUNCTIONS:
            assert getattr(ref, n) is getattr(ops, n)
        import inspect
        for n in inst.PATCHED_FUNCTIONS:  # same parameter names and defaults as the reference
            a = inspect.signature(ref.__yolo_b200_saved__[n])
            b = inspect.signature(getattr(ops, n))
            assert list(a.parameters) == list(b.parameters), n
            assert [p.default for p in a.parameters.values()] == [p.default for p in b.parameters.values()], n
        a, b = inspect.signature(ref.__yolo_b200_saved__["predict"]), inspect.signature(ref.predict)   # f-3
        assert str(a) == str(b) and ref.predict is not ref.__yolo_b200_saved__["predict"]
    finally:
        inst.uninstall(ref)


def test_channels_last_option_removes_the_head_permute_copy(yb):
    """f-2 in the drop-in flow: install(..., channels_last=True) makes every model built afterwards run NHWC, so the
    reference's view/permute/contiguous of a head conv's output (train.py:608-609) returns an alias of the conv's
    output; uninstall restores the constructor.  Host logic only (a stand-in model with the reference's head code)."""
    import torch
    from yolo_from_scratch_b200 import install as inst
    m, _ = fake_train_module()

    class YOLO(torch.nn.Module):
        def __init__(self, nc=2):
            super().__init__()
            self.nc = nc
            self.body = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3, padding=1), torch.nn.BatchNorm2d(8), torch.nn.SiLU())
            self.head = torch.nn.Conv2d(8, 3 * (5 + nc), 1)

        def forward(self, x):
            self.raw = self.head(self.body(x))
            b, _, h, w = self.raw.shape
            return self.raw.view(b, 3, 5 + self.nc, h, w).permute(0, 3, 4, 1, 2).contiguous()
    m.YOLO = YOLO
    orig_init = YOLO.__init__
    x = torch.randn(2, 3, 16, 16)
    torch.manual_seed(0)
    plain = YOLO()
    out_plain = plain(x)
    assert out_plain.data_ptr() != plain.raw.data_ptr()          # the reference pays a copy here
    inst.install(m, channels_last=True)
    try:
        model = m.YOLO()
        model.load_state_dict(plain.state_dict())
        out = model(x)
        assert out.is_contiguous() and out.shape == (2, 16, 16, 3, 7)
        assert out.data_ptr() == model.raw.data_ptr()             # alias of the conv output: no copy
        assert torch.allclose(out, out_plain, atol=1e-5)
        out.sum().backward()
        assert model.head.weight.grad is not None
        assert inst.channels_last_heads(model) is model           # idempotent
    finally:
        inst.uninstall(m)
    assert YOLO.__init__ is orig_init


def test_eval_epoch_is_rebound_and_restored(yb):
    from yolo_from_scratch_b200 import install as inst, ops
    m, _ = fake_train_module()
    m.eval_epoch = lambda model, loader, device, num_classes=1, iou_threshold=0.5, conf_threshold=0.5: "ref"
    orig = m.eval_epoch
    inst.install(m)
    try:
        assert m.eval_epoch is ops.eval_epoch
    finally:
        inst.uninstall(m)
    assert m.eval_epoch is orig
    m2, _ = fake_train_module()
    m2.eval_epoch = orig
    inst.install(m2, patch_eval=False)
    try:
        assert m2.eval_epoch is orig
    finally:
        inst.uninstall(m2)


def test_eval_epoch_signature_matches_reference(yb):
    import inspect
    from yolo_from_scratch_b200 import ops
    assert str(inspect.signature(ops.eval_epoch)) == reference_signatures()["eval_epoch"]


def test_label_packing_and_layout_helpers_on_cpu(yb):
    """Host-side helpers of the f-2 / f-4 entry points need no GPU."""
    from yolo_from_scratch_b200 import ops
    labels = [np.array([[1, .5, .5, .2, .3], [0, .1, .2, .05, .05]]), np.zeros((0, 5)), np.array([[2, .9, .9, .1, .1]])]
    lab, n_gt, lb = ops.pack_labels_host(labels, 320)
    assert lab.shape == (3, 2, 5) and lab.dtype == torch.float64 and n_gt.tolist() == [2, 0, 1]
    assert lb.tolist() == [[320.0, 320.0, 1.0, 0.0, 0.0]] * 3
    assert float(lab[2, 0, 1]) == 0.9 and float(lab[1].abs().sum()) == 0.0
    lab, n_gt, lb = ops.pack_labels_host(labels, 320, letterbox=[(500, 375, 0.64, 40, 0)] * 3, max_gt=7)
    assert lab.shape == (3, 7, 5) and lb[0].tolist() == [500.0, 375.0, 0.64, 40.0, 0.0]
    with pytest.raises(ValueError):
        ops.pack_labels_host(labels, 320, max_gt=1)
    assert ops.pack_labels_host([], 320)[0].shape == (0, 1, 5)
    # heads_from_nchw is exactly the reference's reshape (train.py:608-609)
    B, A, nc, G = 2, 3, 4, 5
    raw = torch.arange(B * A * (5 + nc) * G * G, dtype=torch.float32).reshape(B, A * (5 + nc), G, G)
    want = raw.view(B, A, 5 + nc, G, G).permute(0, 3, 4, 1, 2).contiguous()
    got = ops.heads_from_nchw(raw, A)
    assert got.shape == (B, G, G, A, 5 + nc) and got.is_contiguous() and torch.equal(got, want)
    assert float(got[1, 2, 3, 1, 4]) == float(raw[1, 1 * (5 + nc) + 4, 2, 3])


def test_desc_layout_field_defaults_to_reference_layout(yb):
    L, H = yb._lib.LossDesc(), yb._lib.HeadsDesc()
    assert L.layout == yb._lib.LAYOUT_BHWAC == 0 and H.layout == 0 and yb._lib.LAYOUT_NCHW == 1
