"""north_star: "train.py, eval.py and the existing pytest suite run unchanged with the new path swapped in".

These tests run the UNMODIFIED reference (a checkout of the original yolo-from-scratch, see conftest.REFERENCE_DIR)
through the drop-in boundary on a real GPU:
  * its own pytest suite (everything except tests/test_cli.py, which shells out to `python train.py` without the swap)
    under `-p yolo_from_scratch_b200.pytest_plugin`;
  * its CLI (`train.py data.yaml --epochs 1`, eval mode, inference mode) under `python -m yolo_from_scratch_b200.run`;
  * the unchanged model in NHWC through the swap.
They execute the original's own code, which is not part of this repository and cannot be stored as data, so they
skip from a clean checkout.  `predict` through the rebinding is checked without the original,
against the golden detections the reference itself produced (tests/golden/predict.npz).
Logs go to $YOLO_B200_TEST_LOGS when it is set.
"""
import os
import re
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from conftest import REFERENCE_DIR as REF

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOGDIR = os.environ.get("YOLO_B200_TEST_LOGS", "")


def _need_ref():
    if not os.path.exists(os.path.join(REF, "train.py")):
        pytest.skip("runs the original yolo-from-scratch's own code, which is not part of this repository "
                    "(YOLO_FROM_SCRATCH_REFERENCE names a checkout of it)")


def _env():
    e = dict(os.environ)
    e["PYTHONPATH"] = ROOT + os.pathsep + e.get("PYTHONPATH", "")
    return e


def _log(name, text):
    if not LOGDIR:
        return
    try:
        os.makedirs(LOGDIR, exist_ok=True)
        with open(os.path.join(LOGDIR, name), "w") as f:
            f.write(text)
    except OSError:
        pass


def test_reference_suite_runs_unchanged_through_the_swap():
    """116 non-CLI tests of the reference, every hot-path call landing in libyolo_b200.so."""
    _need_ref()
    cmd = [sys.executable, "-m", "pytest", "-p", "yolo_from_scratch_b200.pytest_plugin", os.path.join(REF, "tests"),
           f"--ignore={os.path.join(REF, 'tests', 'test_cli.py')}", "-q", "-p", "no:cacheprovider", "-n", "4",
           "--timeout", "900"]
    p = subprocess.run(cmd, capture_output=True, text=True, env=_env(), cwd=REF, timeout=3000)
    _log("reference_suite_through_swap.log", "$ " + " ".join(cmd) + "\n" + p.stdout[-20000:] + "\n--- stderr ---\n" + p.stderr[-5000:])
    assert p.returncode == 0, p.stdout[-6000:] + p.stderr[-2000:]
    m = re.search(r"(\d+) passed", p.stdout)
    assert m and int(m.group(1)) >= 116, p.stdout[-2000:]
    assert "failed" not in p.stdout.splitlines()[-1]


def test_the_swap_really_is_active_inside_the_reference_suite(tmp_path):
    """Same plugin, one reference test module, plus a conftest-level check that `train`'s names are the B200 ones
    and that the library's launch counter moved."""
    _need_ref()
    check = tmp_path / "test_swap_active.py"
    check.write_text(
        "import sys\n"
        f"sys.path.insert(0, {REF!r})\n"
        "import train\n"
        "from yolo_from_scratch_b200 import ops, _lib\n"
        "import torch\n"
        "def test_active():\n"
        "    assert train.yolo_loss_multiscale is ops.yolo_loss_multiscale and train.decode_predictions is ops.decode_predictions\n"
        "    assert train.predict.__doc__.startswith('Drop-in') and train.eval_epoch is ops.eval_epoch\n"
        "    n0 = _lib.lib().yb_launch_count()\n"
        "    m = train.YOLO(num_classes=1, img_size=320)\n"
        "    preds = m(torch.randn(1, 3, 320, 320))\n"
        "    tg = [torch.zeros_like(p) for p in preds]\n"
        "    loss = train.yolo_loss_multiscale(preds, tg, m.anchors, 1)[0]\n"
        "    loss.backward()\n"
        "    assert _lib.lib().yb_launch_count() > n0 and any(p.grad is not None for p in m.parameters())\n")
    p = subprocess.run([sys.executable, "-m", "pytest", "-p", "yolo_from_scratch_b200.pytest_plugin", str(check), "-q",
                        "-p", "no:cacheprovider"], capture_output=True, text=True, env=_env(), cwd=str(tmp_path), timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]


def _make_dataset(root, n_train=5, n_val=2, seed=0):
    """A tiny YOLO-format dataset + YAML like the reference's own CLI fixture (tests/test_cli.py:18-60)."""
    import yaml
    from PIL import Image
    rng = np.random.default_rng(seed)
    out = {}
    for split, n in (("train", n_train), ("val", n_val)):
        imgs, labels = root / split / "images", root / split / "labels"
        imgs.mkdir(parents=True)
        labels.mkdir(parents=True)
        for i in range(n):
            Image.fromarray(rng.integers(0, 255, (480, 640, 3), dtype=np.uint8)).save(imgs / f"{split}{i}.jpg")
            with open(labels / f"{split}{i}.txt", "w") as f:
                for _ in range(int(rng.integers(1, 4))):
                    f.write(f"0 {rng.uniform(0.2, 0.8)} {rng.uniform(0.2, 0.8)} {rng.uniform(0.1, 0.3)} {rng.uniform(0.1, 0.3)}\n")
        out[split] = str(imgs)
    cfg = root / "dataset.yaml"
    with open(cfg, "w") as f:
        yaml.dump({"nc": 1, "names": ["object"], "train": out["train"], "val": out["val"]}, f)
    return str(cfg), out


def test_reference_cli_through_the_launcher(tmp_path):
    """train.py:1520-1522 (training loop), :1476-1477 (eval mode) and :1444 (inference mode) through
    `python -m yolo_from_scratch_b200.run train.py ...`, on the GPU, file on disk unchanged; the inference mode's
    printed detections are compared with the UNPATCHED reference run on the same checkpoint."""
    _need_ref()
    cfg, dirs = _make_dataset(tmp_path)
    train_py = os.path.join(REF, "train.py")
    run = [sys.executable, "-m", "yolo_from_scratch_b200.run", train_py]
    log = []

    def sh(cmd, timeout=1500):
        p = subprocess.run(cmd, capture_output=True, text=True, env=_env(), cwd=str(tmp_path), timeout=timeout)
        log.append("$ " + " ".join(cmd) + "\n" + p.stdout[-6000:] + "\n--- stderr ---\n" + p.stderr[-3000:])
        _log("reference_cli_through_swap.log", "\n\n".join(log))
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        return p.stdout

    out = sh(run + [cfg, "--epochs", "1", "--img-size", "320", "--size", "n"])
    assert "Training YOLO model" in out and "Epoch 1:" in out and "Training complete" in out and "Device: cuda" in out
    ckpts = sorted(f for f in os.listdir(tmp_path) if f.startswith("yolo_") and f.endswith(".pt"))
    assert len(ckpts) == 1
    ckpt = str(tmp_path / ckpts[0])
    out = sh(run + [cfg, ckpt, "--size", "n"])
    assert "Validation Set:" in out and "F1 Score:" in out
    img = os.path.join(dirs["val"], "val0.jpg")
    patched = sh(run + [img, ckpt, "--size", "n"])
    plain = sh([sys.executable, train_py, img, ckpt, "--size", "n"])
    take = lambda s: [ln for ln in s.splitlines() if "Box:" in ln or "No objects" in ln or "Detected" in ln]
    assert take(patched) == take(plain), (take(patched)[:5], take(plain)[:5])


class _PresetHeads:
    def __init__(self, heads, img_size, anchors):
        self.heads, self.img_size, self.anchors = heads, img_size, anchors

    def eval(self):
        return self

    def __call__(self, img):
        n = img.shape[0]
        return [h[:n] for h in self.heads]


def _canon(dets):
    a = np.array(dets, dtype=np.float64).reshape(-1, 6)
    return a[np.lexsort((a[:, 3], a[:, 2], a[:, 1], a[:, 0], -a[:, 4]))]


def _train_stand_in(scale, pad_top, pad_left):
    """A module with the names install() rebinds in the reference's `train`.  Its letterbox_resize returns the
    scale and padding the reference's own letterbox_resize gave for the golden image (oracle/make_golden.py:
    golden_predict stores them in <name>_cfg); everything predict() does after it is the B200 path."""
    from PIL import Image
    from yolo_from_scratch_b200.install import PATCHED_FUNCTIONS
    m = types.ModuleType("train")
    m.Image = Image
    m.letterbox_resize = lambda pil_img, img_size: (pil_img, scale, pad_top, pad_left)
    for n in PATCHED_FUNCTIONS + ("predict",):
        setattr(m, n, lambda *a, **k: "ref")
    return m


@pytest.mark.parametrize("device", ["cpu", "cuda"])
@pytest.mark.parametrize("name,wh", [("p_nc1", (200, 160)), ("p_nc3", (224, 224)), ("p_nc80", (100, 128)), ("p_nc1_dense", (160, 160))])
def test_rebound_predict_reproduces_the_reference_goldens(tmp_path, golden, name, wh, device):
    """f-3: `train.predict` rebound by install() — same signature, the module's own image loading and
    letterbox, everything after the model call on the B200 path — against the detections the unmodified
    predict() produced (oracle/make_golden.py: golden_predict), for a CPU model (the reference tests' case)
    and a CUDA model; predict_batch gives the same per image."""
    from PIL import Image
    from yolo_from_scratch_b200.install import install, uninstall
    from oracle import ref_path as R
    g = golden("predict")
    img, nc, conf, iou, scale, pt, pl = g[f"{name}_cfg"]
    train = install(_train_stand_in(float(scale), int(pt), int(pl)))
    assert train.predict.__doc__.startswith("Drop-in")
    path = str(tmp_path / f"{name}.png")
    Image.fromarray(np.zeros((wh[1], wh[0], 3), dtype=np.uint8)).save(path)
    dev = torch.device(device)
    heads = [torch.from_numpy(g[f"{name}_head{s}"]).to(dev) for s in range(3)]
    model = _PresetHeads(heads, int(img), [a.to(dev) for a in R.default_anchors()])
    try:
        dets = train.predict(model, path, dev, num_classes=int(nc), conf_threshold=float(conf), iou_threshold=float(iou))
        many = train.predict_batch(_PresetHeads([torch.cat([h, h]) for h in heads], int(img), model.anchors), [path, path],
                                   dev, num_classes=int(nc), conf_threshold=float(conf), iou_threshold=float(iou))
    finally:
        uninstall(train)
    want = g[f"{name}_dets"]
    assert isinstance(dets, list) and all(isinstance(d, tuple) and len(d) == 6 and isinstance(d[5], int) for d in dets)
    # the golden ran torchvision's CPU kernel; candidates within a few ulp of the confidence threshold may differ
    assert abs(len(dets) - len(want)) <= max(2, len(want) // 200), (len(dets), len(want))
    if len(dets) == len(want):
        a, b = _canon(dets), _canon(want)
        assert np.array_equal(a[:, 5], b[:, 5])
        assert np.allclose(a[:, :4], b[:, :4], rtol=1e-4, atol=1e-2) and np.allclose(a[:, 4], b[:, 4], rtol=1e-4, atol=1e-6)
    assert len(many) == 2 and many[0] == dets and many[1] == dets


@pytest.mark.parametrize("nc", [1, 80])
def test_channels_last_model_hands_over_heads_without_the_permute_copy(nc, monkeypatch):
    """f-2 inside the drop-in flow: with install(..., channels_last=True) the UNCHANGED `train.YOLO` runs in NHWC,
    the three tensors `forward` returns (train.py:608-609) alias the head convs' outputs (no view/permute/contiguous
    copy), and loss + gradients through the swap equal the default NCHW model's and the oracle's on the same heads."""
    _need_ref()
    sys.path.insert(0, REF)
    from yolo_from_scratch_b200.install import enable_import_hook, channels_last_heads
    enable_import_hook()
    import train
    from oracle import ref_path as R
    dev = torch.device("cuda")
    torch.manual_seed(3)
    # full-precision convolutions for the NCHW-vs-NHWC comparison below (cuDNN's TF32 kernels differ by ~1e-3 per layer)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    plain = train.YOLO(num_classes=nc, img_size=320).to(dev).train()
    nhwc = train.YOLO(num_classes=nc, img_size=320).to(dev).train()
    nhwc.load_state_dict(plain.state_dict())
    channels_last_heads(nhwc)
    last_conv = lambda m: [c for c in m.head_p3.modules() if isinstance(c, torch.nn.Conv2d)][-1]
    assert last_conv(nhwc).weight.dim() == 4 and getattr(nhwc, "__yolo_b200_channels_last__", False)
    seen = {}
    hooks = [h.register_forward_hook(lambda m, i, o, k=k: seen.__setitem__(k, o))
             for k, h in enumerate((nhwc.head_p3, nhwc.head_p4, nhwc.head_p5))]
    x = torch.rand(4, 3, 320, 320, device=dev)
    heads = nhwc(x)
    for k, h in enumerate(heads):
        assert h.is_contiguous() and h.shape[-1] == 5 + nc
        assert h.data_ptr() == seen[k].data_ptr(), "head %d was copied" % k
    for h in hooks:
        h.remove()
    heads_plain = plain(x)
    for a, b in zip(heads, heads_plain):
        assert torch.allclose(a, b, rtol=5e-3, atol=5e-3), float((a - b).abs().max())
    rng = np.random.default_rng(5)
    labels = [np.column_stack([rng.integers(0, nc, 3), rng.uniform(0.2, 0.8, (3, 2)), rng.uniform(0.05, 0.4, (3, 2))]).astype(np.float64)
              for _ in range(4)]
    grids = [h.shape[1] for h in heads]
    tg = [torch.from_numpy(np.stack(t)).to(dev) for t in zip(*[R.assign_targets(l, R.default_anchors(), grids, nc, 320) for l in labels])]
    out = train.yolo_loss_multiscale(heads, tg, nhwc.anchors, nc)
    out[0].backward()
    out_plain = train.yolo_loss_multiscale(heads_plain, tg, plain.anchors, nc)
    out_plain[0].backward()
    want = R.multiscale_loss([h.detach().cpu() for h in heads], [t.cpu() for t in tg], R.default_anchors(), nc)
    for got, w in zip(out, want[:4]):
        assert abs(float(got) - float(w)) <= 2e-5 * max(1.0, abs(float(w)))
    for got, w in zip(out, out_plain):
        assert abs(float(got) - float(w)) <= 2e-3 * max(1.0, abs(float(w)))
    ga, gb = last_conv(nhwc).weight.grad, last_conv(plain).weight.grad
    assert ga is not None and torch.isfinite(ga).all()
    assert float((ga - gb).abs().max()) <= 2e-2 * float(gb.abs().max()) + 1e-6


def test_reference_cli_trains_with_channels_last_heads(tmp_path):
    """The unchanged CLI (train.py:1520-1522) with YOLO_B200_CHANNELS_LAST=1: one epoch, finite losses, checkpoint
    written and readable by the UNPATCHED reference's eval mode (the state dict keeps the reference's shapes)."""
    _need_ref()
    cfg, dirs = _make_dataset(tmp_path)
    train_py = os.path.join(REF, "train.py")
    env = _env()
    env["YOLO_B200_CHANNELS_LAST"] = "1"
    p = subprocess.run([sys.executable, "-m", "yolo_from_scratch_b200.run", train_py, cfg, "--epochs", "1", "--img-size", "320",
                        "--size", "n"], capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=1500)
    _log("reference_cli_channels_last.log", p.stdout[-6000:] + "\n--- stderr ---\n" + p.stderr[-3000:])
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "Epoch 1:" in p.stdout and "Training complete" in p.stdout and "nan" not in p.stdout.lower()
    ckpts = sorted(f for f in os.listdir(tmp_path) if f.startswith("yolo_") and f.endswith(".pt"))
    assert len(ckpts) == 1
    q = subprocess.run([sys.executable, train_py, cfg, str(tmp_path / ckpts[0]), "--size", "n"], capture_output=True, text=True,
                       env=_env(), cwd=str(tmp_path), timeout=1500)
    assert q.returncode == 0 and "F1 Score:" in q.stdout, q.stdout[-2000:] + q.stderr[-2000:]
