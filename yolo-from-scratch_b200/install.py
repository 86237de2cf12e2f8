"""Drop-in boundary (SURVEY 8b): swap the B200 path in under the reference's own names.

The reference (`train.py`) has no plugin API; its callers resolve `decode_predictions`,
`ciou_loss`, `yolo_loss`, `yolo_loss_multiscale` through module globals at call time
(train.py:796, :818, :874, :909, :987, :993, :1154), the CLI resolves `eval_epoch` and `predict` the same way
(:1413, :1436, :1523; :1444, eval.py:8 via `from train import predict`), and target assignment lives in
`YOLODataset.__getitem__` / `compute_anchor_iou` (:108-131, :147-205).  `install(train_module)`
rebinds exactly those names; the file on disk is untouched.  `predict` is rebound as a whole
(SURVEY 8f-3), so the swap no longer touches `torchvision.ops.batched_nms` for the rest of the process
(`patch_torchvision=True` restores the round-1 behaviour for callers that use the reference's own predict).

  import train; from yolo_from_scratch_b200.install import install; install(train)
  pytest -p yolo_from_scratch_b200.pytest_plugin /path/to/reference/tests     # unchanged suite
  python -m yolo_from_scratch_b200.run /path/to/train.py data.yaml            # unchanged CLI
"""
import importlib.abc
import importlib.machinery
import sys

from . import ops

PATCHED_FUNCTIONS = ("decode_predictions", "ciou_loss", "yolo_loss", "yolo_loss_multiscale")
_MARK = "__yolo_b200_installed__"


def looks_like_reference(module) -> bool:
    return all(hasattr(module, n) for n in PATCHED_FUNCTIONS + ("YOLODataset", "predict"))


def _read_labels(train_module, label_file):
    """The label lines of one image as YOLODataset.__getitem__ reads them (train.py:148-154): (n,5) fp64
    [class, xc, yc, w, h]; a missing file is an image without objects."""
    import numpy as np
    rows = []
    label_path = train_module.__dict__["Path"](label_file)
    if label_path.exists():
        with open(label_path, encoding="utf-8") as f:
            for line in f:
                parts = line.strip().split()
                if len(parts) == 5:
                    rows.append([float(int(float(parts[0])))] + [float(x) for x in parts[1:]])
    return np.array(rows, dtype=np.float64).reshape(-1, 5)


def _make_getitem(train_module):
    """Replacement for YOLODataset.__getitem__ (train.py:133-207): image loading and letterbox stay
    the reference's (host image I/O is out of scope); the label loop runs in yb_build_targets."""
    def __getitem__(self, idx):
        import numpy as np
        import torch
        if _in_dataloader_worker():
            raise RuntimeError(
                "YOLODataset.__getitem__ on the B200 path runs its label loop on the GPU and cannot be used from "
                "DataLoader worker processes (CUDA after fork); use num_workers=0 like the reference (train.py:1471-1474) "
                "or install(..., patch_dataset=False) to keep the reference's CPU label loop")
        g = train_module.__dict__
        pil_img = g["Image"].open(self.imgs[idx]).convert("RGB")                      # :135
        orig_w, orig_h = pil_img.size
        pil_img, scale, pad_top, pad_left = g["letterbox_resize"](pil_img, self.img_size)   # :137
        img = torch.from_numpy(np.array(pil_img)).permute(2, 0, 1).float() / 255.0    # :138
        targets = ops.build_targets([_read_labels(train_module, self.labels[idx])], self.anchors, self.grid_sizes,
                                    self.num_classes, self.img_size,
                                    letterbox=[(orig_w, orig_h, scale, pad_top, pad_left)])
        return img, [t[0].cpu() for t in targets]
    return __getitem__


def _make_predict(train_module):
    """Signature-identical replacements for predict() (train.py:1114-1250) plus a batched variant.  Image
    loading and letterbox stay the reference's (host image I/O is out of scope); the model call is the
    caller's model; everything after it (:1140-1246) is ops.predict_heads."""
    def _load(image_path, img_size, device):
        import numpy as np
        import torch
        g = train_module.__dict__
        pil_img = g["Image"].open(image_path).convert("RGB")                                   # :1134
        pil_img, scale, pad_top, pad_left = g["letterbox_resize"](pil_img, img_size)           # :1137
        img = torch.from_numpy(np.array(pil_img)).permute(2, 0, 1).float() / 255.0             # :1138
        return img, (scale, pad_top, pad_left)

    def predict(model, image_path, device, num_classes=1, conf_threshold=0.5, iou_threshold=0.4):
        return predict_batch(model, [image_path], device, num_classes, conf_threshold, iou_threshold)[0]

    def predict_batch(model, image_paths, device, num_classes=1, conf_threshold=0.5, iou_threshold=0.4):
        """predict() for a list of images with ONE model call and one pass of the detection path; returns
        a list (per image) of the reference's detection lists."""
        import torch
        model.eval()                                                                            # :1131
        img_size = model.img_size
        if len(image_paths) == 0:
            return []
        loaded = [_load(p, img_size, device) for p in image_paths]
        imgs = torch.stack([im for im, _ in loaded]).to(device)                                 # :1139
        with torch.no_grad():
            preds = model(imgs)                                                                 # :1141-1142
        return ops.predict_heads(preds, model.anchors, img_size, num_classes, conf_threshold, iou_threshold,
                                 letterbox=[lb for _, lb in loaded])
    predict.__doc__ = "Drop-in for train.predict (train.py:1114-1250): same arguments, same return value."
    return predict, predict_batch


def _evaluate_dataset(train_module, metric, model, dataset, device, num_classes, conf_threshold, iou_threshold,
                      batch_size, group, multi_label=False, agnostic=False, max_candidates=None):
    """Feed `metric` (DetectionMAP, COCODetectionEval or DetectionReport) the detections of `model` on `dataset` (its imgs and labels
    lists) batch by batch and return metric.compute().  Images are loaded and letterboxed by the module's own Image
    and letterbox_resize, as predict() does (train.py:1134-1138).  With a torch.distributed `group` this rank takes
    only its contiguous block of images, dist.shard_range(len(dataset.imgs), rank, world), and returns
    metric.compute(group): every rank of the group must call it, and every rank gets the result over all images.
    multi_label, agnostic and max_candidates go to ops.detect_batch."""
    import numpy as np
    import torch
    from .dist import shard_range
    g = train_module.__dict__
    model.eval()
    img_size = model.img_size
    lo, hi = 0, len(dataset.imgs)
    if group is not None:
        import torch.distributed as dist
        lo, hi = shard_range(hi, dist.get_rank(group), dist.get_world_size(group))
    with torch.no_grad():
        for i0 in range(lo, hi, batch_size):
            imgs, letterbox, labels = [], [], []
            for i in range(i0, min(i0 + batch_size, hi)):
                pil_img = g["Image"].open(dataset.imgs[i]).convert("RGB")
                orig_w, orig_h = pil_img.size
                pil_img, scale, pad_top, pad_left = g["letterbox_resize"](pil_img, img_size)
                imgs.append(torch.from_numpy(np.array(pil_img)).permute(2, 0, 1).float() / 255.0)
                letterbox.append((orig_w, orig_h, scale, pad_top, pad_left))
                labels.append(_read_labels(train_module, dataset.labels[i]))
            preds = model(torch.stack(imgs).to(device))
            det = ops.detect_batch(list(preds), model.anchors, img_size, num_classes, conf_threshold, iou_threshold,
                                   letterbox=[lb[2:] for lb in letterbox], multi_label=multi_label,
                                   max_candidates=max_candidates, agnostic=agnostic)
            metric.update(det, ops.pack_labels(labels, img_size, letterbox))
    return metric.compute(group)


def _make_evaluate_map(train_module):
    """`evaluate_map`, a name the reference does not have: COCO-style mAP of a model over a YOLODataset's images
    and label files (ops.DetectionMAP)."""
    def evaluate_map(model, dataset, device, num_classes=1, conf_threshold=0.001, iou_threshold=0.4, batch_size=8,
                     max_det=300, group=None, *, multi_label=False, agnostic=False, max_candidates=None):
        """mAP@[.5:.95] / mAP@0.5 of `model` on `dataset` (its imgs and labels lists).  Returns DetectionMAP.compute()'s
        dict: map, map50, ap (nc,T), precision (T,R,nc), recall (T,nc), n_gt (nc), n_det (nc).  group: a
        torch.distributed process group; every rank calls evaluate_map, scores only its block of the images
        (dist.shard_range) and gets the result over all of them (DetectionMAP.compute(group)).
        multi_label=True scores the multi-label candidates of YOLO validation tools (one per (row, class) pair above
        conf_threshold, at most max_candidates per image, None = ops.MAX_CANDIDATES); agnostic=True suppresses across
        classes (ops.detect_batch)."""
        metric = ops.DetectionMAP(num_classes, max_det=max_det)
        return _evaluate_dataset(train_module, metric, model, dataset, device, num_classes, conf_threshold,
                                 iou_threshold, batch_size, group, multi_label, agnostic, max_candidates)
    return evaluate_map


def _make_evaluate_coco(train_module):
    """`evaluate_coco`, a name the reference does not have: COCO's twelve bbox stats of a model over a YOLODataset's
    images and label files (ops.COCODetectionEval)."""
    def evaluate_coco(model, dataset, device, num_classes=1, conf_threshold=0.001, iou_threshold=0.4, batch_size=8,
                      max_det=300, max_dets=ops.COCO_MAX_DETS, group=None, *, multi_label=False, agnostic=False,
                      max_candidates=None):
        """COCO's bbox summary of `model` on `dataset` (its imgs and labels lists).  Returns
        COCODetectionEval.compute()'s dict: stats (12,), precision (T,R,nc,A,M), recall (T,nc,A,M), n_gt (nc,A),
        n_det (nc), ap (nc,T), map, map50; ops.format_coco_stats(stats) gives pycocotools' printed lines.  group,
        multi_label, agnostic, max_candidates: as evaluate_map's."""
        metric = ops.COCODetectionEval(num_classes, max_det=max_det, max_dets=max_dets)
        return _evaluate_dataset(train_module, metric, model, dataset, device, num_classes, conf_threshold,
                                 iou_threshold, batch_size, group, multi_label, agnostic, max_candidates)
    return evaluate_coco


def _make_evaluate_report(train_module):
    """`evaluate_report`, a name the reference does not have: the validation report of a model over a YOLODataset's
    images and label files (ops.DetectionReport)."""
    def evaluate_report(model, dataset, device, num_classes=1, conf_threshold=0.001, iou_threshold=0.4, batch_size=8,
                        max_det=300, group=None, *, multi_label=False, agnostic=False, max_candidates=None):
        """Confusion matrix, P/R/F1 curves over the confidence threshold, best-F1 threshold and the AP columns of
        `model` on `dataset` (its imgs and labels lists).  Returns DetectionReport.compute()'s dict;
        ops.format_detection_report(out) gives the per-class table.  group, multi_label, agnostic, max_candidates: as
        evaluate_map's."""
        metric = ops.DetectionReport(num_classes, max_det=max_det)
        return _evaluate_dataset(train_module, metric, model, dataset, device, num_classes, conf_threshold,
                                 iou_threshold, batch_size, group, multi_label, agnostic, max_candidates)
    return evaluate_report


def channels_last_heads(model):
    """SURVEY 8f-2 for the UNCHANGED model: run the network in NHWC (`torch.channels_last`).  The head convs
    then write (B, H, W, A*(5+nc)) in memory, on which train.py:608-609's view/permute is a pure stride change and
    `.contiguous()` returns its argument: the three heads reach the loss / decode kernels in the reference's
    (B,H,W,A,5+nc) layout WITHOUT the copy pass (the returned tensors alias the conv outputs), and the
    gradient flows back to the conv the same way.  Idempotent; returns the model."""
    import torch
    if getattr(model, "__yolo_b200_channels_last__", False):
        return model
    model.to(memory_format=torch.channels_last)

    def _nhwc_input(_module, args):
        x = args[0]
        if x.dim() == 4 and not x.is_contiguous(memory_format=torch.channels_last):
            return (x.contiguous(memory_format=torch.channels_last),) + tuple(args[1:])
        return None
    model.register_forward_pre_hook(_nhwc_input)
    model.__yolo_b200_channels_last__ = True
    return model


def _wrap_model_init(train_module):
    cls = train_module.YOLO
    orig = cls.__init__

    def __init__(self, *args, **kwargs):
        orig(self, *args, **kwargs)
        channels_last_heads(self)
    __init__.__wrapped__ = orig
    cls.__init__ = __init__
    return orig


def _in_dataloader_worker():
    try:
        import torch.utils.data
        return torch.utils.data.get_worker_info() is not None
    except Exception:  # pragma: no cover
        return False


def install(train_module, patch_torchvision=False, patch_dataset=True, patch_eval=True, patch_predict=True,
            channels_last=None):
    """Rebind the hot-path names of an imported reference `train` module.  Idempotent.
    channels_last (default: environment YOLO_B200_CHANNELS_LAST=1) makes every `train.YOLO` built afterwards
    run in NHWC, so that the head layout conversion of train.py:608-609 costs nothing (channels_last_heads).
    patch_eval also swaps `eval_epoch` (SURVEY 8f-1: its per-anchor python loop becomes one kernel);
    patch_predict swaps `predict` and adds `predict_batch` (SURVEY 8f-3); `evaluate_map` (COCO-style mAP),
    `evaluate_coco` (COCO's twelve bbox stats) and `evaluate_report` (confusion matrix, P/R/F1 curves, per-class
    table), names the reference does not have, are always added; patch_torchvision additionally
    rebinds torchvision.ops.batched_nms process-wide (off by default: predict no longer needs it)."""
    if getattr(train_module, _MARK, False):
        return train_module
    saved = {}
    for name in PATCHED_FUNCTIONS:
        saved[name] = getattr(train_module, name)
        setattr(train_module, name, getattr(ops, name))
    if patch_eval and hasattr(train_module, "eval_epoch"):
        saved["eval_epoch"] = train_module.eval_epoch
        train_module.eval_epoch = ops.eval_epoch
    if patch_predict and hasattr(train_module, "predict"):
        saved["predict"] = train_module.predict
        train_module.predict, train_module.predict_batch = _make_predict(train_module)
    if not hasattr(train_module, "evaluate_map"):
        saved["evaluate_map"] = None
        train_module.evaluate_map = _make_evaluate_map(train_module)
    if not hasattr(train_module, "evaluate_coco"):
        saved["evaluate_coco"] = None
        train_module.evaluate_coco = _make_evaluate_coco(train_module)
    if not hasattr(train_module, "evaluate_report"):
        saved["evaluate_report"] = None
        train_module.evaluate_report = _make_evaluate_report(train_module)
    if patch_dataset and hasattr(train_module, "YOLODataset"):
        cls = train_module.YOLODataset
        saved["YOLODataset.__getitem__"] = cls.__getitem__
        saved["YOLODataset.compute_anchor_iou"] = cls.compute_anchor_iou
        cls.__getitem__ = _make_getitem(train_module)
        cls.compute_anchor_iou = lambda self, box_wh, anchors: ops.compute_anchor_iou(box_wh, anchors)
    if channels_last is None:
        import os
        channels_last = os.environ.get("YOLO_B200_CHANNELS_LAST", "0") == "1"
    if channels_last and hasattr(train_module, "YOLO"):
        saved["YOLO.__init__"] = _wrap_model_init(train_module)
    if patch_torchvision:
        import torchvision
        import torchvision.ops.boxes as tvb
        saved["torchvision.ops.batched_nms"] = torchvision.ops.batched_nms
        torchvision.ops.batched_nms = ops.batched_nms
        tvb.batched_nms = ops.batched_nms
    setattr(train_module, "__yolo_b200_saved__", saved)
    setattr(train_module, _MARK, True)
    return train_module


def uninstall(train_module):
    saved = getattr(train_module, "__yolo_b200_saved__", None)
    if not saved:
        return
    for name in PATCHED_FUNCTIONS:
        setattr(train_module, name, saved[name])
    if "eval_epoch" in saved:
        train_module.eval_epoch = saved["eval_epoch"]
    if "predict" in saved:
        train_module.predict = saved["predict"]
        if hasattr(train_module, "predict_batch"):
            del train_module.predict_batch
    if "evaluate_map" in saved:
        del train_module.evaluate_map
    if "evaluate_coco" in saved:
        del train_module.evaluate_coco
    if "evaluate_report" in saved:
        del train_module.evaluate_report
    if "YOLODataset.__getitem__" in saved:
        train_module.YOLODataset.__getitem__ = saved["YOLODataset.__getitem__"]
        train_module.YOLODataset.compute_anchor_iou = saved["YOLODataset.compute_anchor_iou"]
    if "YOLO.__init__" in saved:
        train_module.YOLO.__init__ = saved["YOLO.__init__"]
    if "torchvision.ops.batched_nms" in saved:
        import torchvision
        import torchvision.ops.boxes as tvb
        torchvision.ops.batched_nms = saved["torchvision.ops.batched_nms"]
        tvb.batched_nms = saved["torchvision.ops.batched_nms"]
    setattr(train_module, _MARK, False)


class _PatchingLoader(importlib.abc.Loader):
    def __init__(self, inner):
        self.inner = inner

    def create_module(self, spec):
        return self.inner.create_module(spec)

    def exec_module(self, module):
        self.inner.exec_module(module)
        if looks_like_reference(module):
            install(module)


class _TrainFinder(importlib.abc.MetaPathFinder):
    """Patches a module called `train` right after it is executed, so that
    `from train import yolo_loss_multiscale` in a test module already binds the B200 path."""

    def find_spec(self, fullname, path, target=None):
        if fullname != "train":
            return None
        spec = importlib.machinery.PathFinder.find_spec(fullname, path)
        if spec is None or spec.loader is None:
            return None
        spec.loader = _PatchingLoader(spec.loader)
        return spec


_finder = None


def enable_import_hook():
    global _finder
    if _finder is None:
        _finder = _TrainFinder()
        sys.meta_path.insert(0, _finder)
    mod = sys.modules.get("train")
    if mod is not None and looks_like_reference(mod):
        install(mod)


def disable_import_hook():
    global _finder
    if _finder is not None and _finder in sys.meta_path:
        sys.meta_path.remove(_finder)
    _finder = None
