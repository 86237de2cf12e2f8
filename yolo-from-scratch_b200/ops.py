"""Host-side mirror of the reference's per-box hot-path functions (reference `train.py`).

Same names, argument meaning and return values as the reference so that callers and tests read
the same; the arithmetic runs in libyolo_b200.so (hand-written sm_100a kernels, C-ABI in
include/yolo_b200.h).  PyTorch is used only for device memory, streams and autograd plumbing.

  decode_predictions      train.py:712-779
  ciou_loss               train.py:634-710
  yolo_loss               train.py:781-838
  yolo_loss_multiscale    train.py:840-886
  compute_anchor_iou      train.py:108-131
  build_targets           train.py:147-205 (label loop of YOLODataset.__getitem__), batched
  filter_candidates       train.py:1152-1229 (per-scale body of predict), batched
  nms / batched_nms       torchvision.ops as called at train.py:1232-1233
  detect_batch            filter_candidates + batched_nms + gather (predict :1152-1238 for a batch)
  filter_candidates_multilabel  multi-label candidates with a per-image top-K cap (new; YOLO validation's candidate set)
  DetectionMAP            COCO-style mAP of detect_batch's detections (new; no reference equivalent)
  DetectionReport         confusion matrix, P/R/F1 over confidence, best-F1 threshold, per-class table (new)

CPU tensors are accepted (the reference's tests pass CPU tensors): they are staged to the GPU,
computed there, and staged back.  That is staging, not a fallback: without CUDA every function
raises.
"""
import ctypes
import math
import zlib
from typing import List, NamedTuple, Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import HeadsDesc, LossDesc, MAX_ANCHORS, MAX_SCALES

# reference constants
BOX_WEIGHT = 0.05                 # train.py:836
CLS_WEIGHT = 0.5                  # train.py:836
MULTISCALE_OBJ_WEIGHTS = (4.0, 1.0, 0.4)  # train.py:865
LOSS_DECODE_IMG_SIZE = 640.0      # train.py:796 — yolo_loss always decodes with the default
CIOU_EPS = 1e-7                   # train.py:634
DEFAULT_ANCHORS = (               # train.py:372-374 (model) / :81-83 (dataset): P3, P4, P5 anchors in pixels
    ((10, 13), (16, 30), (33, 23)),
    ((30, 61), (62, 45), (59, 119)),
    ((116, 90), (156, 198), (373, 326)),
)
TRICK_MAX_NUMEL_CUDA = 100_000    # torchvision/ops/boxes.py:80
TRICK_MAX_NUMEL_CPU = 4_000


# --------------------------------------------------------------------------------------------
# plumbing
# --------------------------------------------------------------------------------------------
def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError(
            "yolo_from_scratch_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def dist_global_batch(local_batch, group):
    from .dist import global_batch
    return global_batch(local_batch, group)


def _ptr(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.data_ptr()


_HEAD_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16}


def _contig(t: torch.Tensor, dev: torch.device, half: bool = False) -> torch.Tensor:
    """`t` as the kernels read it: on `dev`, contiguous, 16-byte aligned (differentiable); fp32, or with half=True
    bf16 and fp16 kept as they are (a CPU half tensor is staged as half) and any other dtype made fp32."""
    if t.device != dev:
        t = t.to(dev)
    if t.dtype != torch.float32 and not (half and t.dtype in _HEAD_DTYPES):
        t = t.float()
    t = t.contiguous()
    if t.data_ptr() % 16:
        t = t.clone()
    return t


_anchor_cache = {}


def _anchors_dev(anchors, dev: torch.device) -> torch.Tensor:
    """(A,2) fp32 anchors on the device; small host-side cache so a CPU anchor tensor is not
    re-uploaded on every call."""
    if isinstance(anchors, torch.Tensor):
        if anchors.device == dev and anchors.dtype == torch.float32 and anchors.is_contiguous():
            return anchors.detach()
        key = (anchors.data_ptr(), anchors._version, tuple(anchors.shape), str(anchors.dtype), dev.index)
        hit = _anchor_cache.get(key)
        if hit is not None and torch.equal(hit[0], anchors.detach().cpu() if anchors.device.type != "cpu" else anchors.detach()):
            return hit[1]
        host = anchors.detach().to("cpu", torch.float32).contiguous()
        out = host.to(dev)
        if len(_anchor_cache) > 64:
            _anchor_cache.clear()
        _anchor_cache[key] = (host.clone(), out)
        return out
    return torch.tensor(anchors, dtype=torch.float32, device=dev).reshape(-1, 2).contiguous()


def default_anchors(device=None) -> List[torch.Tensor]:
    """The reference's default anchors as three (3,2) fp32 tensors (train.py:372-374)."""
    return [torch.tensor(a, dtype=torch.float32, device=device) for a in DEFAULT_ANCHORS]


LAYOUT_BHWAC, LAYOUT_NCHW = _lib.LAYOUT_BHWAC, _lib.LAYOUT_NCHW


def _grid(p: torch.Tensor, layout: int):
    """(H, W) of a head tensor: (B,H,W,A,5+nc) or, NCHW, (B, A*(5+nc), H, W)."""
    return (p.shape[2], p.shape[3]) if layout == LAYOUT_NCHW else (p.shape[1], p.shape[2])


def _stage_heads(predictions, anchors_list, num_classes, layout, targets=None, *, half=True, detach=True, dev=None):
    """Heads, anchors and dense targets as the kernels read them: every op that reads head tensors stages them here.

    The kernels receive pointers and the sizes of one descriptor: B of scale 0, A of the first anchor set and rows
    of 5+nc.  So every scale's shapes are checked first, on the host, before anything touches the device; a
    mismatch raises ValueError naming the scale.

    predictions: S heads (B,H,W,A,5+nc), or (B,A*(5+nc),H,W) with layout=LAYOUT_NCHW.  num_classes: None takes nc
    from scale 0's rows (reference layout).  targets: None, S dense targets (B,H,W,A,5+nc) in either layout, or a
    PackedLabels.  half: bf16 / fp16 heads are kept (heads of mixed dtypes are all read as fp32); False reads every
    head as fp32.  detach: drop the heads' autograd history (the filters do; the loss and decode keep it).
    dev: where to stage, None = the current CUDA device.
    Returns (preds, tgts, ancs), S device tensors each; tgts is None unless dense targets were given."""
    S = len(predictions)
    if not 1 <= S <= MAX_SCALES:
        raise ValueError(f"1..{MAX_SCALES} scales supported, got {S}")
    dense = targets is not None and not isinstance(targets, PackedLabels)
    if len(anchors_list) < S:
        raise ValueError(f"scale {len(anchors_list)}: no anchor set ({S} heads, {len(anchors_list)} anchor sets)")
    if dense and len(targets) < S:
        raise ValueError(f"scale {len(targets)}: no targets ({S} heads, {len(targets)} targets)")
    nc = None if num_classes is None else int(num_classes)
    if nc is not None and nc < 0:
        raise ValueError(f"num_classes must be >= 0, got {nc}")
    for s, p in enumerate(predictions):
        a = anchors_list[s]
        a_shape = a.shape if isinstance(a, torch.Tensor) else np.shape(a)
        if len(a_shape) != 2 or a_shape[1] != 2:
            raise ValueError(f"scale {s}: anchors must be (A, 2), got shape {tuple(a_shape)}")
        A = a_shape[0]
        if A > MAX_ANCHORS:
            raise ValueError(f"scale {s}: at most {MAX_ANCHORS} anchors per scale, got {A}")
        shape = p.shape
        if layout == LAYOUT_NCHW:
            if len(shape) != 4 or shape[1] != A * (5 + nc):
                raise ValueError(f"scale {s}: NCHW head must be (B, {A}*(5+num_classes), H, W), got {tuple(shape)}")
            B, _, H, W = shape
        else:
            if len(shape) != 5:
                raise ValueError(f"scale {s}: head must be (B, H, W, A, 5+nc), got {tuple(shape)}")
            B, H, W, A_head, row = shape
            if row < 5:
                raise ValueError(f"scale {s}: last dimension must be 5+nc, got {row}")
            if nc is None:
                nc = row - 5
            if A_head != A:
                raise ValueError(f"scale {s}: head has {A_head} anchors, its anchor set {A}")
            if row != 5 + nc:
                raise ValueError(f"scale {s}: last dimension {row} != 5+num_classes = {5 + nc}")
        if s == 0:
            B0, A0 = B, A
        elif B != B0:
            raise ValueError(f"scale {s}: batch {B}, scale 0 has {B0}")
        elif A != A0:
            raise ValueError(f"scale {s}: {A} anchors, scale 0 has {A0}")
        if dense:
            t = targets[s]
            if not isinstance(t, torch.Tensor) or t.shape != (B, H, W, A, 5 + nc):
                got = tuple(t.shape) if isinstance(t, torch.Tensor) else t
                raise ValueError(f"scale {s}: targets {got} do not match the head, expected {(B, H, W, A, 5 + nc)}")
    if isinstance(targets, PackedLabels) and targets.labels.shape[0] != B0:
        raise ValueError(f"labels of {targets.labels.shape[0]} images, the heads' batch is {B0} (scale 0)")
    if dev is None:
        dev = _device()
    preds = [_contig(p.detach() if detach else p, dev, half) for p in predictions]
    if len({p.dtype for p in preds}) > 1:
        preds = [p.float() for p in preds]
    tgts = [_contig(t.detach(), dev) for t in targets[:S]] if dense else None
    ancs = [_anchors_dev(a, dev) for a in anchors_list[:S]]
    return preds, tgts, ancs


def _heads_desc(d, preds, ancs, nc, img_size, layout):
    """Fill the fields yb_heads_desc and yb_loss_desc share (S, B, A, nc, img_size, layout, dtype, H, W, pred,
    anchors) of `d` from staged heads; returns d."""
    d.S, d.B, d.A, d.nc = len(preds), preds[0].shape[0], ancs[0].shape[0], nc
    d.img_size = float(img_size)
    d.layout = layout
    d.dtype = _HEAD_DTYPES[preds[0].dtype]
    for s, p in enumerate(preds):
        d.H[s], d.W[s] = _grid(p, layout)
        d.pred[s] = p.data_ptr()
        d.anchors[s] = ancs[s].data_ptr()
    return d


# --------------------------------------------------------------------------------------------
# a-1 decode_predictions
# --------------------------------------------------------------------------------------------
class _DecodeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, anchors, img_size):
        B, H, W, A, row = pred.shape
        out = torch.empty_like(pred)
        _lib.check(_lib.lib().yb_decode_fwd_t(pred.data_ptr(), anchors.data_ptr(), out.data_ptr(), B, H, W, A, row - 5,
                                              float(img_size), _HEAD_DTYPES[pred.dtype], _stream()), "yb_decode_fwd_t")
        ctx.save_for_backward(pred, anchors)
        ctx.img_size = float(img_size)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        pred, anchors = ctx.saved_tensors
        B, H, W, A, row = pred.shape
        grad_out = _contig(grad_out.to(pred.dtype), pred.device, half=True)
        grad_in = torch.empty_like(pred)
        _lib.check(_lib.lib().yb_decode_bwd_t(pred.data_ptr(), anchors.data_ptr(), grad_out.data_ptr(),
                                              grad_in.data_ptr(), B, H, W, A, row - 5, ctx.img_size,
                                              _HEAD_DTYPES[pred.dtype], _stream()), "yb_decode_bwd_t")
        return grad_in, None, None


def decode_predictions(raw_preds: torch.Tensor, anchors, img_size=640) -> torch.Tensor:
    """train.py:712-779.  (B,H,W,A,5+nc) raw logits -> same shape with xywh decoded to
    normalised coordinates; objectness/class logits unchanged.  Differentiable.  bf16 / fp16 heads are
    decoded natively: the result is the fp32 decode of the upcast heads rounded to the head dtype."""
    (pred,), _, (anc,) = _stage_heads([raw_preds], [anchors], None, LAYOUT_BHWAC, detach=False)
    dev = pred.device
    orig_dev, orig_dtype = raw_preds.device, raw_preds.dtype
    with torch.cuda.device(dev):
        out = _DecodeFn.apply(pred, anc, img_size)
    if out.dtype != orig_dtype:
        out = out.to(orig_dtype)
    return out if orig_dev == dev else out.to(orig_dev)


# --------------------------------------------------------------------------------------------
# a-2 ciou_loss
# --------------------------------------------------------------------------------------------
class _CiouFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred_boxes, target_boxes, eps):
        N = pred_boxes.shape[0]
        L = _lib.lib()
        loss = torch.empty(1, dtype=torch.float32, device=pred_boxes.device)
        need_p, need_t = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gp = torch.empty_like(pred_boxes) if need_p else None
        gt = torch.empty_like(target_boxes) if need_t else None
        scratch = torch.empty(16, dtype=torch.uint8, device=pred_boxes.device)
        _lib.check(L.yb_ciou_fwd_bwd(pred_boxes.data_ptr(), target_boxes.data_ptr(), N, float(eps),
                                     loss.data_ptr(), _ptr(gp), _ptr(gt), scratch.data_ptr(), 16, _stream()),
                   "yb_ciou_fwd_bwd")
        ctx.grads = (gp, gt)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        gp, gt = ctx.grads
        return (None if gp is None else gp * g), (None if gt is None else gt * g), None


def ciou_loss(pred_boxes: torch.Tensor, target_boxes: torch.Tensor, eps=CIOU_EPS) -> torch.Tensor:
    """train.py:634-710.  mean(1 - CIoU) over N (x,y,w,h) pairs."""
    if pred_boxes.dim() != 2 or pred_boxes.shape[1] != 4 or pred_boxes.shape != target_boxes.shape:
        raise ValueError("ciou_loss expects two (N,4) tensors")
    dev = _device()
    orig_dev = pred_boxes.device
    with torch.cuda.device(dev):
        p = _contig(pred_boxes, dev)
        t = _contig(target_boxes, dev)
        out = _CiouFn.apply(p, t, eps)
    return out if orig_dev == dev else out.to(orig_dev)


# --------------------------------------------------------------------------------------------
# a-3 / a-4 fused loss
# --------------------------------------------------------------------------------------------
def heads_from_nchw(raw: torch.Tensor, num_anchors: int = 3) -> torch.Tensor:
    """The reference's own head reshape (train.py:608-609): (B, A*(5+nc), H, W) -> contiguous
    (B, H, W, A, 5+nc).  The *_nchw entry points make this pass unnecessary; tests use it."""
    B, C, H, W = raw.shape
    return raw.view(B, num_anchors, C // num_anchors, H, W).permute(0, 3, 4, 1, 2).contiguous()


class _LossCfg(NamedTuple):
    """The fused loss's configuration besides its tensors."""
    nc: int
    obj_weights: tuple   # objectness weight of each scale
    group: object        # torch.distributed process group of an image-sharded batch, or None
    sparse: object       # PackedLabels: targets assigned on the device from label lists; None: dense targets
    layout: int
    S: int


def _fill_loss_desc(preds, tgts, ancs, grads, cfg, coef, B_global):
    d = _heads_desc(LossDesc(), preds, ancs, cfg.nc, LOSS_DECODE_IMG_SIZE, cfg.layout)
    d.B_global = B_global
    d.eps = CIOU_EPS
    d.w_box, d.w_cls = BOX_WEIGHT, CLS_WEIGHT
    for s in range(cfg.S):
        d.w_obj[s] = cfg.obj_weights[s]
        d.coef_box[s], d.coef_obj[s], d.coef_cls[s] = coef[s]
        d.tgt[s] = 0 if tgts is None else _ptr(tgts[s])
        d.grad[s] = _ptr(grads[s])
    return d


def loss_forward_backward(preds, tgts, ancs, nc, obj_weights, want_grad, coef=None, group=None, equal_shards=True,
                          b_global=None, reduce_fn=None, sparse=None, layout=LAYOUT_BHWAC, grad_scale=None):
    """Run the fused kernels on device tensors.  Returns (out4, per_scale(S,3), grads list).

    `group`: optional torch.distributed process group; the batch is then a shard of a global
    batch and the S*4 partial sums are all-reduced once (SURVEY 8e) between the two stages.
    `sparse`: a `PackedLabels` — targets are assigned on the device from the label lists and handed
    to the loss in sparse form (SURVEY 8f-4); `tgts` is then ignored (pass None).
    `grad_scale`: bf16 / fp16 heads only, an optional (1,) fp32 device tensor s; the gradients are then those
    of s * total (what `GradScaler.scale(total).backward()` gives), rounded to the head dtype after the scaling.
    """
    preds, tgts, ancs = _stage_heads(preds, ancs, nc, layout, tgts if sparse is None else sparse, detach=False,
                                     dev=preds[0].device if len(preds) else None)
    cfg = _LossCfg(int(nc), tuple(float(w) for w in obj_weights), group, sparse, layout, len(preds))
    out4, per_scale, grads, emit = _loss_run(cfg, preds, tgts, ancs, want_grad, coef, equal_shards, b_global, reduce_fn)
    if emit is not None:
        grads = emit(torch.ones(1, dtype=torch.float32, device=preds[0].device) if grad_scale is None else grad_scale)
    return out4, per_scale, grads


def _loss_run(cfg, preds, tgts, ancs, want, coef=None, equal_shards=True, b_global=None, reduce_fn=None):
    """Both stages on staged tensors: (out4, per_scale, grads, emit).  fp32 heads: stage 1 writes the gradients into
    grads and emit is None.  Half heads: grads is [None]*S and, when a gradient is wanted, emit(grad_scale) writes and
    returns the gradients of grad_scale * total ((1,) fp32, read on the device) from this call's partials; the
    descriptor it launches with points at preds, tgts and ancs, so they must still be alive then."""
    L = _lib.lib()
    S, sparse = cfg.S, cfg.sparse
    dev = preds[0].device
    half = preds[0].dtype != torch.float32
    if coef is None:
        coef = [(BOX_WEIGHT, cfg.obj_weights[s], CLS_WEIGHT) for s in range(S)]
    grads = [torch.empty_like(p) if w and not half else None for p, w in zip(preds, want)]
    world, B = 1, preds[0].shape[0]
    if b_global is None and cfg.group is not None:
        import torch.distributed as dist
        world = dist.get_world_size(cfg.group)
        b_global = B * world if equal_shards else dist_global_batch(B, cfg.group)
    d = _fill_loss_desc(preds, tgts, ancs, grads, cfg, coef, B if b_global is None else int(b_global))
    if sparse is None:
        ws_bytes = L.yb_loss_workspace_bytes(ctypes.byref(d))
    else:
        ws_bytes = L.yb_loss_sparse_workspace_bytes(ctypes.byref(d), sparse.max_gt)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    partials = torch.empty(S * 4, dtype=torch.float64, device=dev)
    out4 = torch.empty(4, dtype=torch.float32, device=dev)
    per_scale = torch.empty(S, 3, dtype=torch.float32, device=dev)
    st = _stream()
    if sparse is None:
        _lib.check(L.yb_loss_partials(ctypes.byref(d), partials.data_ptr(), ws.data_ptr(), ws_bytes, st),
                   "yb_loss_partials")
    else:
        anc_all = torch.stack(list(ancs)).contiguous()  # (S,A,2)
        _lib.check(L.yb_loss_partials_sparse(ctypes.byref(d), sparse.labels.data_ptr(), sparse.n_gt.data_ptr(),
                                             sparse.letterbox.data_ptr(), anc_all.data_ptr(), sparse.max_gt,
                                             int(sparse.img_size), sparse.status.data_ptr(), partials.data_ptr(),
                                             ws.data_ptr(), ws_bytes, st), "yb_loss_partials_sparse")
    if reduce_fn is not None:
        partials = reduce_fn(partials)          # test hook: emulate the collective on one GPU
    elif world > 1:
        from .dist import allreduce_partials
        allreduce_partials(partials, cfg.group)
    _lib.check(L.yb_loss_finalize(ctypes.byref(d), partials.data_ptr(), out4.data_ptr(), per_scale.data_ptr(),
                                  ws.data_ptr(), ws_bytes, st), "yb_loss_finalize")
    if not (half and any(want)):
        return out4, per_scale, grads, None

    def emit(grad_scale):
        grads = [torch.empty_like(p) if w else None for p, w in zip(preds, want)]
        for s, g in enumerate(grads):
            d.grad[s] = _ptr(g)
        _lib.check(L.yb_loss_grad_emit(ctypes.byref(d), partials.data_ptr(), grad_scale.data_ptr(),
                                       -1 if sparse is None else sparse.max_gt, ws.data_ptr(), ws.numel(), _stream()),
                   "yb_loss_grad_emit")
        return grads
    return out4, per_scale, grads, emit


class _YoloLossFn(torch.autograd.Function):
    """(total, bbox, obj, cls) = f(cfg, preds..., targets..., anchors...), S of each (targets None with label
    lists), with the gradient of `total` produced in the same pass.  Gradients that arrive on bbox/obj/cls as well are
    honoured by re-running the kernels with the combined coefficients (rare: the reference only calls
    total.backward())."""

    @staticmethod
    def forward(ctx, cfg, *tensors):
        S = cfg.S
        want = list(ctx.needs_input_grad[1:1 + S])
        out4, _, grads, emit = _loss_run(cfg, tensors[:S], tensors[S:2 * S], tensors[2 * S:], want)
        ctx.set_materialize_grads(False)
        ctx.cfg, ctx.want = cfg, want
        ctx.fused = (grads, emit)   # fp32: stage 1's gradients; half: emit, run once the upstream gradient is known
        ctx.save_for_backward(*tensors)
        return out4[0], out4[1], out4[2], out4[3]

    @staticmethod
    def backward(ctx, g_total, g_bbox, g_obj, g_cls):
        cfg, want, S = ctx.cfg, ctx.want, ctx.cfg.S
        fused, ctx.fused = ctx.fused, None
        if not any(want):
            grads = [None] * S
        elif fused is not None and g_bbox is None and g_obj is None and g_cls is None:
            # the first backward, with a gradient on `total` only (or none)
            grads, emit = fused
            if g_total is None:
                grads = [torch.zeros_like(p) if w else None for p, w in zip(ctx.saved_tensors[:S], want)]
            else:
                f = g_total.detach().to(torch.float32).reshape(1).contiguous()   # read on the device: no sync
                if emit is not None:   # half heads: written now, rounded to the head dtype after the scaling
                    grads = emit(f)
                else:                  # fp32: stage 1's gradients, scaled in place
                    for g in grads:
                        if g is not None:
                            _lib.check(_lib.lib().yb_scale_inplace(g.data_ptr(), g.numel(), f.data_ptr(), _stream()),
                                       "yb_scale_inplace")
        else:
            # gradients on bbox/obj/cls as well, or a second backward through the same graph (retain_graph=True:
            # the fused buffers were handed out, and possibly scaled in place, by the first one): recompute
            tensors = ctx.saved_tensors
            z = lambda g: 0.0 if g is None else float(g)
            gt_, gb_, go_, gc_ = z(g_total), z(g_bbox), z(g_obj), z(g_cls)
            coef = [(BOX_WEIGHT * gt_ + gb_, cfg.obj_weights[s] * gt_ + go_, CLS_WEIGHT * gt_ + gc_) for s in range(S)]
            _, _, grads = loss_forward_backward(tensors[:S], tensors[S:2 * S], tensors[2 * S:], cfg.nc, cfg.obj_weights,
                                                want, coef=coef, group=cfg.group, sparse=cfg.sparse, layout=cfg.layout)
        return (None,) + tuple(grads) + (None,) * (2 * S)


def _loss_common(predictions, targets, anchors_list, num_classes, obj_weights, group=None, sparse=None,
                 layout=LAYOUT_BHWAC):
    preds, tgts, ancs = _stage_heads(predictions, anchors_list, num_classes, layout,
                                     targets if sparse is None else sparse, detach=False)
    S, dev, orig_dev = len(preds), preds[0].device, predictions[0].device
    cfg = _LossCfg(int(num_classes), tuple(float(w) for w in obj_weights), group, sparse, layout, S)
    with torch.cuda.device(dev):
        outs = _YoloLossFn.apply(cfg, *preds, *(tgts or [None] * S), *ancs)
    if orig_dev != dev:
        outs = tuple(o.to(orig_dev) for o in outs)
    return outs


class PackedLabels:
    """Label lists of a batch on the device, the input of the sparse-target loss (SURVEY 8f-4):
    labels (B,max_gt,5) fp64 [class, xc, yc, w, h], n_gt (B) int32, letterbox (B,5) fp64
    [orig_w, orig_h, scale, pad_top, pad_left] (train.py:136-137), the dataset's img_size."""

    def __init__(self, labels, n_gt, letterbox, img_size):
        self.labels, self.n_gt, self.letterbox, self.img_size = labels, n_gt, letterbox, int(img_size)
        self.max_gt = int(labels.shape[1])
        self.status = torch.zeros(1, dtype=torch.int32, device=labels.device)

    def check(self):
        """Raise like the reference (IndexError, train.py:193-205) if a label mapped outside the grid."""
        if int(self.status.item()) != 0:
            raise IndexError("a label maps outside the grid or the class range (train.py:193-205)")


def pack_labels_host(labels: Sequence, img_size: int, letterbox: Optional[Sequence] = None, pin: bool = False,
                     max_gt: Optional[int] = None):
    """Host-side packing of per-image label arrays [(n_i,5)] into (labels (B,max_gt,5) f64, n_gt (B) i32,
    letterbox (B,5) f64) — 40 bytes per ground truth instead of three dense target tensors."""
    B = len(labels)
    rows = [torch.as_tensor(l, dtype=torch.float64).reshape(-1, 5) for l in labels]
    need = max([r.shape[0] for r in rows], default=0)
    if max_gt is None:
        max_gt = need
    elif max_gt < need:
        raise ValueError(f"max_gt={max_gt} < {need} labels in one image")
    lab = torch.zeros(B, max(max_gt, 1), 5, dtype=torch.float64)
    n_gt = torch.zeros(B, dtype=torch.int32)
    for i, r in enumerate(rows):
        lab[i, :r.shape[0]] = r
        n_gt[i] = r.shape[0]
    if letterbox is None:
        lb = torch.tensor([[img_size, img_size, 1.0, 0.0, 0.0]] * B, dtype=torch.float64).reshape(B, 5)
    else:
        lb = torch.as_tensor(np.asarray(letterbox, dtype=np.float64)).reshape(B, 5)
    if pin:
        lab, n_gt, lb = lab.pin_memory(), n_gt.pin_memory(), lb.pin_memory()
    return lab, n_gt, lb


def pack_labels(labels: Sequence, img_size: int, letterbox: Optional[Sequence] = None) -> PackedLabels:
    dev = _device()
    lab, n_gt, lb = pack_labels_host(labels, img_size, letterbox)
    return PackedLabels(lab.to(dev), n_gt.to(dev), lb.to(dev), img_size)


def yolo_loss_multiscale_labels(predictions, labels, anchors_list, num_classes=1, img_size=640, letterbox=None,
                                group=None, check=False):
    """yolo_loss_multiscale (train.py:840-886) fed by LABEL LISTS instead of dense targets: the
    assignment of YOLODataset.__getitem__ (:147-205) runs on the device and reaches the loss in
    sparse form.  `labels`: per-image (n_i,5) arrays, or a PackedLabels already on the device.
    Returns the same (total, sum bbox, sum obj, sum cls) as the dense call on the reference's targets.

    A label that maps outside the grid or the class range makes the reference (and `build_targets`) raise
    IndexError (train.py:193-205); here it is dropped on the device and recorded in `PackedLabels.status`.
    `check=True` reads that flag right after the call (one host synchronisation) and raises like the
    reference; asynchronous callers (CUDA graphs, pipelined loops) must call `PackedLabels.check()` at their
    own synchronisation point instead."""
    S = min(len(predictions), len(anchors_list), len(MULTISCALE_OBJ_WEIGHTS))
    packed = labels if isinstance(labels, PackedLabels) else pack_labels(labels, img_size, letterbox)
    out = _loss_common(list(predictions[:S]), [None] * S, list(anchors_list[:S]), num_classes,
                       MULTISCALE_OBJ_WEIGHTS[:S], group=group, sparse=packed)
    if check:
        packed.check()
    return out


def yolo_loss_multiscale_nchw(raw_heads, targets, anchors_list, num_classes=1, img_size=640, letterbox=None,
                              group=None, check=False):
    """yolo_loss_multiscale on the head convs' OWN outputs (B, A*(5+nc), H, W) — SURVEY 8f-2: the
    view/permute/contiguous of train.py:608-609 (a full read+write of every head, plus its backward)
    is not needed; the gradient comes back in the same NCHW layout, ready for the conv backward.
    `targets`: the reference's dense targets [(B,G,G,A,5+nc)], or label lists / PackedLabels (then
    the assignment runs on the device, as in yolo_loss_multiscale_labels)."""
    S = min(len(raw_heads), len(anchors_list), len(MULTISCALE_OBJ_WEIGHTS))
    is_packed = isinstance(targets, PackedLabels)
    dense = (not is_packed) and len(targets) > 0 and isinstance(targets[0], torch.Tensor) and targets[0].dim() == 5
    if not dense:
        packed = targets if is_packed else pack_labels(targets, img_size, letterbox)
        out = _loss_common(list(raw_heads[:S]), [None] * S, list(anchors_list[:S]), num_classes,
                           MULTISCALE_OBJ_WEIGHTS[:S], group=group, sparse=packed, layout=LAYOUT_NCHW)
        if check:
            packed.check()   # see yolo_loss_multiscale_labels
        return out
    S = min(S, len(targets))
    return _loss_common(list(raw_heads[:S]), list(targets[:S]), list(anchors_list[:S]), num_classes,
                        MULTISCALE_OBJ_WEIGHTS[:S], group=group, layout=LAYOUT_NCHW)


def yolo_loss(predictions, targets, anchors, num_classes=1):
    """train.py:781-838.  Returns (total, bbox, obj, cls) for one scale."""
    return _loss_common([predictions], [targets], [anchors], num_classes, (1.0,))


def yolo_loss_multiscale(predictions, targets, anchors_list, num_classes=1):
    """train.py:840-886.  Returns (total, sum bbox, sum obj (unweighted), sum cls)."""
    S = min(len(predictions), len(targets), len(anchors_list), len(MULTISCALE_OBJ_WEIGHTS))  # zip() semantics (:873)
    return _loss_common(list(predictions[:S]), list(targets[:S]), list(anchors_list[:S]), num_classes,
                        MULTISCALE_OBJ_WEIGHTS[:S])


# --------------------------------------------------------------------------------------------
# f-1 eval_epoch's detection counting
# --------------------------------------------------------------------------------------------
EVAL_DECODE_IMG_SIZE = 640.0  # train.py:993 — eval_epoch decodes with the default img_size


def eval_counts(predictions, targets, anchors_list, conf_threshold=0.5, iou_threshold=0.5, out=None):
    """The TP/FP/FN loop of eval_epoch (train.py:993-1024) for one batch, all scales, in one kernel.
    Returns an int64 device tensor [TP, FP, FN]; pass `out` to accumulate over batches (no sync)."""
    S = min(len(predictions), len(targets), len(anchors_list))
    preds, tgts, ancs = _stage_heads(predictions[:S], anchors_list[:S], None, LAYOUT_BHWAC, targets[:S], half=False)
    dev = preds[0].device
    with torch.cuda.device(dev):
        d = _heads_desc(HeadsDesc(), preds, ancs, preds[0].shape[4] - 5, EVAL_DECODE_IMG_SIZE, LAYOUT_BHWAC)
        if out is None:
            out = torch.zeros(3, dtype=torch.int64, device=dev)
        tptr = (ctypes.c_void_p * MAX_SCALES)(*[t.data_ptr() for t in tgts])
        _lib.check(_lib.lib().yb_eval_counts(ctypes.byref(d), tptr, float(conf_threshold), float(iou_threshold),
                                             out.data_ptr(), _stream()), "yb_eval_counts")
    return out


def eval_epoch(model, loader, device, num_classes=1, iou_threshold=0.5, conf_threshold=0.5):
    """Drop-in for train.eval_epoch (train.py:960-1032): same arguments, same four return values
    (avg_loss, precision %, recall %, F1 %).  The loss and the detection counting run on the GPU
    path; the counters stay on the device until the end of the epoch (one synchronisation instead of
    2 x rows `.item()` calls per batch)."""
    model.eval()
    anchors_list = model.anchors
    counts = None
    loss_sum = None
    n_batches = 0
    with torch.no_grad():
        for imgs, targets in loader:
            imgs = imgs.to(device)
            S = len(targets[0])
            targets_batch = [torch.stack([t[s] for t in targets]).to(device) for s in range(S)]  # :973-977
            preds = model(imgs)
            loss = yolo_loss_multiscale(preds, targets_batch, anchors_list, num_classes)[0]        # :987
            loss_sum = loss.detach().double().cuda() if loss_sum is None else loss_sum + loss.detach().double().cuda()
            counts = eval_counts(preds, targets_batch, anchors_list, conf_threshold, iou_threshold, out=counts)
            n_batches += 1
    tp, fp, fn = (0, 0, 0) if counts is None else [int(v) for v in counts.cpu().tolist()]
    precision = tp / (tp + fp) if (tp + fp) > 0 else 0                                            # :1026-1029
    recall = tp / (tp + fn) if (tp + fn) > 0 else 0
    f1 = 2 * precision * recall / (precision + recall) if (precision + recall) > 0 else 0
    avg_loss = (float(loss_sum) if loss_sum is not None else 0.0) / n_batches                      # :1031 (ZeroDivisionError on an empty loader, like the reference)
    return avg_loss, precision * 100, recall * 100, f1 * 100


# --------------------------------------------------------------------------------------------
# a-5 target assignment
# --------------------------------------------------------------------------------------------
def compute_anchor_iou(box_wh, anchors) -> torch.Tensor:
    """train.py:108-131.  box_wh (2,) or (n,2) pixels, anchors (A,2) -> (A,) or (n,A) IoU."""
    dev = _device()
    box_wh = torch.as_tensor(box_wh)
    orig_dev = box_wh.device
    single = box_wh.dim() == 1
    with torch.cuda.device(dev):
        b = _contig(box_wh.reshape(-1, 2), dev)
        a = _anchors_dev(anchors, dev)
        out = torch.empty(b.shape[0], a.shape[0], dtype=torch.float32, device=dev)
        _lib.check(_lib.lib().yb_anchor_iou(b.data_ptr(), a.data_ptr(), out.data_ptr(), b.shape[0], a.shape[0], _stream()),
                   "yb_anchor_iou")
    out = out[0] if single else out
    return out if orig_dev == dev else out.to(orig_dev)


def build_targets(labels: Sequence, anchors_list, grid_sizes: Sequence[int], num_classes: int, img_size: int,
                  letterbox: Optional[Sequence] = None, check: bool = True) -> List[torch.Tensor]:
    """Label loop of YOLODataset.__getitem__ (train.py:147-205) for a batch of images.

    labels: per image an (n_i, 5) array-like of raw label lines [class, xc, yc, w, h] (fp64)
    letterbox: per image (orig_w, orig_h, scale, pad_top, pad_left) as returned by the
               reference's letterbox_resize (:136-137); None = an img_size x img_size original.
    Returns dense targets [ (B,G,G,A,5+nc) fp32 on the GPU for each scale ].
    """
    dev = _device()
    B = len(labels)
    S = len(grid_sizes)
    with torch.cuda.device(dev):
        anc = torch.stack([_anchors_dev(a, dev) for a in anchors_list]).contiguous()  # (S,A,2)
        A = anc.shape[1]
        lab, n_gt, lb = pack_labels_host(labels, img_size, letterbox)
        max_gt = int(n_gt.max()) if B > 0 else 0   # the kernel's bound: the largest label count, read on the host
        packed = PackedLabels(lab.to(dev), n_gt.to(dev), lb.to(dev), img_size)
        row = 5 + num_classes
        targets = [torch.empty(B, g, g, A, row, dtype=torch.float32, device=dev) for g in grid_sizes]
        tptr = (ctypes.c_void_p * MAX_SCALES)(*[t.data_ptr() for t in targets])
        G = (ctypes.c_int * S)(*[int(g) for g in grid_sizes])
        _lib.check(_lib.lib().yb_build_targets(packed.labels.data_ptr(), packed.n_gt.data_ptr(),
                                               packed.letterbox.data_ptr(), anc.data_ptr(), tptr, B, max_gt, S, G, A,
                                               int(num_classes), int(img_size), packed.status.data_ptr(), _stream()),
                   "yb_build_targets")
        if check and int(packed.status.item()) != 0:
            raise IndexError("build_targets: a label maps outside the grid or the class range "
                             "(the reference raises IndexError on the same input, train.py:193-205)")
    return targets


# --------------------------------------------------------------------------------------------
# a-6 candidate filter, a-7 NMS
# --------------------------------------------------------------------------------------------
def _letterbox_dev(letterbox, B, dev):
    if letterbox is None:
        return None
    return torch.as_tensor(letterbox, dtype=torch.float32).reshape(B, 3).to(dev).contiguous()


def filter_candidates(predictions, anchors_list, img_size, num_classes=1, conf_threshold=0.5, letterbox=None,
                      layout=LAYOUT_BHWAC):
    """Per-scale body of predict() (train.py:1152-1229) for a batch: decode, sigmoid, objectness
    filter, class max, pixel xyxy with letterbox reverse, score; P3->P4->P5 order preserved.
    bf16 / fp16 heads are read natively; the candidates are those of the fp32 filter on the upcast heads.

    letterbox: (B,3) [scale, pad_top, pad_left] or None.
    Returns (boxes (B,cap,4), scores (B,cap), classes (B,cap) int64, counts (B,) int32) on the GPU,
    cap = rows per image.
    """
    preds, _, ancs = _stage_heads(predictions, anchors_list, num_classes, layout)
    dev = preds[0].device
    with torch.cuda.device(dev):
        B = preds[0].shape[0]
        d = _heads_desc(HeadsDesc(), preds, ancs, int(num_classes), img_size, layout)
        cap = d.A * sum(d.H[s] * d.W[s] for s in range(d.S))   # rows per image
        L = _lib.lib()
        ws_bytes = L.yb_filter_workspace_bytes(ctypes.byref(d))
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        boxes = torch.empty(B, cap, 4, dtype=torch.float32, device=dev)
        scores = torch.empty(B, cap, dtype=torch.float32, device=dev)
        classes = torch.empty(B, cap, dtype=torch.int64, device=dev)
        counts = (torch.empty if B > 0 else torch.zeros)(B, dtype=torch.int32, device=dev)   # every image's count is written by the kernel
        lb = _letterbox_dev(letterbox, B, dev)
        _lib.check(L.yb_filter_compact(ctypes.byref(d), float(conf_threshold), _ptr(lb), boxes.data_ptr(),
                                       scores.data_ptr(), classes.data_ptr(), counts.data_ptr(), cap,
                                       ws.data_ptr(), ws.numel(), _stream()), "yb_filter_compact")
    return boxes, scores, classes, counts


MAX_CANDIDATES = 30000   # max_nms of YOLO validation tools: candidates per image kept before NMS


def filter_candidates_multilabel(predictions, anchors_list, img_size, num_classes=1, conf_threshold=0.001,
                                 letterbox=None, layout=LAYOUT_BHWAC, max_candidates=MAX_CANDIDATES):
    """Multi-label candidates of a batch (include/yolo_b200.h, yb_filter_multilabel): every (row, class) pair with
    sigmoid(obj) > conf and score = sigmoid(obj) * sigmoid(cls_c) > conf, in (row, class) order, each with the box
    filter_candidates gives its row.  An image with more than max_candidates keeps the best max_candidates by (score
    descending, candidate order), still in candidate order.  Inputs, layouts and dtypes as filter_candidates.

    Returns (boxes (B,cap,4), scores (B,cap), classes (B,cap) int64, counts (B,) int32, totals (B,) int32) on the GPU:
    cap = min(max_candidates, rows * nc), counts = kept candidates, totals = candidates before the cap.  Nothing is
    synchronised; the call is capturable in a CUDA graph.
    """
    K = int(max_candidates)
    if K < 1:
        raise ValueError(f"max_candidates must be >= 1, got {max_candidates}")
    preds, _, ancs = _stage_heads(predictions, anchors_list, num_classes, layout)
    dev = preds[0].device
    with torch.cuda.device(dev):
        B = preds[0].shape[0]
        d = _heads_desc(HeadsDesc(), preds, ancs, int(num_classes), img_size, layout)
        cap = min(K, d.A * sum(d.H[s] * d.W[s] for s in range(d.S)) * int(num_classes))
        L = _lib.lib()
        ws = torch.empty(max(L.yb_filter_multilabel_workspace_bytes(ctypes.byref(d), K), 16), dtype=torch.uint8,
                         device=dev)
        boxes = torch.empty(B, cap, 4, dtype=torch.float32, device=dev)
        scores = torch.empty(B, cap, dtype=torch.float32, device=dev)
        classes = torch.empty(B, cap, dtype=torch.int64, device=dev)
        counts = (torch.empty if B > 0 else torch.zeros)(B, dtype=torch.int32, device=dev)
        totals = (torch.empty if B > 0 else torch.zeros)(B, dtype=torch.int32, device=dev)
        lb = _letterbox_dev(letterbox, B, dev)
        _lib.check(L.yb_filter_multilabel(ctypes.byref(d), float(conf_threshold), _ptr(lb), K, boxes.data_ptr(),
                                          scores.data_ptr(), classes.data_ptr(), counts.data_ptr(), totals.data_ptr(),
                                          cap, ws.data_ptr(), ws.numel(), _stream()), "yb_filter_multilabel")
    return boxes, scores, classes, counts, totals


NMS_GRAPH, NMS_BITMASK = _lib.NMS_GRAPH, _lib.NMS_BITMASK
GRAPH_EDGES_PER_BOX = 16  # edge-list capacity of the default workspace (dense random heads need ~3)


def batched_nms_padded(boxes, scores, classes, counts, iou_threshold, trick_max_numel=TRICK_MAX_NUMEL_CUDA,
                       algo=NMS_GRAPH, return_workspace=False):
    """NMS for B images at once.  boxes (B,cap,4), scores (B,cap), classes (B,cap) int64 or None,
    counts (B,) int32 or None.  Returns (keep (B,cap) int64, n_keep (B,) int32) on the GPU, nothing
    synchronised.  The default sparse-graph algorithm resolves an image whose suppression graph does
    not fit the workspace on the device, in the same launch (blocked greedy pass), so n_keep is never
    negative; only the dense bitmask algorithm with an undersized workspace can report n_keep = -1,
    which `pack_detections` turns into a total of -1 and `detections_to_lists` into an exception."""
    dev = boxes.device
    B, cap = boxes.shape[0], boxes.shape[1]
    L = _lib.lib()
    keep = torch.empty(B, cap, dtype=torch.int64, device=dev)
    if B == 0 or cap == 0:
        z = torch.zeros(B, dtype=torch.int32, device=dev)
        return (keep, z, None) if return_workspace else (keep, z)
    n_keep = torch.empty(B, dtype=torch.int32, device=dev)   # written for every image (no fill kernel on the critical path)
    need = (L.yb_nms_graph_workspace_bytes(B, cap, GRAPH_EDGES_PER_BOX) if algo == NMS_GRAPH
            else L.yb_nms_workspace_bytes(B, cap))
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    _lib.check(L.yb_batched_nms(boxes.data_ptr(), scores.data_ptr(), _ptr(classes), _ptr(counts), B, cap,
                                float(iou_threshold), int(trick_max_numel), int(algo), keep.data_ptr(),
                                n_keep.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "yb_batched_nms")
    if return_workspace:
        return keep, n_keep, ws
    return keep, n_keep


def nms_graph_stats(det):
    """(pair tests executed by the half-precision filter, edges, pairs decided exactly in fp32) of the graph NMS
    behind a `detect_batch` result, summed over the batch; None for the bitmask algorithm.  Synchronises.
    For bench.py / tests."""
    ws = det.get("nms_ws")
    if ws is None or det.get("algo", NMS_GRAPH) != NMS_GRAPH:
        return None
    B, cap = det["boxes"].shape[0], det["boxes"].shape[1]
    ev, ed, ca = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
    with torch.cuda.device(ws.device):
        _lib.check(_lib.lib().yb_nms_graph_stats(ws.data_ptr(), ws.numel(), B, cap, ctypes.byref(ev), ctypes.byref(ed),
                                                 ctypes.byref(ca), _stream()), "yb_nms_graph_stats")
    return int(ev.value), int(ed.value), int(ca.value)


def nms_retry_overflow(boxes, scores, classes, counts, iou_threshold, trick_max_numel, keep, n_keep):
    """Re-run, with the dense bitmask algorithm, the images the graph algorithm gave up on
    (n_keep == -1).  Synchronises (reads n_keep).  Returns (keep, n_keep), updated in place."""
    bad = (n_keep < 0).nonzero().flatten()
    if bad.numel() == 0:
        return keep, n_keep
    sel = lambda t: None if t is None else t.index_select(0, bad).contiguous()
    k2, n2 = batched_nms_padded(sel(boxes), sel(scores), sel(classes), sel(counts), iou_threshold, trick_max_numel,
                                algo=NMS_BITMASK)
    if bool((n2 < 0).any()):
        raise ValueError("batched_nms: class ids must be in [0, 65536)")
    keep.index_copy_(0, bad, k2)
    n_keep.index_copy_(0, bad, n2)
    return keep, n_keep


def _nms_single(boxes, scores, idxs, iou_threshold, algo=NMS_GRAPH):
    if boxes.dim() != 2 or boxes.shape[1] != 4:
        raise ValueError("boxes must be (N,4)")
    dev = _device()
    orig_dev = boxes.device
    n = boxes.shape[0]
    if n == 0:
        return torch.empty(0, dtype=torch.int64, device=orig_dev)
    with torch.cuda.device(dev):
        b = _contig(boxes.detach(), dev).unsqueeze(0)
        s = _contig(scores.detach(), dev).unsqueeze(0)
        c = None
        if idxs is not None:
            c = idxs.detach().to(dev, torch.int64).contiguous().unsqueeze(0)
        # torchvision picks its algorithm from the caller's device (boxes.py:80)
        trick = TRICK_MAX_NUMEL_CPU if orig_dev.type == "cpu" else TRICK_MAX_NUMEL_CUDA
        keep, n_keep = batched_nms_padded(b, s, c, None, iou_threshold, trick, algo)
        k = int(n_keep[0].item())
        if k < 0:
            keep, n_keep = nms_retry_overflow(b, s, c, None, iou_threshold, trick, keep, n_keep)
            k = int(n_keep[0].item())
        out = keep[0, :k].clone()
    return out if orig_dev == dev else out.to(orig_dev)


def batched_nms(boxes, scores, idxs, iou_threshold, algo=NMS_GRAPH):
    """Drop-in for torchvision.ops.batched_nms (train.py:1232-1233): int64 indices of the kept
    boxes in descending score order."""
    return _nms_single(boxes, scores, idxs, iou_threshold, algo)


def nms(boxes, scores, iou_threshold, algo=NMS_GRAPH):
    """Drop-in for torchvision.ops.nms."""
    return _nms_single(boxes, scores, None, iou_threshold, algo)


def detect_batch(predictions, anchors_list, img_size, num_classes=1, conf_threshold=0.5, iou_threshold=0.4,
                 letterbox=None, trick_max_numel=TRICK_MAX_NUMEL_CUDA, algo=NMS_GRAPH, layout=LAYOUT_BHWAC, *,
                 multi_label=False, max_candidates=None, agnostic=False, max_det=None):
    """predict() lines 1152-1238 for a whole batch on the GPU: decode + filter + global NMS.

    Returns a dict of device tensors: boxes (B,cap,4), scores, classes, counts (candidates per
    image), keep (B,cap) indices into the candidates in descending score order, n_keep (B,).
    Nothing is synchronised; use `detections_to_lists` for the reference's list-of-tuples form.

    multi_label=True takes the candidates of filter_candidates_multilabel (one per (row, class) pair that passes
    conf; at most max_candidates per image, None = MAX_CANDIDATES) and adds "totals", the candidates before the cap.
    The default single-label filter is bounded by the rows and takes no max_candidates.  agnostic and max_det are
    nms_candidates'.  The dict records the options.
    """
    if multi_label:
        K = MAX_CANDIDATES if max_candidates is None else int(max_candidates)
        boxes, scores, classes, counts, totals = filter_candidates_multilabel(
            predictions, anchors_list, img_size, num_classes, conf_threshold, letterbox, layout, K)
    else:
        if max_candidates is not None:
            raise ValueError("max_candidates applies to multi_label=True only: the single-label filter keeps at most "
                             "one candidate per row")
        boxes, scores, classes, counts = filter_candidates(predictions, anchors_list, img_size, num_classes,
                                                           conf_threshold, letterbox, layout)
    det = nms_candidates(boxes, scores, classes, counts, iou_threshold, trick_max_numel, algo, agnostic=agnostic,
                         max_det=max_det)
    det["multi_label"] = bool(multi_label)
    if multi_label:
        det["totals"] = totals
        det["max_candidates"] = K
    return det


def nms_candidates(boxes, scores, classes, counts, iou_threshold=0.4, trick_max_numel=TRICK_MAX_NUMEL_CUDA, algo=NMS_GRAPH,
                   *, agnostic=False, max_det=None):
    """Second half of detect_batch: global NMS (train.py:1232-1233) over the padded candidates of filter_candidates.
    agnostic=True suppresses across classes (torchvision.ops.nms on the candidates; the detections keep their
    classes).  max_det keeps the first max_det detections of every image (n_keep = min(n_keep, max_det), torchvision's
    keep[:max_det]; a failed image's -1 stays -1)."""
    if max_det is not None and int(max_det) < 0:
        raise ValueError(f"max_det must be >= 0, got {max_det}")
    with torch.cuda.device(boxes.device):
        keep, n_keep, ws = batched_nms_padded(boxes, scores, None if agnostic else classes, counts, iou_threshold,
                                              trick_max_numel, algo, return_workspace=True)
        if max_det is not None:
            n_keep = n_keep.clamp(max=int(max_det))
    return {"boxes": boxes, "scores": scores, "classes": classes, "counts": counts, "keep": keep, "n_keep": n_keep,
            "iou_threshold": float(iou_threshold), "trick_max_numel": int(trick_max_numel), "algo": algo, "nms_ws": ws,
            "agnostic": bool(agnostic), "max_det": None if max_det is None else int(max_det)}


def detect_batch_nchw(raw_heads, anchors_list, img_size, num_classes=1, conf_threshold=0.5, iou_threshold=0.4,
                      letterbox=None, trick_max_numel=TRICK_MAX_NUMEL_CUDA, algo=NMS_GRAPH, *, multi_label=False,
                      max_candidates=None, agnostic=False, max_det=None):
    """detect_batch on the head convs' own outputs (B, A*(5+nc), H, W) (SURVEY 8f-2); same candidates,
    same order, same keep sets as detect_batch on the permuted heads."""
    return detect_batch(raw_heads, anchors_list, img_size, num_classes, conf_threshold, iou_threshold, letterbox,
                        trick_max_numel, algo, layout=LAYOUT_NCHW, multi_label=multi_label,
                        max_candidates=max_candidates, agnostic=agnostic, max_det=max_det)


def pack_detections(det):
    """Device-side detection list: (rows (B*cap,6) fp32 [x1,y1,x2,y2,conf,class], offsets (B+1,) int32).
    Only the first offsets[B] rows are meaningful."""
    boxes, keep = det["boxes"], det["keep"]
    B, cap = boxes.shape[0], boxes.shape[1]
    with torch.cuda.device(boxes.device):
        rows = torch.empty(B * cap, 6, dtype=torch.float32, device=boxes.device)
        offsets = (torch.empty if B > 0 and cap > 0 else torch.zeros)(B + 1, dtype=torch.int32, device=boxes.device)
        _lib.check(_lib.lib().yb_pack_detections(boxes.data_ptr(), det["scores"].data_ptr(), det["classes"].data_ptr(),
                                                 keep.data_ptr(), det["n_keep"].data_ptr(), B, cap, rows.data_ptr(),
                                                 offsets.data_ptr(), _stream()), "yb_pack_detections")
    return rows, offsets


def detections_to_lists(det):
    """[(x1, y1, x2, y2, conf, class_id), ...] per image (train.py:1242-1246): one pack kernel and
    two D2H copies instead of K*6 `.item()` syncs."""
    rows, offsets = pack_detections(det)
    off = offsets.cpu().tolist()
    if off[-1] < 0:
        raise RuntimeError("NMS failed for an image (n_keep < 0: bitmask algorithm with too small a workspace)")
    host = rows[:off[-1]].cpu().tolist()
    return [[(r[0], r[1], r[2], r[3], r[4], int(r[5])) for r in host[off[b]:off[b + 1]]] for b in range(len(off) - 1)]


def predict_heads(preds, anchors_list, img_size, num_classes=1, conf_threshold=0.5, iou_threshold=0.4, letterbox=None):
    """Everything predict() does after the model call (train.py:1140-1246), for a batch of B images: decode,
    objectness filter, class max, pixel xyxy, letterbox reverse, global NMS, detection list.  preds are the
    model's heads [(B,G,G,A,5+nc)], letterbox per image (scale, pad_top, pad_left) as returned by the
    reference's letterbox_resize.  Returns, per image, [(x1, y1, x2, y2, conf, class_id), ...] in original
    image coordinates, descending score — the reference's return value, one host synchronisation per batch
    instead of a `nonzero` per scale (:1170) and K x 6 `.item()` calls (:1242-1246) per image."""
    # torchvision picks batched_nms' algorithm from the device its inputs live on (boxes.py:80); in
    # predict() that is the device the model ran on
    on_cpu = preds[0].device.type == "cpu"
    det = detect_batch(list(preds), anchors_list, img_size, num_classes, conf_threshold, iou_threshold, letterbox=letterbox,
                       trick_max_numel=TRICK_MAX_NUMEL_CPU if on_cpu else TRICK_MAX_NUMEL_CUDA)
    return detections_to_lists(det)


# --------------------------------------------------------------------------------------------
# COCO-style mAP (no reference equivalent: the reference's eval_epoch reports precision/recall only)
# --------------------------------------------------------------------------------------------
COCO_IOU_THRESHOLDS = tuple(np.linspace(0.5, 0.95, 10).tolist())      # COCOeval Params.iouThrs
COCO_RECALL_THRESHOLDS = tuple(np.linspace(0.0, 1.0, 101).tolist())   # COCOeval Params.recThrs


def _sort_records(rec, nc):
    """Records (N, words) int32 whose first two words are (score f32, class i32) -> (records sorted by class
    ascending, then score descending, stably; seg (nc+1) int64: class c is rows [seg[c], seg[c+1])).  Unused slots
    (class -1) go last."""
    # key = class << 32 | order-reversed score bits: ascending key = class ascending, score descending;
    # the stable sort keeps image and keep order among equal keys.
    score = rec[:, 0].view(torch.float32) + 0.0          # -0.0 -> +0.0: equal scores must tie
    bits = score.view(torch.int32).to(torch.int64)
    asc = bits ^ ((bits >> 31) & 0x7FFFFFFF)              # monotone in the float value
    cls = rec[:, 1].to(torch.int64)
    key = torch.where(cls >= 0, cls, nc) * (1 << 32) + (0x7FFFFFFF - asc)
    key, order = torch.sort(key, stable=True)
    rec = rec.index_select(0, order).contiguous()
    seg = torch.searchsorted(key, torch.arange(nc + 1, dtype=torch.int64, device=rec.device) * (1 << 32))
    return rec, seg


def _eval_fingerprint(kind, nc, T, R, A, M, K, max_det, arrays):
    """The configuration words compute(group) requires to be equal on every rank (dist.FINGERPRINT_FIELDS; kind 1
    DetectionMAP, 2 COCODetectionEval, 3 DetectionReport): the sizes, and one CRC-32 over the float64 bytes of every
    threshold, grid, area range and limit."""
    crc = 0
    for a in arrays:
        crc = zlib.crc32(np.ascontiguousarray(a, dtype=np.float64).tobytes(), crc)
    return kind, nc, T, R, A, M, K, max_det, crc


def _raise_status(status, who):
    """The errors of the mAP kernels' status bits (YB_MAP_*)."""
    if status & _lib.MAP_BAD_CLASS:
        raise IndexError(f"{who}: a ground-truth or detection class id is outside [0, num_classes)")
    if status & _lib.MAP_NMS_FAILED:
        raise RuntimeError(f"{who}: NMS failed for an image (n_keep < 0: bitmask algorithm with too small a "
                           "workspace)")
    if status & _lib.MAP_INCONSISTENT:
        raise RuntimeError(f"{who}: a class has more true positives than ground truths")


def _unpack(host, shapes):
    """The consecutive pieces of the flat array `host` with the given shapes, as views."""
    out, o = [], 0
    for shape in shapes:
        n = math.prod(shape)
        out.append(host[o:o + n].reshape(shape))
        o += n
    return out


def _mean_valid(s):
    """The mean of the entries > -1, -1 when there are none (COCOeval.summarize)."""
    s = s[s > -1]
    return float(np.mean(s)) if s.size else -1.0


def _compute_metric(metric, group):
    """compute(group) of the three metrics: _local_state(), merged over `group` by dist.gather_eval_state, goes
    through _compute_device into flat float64 device tensors, which _copy_back copies to the host with the status
    word appended (the one synchronisation, the second with a group); _compute_host reads their _host_shapes()."""
    with torch.cuda.device(metric.device):
        state = metric._local_state()
        if group is not None:
            from .dist import gather_eval_state
            state = gather_eval_state(metric._fingerprint(), *state, group)
        host = metric._copy_back(metric._compute_device(state) + [state[-1].double()])
    _raise_status(int(host[-1]), type(metric).__name__)
    return metric._compute_host(_unpack(host, metric._host_shapes()), state)


class _MatchMetric:
    """What DetectionMAP and COCODetectionEval share: the common arguments, update() and the state compute(group)
    starts from.  A subclass sets _RECORD_WORDS, creates _gt_count and provides _match and the hooks of
    _compute_metric.  DetectionReport drives its DetectionMAP through update(), _match_prefix, the hooks and _status,
    the device word every kernel of the metric ORs its YB_MAP_* bits into."""

    def __init__(self, num_classes, iou_thresholds, recall_thresholds, max_det):
        self.nc = int(num_classes)
        self.iou_thresholds = np.asarray(iou_thresholds, dtype=np.float64).reshape(-1)
        self.recall_thresholds = np.asarray(recall_thresholds, dtype=np.float64).reshape(-1)
        self.max_det = int(max_det)
        if self.nc < 1:
            raise ValueError("num_classes must be >= 1")
        if not 1 <= len(self.iou_thresholds) <= _lib.MAP_MAX_T:
            raise ValueError(f"1..{_lib.MAP_MAX_T} IoU thresholds supported, got {len(self.iou_thresholds)}")
        if len(self.recall_thresholds) < 1:
            raise ValueError("at least one recall threshold is needed")
        if self.max_det < 0:
            raise ValueError("max_det must be >= 0")
        self.device = _device()
        with torch.cuda.device(self.device):
            self._iou_thr = torch.tensor(self.iou_thresholds, dtype=torch.float64, device=self.device)
            self._rec_thr = torch.tensor(self.recall_thresholds, dtype=torch.float64, device=self.device)
            self._status = torch.zeros(1, dtype=torch.int32, device=self.device)

    def reset(self):
        """Forget every batch seen so far."""
        self._records = []
        self._gt_total = 0   # upper bound on the ground truths seen: sum of B * max_gt (sizes DetectionMAP's workspace)
        with torch.cuda.device(self.device):
            self._gt_count.zero_()
            self._status.zero_()

    def update(self, det, labels: PackedLabels):
        """Match one batch: `det` is a detect_batch result (letterbox reversed, original-image pixels) and `labels`
        the batch's PackedLabels (labels normalised to the original image, letterbox rows [orig_w, orig_h, ...]).
        Returns the batch's records on the device."""
        B, cap = self._check_batch(det, labels)
        with torch.cuda.device(self.device):
            rec = torch.empty(B * min(self.max_det, cap), self._RECORD_WORDS, dtype=torch.int32, device=self.device)
            self._match(self._match_prefix(det, labels), rec)
        self._records.append(rec)
        self._gt_total += B * labels.max_gt
        return rec

    def _check_batch(self, det, labels):
        """update()'s checks of one batch; returns (B, cap)."""
        boxes = det["boxes"]
        if boxes.device != self.device:
            raise ValueError(f"detections on {boxes.device}, {type(self).__name__} on {self.device}")
        B, cap = boxes.shape[0], boxes.shape[1]
        if labels.labels.shape[0] != B or labels.labels.device != self.device:
            raise ValueError("labels and detections disagree on the batch size or the device")
        if labels.max_gt > _lib.MAP_MAX_GT:
            raise ValueError(f"at most {_lib.MAP_MAX_GT} ground truths per image, got max_gt={labels.max_gt}")
        return B, cap

    def _match_prefix(self, det, labels):
        """The arguments every yb_*_match entry point starts with: the batch's candidates and kept lists, max_det, its
        labels and num_classes."""
        B, cap = det["boxes"].shape[0], det["boxes"].shape[1]
        return (det["boxes"].data_ptr(), det["scores"].data_ptr(), det["classes"].data_ptr(), det["keep"].data_ptr(),
                det["n_keep"].data_ptr(), B, cap, self.max_det, labels.labels.data_ptr(), labels.n_gt.data_ptr(),
                labels.letterbox.data_ptr(), labels.max_gt, self.nc)

    def _local_state(self):
        """(records in image order, gt_count, gt_total, images_total, status) of this process."""
        rec = (torch.cat(self._records) if self._records
               else torch.empty(0, self._RECORD_WORDS, dtype=torch.int32, device=self.device))
        return rec, self._gt_count, self._gt_total, 0, self._status

    def _copy_back(self, tensors):
        return torch.cat(tensors).cpu().numpy()


class DetectionMAP(_MatchMetric):
    """mAP@[.5:.95] and mAP@0.5 of the kept detections of `detect_batch`, accumulated over batches on the device.
    COCO's bbox protocol (evaluateImg + accumulate, area range "all", no crowd) with one overall cap of `max_det`
    detections per image instead of COCO's per-category maxDets; include/yolo_b200.h states the semantics.

    update(det, labels) enqueues one matching kernel per batch and keeps its records; it never synchronises.
    compute() sorts the records once, runs the precision kernel and synchronises once.

    compute(group) evaluates an image-sharded run: a collective over the torch.distributed process group `group`
    (every rank calls it) that returns on every rank the dict one process would return after update() with every
    rank's batches in rank order (DESIGN §3.11).  It synchronises twice and leaves the local state unchanged.  The
    result is bit-identical to that process when rank r updated the r-th contiguous block of images
    (dist.shard_range) in image order.  With any other assignment, such as DistributedSampler's interleaving,
    n_gt, n_det and recall are still identical, and the precision table (with the AP values taken from it) can
    differ only through the order of equal-score detections of different images."""
    _RECORD_WORDS = 3   # yb_map_record: score, class, tp

    def __init__(self, num_classes, iou_thresholds=COCO_IOU_THRESHOLDS, recall_thresholds=COCO_RECALL_THRESHOLDS,
                 max_det=300):
        super().__init__(num_classes, iou_thresholds, recall_thresholds, max_det)
        with torch.cuda.device(self.device):
            self._gt_count = torch.zeros(self.nc, dtype=torch.int64, device=self.device)
        self.reset()

    def _match(self, prefix, rec):
        _lib.check(_lib.lib().yb_map_match(*prefix, self._iou_thr.data_ptr(), len(self.iou_thresholds), rec.data_ptr(),
                                           self._gt_count.data_ptr(), self._status.data_ptr(), _stream()),
                   "yb_map_match")

    def compute(self, group=None):
        """{map, map50, ap (nc,T), precision (T,R,nc), recall (T,nc), n_gt (nc), n_det (nc)} on the host (float64 /
        int64; map50 is None when 0.5 is not a threshold).  Entries of a class without ground truth are -1, and
        map / map50 are the means of the entries > -1 (-1 when there are none), as COCOeval.summarize.
        group: a torch.distributed process group to merge over (see the class docstring)."""
        return _compute_metric(self, group)

    def _fingerprint(self):
        return _eval_fingerprint(1, self.nc, len(self.iou_thresholds), len(self.recall_thresholds), 0, 0, 0,
                                 self.max_det, (self.iou_thresholds, self.recall_thresholds))

    def _compute_device(self, state):
        """Sort the records and run the precision kernel: precision, recall, gt_count and seg as flat float64."""
        rec, gt_count, gt_total, _, status = state
        T, R, nc = len(self.iou_thresholds), len(self.recall_thresholds), self.nc
        dev = self.device
        rec, seg = _sort_records(rec, nc)
        n = rec.shape[0]
        ws_bytes = _lib.lib().yb_map_workspace_bytes(n, gt_total, T)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        precision = torch.empty(T, R, nc, dtype=torch.float64, device=dev)
        recall = torch.empty(T, nc, dtype=torch.float64, device=dev)
        _lib.check(_lib.lib().yb_map_precision(rec.data_ptr(), seg.data_ptr(), gt_count.data_ptr(), nc, T,
                                               self._rec_thr.data_ptr(), R, precision.data_ptr(), recall.data_ptr(),
                                               ws.data_ptr(), ws_bytes, status.data_ptr(), _stream()),
                   "yb_map_precision")
        return [precision.reshape(-1), recall.reshape(-1), gt_count.double(), seg.double()]

    def _host_shapes(self):
        T, R, nc = len(self.iou_thresholds), len(self.recall_thresholds), self.nc
        return [(T, R, nc), (T, nc), (nc,), (nc + 1,)]

    def _compute_host(self, parts, state):
        precision, recall, n_gt, seg = parts[:4]
        return dict(summarize_precision(precision, self.iou_thresholds), precision=precision, recall=recall,
                    n_gt=n_gt.astype(np.int64), n_det=np.diff(seg).astype(np.int64))


def summarize_precision(precision, iou_thresholds):
    """map, map50 and ap (nc,T) from a (T,R,nc) precision table, as COCOeval.summarize averages it."""
    hit = np.flatnonzero(np.asarray(iou_thresholds) == 0.5)
    ap = np.where(precision.min(axis=1) > -1, precision.mean(axis=1), -1.0).T   # (nc,T)
    return {"map": _mean_valid(precision), "map50": _mean_valid(precision[hit]) if hit.size else None, "ap": ap}


COCO_AREA_RANGES = ((0.0, 1e5 ** 2), (0.0, 32.0 ** 2), (32.0 ** 2, 96.0 ** 2), (96.0 ** 2, 1e5 ** 2))   # Params.areaRng
COCO_AREA_LABELS = ("all", "small", "medium", "large")                                                # Params.areaRngLbl
COCO_MAX_DETS = (1, 10, 100)                                                                          # Params.maxDets


class COCODetectionEval(_MatchMetric):
    """COCO's bbox summary of the kept detections of `detect_batch`, accumulated over batches on the device: the
    twelve numbers pycocotools prints (AP, AP50, AP75, AP_S/M/L, AR@maxDets, AR_S/M/L) and COCOeval.eval's
    precision (T,R,nc,A,M) and recall (T,nc,A,M) tables.  COCO's protocol (evaluateImg + accumulate + summarize,
    area ranges all/small/medium/large, per-(image, category) maxDets, no crowd) on the first `max_det` kept
    detections of each image; include/yolo_b200.h states the semantics.  A NaN IoU never matches, where
    pycocotools' `iou < best` test would let it through.

    max_det caps the detections of an image (the records kept per image, YOLOv5's NMS cap); max_dets are COCO's
    three per-(image, category) limits.  stats[0] (AP) reads maxDets = 100 literally, as pycocotools does, so it is
    -1 when max_dets lacks 100; every other stat uses max_dets[0..2].

    update(det, labels) enqueues one matching kernel per batch and keeps its records; it never synchronises.
    compute() sorts the records once, runs the precision kernel and synchronises once.

    compute(group) evaluates an image-sharded run as DetectionMAP.compute(group) does: a collective over `group` that
    returns on every rank the dict of one process that saw every rank's batches in rank order, bit-identical when
    rank r updated the r-th contiguous block of images in image order.  With any other assignment n_gt, n_det and
    recall are still identical, and precision (with the stats and AP values taken from it) can differ only through
    the order of equal-score detections of different images."""
    _RECORD_WORDS = 8   # yb_coco_record, 32 bytes

    def __init__(self, num_classes, iou_thresholds=COCO_IOU_THRESHOLDS, recall_thresholds=COCO_RECALL_THRESHOLDS,
                 max_det=300, max_dets=COCO_MAX_DETS):
        super().__init__(num_classes, iou_thresholds, recall_thresholds, max_det)
        self.max_dets = tuple(int(m) for m in max_dets)
        self.area_ranges = np.asarray(COCO_AREA_RANGES, dtype=np.float64)
        if not np.all(np.diff(self.recall_thresholds) >= 0):
            raise ValueError("recall_thresholds must be a non-empty ascending sequence")
        if len(self.max_dets) != 3 or not all(1 <= m <= 65535 for m in self.max_dets):
            raise ValueError(f"max_dets must be three values in [1, 65535], got {max_dets}")
        with torch.cuda.device(self.device):
            self._gt_count = torch.zeros(len(self.area_ranges), self.nc, dtype=torch.int64, device=self.device)
        self._rng_host = (ctypes.c_double * self.area_ranges.size)(*self.area_ranges.reshape(-1).tolist())
        self._md_host = (ctypes.c_int * len(self.max_dets))(*self.max_dets)
        self.reset()

    def _match(self, prefix, rec):
        _lib.check(_lib.lib().yb_coco_match(*prefix, self._iou_thr.data_ptr(), len(self.iou_thresholds),
                                            self._rng_host, len(self.area_ranges), rec.data_ptr(),
                                            self._gt_count.data_ptr(), self._status.data_ptr(), _stream()),
                   "yb_coco_match")

    def compute(self, group=None):
        """{stats (12,), precision (T,R,nc,A,M), recall (T,nc,A,M), n_gt (nc,A), n_det (nc), and ap (nc,T), map,
        map50 at area "all" and max_dets[-1]} on the host (float64 / int64).  Entries of a (class, area) without
        ground truth are -1; stats are pycocotools' _summarizeDets, map / map50 DetectionMAP's means.  n_gt counts
        the ground truths inside each area range, n_det the records of each class (at most max_det per image).
        group: a torch.distributed process group to merge over (see the class docstring)."""
        return _compute_metric(self, group)

    def _fingerprint(self):
        return _eval_fingerprint(2, self.nc, len(self.iou_thresholds), len(self.recall_thresholds),
                                 len(self.area_ranges), len(self.max_dets), 0, self.max_det,
                                 (self.iou_thresholds, self.recall_thresholds, self.area_ranges, self.max_dets))

    def _compute_device(self, state):
        """Sort the records and run the precision kernel: precision, recall, gt_count and seg as flat float64."""
        rec, gt_count, _, _, status = state
        T, R, nc, dev = len(self.iou_thresholds), len(self.recall_thresholds), self.nc, self.device
        A, M = len(self.area_ranges), len(self.max_dets)
        rec, seg = _sort_records(rec, nc)
        precision = torch.empty(T, R, nc, A, M, dtype=torch.float64, device=dev)
        recall = torch.empty(T, nc, A, M, dtype=torch.float64, device=dev)
        _lib.check(_lib.lib().yb_coco_precision(rec.data_ptr(), seg.data_ptr(), gt_count.data_ptr(), nc, A, T,
                                                self._rec_thr.data_ptr(), R, self._md_host, M, precision.data_ptr(),
                                                recall.data_ptr(), status.data_ptr(), _stream()),
                   "yb_coco_precision")
        return [precision.reshape(-1), recall.reshape(-1), gt_count.reshape(-1).double(), seg.double()]

    def _host_shapes(self):
        T, R, nc = len(self.iou_thresholds), len(self.recall_thresholds), self.nc
        A, M = len(self.area_ranges), len(self.max_dets)
        return [(T, R, nc, A, M), (T, nc, A, M), (A, nc), (nc + 1,)]

    def _compute_host(self, parts, state):
        precision, recall, n_gt, seg = parts
        stats = summarize_coco(precision, recall, self.iou_thresholds, self.max_dets)
        return dict(summarize_precision(precision[..., 0, -1], self.iou_thresholds), stats=stats,
                    precision=precision, recall=recall, n_gt=n_gt.T.astype(np.int64),
                    n_det=np.diff(seg).astype(np.int64))


def summarize_coco(precision, recall, iou_thresholds, max_dets, area_labels=COCO_AREA_LABELS):
    """pycocotools' COCOeval.summarize / _summarizeDets on COCOeval.eval's tables: the 12 stats.  Thresholds are
    selected by exact float equality and maxDets by value, as there; stats[0] reads maxDets = 100 literally."""
    iou_thresholds = np.asarray(iou_thresholds)

    def summ(ap, iou_thr=None, area="all", md=100):
        aind = [i for i, lbl in enumerate(area_labels) if lbl == area]
        mind = [i for i, m in enumerate(max_dets) if m == md]
        s = precision if ap else recall
        if iou_thr is not None:
            s = s[np.where(iou_thr == iou_thresholds)[0]]
        s = s[:, :, :, aind, mind] if ap else s[:, :, aind, mind]
        return _mean_valid(s)

    md = max_dets
    return np.array([summ(1), summ(1, .5, md=md[2]), summ(1, .75, md=md[2]), summ(1, area="small", md=md[2]),
                     summ(1, area="medium", md=md[2]), summ(1, area="large", md=md[2]), summ(0, md=md[0]),
                     summ(0, md=md[1]), summ(0, md=md[2]), summ(0, area="small", md=md[2]),
                     summ(0, area="medium", md=md[2]), summ(0, area="large", md=md[2])])


def format_coco_stats(stats, iou_thresholds=COCO_IOU_THRESHOLDS, max_dets=COCO_MAX_DETS):
    """The twelve lines pycocotools' summarize() prints for `stats` (COCODetectionEval.compute()["stats"])."""
    line = " {:<18} {} @[ IoU={:<9} | area={:>6s} | maxDets={:>3d} ] = {:0.3f}"
    every = "{:0.2f}:{:0.2f}".format(iou_thresholds[0], iou_thresholds[-1])
    md = max_dets
    rows = [(1, None, "all", 100), (1, .5, "all", md[2]), (1, .75, "all", md[2]), (1, None, "small", md[2]),
            (1, None, "medium", md[2]), (1, None, "large", md[2]), (0, None, "all", md[0]), (0, None, "all", md[1]),
            (0, None, "all", md[2]), (0, None, "small", md[2]), (0, None, "medium", md[2]), (0, None, "large", md[2])]
    return [line.format("Average Precision" if ap else "Average Recall", "(AP)" if ap else "(AR)",
                        every if thr is None else "{:0.2f}".format(thr), area, m, float(v))
            for (ap, thr, area, m), v in zip(rows, stats)]


# --------------------------------------------------------------------------------------------
# validation report: confusion matrix, P/R/F1 over the confidence threshold, per-class table
# --------------------------------------------------------------------------------------------
DEFAULT_CONF_GRID = tuple(np.linspace(0.0, 1.0, 1000).tolist())


class DetectionReport:
    """The validation report YOLO tools print, of the kept detections of `detect_batch`, accumulated over batches on
    the device: a confusion matrix with a background row and column, precision / recall / F1 curves over the
    confidence threshold at IoU `curve_iou`, the threshold with the best mean F1, and DetectionMAP's AP columns for a
    per-class table (format_detection_report).  include/yolo_b200.h states the matrix and histogram semantics.

    conf_grid: the thresholds of the curves, strictly ascending and finite; a detection counts at grid[k] when its
    score is > grid[k].  cm_conf / cm_iou: the matrix's score and IoU thresholds (both strict).

    update(det, labels) runs DetectionMAP.update and one report kernel on the records it wrote; it never
    synchronises.  compute() runs DetectionMAP's compute path plus the histograms' suffix sums and synchronises
    once.

    compute(group) evaluates an image-sharded run as DetectionMAP.compute(group) does: a collective over `group` that
    returns on every rank the dict of one process that saw every rank's batches in rank order, bit-identical when
    rank r updated the r-th contiguous block of images in image order.  With any other assignment the counts (n_gt,
    n_det, confusion, images, images_total, the histograms and so the curves and best_conf) and recall are still
    identical, and precision (with the AP values taken from it) can differ only through the order of equal-score
    detections of different images."""

    def __init__(self, num_classes, max_det=300, iou_thresholds=COCO_IOU_THRESHOLDS, conf_grid=DEFAULT_CONF_GRID,
                 curve_iou=0.5, cm_conf=0.25, cm_iou=0.45):
        self.map = DetectionMAP(num_classes, iou_thresholds=iou_thresholds, max_det=max_det)
        self.nc = self.map.nc
        self.conf_grid = np.asarray(conf_grid, dtype=np.float64).reshape(-1)
        self.curve_iou, self.cm_conf, self.cm_iou = float(curve_iou), float(cm_conf), float(cm_iou)
        hit = np.flatnonzero(self.map.iou_thresholds == self.curve_iou)
        if hit.size == 0:
            raise ValueError(f"curve_iou={curve_iou} is not one of iou_thresholds {self.map.iou_thresholds.tolist()}")
        self._t_curve = int(hit[0])
        if (self.conf_grid.size < 1 or not np.all(np.isfinite(self.conf_grid))
                or not np.all(np.diff(self.conf_grid) > 0)):
            raise ValueError("conf_grid must be a non-empty, strictly ascending sequence of finite values")
        if not (np.isfinite(self.cm_conf) and np.isfinite(self.cm_iou)):
            raise ValueError("cm_conf and cm_iou must be finite")
        nc, K, dev = self.nc, self.conf_grid.size, self.map.device
        self.device = dev
        with torch.cuda.device(dev):
            self._grid = torch.tensor(self.conf_grid, dtype=torch.float64, device=dev)
            # one buffer, zeroed at once: confusion (nc+1)^2, images (nc), det_hist (nc,K), tp_hist (nc,K)
            self._counts = torch.zeros((nc + 1) ** 2 + nc + 2 * nc * K, dtype=torch.int64, device=dev)
        # compute()'s one copy back goes to page-locked memory: about 16 bytes per class and grid point
        self._host = torch.empty(sum(map(math.prod, self._host_shapes())) + 1, dtype=torch.float64,
                                 pin_memory=True)
        self._confusion, self._images, self._det_hist, self._tp_hist = _unpack(
            self._counts, [(nc + 1, nc + 1), (nc,), (nc, K), (nc, K)])
        self.reset()

    def reset(self):
        """Forget every batch seen so far."""
        self.map.reset()
        self.images_total = 0
        with torch.cuda.device(self.device):
            self._counts.zero_()

    def update(self, det, labels: PackedLabels):
        """Match one batch: the arguments of DetectionMAP.update.  After an error, reset() before the next update."""
        rec = self.map.update(det, labels)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().yb_report_match(
                *self.map._match_prefix(det, labels), rec.data_ptr(), self._t_curve, self._grid.data_ptr(),
                self.conf_grid.size, self.cm_conf, self.cm_iou, self._confusion.data_ptr(), self._images.data_ptr(),
                self._det_hist.data_ptr(), self._tp_hist.data_ptr(), self.map._status.data_ptr(), _stream()),
                "yb_report_match")
        self.images_total += det["boxes"].shape[0]

    def compute(self, group=None):
        """DetectionMAP.compute()'s dict plus, on the host:
        px (K,) the grid; p_curve, r_curve, f1_curve (nc,K) at curve_iou (P = TP/D, 1 where D = 0; R = TP/n_gt;
        F1 = 2PR/(P+R), 0 where P+R = 0; rows of classes without ground truth -1); best_conf = px[k*] with k* the
        first arg-max of the mean F1 over the classes with ground truth (None when there are none); p, r, f1 (nc,)
        at k*; confusion (nc+1,nc+1) and images (nc) int64; images_total; iou_thresholds (the columns of ap).
        group: a torch.distributed process group to merge over (see the class docstring)."""
        return _compute_metric(self, group)

    def _local_state(self):
        """The map's state with this report's counts appended to gt_count, and images_total."""
        rec, gt_count, gt_total, _, status = self.map._local_state()
        return rec, torch.cat([gt_count, self._counts]), gt_total, self.images_total, status

    def _fingerprint(self):
        mp = self.map
        return _eval_fingerprint(3, self.nc, len(mp.iou_thresholds), len(mp.recall_thresholds), 0, 0, self.conf_grid.size,
                                 mp.max_det, (mp.iou_thresholds, mp.recall_thresholds, self.conf_grid,
                                              (self.curve_iou, self.cm_conf, self.cm_iou)))

    def _compute_device(self, state):
        """The map's tensors, then the confusion matrix and images, then the histograms' suffix sums."""
        rec, counts, gt_total, images_total, status = state
        nc, K = self.nc, self.conf_grid.size
        gt_count, counts = counts[:nc], counts[nc:]
        hist = counts[(nc + 1) ** 2 + nc:].view(2, nc, K)   # det_hist, tp_hist
        rev = hist.flip(2).cumsum(2)   # [.., K-1-k] = detections / TPs with score > grid[k]
        return (self.map._compute_device((rec, gt_count, gt_total, images_total, status))
                + [counts[:(nc + 1) ** 2 + nc].double(), rev.reshape(-1).double()])

    def _copy_back(self, tensors):
        self._host.copy_(torch.cat(tensors), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._host.numpy()

    def _host_shapes(self):
        nc, K = self.nc, self.conf_grid.size
        return self.map._host_shapes() + [(nc + 1, nc + 1), (nc,), (2, nc, K)]

    def _compute_host(self, parts, state):
        m = len(self.map._host_shapes())
        out = self.map._compute_host([p.copy() for p in parts[:m]], state)   # it returns views; the buffer is reused
        confusion, images, hist = parts[m:]
        n_det, n_tp = hist.astype(np.int64)[:, :, ::-1]
        out.update(report_curves(n_det, n_tp, out["n_gt"], self.conf_grid), confusion=confusion.astype(np.int64),
                   images=images.astype(np.int64), images_total=state[3], iou_thresholds=self.map.iou_thresholds.copy())
        return out


def report_curves(n_det, n_tp, n_gt, px):
    """px, p_curve, r_curve, f1_curve, best_conf, p, r, f1 (DetectionReport.compute's fields) from the detections
    n_det (nc,K) and TPs n_tp (nc,K) with score > px[k] and the ground truths n_gt (nc) per class."""
    tp, d = n_tp.astype(np.float64), n_det.astype(np.float64)
    n = np.asarray(n_gt, dtype=np.float64)[:, None]
    has_gt = np.asarray(n_gt) > 0
    with np.errstate(divide="ignore", invalid="ignore"):   # 0/0 where D = 0, P + R = 0 or n_gt = 0: replaced
        p = tp / d
        p[d == 0] = 1.0
        r = tp / n
        s = p + r
        f1 = 2 * p * r / s
    f1[s == 0] = 0.0
    p[~has_gt], r[~has_gt], f1[~has_gt] = -1.0, -1.0, -1.0
    if has_gt.any():
        k = int(np.argmax(f1[has_gt].mean(axis=0)))
        best_conf = float(px[k])
        at = (p[:, k].copy(), r[:, k].copy(), f1[:, k].copy())
    else:
        best_conf = None
        at = tuple(np.full(len(has_gt), -1.0) for _ in range(3))
    return {"px": np.asarray(px, dtype=np.float64).copy(), "p_curve": p, "r_curve": r, "f1_curve": f1,
            "best_conf": best_conf, "p": at[0], "r": at[1], "f1": at[2]}


def format_detection_report(out, names=None):
    """The per-class table of DetectionReport.compute()'s dict `out`, as YOLO validators print it: a header, an
    `all` row (images, ground truths, mean P and R at best_conf over the classes with ground truth, map50, map) and
    one row per class with ground truth (its images, ground truths, P, R, AP50, AP50-95).  names: class names
    (default: the class indices).  A value that does not exist (no class with ground truth, no 0.5 threshold) is
    printed as -1."""
    n_gt, ap = np.asarray(out["n_gt"]), np.asarray(out["ap"])
    has_gt = n_gt > 0
    mean = lambda v: float(np.mean(v[has_gt])) if has_gt.any() else -1.0
    hit = np.flatnonzero(np.asarray(out["iou_thresholds"]) == 0.5)
    neg = lambda v: -1.0 if v is None else v
    row = "%22s" + "%11i" * 2 + "%11.3g" * 4
    lines = [("%22s" + "%11s" * 6) % ("Class", "Images", "Instances", "P", "R", "mAP50", "mAP50-95"),
             row % ("all", out["images_total"], int(n_gt.sum()), mean(out["p"]), mean(out["r"]), neg(out["map50"]),
                    out["map"])]
    for c in np.flatnonzero(has_gt):
        name = str(names[c]) if names is not None else str(c)
        lines.append(row % (name, out["images"][c], n_gt[c], out["p"][c], out["r"][c],
                            ap[c, hit[0]] if hit.size else -1.0, ap[c].mean()))
    return lines


# --------------------------------------------------------------------------------------------
# the whole step as one CUDA graph
# --------------------------------------------------------------------------------------------
class HotPathGraph:
    """loss forward+backward + decode/filter/global NMS + detection packing for a fixed batch shape,
    captured once as a CUDA graph (about twenty kernel launches, memsets and workspace allocations
    replayed with a single launch; the per-step host cost drops from ~1 ms of Python to microseconds).

    Static inputs (fill them, e.g. with `copy_` from pinned host memory, then call `replay()`):
      heads[s]   (B,G,G,A,5+nc), or (B,A*(5+nc),G,G) with layout=LAYOUT_NCHW
      labels     PackedLabels (targets="labels": assignment on the device, SURVEY 8f-4), or
      targets[s] dense (B,G,G,A,5+nc) (targets="dense": the reference's call signature)
    Static outputs: losses (4,) [total, bbox, obj, cls], grads[s] (gradient of `total`), det (the
    detect_batch dict), rows (B*cap,6) + offsets (B+1,) from pack_detections.
    An image whose NMS graph overflows the edge list is resolved exactly inside the same launch.

    dtype: element type of the static heads and gradients, torch.float32, torch.bfloat16 or torch.float16.  A half
    graph also owns `grad_scale`, a (1,) fp32 device tensor (1.0 at first) that the captured kernels read at every
    replay: grads[s] are the gradients of grad_scale * total, rounded to dtype after the scaling — what
    `scaler.scale(total).backward()` gives.  Copy a GradScaler's scale into it between replays."""

    def __init__(self, batch, img_size, num_classes, anchors_list, conf_threshold=0.5, iou_threshold=0.4, max_gt=50,
                 targets="labels", layout=LAYOUT_BHWAC, num_anchors=3, device=None, adopt_heads=None,
                 adopt_targets=None, group=None, overlap_loss=True, fork_loss="auto", dtype=torch.float32):
        """adopt_heads / adopt_targets: existing device tensors (or a PackedLabels) to use as the static
        inputs instead of allocating new ones.  group: torch.distributed process group of an image-sharded
        job; the all-reduce of the loss partials is then captured inside the graph (NCCL).
        overlap_loss: the loss kernels (HBM-bound, few resident warps) and the filter/NMS kernels (issue-bound)
        are independent readers of the heads; they are captured as two parallel branches of the graph."""
        if dtype not in _HEAD_DTYPES:
            raise ValueError(f"dtype must be torch.float32, torch.bfloat16 or torch.float16, got {dtype}")
        if adopt_heads is not None:
            for s, h in enumerate(adopt_heads):
                if h.dtype != dtype:
                    raise ValueError(f"adopt_heads[{s}] is {h.dtype}, the graph's dtype is {dtype}")
        self.dtype = dtype
        self.group = group
        self.overlap_loss = bool(overlap_loss)
        if fork_loss not in ("auto", "start", "after_filter"):
            raise ValueError("fork_loss must be 'auto', 'start' or 'after_filter'")
        self.fork_loss = fork_loss   # "auto" is resolved below, once the kind of targets is known
        dev = _device() if device is None else torch.device(device)
        self.device, self.nc, self.img, self.layout = dev, int(num_classes), int(img_size), layout
        row = 5 + self.nc
        grids = [img_size // 8, img_size // 16, img_size // 32]
        with torch.cuda.device(dev):
            self.anchors = [_anchors_dev(a, dev) for a in anchors_list]
            A = num_anchors
            if adopt_heads is not None:
                self.heads = list(adopt_heads)
            elif layout == LAYOUT_NCHW:
                self.heads = [torch.zeros(batch, A * row, g, g, device=dev, dtype=dtype) for g in grids]
            else:
                self.heads = [torch.zeros(batch, g, g, A, row, device=dev, dtype=dtype) for g in grids]
            self.grad_scale = None if dtype == torch.float32 else torch.ones(1, dtype=torch.float32, device=dev)
            self.labels = self.targets = None
            if adopt_targets is not None:
                if isinstance(adopt_targets, PackedLabels):
                    self.labels = adopt_targets
                else:
                    self.targets = list(adopt_targets)
            elif targets == "labels":
                lab, n_gt, lb = pack_labels_host([()] * batch, img_size, max_gt=max_gt)
                self.labels = PackedLabels(lab.to(dev), n_gt.to(dev), lb.to(dev), img_size)
            elif targets == "dense":
                self.targets = [torch.zeros(batch, g, g, A, row, device=dev) for g in grids]
            else:
                raise ValueError("targets must be 'labels' or 'dense'")
            self.conf, self.iou = float(conf_threshold), float(iou_threshold)
            if self.fork_loss == "auto":
                # Where the loss branch leaves the detection chain.  Short rows (nc <= 3) with dense targets: the loss
                # kernels take about as long as the two one-CTA-per-image kernels after the filter, so they start there
                # and the filter has the memory system to itself (B200, nc=1: 295.5 -> 289.2 us per step).  Long rows
                # or label-list targets (assignment kernels first): the loss is the longer branch, would still be
                # running when the persistent edge kernel takes every SM, and starts with the filter instead
                # (nc=80: 572 against 578 us; nc=1 with labels: 291.6 against 294.0 us).
                self.fork_loss = "after_filter" if (5 + self.nc <= 8 and self.labels is None) else "start"
            self._branch = torch.cuda.Stream(device=dev) if self.overlap_loss else None
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):  # warm-up outside the capture (function attributes, allocator pools)
                    self._step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.losses, self.grads, self.det, self.rows, self.offsets = self._step()

    def _loss(self):
        out4, _, grads = loss_forward_backward(self.heads, self.targets, self.anchors, self.nc, MULTISCALE_OBJ_WEIGHTS,
                                               [True] * len(self.heads), sparse=self.labels, layout=self.layout,
                                               group=self.group, grad_scale=self.grad_scale)
        return out4, grads

    def _step(self):
        cur = torch.cuda.current_stream()
        fork_late = self._branch is not None and self.fork_loss == "after_filter"
        if self._branch is not None and not fork_late:   # fork: loss on a second stream, joined before the step ends
            self._branch.wait_stream(cur)
            with torch.cuda.stream(self._branch):
                out4, grads = self._loss()
        elif self._branch is None:
            out4, grads = self._loss()
        cand = filter_candidates(self.heads, self.anchors, self.img, self.nc, self.conf, None, self.layout)
        if fork_late:
            # the filter and the loss both stream the heads from HBM, while the two kernels after the filter run
            # one CTA per image: forking here gives the filter the whole memory system and the loss the idle SMs
            self._branch.wait_stream(cur)
            with torch.cuda.stream(self._branch):
                out4, grads = self._loss()
        det = nms_candidates(*cand, self.iou)
        rows, offsets = pack_detections(det)
        if self._branch is not None:
            cur.wait_stream(self._branch)
        return out4, grads, det, rows, offsets

    def replay(self):
        """Enqueue the captured step on the current stream."""
        self.graph.replay()
        return self.losses, self.grads, self.det
