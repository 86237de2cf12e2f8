"""yolo_from_scratch_b200 — B200-native per-box detection hot path of KhaledSharif/yolo-from-scratch.

decode -> (target assignment + CIoU/objectness/class loss, forward+backward) -> cross-scale global
NMS, as hand-written sm_100a CUDA kernels in libyolo_b200.so (C-ABI: include/yolo_b200.h), with
the reference's own Python function signatures on top (ops.py) and an installer that swaps them
into the reference's `train` module (install.py).
"""
from . import _lib
from .ops import (COCO_AREA_LABELS, COCO_AREA_RANGES, COCO_IOU_THRESHOLDS, COCO_MAX_DETS, COCO_RECALL_THRESHOLDS,
                  COCODetectionEval, DetectionMAP, DetectionReport, format_coco_stats, format_detection_report, batched_nms, batched_nms_padded, build_targets, ciou_loss, compute_anchor_iou,
                  decode_predictions, default_anchors, detect_batch, detect_batch_nchw, detections_to_lists, heads_from_nchw, eval_counts, eval_epoch,
                  filter_candidates, filter_candidates_multilabel, MAX_CANDIDATES,
                  loss_forward_backward, nms, nms_retry_overflow, pack_detections, predict_heads,
                  NMS_GRAPH, NMS_BITMASK, HotPathGraph, LAYOUT_BHWAC, LAYOUT_NCHW, PackedLabels, pack_labels, pack_labels_host, yolo_loss,
                  yolo_loss_multiscale, yolo_loss_multiscale_labels, yolo_loss_multiscale_nchw)

__all__ = [
    "decode_predictions", "ciou_loss", "yolo_loss", "yolo_loss_multiscale", "compute_anchor_iou",
    "build_targets", "filter_candidates", "nms", "batched_nms", "batched_nms_padded", "detect_batch",
    "detections_to_lists", "pack_detections", "loss_forward_backward", "yolo_loss_multiscale_labels",
    "PackedLabels", "pack_labels", "pack_labels_host", "eval_counts", "eval_epoch", "yolo_loss_multiscale_nchw",
    "detect_batch_nchw", "heads_from_nchw", "predict_heads", "HotPathGraph", "LAYOUT_BHWAC", "LAYOUT_NCHW", "default_anchors",
    "DetectionMAP", "COCO_IOU_THRESHOLDS", "COCO_RECALL_THRESHOLDS",
    "COCODetectionEval", "COCO_AREA_RANGES", "COCO_AREA_LABELS", "COCO_MAX_DETS", "format_coco_stats",
    "DetectionReport", "format_detection_report", "filter_candidates_multilabel", "MAX_CANDIDATES",
]
