/*
 * yolo_b200.h — C-ABI of libyolo_b200.so: the per-box detection hot path of
 * KhaledSharif/yolo-from-scratch as hand-written sm_100a CUDA kernels.
 *
 * The reference has no FFI of its own (it is pure Python on PyTorch); each entry point below
 * replaces one Python-level function of reference `train.py` (cited as file:line) and is what a
 * ctypes binding in that file would call.  INTEGRATION.md shows the binding.
 *
 * Conventions (all entry points):
 *   - every pointer is a CALLER-OWNED DEVICE pointer unless the name ends in `_host`;
 *     the library never allocates, frees or retains memory (the tests-only yb_selftest_sigmoid aside);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy default
 *     stream); no entry point synchronises the device or the stream.  One entry point,
 *     yb_batched_nms with YB_NMS_GRAPH, additionally uses a library-owned side stream between two
 *     events (fork after the work already enqueued on `stream`, join before its last kernel): its
 *     score sort overlaps with the rest; every result is still ordered after `stream`, and under
 *     stream capture the fork/join becomes two parallel branches of the captured graph;
 *   - return value 0 = success, otherwise a cudaError_t or a negative YB_E* code;
 *     yb_last_error() returns a thread-local, human readable message for the last failure;
 *   - head tensors use the model-output layout of train.py:608-609: contiguous fp32
 *     (B, H, W, A, 5+nc), row = [tx, ty, tw, th, obj, cls...] raw logits; the loss, decode and
 *     filter entry points also take bf16 or fp16 heads (YB_DTYPE_*, below);
 *   - `anchors` are fp32 (A,2) = [w,h] in pixels (train.py:372-374, 386-388);
 *   - tensors must be 16-byte aligned (every torch allocation is).
 */
#ifndef YOLO_B200_H
#define YOLO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YB_MAX_SCALES 4
#define YB_MAX_ANCHORS 8

/* Layout of head tensors (pred / grad): the model-output contract of train.py:608-609,
 * (B, H, W, A, 5+nc), or — f-2, SURVEY 8f — the head conv's own output (B, A*(5+nc), H, W), i.e. the
 * tensor BEFORE the reference's view/permute/contiguous: the path then reads the conv output directly
 * and that full read+write pass (and its backward) disappears.  Dense targets always keep the
 * reference layout; row indices, candidate order and all results are identical in both layouts. */
#define YB_LAYOUT_BHWAC 0
#define YB_LAYOUT_NCHW 1

/* Element type of head tensors (pred / grad / decode output).  A zero-filled descriptor means fp32.
 * Half heads are read as they are: every value widens exactly to fp32 and all arithmetic is the fp32
 * path's, so every result equals the fp32 path on the upcast heads.  Half results (decode output,
 * loss gradients) are the fp32 values rounded to nearest even (__float2bfloat16_rn / __float2half_rn;
 * overflow in fp16 gives +-inf).  Targets, anchors, candidates and boxes stay fp32. */
#define YB_DTYPE_F32 0
#define YB_DTYPE_BF16 1
#define YB_DTYPE_F16 2

#define YB_EINVAL (-1)   /* bad argument (shape, null pointer, alignment) */
#define YB_EWORKSPACE (-2) /* workspace too small */

/* Library/ABI version (major*100+minor) and last error text (thread local). */
int yb_version(void);
const char* yb_last_error(void);

/* ------------------------------------------------------------------------------------------
 * a-1  decode_predictions(raw_preds, anchors, img_size=640)            train.py:712-779
 *   out[...,0] = ((2*sigmoid(tx) - 0.5) + gx) / W        (:758)
 *   out[...,1] = ((2*sigmoid(ty) - 0.5) + gy) / H        (:759)
 *   out[...,2] = (aw/img) * (2*sigmoid(tw))^2            (:773)
 *   out[...,3] = (ah/img) * (2*sigmoid(th))^2            (:774)
 *   out[...,4:] = pred[...,4:]                            (:737, clone)
 * yb_decode_bwd is its vector-Jacobian product: grad_in = J^T grad_out (autograd of the above).
 * ---------------------------------------------------------------------------------------- */
int yb_decode_fwd(const float* pred, const float* anchors, float* out,
                  int B, int H, int W, int A, int nc, float img_size, void* stream);
int yb_decode_bwd(const float* pred, const float* anchors, const float* grad_out, float* grad_in,
                  int B, int H, int W, int A, int nc, float img_size, void* stream);
/* The same on heads of element type `dtype` (YB_DTYPE_*): pred, out, grad_out and grad_in all have that
 * type.  out = round(fp32 decode of the widened pred); grad_in = round(fp32 vector-Jacobian product of the
 * widened pred and grad_out).  yb_decode_fwd / yb_decode_bwd are the fp32 case. */
int yb_decode_fwd_t(const void* pred, const float* anchors, void* out, int B, int H, int W, int A, int nc,
                    float img_size, int dtype, void* stream);
int yb_decode_bwd_t(const void* pred, const float* anchors, const void* grad_out, void* grad_in, int B, int H,
                    int W, int A, int nc, float img_size, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * a-2  ciou_loss(pred_boxes, target_boxes, eps=1e-7)                    train.py:634-710
 *   boxes are (N,4) xywh.  loss_out[0] = mean_i(1 - CIoU_i)  (NaN when N == 0, like torch).
 *   grad_pred / grad_tgt (nullable) receive d loss / d box (alpha is a constant, :701-702).
 *   `partials` is a caller-provided scratch of yb_ciou_scratch_bytes(N) bytes.
 * ---------------------------------------------------------------------------------------- */
size_t yb_ciou_scratch_bytes(long long N);
int yb_ciou_fwd_bwd(const float* pred_boxes, const float* tgt_boxes, long long N, float eps,
                    float* loss_out, float* grad_pred, float* grad_tgt,
                    void* scratch, size_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a-3 / a-4  yolo_loss (train.py:781-838) and yolo_loss_multiscale (train.py:840-886),
 *            forward and backward fused.
 *
 * Stage 1  yb_loss_partials: one pass over every scale.
 *   For each scale s it accumulates partials[s] = { sum_pos(1-CIoU), n_pos, sum_all BCE(obj),
 *   sum_pos,cls BCE(cls) } (4 doubles per scale) over the LOCAL batch, and when grad[s] != NULL
 *   writes the dense gradient: the objectness column fully normalised by
 *   coef_obj[s] / (B_global*H*W*A), box/class columns of positive rows UN-normalised, zeros
 *   elsewhere.  Positive = target objectness > 0.5 (:809).  Decode uses `img_size` (the
 *   reference always passes its default 640 here, :796).
 * Between the stages a data-parallel caller all-reduces(sum) the S*4 doubles (SURVEY 8e).
 * Stage 2  yb_loss_finalize: takes the (globally reduced) partials, scales the box/class
 *   gradient entries of the local positive rows by coef_box[s]/P_s and coef_cls[s]/(P_s*nc),
 *   and writes out4 = { total, sum_s bbox_s, sum_s obj_s, sum_s cls_s } plus, if per_scale != NULL,
 *   per_scale[s] = { bbox_s, obj_s, cls_s } (means, exactly the three values yolo_loss returns).
 *   total = sum_s (w_box*bbox_s + w_obj[s]*obj_s + w_cls*cls_s)   (:836, :879).
 *
 * coef_* are d(final scalar)/d(term_s): for `total.backward()` they are w_box, w_obj[s], w_cls.
 * `ws` is a caller-provided workspace of yb_loss_workspace_bytes(...) bytes shared by both stages.
 * ---------------------------------------------------------------------------------------- */
typedef struct yb_loss_desc {
    int S;                          /* number of scales, 1..YB_MAX_SCALES */
    int B;                          /* local batch */
    long long B_global;             /* global batch (== B on one GPU): obj mean normaliser */
    int A, nc;
    int H[YB_MAX_SCALES], W[YB_MAX_SCALES];
    float img_size;                 /* decode img_size, 640 in the reference's loss (:796) */
    float eps;                      /* CIoU eps, 1e-7 (:634) */
    float w_box, w_cls;             /* 0.05, 0.5 (:836) */
    float w_obj[YB_MAX_SCALES];     /* 1.0 for yolo_loss; [4.0,1.0,0.4] multiscale (:865) */
    float coef_box[YB_MAX_SCALES];  /* upstream coefficients for the gradient */
    float coef_obj[YB_MAX_SCALES];
    float coef_cls[YB_MAX_SCALES];
    const float* pred[YB_MAX_SCALES];
    const float* tgt[YB_MAX_SCALES];
    const float* anchors[YB_MAX_SCALES];
    float* grad[YB_MAX_SCALES];     /* nullable: forward only (torch.no_grad callers) */
    int layout;                     /* YB_LAYOUT_* of pred and grad */
    int dtype;                      /* YB_DTYPE_* of pred and grad (tgt stays fp32) */
} yb_loss_desc;

/* Half heads (dtype bf16 / fp16).  The gradient of `total` depends on its upstream gradient s, which is
 * known only at backward, and s has to be applied BEFORE the rounding to half (fp16 objectness gradients,
 * ~coef/(B*H*W*A), are subnormal or zero in fp16 until a GradScaler's s lifts them).  So stage 1 writes
 * no dense gradient for half heads (grad[] is ignored there): it keeps the fp32 objectness gradient, one
 * float per row, and the positive lists in `ws` (the workspace is rows*4 bytes larger than for fp32).
 * yb_loss_grad_emit then writes grad[s] completely, after stage 2, from the same workspace and the
 * same reduced partials (max_gt: the value given to yb_loss_partials_sparse, or -1 after yb_loss_partials):
 *   grad = round(s == 1 ? G : round_f32(G * s)),  s = *grad_scale (device fp32),
 * where G is the fp32 path's gradient for upstream 1 (positive rows: g, then g * coef/P, each rounded
 * to fp32) and round() rounds to nearest even in the head dtype — exactly what the fp32 path followed by
 * yb_scale_inplace and a cast to the head dtype gives, for every s.  It may be called again (the
 * workspace is read only) and is capturable; *grad_scale is read when the kernels run. */
int yb_loss_grad_emit(const yb_loss_desc* d, const double* partials /* S*4, reduced */,
                      const float* grad_scale, int max_gt, void* ws, size_t ws_bytes, void* stream);

size_t yb_loss_workspace_bytes(const yb_loss_desc* d);
int yb_loss_partials(const yb_loss_desc* d, double* partials /* S*4 */,
                     void* ws, size_t ws_bytes, void* stream);
int yb_loss_finalize(const yb_loss_desc* d, const double* partials /* S*4, reduced */,
                     float* out4, float* per_scale /* S*3, nullable */,
                     void* ws, size_t ws_bytes, void* stream);

/* f-4 (SURVEY 8f): the same stage 1 fed by label lists instead of dense targets — the label loop of
 * YOLODataset.__getitem__ (train.py:147-205, as yb_build_targets) runs on the device and hands the
 * loss a sparse form of its result: per-scale lists of the assigned rows, their 32-byte target rows
 * and a 1-bit-per-row positive map.  Neither the dense targets (3 tensors the size of the heads) nor
 * their host->device copy (train.py:900-902) exist on this path; d->tgt[] is ignored.
 *   labels (B,max_gt,5) fp64, n_gt (B) int32, letterbox (B,5) fp64, anchors_all (S,A,2) fp32,
 *   assign_img_size = the dataset's img_size (:159-167); status as in yb_build_targets.
 * Results equal yb_loss_partials on the dense targets yb_build_targets would have produced.
 * Stage 2 is yb_loss_finalize with the same workspace. */
size_t yb_loss_sparse_workspace_bytes(const yb_loss_desc* d, int max_gt);
int yb_loss_partials_sparse(const yb_loss_desc* d, const double* labels, const int* n_gt,
                            const double* letterbox, const float* anchors_all, int max_gt,
                            int assign_img_size, int* status, double* partials /* S*4 */,
                            void* ws, size_t ws_bytes, void* stream);

/* x[i] *= *factor for i < n, skipped entirely (no memory traffic) when *factor == 1.0f.
 * Used by the autograd wrapper to apply the upstream gradient of `total` to the gradient the
 * fused kernel already produced (loss.backward() passes exactly 1.0).  factor is a device pointer. */
int yb_scale_inplace(float* x, long long n, const float* factor, void* stream);

/* ------------------------------------------------------------------------------------------
 * a-5  target assignment                                         train.py:108-131, 147-205
 *   yb_anchor_iou: YOLODataset.compute_anchor_iou for n boxes x A anchors (fp32, +1e-16).
 *   yb_build_targets: the label loop of YOLODataset.__getitem__ for a batch.
 *     labels   (B, max_gt, 5) fp64 = raw label lines [class, xc, yc, w, h]
 *     n_gt     (B) int32
 *     letterbox(B, 5) fp64 = [orig_w, orig_h, scale, pad_top, pad_left]  (:136-137)
 *     anchors  (S, A, 2) fp32
 *     targets[s] (B, G_s, G_s, A, 5+nc) fp32, fully written (zero-filled then assigned)
 *   Bit-exact with the reference: fp64 letterbox/cell math (:159-166,:184-189), fp32 shape IoU,
 *   strict '>' across scales then first argmax (:177-180), first GT wins a slot (:193),
 *   nc==1 writes class slot 5 irrespective of label id (:201-202).  Python's negative-index
 *   wrap-around for cells in [-G, 0) is reproduced; rows the reference would reject
 *   (IndexError) set bit 0 of *status (device int32, nullable).
 * ---------------------------------------------------------------------------------------- */
int yb_anchor_iou(const float* box_wh, const float* anchors, float* iou_out,
                  int n, int A, void* stream);
int yb_build_targets(const double* labels, const int* n_gt, const double* letterbox,
                     const float* anchors, float* const targets_host[YB_MAX_SCALES],
                     int B, int max_gt, int S, const int* G_host, int A, int nc, int img_size,
                     int* status, void* stream);

/* ------------------------------------------------------------------------------------------
 * a-6  candidate filter + box build of predict()                  train.py:1152-1222, 1227-1229
 *   For every image b and every row in P3->P4->P5, row-major (gy,gx,a) order:
 *     keep rows with sigmoid(obj) > conf  (:1166-1167, objectness only)
 *     class prob/id = max sigmoid(cls) (first max; nc==1: slot 5, id 0)  (:1184-1189)
 *     xyxy in pixels, minus (pad_left,pad_top), divided by scale  (:1192-1213)
 *     score = sigmoid(obj) * class prob  (:1216)
 *   One pass over the heads (decoupled look-back over groups of 1,024 rows; the workspace is zeroed by a
 *   memset node of the same call).
 *   Output is per image, order preserving, with a fixed stride of `cap` candidates per image:
 *     boxes (B,cap,4) fp32, scores (B,cap) fp32, classes (B,cap) int64, counts (B) int32.
 *   letterbox (B,3) fp32 = [scale, pad_top, pad_left], NULL = identity.
 *   cap must be >= total rows per image (sum_s H_s*W_s*A) unless the caller knows better;
 *   candidates beyond cap are dropped and counts[b] saturates at cap.
 * ---------------------------------------------------------------------------------------- */
typedef struct yb_heads_desc {
    int S, B, A, nc;
    int H[YB_MAX_SCALES], W[YB_MAX_SCALES];
    float img_size;
    const float* pred[YB_MAX_SCALES];
    const float* anchors[YB_MAX_SCALES];
    int layout;                     /* YB_LAYOUT_* of pred (filter: both; decode/eval: BHWAC only) */
    int dtype;                      /* YB_DTYPE_* of pred (filter: all three; eval: fp32 only) */
} yb_heads_desc;

size_t yb_filter_workspace_bytes(const yb_heads_desc* d);
int yb_filter_compact(const yb_heads_desc* d, float conf_thres, const float* letterbox,
                      float* boxes, float* scores, int64_t* classes, int* counts, int cap,
                      void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * a-7  torchvision.ops.batched_nms(boxes, scores, idxs, iou_threshold)       train.py:1232-1233
 *      (torchvision 0.26.0, torchvision/ops/boxes.py:51-120 and its CUDA nms kernel)
 *   Batched over B independent images with a fixed stride of `cap` candidates per image and
 *   counts[b] valid entries (counts == NULL: every image has `cap`).
 *   classes == NULL gives plain torchvision.ops.nms.
 *   Arithmetic is torchvision's CUDA kernel bit for bit: fp32,
 *     inter = max(0, min(ax2,bx2)-max(ax1,bx1)) * max(0, min(ay2,by2)-max(ay1,by1))
 *     iou   = inter / ( fma(bx2-bx1, by2-by1, (ax2-ax1)*(ay2-ay1)) - inter ),  a = higher score
 *     suppress when iou > (float)iou_threshold; stable descending score order (lower index wins
 *     ties).
 *   trick_max_numel reproduces batched_nms' size dispatch (boxes.py:80): an image with
 *   4*counts[b] <= trick_max_numel uses the coordinate-offset trick (boxes + cls*(max+1), fp32,
 *   boxes.py:98-101), larger ones the per-class loop (boxes.py:113-120).  Pass 100000 for CUDA
 *   callers, 4000 for CPU callers, -1 to force per-class, LLONG_MAX to force the trick.
 *   Output: keep (B,cap) int64 = kept candidate indices (0..counts[b]) in descending score order,
 *   n_keep (B) int32.
 *
 *   algo selects how the same result is computed:
 *     YB_NMS_GRAPH    (default) sparse suppression graph: spatial/area-ordered tile culling, edge
 *                     list, parallel fixed-point resolve.  Workspace holds the edge list; an image
 *                     with more edges than fit (heavily clustered boxes) or class ids >= 512 is
 *                     resolved inside the same launch by a blocked greedy pass (M x kept pair
 *                     tests, exact arithmetic), so n_keep[b] is never negative for this algorithm.
 *     YB_NMS_BITMASK  dense blocked IoU bitmask + serial scan (torchvision's structure, batched);
 *                     class ids < 65536; never overflows with yb_nms_workspace_bytes().
 * ---------------------------------------------------------------------------------------- */
#define YB_NMS_GRAPH 0
#define YB_NMS_BITMASK 1
size_t yb_nms_workspace_bytes(int B, int cap);      /* enough for either algorithm, worst case */
size_t yb_nms_min_workspace_bytes(int B, int cap);  /* fixed part; the rest holds mask rows / edges */
size_t yb_nms_graph_workspace_bytes(int B, int cap, int edges_per_box); /* graph algo, sized edge list */
int yb_batched_nms(const float* boxes, const float* scores, const int64_t* classes,
                   const int* counts, int B, int cap, double iou_threshold,
                   long long trick_max_numel, int algo, int64_t* keep, int* n_keep,
                   void* ws, size_t ws_bytes, void* stream);

/* Statistics of the last YB_NMS_GRAPH call that used workspace `ws` (bench/tests; synchronises the
 * stream), summed over the B images: IoU pair tests executed by the half-precision filter, edges found, and
 * pairs that passed the filter and were decided exactly in fp32.  Outputs are HOST pointers (nullable). */
int yb_nms_graph_stats(const void* ws, size_t ws_bytes, int B, int cap, unsigned long long* evals_host,
                       unsigned long long* edges_host, unsigned long long* cands_host, void* stream);

/* ------------------------------------------------------------------------------------------
 * detection list of predict()                                              train.py:1236-1246
 *   Packs the kept detections of a batch as rows (x1, y1, x2, y2, conf, class) fp32, image after
 *   image, each image in descending score order.  out must hold sum(n_keep)*6 floats
 *   (<= B*cap*6); offsets (B+1) int32 receives the first row of every image and the total.
 *   If any n_keep[b] is negative (NMS reported a failure for that image) the total offsets[B] is -1:
 *   a failed image never reads as "no detections".
 * ---------------------------------------------------------------------------------------- */
int yb_pack_detections(const float* boxes, const float* scores, const int64_t* classes,
                       const int64_t* keep, const int* n_keep, int B, int cap, float* out,
                       int* offsets, void* stream);

/* ------------------------------------------------------------------------------------------
 * f-1 (SURVEY 8f)  detection counting of eval_epoch                      train.py:993-1024, 928-958
 *   For every row of every scale: p = sigmoid(pred obj), t = target obj (both compared with
 *   conf_threshold in double, as `.item()` values are in the reference);
 *     p > conf and t > conf : IoU(decoded pred xywh, target xywh; compute_box_iou, eps 1e-6, fp32)
 *                              > (float)iou_threshold ? TP : FP
 *     p > conf only         : FP          t > conf only : FN
 *   d->img_size is the decode img_size (the reference always uses its default 640 here, :993).
 *   targets_host: HOST array of S device pointers, same layout as d->pred.
 *   counts3 (device, int64[3]) += {TP, FP, FN}: the caller zeroes it once per epoch.
 * ---------------------------------------------------------------------------------------- */
int yb_eval_counts(const yb_heads_desc* d, const float* const* targets_host, double conf_threshold,
                   double iou_threshold, long long* counts3, void* stream);

/* ------------------------------------------------------------------------------------------
 * mAP (COCO bbox protocol: COCOeval.evaluateImg + accumulate, area "all", no crowd)
 *   No reference equivalent: the reference scores a model with eval_epoch's precision/recall only.
 *   Stage 1, yb_map_match, once per batch, on the output of yb_filter_compact + yb_batched_nms:
 *     detections of image b = the first min(n_keep[b], max_det) entries of keep[b] (one overall cap);
 *     ground truth = labels (B,max_gt,5) fp64 [cls, xc, yc, w, h] normalised to the original image,
 *       n_gt (B) int32, letterbox (B,5) fp64 [orig_w, orig_h, ...] (yb_build_targets' inputs):
 *       x1 = (xc - w/2)*orig_w, y1 = (yc - h/2)*orig_h, x2 = (xc + w/2)*orig_w, y2 = (yc + h/2)*orig_h;
 *       nc == 1: every ground truth is class 0 (train.py:201-202);
 *     IoU = compute_iou_corners (train.py:1064-1084) in fp64 on the fp32 detection corners, 0 if union <= 0;
 *     per image, class and threshold t: each detection in keep order takes the not yet matched ground truth
 *       of its class with the highest IoU >= iou_thr[t] (the later one on equal IoU) -> TP, else FP.
 *   records (B, min(max_det,cap)) receive {score, class, TP bit t of tp}; unused slots have class -1.
 *   gt_count (nc) int64 += ground truths per class (the caller zeroes it once per evaluation);
 *   *status |= YB_MAP_BAD_CLASS (ground-truth id outside [0,nc) with nc > 1, or a detection class outside
 *   [0,nc)), YB_MAP_NMS_FAILED (n_keep[b] < 0; that image contributes no detections).
 * Between the stages the CALLER orders the records of all batches stably by (class ascending, score
 *   descending), keeping image order (batch after batch, then batch position) and keep order among equal
 *   scores — COCO's argsort(-scores, kind="mergesort") over the images in order; class -1 last.  ops.py does it
 *   with one torch.sort(stable=True) on an int64 key.  seg (nc+1) int64: class c is records [seg[c], seg[c+1]).
 *   Image-sharded runs (ops' compute(group), dist.gather_eval_state): each rank runs stage 1 on its images, and
 *   the records of ranks 0, 1, ... are concatenated before the sort, gt_count summed and status ORed.  When rank r
 *   holds the r-th contiguous block of images in image order this is exactly one process's order, so the tables
 *   are bit-identical.  With any other assignment (an interleaving sampler) the counts are still identical and the
 *   precision table can differ only through the order of equal-score records of different images.  The same holds
 *   for yb_coco_precision's records and yb_report_match's counts below.
 * Stage 2, yb_map_precision, once per evaluation, one CTA per class:
 *   tp, fp = cumulative counts (doubles), rc = tp / n_gt_c, pr = tp / (fp + tp + 2^-52);
 *   precision[t][r][c] = max of pr over positions with rc >= recall_thr[r] (0 if none), recall[t][c] = rc at the
 *   last detection (0 without detections); both tables -1 for a class without ground truth.
 *   ws: yb_map_workspace_bytes(number of records, total ground truths or an upper bound, T) bytes;
 *   *status |= YB_MAP_INCONSISTENT when a class has more TPs than ground truths or ws is too small.
 * ---------------------------------------------------------------------------------------- */
#define YB_MAP_MAX_T 16
#define YB_MAP_MAX_GT 4096
#define YB_MAP_BAD_CLASS 1
#define YB_MAP_NMS_FAILED 2
#define YB_MAP_INCONSISTENT 4
typedef struct yb_map_record {
    float score;
    int32_t cls;     /* -1: unused slot */
    uint16_t tp;     /* bit t: TP at iou_thr[t] */
    uint16_t pad;
} yb_map_record;

int yb_map_match(const float* boxes, const float* scores, const int64_t* classes, const int64_t* keep,
                 const int* n_keep, int B, int cap, int max_det, const double* labels, const int* n_gt,
                 const double* letterbox, int max_gt, int nc, const double* iou_thr, int T,
                 yb_map_record* records, long long* gt_count, int* status, void* stream);
size_t yb_map_workspace_bytes(long long n_records, long long n_gt_total, int T);
int yb_map_precision(const yb_map_record* records, const long long* seg, const long long* gt_count, int nc,
                     int T, const double* recall_thr, int R, double* precision, double* recall, void* ws,
                     size_t ws_bytes, int* status, void* stream);

/* ------------------------------------------------------------------------------------------
 * COCO bbox summary (pycocotools 2.0 COCOeval.evaluateImg + accumulate with area ranges and per-(image, category)
 *   maxDets, no crowd).  Detections, ground truths, classes, status bits and the IoU are yb_map_match's.
 *   area of a ground truth = (x2-x1)*(y2-y1) of its fp64 corners; of a detection the same on its fp32 corners
 *     widened to fp64.  An object is outside range a iff area < area_rng[2a] || area > area_rng[2a+1]
 *     (an area equal to a bound is inside; a NaN area is never outside).
 * Stage 1, yb_coco_match, once per batch, one CTA per (image, area range):
 *   per image, class, range a and threshold t (thr = min(iou_thr[t], 1-1e-10)): a ground truth outside range a
 *     is ignored; each detection in keep order takes the not yet taken ground truth of its class that is best by
 *     (not ignored first, higher IoU, later index) among those with IoU >= thr (COCO's ignored-last order with its
 *     `break` and `iou < best: continue`).  Matched to an ignored one -> ignored, else TP; unmatched -> ignored
 *     when the detection is outside range a, else FP.  A NaN IoU never matches (pycocotools' `iou < best` would let
 *     it through: the one deliberate departure).
 *   rank = number of earlier detections of the same image and class (saturating at 65535); COCO's dt[:maxDet] is
 *     rank < maxDet, since a detection's matching depends only on earlier ones of its image and class.
 *   records (B, min(max_det,cap)) receive {score, class, rank, TP bit t of tp[a], ignored bit t of ig[a]}; unused
 *     slots have class -1; tp/ig of ranges >= A are 0.
 *   gt_count (A, nc) int64 += ground truths per range and class that are not ignored (zeroed by the caller).
 *   area_rng: HOST array of A <= YB_COCO_MAX_A (lo, hi) pairs; nc * 4 bytes of class counters, the ground truths
 *   and the thresholds' taken bitmaps must fit one CTA's shared memory (YB_EINVAL otherwise).
 * Between the stages the CALLER sorts the records as for yb_map_precision (seg (nc+1) as there).
 * Stage 2, yb_coco_precision, once per evaluation, one CTA per (class, range), the M maxDets side by side:
 *   a record counts for maxDets[m] iff rank < maxDets[m]; npig = gt_count[a][c]; ignored records count as neither TP
 *   nor FP; tp, fp cumulative (doubles), rc = tp / npig, pr = tp / (fp + tp + 2^-52);
 *   precision[t][r][c][a][m] = max of pr over positions with rc >= recall_thr[r] (0 if none),
 *   recall[t][c][a][m] = rc at the end (0 without detections); both -1 when npig == 0 (COCOeval.eval's layout).
 *   max_dets: HOST array of 1 <= M <= YB_COCO_MAX_M values in [1, 65535].  recall_thr must be ascending;
 *   T*R*M*8 + R*8 bytes of shared memory must fit one CTA.
 *   *status |= YB_MAP_INCONSISTENT when a class and range has more TPs than ground truths.
 * ---------------------------------------------------------------------------------------- */
#define YB_COCO_MAX_A 4
#define YB_COCO_MAX_M 4
typedef struct yb_coco_record {
    float score;
    int32_t cls;      /* -1: unused slot */
    uint16_t rank;    /* among the image's detections of the same class, saturating */
    uint16_t pad;
    uint16_t tp[YB_COCO_MAX_A];   /* bit t: TP at iou_thr[t] in area range a */
    uint16_t ig[YB_COCO_MAX_A];   /* bit t: ignored at iou_thr[t] in area range a */
    uint32_t pad2;    /* 32 bytes */
} yb_coco_record;

int yb_coco_match(const float* boxes, const float* scores, const int64_t* classes, const int64_t* keep,
                  const int* n_keep, int B, int cap, int max_det, const double* labels, const int* n_gt,
                  const double* letterbox, int max_gt, int nc, const double* iou_thr, int T,
                  const double* area_rng, int A, yb_coco_record* records, long long* gt_count, int* status,
                  void* stream);
int yb_coco_precision(const yb_coco_record* records, const long long* seg, const long long* gt_count, int nc,
                      int A, int T, const double* recall_thr, int R, const int* max_dets, int M,
                      double* precision, double* recall, int* status, void* stream);

/* ------------------------------------------------------------------------------------------
 * Validation report (confusion matrix, images per class, confidence histograms of the P/R/F1 curves)
 *   yb_report_match, once per batch, after yb_map_match on the same batch and stream, one CTA per image.
 *   Detections, ground truths (corners, classes, nc == 1 -> class 0), the IoU and the status bits are yb_map_match's;
 *   records are the (B, min(max_det,cap)) records yb_map_match just wrote for this batch.
 *   Confusion matrix (nc+1, nc+1) int64, row = predicted class, column = true class, index nc = background:
 *     D = the first min(n_keep[b], max_det) keep entries with a class in [0,nc) and (double)score > cm_conf (a NaN
 *       score never passes); G = the ground truths with a class in [0,nc).  The matching is class-agnostic:
 *     step 1: each d in D picks the g with the largest IoU among those with IoU > cm_iou (strict; a NaN IoU never
 *       matches), the lower g on equal IoU;
 *     step 2: each g picked by some d keeps the d with the largest IoU, the earlier keep position on equal IoU;
 *     confusion[cls_d][cls_g] += 1 per kept pair, [nc][cls_g] += 1 per g nobody picked, [cls_d][nc] += 1 per d not
 *       kept.  (The Ultralytics ConfusionMatrix's layout and two-step unique matching; the tie rules and the
 *       counting of unmatched detections are defined here, not claimed equal to any Ultralytics release.)
 *   images (nc) int64 += 1 per class with at least one ground truth in the image.
 *   det_hist / tp_hist (nc, K) int64: each record with class c >= 0 and a non-NaN score s, with
 *     j = #{k : grid[k] < (double)s} - 1 >= 0, adds 1 to det_hist[c][j], and to tp_hist[c][j] when its TP bit t_curve
 *     is set.  The suffix sum over j >= k is the number of detections (TPs) with score > grid[k].
 *   grid: DEVICE array of K strictly ascending finite doubles (not checked here); cm_conf, cm_iou finite.
 *   The caller zeroes every output once per evaluation; they accumulate over batches.
 *   The ground truths (48 B each), 16 B per detection slot and nc * 4 bytes must fit one CTA's shared memory
 *   (YB_EINVAL otherwise).  *status |= YB_MAP_BAD_CLASS, YB_MAP_NMS_FAILED as yb_map_match.
 * ---------------------------------------------------------------------------------------- */
int yb_report_match(const float* boxes, const float* scores, const int64_t* classes, const int64_t* keep,
                    const int* n_keep, int B, int cap, int max_det, const double* labels, const int* n_gt,
                    const double* letterbox, int max_gt, int nc, const yb_map_record* records, int t_curve,
                    const double* grid, int K, double cm_conf, double cm_iou, long long* confusion,
                    long long* images, long long* det_hist, long long* tp_hist, int* status, void* stream);

/* Per-launch CUDA-event timing for bench.py: when enabled every kernel launch of the library is
 * bracketed by two events on its stream; yb_timing_collect synchronises them, writes
 * "name count total_ms" lines into buf (NUL terminated, truncated to n) and resets. */
void yb_timing_enable(int on);
int yb_timing_collect(char* buf, size_t n);

/* Counters for tests/bench: number of kernel launches this library has enqueued (process wide). */
unsigned long long yb_launch_count(void);

/* Self-test of the batched sigmoid (tests only; synchronises the stream).  The filter and the long-row decode
 * evaluate the reference's 1/(1+expf(-x)) (train.py:758-759,773-774,1157; ATen's sigmoid) with the IEEE
 * division's own fast path but without its range-check branch.  This runs both forms on the device over
 *   [0] every float y with 2^-126 <= |y| < 2^126 : 1.0f / y against the branch-free reciprocal,
 *   [1] every non-NaN float x whose 1+expf(-x) is inside that range : the two sigmoid forms,
 * and writes the number of differing bit patterns to mismatches_host[0..1] (both must be 0). */
int yb_selftest_sigmoid(unsigned long long* mismatches_host /* [2] */, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* YOLO_B200_H */
