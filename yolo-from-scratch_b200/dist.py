"""Data-parallel use of the hot path (SURVEY 8e): the path shards by image.

Decode, candidate filter, NMS and target assignment are independent per image: no collective.
The loss terms are means over the GLOBAL batch (train.py:710, :823, :827), so every rank
produces S x {sum(1-CIoU), n_pos, sum BCE_obj, sum BCE_cls} for its images and one all-reduce(sum)
of those S*4 doubles (96 bytes for three scales) gives the global values; the objectness normaliser
B_global*H*W*A is known without communication and the positive rows' gradients are scaled by the
reduced 1/n_pos afterwards (yb_loss_finalize).  One process per GPU, torch.distributed / NCCL.

Evaluation shards the same way: every rank matches its own images (DetectionMAP / COCODetectionEval /
DetectionReport.update), and compute(group) merges the ranks' records and counts with gather_eval_state before
the one sort and precision pass (DESIGN §3.11).
"""
from typing import Tuple

import torch

# The configuration words of gather_eval_state's header, which must be equal on every rank.  gather_eval_state
# appends the record width and the number of counts, which size its own collectives.
FINGERPRINT_FIELDS = ("metric", "nc", "T", "R", "A", "M", "K", "max_det", "crc")
_CHECKED = FINGERPRINT_FIELDS + ("record width", "counts")
_ROWS, _GT_TOTAL, _IMAGES_TOTAL, _STATUS = range(len(_CHECKED), len(_CHECKED) + 4)


def shard_range(n_images: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous block of images owned by `rank` (first n % world ranks get one extra)."""
    if not 0 <= rank < world:
        raise ValueError("rank out of range")
    base, extra = divmod(n_images, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def allreduce_partials(partials: torch.Tensor, group=None) -> torch.Tensor:
    """In-place sum of the (S*4,) float64 partial sums over the ranks; a single small collective."""
    import torch.distributed as dist
    if partials.dtype != torch.float64:
        raise TypeError("partials must be float64")
    dist.all_reduce(partials, op=dist.ReduceOp.SUM, group=group)
    return partials


def global_batch(local_batch: int, group=None) -> int:
    """Sum of the ranks' local batch sizes (ranks may own different numbers of images)."""
    import torch.distributed as dist
    t = torch.tensor([local_batch], dtype=torch.int64)
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return int(t.item())


def yolo_loss_multiscale_sharded(predictions, targets, anchors_list, num_classes=1, group=None):
    """yolo_loss_multiscale (train.py:840-886) over a batch sharded by image across the ranks of
    `group`: every rank passes ITS images and receives the GLOBAL losses; `total.backward()` leaves
    on every rank exactly the gradient rows of its own images of the global-batch loss."""
    from . import ops
    S = min(len(predictions), len(targets), len(anchors_list), len(ops.MULTISCALE_OBJ_WEIGHTS))
    return ops._loss_common(list(predictions[:S]), list(targets[:S]), list(anchors_list[:S]), num_classes,
                            ops.MULTISCALE_OBJ_WEIGHTS[:S], group=group)


def gather_eval_state(fingerprint, records, counts, gt_total, images_total, status, group=None):
    """Merge an evaluation metric's accumulated state over the ranks of `group`.  A collective: every rank calls it.

    fingerprint: len(FINGERPRINT_FIELDS) ints describing the metric's configuration; records (n, W) int32, the local
    records in image order (word 1 is the class, -1 for an unused row); counts: the fixed-size int64 counts (any
    shape); gt_total, images_total: host ints; status: (1,) int32 status word.  The tensors live on one device, CUDA
    for NCCL, CUDA or CPU for gloo.

    Step 1 gathers a fixed-size int64 header (the fingerprint, W, counts.numel(), n, gt_total, images_total, status)
    and reads it on the host, the one synchronisation here.  If any rank's configuration words differ from rank 0's,
    every rank raises ValueError before any variable-size collective, so none is left waiting.  Step 2 gathers the
    counts and, unless every rank has n = 0, the records padded to the largest n with rows of -1 (class -1).

    Returns (records, counts, gt_total, images_total, status) as one process holding every rank's updates would
    hold them: the records of rank 0, 1, ... concatenated without the padding, counts summed (counts' shape),
    gt_total and images_total summed, status the OR of the words, as a (1,) tensor like `status`.  The inputs are
    not changed."""
    import torch.distributed as dist
    fingerprint = [int(v) for v in fingerprint]
    if len(fingerprint) != len(FINGERPRINT_FIELDS):
        raise ValueError(f"fingerprint needs the {len(FINGERPRINT_FIELDS)} words {FINGERPRINT_FIELDS}, "
                         f"got {len(fingerprint)}")
    if records.dim() != 2 or records.dtype != torch.int32 or counts.dtype != torch.int64:
        raise TypeError("records must be (n, W) int32 and counts int64")
    world = dist.get_world_size(group)
    n, width = records.shape
    header = torch.tensor(fingerprint + [width, counts.numel(), n, int(gt_total), int(images_total), 0],
                          dtype=torch.int64).to(records.device)
    header[_STATUS:].copy_(status.reshape(1))   # on the device: the status word is not read before the exchange
    headers = [torch.empty_like(header) for _ in range(world)]
    dist.all_gather(headers, header, group=group)
    h = torch.stack(headers).cpu()
    for r in range(1, world):
        diff = [name for i, name in enumerate(_CHECKED) if h[r, i] != h[0, i]]
        if diff:
            raise ValueError(f"evaluation configurations differ across ranks: rank {r} and rank 0 disagree on "
                             f"{', '.join(diff)}; every rank must build the metric with the same arguments")
    parts = [torch.empty_like(counts) for _ in range(world)]
    dist.all_gather(parts, counts.contiguous(), group=group)
    counts = torch.stack(parts).sum(0)
    rows = h[:, _ROWS].tolist()
    if max(rows) == 0:
        merged = records.new_empty((0, width))
    else:
        padded = records.new_full((max(rows), width), -1)
        padded[:n] = records
        parts = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(parts, padded, group=group)
        merged = torch.cat([p[:r] for p, r in zip(parts, rows)])
    word = 0
    for s in h[:, _STATUS].tolist():
        word |= s
    return (merged, counts, int(h[:, _GT_TOTAL].sum()), int(h[:, _IMAGES_TOTAL].sum()),
            torch.tensor([word], dtype=status.dtype).to(status.device))
