"""Every op that reads head tensors checks all scales' shapes on the host before it touches the device.

The library receives pointers and the sizes of one descriptor (B of scale 0, A of the first anchor set, rows of
5+nc), so a shape the host does not check becomes a read past the end of a head.  Here each entry point gets CPU
tensors with one mismatch and must raise ValueError naming the scale.  ops._device and the library loader are
replaced by functions that raise RuntimeError: a missing check fails the test and can never launch a kernel."""
import pytest
import torch

from yolo_from_scratch_b200 import dist, ops

B, NC, A, GRIDS = 2, 2, 3, (4, 2)
ANCH = [torch.tensor([[10., 13.], [16., 30.], [33., 23.]]), torch.tensor([[30., 61.], [62., 45.], [59., 119.]])]
W = ops.MULTISCALE_OBJ_WEIGHTS[:2]
MISMATCHES = ["row", "head A", "batch", "A across scales", "targets"]


@pytest.fixture(autouse=True)
def no_device(monkeypatch):
    def reached(*args, **kwargs):
        raise RuntimeError("reached the device")
    monkeypatch.setattr(ops, "_device", reached)
    monkeypatch.setattr(ops._lib, "lib", reached)


def to_nchw(h):
    return h.permute(0, 3, 4, 1, 2).reshape(h.shape[0], -1, h.shape[1], h.shape[2])


def case(bad=None):
    """Heads (reference layout), dense targets, anchors and label lists of two scales; `bad` breaks scale 1 (the
    label lists: their batch)."""
    heads = [torch.zeros(B, g, g, A, 5 + NC) for g in GRIDS]
    tgts = [torch.zeros(B, g, g, A, 5 + NC) for g in GRIDS]
    anchors = list(ANCH)
    n_img, g = B, GRIDS[1]
    if bad == "row":
        heads[1] = torch.zeros(B, g, g, A, 4 + NC)
    elif bad == "head A":
        anchors[1] = ANCH[1][:A - 1]
    elif bad == "batch":
        heads[1], tgts[1] = torch.zeros(B - 1, g, g, A, 5 + NC), torch.zeros(B - 1, g, g, A, 5 + NC)
    elif bad == "A across scales":
        heads[1], tgts[1] = torch.zeros(B, g, g, A - 1, 5 + NC), torch.zeros(B, g, g, A - 1, 5 + NC)
        anchors[1] = ANCH[1][:A - 1]
    elif bad == "targets":
        tgts[1] = torch.zeros(B, g + 1, g + 1, A, 5 + NC)
        n_img = B + 1
    labels = ops.PackedLabels(torch.zeros(n_img, 1, 5, dtype=torch.float64), torch.zeros(n_img, dtype=torch.int32),
                              torch.zeros(n_img, 5, dtype=torch.float64), 64)
    return heads, tgts, anchors, labels


def nchw(hs):
    return [to_nchw(h) for h in hs]


# name -> (call(heads, targets, anchors, labels), takes targets: "dense", "labels" or None)
ENTRIES = {
    "yolo_loss_multiscale": (lambda h, t, a, lab: ops.yolo_loss_multiscale(h, t, a, NC), "dense"),
    "yolo_loss_multiscale_nchw": (lambda h, t, a, lab: ops.yolo_loss_multiscale_nchw(nchw(h), t, a, NC), "dense"),
    "yolo_loss_multiscale_labels": (lambda h, t, a, lab: ops.yolo_loss_multiscale_labels(h, lab, a, NC), "labels"),
    "yolo_loss_multiscale_nchw_labels": (lambda h, t, a, lab: ops.yolo_loss_multiscale_nchw(nchw(h), lab, a, NC),
                                         "labels"),
    "yolo_loss_multiscale_sharded": (lambda h, t, a, lab: dist.yolo_loss_multiscale_sharded(h, t, a, NC), "dense"),
    "loss_forward_backward": (lambda h, t, a, lab: ops.loss_forward_backward(h, t, a, NC, W, [True] * 2), "dense"),
    "loss_forward_backward_nchw": (lambda h, t, a, lab: ops.loss_forward_backward(
        nchw(h), t, a, NC, W, [True] * 2, layout=ops.LAYOUT_NCHW), "dense"),
    "loss_forward_backward_labels": (lambda h, t, a, lab: ops.loss_forward_backward(
        h, None, a, NC, W, [True] * 2, sparse=lab), "labels"),
    "loss_forward_backward_nchw_labels": (lambda h, t, a, lab: ops.loss_forward_backward(
        nchw(h), None, a, NC, W, [True] * 2, sparse=lab, layout=ops.LAYOUT_NCHW), "labels"),
    "filter_candidates": (lambda h, t, a, lab: ops.filter_candidates(h, a, 64, NC), None),
    "filter_candidates_nchw": (lambda h, t, a, lab: ops.filter_candidates(nchw(h), a, 64, NC,
                                                                          layout=ops.LAYOUT_NCHW), None),
    "filter_candidates_multilabel": (lambda h, t, a, lab: ops.filter_candidates_multilabel(h, a, 64, NC), None),
    "filter_candidates_multilabel_nchw": (lambda h, t, a, lab: ops.filter_candidates_multilabel(
        nchw(h), a, 64, NC, layout=ops.LAYOUT_NCHW), None),
    "detect_batch": (lambda h, t, a, lab: ops.detect_batch(h, a, 64, NC), None),
    "detect_batch_nchw": (lambda h, t, a, lab: ops.detect_batch_nchw(nchw(h), a, 64, NC), None),
    "detect_batch_multilabel": (lambda h, t, a, lab: ops.detect_batch(h, a, 64, NC, multi_label=True), None),
    "eval_counts": (lambda h, t, a, lab: ops.eval_counts(h, t, a), "dense"),
}


@pytest.mark.parametrize("entry,bad", [(e, b) for e in ENTRIES for b in MISMATCHES
                                       if b != "targets" or ENTRIES[e][1] is not None])
def test_mismatch_raises_before_the_device(entry, bad):
    call, takes = ENTRIES[entry]
    scale = 0 if (bad == "targets" and takes == "labels") else 1
    with pytest.raises(ValueError, match=f"scale {scale}"):
        call(*case(bad))


@pytest.mark.parametrize("entry", list(ENTRIES))
def test_valid_shapes_pass_the_checks(entry):
    """The same calls with matching shapes get past staging's checks, to the (replaced) device."""
    with pytest.raises(RuntimeError, match="reached the device"):
        ENTRIES[entry][0](*case())


@pytest.mark.parametrize("bad", ["row", "head A", "targets"])
def test_single_scale_entry_points(bad):
    heads, tgts, anchors, _ = case()
    h, t, a = heads[0], tgts[0], anchors[0]
    if bad == "row":
        h = torch.zeros(B, 4, 4, A, 4 + NC)
    elif bad == "head A":
        a = a[:A - 1]
    else:
        t = torch.zeros(B, 5, 5, A, 5 + NC)
    with pytest.raises(ValueError, match="scale 0"):
        ops.yolo_loss(h, t, a, NC)
    if bad == "head A":
        with pytest.raises(ValueError, match="scale 0"):
            ops.decode_predictions(h, a)


def test_scale_count_and_anchor_shape():
    heads, tgts, anchors, _ = case()
    with pytest.raises(ValueError, match="scales"):
        ops.filter_candidates([], anchors, 64, NC)
    with pytest.raises(ValueError, match="scales"):
        ops.filter_candidates(heads * 3, anchors * 3, 64, NC)
    with pytest.raises(ValueError, match="scale 1"):
        ops.filter_candidates(heads, anchors[:1], 64, NC)
    with pytest.raises(ValueError, match="scale 1"):
        ops.filter_candidates(heads, [anchors[0], anchors[1].reshape(-1)], 64, NC)
