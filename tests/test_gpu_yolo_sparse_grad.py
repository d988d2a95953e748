"""Backward pass of the sparse-target YOLO loss (GetLossFromBoxesAndGrad / b200_yolo_loss_from_boxes_grad).

d loss / d y_pred from the per-image box lists must be bit-identical to the dense training step
GetTargetsBatch + GetLossAndGrad: both use the same target arithmetic, the same ignore decisions, obj = 1 with 0/1 class
rows, and no summation inside a record's gradient.  Each form of the ignore pass (16-byte aligned device y_pred: lean
filter + exact pass; a 4-byte offset: single kernel) must match its dense counterpart.  The argument checks at the end run
without a device.
"""
import ctypes

import numpy as np
import pytest

from test_gpu_core import _t, assert_bits_equal
from test_gpu_yolo_loss import _offset_copy
from test_gpu_yolo_shapes import BOX_CASES, _anchors, _heads, _plant, _rng

F = np.float32
LOSS_RTOL = 1e-4
gpu = pytest.mark.gpu

# (image_wh, C, B, iou_type, target anchors normalised by the image size)
CASES = [((416, 416), 80, 3, "ciou", False), ((608, 608), 80, 2, "iou", False), ((96, 96), 80, 4, "diou", True)] + \
        [c + (False,) for c in BOX_CASES]


def _case_id(c):
    return "%dx%d-C%d-B%d-%s" % (c[0] + c[1:4]) + ("-normalised" if c[4] else "")


def _inputs(case):
    """Ragged boxes with a triple collision in image 0 (all three dropped), image 1 without boxes when B > 2 and an
    out-of-range class on the last box; the oracle's dense targets; heads with a prediction planted on every target."""
    from oracle import yolo as oy
    from tfmv_b200 import synth
    image_wh, C, B, _, normalised = case
    rng = _rng("sparse-grad", case)
    anc = _anchors(3)
    tanc = anc / F(image_wh[0]) if normalised else anc
    boxes, classes, off = synth.gt_batch(rng, B, image_wh, max_boxes=40, classes=C, min_boxes=3)
    boxes[1] = boxes[0]
    boxes[2] = boxes[0]
    classes[-1] = C + 5
    if B > 2:
        keep = np.ones(len(boxes), bool)
        keep[off[1]:off[2]] = False
        cnt = np.diff(off)
        cnt[1] = 0
        boxes, classes, off = boxes[keep], classes[keep], np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    y_true = [np.stack(t, 0) for t in zip(*[oy.get_targets(boxes[off[b]:off[b + 1]], classes[off[b]:off[b + 1]], tanc, image_wh, C)
                                             for b in range(B)])]
    y_pred = _heads(rng, B, image_wh, 3, C)
    _plant(rng, y_true, y_pred, anc, image_wh[::-1])
    return boxes, classes, off, y_true, y_pred, anc, tanc


def _layout(heads, layout):
    if layout == "offset":
        return [_offset_copy(h) for h in heads]
    if layout == "pinned":
        return [h.cpu().pin_memory() for h in heads]
    assert all(h.data_ptr() % 16 == 0 for h in heads)
    return heads


def _dense_step(classes, boxes, off, dp, image_wh, anc, tanc, C, iou_type, cuda):
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossAndGrad
    y_true = DataGenerator(C, tanc, image_wh).GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda))
    return GetLossAndGrad(y_true, dp, image_wh, anc, 0.5, iou_type)


@gpu
@pytest.mark.parametrize("layout", ["aligned", "offset", "pinned"])
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_grad_bits_equal_dense_training_step(lib, cuda, case, layout):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, y_true, y_pred, anc, tanc = _inputs(case)
    dp = _layout([_t(h, cuda) for h in y_pred], layout)
    loss, grads = GetLossFromBoxesAndGrad(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), dp, image_wh, anc, C, 0.5, iou_type,
                                          target_anchors=tanc)
    want_loss, want = _dense_step(classes, boxes, off, dp, image_wh, anc, tanc, C, iou_type, cuda)
    for l in range(3):
        assert grads[l].shape == dp[l].shape and grads[l].is_cuda
        assert_bits_equal(grads[l].cpu().numpy(), want[l].cpu().numpy())
    assert abs(float(loss) - float(want_loss)) <= 1e-6 * abs(float(want_loss))


@gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_grad_matches_oracle(lib, cuda, case):
    """Against the oracle's get_targets -> get_loss_grad; non-object records carry a gradient only in the conf channel."""
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, y_true, y_pred, anc, tanc = _inputs(case)
    _, _, want_ign = oy.get_loss(y_true, y_pred, image_wh, anc, 0.5, iou_type, return_ignore=True)
    assert 0 < int(want_ign.sum()) < want_ign.size   # the planted predictions clear some ignore bits
    want_loss, want = oy.get_loss_grad(y_true, y_pred, image_wh, anc, 0.5, iou_type)
    loss, parts, grads = GetLossFromBoxesAndGrad(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), [_t(h, cuda) for h in y_pred],
                                                 image_wh, anc, C, 0.5, iou_type, target_anchors=tanc, return_parts=True)
    assert tuple(parts.shape) == (3, 4)
    assert abs(float(loss) - float(want_loss)) <= LOSS_RTOL * abs(float(want_loss)), (float(loss), float(want_loss))
    for l in range(3):
        g = grads[l].cpu().numpy().reshape(want[l].shape)
        np.testing.assert_allclose(g, want[l], rtol=1e-4, atol=1e-7)
        nobj = y_true[l][..., 4] == 0
        assert np.count_nonzero(np.delete(g[nobj], 4, axis=-1)) == 0
        assert np.count_nonzero(g[~nobj][:, 5:]) > 0 or not (~nobj).any()


@gpu
@pytest.mark.parametrize("layout", ["aligned", "offset"])
def test_batch_without_boxes(lib, cuda, layout):
    """No boxes at all: only the conf channel is non-zero, as the dense step and the oracle on an all-zero y_true."""
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad
    image_wh, C, B = (96, 96), 80, 3
    anc = _anchors(3)
    y_pred = _heads(_rng("sparse-grad-empty"), B, image_wh, 3, C)
    boxes, classes, off = np.zeros((0, 4), F), np.zeros((0,), np.int32), np.zeros(B + 1, np.int32)
    dp = _layout([_t(h, cuda) for h in y_pred], layout)
    loss, grads = GetLossFromBoxesAndGrad(classes, boxes, off, dp, image_wh, anc, C, 0.5, "ciou")
    want_loss, want = _dense_step(classes, boxes, off, dp, image_wh, anc, anc, C, "ciou", cuda)
    zeros = [np.zeros((B, h.shape[1], h.shape[2], 3, 5 + C), F) for h in y_pred]
    o_loss, o_grads = oy.get_loss_grad(zeros, y_pred, image_wh, anc, 0.5, "ciou")
    assert abs(float(loss) - float(o_loss)) <= LOSS_RTOL * abs(float(o_loss))
    for l in range(3):
        g = grads[l].cpu().numpy()
        assert_bits_equal(g, want[l].cpu().numpy())
        g = g.reshape(o_grads[l].shape)
        np.testing.assert_allclose(g, o_grads[l], rtol=1e-4, atol=1e-7)
        assert np.count_nonzero(np.delete(g, 4, axis=-1)) == 0


@gpu
def test_sharded_calls_concatenate_to_the_full_batch(lib, cuda):
    """Data parallel: images [0,k) and [k,B) in two calls with batch_divisor = B give the full call's gradients bit for
    bit (no exchange needed); combine_loss_parts of the two parts gives the full loss."""
    import torch
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad, combine_loss_parts
    case = ((416, 416), 80, 4, "ciou", False)
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, _, y_pred, anc, tanc = _inputs(case)
    dp = [_t(h, cuda) for h in y_pred]
    loss, grads = GetLossFromBoxesAndGrad(classes, boxes, off, dp, image_wh, anc, C, 0.5, iou_type)
    k = 1
    shards = [(0, k), (k, B)]
    got, parts = [[], [], []], []
    for lo, hi in shards:
        s_off = (off[lo:hi + 1] - off[lo]).astype(np.int32)
        sb, sc = boxes[off[lo]:off[hi]], classes[off[lo]:off[hi]]
        s_loss, s_parts, s_grads = GetLossFromBoxesAndGrad(sc, sb, s_off, [h[lo:hi].clone() for h in dp], image_wh, anc, C, 0.5,
                                                           iou_type, batch_divisor=B, return_parts=True)
        parts.append(s_parts)
        for l in range(3):
            got[l].append(s_grads[l])
    for l in range(3):
        assert_bits_equal(torch.cat(got[l], 0).cpu().numpy(), grads[l].cpu().numpy())
    total = combine_loss_parts(parts[0] + parts[1])
    assert abs(float(total) - float(loss)) <= 1e-6 * abs(float(loss))


@gpu
def test_graph_replay_after_rewriting_the_boxes(lib, cuda):
    """Captured once, replayed after boxes / classes / offsets are rewritten in place (same total): equals an eager call."""
    from tfmv_b200 import runtime, synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad
    case = ((416, 416), 80, 3, "ciou", False)
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, _, y_pred, anc, _ = _inputs(case)
    dp = [_t(h, cuda) for h in y_pred]
    bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    step = runtime.capture(lambda: GetLossFromBoxesAndGrad(cd, bd, od, dp, image_wh, anc, C, 0.5, iou_type))
    rng = _rng("sparse-grad-replay")
    total = len(boxes)
    b2, c2, _ = synth.gt_batch(rng, 1, image_wh, max_boxes=total, min_boxes=total, classes=C)
    o2 = np.concatenate([[0], np.sort(rng.integers(0, total + 1, B - 1)), [total]]).astype(np.int32)
    assert not np.array_equal(o2, off)
    bd.copy_(_t(b2, cuda))
    cd.copy_(_t(c2, cuda))
    od.copy_(_t(o2, cuda))
    r_loss, r_grads = step()
    e_loss, e_grads = GetLossFromBoxesAndGrad(c2, b2, o2, dp, image_wh, anc, C, 0.5, iou_type)
    assert float(r_loss) == float(e_loss)
    for l in range(3):
        assert_bits_equal(r_grads[l].cpu().numpy(), e_grads[l].cpu().numpy())


def _call_args(anc, img, hw, B, C, total, y_pred, out_grad, workspace, ws_bytes, loss_ptr, parts_ptr, stream, boxes=0,
               classes=0, offsets=0):
    return (boxes, classes, offsets, total, anc.ctypes.data_as(ctypes.c_void_p), y_pred, hw, B, 3, C,
            anc.ctypes.data_as(ctypes.c_void_p), img.ctypes.data_as(ctypes.c_void_p), ctypes.c_float(0.5), 2, 0,
            ctypes.c_float(B), parts_ptr, loss_ptr, out_grad, workspace, ws_bytes, stream)


@gpu
def test_workspace_size_and_refusals_enqueue_nothing(lib, cuda):
    """b200_yolo_loss_from_boxes_workspace_bytes suffices for the backward and one byte less is refused; a refused call
    (short workspace, misaligned gradient level) leaves every output untouched, for the dense entry too."""
    import torch
    from tfmv_b200 import _tensors as T
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad
    case = ((96, 96), 80, 3, "ciou", False)
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, y_true, y_pred, anc, _ = _inputs(case)
    dp = [_t(h, cuda) for h in y_pred]
    bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    hw = (ctypes.c_int32 * 6)(*[d for h in dp for d in (h.shape[1], h.shape[2])])
    ws_bytes = lib.b200_yolo_loss_from_boxes_workspace_bytes(hw, B, 3, len(boxes))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=cuda)
    loss, grads = GetLossFromBoxesAndGrad(cd, bd, od, dp, image_wh, anc, C, 0.5, iou_type, workspace=ws)
    loss2, grads2 = GetLossFromBoxesAndGrad(cd, bd, od, dp, image_wh, anc, C, 0.5, iou_type)
    assert float(loss) == float(loss2)
    for l in range(3):
        assert_bits_equal(grads[l].cpu().numpy(), grads2[l].cpu().numpy())
    img = np.asarray(image_wh, F)
    ancf = np.ascontiguousarray(anc, F)
    pp = (ctypes.c_void_p * 3)(*[h.data_ptr() for h in dp])
    out = [torch.full_like(h, 7.0) for h in dp]
    gp = (ctypes.c_void_p * 3)(*[g.data_ptr() for g in out])
    parts = torch.full((3, 4), 7.0, device=cuda)
    lo = torch.full((), 7.0, device=cuda)
    args = lambda g, n: _call_args(ancf, img, hw, B, C, len(boxes), pp, g, ws.data_ptr(), n, lo.data_ptr(), parts.data_ptr(),
                                   T.stream_ptr(), bd.data_ptr(), cd.data_ptr(), od.data_ptr())
    assert lib.b200_yolo_loss_from_boxes_grad(*args(gp, ws_bytes - 1)) == -2
    assert b"workspace" in lib.b200_last_error()
    gbad = (ctypes.c_void_p * 3)(gp[0], gp[1] + 4, gp[2])
    assert lib.b200_yolo_loss_from_boxes_grad(*args(gbad, ws_bytes)) == -1
    assert b"grad level 1" in lib.b200_last_error()
    # the dense entry checks its gradient levels before the forward is queued, with the same code and message
    tp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in (_t(y, cuda) for y in y_true)])
    dws = torch.empty((lib.b200_yolo_loss_workspace_bytes(hw, B, 3),), dtype=torch.uint8, device=cuda)
    assert lib.b200_yolo_loss_grad(tp, pp, hw, B, 3, C, ancf.ctypes.data_as(ctypes.c_void_p), img.ctypes.data_as(ctypes.c_void_p),
                                   ctypes.c_float(0.5), 2, 0, ctypes.c_float(B), parts.data_ptr(), lo.data_ptr(), gbad,
                                   dws.data_ptr(), dws.numel(), T.stream_ptr()) == -1
    assert b"b200_yolo_loss_grad: grad level 1 null or not 16-byte aligned" in lib.b200_last_error()
    torch.cuda.synchronize()
    assert float(lo) == 7.0 and bool((parts == 7.0).all())
    assert all(bool((g == 7.0).all()) for g in out)


def test_grad_entry_refuses_bad_arguments_without_a_device(lib):
    """Null y_pred, null out_grad, a null y_pred level and a null or misaligned gradient level are refused with
    B200_ERR_BAD_ARG before anything touches the device."""
    from tfmv_b200 import synth
    anc = np.ascontiguousarray(synth.yolo_anchors(), F)
    img = np.asarray([416, 416], F)
    hw = (ctypes.c_int32 * 6)(13, 13, 26, 26, 52, 52)
    fake = 1 << 20     # 256-byte aligned and never dereferenced: every refusal below happens before the first CUDA call
    P3 = ctypes.c_void_p * 3
    call = lambda y_pred, out_grad: lib.b200_yolo_loss_from_boxes_grad(
        *_call_args(anc, img, hw, 2, 80, 10, y_pred, out_grad, fake, 1 << 40, fake, 0, 0, fake, fake, fake))
    assert call(None, P3(fake, fake, fake)) == -1
    assert call(P3(fake, fake, fake), None) == -1
    assert b"null out_grad" in lib.b200_last_error()
    assert call(P3(fake, 0, fake), P3(fake, fake, fake)) == -1
    assert b"bad level 1" in lib.b200_last_error()
    assert call(P3(fake, fake, fake), P3(fake, 0, fake)) == -1
    assert b"b200_yolo_loss_from_boxes_grad: grad level 1" in lib.b200_last_error()
    assert call(P3(fake, fake, fake), P3(fake, fake, fake + 4)) == -1
    assert b"grad level 2" in lib.b200_last_error()
