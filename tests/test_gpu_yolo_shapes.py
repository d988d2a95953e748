"""YOLO parity at rectangular images, A != 3 anchors per level and C != 80 classes, against the oracle.

The other YOLO tests run square images (H == W at every level, img_w == img_h) with A = 3, so a kernel that swaps a
width for a height passes them.  The cases here cross rectangular sizes, one of them transposed, grids that do not
double from level to level and a level with W == 1, with C in {1, 2, 3, 20, 80} (record sizes 5 + C = 6 and 7 take
the ignore pass's scalar load, 8, 25 and 85 the aligned one) and A in {1, 2, 3, 5, 8}.  The CPU tests at the end check
on the oracle alone that every rectangular case can tell (w, h) from (h, w), so that the GPU cases mean something.
"""
import zlib

import numpy as np
import pytest

from test_gpu_core import _t, assert_bits_equal
from test_gpu_yolo_decode import _check_image
from test_gpu_yolo_loss import _offset_copy

F = np.float32
LOSS_RTOL = 1e-4
gpu = pytest.mark.gpu


def _grids(image_wh):
    """(h, w) of the three levels, coarsest first (DataGenerator.layers_hw)."""
    return [(int(image_wh[1]) // s, int(image_wh[0]) // s) for s in (32, 16, 8)]


def _rng(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def _anchors(A):
    """(3, A, 2) pixel anchors, coarsest level first: the COCO set for A = 3, else seeded non-square anchors of 0.7 to 4
    strides."""
    from tfmv_b200 import synth
    if A == 3:
        return synth.yolo_anchors().astype(F)
    rng = _rng("anchors", A)
    s = np.array([32, 16, 8], np.float64).reshape(3, 1, 1)
    return np.round(s * np.exp(rng.uniform(np.log(0.7), np.log(4.0), (3, A, 2)))).astype(F)


def _heads(rng, B, image_wh, A, C, sigma=1.0):
    return [rng.standard_normal((B, h, w, A * (5 + C)), dtype=F) * F(sigma) for h, w in _grids(image_wh)]


def _planted_targets(rng, B, image_wh, A, C, max_objects=40):
    """Dense y_true written record by record (defined for any A): obj = 1, centre inside the record's cell, positive
    w and h, one-hot class.  In a batch of more than two images the last one has no ground truth."""
    y_true = [np.zeros((B, h, w, A, 5 + C), F) for h, w in _grids(image_wh)]
    for b in range(B if B <= 2 else B - 1):
        for _ in range(int(rng.integers(1, max_objects + 1))):
            l = int(rng.integers(0, 3))
            h, w = y_true[l].shape[1:3]
            gy, gx, a = int(rng.integers(0, h)), int(rng.integers(0, w)), int(rng.integers(0, A))
            rec = y_true[l][b, gy, gx, a]
            rec[:] = 0
            rec[0] = (gx + rng.uniform(0.02, 0.98)) / w
            rec[1] = (gy + rng.uniform(0.02, 0.98)) / h
            rec[2:4] = np.exp(rng.uniform(np.log(0.02), np.log(0.6), 2))
            rec[4] = 1
            rec[5 + int(rng.integers(0, C))] = 1
    return y_true


def _plant(rng, y_true, y_pred, anc, wh_div):
    """Puts a prediction on top of every target (IoU near 1, so that the ignore mask has zeros): same cell, an anchor of
    that cell, width logit log(t_w * wh_div[0] / anchor_w).  wh_div is the divisor of the predicted width and height:
    image_wh[::-1] for GetLoss (tyu:57), (W, H) for Yolov4Loss."""
    div = np.asarray(wh_div, F)
    for l in range(3):
        yt = y_true[l]
        yp = y_pred[l].reshape(yt.shape)
        h, w, A = yt.shape[1:4]
        bb, gy, gx, aa = np.nonzero(yt[..., 4] > 0)
        for k in range(len(bb)):
            t = yt[bb[k], gy[k], gx[k], aa[k]]
            a2 = (aa[k] + k) % A
            fx = min(max(float(t[0]) * w - gx[k], 1e-3), 1 - 1e-3)
            fy = min(max(float(t[1]) * h - gy[k], 1e-3), 1 - 1e-3)
            s = 1.0 + rng.normal(0, 0.05)
            rec = yp[bb[k], gy[k], gx[k], a2]
            rec[0], rec[1] = np.log(fx / (1 - fx)), np.log(fy / (1 - fy))
            rec[2:4] = np.log(np.maximum(t[2:4] * div * F(s), 1e-3) / anc[l][a2])


# ------------------------------------------------------------------------------------------------------------------------
# dense loss cases: (image_wh, A, C, B, iou_type, thr)
LOSS_CASES = [
    ((416, 256), 3, 80, 2, "ciou", 0.5),
    ((256, 416), 3, 1, 3, "iou", 0.5),     # RF 6: scalar record loads
    ((320, 200), 2, 2, 3, "diou", 0.5),    # RF 7; grids 6x10, 12x20, 25x40
    ((40, 96), 1, 20, 4, "ciou", 0.5),     # W == 1 and A == 1: both fast-division constants are 0
    ((416, 256), 5, 3, 2, "iou", 0.5),     # RF 8: aligned record
    ((256, 416), 8, 20, 2, "ciou", 0.5),
    ((320, 200), 3, 80, 2, "ciou", 0.3),   # thr < 0.5: no decode-free filter, exact test only
    ((40, 96), 8, 2, 2, "diou", 0.5),
    ((416, 416), 1, 1, 2, "ciou", 0.5),    # square controls
    ((416, 416), 3, 80, 2, "iou", 0.5),
]
# gradient cases: (image_wh, A, C, B, iou_type)
GRAD_CASES = [((416, 256), 3, 80, 2, "ciou"), ((40, 96), 1, 2, 3, "iou"), ((256, 416), 5, 20, 2, "diou"),
              ((320, 200), 3, 3, 2, "ciou")]
# sparse-target loss cases (A = 3): (image_wh, C, B, iou_type)
BOX_CASES = [((416, 256), 80, 2, "ciou"), ((256, 416), 3, 3, "iou"), ((40, 96), 1, 4, "diou"), ((320, 200), 20, 3, "ciou")]


def _case_id(c):
    return "%dx%d-A%d-C%d-B%d-%s" % (c[0][0], c[0][1], c[1], c[2], c[3], c[4]) + ("-thr%g" % c[5] if len(c) > 5 else "")


def _loss_inputs(case, sigma):
    """y_true, y_pred (wide logits for sigma > 1: boxes of every size, many overlapping), anchors."""
    image_wh, A, C, B = case[:4]
    rng = _rng("loss", case, sigma)
    anc = _anchors(A)
    y_true = _planted_targets(rng, B, image_wh, A, C)
    y_pred = _heads(rng, B, image_wh, A, C, sigma)
    _plant(rng, y_true, y_pred, anc, image_wh[::-1])
    return y_true, y_pred, anc


def _box_inputs(case):
    """Ragged ground truth with a collision in image 0 and an out-of-range class, its oracle targets and planted heads."""
    from oracle import yolo as oy
    from tfmv_b200 import synth
    image_wh, C, B = case[:3]
    rng = _rng("boxes", case)
    anc = _anchors(3)
    boxes, classes, off = synth.gt_batch(rng, B, image_wh, max_boxes=40, classes=C)
    if off[1] >= 2:
        boxes[1] = boxes[0]
    classes[-1] = C + 5
    y_true = [np.stack(t, 0) for t in zip(*[oy.get_targets(boxes[off[b]:off[b + 1]], classes[off[b]:off[b + 1]], anc, image_wh, C)
                                             for b in range(B)])]
    y_pred = _heads(rng, B, image_wh, 3, C)
    _plant(rng, y_true, y_pred, anc, image_wh[::-1])
    return boxes, classes, off, y_true, y_pred, anc


@gpu
@pytest.mark.parametrize("layout", ["aligned", "offset"])
@pytest.mark.parametrize("case", LOSS_CASES, ids=_case_id)
def test_get_loss_shapes(lib, cuda, case, layout):
    """GetLoss in both ignore-pass forms: a 16-byte aligned device y_pred takes the lean filter + exact pass when
    RF >= 8, the same values at a 4-byte offset take the single kernel.  Ignore mask bit-exact, loss parts within 1e-4."""
    import torch
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLoss, _loss_call
    image_wh, A, C, B, iou_type, thr = case
    y_true, y_pred, anc = _loss_inputs(case, 2.5)
    want, want_parts, want_ign = oy.get_loss(y_true, y_pred, image_wh, anc, thr, iou_type, return_ignore=True)
    assert 0 < int(want_ign.sum()) < want_ign.size
    ign = torch.full(want_ign.shape, 7, dtype=torch.uint8, device=cuda)
    dt, dp = [_t(t, cuda) for t in y_true], [_t(t, cuda) for t in y_pred]
    if layout == "offset":
        dp = [_offset_copy(t) for t in dp]
    got, parts = _loss_call(dt, dp, image_wh, anc, thr, iou_type, 0, return_parts=True, ignore_out=ign)
    g = ign.cpu().numpy()
    assert np.array_equal(g, want_ign), "%d ignore bits differ" % int((g != want_ign).sum())
    np.testing.assert_allclose(parts.cpu().numpy(), want_parts, rtol=LOSS_RTOL, atol=1e-6)
    assert abs(float(got) - float(want)) <= LOSS_RTOL * abs(float(want)), (float(got), float(want))
    assert float(GetLoss(dt, dp, image_wh, anc, thr, iou_type)) == float(got)


@gpu
@pytest.mark.parametrize("case", GRAD_CASES, ids=_case_id)
def test_get_loss_and_grad_shapes(lib, cuda, case):
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossAndGrad
    image_wh, A, C, B, iou_type = case
    y_true, y_pred, anc = _loss_inputs(case, 1.0)
    want_loss, want = oy.get_loss_grad(y_true, y_pred, image_wh, anc, 0.5, iou_type)
    got_loss, got = GetLossAndGrad([_t(t, cuda) for t in y_true], [_t(t, cuda) for t in y_pred], image_wh, anc, 0.5, iou_type)
    assert abs(float(got_loss) - float(want_loss)) <= LOSS_RTOL * abs(float(want_loss)), (float(got_loss), float(want_loss))
    for l in range(3):
        g = got[l].cpu().numpy().reshape(want[l].shape)
        np.testing.assert_allclose(g, want[l], rtol=1e-4, atol=1e-7)


@gpu
@pytest.mark.parametrize("case", BOX_CASES, ids=lambda c: "%dx%d-C%d-B%d-%s" % (c[0] + c[1:]))
def test_loss_from_boxes_shapes(lib, cuda, case):
    """GetLossFromBoxes == the oracle's get_targets -> get_loss: the target step keeps image_wh in (w, h) order, the
    loss step reverses it.  Also == the dense GPU path (GetTargetsBatch + GetLoss)."""
    import torch
    from oracle import yolo as oy
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxes, _loss_call
    image_wh, C, B, iou_type = case
    boxes, classes, off, y_true, y_pred, anc = _box_inputs(case)
    want, want_parts, want_ign = oy.get_loss(y_true, y_pred, image_wh, anc, 0.5, iou_type, return_ignore=True)
    assert 0 < int(want_ign.sum()) < want_ign.size
    ign = torch.full(want_ign.shape, 7, dtype=torch.uint8, device=cuda)
    dp = [_t(t, cuda) for t in y_pred]
    got, parts = GetLossFromBoxes(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), dp, image_wh, anc, C, 0.5, iou_type,
                                  return_parts=True, ignore_out=ign)
    g = ign.cpu().numpy()
    assert np.array_equal(g, want_ign), "%d ignore bits differ" % int((g != want_ign).sum())
    np.testing.assert_allclose(parts.cpu().numpy(), want_parts, rtol=LOSS_RTOL, atol=1e-6)
    assert abs(float(got) - float(want)) <= LOSS_RTOL * abs(float(want)), (float(got), float(want))
    dense = DataGenerator(C, anc, image_wh).GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda))
    _, parts_d = _loss_call(dense, dp, image_wh, anc, 0.5, iou_type, 0, return_parts=True)
    np.testing.assert_allclose(parts.cpu().numpy(), parts_d.cpu().numpy(), rtol=1e-6, atol=1e-9)


@gpu
@pytest.mark.parametrize("grid0,C", [((8, 13), 80), ((13, 8), 1), ((3, 1), 20)])
def test_yolov4_loss_rectangular_grids(lib, cuda, grid0, C):
    """Yolov4Loss derives input_shape = grid0 * 32 and divides the predicted width by input_shape[::-1][0] == W."""
    from oracle import yolo as oy
    from tfmv_b200.ai_models.losses.yolo_loss import Yolov4Loss
    image_wh = (grid0[1] * 32, grid0[0] * 32)
    rng = _rng("v4", grid0, C)
    anc = oy.load_anchors_order(oy.COCO_ANCHORS_FLAT.reshape(-1)).astype(F)
    y_true = _planted_targets(rng, 3, image_wh, 3, C)
    y_pred = _heads(rng, 3, image_wh, 3, C, 2.0)
    _plant(rng, y_true, y_pred, anc, image_wh)
    assert [t.shape[1:3] for t in y_true] == [grid0, (2 * grid0[0], 2 * grid0[1]), (4 * grid0[0], 4 * grid0[1])]
    want = oy.yolov4_loss(oy.COCO_ANCHORS_FLAT, C, y_true, y_pred)
    got = Yolov4Loss(oy.COCO_ANCHORS_FLAT, C)([_t(t, cuda) for t in y_true], [_t(t, cuda) for t in y_pred])
    assert abs(float(got) - float(want)) <= LOSS_RTOL * abs(float(want)), (float(got), float(want))


# ------------------------------------------------------------------------------------------------------------------------
TARGET_CASES = [((416, 256), 80, 3, False), ((256, 416), 1, 3, True), ((320, 200), 20, 2, False), ((40, 96), 2, 4, True),
                ((416, 416), 3, 2, False)]


def _target_draw(rng, image_wh, C, B, anc, max_boxes):
    from oracle import yolo as oy
    from tfmv_b200 import synth
    boxes, classes, off = synth.gt_batch(rng, B, image_wh, max_boxes=max_boxes, classes=C)
    if off[1] >= 3:
        boxes[1:3] = boxes[0]   # three boxes on one record: all dropped (cds:279-284)
    per = [oy.get_targets(boxes[off[b]:off[b + 1]], classes[off[b]:off[b + 1]], anc, image_wh, C) for b in range(B)]
    return boxes, classes, off, [np.stack([p[l] for p in per], 0) for l in range(3)]


@gpu
@pytest.mark.parametrize("image_wh,C,B,normalised", TARGET_CASES)
def test_get_targets_shapes(lib, cuda, image_wh, C, B, normalised):
    """GetTargetsBatch and the TargetBuffers reuse path, bit-exact (A = 3: the reference's idx // layers_num rule)."""
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator, TargetBuffers
    rng = _rng("targets", image_wh, C, B, normalised)
    anc = _anchors(3) / np.asarray(image_wh, F) if normalised else _anchors(3)
    gen = DataGenerator(C, anc, image_wh)
    boxes, classes, off, want = _target_draw(rng, image_wh, C, B, anc, 60)
    got = gen.GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda))
    for l in range(3):
        assert_bits_equal(got[l].cpu().numpy(), want[l])
    assert sum(float(w[..., 4].sum()) for w in want) > 0
    buf = TargetBuffers()
    for max_boxes in (40, 80, 5):
        boxes, classes, off, want = _target_draw(rng, image_wh, C, B, anc, max_boxes)
        got = gen.GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), buffers=buf)
        for l in range(3):
            assert_bits_equal(got[l].cpu().numpy(), want[l])


# ------------------------------------------------------------------------------------------------------------------------
# decode + NMS cases: (image_wh, A, C, B, metric)
NMS_CASES = [
    ((416, 256), 3, 80, 2, "iou"),
    ((256, 416), 3, 20, 2, "diou"),
    ((320, 200), 5, 1, 2, "ciou"),
    ((40, 96), 1, 3, 3, "iou"),
    ((40, 96), 8, 80, 2, "diou"),
    ((256, 416), 2, 2, 2, "ciou"),
    ((416, 416), 3, 1, 2, "diou"),
]
NMS_THR = (0.5, 0.3, 0.5)


def _nms_inputs(case):
    image_wh, A, C, B = case[:4]
    return _heads(_rng("nms", case), B, image_wh, A, C), _anchors(A)


@gpu
@pytest.mark.parametrize("case", NMS_CASES, ids=_case_id)
def test_get_nms_boxes_shapes(lib, cuda, case):
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxesBatch
    image_wh, A, C, B, metric = case
    heads, anc = _nms_inputs(case)
    r = GetNMSBoxesBatch(*[_t(h, cuda) for h in heads], anc, image_wh, C, *NMS_THR, metric, with_indices=True)
    r = {k: v.cpu().numpy() for k, v in r.items()}
    for b in range(B):
        want = oy.get_nms_boxes_ex(*[h[b:b + 1] for h in heads], anc, image_wh, C, *NMS_THR, metric)
        assert want["selected"].shape[0] > 0
        _check_image(r, b, want, C)


@gpu
@pytest.mark.parametrize("shape", [(2, 8, 13, 3, 1), (3, 13, 8, 5, 2), (2, 6, 1, 1, 20)])
def test_get_boxes_shapes(lib, cuda, shape):
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetBoxes
    B, h, w, A, C = shape
    rng = _rng("boxes-dense", shape)
    y = rng.standard_normal((B, h, w, A, 5 + C), dtype=F) * F(2)
    y[0, 0, 0, 0, 2] = 150.0   # inf width -> 0 -> row dropped
    anc = (_anchors(A)[0] / np.array([w * 32, h * 32], F)).astype(F)
    want = oy.get_boxes(y, anc, C)
    got = GetBoxes(_t(y, cuda), _t(anc, cuda), C)
    assert 0 < want[0].shape[0] < B * h * w * A
    for g, wv in zip(got, want):
        assert_bits_equal(g.cpu().numpy(), wv)


@gpu
@pytest.mark.parametrize("image_wh,A,C", [((416, 256), 3, 1), ((40, 96), 1, 2)])
def test_get_ground_truth_shapes(lib, cuda, image_wh, A, C):
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetGroudTruth
    y_true = _planted_targets(_rng("gt", image_wh, A, C), 3, image_wh, A, C)
    for l in range(3):
        want = oy.get_ground_truth(y_true[l])
        got = GetGroudTruth(_t(y_true[l], cuda)).cpu().numpy()
        assert_bits_equal(got, want)


@gpu
@pytest.mark.parametrize("refill", ["late", "early"])
def test_decode_filter_refill_forms(lib, cuda, refill):
    """A warp of the persistent decode filter refills its slab before its append on long streams (>= 32 tiles per warp:
    4 warps per CTA at C = 80, one CTA per SM) and after it on short ones.  A batch large enough for the early refill and
    its first 8 images, which take the late one, must both give the oracle's per-image results."""
    import torch
    from oracle import yolo as oy
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxesBatch
    image = 416
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = lambda b: sum((b * g * g * 3 + 31) // 32 for g in synth.yolo_grids(image))
    B = 8
    while tiles(B) < 32 * 4 * sms:
        B += 8
    rng = _rng("refill", image)
    heads = synth.yolo_heads(rng, B, image)
    if refill == "late":
        B = 8
        heads = [h[:B] for h in heads]
        assert tiles(B) < 32 * 2 * sms   # short even if the filter ran 2 warps per CTA
    anc = synth.yolo_anchors()
    r = GetNMSBoxesBatch(*[_t(h, cuda) for h in heads], anc, (image, image), 80, *NMS_THR, "diou", with_indices=True)
    r = {k: v.cpu().numpy() for k, v in r.items()}
    for b in sorted({0, B // 2, B - 1} | set(int(x) for x in rng.choice(B, 3, replace=False))):
        want = oy.get_nms_boxes_ex(*[h[b:b + 1] for h in heads], anc, (image, image), 80, *NMS_THR, "diou")
        _check_image(r, b, want, 80)


# ------------------------------------------------------------------------------------------------------------------------
LN_IMAGE_WH, LN_A, LN_C, LN_B = (416, 256), 3, 80, 3


def _ln_draw(seed):
    rng = _rng("loss-nms", seed)
    anc = _anchors(LN_A)
    y_true = _planted_targets(rng, LN_B, LN_IMAGE_WH, LN_A, LN_C)
    heads = _heads(rng, LN_B, LN_IMAGE_WH, LN_A, LN_C)
    _plant(rng, y_true, heads, anc, LN_IMAGE_WH[::-1])
    return y_true, heads, anc


def _same_nms(r, s):
    import torch
    assert torch.equal(r["count"], s["count"])
    for b, k in enumerate(s["count"].tolist()):
        for key in s:
            if key != "count":
                assert torch.equal(r[key][b, :k], s[key][b, :k]), (key, b)


@gpu
@pytest.mark.parametrize("other_units,global_batch", [(False, None), (True, 2 * LN_B + 1)])
def test_loss_and_nms_batch(lib, cuda, other_units, global_batch):
    """LossAndNMSBoxesBatch (loss and NMS on two streams) == GetLoss + GetNMSBoxesBatch bit for bit, and == the oracle;
    with the loss's anchors in other units than the decode's and a global batch divisor."""
    from oracle import yolo as oy
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxesBatch, LossAndNMSBoxesBatch, _loss_call
    y_true, heads, anc = _ln_draw(1)
    loss_anc = (anc / F(LN_IMAGE_WH[0])).astype(F) if other_units else anc
    dt, dh = [_t(t, cuda) for t in y_true], [_t(h, cuda) for h in heads]
    loss, r = LossAndNMSBoxesBatch(dt, dh, LN_IMAGE_WH, anc, LN_C, 0.5, "ciou", *NMS_THR, "diou", with_indices=True,
                                   global_batch=global_batch, loss_anchors_wh=loss_anc if other_units else None)
    div = LN_B if global_batch is None else global_batch
    sep = _loss_call(dt, dh, LN_IMAGE_WH, loss_anc, 0.5, "ciou", 0, batch_divisor=div)
    assert float(loss) == float(sep)
    _same_nms(r, GetNMSBoxesBatch(*dh, anc, LN_IMAGE_WH, LN_C, *NMS_THR, "diou", with_indices=True))
    want = float(oy.get_loss(y_true, heads, LN_IMAGE_WH, loss_anc, 0.5, "ciou")) * LN_B / div
    assert abs(float(loss) - want) <= LOSS_RTOL * abs(want), (float(loss), want)
    r = {k: v.cpu().numpy() for k, v in r.items()}
    for b in range(LN_B):
        _check_image(r, b, oy.get_nms_boxes_ex(*[h[b:b + 1] for h in heads], anc, LN_IMAGE_WH, LN_C, *NMS_THR, "diou"), LN_C)


@gpu
def test_loss_and_nms_batch_graph_replay(lib, cuda):
    """Captured once, inputs refilled in place with a second draw, replayed: the eager results of that draw."""
    import torch
    from oracle import yolo as oy
    from tfmv_b200 import runtime
    from tfmv_b200.ai_models.utils.tf_yolo_utils import LossAndNMSBoxesBatch
    y_true, heads, anc = _ln_draw(1)
    loss_anc = (anc / F(LN_IMAGE_WH[0])).astype(F)
    dt, dh = [_t(t, cuda) for t in y_true], [_t(h, cuda) for h in heads]
    run = lambda: LossAndNMSBoxesBatch(dt, dh, LN_IMAGE_WH, anc, LN_C, 0.5, "ciou", *NMS_THR, "diou", with_indices=True,
                                       global_batch=2 * LN_B, loss_anchors_wh=loss_anc)
    step = runtime.capture(run)
    y_true2, heads2, _ = _ln_draw(2)
    for dst, src in zip(dt + dh, y_true2 + heads2):
        dst.copy_(torch.from_numpy(src))
    loss_g, r_g = step()
    loss_g, r_g = loss_g.clone(), {k: v.clone() for k, v in r_g.items()}
    loss_e, r_e = run()
    torch.cuda.synchronize()
    assert float(loss_g) == float(loss_e)
    _same_nms(r_g, r_e)
    want = float(oy.get_loss(y_true2, heads2, LN_IMAGE_WH, loss_anc, 0.5, "ciou")) / 2
    assert abs(float(loss_g) - want) <= LOSS_RTOL * abs(want), (float(loss_g), want)
    r_g = {k: v.cpu().numpy() for k, v in r_g.items()}
    b = LN_B - 1
    _check_image(r_g, b, oy.get_nms_boxes_ex(*[h[b:b + 1] for h in heads2], anc, LN_IMAGE_WH, LN_C, *NMS_THR, "diou"), LN_C)


# ------------------------------------------------------------------------------------------------------------------------
# CPU guards (no GPU): the cases above are able to fail
def _rect(image_wh):
    return image_wh[0] != image_wh[1]


def _swapped_loss_cases():
    out = [("dense", c) for c in LOSS_CASES if _rect(c[0])] + [("grad", c) for c in GRAD_CASES if _rect(c[0])]
    return out + [("boxes", c) for c in BOX_CASES if _rect(c[0])]


@pytest.mark.parametrize("kind,case", _swapped_loss_cases(), ids=lambda v: v if isinstance(v, str) else repr(v).replace(" ", ""))
def test_rectangular_loss_cases_tell_w_from_h(kind, case):
    """On the oracle alone: image_wh and image_wh[::-1] give losses far apart and different ignore masks."""
    from oracle import yolo as oy
    if kind == "boxes":
        _, _, _, y_true, y_pred, anc = _box_inputs(case)
        iou_type, thr = case[3], 0.5
    else:
        y_true, y_pred, anc = _loss_inputs(case, 2.5 if kind == "dense" else 1.0)
        iou_type, thr = case[4], (case[5] if kind == "dense" else 0.5)
    image_wh = case[0]
    _, pa, ia = oy.get_loss(y_true, y_pred, image_wh, anc, thr, iou_type, return_ignore=True)
    _, pb, ib = oy.get_loss(y_true, y_pred, image_wh[::-1], anc, thr, iou_type, return_ignore=True)
    assert not np.array_equal(ia, ib)
    # the total is dominated by the background objectness terms; the wh parts, which the GPU cases compare within
    # LOSS_RTOL, and the gradients are where the order shows
    if kind == "grad":
        _, ga = oy.get_loss_grad(y_true, y_pred, image_wh, anc, thr, iou_type)
        _, gb = oy.get_loss_grad(y_true, y_pred, image_wh[::-1], anc, thr, iou_type)
        assert any(np.max(np.abs(x - y) - 1e-4 * np.abs(x)) > 100 * 1e-7 for x, y in zip(ga, gb))
    else:
        assert np.max(np.abs(pa - pb) / np.maximum(np.abs(pa), 1e-6)) > 100 * LOSS_RTOL, (pa, pb)


@pytest.mark.parametrize("case", [c for c in NMS_CASES if _rect(c[0])], ids=_case_id)
def test_rectangular_decode_cases_tell_w_from_h(case):
    """On the oracle alone: the NMS output of every image changes when the decode takes (h, w) for (w, h)."""
    from oracle import yolo as oy
    image_wh, A, C, B, metric = case
    heads, anc = _nms_inputs(case)
    for b in range(B):
        hb = [h[b:b + 1] for h in heads]
        a = oy.get_nms_boxes_ex(*hb, anc, image_wh, C, *NMS_THR, metric)["boxes"]
        s = oy.get_nms_boxes_ex(*hb, anc, image_wh[::-1], C, *NMS_THR, metric)["boxes"]
        assert a.shape != s.shape or not np.array_equal(a, s)


def test_cases_cover_the_special_paths():
    """The loss cases include a scalar-load record (RF < 8), a W == 1 level and A == 1, and every record size the
    ignore pass distinguishes; the decode cases include W == 1, A == 1 and C == 1."""
    loss_inputs = [_loss_inputs(c, 2.5)[0] for c in LOSS_CASES]
    assert any(t[0].shape[-1] < 8 for t in loss_inputs)
    assert any(t.shape[2] == 1 for y in loss_inputs for t in y)
    assert any(t[0].shape[3] == 1 for t in loss_inputs)
    assert {t[0].shape[-1] for t in loss_inputs} >= {6, 7, 8, 25, 85}
    assert {c[1] for c in LOSS_CASES} >= {1, 2, 5, 8}
    assert any(_rect(c[0]) and c[2] < 3 for c in LOSS_CASES)
    nms_heads = [_nms_inputs(c)[0] for c in NMS_CASES]
    assert any(h.shape[2] == 1 for hs in nms_heads for h in hs)
    assert {c[1] for c in NMS_CASES} >= {1, 8} and {c[2] for c in NMS_CASES} >= {1, 2, 80}
    shapes = {(416, 256), (256, 416), (320, 200), (40, 96), (416, 416)}
    assert {c[0] for c in LOSS_CASES} == shapes and {c[0] for c in NMS_CASES} == shapes
    assert {c[0] for c in TARGET_CASES} == shapes
