"""GPU parity: GetTargets (bit-exact) and GetLoss / Yolov4Loss (<= 1e-4 relative, BASELINE.md §5) vs the oracle."""
import numpy as np
import pytest

from test_gpu_core import _t, assert_bits_equal

pytestmark = pytest.mark.gpu
F = np.float32
LOSS_RTOL = 1e-4


def _dense_targets(rng, batch, image, anc, max_boxes=100, normalised_anchors=False):
    from oracle import yolo as oy
    from tfmv_b200 import synth
    boxes, classes, off = synth.gt_batch(rng, batch, (image, image), max_boxes=max_boxes)
    a = anc / F(image) if normalised_anchors else anc
    per = [oy.get_targets(boxes[off[b]:off[b + 1]], classes[off[b]:off[b + 1]], a, (image, image), 80) for b in range(batch)]
    return boxes, classes, off, [np.stack([p[l] for p in per], 0) for l in range(3)]


@pytest.mark.parametrize("image,batch,normalised", [(416, 3, False), (608, 2, False), (416, 4, True), (96, 6, True)])
def test_get_targets_bit_exact(lib, cuda, image, batch, normalised):
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    rng = np.random.default_rng(20261018 + 2 + image)
    anc = synth.yolo_anchors().astype(F)
    boxes, classes, off, want = _dense_targets(rng, batch, image, anc, normalised_anchors=normalised)
    if batch >= 3:  # force collisions: duplicate the first boxes of image 0 inside image 0
        n0 = off[1]
        boxes[1:min(3, n0)] = boxes[0]
        a = anc / F(image) if normalised else anc
        from oracle import yolo as oy
        p0 = oy.get_targets(boxes[:n0], classes[:n0], a, (image, image), 80)
        for l in range(3):
            want[l][0] = p0[l]
    gen = DataGenerator(80, anc / F(image) if normalised else anc, (image, image))
    got = gen.GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda))
    for l in range(3):
        assert tuple(got[l].shape) == want[l].shape
        assert_bits_equal(got[l].cpu().numpy(), want[l])
    if normalised:
        assert sum(float(w[..., 4].sum()) for w in want[:2]) > 0  # real argmax spreads over the layers
    # single-image reference signature, including the empty image
    img, t1 = gen.GetTargets("img", classes[:off[1]], _t(boxes[:off[1]], cuda))
    assert img == "img"
    assert_bits_equal(t1[2].cpu().numpy(), want[2][0])
    _, te = gen.GetTargets(None, np.zeros((0,), np.int32), np.zeros((0, 4), F))
    assert all(float(x.abs().sum()) == 0.0 for x in te)


@pytest.mark.parametrize("image,batch", [(416, 3), (96, 6)])
def test_get_targets_persistent_buffers(lib, cuda, image, batch):
    """TargetBuffers: dense fill once, then sparse reset of the previous step's records — every step's tensors must
    equal a fresh assignment bit for bit (different GT sets, collisions, an empty step, a shrinking/growing total)."""
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator, TargetBuffers
    anc = synth.yolo_anchors().astype(F)
    gen = DataGenerator(80, anc, (image, image))
    buf = TargetBuffers()
    ptrs = None
    for step, max_boxes in enumerate([40, 100, 0, 7, 100]):
        rng = np.random.default_rng(20261018 + 50 + step)
        if max_boxes == 0:
            boxes, classes, off = np.zeros((0, 4), F), np.zeros((0,), np.int32), np.zeros(batch + 1, np.int32)
            want = [np.zeros((batch, image // s, image // s, 3, 85), F) for s in (32, 16, 8)]
        else:
            boxes, classes, off, want = _dense_targets(rng, batch, image, anc, max_boxes=max_boxes)
            n0 = off[1]
            if n0 >= 2:  # collision inside image 0
                boxes[1] = boxes[0]
                from oracle import yolo as oy
                p0 = oy.get_targets(boxes[:n0], classes[:n0], anc, (image, image), 80)
                for l in range(3):
                    want[l][0] = p0[l]
        got = gen.GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), buffers=buf)
        if ptrs is None:
            ptrs = [t.data_ptr() for t in got]
        assert [t.data_ptr() for t in got] == ptrs  # same tensors every step
        for l in range(3):
            assert_bits_equal(got[l].cpu().numpy(), want[l])
    buf.invalidate()
    got[0].fill_(3.0)
    got = gen.GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), buffers=buf)
    assert_bits_equal(got[0].cpu().numpy(), want[0])


@pytest.mark.parametrize("image,batch,iou_type,normalised", [
    (416, 2, "iou", False), (416, 2, "ciou", True), (608, 2, "ciou", False), (416, 3, "diou", True), (96, 5, "ciou", True)])
def test_get_loss_matches_oracle(lib, cuda, image, batch, iou_type, normalised):
    from oracle import yolo as oy
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLoss, _loss_call
    rng = np.random.default_rng(20261018 + 2 + batch)
    anc = synth.yolo_anchors().astype(F)
    _, _, _, y_true = _dense_targets(rng, batch, image, anc, normalised_anchors=normalised)
    if batch > 2:
        for l in range(3):
            y_true[l][batch - 1] = 0  # an image without ground truth: ignore mask all ones (reduce_max of empty)
    y_pred = synth.yolo_heads(rng, batch, image)
    # make some predictions overlap their targets so the ignore mask has zeros
    for l in range(3):
        yt = y_true[l]
        yp = y_pred[l].reshape(yt.shape)
        m = yt[..., 4] > 0
        yp[m, 2:4] = np.log(np.maximum(yt[m, 2:4] * image, 1e-3) / anc[l][np.nonzero(m)[3]]) + rng.normal(0, 0.1, (int(m.sum()), 2))
    import torch
    want, want_parts, want_ign = oy.get_loss(y_true, y_pred, (image, image), anc, 0.5, iou_type, return_ignore=True)
    ign = torch.full(want_ign.shape, 7, dtype=torch.uint8, device=cuda)
    got, parts = _loss_call([_t(t, cuda) for t in y_true], [_t(t, cuda) for t in y_pred], (image, image), anc, 0.5, iou_type, 0,
                            return_parts=True, ignore_out=ign)
    # the ignore mask is a discrete output: bit-exact, and it must contain both values to mean anything
    assert np.array_equal(ign.cpu().numpy(), want_ign)
    assert 0 < int(want_ign.sum()) < want_ign.size
    np.testing.assert_allclose(parts.cpu().numpy(), want_parts, rtol=LOSS_RTOL, atol=1e-6)
    assert abs(float(got) - float(want)) <= LOSS_RTOL * abs(float(want))
    got2 = GetLoss([_t(t, cuda) for t in y_true], [_t(t, cuda) for t in y_pred], image_wh=(image, image), anchors_wh=anc,
                   iou_thresh=0.5, iou_type=iou_type)
    assert float(got2) == float(got)  # deterministic reduction: bit-identical run to run


@pytest.mark.parametrize("image,batch,iou_type,normalised", [(416, 3, "ciou", False), (608, 2, "iou", False), (416, 4, "diou", True),
                                                             (96, 6, "ciou", True)])
def test_loss_from_boxes_matches_dense_path_and_oracle(lib, cuda, image, batch, iou_type, normalised):
    """SURVEY §8f N3: GetTargets + GetLoss fused without the dense y_true == the oracle's get_targets -> get_loss
    (loss within 1e-4, ignore mask bit-exact), including colliding boxes, an image without boxes and out-of-range
    classes; and == the dense GPU path."""
    import torch
    from oracle import yolo as oy
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxes, _loss_call
    rng = np.random.default_rng(20261018 + 70 + batch)
    anc = synth.yolo_anchors().astype(F)
    tanc = anc / F(image) if normalised else anc
    boxes, classes, off = synth.gt_batch(rng, batch, (image, image), max_boxes=60)
    n0 = off[1]
    if n0 >= 3:
        boxes[1] = boxes[0]; boxes[2] = boxes[0]           # triple collision in image 0: all three dropped
    classes[-1] = 200                                       # out of range -> all-zero class row
    if batch > 2:                                           # image 1 without ground truth
        keep = np.ones(len(boxes), bool); keep[off[1]:off[2]] = False
        cnt = np.diff(off); cnt[1] = 0
        boxes, classes, off = boxes[keep], classes[keep], np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    per = [oy.get_targets(boxes[off[b]:off[b + 1]], classes[off[b]:off[b + 1]], tanc, (image, image), 80) for b in range(batch)]
    y_true = [np.stack([p[l] for p in per], 0) for l in range(3)]
    y_pred = synth.yolo_heads(rng, batch, image)
    for l in range(3):  # some predictions overlap their targets so the ignore mask has zeros
        yt = y_true[l]
        yp = y_pred[l].reshape(yt.shape)
        m = yt[..., 4] > 0
        yp[m, 2:4] = np.log(np.maximum(yt[m, 2:4] * image, 1e-3) / anc[l][np.nonzero(m)[3]]) + rng.normal(0, 0.1, (int(m.sum()), 2))
    want, want_parts, want_ign = oy.get_loss(y_true, y_pred, (image, image), anc, 0.5, iou_type, return_ignore=True)
    ign = torch.full(want_ign.shape, 7, dtype=torch.uint8, device=cuda)
    dp = [_t(t, cuda) for t in y_pred]
    got, parts = GetLossFromBoxes(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), dp, (image, image), anc, 80, 0.5, iou_type,
                                  target_anchors=tanc, return_parts=True, ignore_out=ign)
    assert np.array_equal(ign.cpu().numpy(), want_ign)
    assert sum(float(t[..., 4].sum()) for t in y_true) > 0 and 0 < int(want_ign.sum()) < want_ign.size
    np.testing.assert_allclose(parts.cpu().numpy(), want_parts, rtol=LOSS_RTOL, atol=1e-6)
    assert abs(float(got) - float(want)) <= LOSS_RTOL * abs(float(want))
    gen = DataGenerator(80, tanc, (image, image))
    dense = gen.GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda))
    got_d, parts_d = _loss_call(dense, dp, (image, image), anc, 0.5, iou_type, 0, return_parts=True)
    np.testing.assert_allclose(parts.cpu().numpy(), parts_d.cpu().numpy(), rtol=1e-6, atol=1e-9)
    # no boxes at all
    e = GetLossFromBoxes(np.zeros((0,), np.int32), np.zeros((0, 4), F), np.zeros(batch + 1, np.int32), dp, (image, image), anc, 80,
                         0.5, iou_type)
    want_e = oy.get_loss([np.zeros_like(t) for t in y_true], y_pred, (image, image), anc, 0.5, iou_type)
    assert abs(float(e) - float(want_e)) <= LOSS_RTOL * abs(float(want_e))


def test_get_loss_reads_pinned_host_predictions_in_place(lib, cuda):
    """y_pred handed over as pinned host tensors is consumed in place (no staging copy): same bits as device tensors."""
    import torch
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLoss, GetLossFromBoxes, _loss_call
    rng = np.random.default_rng(20261018 + 33)
    image, batch = 416, 3
    anc = synth.yolo_anchors().astype(F)
    boxes, classes, off, y_true = _dense_targets(rng, batch, image, anc, normalised_anchors=True)
    y_pred = synth.yolo_heads(rng, batch, image)
    dt = [_t(t, cuda) for t in y_true]
    pinned = [torch.from_numpy(np.ascontiguousarray(h)).pin_memory() for h in y_pred]
    ign_a = torch.full((batch, 10647), 7, dtype=torch.uint8, device=cuda)
    ign_b = torch.full((batch, 10647), 9, dtype=torch.uint8, device=cuda)
    a, pa = _loss_call(dt, [_t(h, cuda) for h in y_pred], (image, image), anc, 0.5, "ciou", 0, return_parts=True, ignore_out=ign_a)
    b, pb = _loss_call(dt, pinned, (image, image), anc, 0.5, "ciou", 0, return_parts=True, ignore_out=ign_b)
    assert float(a) == float(b) and torch.equal(pa, pb) and torch.equal(ign_a, ign_b)
    assert float(GetLoss(dt, pinned, (image, image), anc, 0.5, "ciou")) == float(a)
    tanc = anc / F(image)
    s_dev = GetLossFromBoxes(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), [_t(h, cuda) for h in y_pred], (image, image), anc, 80,
                             0.5, "ciou", target_anchors=tanc)
    s_pin = GetLossFromBoxes(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), pinned, (image, image), anc, 80, 0.5, "ciou",
                             target_anchors=tanc)
    assert float(s_dev) == float(s_pin) and abs(float(s_dev) - float(a)) <= 1e-6 * abs(float(a))


def test_reference_unit_test_relation_on_gpu(lib, cuda):
    """yolo_v3/unit_test/loss_test.py:152-172 on the GPU: GetLoss-copy == Yolov4Loss on uniform-random tensors."""
    from oracle import yolo as oy
    from tfmv_b200.ai_models.losses.yolo_loss import Yolov4Loss
    from tfmv_b200.ai_models.utils.tf_yolo_utils import _loss_call
    rng = np.random.default_rng(5)
    grids = (2, 4, 8)
    yt = [rng.random((2, g, g, 3, 85), dtype=F) for g in grids]
    yp = [rng.random((2, g, g, 255), dtype=F) for g in grids]
    anc = oy.load_anchors_order(oy.COCO_ANCHORS_FLAT.reshape(-1))
    a = Yolov4Loss(oy.COCO_ANCHORS_FLAT, 80)([_t(t, cuda) for t in yt], [_t(t, cuda) for t in yp])
    b = _loss_call([_t(t, cuda) for t in yt], [_t(t, cuda) for t in yp], (64, 64), anc, 0.5, "iou", 1)
    assert float(a) == float(b)
    want = oy.yolov4_loss(oy.COCO_ANCHORS_FLAT, 80, yt, yp)
    assert abs(float(a) - float(want)) <= LOSS_RTOL * abs(float(want))
    # the tf_yolo_utils variant differs on non-binary obj (Q10, Q11) and must follow the oracle too
    c = _loss_call([_t(t, cuda) for t in yt], [_t(t, cuda) for t in yp], (64, 64), anc, 0.5, "ciou", 0)
    want_c = oy.get_loss(yt, yp, (64, 64), anc, 0.5, "ciou")
    assert abs(float(c) - float(want_c)) <= LOSS_RTOL * abs(float(want_c))


@pytest.mark.parametrize("iou_type,thr,sigma", [("ciou", 0.5, 2.5), ("iou", 0.5, 2.0), ("diou", 0.7, 2.5), ("ciou", 0.3, 2.0),
                                                ("iou", 0.05, 1.0), ("ciou", 0.5, 6.0)])
def test_ignore_mask_stress_bit_exact(lib, cuda, iou_type, thr, sigma):
    """The ignore mask decides on exact metric >= thr comparisons; the kernel's decode-free filters (cell / logit-sum
    windows, thr >= 0.5) and the exact fall-back paths (thr < 0.5, out-of-range logits) must agree with the oracle
    bit for bit.  Wide logits make predicted boxes of every size, many of them overlapping ground truth."""
    import torch
    from oracle import yolo as oy
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import _loss_call
    image, batch = 256, 3
    rng = np.random.default_rng(int(thr * 100) + int(sigma * 10))
    anc = (synth.yolo_anchors().astype(F) * F(image / 608.0)).astype(F)
    _, _, _, y_true = _dense_targets(rng, batch, image, anc, max_boxes=60, normalised_anchors=True)
    y_pred = [h * F(sigma) for h in synth.yolo_heads(rng, batch, image)]
    # plant predictions that sit right on their targets (IoU near 1) and near-threshold rescaled copies
    for l in range(3):
        yt = y_true[l]
        yp = y_pred[l].reshape(yt.shape)
        b, yy, xx, aa = np.nonzero(yt[..., 4] > 0)
        for k in range(len(b)):
            g = yt.shape[1]
            t = yt[b[k], yy[k], xx[k], aa[k]]
            s = [1.0, 1.0, np.sqrt(thr), 1.0 / np.sqrt(max(thr, 1e-3))][k % 4] * (1.0 + rng.normal(0, 0.01))
            a2 = (aa[k] + k) % 3
            fx, fy = t[0] * g - xx[k], t[1] * g - yy[k]
            fx, fy = min(max(fx, 1e-3), 1 - 1e-3), min(max(fy, 1e-3), 1 - 1e-3)
            yp[b[k], yy[k], xx[k], a2, 0] = np.log(fx / (1 - fx))
            yp[b[k], yy[k], xx[k], a2, 1] = np.log(fy / (1 - fy))
            yp[b[k], yy[k], xx[k], a2, 2:4] = np.log(np.maximum(t[2:4] * image * s, 1e-3) / anc[l][a2])
    want, _, want_ign = oy.get_loss(y_true, y_pred, (image, image), anc, thr, iou_type, return_ignore=True)
    ign = torch.full(want_ign.shape, 7, dtype=torch.uint8, device=cuda)
    got = _loss_call([_t(t, cuda) for t in y_true], [_t(t, cuda) for t in y_pred], (image, image), anc, thr, iou_type, 0,
                     ignore_out=ign)
    g = ign.cpu().numpy()
    assert np.array_equal(g, want_ign), "%d ignore bits differ" % int((g != want_ign).sum())
    assert int((want_ign == 0).sum()) > 20
    if np.isfinite(want):
        assert abs(float(got) - float(want)) <= LOSS_RTOL * abs(float(want))


def test_get_ground_truth_and_boolean_mask_order(lib, cuda):
    """yolo_v4/model.py:380-395 GetGroudTruth: rows in row-major order, corners bit-exact, class = first argmax."""
    from oracle import yolo as oy
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetGroudTruth
    rng = np.random.default_rng(13)
    anc = (synth.yolo_anchors().astype(F) / F(416)).astype(F)
    _, _, _, y_true = _dense_targets(rng, 3, 416, synth.yolo_anchors().astype(F), normalised_anchors=True)
    for l in range(3):
        want = oy.get_ground_truth(y_true[l])
        got = GetGroudTruth(_t(y_true[l], cuda)).cpu().numpy()
        assert got.shape == want.shape
        assert_bits_equal(got, want)
    empty = GetGroudTruth(_t(np.zeros((1, 13, 13, 3, 85), F), cuda))
    assert tuple(empty.shape) == (0, 5)


def test_class_focal_loss_variant(lib, cuda):
    """losses/class_loss.py:25-60 ClassFocalLoss (demo-only variant): per level sum / (sum(mask)/B), divide_no_nan."""
    from oracle import effdet as oe
    from tfmv_b200.ai_models.losses.class_loss import ClassFocalLoss
    rng = np.random.default_rng(17)
    shapes = [(4, 8, 8, 9, 11), (4, 4, 4, 9, 11), (4, 2, 2, 9, 11)]
    tc = [(rng.random(s) < 0.05).astype(F) for s in shapes]
    pc = [rng.standard_normal(s).astype(F) for s in shapes]
    tm = [(rng.random(s[:-1] + (1,)) < 0.1) for s in shapes]
    tm[2][:] = False   # normalizer 0 -> divide_no_nan -> that level contributes 0
    want = oe.class_focal_loss(tc, pc, tm, 0.25, 1.5)
    got = ClassFocalLoss(0.25, 1.5)([_t(t, cuda) for t in tc], ([_t(p, cuda) for p in pc], [_t(m, cuda) for m in tm]))
    assert abs(float(got) - float(want)) <= LOSS_RTOL * abs(float(want))


@pytest.mark.parametrize("image,batch,iou_type", [(416, 2, "ciou"), (96, 5, "iou"), (608, 2, "ciou")])
def test_get_loss_gradient_matches_oracle(lib, cuda, image, batch, iou_type):
    """SURVEY §8f N1: d GetLoss / d y_pred, dense like y_pred, against the oracle's analytic gradient (itself pinned
    to fp64 finite differences on the CPU)."""
    from oracle import yolo as oy
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossAndGrad
    rng = np.random.default_rng(29 + batch)
    anc = synth.yolo_anchors().astype(F)
    _, _, _, y_true = _dense_targets(rng, batch, image, anc, normalised_anchors=True)
    y_pred = synth.yolo_heads(rng, batch, image)
    for l in range(3):   # overlapping predictions so the ignore mask has zeros
        yt = y_true[l]
        yp = y_pred[l].reshape(yt.shape)
        m = yt[..., 4] > 0
        yp[m, 2:4] = np.log(np.maximum(yt[m, 2:4] * image, 1e-3) / (anc[l] / 1.0)[np.nonzero(m)[3]]) + rng.normal(0, 0.1, (int(m.sum()), 2))
    a = anc / F(image)
    want_loss, want = oy.get_loss_grad(y_true, y_pred, (image, image), a * F(image), 0.5, iou_type)
    got_loss, got = GetLossAndGrad([_t(t, cuda) for t in y_true], [_t(t, cuda) for t in y_pred], (image, image), a * F(image), 0.5, iou_type)
    assert abs(float(got_loss) - float(want_loss)) <= LOSS_RTOL * abs(float(want_loss))
    for l in range(3):
        g = got[l].cpu().numpy().reshape(want[l].shape)
        assert g.shape == want[l].shape
        np.testing.assert_allclose(g, want[l], rtol=1e-4, atol=1e-7)
        # structure: non-object records carry a gradient only in the conf channel
        nobj = y_true[l][..., 4] == 0
        assert np.count_nonzero(np.delete(g[nobj], 4, axis=-1)) == 0


def _offset_copy(t):
    """The values of device tensor t in a new device buffer, 4 bytes past a 16-byte boundary.  GetLoss reads such a y_pred
    with the single ignore kernel's scalar loads."""
    import torch
    buf = torch.empty(t.numel() + 4, dtype=t.dtype, device=t.device)
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


def _ignore_layouts(heads):
    """The same y_pred in the three layouts that select the forms of the ignore pass: 16-byte aligned device tensors (the
    split form), device tensors at a 4-byte offset (the single kernel, scalar loads) and pinned host tensors (the single
    kernel, paired loads)."""
    assert all(h.is_cuda and h.data_ptr() % 16 == 0 for h in heads)
    pinned = [h.cpu().pin_memory() for h in heads]
    assert all(h.is_pinned() and h.data_ptr() % 16 == 0 for h in pinned)
    return {"split": heads, "offset": [_offset_copy(h) for h in heads], "pinned": pinned}


def test_split_ignore_pass_is_bit_identical(lib, cuda):
    """The split form of the ignore pass (K4b-lean streams and filters, K4b-exact resolves the undecided records) must
    give the ignore mask of the single kernel bit for bit and the same loss (the undecided records' terms go through a
    2^-32 fixed-point sum).  The single kernel is reached through its real triggers: an unaligned y_pred and a pinned
    host y_pred."""
    import torch
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.utils.tf_yolo_utils import _loss_call
    rng = np.random.default_rng(77)
    image, batch = 256, 5
    anc = synth.yolo_anchors().astype(F)
    heads = [torch.from_numpy(h).to(cuda) for h in synth.yolo_heads(rng, batch, image)]
    # plant predictions on their targets so that the mask has zeros, and one NaN logit
    boxes, classes, off = synth.gt_batch(rng, batch, (image, image), max_boxes=40)
    gen = DataGenerator(80, anc / F(image), (image, image))
    y_true = gen.GetTargetsBatch(classes, boxes, off)
    for l in range(3):
        yt = y_true[l]
        hp = heads[l].view(yt.shape)
        m = yt[..., 4] > 0
        g = yt.shape[1]
        idx = m.nonzero()
        for b, yy, xx, a in idx.tolist()[::2]:
            t = yt[b, yy, xx, a]
            fx = min(max(float(t[0]) * g - xx, 1e-3), 1 - 1e-3)
            fy = min(max(float(t[1]) * g - yy, 1e-3), 1 - 1e-3)
            hp[b, yy, xx, a, 0] = float(np.log(fx / (1 - fx)))
            hp[b, yy, xx, a, 1] = float(np.log(fy / (1 - fy)))
            hp[b, yy, xx, a, 2] = float(np.log(max(float(t[2]) * image / anc[l][a][0], 1e-6)))
            hp[b, yy, xx, a, 3] = float(np.log(max(float(t[3]) * image / anc[l][a][1], 1e-6)))
    n_img = sum(int(t.shape[1] * t.shape[2] * 3) for t in y_true)
    out = {}
    for form, hp in _ignore_layouts(heads).items():
        ign = torch.zeros((batch, n_img), dtype=torch.uint8, device=cuda)
        loss, parts = _loss_call(y_true, hp, (image, image), anc, 0.5, "ciou", 0, return_parts=True, ignore_out=ign)
        out[form] = (float(loss), parts.cpu().numpy(), ign.cpu().numpy())
    assert out["split"][2].min() == 0 and out["split"][2].max() == 1          # the mask has both values
    for form in ("offset", "pinned"):
        assert np.array_equal(out[form][2], out["split"][2]), form
        assert abs(out[form][0] - out["split"][0]) <= 2e-6 * abs(out["split"][0]), (form, out[form][0], out["split"][0])
    # a NaN logit reaches the loss in both forms
    heads[2].view(y_true[2].shape)[0, 1, 1, 0, 4] = float("nan")
    for form, hp in _ignore_layouts(heads).items():
        assert np.isnan(float(_loss_call(y_true, hp, (image, image), anc, 0.5, "ciou", 0))), form
