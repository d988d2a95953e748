"""GPU: the YOLO loss and its gradient from bf16 / fp16 y_pred read in place.  Every half call is held to the fp32 call
on the widened heads (y.float()) in the same memory layout, so both take the same form of the ignore pass: loss, parts
and ignore mask bit-identical, and gradients equal to (g32 * s).to(grad_dtype) bit for bit (NaN positions equal, payloads
not compared), where g32 is the fp32 gradient and s the gradient scale.

Cases: those of test_gpu_yolo_sparse_grad plus C = 6 at 160x96, B = 1 (RF 11: the last record of level 0 starts 4
elements into a 16-byte chunk and the next chunk would end past the tensor) and C = 7 (RF 12: that chunk ends exactly at
the tensor's end)."""
import functools
import zlib

import numpy as np
import pytest
import torch

from test_gpu_core import _t, assert_bits_equal
from test_gpu_half_heads import _assert_same_rows
from test_gpu_yolo_sparse_grad import CASES, _case_id, _inputs, _layout

pytestmark = pytest.mark.gpu
HALF = {"bf16": torch.bfloat16, "fp16": torch.float16}
HALF_CASES = CASES + [((160, 96), 6, 1, "ciou", False), ((160, 96), 7, 2, "iou", False)]
SCALES = (None, 1024.0, 2.0 ** -4)


@functools.lru_cache(maxsize=None)
def _case_inputs(case):
    return _inputs(case)


def _plant_half(y_pred, case, dtype, dev):
    """The case's fp32 heads with values planted in a few per cent of the records, then cast to the half type: tw / th at
    the edges of the ignore filter's logit window (4, just above 4, -6, just below -6), outside the safe range and +-inf;
    conf logits near 0; NaN in box, conf and class channels; fp16 subnormals."""
    g = torch.Generator(device=dev).manual_seed(zlib.crc32(_case_id(case).encode()))
    C = case[1]
    out = []
    for h in y_pred:
        x = _t(h, dev).reshape(h.shape[0], h.shape[1], h.shape[2], 3, 5 + C).clone()
        u = lambda: torch.rand(x.shape[:-1], device=dev, generator=g)
        for k in (2, 3):
            for val in (4.0, 4.03125, -6.0, -6.0625, -40.0, 80.5, float("inf"), float("-inf")):
                x[..., k][u() < 0.004] = val
        for val in (0.0, 1e-7, -1e-7, 3e-6, -3e-6):
            x[..., 4][u() < 0.005] = val
        for k in (0, 1, 4):
            x[..., k][u() < 0.002] = float("nan")
        x[..., 5:][u() < 0.005] = float("nan")
        x[..., 0][u() < 0.005] = 3e-8
        x[..., 5][u() < 0.005] = 2e-7
        out.append(x.reshape(h.shape).to(dtype).contiguous())
    return out


def _half_layout(heads, layout):
    """aligned: 16-byte aligned device tensors (split ignore pass when RF >= 8); offset: 2 bytes past a 16-byte boundary
    (single kernel, scalar loads); pinned: page-locked host memory (single kernel, read in place)."""
    if layout == "offset":
        out = []
        for h in heads:
            buf = torch.empty(h.numel() + 8, dtype=h.dtype, device=h.device)
            v = buf[1:1 + h.numel()].view(h.shape)
            v.copy_(h)
            assert v.data_ptr() % 16 == 2
            out.append(v)
        return out
    return _layout(heads, layout)


def _wide_layout(heads, layout):
    """The fp32 heads y.float() in the layout of the same name (4-byte offset for "offset")."""
    return _layout([h.float() for h in heads], layout)


def _bits(x):
    return x.detach().reshape(-1).cpu().float().numpy()


def _expect_grads(got, g32, grad_dtype, scale):
    for a, b in zip(got, g32):
        assert a.dtype == grad_dtype and a.shape == b.shape
        want = (b if scale is None else b * scale).to(grad_dtype)
        assert_bits_equal(_bits(a), _bits(want))


def _dense_call(y_true, heads, case, **kw):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import _loss_call
    image_wh, C, B, iou_type, _ = case
    _, _, _, _, _, anc, _ = _case_inputs(case)
    return _loss_call(y_true, heads, image_wh, anc, 0.5, iou_type, 0, return_parts=True, **kw)


def _boxes_call(heads, case, cuda, **kw):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxes, GetLossFromBoxesAndGrad
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, _, _, anc, tanc = _case_inputs(case)
    args = (_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), heads, image_wh, anc, C, 0.5, iou_type)
    if "grad_dtype" in kw:
        return GetLossFromBoxesAndGrad(*args, target_anchors=tanc, return_parts=True, **kw)
    return GetLossFromBoxes(*args, target_anchors=tanc, return_parts=True, **kw)


def _n_img(heads):
    return sum(h.shape[1] * h.shape[2] * 3 for h in heads)


@pytest.mark.parametrize("layout", ["aligned", "offset", "pinned"])
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("case", HALF_CASES, ids=_case_id)
def test_forward_bit_identical(lib, cuda, case, dtype, layout):
    _, _, _, y_true, y_pred, _, _ = _case_inputs(case)
    heads = _plant_half(y_pred, case, HALF[dtype], cuda)
    half, wide = _half_layout(heads, layout), _wide_layout(heads, layout)
    yt = [_t(y, cuda) for y in y_true]
    B, n = heads[0].shape[0], _n_img(heads)
    ign = [torch.full((B, n), 7, dtype=torch.uint8, device=cuda) for _ in range(4)]
    lh, ph = _dense_call(yt, half, case, ignore_out=ign[0])
    lf, pf = _dense_call(yt, wide, case, ignore_out=ign[1])
    assert_bits_equal(_bits(lh), _bits(lf))
    assert_bits_equal(_bits(ph), _bits(pf))
    assert torch.equal(ign[0], ign[1]) and int(ign[0].max()) <= 1
    lh, ph = _boxes_call(half, case, cuda, ignore_out=ign[2])
    lf, pf = _boxes_call(wide, case, cuda, ignore_out=ign[3])
    assert_bits_equal(_bits(lh), _bits(lf))
    assert_bits_equal(_bits(ph), _bits(pf))
    assert torch.equal(ign[2], ign[3]) and int(ign[2].max()) <= 1
    assert 0 < int(ign[2].sum()) < ign[2].numel()   # the planted predictions clear some ignore bits


@pytest.mark.parametrize("layout", ["aligned", "offset"])
@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("case", HALF_CASES, ids=_case_id)
def test_backward_bit_identical(lib, cuda, case, dtype, layout):
    _, _, _, y_true, y_pred, _, _ = _case_inputs(case)
    heads = _plant_half(y_pred, case, HALF[dtype], cuda)
    half, wide = _half_layout(heads, layout), _wide_layout(heads, layout)
    yt = [_t(y, cuda) for y in y_true]
    l32, p32, g32 = _dense_call(yt, wide, case, with_grad=True)
    b32, q32, h32 = _boxes_call(wide, case, cuda, grad_dtype=torch.float32)
    for gd in (torch.float32, HALF[dtype]):
        for s in SCALES:
            st = None if s is None else torch.full((1,), s, dtype=torch.float32, device=cuda)
            lh, ph, gh = _dense_call(yt, half, case, with_grad=True, grad_dtype=gd, grad_scale=st)
            assert_bits_equal(_bits(lh), _bits(l32))
            assert_bits_equal(_bits(ph), _bits(p32))
            _expect_grads(gh, g32, gd, s)
            lh, ph, gh = _boxes_call(half, case, cuda, grad_dtype=gd, grad_scale=s)   # a Python float here
            assert_bits_equal(_bits(lh), _bits(b32))
            assert_bits_equal(_bits(ph), _bits(q32))
            _expect_grads(gh, h32, gd, s)


def test_default_gradient_type_is_fp32(lib, cuda):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossAndGrad
    case = CASES[0]
    image_wh, C, B, iou_type, _ = case
    _, _, _, y_true, y_pred, anc, _ = _case_inputs(case)
    heads = _plant_half(y_pred, case, torch.bfloat16, cuda)
    yt = [_t(y, cuda) for y in y_true]
    loss, grads = GetLossAndGrad(yt, heads, image_wh, anc, 0.5, iou_type)
    want_loss, want = GetLossAndGrad(yt, [h.float() for h in heads], image_wh, anc, 0.5, iou_type)
    assert_bits_equal(_bits(loss), _bits(want_loss))
    _expect_grads(grads, want, torch.float32, None)


def test_mixed_levels_fall_back_to_fp32(lib, cuda):
    case = CASES[0]
    _, _, _, y_true, y_pred, _, _ = _case_inputs(case)
    hb = _plant_half(y_pred, case, torch.bfloat16, cuda)
    hf = _plant_half(y_pred, case, torch.float16, cuda)
    mixed = [hb[0], hf[1], hb[2]]
    wide = [h.float() for h in mixed]
    yt = [_t(y, cuda) for y in y_true]
    lm, pm, gm = _dense_call(yt, mixed, case, with_grad=True)
    lw, pw, gw = _dense_call(yt, wide, case, with_grad=True)
    assert_bits_equal(_bits(lm), _bits(lw))
    _expect_grads(gm, gw, torch.float32, None)
    lm, pm = _boxes_call(mixed, case, cuda)
    lw, pw = _boxes_call(wide, case, cuda)
    assert_bits_equal(_bits(pm), _bits(pw))


def test_composite_calls_on_bf16_heads(lib, cuda):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import EvalStepFromBoxes, LossAndNMSBoxesBatch
    case = CASES[0]
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, y_true, y_pred, anc, tanc = _case_inputs(case)
    heads = _plant_half(y_pred, case, torch.bfloat16, cuda)
    wide = [h.float() for h in heads]
    yt = [_t(y, cuda) for y in y_true]
    kw = dict(confidence_thresh=0.3, scores_thresh=0.2, with_indices=True)
    lh, rh = LossAndNMSBoxesBatch(yt, heads, image_wh, anc, C, 0.5, iou_type, **kw)
    lf, rf = LossAndNMSBoxesBatch(yt, wide, image_wh, anc, C, 0.5, iou_type, **kw)
    assert_bits_equal(_bits(lh), _bits(lf))
    _assert_same_rows(rh, rf)
    args = (_t(classes, cuda), _t(boxes, cuda), _t(off, cuda))
    lh, ph, rh, mh = EvalStepFromBoxes(*args, heads, image_wh, anc, C, 0.5, iou_type, target_anchors=tanc, return_parts=True, **kw)
    lf, pf, rf, mf = EvalStepFromBoxes(*args, wide, image_wh, anc, C, 0.5, iou_type, target_anchors=tanc, return_parts=True, **kw)
    assert_bits_equal(_bits(lh), _bits(lf))
    assert_bits_equal(_bits(ph), _bits(pf))
    _assert_same_rows(rh, rf)
    assert np.array_equal(mh.cpu().numpy(), mf.cpu().numpy(), equal_nan=True)


def test_graph_replay_after_rewriting_heads_and_scale(lib, cuda):
    from tfmv_b200 import runtime
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad
    case = CASES[0]
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, _, y_pred, anc, tanc = _case_inputs(case)
    heads = _plant_half(y_pred, case, torch.bfloat16, cuda)
    scale = torch.full((1,), 1024.0, dtype=torch.float32, device=cuda)
    bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    step = runtime.capture(lambda: GetLossFromBoxesAndGrad(cd, bd, od, heads, image_wh, anc, C, 0.5, iou_type, target_anchors=tanc,
                                                           grad_dtype=torch.bfloat16, grad_scale=scale))
    for h in heads:
        h.copy_((torch.randn(h.shape, device=cuda) * 2.0).to(torch.bfloat16))
    scale.fill_(0.125)
    r_loss, r_grads = step()
    e_loss, e_grads = GetLossFromBoxesAndGrad(cd, bd, od, [h.float() for h in heads], image_wh, anc, C, 0.5, iou_type,
                                              target_anchors=tanc)
    assert_bits_equal(_bits(r_loss), _bits(e_loss))
    _expect_grads(r_grads, e_grads, torch.bfloat16, 0.125)


@pytest.mark.parametrize("call", ["forward", "backward"])
def test_half_call_makes_no_fp32_copy(lib, cuda, call):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLoss, GetLossFromBoxesAndGrad
    case = ((416, 416), 80, 3, "ciou", False)
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, y_true, y_pred, anc, tanc = _case_inputs(case)
    heads = [h.repeat(8, 1, 1, 1) for h in _plant_half(y_pred, case, torch.float16, cuda)]
    if call == "forward":
        yt = [_t(y, cuda).repeat(8, 1, 1, 1, 1) for y in y_true]
        run = lambda: GetLoss(yt, heads, image_wh, anc, 0.5, iou_type)
    else:
        bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
        heads = [h[:B].contiguous() for h in heads]
        run = lambda: GetLossFromBoxesAndGrad(cd, bd, od, heads, image_wh, anc, C, 0.5, iou_type, target_anchors=tanc,
                                              grad_dtype=torch.float16)
    run()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    run()
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < sum(h.numel() for h in heads) * 4
