"""CPU: argument checks of the typed EfficientDet loss entries that read bf16 / fp16 heads in place and write the
gradients in the caller's type (b200_focal_box_partial_sums_typed, b200_focal_box_partial_sums_indexed_typed,
b200_focal_box_grad_typed, b200_focal_box_grad_indexed_typed, b200_effdet_loss_from_boxes_grad_typed), and the shims'
grad_dtype / grad_scale refusals.  Every refusal below is decided before the first CUDA call, so none needs a device;
messages name the entry and the offending level."""
import ctypes

import numpy as np
import pytest

FAKE = 1 << 20   # 256-byte aligned and never dereferenced
F32, BF16, F16 = 0, 1, 2
L = 5
P = ctypes.c_void_p * L
f = ctypes.c_float
D0 = (64, 64, 32, 32, 16, 16, 8, 8, 4, 4)
ANCHORS = (ctypes.c_ulonglong * L)(*[2 * h * w * 9 for h, w in zip(D0[::2], D0[1::2])])
NUMEL = (ctypes.c_double * L)(*[1.0] * L)


def _err(lib):
    return lib.b200_last_error().decode()


def _p(levels=None):
    return P(*(levels if levels is not None else [FAKE] * L))


def _sums(lib, indexed=False, pred_boxes=None, pred_classes=None, pred_dtype=BF16, ws_bytes=1 << 40, C=81):
    fn = lib.b200_focal_box_partial_sums_indexed_typed if indexed else lib.b200_focal_box_partial_sums_typed
    return fn(L, ANCHORS, C, _p(), _p(), _p(), _p(pred_boxes), _p(pred_classes), pred_dtype, f(0.25), f(1.5), f(0.1), f(0.0),
              FAKE, FAKE, ws_bytes, None)


def _grad(lib, indexed=False, pred_classes=None, pred_dtype=BF16, grad_boxes=(), grad_classes=(), grad_dtype=BF16, C=81):
    fn = lib.b200_focal_box_grad_indexed_typed if indexed else lib.b200_focal_box_grad_typed
    gb = None if grad_boxes is None else _p(grad_boxes if grad_boxes != () else None)
    gc = None if grad_classes is None else _p(grad_classes if grad_classes != () else None)
    return fn(L, ANCHORS, C, _p(), _p(), _p(), _p(pred_classes), pred_dtype, f(0.25), f(1.5), f(0.1), f(0.0), FAKE, NUMEL, gb, gc,
              grad_dtype, FAKE, None)


def _boxes(lib, pred_boxes=None, pred_dtype=F16, grad_boxes=(), grad_classes=(), grad_dtype=F16, ws_bytes=1 << 40, C=81):
    gb = None if grad_boxes is None else _p(grad_boxes if grad_boxes != () else None)
    gc = None if grad_classes is None else _p(grad_classes if grad_classes != () else None)
    return lib.b200_effdet_loss_from_boxes_grad_typed(L, (ctypes.c_int32 * 10)(*D0), 9, FAKE, C, 2, FAKE, FAKE, 10, _p(pred_boxes),
                                                      _p(), pred_dtype, f(0.25), f(1.5), f(0.1), f(0.0), NUMEL, FAKE, gb, gc,
                                                      grad_dtype, FAKE, FAKE, ws_bytes, None)


@pytest.mark.parametrize("code", [-1, 3, 7])
def test_dtype_codes_outside_the_enum_are_refused(lib, code):
    for indexed in (False, True):
        assert _sums(lib, indexed, pred_dtype=code) == -1
        assert "b200_focal_box_partial_sums: pred_dtype %d is not a B200_DTYPE_* code" % code in _err(lib)
        assert _grad(lib, indexed, pred_dtype=code) == -1 and "b200_focal_box_grad: pred_dtype %d" % code in _err(lib)
        assert _grad(lib, indexed, grad_dtype=code) == -1 and "b200_focal_box_grad: grad_dtype %d" % code in _err(lib)
    assert _boxes(lib, pred_dtype=code) == -1 and "b200_effdet_loss_from_boxes_grad: pred_dtype %d" % code in _err(lib)
    assert _boxes(lib, grad_dtype=code) == -1 and "b200_effdet_loss_from_boxes_grad: grad_dtype %d" % code in _err(lib)


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
def test_null_arguments(lib, dtype):
    fn = lib.b200_focal_box_partial_sums_typed
    assert fn(L, ANCHORS, 81, _p(), None, _p(), _p(), _p(), dtype, f(0.25), f(1.5), f(0.1), f(0.0), FAKE, FAKE, 1 << 40, None) == -1
    assert "b200_focal_box_partial_sums: null argument" in _err(lib)
    fn = lib.b200_focal_box_partial_sums_indexed_typed
    assert fn(L, ANCHORS, 81, _p(), None, _p(), _p(), _p(), dtype, f(0.25), f(1.5), f(0.1), f(0.0), FAKE, FAKE, 1 << 40, None) == -1
    assert "b200_focal_box_partial_sums_indexed: null argument" in _err(lib)
    # a level without its class half and its box half
    assert _sums(lib, pred_boxes=[FAKE, FAKE, 0, FAKE, FAKE], pred_classes=[FAKE, FAKE, 0, FAKE, FAKE], pred_dtype=dtype) == -1
    assert "null level 2" in _err(lib)
    assert _grad(lib, pred_classes=[FAKE, 0, FAKE, FAKE, FAKE], pred_dtype=dtype) == -1
    assert "b200_focal_box_grad: null class tensors at level 1" in _err(lib)
    assert _boxes(lib, pred_boxes=[FAKE, FAKE, FAKE, 0, FAKE], pred_dtype=dtype) == -1
    assert "b200_effdet_loss_from_boxes_grad: null prediction at level 3" in _err(lib)
    assert _boxes(lib, grad_classes=[FAKE, FAKE, FAKE, FAKE, 0], grad_dtype=dtype) == -1
    assert "b200_effdet_loss_from_boxes_grad: null grad_classes at level 4" in _err(lib)


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
def test_two_byte_tensors_keep_the_16_byte_rule(lib, dtype):
    """Half heads and gradients are still read and written in 4-element groups: every level must be 16-byte aligned."""
    assert _sums(lib, pred_classes=[FAKE, FAKE + 2, FAKE, FAKE, FAKE], pred_dtype=dtype) == -1
    assert "b200_focal_box_partial_sums: level 1 tensors must be 16-byte aligned" in _err(lib)
    assert _sums(lib, True, pred_boxes=[FAKE, FAKE, FAKE, FAKE, FAKE + 8], pred_dtype=dtype) == -1
    assert "level 4 tensors must be 16-byte aligned" in _err(lib)
    assert _grad(lib, grad_classes=[FAKE + 8, FAKE, FAKE, FAKE, FAKE], grad_dtype=dtype) == -1
    assert "b200_focal_box_grad: level 0 class tensors must be 16-byte aligned" in _err(lib)
    assert _grad(lib, True, grad_boxes=[FAKE, FAKE, FAKE + 2, FAKE, FAKE], grad_dtype=dtype) == -1
    assert "b200_focal_box_grad: level 2 box tensors must be 16-byte aligned" in _err(lib)
    assert _boxes(lib, pred_boxes=[FAKE, FAKE + 4, FAKE, FAKE, FAKE], pred_dtype=dtype) == -1
    assert "b200_effdet_loss_from_boxes_grad: level 1 tensors must be 16-byte aligned" in _err(lib)
    assert _boxes(lib, grad_boxes=[FAKE, FAKE, FAKE, FAKE, FAKE + 2], grad_dtype=dtype) == -1
    assert "b200_effdet_loss_from_boxes_grad: level 4 tensors must be 16-byte aligned" in _err(lib)


def test_workspace_and_class_count(lib):
    assert _sums(lib, ws_bytes=8) == -2 and "b200_focal_box_partial_sums: workspace 8 < required" in _err(lib)
    assert _boxes(lib, ws_bytes=8) == -2 and "b200_effdet_loss_from_boxes_grad: workspace 8 < required" in _err(lib)
    assert _boxes(lib, C=3) == -4 and "needs classes_num >= 4 (got 3)" in _err(lib)
    assert _grad(lib, True, C=3) == -4 and "b200_focal_box_grad_indexed: needs classes_num >= 4" in _err(lib)


def _d0_heads():
    shapes = [(1, h, w, 9) for h, w in zip(D0[::2], D0[1::2])]
    return shapes, [np.zeros(s + (4,), np.float32) for s in shapes], [np.zeros(s + (81,), np.float32) for s in shapes]


@pytest.mark.parametrize("bad", ["float64", "int32", "float32-string"])
def test_shims_refuse_other_gradient_types(lib, bad):
    import torch
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_and_grad, get_loss_from_boxes_and_grad
    from tfmv_b200.ai_models.efficientnet.utils.anchors import Anchors
    dtype = {"float64": torch.float64, "int32": torch.int32, "float32-string": "float32"}[bad]
    shapes, pb, pc = _d0_heads()
    masks = [np.zeros(s, bool) for s in shapes]
    with pytest.raises(ValueError, match="grad_dtype"):
        get_loss_and_grad(pb, pc, masks, pb, pc, grad_dtype=dtype)
    a = Anchors(3, 7, (512, 512), 3, [(1.0, 1.0), (1.4, 0.7), (0.7, 1.4)], 4.0)
    boxes, classes, off = np.zeros((1, 4), np.float32), np.ones(1, np.int32), np.array([0, 1], np.int32)
    with pytest.raises(ValueError, match="grad_dtype"):
        get_loss_from_boxes_and_grad(a, boxes, classes, off, pb, pc, grad_dtype=dtype)


def test_gradient_scale_must_be_one_fp32_element_on_the_heads_device():
    import torch
    from tfmv_b200 import _tensors as T
    heads = [torch.zeros((2, 4), dtype=torch.bfloat16)]
    for bad in (torch.ones(1, dtype=torch.float64), torch.ones(2), torch.ones((1, 1), dtype=torch.float16)):
        with pytest.raises(ValueError, match="grad_scale"):
            T.grad_out(heads, torch.bfloat16, bad)
    grads, code, scale = T.grad_out(heads, torch.float16, 1024.0)
    assert code == F16 and grads[0].dtype == torch.float16 and grads[0].shape == heads[0].shape
    assert scale.dtype == torch.float32 and scale.numel() == 1 and float(scale) == 1024.0
    assert T.grad_out(heads, torch.float32, None)[2] is None
