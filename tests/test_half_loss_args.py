"""CPU: argument checks of the typed YOLO loss entries that read bf16 / fp16 y_pred in place and write the gradient in
the caller's type (b200_yolo_loss_typed, b200_yolo_loss_grad_typed, b200_yolo_loss_from_boxes_typed,
b200_yolo_loss_from_boxes_grad_typed), and the shims' grad_dtype refusal.  Every refusal below is decided before the
first CUDA call, so none needs a device; messages name the entry and the offending level."""
import ctypes

import numpy as np
import pytest

FAKE = 1 << 20   # 256-byte aligned and never dereferenced
F32, BF16, F16 = 0, 1, 2
P3 = ctypes.c_void_p * 3
f = ctypes.c_float
HW = (ctypes.c_int32 * 6)(13, 13, 26, 26, 52, 52)
ANC = (ctypes.c_float * 18)(*[10.0] * 18)
IMG = (ctypes.c_float * 2)(416.0, 416.0)


def _err(lib):
    return lib.b200_last_error().decode()


def _p3(levels):
    return P3(*(levels if levels is not None else (FAKE, FAKE, FAKE)))


def _dense(lib, pred=None, pred_dtype=BF16):
    return lib.b200_yolo_loss_typed(_p3(None), _p3(pred), pred_dtype, HW, 2, 3, 80, ctypes.addressof(ANC), ctypes.addressof(IMG),
                                    f(0.5), 2, 0, f(2), FAKE, FAKE, None, FAKE, 1 << 40, None)


def _dense_grad(lib, pred=None, pred_dtype=BF16, grad=(), grad_dtype=BF16):
    g = None if grad is None else _p3(grad if grad != () else None)
    return lib.b200_yolo_loss_grad_typed(_p3(None), _p3(pred), pred_dtype, HW, 2, 3, 80, ctypes.addressof(ANC),
                                         ctypes.addressof(IMG), f(0.5), 2, 0, f(2), FAKE, FAKE, g, grad_dtype, None, FAKE,
                                         1 << 40, None)


def _boxes(lib, pred=None, pred_dtype=F16):
    return lib.b200_yolo_loss_from_boxes_typed(FAKE, FAKE, FAKE, 10, ctypes.addressof(ANC), _p3(pred), pred_dtype, HW, 2, 3, 80,
                                               ctypes.addressof(ANC), ctypes.addressof(IMG), f(0.5), 2, 0, f(2), FAKE, FAKE,
                                               None, FAKE, 1 << 40, None)


def _boxes_grad(lib, pred=None, pred_dtype=F16, grad=(), grad_dtype=F16):
    g = None if grad is None else _p3(grad if grad != () else None)
    return lib.b200_yolo_loss_from_boxes_grad_typed(FAKE, FAKE, FAKE, 10, ctypes.addressof(ANC), _p3(pred), pred_dtype, HW, 2, 3,
                                                    80, ctypes.addressof(ANC), ctypes.addressof(IMG), f(0.5), 2, 0, f(2), FAKE,
                                                    FAKE, g, grad_dtype, FAKE, FAKE, 1 << 40, None)


@pytest.mark.parametrize("code", [-1, 3, 7])
def test_dtype_codes_outside_the_enum_are_refused(lib, code):
    assert _dense(lib, pred_dtype=code) == -1 and "b200_yolo_loss: pred_dtype %d" % code in _err(lib)
    assert _boxes(lib, pred_dtype=code) == -1 and "b200_yolo_loss_from_boxes: pred_dtype %d" % code in _err(lib)
    assert _dense_grad(lib, pred_dtype=code) == -1 and "b200_yolo_loss_grad: pred_dtype %d" % code in _err(lib)
    assert _dense_grad(lib, grad_dtype=code) == -1 and "b200_yolo_loss_grad: grad_dtype %d" % code in _err(lib)
    assert _boxes_grad(lib, pred_dtype=code) == -1 and "b200_yolo_loss_from_boxes_grad: pred_dtype %d" % code in _err(lib)
    assert _boxes_grad(lib, grad_dtype=code) == -1 and "b200_yolo_loss_from_boxes_grad: grad_dtype %d" % code in _err(lib)


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
def test_null_prediction_levels(lib, dtype):
    assert _dense(lib, pred=(FAKE, 0, FAKE), pred_dtype=dtype) == -1 and "bad level 1" in _err(lib)
    assert _boxes(lib, pred=(FAKE, FAKE, 0), pred_dtype=dtype) == -1 and "bad level 2" in _err(lib)
    assert _dense_grad(lib, pred=(0, FAKE, FAKE), pred_dtype=dtype) == -1 and "bad level 0" in _err(lib)
    assert _boxes_grad(lib, pred=(FAKE, 0, FAKE), pred_dtype=dtype) == -1 and "bad level 1" in _err(lib)
    assert lib.b200_yolo_loss_typed(_p3(None), None, dtype, HW, 2, 3, 80, ctypes.addressof(ANC), ctypes.addressof(IMG), f(0.5), 2,
                                    0, f(2), FAKE, FAKE, None, FAKE, 1 << 40, None) == -1
    assert "null argument" in _err(lib)


@pytest.mark.parametrize("grad_dtype", [F32, BF16, F16])
def test_gradient_levels(lib, grad_dtype):
    assert _dense_grad(lib, grad=None, grad_dtype=grad_dtype) == -1 and "b200_yolo_loss_grad: null out_grad" in _err(lib)
    assert _boxes_grad(lib, grad=None, grad_dtype=grad_dtype) == -1
    assert "b200_yolo_loss_from_boxes_grad: null out_grad" in _err(lib)
    assert _dense_grad(lib, grad=(FAKE, 0, FAKE), grad_dtype=grad_dtype) == -1
    assert "b200_yolo_loss_grad: grad level 1 null or not 16-byte aligned" in _err(lib)
    # a 2-byte gradient is still written with 16-byte stores: every level must be 16-byte aligned
    assert _dense_grad(lib, grad=(FAKE, FAKE, FAKE + 2), grad_dtype=grad_dtype) == -1
    assert "b200_yolo_loss_grad: grad level 2 null or not 16-byte aligned" in _err(lib)
    assert _boxes_grad(lib, grad=(FAKE + 8, FAKE, FAKE), grad_dtype=grad_dtype) == -1
    assert "b200_yolo_loss_from_boxes_grad: grad level 0 null or not 16-byte aligned" in _err(lib)


def test_typed_entries_keep_the_shape_checks(lib):
    assert lib.b200_yolo_loss_typed(_p3(None), _p3(None), BF16, HW, 2, 9, 80, ctypes.addressof(ANC), ctypes.addressof(IMG), f(0.5),
                                    2, 0, f(2), FAKE, FAKE, None, FAKE, 1 << 40, None) == -1
    assert "unsupported shape" in _err(lib)
    assert lib.b200_yolo_loss_from_boxes_grad_typed(FAKE, FAKE, FAKE, 10, ctypes.addressof(ANC), _p3(None), F16, HW, 2, 3, 80,
                                                    ctypes.addressof(ANC), ctypes.addressof(IMG), f(0.5), 5, 0, f(2), FAKE, FAKE,
                                                    _p3(None), F16, None, FAKE, 1 << 40, None) == -1
    assert "iou_type must be iou/diou/ciou" in _err(lib)


@pytest.mark.parametrize("bad", ["float64", "int32", "float32-string"])
def test_shims_refuse_other_gradient_types(lib, bad):
    import torch
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossAndGrad, GetLossFromBoxesAndGrad
    dtype = {"float64": torch.float64, "int32": torch.int32, "float32-string": "float32"}[bad]
    anc = np.ones((3, 3, 2), np.float32) * 10
    heads = [np.zeros((1, s, s, 255), np.float32) for s in (13, 26, 52)]
    y_true = [np.zeros((1, s, s, 3, 85), np.float32) for s in (13, 26, 52)]
    with pytest.raises(ValueError, match="grad_dtype"):
        GetLossAndGrad(y_true, heads, (416, 416), anc, grad_dtype=dtype)
    boxes, classes, off = np.zeros((1, 4), np.float32), np.ones(1, np.int32), np.array([0, 1], np.int32)
    with pytest.raises(ValueError, match="grad_dtype"):
        GetLossFromBoxesAndGrad(classes, boxes, off, heads, (416, 416), anc, 80, grad_dtype=dtype)
