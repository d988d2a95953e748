"""CPU: argument checks and workspace size of the EfficientDet loss from box lists (b200_effdet_loss_from_boxes_*).
Every refusal below is decided before the first CUDA call, so none needs a device; messages name the offending level."""
import ctypes

import pytest

FAKE = 1 << 20   # 256-byte aligned and never dereferenced
D0 = (64, 64, 32, 32, 16, 16, 8, 8, 4, 4)
D7 = (192, 192, 96, 96, 48, 48, 24, 24, 12, 12)
L = 5
P = ctypes.c_void_p * L


def _hw(levels=D0):
    return (ctypes.c_int32 * len(levels))(*levels)


def _err(lib):
    return lib.b200_last_error().decode()


def _match(lib, hw=None, B=2, total=10, gt_boxes=FAKE, sums=FAKE, ws=FAKE, ws_bytes=1 << 40, num_levels=L):
    hw = _hw() if hw is None else hw
    return lib.b200_effdet_loss_from_boxes_match(num_levels, hw, 9, FAKE, B, gt_boxes, FAKE, total, ctypes.c_float(0.5), sums, ws,
                                                 ws_bytes, None)


def _grad(lib, C=81, B=2, total=10, pred_boxes=None, pred_classes=None, grad_boxes=None, grad_classes=None, numel=None,
          ws=FAKE, ws_bytes=1 << 40, gt_boxes=FAKE):
    nm = numel if numel is not None else (ctypes.c_double * L)(*[1.0] * L)
    f = ctypes.c_float
    return lib.b200_effdet_loss_from_boxes_grad(L, _hw(), 9, FAKE, C, B, gt_boxes, FAKE, total,
                                                pred_boxes if pred_boxes is not None else P(*[FAKE] * L),
                                                pred_classes if pred_classes is not None else P(*[FAKE] * L),
                                                f(0.25), f(1.5), f(0.1), f(0.0), nm, FAKE, grad_boxes, grad_classes, ws, ws_bytes,
                                                None)


# (levels, B) -> bytes: int32 match per anchor (256-aligned) + 3 doubles for each of at most 16384 + L CTAs
@pytest.mark.parametrize("levels,B,want", [
    (D0, 1, 196608 + 393472), (D0, 128, 25141248 + 393472), (D7, 1, 1767936 + 393472), (D7, 16, 28283904 + 393472),
])
def test_workspace_bytes_pinned(lib, levels, B, want):
    assert lib.b200_effdet_loss_from_boxes_workspace_bytes(L, _hw(levels), 9, B) == want


def test_workspace_bytes_of_a_bad_spec_is_zero(lib):
    assert lib.b200_effdet_loss_from_boxes_workspace_bytes(0, _hw(), 9, 2) == 0
    assert lib.b200_effdet_loss_from_boxes_workspace_bytes(L, _hw(), 0, 2) == 0
    assert lib.b200_effdet_loss_from_boxes_workspace_bytes(L, _hw(), 9, -1) == 0
    assert lib.b200_effdet_loss_from_boxes_workspace_bytes(L, None, 9, 2) == 0


def test_match_refusals(lib):
    need = lib.b200_effdet_loss_from_boxes_workspace_bytes(L, _hw(), 9, 2)
    assert _match(lib, sums=0) == -1 and "null argument" in _err(lib)
    assert _match(lib, hw=_hw((64, 0) + D0[2:])) == -1 and "bad level spec" in _err(lib)
    assert _match(lib, num_levels=9) == -1 and "bad level spec" in _err(lib)
    assert _match(lib, B=-1) == -1 and "negative" in _err(lib)
    assert _match(lib, gt_boxes=0) == -1 and "null gt_boxes" in _err(lib)
    assert _match(lib, ws_bytes=need - 1) == -2 and "workspace" in _err(lib)
    assert _match(lib, ws=0) == -2
    assert _match(lib, ws=FAKE + 16, ws_bytes=need) == -1 and "256-byte" in _err(lib)


def test_grad_refusals(lib):
    need = lib.b200_effdet_loss_from_boxes_workspace_bytes(L, _hw(), 9, 2)
    assert _grad(lib, C=3) == -4 and "classes_num >= 4" in _err(lib)
    assert _grad(lib, C=0) == -4
    assert _grad(lib, numel=0) == -1 and "null argument" in _err(lib)
    assert _grad(lib, B=-1) == -1
    assert _grad(lib, gt_boxes=0) == -1 and "null gt_boxes" in _err(lib)
    assert _grad(lib, gt_boxes=FAKE + 4) == -1 and "gt_boxes not 16-byte aligned" in _err(lib)
    assert _grad(lib, pred_classes=P(FAKE, FAKE, 0, FAKE, FAKE)) == -1 and "level 2" in _err(lib)
    assert _grad(lib, pred_boxes=P(FAKE, FAKE, FAKE, FAKE + 8, FAKE)) == -1 and "level 3" in _err(lib)
    assert _grad(lib, grad_classes=P(FAKE, 0, FAKE, FAKE, FAKE)) == -1 and "grad_classes at level 1" in _err(lib)
    assert _grad(lib, grad_boxes=P(FAKE, FAKE, FAKE, FAKE, FAKE + 4)) == -1 and "level 4" in _err(lib)
    assert _grad(lib, numel=(ctypes.c_double * L)(1.0, 1.0, 0.0, 1.0, 1.0)) == -1 and "numel of level 2" in _err(lib)
    assert _grad(lib, ws_bytes=need - 1) == -2 and "workspace" in _err(lib)
    assert _grad(lib, ws=FAKE + 16, ws_bytes=need) == -1 and "256-byte" in _err(lib)


def test_python_entry_points_need_a_device():
    import numpy as np
    import torch
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes, get_loss_from_boxes_and_grad
    from tfmv_b200.ai_models.efficientnet.utils.anchors import Anchors
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    a = Anchors(0, 0, (10, 10), 3, [(1.0, 1.0)], 3.0)
    boxes, classes, off = np.zeros((1, 4), np.float32), np.ones(1, np.int32), np.array([0, 1], np.int32)
    for fn in (get_loss_from_boxes, get_loss_from_boxes_and_grad):
        with pytest.raises(RuntimeError, match="CUDA device"):
            fn(a, boxes, classes, off, [np.zeros((1, 10, 10, 3, 4), np.float32)], [np.zeros((1, 10, 10, 3, 5), np.float32)])
