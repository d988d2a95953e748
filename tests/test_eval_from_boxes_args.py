"""CPU: argument checks and workspace sizes of the validation step from box lists (b200_effdet_eval_step_from_boxes,
b200_yolo_ground_truth_from_boxes) and of the padded mAP (b200_map_padded).  Every refusal below is decided before anything is enqueued, so none needs a device;
messages name the offending argument."""
import ctypes

import numpy as np
import pytest

FAKE = 1 << 20   # 256-byte aligned and never dereferenced
D0 = (64, 64, 32, 32, 16, 16, 8, 8, 4, 4)
D7 = (192, 192, 96, 96, 48, 48, 24, 24, 12, 12)
L = 5
P = ctypes.c_void_p * L
f = ctypes.c_float


def _hw(levels=D0):
    return (ctypes.c_int32 * len(levels))(*levels)


def _err(lib):
    return lib.b200_last_error().decode()


def _step(lib, C=81, B=2, total=10, gt_boxes=FAKE, gt_classes=FAKE, gt_offsets=FAKE, pred_boxes=None, pred_classes=None,
          sums=FAKE, decoded=None, max_out=200, metric=5, out_boxes=FAKE, ws=FAKE, ws_bytes=1 << 40, hw=None, num_levels=L):
    return lib.b200_effdet_eval_step_from_boxes(
        num_levels, _hw() if hw is None else hw, 9, FAKE, C, B, gt_boxes, gt_classes, gt_offsets, total, f(0.5),
        pred_boxes if pred_boxes is not None else P(*[FAKE] * L), pred_classes if pred_classes is not None else P(*[FAKE] * L),
        f(0.25), f(1.5), f(0.1), f(0.0), sums, decoded, max_out, f(0.5), f(1e-4), metric, out_boxes, FAKE, FAKE, None, None,
        FAKE, ws, ws_bytes, None)


def _map(lib, B=2, K=200, id_bytes=8, pred_boxes=FAKE, pred_count=FAKE, gt_boxes=FAKE, gt_classes=FAKE, total_gt=10,
         gt_offsets=FAKE, out=FAKE, class_num=80):
    return lib.b200_map_padded(pred_boxes, FAKE, id_bytes, FAKE, pred_count, B, K, gt_boxes, gt_classes, total_gt, gt_offsets, None,
                               class_num, ctypes.c_double(0.5), out, None)


YOLO_416 = (13, 13, 26, 26, 52, 52)
YOLO_608 = (19, 19, 38, 38, 76, 76)
ANC = np.arange(1, 25, dtype=np.float32)   # 3 levels x up to 4 anchors x (w, h), pixels
IMG = np.array([416, 416], np.float32)


def _yhw(hw=YOLO_416):
    return (ctypes.c_int32 * 6)(*hw)


def _rows(lib, B=2, total=10, boxes=FAKE, classes=FAKE, offsets=FAKE, rows=FAKE, count=FAKE, hw=None, A=3, C=80, anc=ANC, img=IMG,
          ws=FAKE, ws_bytes=1 << 40):
    ptr = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    return lib.b200_yolo_ground_truth_from_boxes(boxes, classes, offsets, total, B, _yhw() if hw is None else hw, A, C, ptr(anc),
                                                 ptr(img), rows, count, ws, ws_bytes, None)


# eval workspace (candidate store + per-CTA partials for 148 SMs) + int32 match per anchor (256-aligned)
@pytest.mark.parametrize("levels,B,want", [
    (D0, 1, 1766144 + 196608), (D0, 128, 189746688 + 25141248), (D7, 1, 12814592 + 1767936), (D7, 16, 200742144 + 28283904),
])
def test_workspace_bytes_pinned(lib, levels, B, want):
    assert lib.b200_effdet_eval_step_from_boxes_workspace_bytes(L, _hw(levels), 9, B, 200) == want


def test_workspace_bytes_of_a_bad_spec_is_zero(lib):
    assert lib.b200_effdet_eval_step_from_boxes_workspace_bytes(0, _hw(), 9, 2, 200) == 0
    assert lib.b200_effdet_eval_step_from_boxes_workspace_bytes(L, _hw(), 0, 2, 200) == 0
    assert lib.b200_effdet_eval_step_from_boxes_workspace_bytes(L, _hw(), 9, -1, 200) == 0
    assert lib.b200_effdet_eval_step_from_boxes_workspace_bytes(L, None, 9, 2, 200) == 0


def test_eval_step_from_boxes_refusals(lib):
    need = lib.b200_effdet_eval_step_from_boxes_workspace_bytes(L, _hw(), 9, 2, 200)
    assert _step(lib, sums=0) == -1 and "null argument" in _err(lib)
    assert _step(lib, gt_offsets=0) == -1 and "null gt_offsets" in _err(lib)
    assert _step(lib, total=-1) == -1 and "negative total_boxes" in _err(lib)
    assert _step(lib, gt_boxes=0) == -1 and "null gt_boxes" in _err(lib)
    assert _step(lib, gt_classes=0) == -1 and "gt_classes" in _err(lib)
    assert _step(lib, gt_boxes=FAKE + 4) == -1 and "gt_boxes not 16-byte aligned" in _err(lib)
    assert _step(lib, hw=_hw((64, 0) + D0[2:])) == -1 and "bad level spec" in _err(lib)
    assert _step(lib, num_levels=9) == -1 and "bad level spec" in _err(lib)
    assert _step(lib, C=3) == -4 and "classes_num 3 < 4" in _err(lib)
    assert _step(lib, C=129) == -4 and "classes_num 129 > 128" in _err(lib)
    assert _step(lib, C=401) == -4 and "outside [1,400]" in _err(lib)
    assert _step(lib, B=-1) == -1 and "negative batch" in _err(lib)
    assert _step(lib, metric=1) == -1 and "iou_type" in _err(lib)
    assert _step(lib, max_out=0) == -4 and "max_out 0" in _err(lib)
    assert _step(lib, max_out=4097) == -4 and "max_out 4097" in _err(lib)
    assert _step(lib, out_boxes=0) == -1 and "null output" in _err(lib)
    assert _step(lib, pred_classes=P(FAKE, FAKE, 0, FAKE, FAKE)) == -1 and "null level 2" in _err(lib)
    assert _step(lib, pred_boxes=P(FAKE, FAKE, FAKE, FAKE + 8, FAKE)) == -1 and "level 3" in _err(lib)
    assert _step(lib, decoded=P(FAKE, FAKE, FAKE, FAKE, FAKE + 4)) == -1 and "level 4" in _err(lib)
    assert _step(lib, ws_bytes=need - 1) == -2 and "workspace" in _err(lib)
    assert _step(lib, ws=0) == -2
    assert _step(lib, ws=FAKE + 16, ws_bytes=need) == -1 and "256-byte" in _err(lib)
    # nothing to do for an empty batch
    assert _step(lib, B=0) == 0


def test_map_padded_refusals(lib):
    assert _map(lib, B=-1) == -1 and "negative num_images" in _err(lib)
    assert _map(lib, class_num=0) == -1 and "class_num 0" in _err(lib)
    assert _map(lib, K=0) == -4 and "max_out 0" in _err(lib)
    assert _map(lib, K=4097) == -4 and "max_out 4097" in _err(lib)
    assert _map(lib, id_bytes=2) == -1 and "class_id_bytes" in _err(lib)
    assert _map(lib, pred_boxes=0) == -1 and "null prediction" in _err(lib)
    assert _map(lib, pred_count=0) == -1 and "null prediction" in _err(lib)
    assert _map(lib, gt_offsets=0) == -1 and "gt_offsets" in _err(lib)
    assert _map(lib, total_gt=-1) == -1 and "negative total_gt" in _err(lib)
    assert _map(lib, gt_boxes=0) == -1 and "null gt_boxes" in _err(lib)
    assert _map(lib, gt_classes=0) == -1 and "gt_classes" in _err(lib)
    assert _map(lib, out=0) == -1 and "out" in _err(lib)
    assert _map(lib, B=0) == 0


# one int32 key per box, 256-byte aligned: independent of the grid and the batch
@pytest.mark.parametrize("hw,B,total,want", [(YOLO_416, 1, 0, 256), (YOLO_416, 64, 100, 512), (YOLO_608, 64, 6400, 25600),
                                             (YOLO_608, 8, 65, 512)])
def test_yolo_ground_truth_workspace_bytes_pinned(lib, hw, B, total, want):
    assert lib.b200_yolo_ground_truth_from_boxes_workspace_bytes(_yhw(hw), B, 3, total) == want


def test_yolo_ground_truth_workspace_bytes_of_a_bad_spec_is_zero(lib):
    assert lib.b200_yolo_ground_truth_from_boxes_workspace_bytes(None, 2, 3, 10) == 0
    assert lib.b200_yolo_ground_truth_from_boxes_workspace_bytes(_yhw((13, 0, 26, 26, 52, 52)), 2, 3, 10) == 0
    assert lib.b200_yolo_ground_truth_from_boxes_workspace_bytes(_yhw(), -1, 3, 10) == 0
    assert lib.b200_yolo_ground_truth_from_boxes_workspace_bytes(_yhw(), 2, 9, 10) == 0
    assert lib.b200_yolo_ground_truth_from_boxes_workspace_bytes(_yhw(), 2, 3, -1) == 0


def test_yolo_ground_truth_from_boxes_refusals(lib):
    assert _rows(lib, B=-1) == -1 and "negative batch" in _err(lib)
    assert _rows(lib, total=-1) == -1 and "negative total_boxes" in _err(lib)
    assert _rows(lib, offsets=0) == -1 and "null offsets" in _err(lib)
    assert _rows(lib, boxes=0) == -1 and "null boxes" in _err(lib)
    assert _rows(lib, classes=0) == -1 and "classes" in _err(lib)
    assert _rows(lib, rows=0) == -1 and "rows" in _err(lib)
    assert _rows(lib, boxes=FAKE + 4) == -1 and "boxes not 16-byte aligned" in _err(lib)
    assert _rows(lib, count=0) == -1 and "null count" in _err(lib)
    assert _rows(lib, A=9) == -1 and "bad geometry" in _err(lib)
    assert _rows(lib, A=0) == -1 and "bad geometry" in _err(lib)
    assert _rows(lib, anc=None) == -1 and "bad geometry" in _err(lib)
    assert _rows(lib, img=None) == -1 and "bad geometry" in _err(lib)
    assert _rows(lib, hw=_yhw((13, 13, 0, 26, 52, 52))) == -1 and "bad geometry" in _err(lib)
    assert _rows(lib, ws_bytes=10) == -2 and "workspace" in _err(lib)
    assert _rows(lib, ws=0) == -2
    assert _rows(lib, B=0) == 0
    assert _rows(lib, B=0, total=0, boxes=0, classes=0, rows=0, count=0) == 0


def test_python_entry_points_need_a_device():
    import torch
    from tfmv_b200.ai_models.efficientnet.utils.anchors import Anchors
    from tfmv_b200.ai_models.utils.mAP import Get_mAP_padded
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    a = Anchors(0, 0, (10, 10), 3, [(1.0, 1.0)], 3.0)
    boxes, classes, off = np.zeros((1, 4), np.float32), np.ones(1, np.int32), np.array([0, 1], np.int32)
    with pytest.raises(RuntimeError, match="CUDA device"):
        a.eval_step_from_boxes(boxes, classes, off, [np.zeros((1, 10, 10, 3, 4), np.float32)],
                               [np.zeros((1, 10, 10, 3, 5), np.float32)])
    nms = dict(boxes=np.zeros((1, 4, 4), np.float32), classes_id=np.zeros((1, 4), np.int64),
               scores=np.zeros((1, 4), np.float32), count=np.zeros(1, np.int32))
    with pytest.raises(RuntimeError, match="CUDA device"):
        Get_mAP_padded(boxes, classes, off, nms, 5)
    from tfmv_b200.ai_models.utils.tf_yolo_utils import EvalStepFromBoxes, GetGroudTruthFromBoxes
    anc = np.ones((3, 3, 2), np.float32) * 10
    with pytest.raises(RuntimeError, match="CUDA device"):
        GetGroudTruthFromBoxes(classes, boxes, off, (416, 416), anc, 80)
    heads = [np.zeros((1, s, s, 255), np.float32) for s in (13, 26, 52)]
    with pytest.raises(RuntimeError, match="CUDA device"):
        EvalStepFromBoxes(classes, boxes, off, heads, (416, 416), anc, 80)
