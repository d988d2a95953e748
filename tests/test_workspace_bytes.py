"""CPU tests: the workspace sizes the post-processing entry points report.  Callers allocate exactly these byte counts,
so a change in the candidate-store layout that moves them is a change of the public API.  Host-only: no device needed."""
import ctypes

import pytest

YOLO_LEVELS = {416: (13, 13, 26, 26, 52, 52), 608: (19, 19, 38, 38, 76, 76)}
EFFDET_LEVELS = {"d0": (64, 64, 32, 32, 16, 16, 8, 8, 4, 4), "d7": (192, 192, 96, 96, 48, 48, 24, 24, 12, 12)}


@pytest.mark.parametrize("image,batch,want", [
    (416, 1, 345344), (416, 8, 2753024), (608, 1, 733952), (608, 8, 5861632),
])
def test_yolo_decode_nms_workspace_bytes(lib, image, batch, want):
    hw = (ctypes.c_int32 * 6)(*YOLO_LEVELS[image])
    assert lib.b200_yolo_decode_nms_workspace_bytes(hw, batch, 3, 500) == want


@pytest.mark.parametrize("model,images,want", [
    ("d0", 1, 1481984), ("d0", 16, 23683584), ("d7", 1, 12530432), ("d7", 16, 200457984),
])
def test_effdet_postprocess_workspace_bytes(lib, model, images, want):
    hw = (ctypes.c_int32 * 10)(*EFFDET_LEVELS[model])
    assert lib.b200_effdet_postprocess_workspace_bytes(5, hw, 9, images, 200) == want
