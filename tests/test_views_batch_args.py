"""CPU: argument checks of the batched serving entry points (b200_letterbox_batch, b200_unletterbox_boxes_batch).
Every check runs before any CUDA call, so a refusal needs no GPU; the error names the offending frame."""
import ctypes

import pytest

# b200_letterbox_batch(N, imgs, hw, channels, out_w, out_h, bg, out_u8, out_f32, padding_out, resized_wh_out, geometry_out, stream)
FAKE = 0x10000  # never dereferenced: every call below fails its checks (or is N == 0) before a launch


def _call(lib, frames, channels=3, out_wh=(416, 416), out_u8=FAKE, padding=True):
    n = len(frames)
    imgs = (ctypes.c_void_p * max(n, 1))(*[p for p, _, _ in frames])
    hw = (ctypes.c_int32 * max(2 * n, 2))(*[v for _, h, w in frames for v in (h, w)])
    bg = (ctypes.c_uint8 * 3)(0, 0, 0)
    pad = (ctypes.c_int32 * max(4 * n, 4))() if padding else None
    return lib.b200_letterbox_batch(n, imgs, hw, channels, out_wh[0], out_wh[1], bg, out_u8, 0, pad, None, None, None)


def _err(lib):
    return lib.b200_last_error().decode()


def test_letterbox_batch_names_the_bad_frame(lib):
    good = (FAKE, 480, 640)
    # an empty resize (2 x 4000 -> 416^2 gives height 0, as cv2.resize would fail) in frame 2
    assert _call(lib, [good, good, (FAKE, 2, 4000), good]) == -1
    assert "image 2" in _err(lib) and "empty" in _err(lib)
    # a null frame pointer in frame 1
    assert _call(lib, [good, (0, 480, 640), good]) == -1
    assert "image 1" in _err(lib) and "null" in _err(lib)
    # a bad size in frame 3
    assert _call(lib, [good, good, good, (FAKE, 0, 640)]) == -1
    assert "image 3" in _err(lib) and "bad sizes" in _err(lib)
    assert _call(lib, [good, (FAKE, 1 << 24, 8)]) == -1
    assert "image 1" in _err(lib) and "too large" in _err(lib)
    # 4 channels: unsupported, reported at the first frame
    assert _call(lib, [good, good], channels=4) == -4
    assert "image 0" in _err(lib) and "3-channel" in _err(lib)


def test_letterbox_batch_whole_call_arguments(lib):
    good = (FAKE, 480, 640)
    assert _call(lib, []) == 0                                      # N == 0: nothing to do, nothing checked
    assert lib.b200_letterbox_batch(0, None, None, 3, 416, 416, None, None, None, None, None, None, None) == 0
    assert lib.b200_letterbox_batch(-1, None, None, 3, 416, 416, None, None, None, None, None, None, None) == -1
    assert "count" in _err(lib)
    assert _call(lib, [good], out_u8=0) == -1 and "no output buffer" in _err(lib)
    assert _call(lib, [good], padding=False) == -1 and "null argument" in _err(lib)
    assert _call(lib, [good], out_wh=(0, 416)) == -1 and "image 0" in _err(lib)
    bg = (ctypes.c_uint8 * 3)()
    assert lib.b200_letterbox_batch(1, None, None, 3, 416, 416, bg, FAKE, None, (ctypes.c_int32 * 4)(), None, None, None) == -1


def test_unletterbox_boxes_batch_arguments(lib):
    size = (ctypes.c_int32 * 2)(416, 416)
    # b200_unletterbox_boxes_batch(boxes, counts, B, max_rows, image_size, geometry, out_boxes, out_index, out_count, stream)
    assert lib.b200_unletterbox_boxes_batch(0, 0, 0, 10, 0, 0, 0, 0, 0, 0) == 0          # B == 0
    assert lib.b200_unletterbox_boxes_batch(0, 0, -1, 10, size, 0, 0, 0, 0, 0) == -1
    assert lib.b200_unletterbox_boxes_batch(FAKE, 0, 2, 10, size, 0, FAKE, FAKE, FAKE, 0) == -1
    assert "geometry" in _err(lib)
    assert lib.b200_unletterbox_boxes_batch(FAKE, 0, 2, 10, None, FAKE, FAKE, FAKE, FAKE, 0) == -1
    assert "null argument" in _err(lib)
    assert lib.b200_unletterbox_boxes_batch(0, 0, 2, 10, size, FAKE, FAKE, FAKE, FAKE, 0) == -1
    assert "null buffer" in _err(lib)
    assert lib.b200_unletterbox_boxes_batch(FAKE + 4, 0, 2, 10, size, FAKE, FAKE, FAKE, FAKE, 0) == -1
    assert "aligned" in _err(lib)


def test_python_batch_entry_points_need_a_device():
    import torch
    from tfmv_b200.ai_models.utils import image_helper as ih
    from tfmv_b200.views.object_detection import prepare_images
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="CUDA device"):
        ih.letterbox_batch([torch.zeros((4, 4, 3), dtype=torch.uint8)], (8, 8), (0, 0, 0), True, False)
    with pytest.raises(RuntimeError, match="CUDA device"):
        prepare_images(torch.zeros((2, 4, 4, 3), dtype=torch.uint8))
