"""CPU: argument checks of the typed post-processing entries that read bf16 / fp16 heads in place
(b200_yolo_decode_nms_typed, b200_effdet_decode_typed, b200_effdet_postprocess_typed,
b200_effdet_decode_postprocess_typed).  Every refusal below is decided before the first CUDA call, so none needs a
device; messages name the offending level."""
import ctypes

import pytest

FAKE = 1 << 20   # 256-byte aligned and never dereferenced
F32, BF16, F16 = 0, 1, 2
D0 = (64, 64, 32, 32, 16, 16, 8, 8, 4, 4)
L = 5
P = ctypes.c_void_p * L
f = ctypes.c_float


def _err(lib):
    return lib.b200_last_error().decode()


def _yolo(lib, heads=None, dtype=BF16, B=2, C=80):
    hw = (ctypes.c_int32 * 6)(13, 13, 26, 26, 52, 52)
    anc = (ctypes.c_float * 18)(*[10.0] * 18)
    img = (ctypes.c_float * 2)(416.0, 416.0)
    hp = (ctypes.c_void_p * 3)(*(heads if heads is not None else (FAKE, FAKE, FAKE)))
    return lib.b200_yolo_decode_nms_typed(hp, dtype, hw, B, 3, C, ctypes.addressof(anc), ctypes.addressof(img), f(0.5), f(0.3),
                                          f(0.5), 0, 500, FAKE, FAKE, FAKE, FAKE, FAKE, None, None, FAKE, FAKE, 1 << 40, None)


def _decode(lib, rel=None, dtype=F16):
    hw = (ctypes.c_int32 * len(D0))(*D0)
    return lib.b200_effdet_decode_typed(L, hw, 9, FAKE, 2, rel if rel is not None else P(*[FAKE] * L), dtype, P(*[FAKE] * L), None)


def _post(lib, boxes=None, box_dtype=F32, classes=None, cls_dtype=BF16):
    hw = (ctypes.c_int32 * len(D0))(*D0)
    return lib.b200_effdet_postprocess_typed(L, hw, 9, 90, 4, 1, 2, boxes if boxes is not None else P(*[FAKE] * L), box_dtype,
                                             classes if classes is not None else P(*[FAKE] * L), cls_dtype, 200, f(0.5),
                                             f(1e-4), 5, FAKE, FAKE, FAKE, None, None, FAKE, FAKE, 1 << 40, None)


def _decode_post(lib, rel=None, rel_dtype=BF16, classes=None, cls_dtype=BF16):
    hw = (ctypes.c_int32 * len(D0))(*D0)
    return lib.b200_effdet_decode_postprocess_typed(L, hw, 9, FAKE, 90, 2, rel if rel is not None else P(*[FAKE] * L), rel_dtype,
                                                    classes if classes is not None else P(*[FAKE] * L), cls_dtype,
                                                    P(*[FAKE] * L), 200, f(0.5), f(1e-4), 5, FAKE, FAKE, FAKE, None, None,
                                                    FAKE, FAKE, 1 << 40, None)


@pytest.mark.parametrize("code", [-1, 3, 7])
def test_dtype_codes_outside_the_enum_are_refused(lib, code):
    assert _yolo(lib, dtype=code) == -1 and "head_dtype %d" % code in _err(lib)
    assert _decode(lib, dtype=code) == -1 and "rel_dtype %d" % code in _err(lib)
    assert _post(lib, box_dtype=code) == -1 and "dtype codes" in _err(lib)
    assert _post(lib, cls_dtype=code) == -1 and "dtype codes" in _err(lib)
    assert _decode_post(lib, rel_dtype=code) == -1 and "dtype codes" in _err(lib)
    assert _decode_post(lib, cls_dtype=code) == -1 and "dtype codes" in _err(lib)


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
def test_yolo_heads_null_or_unaligned(lib, dtype):
    assert _yolo(lib, heads=(FAKE, 0, FAKE), dtype=dtype) == -1 and "bad level 1" in _err(lib)
    assert _yolo(lib, heads=(FAKE, FAKE, FAKE + 2), dtype=dtype) == -1 and "head 2 not 16-byte aligned" in _err(lib)
    assert _yolo(lib, heads=(FAKE + 8, FAKE, FAKE), dtype=dtype) == -1 and "head 0 not 16-byte aligned" in _err(lib)
    hp = None
    hw = (ctypes.c_int32 * 6)(13, 13, 26, 26, 52, 52)
    assert lib.b200_yolo_decode_nms_typed(hp, dtype, hw, 2, 3, 80, FAKE, FAKE, f(0.5), f(0.3), f(0.5), 0, 500, FAKE, FAKE, FAKE,
                                          FAKE, FAKE, None, None, FAKE, FAKE, 1 << 40, None) == -1
    assert "null argument" in _err(lib)


def test_yolo_typed_keeps_the_shape_checks(lib):
    assert _yolo(lib, C=0) == -1 and "unsupported shape" in _err(lib)
    assert _yolo(lib, C=1020) == -1 and "unsupported shape" in _err(lib)


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
def test_effdet_decode_levels(lib, dtype):
    assert _decode(lib, rel=P(FAKE, FAKE, FAKE, 0, FAKE), dtype=dtype) == -1 and "null level 3" in _err(lib)
    assert _decode(lib, rel=P(FAKE, FAKE + 8, FAKE, FAKE, FAKE), dtype=dtype) == -1
    assert "level 1 not 16-byte aligned" in _err(lib)


@pytest.mark.parametrize("dtype", [F32, BF16, F16])
def test_effdet_postprocess_levels(lib, dtype):
    assert _post(lib, boxes=P(FAKE, FAKE, FAKE, FAKE, 0), box_dtype=dtype) == -1 and "null level 4" in _err(lib)
    assert _post(lib, classes=P(FAKE, FAKE, 0, FAKE, FAKE), cls_dtype=dtype) == -1 and "null level 2" in _err(lib)
    assert _post(lib, boxes=P(FAKE, FAKE, FAKE + 8, FAKE, FAKE), box_dtype=dtype) == -1
    assert "boxes level 2 not 16-byte aligned" in _err(lib)
    assert _decode_post(lib, rel=P(FAKE, 0, FAKE, FAKE, FAKE), rel_dtype=dtype) == -1 and "null level 1" in _err(lib)
    assert _decode_post(lib, classes=P(0, FAKE, FAKE, FAKE, FAKE), cls_dtype=dtype) == -1 and "null level 0" in _err(lib)
    assert _decode_post(lib, rel=P(FAKE, FAKE, FAKE, FAKE, FAKE + 4), rel_dtype=dtype) == -1
    assert "boxes level 4 not 16-byte aligned" in _err(lib)
