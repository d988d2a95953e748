"""GPU: the YOLO loss, its (3, 4) parts, the ignore mask and the gradient held to the oracle (oracle/yolo.py, fp64 sums) at
extreme heads, for fp32 / bf16 / fp16 y_pred in every form of the ignore pass.  The reference is always the oracle on the
widened values (y.float()), so a defect that the fp32 and the half paths share cannot hide behind a half-versus-fp32 test.

Regime A (finite extremes): tw / th at the filter's window edges and past exp's range, conf / class logits up to
+-3e38 (+-65504 for fp16), near zero and subnormal, tx / ty at +-30.  Everything finite: loss and parts within 1e-4 of
the oracle, ignore mask bit for bit, the three layouts within 2e-6 of each other, gradients within 1e-4 (plus one ulp of
the gradient type).
Regime B (non-finite inputs in one level): each part finite, +inf or NaN as the oracle's, finite parts as in A.
Fixed-point regressions: the exact pass of the split form sums its object-loss terms in 2^-32 fixed point; terms of
1e9 and more, sums past 2^31 and past 2^32 loss units must still give the oracle's value.

Layouts: aligned (split ignore pass: lean filter + exact pass), offset (single kernel, scalar loads), pinned (single
kernel reading host memory in place; forward only)."""
import functools
import zlib

import numpy as np
import pytest
import torch

from test_gpu_core import _t
from test_gpu_half_loss import HALF_CASES, _half_layout
from test_gpu_yolo_sparse_grad import CASES, _case_id, _inputs, _layout

pytestmark = pytest.mark.gpu
F = np.float32
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
LOSS_RTOL = 1e-4      # the suite's loss tolerance against the oracle
LAYOUT_RTOL = 2e-6    # forms of the ignore pass against each other (test_split_ignore_pass_is_bit_identical)
MANT_BITS = {torch.bfloat16: 7, torch.float16: 10}
MIN_NORMAL = {torch.bfloat16: 2.0 ** -126, torch.float16: 2.0 ** -14}


@functools.lru_cache(maxsize=None)
def _case_inputs(case):
    return _inputs(case)


def _place(heads, layout):
    """Device heads in the layout: "offset" is one element past a 16-byte boundary for every element type."""
    return _layout(heads, layout) if heads[0].dtype == torch.float32 else _half_layout(heads, layout)


def _tmin(case, anc):
    """Per (level, anchor) the lowest tw / th for which the lean filter's area bound holds, computed as the kernel does
    (GetLoss divides the width by image_wh[1])."""
    image_wh = case[0]
    img_w, img_h = float(image_wh[1]), float(image_wh[0])
    a = np.asarray(anc, np.float64)
    tw = np.maximum(np.log(4e-5 * img_w / a[..., 0]), -6.0).astype(F)
    th = np.maximum(np.log(4e-5 * img_h / a[..., 1]), -6.0).astype(F)
    return tw, th


def _records(y_pred, y_true):
    return [h.reshape(y.shape).copy() for h, y in zip(y_pred, y_true)]


def _plant_finite(case, dtype):
    """Regime A on the case's fp32 heads (records of shape (B, H, W, A, 5 + C))."""
    _, C, _, _, _ = case
    _, _, _, y_true, y_pred, anc, _ = _case_inputs(case)
    rng = np.random.default_rng(zlib.crc32(repr(("extremes-A", _case_id(case), dtype)).encode()))
    tmin_w, tmin_h = _tmin(case, anc)
    big = (1e4, 65504.0) if dtype == "fp16" else (1e4, 1e9)
    sub = 3e-7 if dtype == "fp16" else 1e-40
    out = _records(y_pred, y_true)
    for l, x in enumerate(out):
        obj = y_true[l][..., 4] != 0
        u = lambda: rng.random(x.shape[:-1])
        for k, tmin in ((2, tmin_w[l]), (3, tmin_h[l])):
            edge = [tmin, np.nextafter(tmin, F(-np.inf)), F(-6.0), np.nextafter(F(-6.0), F(-np.inf)), F(4.0),
                    np.nextafter(F(4.0), F(np.inf)), F(80.5), F(90.0)]
            for v in edge:
                m = u() < 0.004
                x[..., k][m] = np.broadcast_to(v, x.shape[:-1])[m]   # v: one value per anchor for tmin
        for k in (0, 1):
            x[..., k][u() < 0.004] = 30.0
            x[..., k][u() < 0.004] = -30.0
        for v in (1e4, -1e4, 0.0, 1e-7, -1e-7, sub, -sub):
            x[..., 4][u() < 0.004] = v
            cm = rng.random(x.shape[:-1] + (C,)) < 0.002
            x[..., 5:][cm] = v
        flat = x.reshape(-1, 5 + C)
        objs = np.flatnonzero(obj.reshape(-1))
        n = flat.shape[0]
        # the largest magnitudes in a few records only: two terms of 3e38 already sum past the fp32 range
        for r in rng.choice(n, 2, replace=False):
            flat[r, 4] = big[1] * rng.choice([-1.0, 1.0])
        for r in rng.choice(n, 2, replace=False):
            flat[r, 5 + int(rng.integers(0, C))] = big[1] * rng.choice([-1.0, 1.0])
        if len(objs):
            r = objs[int(rng.integers(0, len(objs)))]
            cls = y_true[l].reshape(-1, 5 + C)[r, 5:]
            flat[r, 4] = -big[1]                       # obj = 1: an object-loss term of big[1]
            flat[r, 5 + int(np.argmin(cls))] = big[1]  # a class whose target is 0: a class term of big[1]
        if dtype != "fp16":
            if l == 0:
                flat[int(rng.integers(0, n)), 4] = 3e38   # one conf term of 3e38 (obj = 0 and ignored: the usual case)
            if l == 2 and len(objs):
                r = objs[-1]
                cls = y_true[l].reshape(-1, 5 + C)[r, 5:]
                flat[r, 5 + int(np.argmin(cls))] = 3e38  # one class term of 3e38 (a class whose target is 0)
        else:
            x[..., 4][u() < 0.002] = 65504.0
            x[..., 4][u() < 0.002] = -65504.0
    return out


NONFINITE = ["tx_nan", "tw_inf", "conf_nan", "conf_inf_obj1", "conf_inf_obj0"]


def _plant_nonfinite(case, kind, level, dtype):
    """Regime B: NaN / inf at a few single positions of one level; the other levels keep the case's finite heads."""
    _, _, _, y_true, y_pred, _, _ = _case_inputs(case)
    rng = np.random.default_rng(zlib.crc32(repr(("extremes-B", _case_id(case), kind, level, dtype)).encode()))
    out = _records(y_pred, y_true)
    x = out[level]
    obj = (y_true[level][..., 4] != 0).reshape(-1)
    flat = x.reshape(-1, x.shape[-1])
    ones, zeros = np.flatnonzero(obj), np.flatnonzero(~obj)
    pick = lambda idx, k: rng.choice(idx, min(k, len(idx)), replace=False) if len(idx) else idx
    nan, inf = float("nan"), float("inf")
    if kind == "tx_nan":
        flat[pick(ones, 2), 0] = nan
        flat[pick(zeros, 3), 0] = nan
    elif kind == "tw_inf":
        flat[pick(ones, 2), 2] = inf
        flat[pick(zeros, 3), 2] = inf
    elif kind == "conf_nan":
        flat[pick(ones, 1), 4] = nan
        flat[pick(zeros, 2), 4] = nan
    elif kind == "conf_inf_obj1":
        r = pick(ones, 2)
        flat[r[:1], 4] = inf
        flat[r[1:], 4] = -inf
    else:
        r = pick(zeros, 2)
        flat[r[:1], 4] = inf
        flat[r[1:], 4] = -inf
    return out


@functools.lru_cache(maxsize=None)
def _planted(case, dtype, thr, regime):
    """The planted heads of the type (host), their widened values, and the oracle's loss, parts and ignore mask on them."""
    from oracle import yolo as oy
    image_wh, _, _, iou_type, _ = case
    _, _, _, y_true, y_pred, anc, _ = _case_inputs(case)
    recs = _plant_finite(case, dtype) if regime is None else _plant_nonfinite(case, *regime, dtype)
    heads = [torch.from_numpy(r.reshape(h.shape)).to(DTYPES[dtype]).contiguous() for r, h in zip(recs, y_pred)]
    wide = [h.float().numpy() for h in heads]
    with np.errstate(all="ignore"):
        loss, parts, ign = oy.get_loss(y_true, wide, image_wh, anc, thr, iou_type, return_ignore=True)
    return heads, wide, loss, parts, ign


@functools.lru_cache(maxsize=None)
def _oracle_grad(case, dtype, thr):
    from oracle import yolo as oy
    image_wh, _, _, iou_type, _ = case
    _, _, _, y_true, _, anc, _ = _case_inputs(case)
    _, wide, _, _, _ = _planted(case, dtype, thr, None)
    with np.errstate(all="ignore"):
        return oy.get_loss_grad(y_true, wide, image_wh, anc, thr, iou_type)[1]


def _forward(entry, heads, case, thr, cuda, ign=None):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxes, _loss_call
    image_wh, C, _, iou_type, _ = case
    boxes, classes, off, y_true, _, anc, tanc = _case_inputs(case)
    if entry == "dense":
        return _loss_call([_t(y, cuda) for y in y_true], heads, image_wh, anc, thr, iou_type, 0, return_parts=True,
                          ignore_out=ign)
    return GetLossFromBoxes(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), heads, image_wh, anc, C, thr, iou_type,
                            target_anchors=tanc, return_parts=True, ignore_out=ign)


def _backward(entry, heads, case, thr, cuda, grad_dtype=torch.float32, grad_scale=None):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetLossFromBoxesAndGrad, _loss_call
    image_wh, C, _, iou_type, _ = case
    boxes, classes, off, y_true, _, anc, tanc = _case_inputs(case)
    if entry == "dense":
        return _loss_call([_t(y, cuda) for y in y_true], heads, image_wh, anc, thr, iou_type, 0, with_grad=True,
                          grad_dtype=grad_dtype, grad_scale=grad_scale)
    return GetLossFromBoxesAndGrad(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), heads, image_wh, anc, C, thr, iou_type,
                                   target_anchors=tanc, return_parts=True, grad_dtype=grad_dtype, grad_scale=grad_scale)


def _np(x):
    return x.detach().reshape(-1).cpu().float().numpy()


def _kind(v):
    v = np.asarray(v, np.float64)
    return np.where(np.isnan(v), 0, np.where(np.isposinf(v), 1, np.where(np.isneginf(v), -1, 2)))


def _assert_close(got, want, rtol, what):
    """Non-finite values equal in kind (NaN, +inf, -inf), finite ones within rtol of each other."""
    got, want = np.asarray(got, np.float64).reshape(-1), np.asarray(want, np.float64).reshape(-1)
    assert np.array_equal(_kind(got), _kind(want)), "%s: non-finite values differ: got %r want %r" % (what, got, want)
    fin = np.isfinite(want)
    err = np.abs(got[fin] - want[fin])
    assert np.all(err <= rtol * np.abs(want[fin])), "%s: got %r want %r" % (what, got, want)


def _assert_grads(got, want, grad_dtype, scale):
    """Against oracle_g * s: non-finite positions equal, finite elements within rtol 1e-4, atol 1e-7 (times s), plus one
    ulp of a half gradient type at the expected value."""
    s = 1.0 if scale is None else float(scale)
    for g, w in zip(got, want):
        assert g.dtype == grad_dtype
        g = g.detach().float().cpu().numpy().reshape(w.shape).astype(np.float64)
        ws = (w * F(s)).astype(F)
        if grad_dtype == torch.float32:
            wr, ulp = ws.astype(np.float64), 0.0
        else:
            wr = torch.from_numpy(ws).to(grad_dtype).float().numpy().astype(np.float64)
            mag = np.maximum(np.abs(ws.astype(np.float64)), MIN_NORMAL[grad_dtype])
            ulp = np.exp2(np.floor(np.log2(mag)) - MANT_BITS[grad_dtype])
        assert np.array_equal(_kind(g), _kind(wr)), "non-finite gradient positions differ"
        fin = np.isfinite(wr)
        err = np.abs(g - ws.astype(np.float64))
        tol = 1e-4 * np.abs(ws.astype(np.float64)) + 1e-7 * s + ulp
        bad = fin & ~(err <= tol)
        assert not bad.any(), "%d gradient elements off, first got %r want %r" % (
            bad.sum(), g[bad][0], ws[bad][0])


# ---- A: finite extremes ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("thr", [0.5, 0.3])
@pytest.mark.parametrize("entry", ["dense", "boxes"])
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("case", HALF_CASES, ids=_case_id)
def test_finite_extremes_forward_match_oracle(lib, cuda, case, dtype, entry, thr):
    heads, _, loss, parts, ign = _planted(case, dtype, thr, None)
    assert np.isfinite(parts).all()     # regime A keeps every part of the oracle's loss finite
    B, n = ign.shape
    got = {}
    for layout in ("aligned", "offset", "pinned"):
        mask = torch.full((B, n), 7, dtype=torch.uint8, device=cuda)
        hl = _place([h.to(cuda) for h in heads], layout)
        gl, gp = _forward(entry, hl, case, thr, cuda, mask)
        assert np.array_equal(mask.cpu().numpy(), ign), layout
        _assert_close(_np(gp), parts, LOSS_RTOL, "parts " + layout)
        _assert_close(_np(gl), [loss], LOSS_RTOL, "loss " + layout)
        got[layout] = np.concatenate([_np(gl), _np(gp)])
    for layout in ("offset", "pinned"):
        _assert_close(got[layout], got["aligned"], LAYOUT_RTOL, "aligned vs " + layout)


@pytest.mark.parametrize("thr", [0.5, 0.3])
@pytest.mark.parametrize("entry", ["dense", "boxes"])
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("case", HALF_CASES, ids=_case_id)
def test_finite_extremes_gradient_matches_oracle(lib, cuda, case, dtype, entry, thr):
    heads, _, loss, parts, _ = _planted(case, dtype, thr, None)
    want = _oracle_grad(case, dtype, thr)
    grad_types = [(torch.float32, None)]
    if dtype != "fp32":
        grad_types += [(DTYPES[dtype], None), (DTYPES[dtype], 1024.0)]
    for layout in ("aligned", "offset"):
        hl = _place([h.to(cuda) for h in heads], layout)
        for gd, s in grad_types:
            st = None if s is None else torch.full((1,), s, dtype=torch.float32, device=cuda)
            gl, gp, grads = _backward(entry, hl, case, thr, cuda, gd, st)
            _assert_close(_np(gp), parts, LOSS_RTOL, "parts " + layout)
            _assert_close(_np(gl), [loss], LOSS_RTOL, "loss " + layout)
            _assert_grads(grads, want, gd, s)


# ---- B: non-finite inputs, one level at a time -------------------------------------------------------------------------
B_CASES = [CASES[2], HALF_CASES[-2]]


@pytest.mark.parametrize("thr", [0.5, 0.3])
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kind", NONFINITE)
@pytest.mark.parametrize("case", B_CASES, ids=_case_id)
def test_nonfinite_inputs_match_oracle(lib, cuda, case, kind, dtype, thr):
    for level in range(3):
        heads, _, loss, parts, ign = _planted(case, dtype, thr, (kind, level))
        assert np.isfinite(np.delete(parts, level, axis=0)).all()
        want = parts.copy()
        if kind in ("tx_nan", "tw_inf") and not (_case_inputs(case)[3][level][..., 4] != 0).any():
            # DESIGN.md section 8: NaN / inf box logits are outside the parity contract.  The oracle's xy / wh term of a
            # non-object record is 0 * NaN = NaN (0 * inf); the kernels sum the xy / wh / class terms over the object
            # records only.  Where the level has object records, some of them carry the planted value and both sides
            # agree (NaN xy, +inf wh); a level without object records keeps a part of 0.
            want[level, 0 if kind == "tx_nan" else 1] = 0.0
        elif kind == "tw_inf":
            want[level, 1] = np.inf   # section 8 as above: +inf from the object records, not the oracle's 0 * inf
        B, n = ign.shape
        got = {}
        for entry in ("dense", "boxes"):
            for layout in ("aligned", "offset", "pinned"):
                mask = torch.full((B, n), 7, dtype=torch.uint8, device=cuda)
                hl = _place([h.to(cuda) for h in heads], layout)
                gl, gp = _forward(entry, hl, case, thr, cuda, mask)
                where = "%s %s level %d" % (entry, layout, level)
                assert np.array_equal(mask.cpu().numpy(), ign), where   # a NaN metric clears the bit (DESIGN.md 6, 8)
                _assert_close(_np(gp), want, LOSS_RTOL, "parts " + where)
                got[(entry, layout)] = np.concatenate([_np(gl), _np(gp)])
        for key, v in got.items():
            _assert_close(v, got[(key[0], "aligned")], LAYOUT_RTOL, "aligned vs %s" % (key,))


# ---- the exact pass's fixed-point object-loss sum ----------------------------------------------------------------------
# conf logits planted on obj = 1 records whose tw = 4.5 (outside the lean filter's window: always queued for the exact
# pass).  Each such record's object-loss term is -logit.
FIXED_CASES = {
    "one_1.5e9": [-1.5e9],
    "three_9e8_past_2^31": [-9e8] * 3,
    "five_9e8_past_2^32": [-9e8] * 5,
    "just_below_2^31": [-170.0 * 2 ** 22] * 3,   # terms below 1e9, sum 2^31 - 2^23 (exact in bf16 too)
    "just_above_2^31": [-171.0 * 2 ** 22] * 3,   # sum 2^31 + 2^22
    "minus_inf": [float("-inf")],
}
FIXED_CASE = CASES[2]   # 96x96, C = 80, B = 4


@functools.lru_cache(maxsize=None)
def _fixed_heads(name, dtype):
    from oracle import yolo as oy
    case = FIXED_CASE
    image_wh, _, _, iou_type, _ = case
    _, _, _, y_true, y_pred, anc, _ = _case_inputs(case)
    recs = _records(y_pred, y_true)
    logits = FIXED_CASES[name]
    counts = [int((y[..., 4] != 0).sum()) for y in y_true]
    level = int(np.argmax(counts))
    assert counts[level] >= len(logits)
    flat = recs[level].reshape(-1, recs[level].shape[-1])
    rows = np.flatnonzero(y_true[level].reshape(-1, flat.shape[-1])[:, 4] != 0)[:len(logits)]
    flat[rows, 2] = 4.5
    flat[rows, 4] = logits
    heads = [torch.from_numpy(r.reshape(h.shape)).to(DTYPES[dtype]).contiguous() for r, h in zip(recs, y_pred)]
    wide = [h.float().numpy() for h in heads]
    with np.errstate(all="ignore"):
        loss, parts = oy.get_loss(y_true, wide, image_wh, anc, 0.5, iou_type, return_parts=True)
        grads = oy.get_loss_grad(y_true, wide, image_wh, anc, 0.5, iou_type)[1]
    return heads, loss, parts, grads


@pytest.mark.parametrize("entry", ["dense", "boxes"])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("name", list(FIXED_CASES))
def test_exact_pass_sum_of_large_terms(lib, cuda, name, dtype, entry):
    case = FIXED_CASE
    heads, loss, parts, grads = _fixed_heads(name, dtype)
    got = []
    for layout in ("aligned", "offset"):
        hl = _place([h.to(cuda) for h in heads], layout)
        gl, gp = _forward(entry, hl, case, 0.5, cuda)
        _assert_close(_np(gp), parts, LOSS_RTOL, "parts " + layout)
        _assert_close(_np(gl), [loss], LOSS_RTOL, "loss " + layout)
        got.append(np.concatenate([_np(gl), _np(gp)]))
        bl, bp, bg = _backward(entry, hl, case, 0.5, cuda)
        _assert_close(_np(bp), parts, LOSS_RTOL, "parts with gradient " + layout)
        _assert_close(_np(bl), [loss], LOSS_RTOL, "loss with gradient " + layout)
        got.append(np.concatenate([_np(bl), _np(bp)]))
        _assert_grads(bg, grads, torch.float32, None)
    for g in got[1:]:
        _assert_close(g, got[0], LAYOUT_RTOL, "layouts / entries")


def test_exact_pass_sum_of_saturated_fp16_conf(lib, cuda):
    """fp16 heads at iou_thresh 0.3 (every record of a level with ground truth goes to the exact pass): conf +65504 on
    every obj = 0 record of level 2 of a 608x608 batch of 2, i.e. over 32 768 terms of 65504 in one level's sum."""
    from oracle import yolo as oy
    case = CASES[1]
    image_wh, _, B, iou_type, _ = case
    _, _, _, y_true, y_pred, anc, _ = _case_inputs(case)
    recs = _records(y_pred, y_true)
    x = recs[2]
    x[..., 4][y_true[2][..., 4] == 0] = 65504.0
    heads = [torch.from_numpy(r.reshape(h.shape)).to(torch.float16).contiguous() for r, h in zip(recs, y_pred)]
    wide = [h.float().numpy() for h in heads]
    loss, parts = oy.get_loss(y_true, wide, image_wh, anc, 0.3, iou_type, return_parts=True)
    assert float(parts[2, 2]) * B > 2.0 ** 31
    got = []
    for layout in ("aligned", "offset"):
        for entry in ("dense", "boxes"):
            gl, gp = _forward(entry, _place([h.to(cuda) for h in heads], layout), case, 0.3, cuda)
            _assert_close(_np(gp), parts, LOSS_RTOL, "parts %s %s" % (layout, entry))
            _assert_close(_np(gl), [loss], LOSS_RTOL, "loss %s %s" % (layout, entry))
            got.append(np.concatenate([_np(gl), _np(gp)]))
    for g in got[1:]:
        _assert_close(g, got[0], LAYOUT_RTOL, "layouts / entries")
