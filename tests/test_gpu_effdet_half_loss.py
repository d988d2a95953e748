"""GPU: the EfficientDet loss and its gradient from bf16 / fp16 heads read in place.  Every half call is held to the fp32
call on the widened heads (y.float()): loss, parts, num_positives and the fp64 sums bit-identical, and gradients equal to
(g32 * s).to(grad_dtype) bit for bit (NaN positions equal, payloads not compared), where g32 is the fp32 gradient and s
the gradient scale.  Two cases are also held to the oracle, so that a defect shared by both paths cannot pass.

Shapes: the cases of test_gpu_effdet_sparse_grad plus dense cases at C = 4, 5 and 7.  At B = 3, C = 81 the "small"
configuration (3069 anchors per image) has a last level of 9 anchors per image, 3 * 9 * 81 = 3 (mod 4) logits, so CTA 0
runs the scalar tail; C = 4, 5 and 7 make 4-element groups straddle two anchors."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from test_gpu_core import _t, assert_bits_equal
from test_gpu_effdet import _pair
from test_gpu_effdet_sparse_grad import CASES, _case_id, _inputs, _oracle_targets

pytestmark = pytest.mark.gpu
HALF = {"bf16": torch.bfloat16, "fp16": torch.float16}
OTHER = {torch.bfloat16: torch.float16, torch.float16: torch.bfloat16}
SCALES = (None, 1024.0, 2.0 ** -4)
BIG = {torch.bfloat16: 3e38, torch.float16: 65504.0}
TINY = {torch.bfloat16: 1e-40, torch.float16: 6e-8}   # subnormals of each type
DENSE = [("small", 3, 81), ("small", 2, 4), ("rect", 2, 5), ("small", 3, 7)]


def _bits(x):
    return x.detach().reshape(-1).cpu().float().numpy()


def _expect_grads(got, g32, grad_dtype, scale):
    for a, b in zip(got, g32):
        assert a.dtype == grad_dtype and a.shape == b.shape
        want = (b if scale is None else b * scale).to(grad_dtype)
        assert_bits_equal(_bits(a), _bits(want))


@functools.lru_cache(maxsize=None)
def _case(name, B, C, many=False, seed=0):
    a, _ = _pair(name)
    return _inputs(a, name, B, C, many, 7600 + 13 * B + C + seed)


def _plant(a, boxes, classes, off, pb, pc, C, thr, dtype, dev, seed):
    """The fp32 heads with planted values, cast to the half type.  Logits: +-inf, NaN, the largest finite values of the
    type, subnormals and +-0 at random anchors (matched and unmatched).  Box outputs: equal to the (rounded) box target of
    a matched anchor, at target +- delta, and NaN."""
    g = torch.Generator(device=dev).manual_seed(seed)
    tb, _, tm = a.generate_targets_batch(_t(boxes, dev), _t(classes, dev), _t(off, dev), C, iou_threshold=thr)
    hb, hc = [], []
    for l in range(len(pb)):
        x = _t(pc[l], dev).clone()
        u = lambda: torch.rand(x.shape, device=dev, generator=g)
        for val in (float("inf"), float("-inf"), float("nan"), BIG[dtype], -BIG[dtype], TINY[dtype], -TINY[dtype], 0.0, -0.0):
            x[u() < 0.002] = val
        o = _t(pb[l], dev).clone()
        t, m = tb[l], tm[l].reshape(o.shape[:-1])
        r = torch.rand(o.shape[:-1], device=dev, generator=g)
        o[m & (r < 0.3)] = t[m & (r < 0.3)]
        o[m & (r >= 0.3) & (r < 0.5)] = t[m & (r >= 0.3) & (r < 0.5)] + 0.1
        o[m & (r >= 0.5) & (r < 0.7)] = t[m & (r >= 0.5) & (r < 0.7)] - 0.1
        o[torch.rand(o.shape, device=dev, generator=g) < 0.002] = float("nan")
        hb.append(o.to(dtype).contiguous())
        hc.append(x.to(dtype).contiguous())
    return hb, hc


def _planted(case, dtype, dev):
    name, B, C, thr, many = case
    a, _ = _pair(name)
    boxes, classes, off, pb, pc = _case(name, B, C, many)
    hb, hc = _plant(a, boxes, classes, off, pb, pc, C, thr, dtype, dev, 31 * B + C)
    return a, boxes, classes, off, hb, hc


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_from_boxes_bit_identical(lib, cuda, case, dtype):
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes, get_loss_from_boxes_and_grad
    thr = case[3]
    a, boxes, classes, off, hb, hc = _planted(case, HALF[dtype], cuda)
    wb, wc = [h.float() for h in hb], [h.float() for h in hc]
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    l32, pb32, pc32 = get_loss_from_boxes_and_grad(a, db, dc, do, wb, wc, iou_threshold=thr)
    f32, p32, n32 = get_loss_from_boxes(a, db, dc, do, wb, wc, iou_threshold=thr, return_parts=True)
    fh, ph, nh = get_loss_from_boxes(a, db, dc, do, hb, hc, iou_threshold=thr, return_parts=True)
    for x, y in ((fh, f32), (ph, p32), (nh, n32)):
        assert_bits_equal(_bits(x), _bits(y))
    assert not np.isfinite(float(f32))   # the planted infinities and NaNs reach the loss
    for gd in (torch.float32, HALF[dtype], OTHER[HALF[dtype]]):
        for s in SCALES:
            st = None if s is None else torch.full((1,), s, dtype=torch.float32, device=cuda)
            lh, gb, gc = get_loss_from_boxes_and_grad(a, db, dc, do, hb, hc, iou_threshold=thr, grad_dtype=gd, grad_scale=st)
            assert_bits_equal(_bits(lh), _bits(l32))
            _expect_grads(gb, pb32, gd, s)
            _expect_grads(gc, pc32, gd, s)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("dense", DENSE, ids=lambda d: "%s-B%d-C%d" % d)
def test_dense_targets_bit_identical(lib, cuda, dense, dtype):
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss, get_loss_and_grad
    name, B, C = dense
    a, boxes, classes, off, hb, hc = _planted((name, B, C, 0.5, False), HALF[dtype], cuda)
    wb, wc = [h.float() for h in hb], [h.float() for h in hc]
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    for index in (False, True):
        tb, tc, tm = a.generate_targets_batch(db, dc, do, C, class_index=index)
        f32, p32, n32 = get_loss(tb, tc, tm, wb, wc, return_parts=True)
        fh, ph, nh = get_loss(tb, tc, tm, hb, hc, return_parts=True)
        for x, y in ((fh, f32), (ph, p32), (nh, n32)):
            assert_bits_equal(_bits(x), _bits(y))
        l32, gb32, gc32 = get_loss_and_grad(tb, tc, tm, wb, wc)
        for gd in (torch.float32, HALF[dtype], OTHER[HALF[dtype]]):
            for s in SCALES:
                lh, gb, gc = get_loss_and_grad(tb, tc, tm, hb, hc, grad_dtype=gd, grad_scale=s)   # a Python float here
                assert_bits_equal(_bits(lh), _bits(l32))
                _expect_grads(gb, gb32, gd, s)
                _expect_grads(gc, gc32, gd, s)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_narrow_heads_take_the_dense_typed_entries(lib, cuda, dtype):
    """classes_num < 4: generate_targets_batch + get_loss, still on the half heads in place."""
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes, get_loss_from_boxes_and_grad
    a, _ = _pair("tiny")
    boxes = np.array([[3, 3, 6, 6], [5, 5, 9, 9], [2, 2, 5, 5]], np.float32)
    classes, off = np.array([1, 2, 1], np.int32), np.array([0, 2, 3], np.int32)
    g = torch.Generator(device=cuda).manual_seed(12)
    hb = [(torch.randn((2, 10, 10, 3, 4), device=cuda, generator=g) * 0.25).to(HALF[dtype])]
    hc = [torch.randn((2, 10, 10, 3, 3), device=cuda, generator=g).to(HALF[dtype])]
    wb, wc = [h.float() for h in hb], [h.float() for h in hc]
    l32, gb32, gc32 = get_loss_from_boxes_and_grad(a, boxes, classes, off, wb, wc)
    lh, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, hb, hc, grad_dtype=HALF[dtype], grad_scale=1024.0)
    assert_bits_equal(_bits(lh), _bits(l32))
    _expect_grads(gb, gb32, HALF[dtype], 1024.0)
    _expect_grads(gc, gc32, HALF[dtype], 1024.0)
    f32, p32, n32 = get_loss_from_boxes(a, boxes, classes, off, wb, wc, return_parts=True)
    fh, ph, nh = get_loss_from_boxes(a, boxes, classes, off, hb, hc, return_parts=True)
    assert_bits_equal(_bits(fh), _bits(f32))
    assert_bits_equal(_bits(ph), _bits(p32))


def test_fp16_gradient_overflows_to_inf(lib, cuda):
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes_and_grad
    case = CASES[0]
    a, boxes, classes, off, hb, hc = _planted(case, torch.float16, cuda)
    wb, wc = [h.float() for h in hb], [h.float() for h in hc]
    _, gb32, gc32 = get_loss_from_boxes_and_grad(a, boxes, classes, off, wb, wc)
    s = 2.0 ** 40
    _, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, hb, hc, grad_dtype=torch.float16, grad_scale=s)
    _expect_grads(gb, gb32, torch.float16, s)
    _expect_grads(gc, gc32, torch.float16, s)
    assert any(bool(torch.isinf(x).any()) for x in gc) and any(bool(torch.isinf(x).any()) for x in gb)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_focal_and_box_loss_helpers(lib, cuda, dtype):
    from tfmv_b200.ai_models.losses.box_loss import BoxLoss
    from tfmv_b200.ai_models.losses.focal_loss import FocalLoss
    name, B, C = "small", 3, 81
    a, boxes, classes, off, hb, hc = _planted((name, B, C, 0.5, False), HALF[dtype], cuda)
    tb, tc, _ = a.generate_targets_batch(_t(boxes, cuda), _t(classes, cuda), _t(off, cuda), C)
    fl = FocalLoss(label_smoothing=0.1)
    for l in (0, 2):
        x = torch.nan_to_num(hc[l].float()).clamp(-30, 30).to(HALF[dtype])   # a finite loss, so the bits say something
        assert_bits_equal(_bits(fl((7.0, tc[l]), x)), _bits(fl((7.0, tc[l]), x.float())))
        bl = BoxLoss(delta=0.1)
        assert_bits_equal(_bits(bl((5.0, tb[l]), hb[l])), _bits(bl((5.0, tb[l]), hb[l].float())))


def test_mixed_families_take_the_cast_path(lib, cuda):
    """bf16 boxes with fp32 logits, bf16 boxes with fp16 logits, and one fp32 box level among bf16 ones: cast to fp32,
    so the results are those of the fp32 call on the widened heads."""
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_and_grad, get_loss_from_boxes_and_grad
    case = CASES[0]
    a, boxes, classes, off, hb, hc = _planted(case, torch.bfloat16, cuda)
    tb, tc, tm = a.generate_targets_batch(_t(boxes, cuda), _t(classes, cuda), _t(off, cuda), case[2])
    wide = lambda xs: [x.float() for x in xs]
    f16 = [h.float().to(torch.float16) for h in hc]
    for mb, mc in ((hb, wide(hc)), (hb, f16), (hb[:1] + wide(hb[1:]), hc)):
        l32, gb32, gc32 = get_loss_from_boxes_and_grad(a, boxes, classes, off, wide(mb), wide(mc))
        lm, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, mb, mc)
        assert_bits_equal(_bits(lm), _bits(l32))
        _expect_grads(gb, gb32, torch.float32, None)
        _expect_grads(gc, gc32, torch.float32, None)
        l32, gb32, gc32 = get_loss_and_grad(tb, tc, tm, wide(mb), wide(mc))
        lm, gb, gc = get_loss_and_grad(tb, tc, tm, mb, mc)
        assert_bits_equal(_bits(lm), _bits(l32))
        _expect_grads(gb, gb32, torch.float32, None)
        _expect_grads(gc, gc32, torch.float32, None)


def test_sharded_stages_concatenate_to_the_full_batch(lib, cuda):
    """Two halves of a bf16 batch through the two ABI stages (the all-reduces played by torch adds): the bf16 gradients
    concatenate to the whole-batch call's bit for bit, and the finalized loss equals it to fp64 summation order."""
    from tfmv_b200 import _tensors as T
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes_and_grad
    a, _ = _pair("small")
    B, C, L = 4, 81, a._num_levels
    boxes, classes, off, pb, pc = _case("small", B, C, False, 1)
    hb, hc = [_t(x, cuda).to(torch.bfloat16) for x in pb], [_t(x, cuda).to(torch.bfloat16) for x in pc]
    scale = torch.full((1,), 1024.0, dtype=torch.float32, device=cuda)
    loss, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, hb, hc, grad_dtype=torch.bfloat16, grad_scale=scale)
    numel = [float(t.numel()) for t in hc]
    arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])
    f = ctypes.c_float
    shards = []
    for lo, hi in ((0, 2), (2, B)):
        s = dict(boxes=_t(boxes[off[lo]:off[hi]], cuda), classes=_t(classes[off[lo]:off[hi]], cuda),
                 off=_t((off[lo:hi + 1] - off[lo]).astype(np.int32), cuda), pb=[t[lo:hi].clone() for t in hb],
                 pc=[t[lo:hi].clone() for t in hc], sums=torch.full((2 * L + 1,), 7.0, dtype=torch.float64, device=cuda))
        s["gb"], s["gc"] = [torch.empty_like(t) for t in s["pb"]], [torch.empty_like(t) for t in s["pc"]]
        s["ws"] = torch.empty((lib.b200_effdet_loss_from_boxes_workspace_bytes(L, a._hw, a._A, hi - lo),), dtype=torch.uint8,
                              device=cuda)
        shards.append(s)
    for s in shards:
        assert lib.b200_effdet_loss_from_boxes_match(L, a._hw, a._A, a._dev_table().data_ptr(), s["off"].numel() - 1,
                                                     s["boxes"].data_ptr(), s["off"].data_ptr(), s["boxes"].shape[0], f(0.5),
                                                     s["sums"].data_ptr(), s["ws"].data_ptr(), s["ws"].numel(), T.stream_ptr()) == 0
    npos = shards[0]["sums"][2 * L:] + shards[1]["sums"][2 * L:]
    for s in shards:
        s["sums"][2 * L:] = npos
        assert lib.b200_effdet_loss_from_boxes_grad_typed(
            L, a._hw, a._A, a._dev_table().data_ptr(), C, s["off"].numel() - 1, s["boxes"].data_ptr(), s["classes"].data_ptr(),
            s["boxes"].shape[0], arr(s["pb"]), arr(s["pc"]), 1, f(0.25), f(1.5), f(0.1), f(0.0), (ctypes.c_double * L)(*numel),
            s["sums"].data_ptr(), arr(s["gb"]), arr(s["gc"]), 1, scale.data_ptr(), s["ws"].data_ptr(), s["ws"].numel(),
            T.stream_ptr()) == 0
    sums = shards[0]["sums"] + shards[1]["sums"]
    sums[2 * L:] = npos
    for l in range(L):
        assert_bits_equal(_bits(torch.cat([shards[0]["gb"][l], shards[1]["gb"][l]])), _bits(gb[l]))
        assert_bits_equal(_bits(torch.cat([shards[0]["gc"][l], shards[1]["gc"][l]])), _bits(gc[l]))
    out = torch.empty((), dtype=torch.float32, device=cuda)
    assert lib.b200_focal_box_finalize(L, sums.data_ptr(), (ctypes.c_double * L)(*numel), None, out.data_ptr(), None, T.stream_ptr()) == 0
    assert abs(float(out) - float(loss)) <= 1e-6 * abs(float(loss))


def test_graph_replay_after_rewriting_heads_and_scale(lib, cuda):
    from tfmv_b200 import runtime
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes_and_grad
    a, _ = _pair("small")
    boxes, classes, off, pb, pc = _case("small", 3, 81, False, 2)
    hb, hc = [_t(x, cuda).to(torch.bfloat16) for x in pb], [_t(x, cuda).to(torch.bfloat16) for x in pc]
    scale = torch.full((1,), 1024.0, dtype=torch.float32, device=cuda)
    bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    step = runtime.capture(lambda: get_loss_from_boxes_and_grad(a, bd, cd, od, hb, hc, grad_dtype=torch.bfloat16, grad_scale=scale))
    for h in hb + hc:
        h.copy_((torch.randn(h.shape, device=cuda) * 2.0).to(torch.bfloat16))
    scale.fill_(0.125)
    r_loss, r_gb, r_gc = step()
    e_loss, e_gb, e_gc = get_loss_from_boxes_and_grad(a, bd, cd, od, [h.float() for h in hb], [h.float() for h in hc])
    assert_bits_equal(_bits(r_loss), _bits(e_loss))
    _expect_grads(r_gb, e_gb, torch.bfloat16, 0.125)
    _expect_grads(r_gc, e_gc, torch.bfloat16, 0.125)


@pytest.mark.parametrize("call", ["forward", "backward"])
def test_half_call_makes_no_fp32_copy(lib, cuda, call):
    """D0 512 x 512, B = 8, C = 81: the call's peak allocation stays below an fp32 copy of the logits."""
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes, get_loss_from_boxes_and_grad
    a, _ = _pair("d0")
    boxes, classes, off, pb, pc = _case("d0", 2, 81)
    hb = [_t(x, cuda).to(torch.bfloat16).repeat(4, 1, 1, 1, 1) for x in pb]
    hc = [_t(x, cuda).to(torch.bfloat16).repeat(4, 1, 1, 1, 1) for x in pc]
    n = len(boxes)
    boxes, classes = np.tile(boxes, (4, 1)), np.tile(classes, 4)
    off = np.concatenate([[0], np.cumsum(np.tile(np.diff(off), 4))]).astype(np.int32)
    args = (a, _t(boxes, cuda), _t(classes, cuda), _t(off, cuda), hb, hc)
    assert off[-1] == 4 * n
    if call == "forward":
        run = lambda: get_loss_from_boxes(*args)
    else:
        run = lambda: get_loss_from_boxes_and_grad(*args, grad_dtype=torch.bfloat16)
    run()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    run()
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < sum(h.numel() for h in hc) * 4


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_half_heads_against_the_oracle(lib, cuda, dtype):
    """The loss and its parts from half heads within 1e-4 of the fp64-summing oracle on the widened heads, with large
    finite logits (+-60) and logits near 0 planted."""
    from oracle import effdet as oe
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes, get_loss_from_boxes_and_grad
    name, B, C, thr = ("small", 3, 81, 0.5) if dtype == "bf16" else ("rect", 2, 7, 0.5)
    a, o = _pair(name)
    boxes, classes, off, pb, pc = _case(name, B, C, False, 3)
    pc = [x.copy() for x in pc]
    rng = np.random.default_rng(91)
    for x in pc:
        x[rng.random(x.shape) < 0.003] = 60.0
        x[rng.random(x.shape) < 0.003] = -60.0
        x[rng.random(x.shape) < 0.003] = 1e-3
    hb, hc = [_t(x, cuda).to(HALF[dtype]) for x in pb], [_t(x, cuda).to(HALF[dtype]) for x in pc]
    loss, parts, npos = get_loss_from_boxes(a, boxes, classes, off, hb, hc, iou_threshold=thr, return_parts=True)
    lg, _, _ = get_loss_from_boxes_and_grad(a, boxes, classes, off, hb, hc, iou_threshold=thr, grad_dtype=HALF[dtype])
    assert_bits_equal(_bits(lg), _bits(loss))
    otb, otc, otm = _oracle_targets(o, boxes, classes, off, C, thr)
    want, o_parts, o_npos = oe.get_loss(otb, otc, otm, [h.float().cpu().numpy() for h in hb], [h.float().cpu().numpy() for h in hc],
                                        return_parts=True)
    assert float(npos) == float(o_npos)
    np.testing.assert_allclose(parts.cpu().numpy(), o_parts, rtol=1e-4, atol=1e-9)
    assert abs(float(loss) - float(want)) <= 1e-4 * abs(float(want))
