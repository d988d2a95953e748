"""GPU: post-processing from bf16 / fp16 heads read in place.  Every output of a half-precision call must be
bit-identical to the fp32 call on the widened heads (heads.float()): widening is exact and every decision is taken in
fp32, so nothing may differ.  NaN positions must match (payloads are not compared); integer outputs and counts are equal."""
import numpy as np
import pytest
import torch

from test_gpu_core import assert_bits_equal

pytestmark = pytest.mark.gpu
F = np.float32
HALF = {"bf16": torch.bfloat16, "fp16": torch.float16}


def _anchors(A):
    from tfmv_b200 import synth
    base = synth.yolo_anchors().astype(F)               # (3, 3, 2)
    reps = (A + 2) // 3
    return np.concatenate([base] * reps, axis=1)[:, :A] * F(1.0 + 0.1 * np.arange(A)[None, :, None])


def _crafted_heads(seed, B, grids, A, C, dtype, dev):
    """Random heads in the given half type, with the inputs the decision paths care about planted in a few per cent
    of the records: exact ties of the class maximum, runner-ups inside the 0.01 guard band, conf logits at the edges of
    the logit-space window around logit(0.5) = 0, tw / th outside the safe range and +-inf, NaN, fp16 subnormals."""
    g = torch.Generator(device=dev).manual_seed(seed)
    heads = []
    for (h, w) in grids:
        x = torch.randn((B, h, w, A, 5 + C), device=dev, generator=g) * 2.0
        u = lambda: torch.rand((B, h, w, A), device=dev, generator=g)
        cls = x[..., 5:]
        m = u() < 0.03     # every class logit equal: the first index must win
        cls[m] = cls[m][:, :1].expand(-1, C).clone()
        m = u() < 0.05     # runner-up just inside the guard band, and an exact tie with a later class
        if C > 1:
            top = cls[m].max(dim=-1).values
            cls[m] = torch.stack([top - 0.005] + [cls[m][:, k] for k in range(1, C)], dim=-1)
            cls[..., C - 1][m] = top
        conf = x[..., 4]
        for val in (0.0, 1e-7, -1e-7, 3e-6, -3e-6, 6e-8, -6e-8, 1e-30):
            conf[u() < 0.01] = val
        for k in (2, 3):
            for val in (-40.0, -16.0, 80.5, 90.0, float("inf"), float("-inf")):
                x[..., k][u() < 0.005] = val
        for k in (0, 1, 4):
            x[..., k][u() < 0.003] = float("nan")
        cls[u() < 0.01] = float("nan")
        x[..., 0][u() < 0.01] = 3e-8           # fp16 subnormal (bf16 keeps it normal)
        cls[..., 0][u() < 0.01] = 2e-7
        heads.append(x.reshape(B, h, w, A * (5 + C)).to(dtype).contiguous())
    return heads


def _assert_same_rows(a, b):
    assert torch.equal(a["count"], b["count"])
    cnt = a["count"].cpu().tolist()
    for k in a:
        if k == "count":
            continue
        for i, n in enumerate(cnt):
            x, y = a[k][i, :n].cpu(), b[k][i, :n].cpu()
            if x.dtype == torch.float32:
                assert_bits_equal(x.numpy(), y.numpy())
            else:
                assert torch.equal(x, y), k


def _yolo_pair(heads, anc, image_wh, C, iou_type, conf=0.5, score=0.3):
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxesBatch
    args = (anc, image_wh, C, conf, score, 0.5, iou_type)
    half = GetNMSBoxesBatch(*heads, *args, with_indices=True)
    full = GetNMSBoxesBatch(*[h.float() for h in heads], *args, with_indices=True)
    _assert_same_rows(half, full)
    return half


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("image,B,iou_type", [(416, 1, "iou"), (608, 3, "diou"), (416, 160, "ciou")])
def test_yolo_half_heads_bit_identical(lib, cuda, dtype, image, B, iou_type):
    from tfmv_b200 import synth
    grids = [(s, s) for s in synth.yolo_grids(image)]
    heads = _crafted_heads(7 + B, B, grids, 3, 80, HALF[dtype], cuda)
    r = _yolo_pair(heads, synth.yolo_anchors().astype(F), (image, image), 80, iou_type)
    assert int(r["count"].min()) > 0


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("A,C", [(1, 1), (2, 20), (4, 300), (1, 300), (4, 1), (2, 80)])
def test_yolo_half_heads_shapes(lib, cuda, dtype, A, C):
    # rectangular grids with 35, 140 and 560 cells per image: the tensors end in ragged tiles (plain-copy fallback)
    grids = [(5, 7), (10, 14), (20, 28)]
    heads = _crafted_heads(100 + A * 1000 + C, 3, grids, A, C, HALF[dtype], cuda)
    _yolo_pair(heads, _anchors(A), (224, 160), C, "diou", conf=0.4, score=0.2)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_yolo_half_heads_low_thresholds(lib, cuda, dtype):
    # thresholds near 0 take the exact sigmoid comparison for every record, and nearly every record is a candidate
    from tfmv_b200 import synth
    heads = _crafted_heads(5, 2, [(13, 13), (26, 26), (52, 52)], 3, 80, HALF[dtype], cuda)
    _yolo_pair(heads, synth.yolo_anchors().astype(F), (416, 416), 80, "iou", conf=1e-4, score=1e-4)


def test_yolo_mixed_family_falls_back_to_fp32(lib, cuda):
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxesBatch
    grids = [(13, 13), (26, 26), (52, 52)]
    hb = _crafted_heads(11, 2, grids, 3, 80, torch.bfloat16, cuda)
    hf = _crafted_heads(12, 2, grids, 3, 80, torch.float16, cuda)
    mixed = [hb[0], hf[1], hb[2].float()]
    args = (synth.yolo_anchors().astype(F), (416, 416), 80, 0.5, 0.3, 0.5, "iou")
    _assert_same_rows(GetNMSBoxesBatch(*mixed, *args, with_indices=True),
                      GetNMSBoxesBatch(*[h.float() for h in mixed], *args, with_indices=True))


def test_yolo_half_heads_graph_capture(lib, cuda):
    from tfmv_b200 import runtime, synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxesBatch
    grids = [(13, 13), (26, 26), (52, 52)]
    heads = _crafted_heads(21, 4, grids, 3, 80, torch.bfloat16, cuda)
    args = (synth.yolo_anchors().astype(F), (416, 416), 80, 0.5, 0.3, 0.5, "diou")
    step = runtime.capture(lambda: GetNMSBoxesBatch(*heads, *args, with_indices=True))
    for h, n in zip(heads, _crafted_heads(22, 4, grids, 3, 80, torch.bfloat16, cuda)):
        h.copy_(n)
    got = {k: v.clone() for k, v in step().items()}
    _assert_same_rows(got, GetNMSBoxesBatch(*heads, *args, with_indices=True))
    _assert_same_rows(got, GetNMSBoxesBatch(*[h.float() for h in heads], *args, with_indices=True))


def test_yolo_half_call_makes_no_fp32_copy(lib, cuda):
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxesBatch
    heads = _crafted_heads(31, 32, [(13, 13), (26, 26), (52, 52)], 3, 80, torch.float16, cuda)
    args = (synth.yolo_anchors().astype(F), (416, 416), 80, 0.5, 0.3, 0.5, "iou")
    GetNMSBoxesBatch(*heads, *args)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    GetNMSBoxesBatch(*heads, *args)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < sum(h.numel() for h in heads) * 4


# ---- EfficientDet ------------------------------------------------------------------------------------------------------
def _effdet(name):
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.efficientnet.utils.anchors import Anchors
    c = synth.EFFDET_CONFIGS[name]
    return Anchors(c["min_level"], c["max_level"], c["image_size"], c["num_scales"], c["aspect_ratios"], c["anchor_scale"])


def _effdet_heads(a, seed, B, C, dtype, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    rel, cls = [], []
    for s in (tuple(b.shape) for b in a.boxes):
        r = torch.randn((B,) + s, device=dev, generator=g) * 0.25
        r.view(-1)[torch.rand(r.numel(), device=dev, generator=g) < 1e-3] = 100.0   # exp overflow -> inf boxes
        c = torch.randn((B,) + s[:-1] + (C,), device=dev, generator=g) * 2.0
        m = torch.rand(c.shape[:-1], device=dev, generator=g) < 0.02                  # all-equal rows: argmax 0, dropped
        c[m] = c[m][:, :1].expand(-1, C).clone()
        c.view(-1)[torch.rand(c.numel(), device=dev, generator=g) < 1e-4] = float("nan")
        rel.append(r.to(dtype))
        cls.append(c.to(dtype))
    return rel, cls


def _assert_same_dense(xs, ys):
    for x, y in zip(xs, ys):
        assert x.dtype == torch.float32 and y.dtype == torch.float32
        assert_bits_equal(x.cpu().numpy(), y.cpu().numpy())


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("name,B,iou_type", [("d0", 2, "diou"), ("d0", 5, "iou"), ("d7", 1, "diou")])
def test_effdet_half_heads_bit_identical(lib, cuda, dtype, name, B, iou_type):
    a = _effdet(name)
    rel, cls = _effdet_heads(a, 3 + B, B, 81, HALF[dtype], cuda)
    kw = dict(iou_type=iou_type, with_indices=True)
    dec_h, out_h = a.decode_and_postprocess(rel, cls, **kw)
    dec_f, out_f = a.decode_and_postprocess([t.float() for t in rel], [t.float() for t in cls], **kw)
    _assert_same_dense(dec_h, dec_f)
    _assert_same_rows(out_h, out_f)
    _assert_same_dense(a.convert_outputs_boxes(rel), dec_f)
    if name == "d7":   # > 65 536 candidates in one image: the multi-CTA pre-selection ran
        assert sum(t.shape[1] * t.shape[2] * t.shape[3] for t in rel) > 65536
    # decoded fp32 boxes with half logits, on a slice of the batch
    first, n = (1, B - 1) if B > 1 else (0, 1)
    got = a.convert_outputs_batch(dec_f, cls, first_image=first, num_images=n, iou_type=iou_type, with_indices=True)
    want = a.convert_outputs_batch(dec_f, [t.float() for t in cls], first_image=first, num_images=n, iou_type=iou_type,
                                   with_indices=True)
    _assert_same_rows(got, want)
    if name == "d0":   # half decoded boxes as well
        dec_half = [t.to(HALF[dtype]) for t in dec_f]
        got = a.convert_outputs_batch(dec_half, cls, iou_type=iou_type, with_indices=True)
        want = a.convert_outputs_batch([t.float() for t in dec_half], [t.float() for t in cls], iou_type=iou_type, with_indices=True)
        _assert_same_rows(got, want)


def test_effdet_mixed_family_falls_back_to_fp32(lib, cuda):
    a = _effdet("d0")
    rel, cls = _effdet_heads(a, 41, 2, 81, torch.bfloat16, cuda)
    cls = [t.half() if i % 2 else t for i, t in enumerate(cls)]
    dec_h, out_h = a.decode_and_postprocess(rel, cls)
    dec_f, out_f = a.decode_and_postprocess([t.float() for t in rel], [t.float() for t in cls])
    _assert_same_dense(dec_h, dec_f)
    _assert_same_rows(out_h, out_f)


def test_effdet_half_call_makes_no_fp32_copy(lib, cuda):
    a = _effdet("d0")
    rel, cls = _effdet_heads(a, 51, 16, 81, torch.bfloat16, cuda)
    a.decode_and_postprocess(rel, cls)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    a.decode_and_postprocess(rel, cls)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < sum(t.numel() for t in rel + cls) * 4
