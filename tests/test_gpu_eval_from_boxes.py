"""Validation step from box lists: Anchors.eval_step_from_boxes (b200_effdet_eval_step_from_boxes), the YOLO
GetGroudTruthFromBoxes (b200_yolo_ground_truth_from_boxes) / EvalStepFromBoxes and the padded mAP (Get_mAP_padded /
b200_map_padded).

eval_step_from_boxes must give, bit for bit, what generate_targets_batch + eval_step give on the same boxes: the decoded
tensors, every NMS output and the loss terms (the match stage is generate_targets' own kernel, the one-hot rows and box
targets are rebuilt with the same values, and the stream sums them in the same order).  The YOLO rows must equal, image by
image, GetGroudTruth of the three levels GetTargetsBatch writes, and EvalStepFromBoxes the separate calls.  Get_mAP_padded
must equal the reference-generated golden values and Get_mAP_batch on the same rows."""
import os
import socket
import sys

import numpy as np
import pytest

from test_gpu_core import _t, assert_bits_equal
from test_gpu_effdet import CFGS, _pair
from test_gpu_effdet_sparse_grad import _inputs
from test_map import _cases, _degenerate_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32
OUT_KEYS = ("boxes", "classes_id", "scores", "count", "sel_idx", "sel_anchor")


def _assert_same_step(got, want):
    loss, dec, out, parts, npos = got
    w_loss, w_dec, w_out, w_parts, w_npos = want
    assert loss.cpu().numpy().tobytes() == w_loss.cpu().numpy().tobytes()
    assert parts.cpu().numpy().tobytes() == w_parts.cpu().numpy().tobytes()
    assert float(npos) == float(w_npos)
    for d, w in zip(dec, w_dec):
        assert_bits_equal(d.cpu().numpy(), w.cpu().numpy())
    assert set(out) == set(w_out)
    cnt = w_out["count"].cpu().numpy()
    assert np.array_equal(out["count"].cpu().numpy(), cnt)
    for k in OUT_KEYS:
        if k not in w_out or k == "count":
            continue
        g, w = out[k].cpu().numpy(), w_out[k].cpu().numpy()
        for b, n in enumerate(cnt):   # rows past count are not written
            assert g[b, :n].tobytes() == w[b, :n].tobytes(), (k, b)


def _two_call(a, db, dc, do, dpb, dpc, C, gamma=1.5, thr=0.5, iou_type="diou"):
    tb, tc, tm = a.generate_targets_batch(db, dc, do, C, iou_threshold=thr)
    return a.eval_step(tb, tc, tm, dpb, dpc, gamma=gamma, iou_type=iou_type, with_indices=True, return_parts=True)


# (config, B, C, gamma, match threshold, NMS metric)
CASES = [("d0", 2, 81, 1.5, 0.5, "diou"), ("small", 3, 81, 1.5, 0.5, "diou"), ("rect", 3, 7, 2.0, 0.5, "ciou"),
         ("small", 2, 90, 2.0, 0.0, "giou"), ("d0", 3, 4, 1.5, 0.9, "iou")]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-B%d-C%d-g%g-thr%g-%s" % c)
def test_effdet_eval_step_from_boxes_bit_identical(lib, cuda, case):
    """Ragged boxes with an image without boxes, out-of-range and negative class ids (from _inputs)."""
    name, B, C, gamma, thr, iou_type = case
    a, _ = _pair(name)
    boxes, classes, off, pb, pc = _inputs(a, name, B, C, False, 8100 + B + C)
    assert off[-1] == off[-2] and (classes >= C).any() and (classes < 0).any()
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    got = a.eval_step_from_boxes(db, dc, do, dpb, dpc, match_iou_threshold=thr, gamma=gamma, iou_type=iou_type,
                                 with_indices=True, return_parts=True)
    _assert_same_step(got, _two_call(a, db, dc, do, dpb, dpc, C, gamma, thr, iou_type))
    assert float(got[4]) > 1 and int(got[2]["count"].sum()) > 0


def test_ragged_level_takes_the_plain_load_path(lib, cuda):
    """B*anchors of a level not a multiple of the 64-anchor tile: the last tile of that level is read without bulk copies."""
    a, _ = _pair("small")
    B, C = 3, 81
    ragged = [B * h * w * a._A % 64 for h, w in a._level_hw]
    assert any(r != 0 for r in ragged), ragged
    boxes, classes, off, pb, pc = _inputs(a, "small", B, C, True, 8200)
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    got = a.eval_step_from_boxes(db, dc, do, dpb, dpc, with_indices=True, return_parts=True)
    _assert_same_step(got, _two_call(a, db, dc, do, dpb, dpc, C))


def test_batch_without_boxes(lib, cuda):
    a, _ = _pair("small")
    B, C = 2, 81
    _, _, _, pb, pc = _inputs(a, "small", B, C, False, 8300)
    boxes, classes, off = np.zeros((0, 4), F), np.zeros((0,), np.int32), np.zeros(B + 1, np.int32)
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    got = a.eval_step_from_boxes(db, dc, do, dpb, dpc, with_indices=True, return_parts=True)
    _assert_same_step(got, _two_call(a, db, dc, do, dpb, dpc, C))
    assert float(got[4]) == 1.0


@pytest.mark.parametrize("C", [3, 129])
def test_narrow_and_wide_heads_take_the_two_call_path(lib, cuda, C):
    a, _ = _pair("small")
    B = 2
    boxes, classes, off, pb, pc = _inputs(a, "small", B, C, False, 8400 + C)
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    got = a.eval_step_from_boxes(db, dc, do, dpb, dpc, with_indices=True, return_parts=True)
    _assert_same_step(got, _two_call(a, db, dc, do, dpb, dpc, C))


# ---- Get_mAP_padded ---------------------------------------------------------------------------------------------------
def _pad(cases, K, cls_dtype, rng, extra_gt=0):
    """Golden cases (gt [n,5], pr [m,6]) as the padded NMS dict + box lists; padding slots and `extra_gt` trailing GT
    rows per image hold junk that count / gt_count must exclude."""
    B = len(cases)
    boxes = rng.uniform(0, 50, (B, K, 4)).astype(F)
    cls = np.zeros((B, K), cls_dtype)
    scores = np.full((B, K), 2.0, F)
    count = np.zeros(B, np.int32)
    gtb, gtc, off, gcnt = [], [], [0], []
    for b, (gt, pr, _, _) in enumerate(cases):
        m = pr.shape[0]
        boxes[b, :m], cls[b, :m], scores[b, :m], count[b] = pr[:, :4], pr[:, 4], pr[:, 5], m
        junk = rng.uniform(0, 50, (extra_gt, 4)).astype(F)
        gtb += [gt[:, :4].astype(F), junk]
        gtc += [gt[:, 4].astype(np.int32), np.zeros(extra_gt, np.int32)]
        gcnt.append(gt.shape[0])
        off.append(off[-1] + gt.shape[0] + extra_gt)
    nms = dict(boxes=boxes, classes_id=cls, scores=scores, count=count)
    return nms, np.concatenate(gtb), np.concatenate(gtc), np.asarray(off, np.int32), np.asarray(gcnt, np.int32)


@pytest.mark.parametrize("cls_dtype", [np.int32, np.int64])
def test_map_padded_matches_reference_generated_golden(lib, cuda, cls_dtype):
    import torch
    from tfmv_b200.ai_models.utils.mAP import Get_mAP_padded
    rng = np.random.default_rng(5)
    for C in sorted({c[2] for c in _cases()}):
        cases = [c for c in _cases() if c[2] == C]
        K = max(1, max(c[1].shape[0] for c in cases)) + 3
        for extra in (0, 2):
            nms, gb, gc, off, gcnt = _pad(cases, K, cls_dtype, rng, extra)
            dnms = {k: _t(v, cuda) for k, v in nms.items()}
            assert dnms["classes_id"].dtype == (torch.int32 if cls_dtype is np.int32 else torch.int64)
            got = Get_mAP_padded(_t(gb, cuda), _t(gc, cuda), _t(off, cuda), dnms, C, 0.5,
                                 gt_count=_t(gcnt, cuda) if extra else None)
            assert got.dtype == torch.float64 and got.shape == (len(cases),)
            for j, c in enumerate(cases):
                assert abs(float(got[j]) - c[3]) < 1e-12, (C, j, extra, float(got[j]), c[3])


def test_map_padded_nan_iou_follows_np_argmax(lib, cuda):
    from oracle import map as om
    from tfmv_b200.ai_models.utils.mAP import Get_mAP_padded
    gt, pr = _degenerate_case()
    rng = np.random.default_rng(6)
    for order in ([0, 1, 2], [1, 0, 2], [2, 1, 0]):
        p = pr[order]
        nms, gb, gc, off, _ = _pad([(gt, p, 3, 0.0)], 4, np.int64, rng)
        got = float(Get_mAP_padded(_t(gb, cuda), _t(gc, cuda), _t(off, cuda), {k: _t(v, cuda) for k, v in nms.items()}, 3)[0])
        assert abs(got - om.get_map_one(gt, p, 3, 0.5)) < 1e-12, order


def _random_image(rng, n_gt, n_pr, C, size=400.0):
    xy = rng.uniform(0, size, (n_gt, 2))
    wh = rng.uniform(4, 60, (n_gt, 2))
    gt = np.concatenate([xy, xy + wh, rng.integers(0, C, (n_gt, 1))], 1).astype(F).astype(np.float64)
    # predictions: jittered copies of some GT boxes (true positives at several IoUs) and random boxes
    src = gt[rng.integers(0, n_gt, n_pr)]
    jit = rng.normal(0, 3, (n_pr, 4))
    pr_boxes = src[:, :4] + jit
    pr_boxes[:, 2:] = np.maximum(pr_boxes[:, 2:], pr_boxes[:, :2] + 1)
    cls = np.where(rng.random(n_pr) < 0.8, src[:, 4], rng.integers(0, C, n_pr))
    score = rng.random(n_pr).astype(F)
    score[::7] = score[0]   # ties
    pr = np.concatenate([pr_boxes, cls[:, None], score[:, None]], 1).astype(F).astype(np.float64)
    return gt, pr


@pytest.mark.parametrize("n_gt,n_pr,K", [(2500, 300, 300), (150, 4000, 4096), (1030, 4096, 4096)])
def test_map_padded_many_boxes(lib, cuda, n_gt, n_pr, K):
    """More ground truth than one shared-memory chunk (1024 rows), and K = NMS_MAX_OUT_LIMIT: equals Get_mAP_batch on the
    same rows and the oracle."""
    from oracle import map as om
    from tfmv_b200.ai_models.utils.mAP import Get_mAP_batch, Get_mAP_padded
    rng = np.random.default_rng(n_gt + n_pr)
    C = 5
    imgs = [_random_image(rng, n_gt, n_pr, C), _random_image(rng, max(1, n_gt // 3), n_pr // 2, C)]
    nms, gb, gc, off, _ = _pad([(g, p, C, 0.0) for g, p in imgs], K, np.int32, rng)
    got = Get_mAP_padded(_t(gb, cuda), _t(gc, cuda), _t(off, cuda), {k: _t(v, cuda) for k, v in nms.items()}, C)
    go = np.cumsum([0] + [g.shape[0] for g, _ in imgs]).astype(np.int32)
    po = np.cumsum([0] + [p.shape[0] for _, p in imgs]).astype(np.int32)
    want = Get_mAP_batch(np.concatenate([g for g, _ in imgs]), go, np.concatenate([p for _, p in imgs]), po, C)
    assert got.cpu().numpy().tobytes() == want.cpu().numpy().tobytes()
    for j, (g, p) in enumerate(imgs):
        assert abs(float(got[j]) - om.get_map_one(g, p, C, 0.5)) < 1e-12
    assert float(got[0]) > 0


def test_map_padded_on_eval_step_output(lib, cuda):
    """The mAP of test_step on eval_step_from_boxes' output with the box lists as ground truth equals Get_mAP_batch on
    the compacted rows."""
    import torch
    from tfmv_b200.ai_models.utils.mAP import Get_mAP_batch, Get_mAP_padded
    a, _ = _pair("small")
    B, C = 3, 81
    boxes, classes, off, pb, pc = _inputs(a, "small", B, C, False, 8500)
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    _, _, out = a.eval_step_from_boxes(db, dc, do, [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc])
    got = Get_mAP_padded(db, dc, do, out, C)
    cnt = out["count"].cpu().numpy()
    pred = torch.cat([torch.cat([out["boxes"][b, :n], out["classes_id"][b, :n, None].float(), out["scores"][b, :n, None]], 1)
                      for b, n in enumerate(cnt)])
    gt = torch.cat([db, dc[:, None].float()], 1)
    want = Get_mAP_batch(gt, off, pred, np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32), C)
    assert got.cpu().numpy().tobytes() == want.cpu().numpy().tobytes()


def test_graph_replay_after_rewriting_the_boxes(lib, cuda):
    """eval_step_from_boxes + Get_mAP_padded captured once and replayed after the box lists are rewritten in place: equal
    to eager calls.  The capture itself shows the step never synchronises with the host."""
    from tfmv_b200 import runtime, synth
    from tfmv_b200.ai_models.utils.mAP import Get_mAP_padded
    a, _ = _pair("small")
    B, C = 3, 81
    boxes, classes, off, pb, pc = _inputs(a, "small", B, C, False, 8600)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)

    def step():
        loss, dec, out, parts, npos = a.eval_step_from_boxes(bd, cd, od, dpb, dpc, with_indices=True, return_parts=True)
        return loss, dec, out, parts, npos, Get_mAP_padded(bd, cd, od, out, C)

    replay = runtime.capture(step)
    rng = np.random.default_rng(8601)
    total = len(boxes)
    ih, iw = CFGS["small"]["image_size"]
    b2, c2, _ = synth.gt_batch(rng, 1, (iw, ih), max_boxes=total, min_boxes=total, order="yxyx")
    c2 = (c2 % 80 + 1).astype(np.int32)
    o2 = np.concatenate([[0], np.sort(rng.integers(0, total + 1, B - 1)), [total]]).astype(np.int32)
    assert not np.array_equal(o2, off)
    bd.copy_(_t(b2, cuda))
    cd.copy_(_t(c2, cuda))
    od.copy_(_t(o2, cuda))
    r = replay()
    e = step()
    _assert_same_step(r[:5], e[:5])
    assert r[5].cpu().numpy().tobytes() == e[5].cpu().numpy().tobytes()


def _worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        sys.path.insert(0, ROOT)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import torch
        import torch.distributed as dist
        import tfmv_b200  # noqa: F401
        from tfmv_b200 import runtime
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", device_id=dev)
        a, _ = _pair("small")
        B, C = 2 * world, 81
        boxes, classes, off, pb, pc = _inputs(a, "small", B, C, False, 8700)
        to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
        loss = a.eval_step_from_boxes(boxes, classes, off, [to(x) for x in pb], [to(x) for x in pc])[0]
        lo, hi = 2 * rank, 2 * rank + 2
        peer = runtime.PeerExchange()
        s_loss = a.eval_step_from_boxes(boxes[off[lo]:off[hi]], classes[off[lo]:off[hi]], off[lo:hi + 1] - off[lo],
                                        [to(x[lo:hi]) for x in pb], [to(x[lo:hi]) for x in pc], exchange=peer)[0]
        torch.cuda.synchronize()
        res = {"loss": float(loss), "shard_loss": float(s_loss), "status": peer.status()}
        dist.barrier()
        peer.close()
        dist.destroy_process_group()
        q.put((rank, res))
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put((rank, {"error": "%s\n%s" % (e, traceback.format_exc())}))


def test_two_gpus_over_peer_mailboxes(lib, cuda):
    import torch
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 2)
    if world < 2:
        pytest.skip("needs two GPUs (one process per GPU)")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=120)
    for r in range(world):
        assert "error" not in res[r], res[r]["error"]
        v = res[r]
        assert abs(v["shard_loss"] - v["loss"]) <= 1e-4 * abs(v["loss"]), v
        assert v["shard_loss"] == res[0]["shard_loss"] and v["status"][1] == 0


# ---- YOLO -------------------------------------------------------------------------------------------------------------
def _yolo_dense_rows(classes, boxes, off, image_wh, tanc, C, cuda):
    """GetGroudTruth of the three levels of GetTargetsBatch, image by image."""
    import torch
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetGroudTruth
    y = DataGenerator(C, tanc, image_wh).GetTargetsBatch(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda))
    return [torch.cat([GetGroudTruth(t[b]) for t in y]) for b in range(len(off) - 1)]


def _assert_rows_equal(rows, count, want, off):
    cnt = count.cpu().numpy()
    assert [len(w) for w in want] == cnt.tolist()
    for b, w in enumerate(want):
        assert_bits_equal(rows[off[b]:off[b] + cnt[b]].cpu().numpy(), w.cpu().numpy())


def _yolo_boxes(rng, B, image_wh, C):
    """Ragged boxes: a triple collision (all three dropped), a box whose centre lies outside the image (rejected by the
    assignment), negative and too-large class ids, and an image without boxes when B > 2."""
    from tfmv_b200 import synth
    boxes, classes, off = synth.gt_batch(rng, B, image_wh, max_boxes=40, classes=C, min_boxes=6)
    boxes[1] = boxes[0]
    boxes[2] = boxes[0]
    w, h = image_wh
    boxes[4] = [w + 10, 5, w + 40, min(30, h)]
    classes[3], classes[-1] = -1, C + 5
    if B > 2:
        keep = np.ones(len(boxes), bool)
        keep[off[1]:off[2]] = False
        cnt = np.diff(off)
        cnt[1] = 0
        boxes, classes, off = boxes[keep], classes[keep], np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    return boxes.astype(F), classes.astype(np.int32), off.astype(np.int32)


# (image_wh, A, C, B, target anchors normalised by the image width)
GT_CASES = [((416, 416), 3, 80, 3, False), ((608, 608), 3, 80, 2, False), ((416, 256), 3, 20, 3, False),
            ((320, 200), 2, 7, 3, False), ((96, 96), 3, 80, 4, True)]


@pytest.mark.parametrize("case", GT_CASES, ids=lambda c: "%dx%d-A%d-C%d-B%d" % (c[0] + c[1:4]) + ("-normalised" if c[4] else ""))
def test_yolo_ground_truth_from_boxes_bit_identical(lib, cuda, case):
    from test_gpu_yolo_shapes import _anchors, _rng
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetGroudTruthFromBoxes
    image_wh, A, C, B, normalised = case
    rng = _rng("gt-from-boxes", case)
    anc = _anchors(A)
    tanc = anc / F(image_wh[0]) if normalised else anc
    boxes, classes, off = _yolo_boxes(rng, B, image_wh, C)
    rows, count = GetGroudTruthFromBoxes(_t(classes, cuda), _t(boxes, cuda), _t(off, cuda), image_wh, tanc, C)
    want = _yolo_dense_rows(classes, boxes, off, image_wh, tanc, C, cuda)
    _assert_rows_equal(rows, count, want, off)
    assert int(count[0]) < off[1] - off[0]          # the collision and the rejected box are gone
    assert sum(len(w) for w in want) > 0


def _yolo_eval_inputs(case, cuda):
    from test_gpu_yolo_sparse_grad import _inputs as yolo_inputs
    boxes, classes, off, _, y_pred, anc, tanc = yolo_inputs(case)
    return boxes, classes, off, [_t(h, cuda) for h in y_pred], anc, tanc


YOLO_EVAL_CASES = [((416, 416), 80, 3, "ciou", False), ((608, 608), 80, 2, "iou", False), ((416, 256), 80, 2, "ciou", False),
                   ((96, 96), 80, 4, "diou", True)]


@pytest.mark.parametrize("case", YOLO_EVAL_CASES, ids=lambda c: "%dx%d-C%d-B%d-%s" % (c[0] + c[1:4]) + ("-normalised" if c[4] else ""))
def test_yolo_eval_step_from_boxes(lib, cuda, case):
    """Loss bit-identical to GetLossFromBoxes, the NMS dict to GetNMSBoxesBatch, the mAP equal in fp64 to Get_mAP_batch on
    the compacted rows and within 1e-12 of the oracle."""
    import torch
    from oracle import map as om
    from tfmv_b200.ai_models.utils.mAP import Get_mAP_batch
    from tfmv_b200.ai_models.utils.tf_yolo_utils import EvalStepFromBoxes, GetLossFromBoxes, GetNMSBoxesBatch
    image_wh, C, B, iou_type, _ = case
    boxes, classes, off, heads, anc, tanc = _yolo_eval_inputs(case, cuda)
    loss, parts, r, m_ap = EvalStepFromBoxes(classes, boxes, off, heads, image_wh, anc, C, 0.5, iou_type, nms_iou_type="diou",
                                             target_anchors=tanc, return_parts=True)
    w_loss, w_parts = GetLossFromBoxes(classes, boxes, off, heads, image_wh, anc, C, 0.5, iou_type, target_anchors=tanc,
                                       return_parts=True)
    assert loss.cpu().numpy().tobytes() == w_loss.cpu().numpy().tobytes()
    assert parts.cpu().numpy().tobytes() == w_parts.cpu().numpy().tobytes()
    w_r = GetNMSBoxesBatch(*heads, anc, image_wh, C, 0.5, 0.3, 0.5, "diou")
    cnt = w_r["count"].cpu().numpy()
    assert set(r) == set(w_r) and np.array_equal(r["count"].cpu().numpy(), cnt) and cnt.sum() > 0
    for k in w_r:
        if k == "count":
            continue
        g, w = r[k].cpu().numpy(), w_r[k].cpu().numpy()
        for b, n in enumerate(cnt):
            assert g[b, :n].tobytes() == w[b, :n].tobytes(), (k, b)
    gt = _yolo_dense_rows(classes, boxes, off, image_wh, tanc, C, cuda)
    pred = [torch.cat([w_r["boxes"][b, :n], w_r["classes_id"][b, :n, None].float(), w_r["scores"][b, :n, None]], 1)
            for b, n in enumerate(cnt)]
    want = Get_mAP_batch(torch.cat(gt), np.cumsum([0] + [len(g) for g in gt]).astype(np.int32), torch.cat(pred),
                         np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32), C)
    assert m_ap.dtype == torch.float64 and m_ap.cpu().numpy().tobytes() == want.cpu().numpy().tobytes()
    for b in range(B):
        assert abs(float(m_ap[b]) - om.get_map_one(gt[b].cpu().numpy(), pred[b].cpu().numpy(), C, 0.5)) < 1e-12


def test_yolo_graph_replay_after_rewriting_the_boxes(lib, cuda):
    from tfmv_b200 import runtime, synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import EvalStepFromBoxes
    case = YOLO_EVAL_CASES[0]
    image_wh, C, B = case[0], case[1], case[2]
    boxes, classes, off, heads, anc, _ = _yolo_eval_inputs(case, cuda)
    bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    step = lambda: EvalStepFromBoxes(cd, bd, od, heads, image_wh, anc, C, 0.5, "ciou", nms_iou_type="diou")
    replay = runtime.capture(step)
    rng = np.random.default_rng(8801)
    total = len(boxes)
    b2, c2, _ = synth.gt_batch(rng, 1, image_wh, max_boxes=total, classes=C, min_boxes=total)
    o2 = np.concatenate([[0], np.sort(rng.integers(0, total + 1, B - 1)), [total]]).astype(np.int32)
    assert not np.array_equal(o2, off)
    bd.copy_(_t(b2.astype(F), cuda))
    cd.copy_(_t(c2.astype(np.int32), cuda))
    od.copy_(_t(o2, cuda))
    r_loss, r_r, r_map = replay()
    e_loss, e_r, e_map = step()
    assert r_loss.cpu().numpy().tobytes() == e_loss.cpu().numpy().tobytes()
    assert r_map.cpu().numpy().tobytes() == e_map.cpu().numpy().tobytes()
    for k in e_r:
        assert r_r[k].cpu().numpy().tobytes() == e_r[k].cpu().numpy().tobytes(), k
