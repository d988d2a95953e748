"""EfficientDet training step from box lists (get_loss_from_boxes[_and_grad] / b200_effdet_loss_from_boxes_*).

The gradients must be bit-identical to generate_targets_batch + get_loss_and_grad on the same boxes, in both target forms
(class ids and one-hot rows): the match stage is generate_targets' own kernel, the box targets come from the same encoder
and the focal derivative from the same device function.  The loss is a sum in another order: within 1e-5 of get_loss on
the same targets and within 1e-4 of the oracle."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

from test_gpu_core import _t, assert_bits_equal
from test_gpu_effdet import CFGS, _pair

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32

# (config, B, C, iou_threshold, GT boxes in image 0 beyond one EF_GT_TILE of 128)
CASES = [("small", 3, 81, 0.5, False), ("rect", 2, 7, 0.5, False), ("d0", 2, 90, 0.5, False), ("small", 4, 4, 0.0, False),
         ("rect", 3, 90, 0.9, False), ("small", 2, 81, 0.5, True), ("d0", 4, 81, 0.9, False), ("small", 3, 7, 0.0, True)]


def _case_id(c):
    return "%s-B%d-C%d-thr%g%s" % (c[:4] + ("-many" if c[4] else "",))


def _inputs(a, name, B, C, many, seed):
    """Ragged boxes: the last image without boxes, an out-of-range and a negative class id, a duplicated GT with another
    class (the tie goes to the first), a GT equal to an anchor (matched, box target components exactly 0), and in
    `many` cases an image with more than 128 boxes; random heads."""
    from tfmv_b200 import synth
    rng = np.random.default_rng(seed)
    ih, iw = CFGS[name]["image_size"]
    boxes, classes, off = synth.gt_batch(rng, B, (iw, ih), max_boxes=30, min_boxes=5, order="yxyx")
    if many:
        b0, c0, _ = synth.gt_batch(rng, 1, (iw, ih), max_boxes=160, min_boxes=140, order="yxyx")
        boxes, classes = np.concatenate([b0, boxes[off[1]:]]), np.concatenate([c0, classes[off[1]:]])
        off = np.concatenate([[0], off[1:] - off[1] + len(b0)]).astype(np.int32)
    classes = (classes % (C - 1) + 1).astype(np.int32)
    classes[0], classes[1] = C + 3, -2
    boxes[3] = boxes[2]
    classes[3] = classes[2] % (C - 1) + 1
    anc = a.boxes[0].cpu().numpy()
    boxes[4] = anc[anc.shape[0] // 2, anc.shape[1] // 2, 0]
    cnt = np.diff(off)
    cnt[-1] = 0
    keep = np.arange(len(boxes)) < off[-2]
    boxes, classes, off = boxes[keep], classes[keep], np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    shapes = [tuple(b.shape) for b in a.boxes]
    pb = [(rng.standard_normal((B,) + s, dtype=F) * F(0.25)) for s in shapes]
    pc = [rng.standard_normal((B,) + s[:-1] + (C,), dtype=F) for s in shapes]
    return boxes, classes, off, pb, pc


def _oracle_targets(o, boxes, classes, off, C, thr):
    """The oracle's generate_targets per image (an image without boxes: all anchors unmatched, class 0)."""
    per = []
    for b in range(len(off) - 1):
        if off[b + 1] > off[b]:
            per.append(o.generate_targets(boxes[off[b]:off[b + 1]], classes[off[b]:off[b + 1]], C, iou_threshold=thr))
        else:
            shp = [s.shape[:-1] for s in o.boxes]
            per.append((tuple(np.zeros(s + (4,), F) for s in shp), tuple(np.eye(1, C, dtype=F)[0] * np.ones(s + (1,), F) for s in shp),
                        tuple(np.zeros(s + (1,), bool) for s in shp)))
    return [[np.stack([p[k][l] for p in per], 0) for l in range(len(o.boxes))] for k in range(3)]


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_grads_bit_identical_and_loss(lib, cuda, case):
    from oracle import effdet as oe
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import (get_loss, get_loss_and_grad, get_loss_from_boxes,
                                                                         get_loss_from_boxes_and_grad)
    name, B, C, thr, many = case
    a, o = _pair(name)
    boxes, classes, off, pb, pc = _inputs(a, name, B, C, many, 7100 + B + C)
    assert off[-1] == off[-2] and (np.diff(off)[:-1] > 0).all()
    assert not many or off[1] > 128
    db, dc, do = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    loss, gb, gc = get_loss_from_boxes_and_grad(a, db, dc, do, dpb, dpc, iou_threshold=thr)
    ib, ic, im = a.generate_targets_batch(db, dc, do, C, iou_threshold=thr, class_index=True)
    tb, tc, tm = a.generate_targets_batch(db, dc, do, C, iou_threshold=thr)
    for targets in ((ib, ic, im), (tb, tc, tm)):
        _, wb, wc = get_loss_and_grad(*targets, dpb, dpc)
        for l in range(len(pb)):
            assert gb[l].shape == dpb[l].shape and gc[l].shape == dpc[l].shape
            assert_bits_equal(gb[l].cpu().numpy(), wb[l].cpu().numpy())
            assert_bits_equal(gc[l].cpu().numpy(), wc[l].cpu().numpy())
    # the GT planted on an anchor: a matched anchor with a box target component exactly 0 (the Huber mask is target != 0)
    assert any(bool((t.reshape(-1, 4)[m.reshape(-1)] == 0).any()) for t, m in zip(tb, tm))
    f_loss, parts, npos = get_loss_from_boxes(a, db, dc, do, dpb, dpc, iou_threshold=thr, return_parts=True)
    assert f_loss.cpu().numpy().tobytes() == loss.cpu().numpy().tobytes()   # forward only: the same sums, bit for bit
    w_loss, w_parts, w_npos = get_loss(tb, tc, tm, dpb, dpc, return_parts=True)
    assert float(npos) == float(w_npos) == 1.0 + sum(int(m.sum()) for m in tm)
    np.testing.assert_allclose(parts.cpu().numpy(), w_parts.cpu().numpy(), rtol=1e-5, atol=1e-12)
    assert abs(float(loss) - float(w_loss)) <= 1e-5 * abs(float(w_loss))
    otb, otc, otm = _oracle_targets(o, boxes, classes, off, C, thr)
    want, o_parts, o_npos = oe.get_loss(otb, otc, otm, pb, pc, return_parts=True)
    assert float(npos) == float(o_npos)
    np.testing.assert_allclose(parts.cpu().numpy(), o_parts, rtol=1e-4, atol=1e-9)
    assert abs(float(loss) - float(want)) <= 1e-4 * abs(float(want))


def test_batch_without_boxes(lib, cuda):
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_and_grad, get_loss_from_boxes_and_grad
    a, _ = _pair("small")
    B, C = 3, 81
    _, _, _, pb, pc = _inputs(a, "small", B, C, False, 7200)
    boxes, classes, off = np.zeros((0, 4), F), np.zeros((0,), np.int32), np.zeros(B + 1, np.int32)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    loss, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, dpb, dpc)
    tb, tc, tm = a.generate_targets_batch(_t(boxes, cuda), _t(classes, cuda), _t(off, cuda), C)
    w_loss, wb, wc = get_loss_and_grad(tb, tc, tm, dpb, dpc)
    assert abs(float(loss) - float(w_loss)) <= 1e-5 * abs(float(w_loss))
    for l in range(len(pb)):
        assert_bits_equal(gc[l].cpu().numpy(), wc[l].cpu().numpy())
        assert not bool(gb[l].any())


def _abi_step(lib, a, boxes, classes, off, pb, pc, sums, gb, gc, ws, numel, stage):
    """One stage of the C ABI on device tensors (stage 'match' or 'grad')."""
    from tfmv_b200 import _tensors as T
    L, B, C = a._num_levels, off.numel() - 1, pc[0].shape[-1]
    arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])
    if stage == "match":
        return lib.b200_effdet_loss_from_boxes_match(L, a._hw, a._A, a._dev_table().data_ptr(), B, boxes.data_ptr(), off.data_ptr(),
                                                     boxes.shape[0], ctypes.c_float(0.5), sums.data_ptr(), ws.data_ptr(), ws.numel(),
                                                     T.stream_ptr())
    f = ctypes.c_float
    return lib.b200_effdet_loss_from_boxes_grad(L, a._hw, a._A, a._dev_table().data_ptr(), C, B, boxes.data_ptr(), classes.data_ptr(),
                                                boxes.shape[0], arr(pb), arr(pc), f(0.25), f(1.5), f(0.1), f(0.0),
                                                (ctypes.c_double * L)(*numel), sums.data_ptr(), arr(gb), arr(gc), ws.data_ptr(),
                                                ws.numel(), T.stream_ptr())


def test_sharded_stages_concatenate_to_the_full_batch(lib, cuda):
    """Two halves through the two ABI stages, the all-reduces played by torch adds: the gradients concatenate to the
    whole-batch call's bit for bit, and the finalized loss equals it to fp64 summation order."""
    import torch
    from tfmv_b200 import _tensors as T
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes_and_grad
    a, _ = _pair("small")
    B, C = 4, 81
    boxes, classes, off, pb, pc = _inputs(a, "small", B, C, False, 7300)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    loss, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, dpb, dpc)
    L = a._num_levels
    numel = [float(t.numel()) for t in dpc]   # global element counts
    shards = []
    for lo, hi in ((0, 2), (2, B)):
        s = dict(boxes=_t(boxes[off[lo]:off[hi]], cuda), classes=_t(classes[off[lo]:off[hi]], cuda),
                 off=_t((off[lo:hi + 1] - off[lo]).astype(np.int32), cuda), pb=[t[lo:hi].clone() for t in dpb],
                 pc=[t[lo:hi].clone() for t in dpc], sums=torch.full((2 * L + 1,), 7.0, dtype=torch.float64, device=cuda))
        s["gb"], s["gc"] = [torch.empty_like(t) for t in s["pb"]], [torch.empty_like(t) for t in s["pc"]]
        s["ws"] = torch.empty((lib.b200_effdet_loss_from_boxes_workspace_bytes(L, a._hw, a._A, hi - lo),), dtype=torch.uint8, device=cuda)
        shards.append(s)
    step = lambda s, stage: _abi_step(lib, a, s["boxes"], s["classes"], s["off"], s["pb"], s["pc"], s["sums"], s["gb"], s["gc"],
                                      s["ws"], numel, stage)
    for s in shards:
        assert step(s, "match") == 0
    npos = shards[0]["sums"][2 * L:] + shards[1]["sums"][2 * L:]
    for s in shards:
        s["sums"][2 * L:] = npos
        assert step(s, "grad") == 0
    sums = shards[0]["sums"] + shards[1]["sums"]
    sums[2 * L:] = npos
    for l in range(L):
        assert_bits_equal(torch.cat([shards[0]["gb"][l], shards[1]["gb"][l]]).cpu().numpy(), gb[l].cpu().numpy())
        assert_bits_equal(torch.cat([shards[0]["gc"][l], shards[1]["gc"][l]]).cpu().numpy(), gc[l].cpu().numpy())
    out = torch.empty((), dtype=torch.float32, device=cuda)
    assert lib.b200_focal_box_finalize(L, sums.data_ptr(), (ctypes.c_double * L)(*numel), None, out.data_ptr(), None, T.stream_ptr()) == 0
    assert abs(float(out) - float(loss)) <= 1e-6 * abs(float(loss))


def test_graph_replay_after_rewriting_the_boxes(lib, cuda):
    """Captured once, replayed after boxes / classes / offsets are rewritten in place (same total): equals an eager call."""
    from tfmv_b200 import runtime, synth
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes_and_grad
    a, _ = _pair("small")
    B, C = 3, 81
    boxes, classes, off, pb, pc = _inputs(a, "small", B, C, False, 7400)
    dpb, dpc = [_t(x, cuda) for x in pb], [_t(x, cuda) for x in pc]
    bd, cd, od = _t(boxes, cuda), _t(classes, cuda), _t(off, cuda)
    step = runtime.capture(lambda: get_loss_from_boxes_and_grad(a, bd, cd, od, dpb, dpc))
    rng = np.random.default_rng(7401)
    total = len(boxes)
    b2, c2, _ = synth.gt_batch(rng, 1, (128, 128), max_boxes=total, min_boxes=total, order="yxyx")
    c2 = (c2 % 80 + 1).astype(np.int32)
    o2 = np.concatenate([[0], np.sort(rng.integers(0, total + 1, B - 1)), [total]]).astype(np.int32)
    assert not np.array_equal(o2, off)
    bd.copy_(_t(b2, cuda))
    cd.copy_(_t(c2, cuda))
    od.copy_(_t(o2, cuda))
    r_loss, r_gb, r_gc = step()
    e_loss, e_gb, e_gc = get_loss_from_boxes_and_grad(a, b2, c2, o2, dpb, dpc)
    assert r_loss.cpu().numpy().tobytes() == e_loss.cpu().numpy().tobytes()
    for l in range(len(pb)):
        assert_bits_equal(r_gb[l].cpu().numpy(), e_gb[l].cpu().numpy())
        assert_bits_equal(r_gc[l].cpu().numpy(), e_gc[l].cpu().numpy())


def test_narrow_heads_take_the_two_call_path(lib, cuda):
    """classes_num < 4 (the reference fixture, tests/test_anchors.py): generate_targets_batch + get_loss, same results."""
    import torch
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import (get_loss, get_loss_and_grad, get_loss_from_boxes,
                                                                         get_loss_from_boxes_and_grad)
    a, _ = _pair("tiny")
    boxes = np.array([[3, 3, 6, 6], [5, 5, 9, 9], [2, 2, 5, 5]], F)
    classes, off = np.array([1, 2, 1], np.int32), np.array([0, 2, 3], np.int32)
    g = torch.Generator(device=cuda).manual_seed(11)
    pb = [torch.randn((2, 10, 10, 3, 4), device=cuda, generator=g) * 0.25]
    pc = [torch.randn((2, 10, 10, 3, 3), device=cuda, generator=g)]
    loss, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, pb, pc)
    tb, tc, tm = a.generate_targets_batch(_t(boxes, cuda), _t(classes, cuda), _t(off, cuda), 3)
    w_loss, wb, wc = get_loss_and_grad(tb, tc, tm, pb, pc)
    assert float(loss) == float(w_loss)
    assert_bits_equal(gb[0].cpu().numpy(), wb[0].cpu().numpy())
    assert_bits_equal(gc[0].cpu().numpy(), wc[0].cpu().numpy())
    f_loss, parts, npos = get_loss_from_boxes(a, boxes, classes, off, pb, pc, return_parts=True)
    w2, wparts, wnpos = get_loss(tb, tc, tm, pb, pc, return_parts=True)
    assert float(f_loss) == float(w2) and float(npos) == float(wnpos) > 1
    assert torch.equal(parts, wparts)


def _worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        sys.path.insert(0, ROOT)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import torch
        import torch.distributed as dist
        import tfmv_b200  # noqa: F401
        from tfmv_b200 import runtime
        from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_from_boxes_and_grad
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", device_id=dev)
        a, _ = _pair("small")
        B, C = 2 * world, 81
        boxes, classes, off, pb, pc = _inputs(a, "small", B, C, False, 7500)
        to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
        loss, gb, gc = get_loss_from_boxes_and_grad(a, boxes, classes, off, [to(x) for x in pb], [to(x) for x in pc])
        lo, hi = 2 * rank, 2 * rank + 2
        peer = runtime.PeerExchange()
        s_loss, s_gb, s_gc = get_loss_from_boxes_and_grad(a, boxes[off[lo]:off[hi]], classes[off[lo]:off[hi]], off[lo:hi + 1] - off[lo],
                                                          [to(x[lo:hi]) for x in pb], [to(x[lo:hi]) for x in pc], exchange=peer)
        torch.cuda.synchronize()
        res = {"loss": float(loss), "shard_loss": float(s_loss),
               "grads_equal": all(torch.equal(x, y[lo:hi]) for x, y in zip(list(s_gb) + list(s_gc), list(gb) + list(gc))),
               "status": peer.status()}
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
        assert v["grads_equal"], r
        assert abs(v["shard_loss"] - v["loss"]) <= 1e-6 * abs(v["loss"]), v
        assert v["shard_loss"] == res[0]["shard_loss"] and v["status"][1] == 0
