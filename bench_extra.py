#!/usr/bin/env python
"""bench_extra.py — device-resident throughput of the other BASELINE.json configs (1, 3, 4, 5-per-GPU).

Not the driver's bench (that is bench.py on config 2); this prints one JSON line per workload so DESIGN.md and
profiles/ can quote measured numbers for every §8 row.  Inputs are generated on the device (synthetic, the shapes
and distributions of BASELINE.md §3); timing: CUDA events, >= 3 warm-up steps, inputs larger than L2 unless noted.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
F = np.float32


def timed(fn, steps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _card():
    """Name and power limit of cuda:0, read next to the measurement (a read-only nvidia-smi query)."""
    import subprocess
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit"] = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        out["power_limit"] = "unknown"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="all")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--graph", action="store_true", help="replay each step as a CUDA graph")
    args = ap.parse_args()
    import torch
    import tfmv_b200  # noqa: F401
    from tfmv_b200 import runtime, synth
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss
    from tfmv_b200.ai_models.efficientnet.utils.anchors import Anchors
    from tfmv_b200.ai_models.utils import tf_yolo_utils as tyu
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    peak = 6466.5
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    g = torch.Generator(device=dev).manual_seed(20261018)
    anc = synth.yolo_anchors().astype(F)

    def yolo_heads(batch, image):
        return [torch.randn((batch, s, s, 255), device=dev, generator=g) for s in synth.yolo_grids(image)]

    def report(name, what, batch, ms, bytes_per_img, extra=None):
        line = {"workload": name, "what": what, "batch": batch, "ms_per_step": ms, "images_per_s": batch / ms * 1e3,
                "algorithmic_bytes_per_image": bytes_per_img, "dense_equiv_gbps": bytes_per_img * batch / ms / 1e6,
                "frac_of_measured_hbm_peak": bytes_per_img * batch / ms / 1e6 / peak, "peak_gbps": peak,
                "launch": "graph" if args.graph else "launch by launch"}
        if extra:
            line.update(extra)
        print(json.dumps(line), flush=True)

    def wrap(fn):
        return runtime.capture(fn) if args.graph else fn

    want = lambda n: args.workload in ("all", n)

    if want("c1_b1"):  # config 1: YOLOv3 416, batch 1, decode + per-class NMS ('iou', 0.5/0.3/0.5): latency
        heads = yolo_heads(1, 416)
        fn = wrap(lambda: tyu.GetNMSBoxesBatch(*heads, anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou"))
        ms = timed(fn, max(args.steps, 50), 10)
        report("c1_b1", "YOLOv3 416 B=1 decode+per-class NMS (latency; input 3.6 MB is L2-resident)", 1, ms, 3619980 + 174000,
               {"latency_us": ms * 1e3})
    if want("c1_b256"):
        heads = yolo_heads(256, 416)
        fn = wrap(lambda: tyu.GetNMSBoxesBatch(*heads, anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou"))
        ms = timed(fn, args.steps, args.warmup)
        report("c1_b256", "YOLOv3 416 B=256 decode+per-class NMS", 256, ms, 3619980 + 174000)
    if want("c1_b256_trained"):  # SURVEY 8d second input set: conf ~ N(-4,1.5), 50 planted objects x 5 duplicates per image
        rng = np.random.default_rng(20261018 + 1)
        base = synth.yolo_heads_trained_like(rng, 32, 416)
        heads = [torch.from_numpy(np.tile(h, (8, 1, 1, 1))).to(dev) for h in base]
        fn = wrap(lambda: tyu.GetNMSBoxesBatch(*heads, anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou"))
        ms = timed(fn, args.steps, args.warmup)
        kept = int(tyu.GetNMSBoxesBatch(*heads, anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou")["count"].sum().item())
        report("c1_b256_trained", "YOLOv3 416 B=256 decode+per-class NMS, trained-like heads (32 generated images tiled x8)", 256, ms,
               3619980 + 174000, {"kept_boxes_total": kept})
    if want("c5_b64"):  # config 5 per GPU: YOLOv4 608, decode + loss + NMS ('diou'), y_true given
        batch, image = 64, 608
        heads = yolo_heads(batch, image)
        rng = np.random.default_rng(20261018 + 5)
        boxes, classes, off = synth.gt_batch(rng, batch, (image, image), max_boxes=100)
        gen = DataGenerator(80, anc, (image, image))
        y_true = gen.GetTargetsBatch(torch.from_numpy(classes).to(dev), torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev))

        def step():
            loss = tyu.GetLoss(y_true, heads, (image, image), anc, 0.5, "ciou")
            r = tyu.GetNMSBoxesBatch(*heads, anc, (image, image), 80, 0.5, 0.3, 0.5, "diou")
            return loss, r
        ms = timed(wrap(step), args.steps, args.warmup)
        report("c5_b64", "YOLOv4 608 B=64 per GPU: GetLoss(ciou) + decode + per-class NMS(diou)", batch, ms, 15639240)
    if want("c2_backward"):  # SURVEY 8f N1 on config 2: GetLoss forward + d loss / d y_pred (dense gradient written)
        batch, image = 64, 608
        heads = yolo_heads(batch, image)
        rng = np.random.default_rng(20261018 + 2)
        boxes, classes, off = synth.gt_batch(rng, batch, (image, image), max_boxes=100)
        gen = DataGenerator(80, anc, (image, image))
        y_true = gen.GetTargetsBatch(torch.from_numpy(classes).to(dev), torch.from_numpy(boxes).to(dev), torch.from_numpy(off).to(dev))
        ms_f = timed(wrap(lambda: tyu.GetLoss(y_true, heads, (image, image), anc, 0.5, "ciou")), args.steps, args.warmup)
        ms = timed(wrap(lambda: tyu.GetLossAndGrad(y_true, heads, (image, image), anc, 0.5, "ciou")), args.steps, args.warmup)
        report("c2_backward", "YOLOv4 608 B=64: GetLossAndGrad(ciou) = forward + dense d loss/d y_pred (y_true given)", batch, ms,
               3 * 7732620, {"forward_only_ms": ms_f, "note": "bytes: read y_true + read y_pred + write the gradient"})
    if want("c2_sparse_backward"):  # SURVEY 8f N3 + N1: the training step from box lists against the drop-in one
        card = _card()
        batch, image = 64, 608
        heads = yolo_heads(batch, image)
        rng = np.random.default_rng(20261018 + 2)
        boxes, classes, off = synth.gt_batch(rng, batch, (image, image), max_boxes=100)
        boxes_d, classes_d, off_d = (torch.from_numpy(x).to(dev) for x in (boxes, classes, off))
        gen = DataGenerator(80, anc, (image, image))
        arms = {
            "dense": lambda: tyu.GetLossAndGrad(gen.GetTargetsBatch(classes_d, boxes_d, off_d), heads, (image, image), anc, 0.5, "ciou"),
            "sparse": lambda: tyu.GetLossFromBoxesAndGrad(classes_d, boxes_d, off_d, heads, (image, image), anc, 80, 0.5, "ciou"),
            "sparse_forward": lambda: tyu.GetLossFromBoxes(classes_d, boxes_d, off_d, heads, (image, image), anc, 80, 0.5, "ciou"),
        }
        loss_a, grads_a = arms["dense"]()
        loss_b, grads_b = arms["sparse"]()
        assert all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(grads_a, grads_b)), \
            "GetLossFromBoxesAndGrad and GetTargetsBatch + GetLossAndGrad disagree on the gradient bits"
        loss_rel = abs(float(loss_b) - float(loss_a)) / abs(float(loss_a))
        del grads_a, grads_b
        fns = {k: wrap(f) for k, f in arms.items()}
        # the arms alternate window by window (order rotated) so that drift of clocks and neighbours hits all of them
        steps, n_win = max(args.steps, 50), 7
        times = {k: [] for k in fns}
        order = list(fns)
        for w in range(n_win):
            for k in order[w % 3:] + order[:w % 3]:
                times[k].append(timed(fns[k], steps, args.warmup))
        ms = {k: float(np.median(v)) for k, v in times.items()}
        report("c2_sparse_backward", "YOLOv4 608 B=64 training step from box lists: GetLossFromBoxesAndGrad(ciou) against "
               "GetTargetsBatch + GetLossAndGrad (gradients asserted bit-identical first) and GetLossFromBoxes alone; median of %d "
               "alternating windows of %d steps" % (n_win, steps), batch, ms["sparse"], 2 * 7732620,
               dict(card, dense_targets_and_grad_ms=ms["dense"], from_boxes_forward_ms=ms["sparse_forward"],
                    speedup_vs_dense=ms["dense"] / ms["sparse"], window_ms={k: [round(t, 5) for t in v] for k, v in times.items()},
                    grads_bit_identical=True, loss_rel_diff=loss_rel,
                    note="bytes: read y_pred + write the gradient (dense equivalent; y_pred and the gradients exceed the 126 MB L2)"))
    if want("c3_sparse_backward"):  # SURVEY 8f N3 + N1 for EfficientDet: the training step from box lists against the two-call ones
        from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import (get_loss_and_grad, get_loss_from_boxes,
                                                                             get_loss_from_boxes_and_grad)
        card = _card()
        c = synth.EFFDET_CONFIGS["d0"]
        batch, C = 128, 81
        a = Anchors(c["min_level"], c["max_level"], c["image_size"], c["num_scales"], c["aspect_ratios"], c["anchor_scale"])
        shapes = [tuple(b.shape) for b in a.boxes]
        rel = [torch.randn((batch,) + s, device=dev, generator=g) * 0.25 for s in shapes]
        cls = [torch.randn((batch,) + s[:-1] + (C,), device=dev, generator=g) for s in shapes]
        n_anchor = sum(s[0] * s[1] * s[2] for s in shapes)
        rng = np.random.default_rng(20261018 + 3)
        boxes, classes, off = synth.gt_batch(rng, batch, (c["image_size"][1], c["image_size"][0]), max_boxes=100, order="yxyx")
        d_boxes, d_cls, d_off = (torch.from_numpy(boxes).to(dev), torch.from_numpy((classes + 1).astype(np.int32)).to(dev),
                                 torch.from_numpy(off).to(dev))
        arms = {
            "one_hot": lambda: get_loss_and_grad(*a.generate_targets_batch(d_boxes, d_cls, d_off, C), rel, cls),
            "class_id": lambda: get_loss_and_grad(*a.generate_targets_batch(d_boxes, d_cls, d_off, C, class_index=True), rel, cls),
            "from_boxes": lambda: get_loss_from_boxes_and_grad(a, d_boxes, d_cls, d_off, rel, cls),
            "from_boxes_forward": lambda: get_loss_from_boxes(a, d_boxes, d_cls, d_off, rel, cls),
        }
        res = {k: arms[k]() for k in ("one_hot", "class_id", "from_boxes")}
        same = lambda x, y: all(torch.equal(p.view(torch.int32), q.view(torch.int32)) for p, q in zip(x[1] + x[2], y[1] + y[2]))
        assert same(res["one_hot"], res["from_boxes"]) and same(res["class_id"], res["from_boxes"]), \
            "get_loss_from_boxes_and_grad and generate_targets_batch + get_loss_and_grad disagree on the gradient bits"
        loss_ref = float(res["one_hot"][0])
        loss_rel = abs(float(res["from_boxes"][0]) - loss_ref) / abs(loss_ref)
        fwd_bits = float(arms["from_boxes_forward"]()) == float(res["from_boxes"][0])
        del res
        fns = {k: wrap(f) for k, f in arms.items()}
        # the arms alternate window by window (order rotated) so that drift of clocks and neighbours hits all of them
        steps, n_win = max(args.steps, 20), 7
        times = {k: [] for k in fns}
        order = list(fns)
        for w in range(n_win):
            for k in order[w % len(order):] + order[:w % len(order)]:
                times[k].append(timed(fns[k], steps, args.warmup))
        ms = {k: float(np.median(v)) for k, v in times.items()}
        report("c3_sparse_backward", "EfficientDet-D0 512 B=128 C=81 training step from box lists: get_loss_from_boxes_and_grad "
               "against generate_targets_batch (one-hot / class ids) + get_loss_and_grad (gradients asserted bit-identical "
               "first) and get_loss_from_boxes alone; median of %d alternating windows of %d steps" % (n_win, steps), batch,
               ms["from_boxes"], n_anchor * (C * 8 + 32 + 8),
               dict(card, one_hot_targets_and_grad_ms=ms["one_hot"], class_id_targets_and_grad_ms=ms["class_id"],
                    from_boxes_forward_ms=ms["from_boxes_forward"], speedup_vs_one_hot=ms["one_hot"] / ms["from_boxes"],
                    speedup_vs_class_id=ms["class_id"] / ms["from_boxes"], window_ms={k: [round(t, 5) for t in v] for k, v in times.items()},
                    grads_bit_identical=True, forward_loss_bit_identical=fwd_bits, loss_rel_diff_vs_one_hot=loss_rel,
                    note="bytes: read logits + box outputs, write both gradients, write + read one int32 match per anchor"))
        del rel, cls
        torch.cuda.empty_cache()
    if want("c3_sparse_eval"):  # test_step of config 3 from box lists against the dense-target eval step
        card = _card()
        c = synth.EFFDET_CONFIGS["d0"]
        batch, C = 128, 81
        a = Anchors(c["min_level"], c["max_level"], c["image_size"], c["num_scales"], c["aspect_ratios"], c["anchor_scale"])
        shapes = [tuple(b.shape) for b in a.boxes]
        rel = [torch.randn((batch,) + s, device=dev, generator=g) * 0.25 for s in shapes]
        cls = [torch.randn((batch,) + s[:-1] + (C,), device=dev, generator=g) for s in shapes]
        n_anchor = sum(s[0] * s[1] * s[2] for s in shapes)
        rng = np.random.default_rng(20261018 + 3)
        boxes, classes, off = synth.gt_batch(rng, batch, (c["image_size"][1], c["image_size"][0]), max_boxes=100, order="yxyx")
        d_boxes, d_cls, d_off = (torch.from_numpy(boxes).to(dev), torch.from_numpy((classes + 1).astype(np.int32)).to(dev),
                                 torch.from_numpy(off).to(dev))
        targets = a.generate_targets_batch(d_boxes, d_cls, d_off, C)
        arms = {
            "from_boxes": lambda: a.eval_step_from_boxes(d_boxes, d_cls, d_off, rel, cls),
            "targets_and_eval": lambda: a.eval_step(*a.generate_targets_batch(d_boxes, d_cls, d_off, C), rel, cls),
            "eval_precomputed": lambda: a.eval_step(*targets, rel, cls),
        }
        # the match stage alone (the same kernel and launch as the first stage of eval_step_from_boxes): separates its time
        # from the stream's
        import ctypes
        from tfmv_b200 import _lib, _tensors as T
        lib = _lib.load()
        L = a._num_levels
        m_sums = torch.empty((2 * L + 1,), dtype=torch.float64, device=dev)
        m_ws = torch.empty((lib.b200_effdet_loss_from_boxes_workspace_bytes(L, a._hw, a._A, batch),), dtype=torch.uint8, device=dev)
        arms["match_stage"] = lambda: lib.b200_effdet_loss_from_boxes_match(
            L, a._hw, a._A, T.ptr(a._dev_table()), batch, T.ptr(d_boxes), T.ptr(d_off), d_boxes.shape[0], ctypes.c_float(0.5),
            T.ptr(m_sums), T.ptr(m_ws), m_ws.numel(), T.stream_ptr())
        got = a.eval_step_from_boxes(d_boxes, d_cls, d_off, rel, cls, with_indices=True, return_parts=True)
        ref = a.eval_step(*targets, rel, cls, with_indices=True, return_parts=True)
        bits = lambda x, y: x.shape == y.shape and torch.equal(x.reshape(-1).view(torch.uint8), y.reshape(-1).view(torch.uint8))
        cnt = ref[2]["count"]
        rows = torch.arange(ref[2]["boxes"].shape[1], device=dev)[None, :] < cnt[:, None]   # rows past count are not written
        assert bits(got[0], ref[0]) and bits(got[3], ref[3]) and bits(got[4], ref[4]), "loss terms differ"
        assert all(bits(x, y) for x, y in zip(got[1], ref[1])), "decoded boxes differ"
        assert bits(got[2]["count"], cnt) and all(bits(got[2][k][rows], ref[2][k][rows]) for k in ref[2] if k != "count"), \
            "NMS outputs differ"
        del got, ref
        fns = {k: wrap(f) for k, f in arms.items()}
        # the arms alternate window by window (order rotated) so that drift of clocks and neighbours hits all of them
        steps, n_win = max(args.steps, 20), 7
        times = {k: [] for k in fns}
        order = list(fns)
        for w in range(n_win):
            for k in order[w % len(order):] + order[:w % len(order)]:
                times[k].append(timed(fns[k], steps, args.warmup))
        ms = {k: float(np.median(v)) for k, v in times.items()}
        report("c3_sparse_eval", "EfficientDet-D0 512 B=128 C=81 eval step from box lists: eval_step_from_boxes against "
               "generate_targets_batch + eval_step and against eval_step on precomputed targets (loss terms, decoded boxes and "
               "NMS outputs asserted bit-identical first); median of %d alternating windows of %d steps" % (n_win, steps), batch,
               ms["from_boxes"], n_anchor * (C * 4 + 16 + 16 + 8),
               dict(card, targets_and_eval_ms=ms["targets_and_eval"], eval_precomputed_targets_ms=ms["eval_precomputed"],
                    match_stage_ms=ms["match_stage"], stream_reduce_nms_ms=ms["from_boxes"] - ms["match_stage"],
                    speedup_vs_targets_and_eval=ms["targets_and_eval"] / ms["from_boxes"],
                    speedup_vs_precomputed=ms["eval_precomputed"] / ms["from_boxes"],
                    window_ms={k: [round(t, 5) for t in v] for k, v in times.items()}, outputs_bit_identical=True,
                    note="bytes: read logits + box outputs, write the decoded boxes, write + read one int32 match per anchor"))
        del rel, cls, targets, m_ws
        torch.cuda.empty_cache()
    if want("c5_sparse_eval"):  # test_step of config 5 from box lists against the dense targets + host-offset mAP
        from tfmv_b200.ai_models.utils.mAP import Get_mAP_batch
        card = _card()
        batch, image, C = 64, 608, 80
        heads = yolo_heads(batch, image)
        rng = np.random.default_rng(20261018 + 5)
        boxes, classes, off = synth.gt_batch(rng, batch, (image, image), max_boxes=100)
        boxes_d, classes_d, off_d = (torch.from_numpy(x).to(dev) for x in (boxes, classes, off))
        gen = DataGenerator(C, anc, (image, image))
        wh = (image, image)

        def dense():
            y = gen.GetTargetsBatch(classes_d, boxes_d, off_d)
            loss, r = tyu.LossAndNMSBoxesBatch(y, heads, wh, anc, C, 0.5, "ciou", nms_iou_type="diou")
            # GetGroudTruth per level (batch-major) regrouped per image, the NMS rows compacted: host offsets for Get_mAP_batch
            per_level = [tyu.GetGroudTruth(t) for t in y]
            n_l = [(t[..., 4] != 0).reshape(batch, -1).sum(1).cpu().numpy() for t in y]
            parts = [torch.split(g, n.tolist()) for g, n in zip(per_level, n_l)]
            gt = torch.cat([p[b] for b in range(batch) for p in parts])
            go = np.concatenate([[0], np.cumsum(sum(n_l))]).astype(np.int32)
            cnt = r["count"].cpu().numpy()
            pred = torch.cat([torch.cat([r["boxes"][b, :n], r["classes_id"][b, :n, None].float(), r["scores"][b, :n, None]], 1)
                              for b, n in enumerate(cnt)])
            return loss, r, Get_mAP_batch(gt, go, pred, np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32), C)

        arms = {
            "from_boxes": lambda: tyu.EvalStepFromBoxes(classes_d, boxes_d, off_d, heads, wh, anc, C, 0.5, "ciou", nms_iou_type="diou"),
            "dense": dense,
        }
        got, ref = arms["from_boxes"](), arms["dense"]()
        loss_rel = abs(float(got[0]) - float(ref[0])) / abs(float(ref[0]))   # dense GetLoss sums in another order
        assert loss_rel < 1e-4, "losses differ"
        assert got[2].cpu().numpy().tobytes() == ref[2].cpu().numpy().tobytes(), "mAP differs"
        assert torch.equal(got[1]["count"], ref[1]["count"])
        m_ap = float(got[2].mean())
        fns = {"from_boxes": wrap(arms["from_boxes"]), "dense": arms["dense"]}   # the dense arm synchronises: no graph
        steps, n_win = max(args.steps, 20), 7
        times = {k: [] for k in fns}
        order = list(fns)
        for w in range(n_win):
            for k in order[w % len(order):] + order[:w % len(order)]:
                times[k].append(timed(fns[k], steps, args.warmup))
        ms = {k: float(np.median(v)) for k, v in times.items()}
        report("c5_sparse_eval", "YOLOv4 608 B=64 eval step from box lists: EvalStepFromBoxes(ciou loss, diou NMS, mAP) against "
               "GetTargetsBatch + LossAndNMSBoxesBatch + GetGroudTruth + Get_mAP_batch (host offsets; mAP asserted bit-identical "
               "and the loss within 1e-4 first); median of %d alternating windows of %d steps" % (n_win, steps), batch, ms["from_boxes"],
               7732620, dict(card, dense_targets_and_host_map_ms=ms["dense"], speedup_vs_dense=ms["dense"] / ms["from_boxes"],
                             mean_map=m_ap, window_ms={k: [round(t, 5) for t in v] for k, v in times.items()},
                             map_bit_identical=True, loss_rel_diff=loss_rel, note="bytes: read y_pred once (dense equivalent)"))
    if want("n4_letterbox"):  # SURVEY 8f N4: the serving view's image pre-processing, one image per call (latency)
        from tfmv_b200.views.object_detection import prepare_image
        for (h, w) in ((1080, 1920), (3024, 4032), (480, 640), (240, 320)):
            img = torch.randint(0, 256, (h, w, 3), device=dev, dtype=torch.uint8, generator=g)
            fn = wrap(lambda: prepare_image(img, (416, 416))[0])
            ms = timed(fn, max(args.steps, 50), 10)
            report("n4_letterbox_%dx%d" % (w, h), "prepare_image: INTER_AREA letterbox to 416x416 + BGR->RGB + /255 (device-resident "
                   "uint8 frame; L2-resident after the first pass)", 1, ms, h * w * 3 + 416 * 416 * 3 * 4, {"latency_us": ms * 1e3})
    if want("n4_letterbox_batch") or want("n4_serving_chain"):
        from tfmv_b200.views.object_detection import prepare_image, prepare_images
        card = _card()
        mix_sizes = ((480, 640), (1080, 1920), (3024, 4032))
        frames_mix = [torch.randint(0, 256, mix_sizes[i % 3] + (3,), device=dev, dtype=torch.uint8, generator=g) for i in range(64)]
    if want("n4_letterbox_batch"):  # SURVEY 8f N4 batched: N frames per call against one call per frame
        cases = [("1920x1080_n%d" % n, [torch.randint(0, 256, (1080, 1920, 3), device=dev, dtype=torch.uint8, generator=g)
                                        for _ in range(n)]) for n in (1, 8, 64)] + [("mix_n64", frames_mix)]
        for tag, frames in cases:
            n = len(frames)
            src = sum(f.numel() for f in frames)
            steps = max(args.steps, 50)
            ms_loop = timed(wrap(lambda: [prepare_image(f, (416, 416))[0] for f in frames]), steps, args.warmup)
            ms = timed(wrap(lambda: prepare_images(frames, (416, 416))[0]), steps, args.warmup)
            report("n4_letterbox_batch_" + tag, "prepare_images (one launch) vs a loop of prepare_image, %d device-resident frames "
                   "to 416x416 + BGR->RGB + /255 (source %.0f MB: %s)" % (n, src / 1e6, "L2-resident" if src < 100e6 else
                                                                          "exceeds the 126 MB L2"), n, ms,
                   src / n + 416 * 416 * 3 * 4,
                   dict(card, us_per_frame=ms * 1e3 / n, frames_per_s=n / ms * 1e3, l2_resident=src < 100e6,
                        per_frame_loop_us_per_frame=ms_loop * 1e3 / n, per_frame_loop_frames_per_s=n / ms_loop * 1e3,
                        speedup_vs_loop=ms_loop / ms))
    if want("n4_serving_chain"):  # decoded frames -> network input ... NMS output -> pixel boxes, backbone not timed
        from tfmv_b200.ai_models.utils import tf_yolo_utils as tyu
        from tfmv_b200.views.object_detection import restore_predictions, restore_predictions_batch
        frames = frames_mix
        n = len(frames)
        base = synth.yolo_heads_trained_like(np.random.default_rng(20261018 + 4), 16, 416)
        heads = [torch.from_numpy(np.tile(h, (n // 16, 1, 1, 1))).to(dev) for h in base]   # the backbone's output, fixed

        def batched():
            _, _, _, geometry = prepare_images(frames, (416, 416))
            nms = tyu.GetNMSBoxesBatch(*heads, anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou")
            return restore_predictions_batch(nms, (416, 416), geometry)

        def per_frame():  # today's single-image calls; GetNMSBoxes and restore_predictions read counts on the host
            out = []
            for i, f in enumerate(frames):
                _, padding, old = prepare_image(f, (416, 416))
                y = tyu.GetNMSBoxes(*[h[i:i + 1] for h in heads], anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou")
                out.append(restore_predictions(*y, np.int32([416, 416]), padding, old))
            return out
        ms = timed(wrap(batched), args.steps, args.warmup)
        ms_loop = timed(per_frame, args.steps, args.warmup)
        kept = int(batched()["count"].sum().item())
        report("n4_serving_chain_mix_n64", "prepare_images -> GetNMSBoxesBatch -> restore_predictions_batch on 64 device frames "
               "(640x480 / 1920x1080 / 4032x3024 mix, source %.0f MB, exceeds the 126 MB L2) against a per-frame loop of prepare_image -> GetNMSBoxes -> "
               "restore_predictions (always launch by launch: it syncs on the counts); trained-like heads stand in for the "
               "backbone, outside the timed region" % (sum(f.numel() for f in frames) / 1e6), n, ms, sum(f.numel() for f in frames) / n + 416 * 416 * 3 * 4,
               dict(card, us_per_frame=ms * 1e3 / n, frames_per_s=n / ms * 1e3, kept_boxes_total=kept,
                    per_frame_loop_us_per_frame=ms_loop * 1e3 / n, per_frame_loop_frames_per_s=n / ms_loop * 1e3,
                    speedup_vs_loop=ms_loop / ms))
    for name, cfgname, batch, with_loss in (("c3_d0_b128", "d0", 128, True), ("c4_d7_b16", "d7", 16, False)):
        if not want(name):
            continue
        c = synth.EFFDET_CONFIGS[cfgname]
        a = Anchors(c["min_level"], c["max_level"], c["image_size"], c["num_scales"], c["aspect_ratios"], c["anchor_scale"])
        shapes = [tuple(b.shape) for b in a.boxes]
        rel = [torch.randn((batch,) + s, device=dev, generator=g) * 0.25 for s in shapes]
        cls = [torch.randn((batch,) + s[:-1] + (81,), device=dev, generator=g) for s in shapes]
        n_anchor = sum(s[0] * s[1] * s[2] for s in shapes)
        if with_loss:
            rng = np.random.default_rng(20261018 + 3)
            boxes, classes, off = synth.gt_batch(rng, batch, (c["image_size"][1], c["image_size"][0]), max_boxes=100, order="yxyx")
            d_boxes, d_cls, d_off = (torch.from_numpy(boxes).to(dev), torch.from_numpy((classes + 1).astype(np.int32)).to(dev),
                                     torch.from_numpy(off).to(dev))
            tb, tc, tm = a.generate_targets_batch(d_boxes, d_cls, d_off, 81)
            ms_t = timed(wrap(lambda: a.generate_targets_batch(d_boxes, d_cls, d_off, 81)), args.steps, args.warmup)

            def step():
                loss = get_loss(tb, tc, tm, rel, cls)
                dec = a.convert_outputs_boxes(rel)
                return loss, a.convert_outputs_batch(dec, cls)
            ms = timed(wrap(step), args.steps, args.warmup)
            bpi = n_anchor * (81 * 4 * 2 + 16 * 2 + 1 + 16)
            ms_loss = timed(wrap(lambda: get_loss(tb, tc, tm, rel, cls)), args.steps, args.warmup)
            # sparse-target mode (SURVEY 8f N3): class ids instead of one-hot rows
            ib, ic, im = a.generate_targets_batch(d_boxes, d_cls, d_off, 81, class_index=True)
            ms_t_idx = timed(wrap(lambda: a.generate_targets_batch(d_boxes, d_cls, d_off, 81, class_index=True)), args.steps, args.warmup)
            ms_loss_idx = timed(wrap(lambda: get_loss(ib, ic, im, rel, cls)), args.steps, args.warmup)
            from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss_and_grad
            ms_bwd = timed(wrap(lambda: get_loss_and_grad(tb, tc, tm, rel, cls)), args.steps, args.warmup)
            loss_rel = abs(float(get_loss(ib, ic, im, rel, cls)) - float(get_loss(tb, tc, tm, rel, cls))) / abs(float(get_loss(tb, tc, tm, rel, cls)))
            ms_dec = timed(wrap(lambda: a.convert_outputs_boxes(rel)), args.steps, args.warmup)
            dec = a.convert_outputs_boxes(rel)
            ms_post = timed(wrap(lambda: a.convert_outputs_batch(dec, cls)), args.steps, args.warmup)
            report(name, "EfficientDet-D0 512 B=128: focal+box loss + decode + post-process (NMS diou, cap 200)", batch, ms, bpi,
                   {"phase_ms": {"loss": ms_loss, "decode": ms_dec, "postprocess": ms_post, "generate_targets": ms_t,
                                 "loss_and_grad": ms_bwd},
                    "sparse_target_mode": {"generate_targets_ms": ms_t_idx, "loss_ms": ms_loss_idx, "loss_rel_diff": loss_rel,
                                           "loss_gbps": n_anchor * (81 * 4 + 37) * batch / ms_loss_idx / 1e6},
                    "loss_gbps": n_anchor * (81 * 8 + 33) * batch / ms_loss / 1e6,
                    "postprocess_gbps": n_anchor * (81 * 4) * batch / ms_post / 1e6})
        else:
            def step():
                dec = a.convert_outputs_boxes(rel)
                return a.convert_outputs_batch(dec, cls)
            ms = timed(wrap(step), args.steps, args.warmup)
            bpi = n_anchor * (81 * 4 + 16 + 16)
            ms_dec = timed(wrap(lambda: a.convert_outputs_boxes(rel)), args.steps, args.warmup)
            dec = a.convert_outputs_boxes(rel)
            ms_post = timed(wrap(lambda: a.convert_outputs_batch(dec, cls)), args.steps, args.warmup)
            report(name, "EfficientDet-D7 1536 B=16: decode + post-process (NMS diou, cap 200, ~436k candidates/image)", batch, ms, bpi,
                   {"phase_ms": {"decode": ms_dec, "postprocess": ms_post},
                    "postprocess_gbps": n_anchor * (81 * 4) * batch / ms_post / 1e6})
        del rel, cls
        torch.cuda.empty_cache()

    if any(want(n) for n in ("c1_half", "c3_half_post", "c4_half")):
        _half_heads(args, dev, g, anc, tyu, Anchors, synth, report, wrap, want)
    if want("c2_half_train"):
        _half_train(args, dev, g, anc, tyu, DataGenerator, synth, report, wrap)
    if want("c3_half_train"):
        _effdet_half_train(args, dev, g, Anchors, synth, report, wrap)


def _half_heads(args, dev, g, anc, tyu, Anchors, synth, report, wrap, want):
    """Post-processing from bf16 / fp16 heads read in place, against fp32 heads holding the same values and against
    "bf16 cast then fp32" (what a mixed-precision user gets from an fp32-only library: a cast pass and an fp32 copy).
    The values are bf16 values that fp16 also holds exactly, so the four arms must give the same bits; that is asserted
    before anything is timed.  The arms alternate window by window (order rotated)."""
    import torch
    card = _card()

    def values(shape, scale=1.0):
        x = (torch.randn(shape, device=dev, generator=g) * scale).to(torch.bfloat16).float()
        x[x.abs() < 1e-4] = 0.0   # below fp16's normal range a bf16 value may not be exact in fp16
        return x

    def run(name, what, batch, fams, call, bytes_f32, bytes_half, same):
        """fams: the fp32 head families; call(families) runs the post-processing."""
        arms = {
            "fp32": [list(f) for f in fams],
            "bf16": [[t.to(torch.bfloat16) for t in f] for f in fams],
            "fp16": [[t.to(torch.float16) for t in f] for f in fams],
        }
        assert all(torch.equal(a.float(), b) for k in ("bf16", "fp16") for fa, fb in zip(arms[k], arms["fp32"]) for a, b in zip(fa, fb))
        fns = {k: (lambda v=v: call(v)) for k, v in arms.items()}
        fns["bf16_cast_then_fp32"] = lambda: call([[t.float() for t in f] for f in arms["bf16"]])
        ref = fns["fp32"]()
        for k in ("bf16", "fp16", "bf16_cast_then_fp32"):
            same(fns[k](), ref)
        del ref
        fns = {k: wrap(f) for k, f in fns.items()}
        steps, n_win = max(args.steps, 20), 5
        times = {k: [] for k in fns}
        order = list(fns)
        for w in range(n_win):
            for k in order[w % len(order):] + order[:w % len(order)]:
                times[k].append(timed(fns[k], steps, args.warmup))
        ms = {k: float(np.median(v)) for k, v in times.items()}
        report(name, what + "; arms bit-identical (asserted); median of %d alternating windows of %d steps" % (n_win, steps),
               batch, ms["bf16"], bytes_half,
               dict(card, arms_ms=ms, algorithmic_bytes_per_image_fp32=bytes_f32, algorithmic_bytes_per_image_half=bytes_half,
                    speedup_bf16_vs_cast_then_fp32=ms["bf16_cast_then_fp32"] / ms["bf16"],
                    speedup_bf16_vs_fp32=ms["fp32"] / ms["bf16"], speedup_fp16_vs_fp32=ms["fp32"] / ms["fp16"],
                    window_ms={k: [round(t, 5) for t in v] for k, v in times.items()}, outputs_bit_identical=True))

    def same_rows(a, b):
        assert torch.equal(a["count"], b["count"])
        cnt = a["count"].cpu().tolist()
        for k in a:
            if k != "count":
                for i, n in enumerate(cnt):
                    x, y = a[k][i, :n], b[k][i, :n]
                    if x.dtype == torch.float32:
                        x, y = x.view(torch.int32), y.view(torch.int32)
                    assert torch.equal(x, y), "%s differs between arms" % k

    if want("c1_half"):
        rec = sum(s * s * 3 for s in synth.yolo_grids(416))
        for batch in (1, 256):
            heads = [values((batch, s, s, 255), 2.0) for s in synth.yolo_grids(416)]
            call = lambda f: tyu.GetNMSBoxesBatch(*f[0], anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou", with_indices=True)
            run("c1_half_b%d" % batch, "YOLOv3 416 B=%d decode + per-class NMS ('iou') from half heads" % batch, batch, [heads], call,
                rec * 85 * 4, rec * 85 * 2, same_rows)
            del heads
    for name, cfg, batch in (("c3_half_post", "d0", 128), ("c4_half", "d7", 16)):
        if not want(name):
            continue
        c = synth.EFFDET_CONFIGS[cfg]
        a = Anchors(c["min_level"], c["max_level"], c["image_size"], c["num_scales"], c["aspect_ratios"], c["anchor_scale"])
        shapes = [tuple(b.shape) for b in a.boxes]
        n_anchor = sum(s[0] * s[1] * s[2] for s in shapes)
        rel = [values((batch,) + s, 0.25) for s in shapes]
        cls = [values((batch,) + s[:-1] + (81,)) for s in shapes]

        def call(f):
            return a.decode_and_postprocess(f[0], f[1])

        def same(x, y):
            for p, q in zip(x[0], y[0]):
                assert torch.equal(p.view(torch.int32), q.view(torch.int32)), "decoded boxes differ between arms"
            same_rows(x[1], y[1])
        run(name, "EfficientDet-%s B=%d decode_and_postprocess (NMS diou, cap 200) from half heads" % (cfg.upper(), batch), batch,
            [rel, cls], call, n_anchor * (81 * 4 + 16 + 16), n_anchor * (81 * 2 + 8 + 16), same)
        del rel, cls
        torch.cuda.empty_cache()


def _half_train(args, dev, g, anc, tyu, DataGenerator, synth, report, wrap):
    """The YOLO training step from box lists (GetLossFromBoxesAndGrad, 'ciou') on YOLOv4 608 B=64 heads in fp32, bf16
    and fp16, each writing its gradient in the heads' type (fp16 with a device loss scale), against "bf16 cast to fp32,
    fp32 call, gradients cast back to bf16" (what a mixed-precision user does with an fp32-only loss).  Beside them a
    dense GetLossAndGrad pair and a forward-only GetLossFromBoxes pair.  The heads hold bf16 values that fp16 also holds
    exactly, so every arm's loss and parts have the same bits and every gradient is round(g32 * s) of the fp32 arm's
    g32: asserted before anything is timed.  7 windows per arm, alternating, the order rotated window by window."""
    import torch
    card = _card()
    batch, image, C = 64, 608, 80
    grids = synth.yolo_grids(image)
    rec = sum(s * s * 3 for s in grids)
    f32 = []
    for s in grids:
        # N(0, 1) logits as the headline's heads (synth.yolo_heads), rounded to bf16
        x = torch.randn((batch, s, s, 3 * (5 + C)), device=dev, generator=g).to(torch.bfloat16).float()
        x[x.abs() < 1e-4] = 0.0   # below fp16's normal range a bf16 value may not be exact in fp16
        f32.append(x)
    heads = {"fp32": f32, "bf16": [t.to(torch.bfloat16) for t in f32], "fp16": [t.to(torch.float16) for t in f32]}
    assert all(torch.equal(a.float(), b) for k in ("bf16", "fp16") for a, b in zip(heads[k], f32))
    rng = np.random.default_rng(20261018 + 2)
    boxes, classes, off = (torch.from_numpy(a).to(dev) for a in synth.gt_batch(rng, batch, (image, image), max_boxes=100))
    y_true = DataGenerator(C, anc, (image, image)).GetTargetsBatch(classes, boxes, off)
    scale = torch.full((1,), 1024.0, dtype=torch.float32, device=dev)   # fp16 loss scale, read on the device
    box_args = (classes, boxes, off)
    kw = dict(iou_thresh=0.5, iou_type="ciou", return_parts=True)

    def train(h, **gkw):
        return tyu.GetLossFromBoxesAndGrad(*box_args, h, (image, image), anc, C, **kw, **gkw)

    def cast_then_fp32():
        loss, parts, grads = train([t.float() for t in heads["bf16"]])
        return loss, parts, [t.to(torch.bfloat16) for t in grads]

    def dense(h):
        loss, parts, grads = tyu._loss_call(y_true, h, (image, image), anc, 0.5, "ciou", 0, return_parts=True, with_grad=True,
                                            grad_dtype=h[0].dtype)
        return loss, parts, grads

    fns = {
        "fp32": lambda: train(heads["fp32"]),
        "bf16": lambda: train(heads["bf16"], grad_dtype=torch.bfloat16),
        "fp16_scaled": lambda: train(heads["fp16"], grad_dtype=torch.float16, grad_scale=scale),
        "bf16_cast_then_fp32": cast_then_fp32,
        "dense_fp32": lambda: dense(heads["fp32"]),
        "dense_bf16": lambda: dense(heads["bf16"]),
        "forward_fp32": lambda: tyu.GetLossFromBoxes(*box_args, heads["fp32"], (image, image), anc, C, **kw),
        "forward_bf16": lambda: tyu.GetLossFromBoxes(*box_args, heads["bf16"], (image, image), anc, C, **kw),
    }
    def same(a, b):   # bit equality, NaN positions equal (payloads not compared)
        a, b = a.float(), b.float()
        return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(torch.nan_to_num(a).view(torch.int32),
                                                                           torch.nan_to_num(b).view(torch.int32))

    def check(name, got, ref, s, dt):
        assert same(got[0], ref[0]) and same(got[1], ref[1]), "%s: loss bits differ from the fp32 arm" % name
        for a, b in zip(got[2], ref[2]):
            assert a.dtype == dt and same(a, (b if s is None else b * s).to(dt)), "%s: gradient bits differ" % name

    ref = fns["fp32"]()
    check("bf16", fns["bf16"](), ref, None, torch.bfloat16)
    check("fp16_scaled", fns["fp16_scaled"](), ref, 1024.0, torch.float16)
    check("bf16_cast_then_fp32", fns["bf16_cast_then_fp32"](), ref, None, torch.bfloat16)
    dref = fns["dense_fp32"]()
    check("dense_bf16", fns["dense_bf16"](), dref, None, torch.bfloat16)
    fref, fh = fns["forward_fp32"](), fns["forward_bf16"]()
    assert same(fh[0], fref[0]) and same(fh[1], fref[1]), "forward: loss bits differ between the arms"
    del ref, dref, fref, fh
    fns = {k: wrap(f) for k, f in fns.items()}
    steps, n_win = max(args.steps, 20), 7
    times = {k: [] for k in fns}
    order = list(fns)
    for w in range(n_win):
        for k in order[w % len(order):] + order[:w % len(order)]:
            times[k].append(timed(fns[k], steps, args.warmup))
    ms = {k: float(np.median(v)) for k, v in times.items()}
    elems = rec * (5 + C)
    report("c2_half_train", "YOLOv4 608 B=64 GetLossFromBoxesAndGrad('ciou') from bf16 / fp16 heads, gradient in the heads' type; "
           "arms bit-identical (asserted); median of %d alternating windows of %d steps" % (n_win, steps), batch, ms["bf16"],
           elems * 4,
           dict(card, arms_ms=ms,
                algorithmic_bytes_per_image_by_type={"fp32": elems * 8, "half": elems * 4,
                                             "what": "y_pred read (dense equivalent) + gradient written"},
                speedup_bf16_vs_cast_then_fp32=ms["bf16_cast_then_fp32"] / ms["bf16"],
                speedup_bf16_vs_fp32=ms["fp32"] / ms["bf16"], speedup_fp16_vs_fp32=ms["fp32"] / ms["fp16_scaled"],
                window_ms={k: [round(t, 5) for t in v] for k, v in times.items()}, outputs_bit_identical=True))



def _effdet_half_train(args, dev, g, Anchors, synth, report, wrap):
    """The EfficientDet training step from box lists (get_loss_from_boxes_and_grad) on D0 512 B=128 C=81 heads in fp32,
    bf16 and fp16, each writing its gradients in the heads' type (fp16 with a device loss scale of 1024), against "bf16
    cast to fp32, fp32 call, gradients cast back to bf16" (what a mixed-precision user does with an fp32-only loss).
    Beside them the dense class-id path (generate_targets_batch(class_index=True) + get_loss_and_grad) in bf16 and a
    forward-only get_loss_from_boxes pair.  Ground truth as in c3_sparse_backward; the heads hold N(0, 1) logits (box
    outputs N(0, 0.25)) rounded to bf16 values that fp16 also holds exactly, so every arm's loss has the same bits and
    every gradient is round(g32 * s) of the fp32 arm's g32: asserted before anything is timed.  7 windows per arm,
    alternating, the order rotated window by window."""
    import torch
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import (get_loss_and_grad, get_loss_from_boxes,
                                                                         get_loss_from_boxes_and_grad)
    card = _card()
    c = synth.EFFDET_CONFIGS["d0"]
    batch, C = 128, 81
    a = Anchors(c["min_level"], c["max_level"], c["image_size"], c["num_scales"], c["aspect_ratios"], c["anchor_scale"])
    shapes = [tuple(b.shape) for b in a.boxes]
    n_anchor = sum(s[0] * s[1] * s[2] for s in shapes)

    def values(shape, sd):
        x = (torch.randn(shape, device=dev, generator=g) * sd).to(torch.bfloat16).float()
        x[x.abs() < 1e-4] = 0.0   # below fp16's normal range a bf16 value may not be exact in fp16
        return x

    f32 = ([values((batch,) + s, 0.25) for s in shapes], [values((batch,) + s[:-1] + (C,), 1.0) for s in shapes])
    heads = {"fp32": f32, "bf16": tuple([t.to(torch.bfloat16) for t in f] for f in f32),
             "fp16": tuple([t.to(torch.float16) for t in f] for f in f32)}
    assert all(torch.equal(x.float(), y) for k in ("bf16", "fp16") for f, w in zip(heads[k], f32) for x, y in zip(f, w))
    rng = np.random.default_rng(20261018 + 3)
    boxes, classes, off = synth.gt_batch(rng, batch, (c["image_size"][1], c["image_size"][0]), max_boxes=100, order="yxyx")
    gt = (torch.from_numpy(boxes).to(dev), torch.from_numpy((classes + 1).astype(np.int32)).to(dev), torch.from_numpy(off).to(dev))
    scale = torch.full((1,), 1024.0, dtype=torch.float32, device=dev)   # fp16 loss scale, read on the device

    def train(h, **gkw):
        return get_loss_from_boxes_and_grad(a, *gt, *h, **gkw)

    def cast_then_fp32():
        loss, gb, gc = train(tuple([t.float() for t in f] for f in heads["bf16"]))
        return loss, tuple(t.to(torch.bfloat16) for t in gb), tuple(t.to(torch.bfloat16) for t in gc)

    def dense(h, **gkw):
        return get_loss_and_grad(*a.generate_targets_batch(*gt, C, class_index=True), *h, **gkw)

    fns = {
        "fp32": lambda: train(heads["fp32"]),
        "bf16": lambda: train(heads["bf16"], grad_dtype=torch.bfloat16),
        "fp16_scaled": lambda: train(heads["fp16"], grad_dtype=torch.float16, grad_scale=scale),
        "bf16_cast_then_fp32": cast_then_fp32,
        "dense_class_id_bf16": lambda: dense(heads["bf16"], grad_dtype=torch.bfloat16),
        "forward_fp32": lambda: get_loss_from_boxes(a, *gt, *heads["fp32"]),
        "forward_bf16": lambda: get_loss_from_boxes(a, *gt, *heads["bf16"]),
    }

    def same(x, y):   # bit equality, NaN positions equal (payloads not compared)
        x, y = x.float(), y.float()
        return torch.equal(torch.isnan(x), torch.isnan(y)) and torch.equal(torch.nan_to_num(x).view(torch.int32),
                                                                           torch.nan_to_num(y).view(torch.int32))

    def check(name, got, ref, s, dt):
        assert same(got[0], ref[0]), "%s: loss bits differ from the fp32 arm" % name
        for x, y in zip(got[1] + got[2], ref[1] + ref[2]):
            assert x.dtype == dt and same(x, (y if s is None else y * s).to(dt)), "%s: gradient bits differ" % name

    ref = fns["fp32"]()
    check("bf16", fns["bf16"](), ref, None, torch.bfloat16)
    check("fp16_scaled", fns["fp16_scaled"](), ref, 1024.0, torch.float16)
    check("bf16_cast_then_fp32", fns["bf16_cast_then_fp32"](), ref, None, torch.bfloat16)
    check("dense_class_id_bf16", fns["dense_class_id_bf16"](), dense(heads["fp32"]), None, torch.bfloat16)
    assert same(fns["forward_bf16"](), fns["forward_fp32"]()) and same(fns["forward_fp32"](), ref[0]), \
        "forward: loss bits differ between the arms"
    del ref
    fns = {k: wrap(f) for k, f in fns.items()}
    steps, n_win = max(args.steps, 20), 7
    times = {k: [] for k in fns}
    order = list(fns)
    for w in range(n_win):
        for k in order[w % len(order):] + order[:w % len(order)]:
            times[k].append(timed(fns[k], steps, args.warmup))
    ms = {k: float(np.median(v)) for k, v in times.items()}
    # per anchor: logits read + gradient written (C each), box outputs read + gradient written (4 each), one int32 match
    # written and read
    by_type = {"fp32": n_anchor * ((2 * C + 8) * 4 + 8), "half": n_anchor * ((2 * C + 8) * 2 + 8)}
    report("c3_half_train", "EfficientDet-D0 512 B=128 C=81 get_loss_from_boxes_and_grad from bf16 / fp16 heads, gradients in "
           "the heads' type; arms bit-identical (asserted); median of %d alternating windows of %d steps" % (n_win, steps), batch,
           ms["bf16"], by_type["half"],
           dict(card, arms_ms=ms, algorithmic_bytes_per_image_by_type=dict(by_type, what="heads read + gradients written + "
                                                                           "one int32 match written and read, per anchor"),
                speedup_bf16_vs_cast_then_fp32=ms["bf16_cast_then_fp32"] / ms["bf16"],
                speedup_bf16_vs_fp32=ms["fp32"] / ms["bf16"], speedup_fp16_vs_fp32=ms["fp32"] / ms["fp16_scaled"],
                speedup_forward_bf16_vs_fp32=ms["forward_fp32"] / ms["forward_bf16"],
                window_ms={k: [round(t, 5) for t in v] for k, v in times.items()}, outputs_bit_identical=True))


if __name__ == "__main__":
    main()
