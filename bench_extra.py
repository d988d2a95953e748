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


if __name__ == "__main__":
    main()
