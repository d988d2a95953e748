#!/usr/bin/env python
"""bench.py — throughput of the detection hot path on B200 (contract: DESIGN.md §5).

Headline workload = BASELINE.json configs[1]: YOLOv4 608x608, batch 64 per GPU, best-anchor target assignment
(GetTargets) + yolo_loss with the CIoU ignore mask (GetLoss), synthetic heads ~ N(0,1) and synthetic ground truth
(1..100 boxes/image).  One "step" = one pass of that path over one batch.  The same run also measures the other four
BASELINE configs (key `configs`): c1 YOLOv3 416 decode + per-class NMS (latency at batch 1, throughput at batch 256),
c3 EfficientDet-D0 batch 128 loss + decode + NMS, c4 EfficientDet-D7 batch 16 decode + NMS, and c5 YOLOv4 608 global
batch 512 loss + decode + NMS sharded by image over the N GPUs with the loss all-reduce (c5 runs at every N; c1/c3/c4
at N = 1), each with its roofline fractions and a parity check against the committed golden fixtures.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
  python bench.py --impl reference ...                      CPU restatement of the reference on the host cores
  python bench.py --only c3 --only-step --no-graph ...      one config, launch by launch (the ncu launch-list runs)
  python bench.py --dump-outputs DIR ...                    also write the headline's last timed step to DIR/<name>.npy

Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F = np.float32
SEED = 20261018
# algorithmic (dense) bytes per image, SURVEY.md §8(d)
BYTES = {
    "c1": 3619980 + 174000,      # heads read once + outputs (<= 500 x 87 floats)
    "c2": 23197860,              # write y_true + read y_true + read y_pred
    "c3": 49104 * (81 * 4 * 2 + 16 * 2 + 1 + 16),   # cls logits + one-hot + box out + box tgt + mask + decoded write
    "c4": 441936 * (81 * 4 + 16 + 16),              # cls logits + box out + decoded write
    "c5": 15639240,              # y_pred + y_true (+ outputs)
}
WHAT = {
    "c1": "YOLOv3 416x416, 80 classes: yolo_head decode + per-class NMS ('iou', 0.5/0.3/0.5, cap 500), N(0,1) heads",
    "c2": "YOLOv4 608x608 batch 64: GetTargets + GetLoss(ciou ignore mask)",
    "c3": "EfficientDet-D0 512x512 batch 128: focal + box loss, anchor decode, NMS ('diou', cap 200) over 49 104 anchors/image",
    "c4": "EfficientDet-D7 1536x1536 batch 16: anchor decode + NMS ('diou', cap 200) over 441 936 anchors/image",
    "c5": "YOLOv4 608x608 global batch 512 sharded by image: GetLoss(ciou) + decode + per-class NMS(diou) + loss all-reduce",
}


def auto_graph_steps(steps, want):
    if want > 0:
        return want if steps % want == 0 else 1
    return max(d for d in range(1, 33) if steps % d == 0)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch of the headline workload (0 = 64)")
    ap.add_argument("--repeats", type=int, default=1,
                    help="timed windows of --steps steps for the headline (median reported; the default times exactly --steps steps)")
    ap.add_argument("--config-repeats", type=int, default=9, help="timed windows per entry of `configs`")
    ap.add_argument("--only", default="", help="comma list out of c1,c2,c3,c4,c5: measure only these")
    ap.add_argument("--c5-global-batch", type=int, default=512, help="global batch of configs.c5 (512 = BASELINE configs[4])")
    ap.add_argument("--cpu-sample", type=int, default=0, help="images per CPU-baseline run (0 = 16)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl", "torch", "local", "peer-idle"],
                    help="transport of the loss all-reduce (N > 1); local = no exchange at all (diagnostic: isolates its cost)")
    ap.add_argument("--graph-steps", type=int, default=0, help="consecutive steps captured in one CUDA graph (0 = the largest divisor of --steps up to 32; 1 = one graph per step)")
    ap.add_argument("--fused-exchange", action="store_true", help="N > 1: keep the exchange inside the step's finalize kernel (one graph, no second stream; ~6 us per step slower)")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="issue every step launch by launch instead of replaying CUDA graphs")
    ap.add_argument("--only-step", action="store_true", help="skip phase timing / e2e / cpu baseline / parity (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the headline's last timed step returned (loss, sampled y_true) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or (args.only and "c2" not in args.only.split(","))):
        ap.error("--dump-outputs writes the outputs of the headline (c2) on the GPU")
    args.graph_steps = auto_graph_steps(args.steps, args.graph_steps)
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm_sorted = sorted(sm)
        top = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []   # the busiest samples are the ones under load
        return {"sm_mhz": statistics.median(top) if top else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


_REAL_STDOUT = None


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def spread(xs):
    xs = sorted(xs)
    n = len(xs)
    return {"n": n, "median": statistics.median(xs), "min": xs[0], "max": xs[-1], "p10": xs[int(0.1 * (n - 1))], "p90": xs[int(round(0.9 * (n - 1)))]}


# ------------------------------------------------------------------------------------------------
# CPU legs (the NumPy restatement of the reference; TensorFlow is not installable in this image)
_CPU_CACHE = {}


def cpu_inputs(image, seed, n_images):
    key = (image, seed, n_images)
    if key not in _CPU_CACHE:
        from tfmv_b200 import synth
        rng = np.random.default_rng(seed)
        _CPU_CACHE.clear()
        _CPU_CACHE[key] = (synth.yolo_anchors().astype(F), synth.yolo_heads(rng, n_images, image),
                           synth.gt_batch(rng, n_images, (image, image), max_boxes=100))
    return _CPU_CACHE[key]


def cpu_step_images(args_tuple):
    """Oracle on a few images: GetTargets + GetLoss.  Inputs are generated once per (worker, seed) and cached, so a timed
    call is compute only.  Returns (seconds of compute, loss)."""
    image, seed, n_images = args_tuple
    from oracle import yolo as oy
    anc, heads, (boxes, classes, off) = cpu_inputs(image, seed, n_images)
    t0 = time.perf_counter()
    per = [oy.get_targets(boxes[off[b]:off[b + 1]], classes[off[b]:off[b + 1]], anc, (image, image), 80) for b in range(n_images)]
    y_true = [np.stack([p[l] for p in per], 0) for l in range(3)]
    loss = oy.get_loss(y_true, heads, (image, image), anc, 0.5, "ciou")
    return time.perf_counter() - t0, float(loss)


def run_reference(args):
    """Reference arm: the oracle port on every host core.  Each worker holds its own fixed images (generated before the
    timed region); a step = every worker computing GetTargets + GetLoss on its images once; the step time is the slowest
    worker's COMPUTE time (input generation and result pickling are outside it)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    per_worker = 4
    image = 608
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        jobs = [(image, SEED + 2 + 7919 * w, per_worker) for w in range(cores)]
        warm = max(1, min(args.warmup, 3))
        for _ in range(warm):
            pool.map(cpu_step_images, jobs, chunksize=1)     # first call also generates and caches the worker's inputs
        steps = max(1, min(args.steps, 30))
        per_step = []
        t0 = time.perf_counter()
        for _ in range(steps):
            res = pool.map(cpu_step_images, jobs, chunksize=1)
            per_step.append(max(r[0] for r in res))
        wall = time.perf_counter() - t0
    imgs_per_step = cores * per_worker
    dt = sum(per_step)
    value = steps * imgs_per_step / dt
    line = {
        "impl": "reference", "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WHAT["c2"], "image": image, "per_gpu_batch": args.batch or 64,
                   "note": "NumPy restatement of the reference (TensorFlow not installable); each step = %d images, %d per host core; "
                           "timed: the slowest worker's compute per step (wall clock incl. pool overhead: %.1f ms/step)" % (
                               imgs_per_step, per_worker, 1e3 * wall / steps)},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": "%d steps x %d images (GetTargets+GetLoss ciou, 608x608), process pool over all host cores, compute only" % (steps, imgs_per_step)},
        "step_spread_ms": spread([1e3 * x for x in per_step]),
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
class Bench(object):
    """Shared state of the GPU arm: device, distributed group, exchange transport, timing helpers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import tfmv_b200  # noqa: F401
        from tfmv_b200 import _lib, runtime
        self.args = args
        self.torch, self.dist, self.runtime = torch, dist, runtime
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback in the product path")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.lib = _lib.load()
        self.tail_hooks = []
        self.exchange, self.exchange_kind = None, "none (single GPU)"
        if self.world > 1:
            kind = args.exchange
            if kind == "peer":
                ok = 1
                try:
                    self.exchange = runtime.PeerExchange()
                except Exception as e:  # noqa: BLE001  (e.g. CUDA IPC not permitted in this container)
                    self.log("peer mailboxes unavailable: %r" % (e,))
                    ok = 0
                t = torch.tensor([ok], device=self.dev)
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
                if int(t.item()) == 0:
                    self.exchange, kind = None, "nccl"
                else:
                    self.exchange_kind = "NVLink peer mailboxes, summed inside the loss-finalize kernel (no collective launch)"
            if kind == "nccl":
                self.exchange = runtime.NcclExchange()
                self.exchange_kind = "b200_allreduce_loss: ncclAllReduce issued by the library on the step's stream"
            if kind == "torch":
                self.exchange_kind = "torch.distributed all_reduce behind the step (outside the CUDA graph)"
            if kind == "local":
                self.exchange_kind = "NONE (diagnostic run: every rank keeps its local loss)"
            if kind == "peer-idle":   # diagnostic: peer mappings exist (CUDA IPC, peer access enabled) but the step never uses them
                self.idle_exchange = runtime.PeerExchange()
                self.exchange_kind = "NONE (diagnostic run: peer mailboxes mapped but unused)"
        self.peaks = {}
        try:
            self.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        self.peak = float(self.peaks.get("hbm_gbs", 6650.0))
        self.peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in self.peaks else "6650 GB/s (of fallback)"
        self.kernels = {}
        try:
            self.kernels = json.load(open(os.path.join(ROOT, "profiles", "r02_kernels.json")))
        except Exception:
            pass

    def log(self, msg):
        if self.args.verbose:
            sys.stderr.write("[rank %d] %s\n" % (self.rank, msg))
            sys.stderr.flush()

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def window(self, fn, steps, unit=1):
        """EXACTLY `steps` calls of fn bracketed by barrier + synchronize on both sides, CUDA events on the launching
        stream, max over ranks.  Returns milliseconds for the window; self.last holds what the last call of fn returned."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps // unit):   # one call of fn = `unit` steps (a CUDA graph of several consecutive steps)
            self.last = fn()
        for hook in self.tail_hooks:   # side streams whose work belongs to the timed region join before the stop event
            hook()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        self.barrier()
        return ms

    def timed(self, fn, steps, warmup, repeats=1, unit=1):
        """Warm-up, then `repeats` windows of `steps` steps.  Returns (median ms per step, per-window ms-per-step list)."""
        for _ in range((max(warmup, 3) + unit - 1) // unit):
            fn()
        per = [self.window(fn, steps, unit) / steps for _ in range(max(1, repeats))]
        return statistics.median(per), per

    def wrap(self, fn):
        return fn if self.args.no_graph else self.runtime.capture(fn)

    def table(self, cfg):
        """ncu launch-list summary of a config (profiles/r02_kernels.json): per-kernel device time and DRAM bytes."""
        return self.kernels.get(cfg) or {}

    def roofline(self, cfg, batch, ms_step, dominant_live=None):
        """Step-level fractions: dense-equivalent (SURVEY 8d bytes) and physical (ncu DRAM bytes of the step's kernels)."""
        dense = BYTES[cfg] * batch
        r = {"bound": "hbm", "peak": self.peak, "unit": "GB/s", "peak_source": self.peak_src,
             "algorithmic_bytes_per_step": dense, "step_gbps_dense": dense / ms_step / 1e6,
             "frac_dense": dense / ms_step / 1e6 / self.peak}
        t = self.table(cfg)
        if t.get("dram_bytes_per_step"):
            scale = batch / float(t.get("batch", batch))
            r["traffic_step"] = t["dram_bytes_per_step"] * scale
            r["frac_dram"] = t["dram_bytes_per_step"] * scale / ms_step / 1e6 / self.peak
            r["traffic_source"] = "profiles/r02_kernels.json (ncu dram__bytes_read.sum + dram__bytes_write.sum, sum over the step's launches)"
        if t.get("dominant"):
            d = t["dominant"]
            r["kernel"] = d["name"]
            r["kernel_share_ncu"] = d.get("share")
            r["traffic"] = d.get("dram_bytes")
        if dominant_live:
            r.update(dominant_live)
        else:
            r["achieved"] = r["step_gbps_dense"]
            r["frac"] = r["frac_dense"]
        return r


def to_dev(b, a, dtype=None):
    t = b.torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(b.dev)


# ------------------------------------------------------------------------------------------------
def headline_c2(b, line):
    """BASELINE configs[1]: the headline.  Fills `line` (value, ms_per_step, roofline, e2e, cpu_baseline, ...)."""
    args, torch, lib = b.args, b.torch, b.lib
    from tfmv_b200 import _tensors as T, synth
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.utils import tf_yolo_utils as tyu
    world, rank, dev = b.world, b.rank, b.dev
    batch, image = args.batch or 64, 608
    anc = synth.yolo_anchors().astype(F)
    # weak scaling: every rank gets the same AMOUNT of work — the ground truth of the per-GPU batch is the same draw on every
    # rank (box counts and geometry decide the loss kernels' work), the head tensors are rank-specific
    heads_h = synth.yolo_heads(np.random.default_rng(SEED + 2 + 1000 * rank), batch, image)
    boxes_h, classes_h, off_h = synth.gt_batch(np.random.default_rng(SEED + 2), batch, (image, image), max_boxes=100)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    heads_p = [pin(h) for h in heads_h]
    boxes_p, classes_p, off_p = pin(boxes_h), pin(classes_h), pin(off_h)
    heads_d = [h.to(dev, non_blocking=True) for h in heads_p]
    boxes_d, classes_d, off_d = boxes_p.to(dev), classes_p.to(dev), off_p.to(dev)
    gen = DataGenerator(80, anc, (image, image))
    A, RF = 3, 85
    y_true = tuple(torch.empty((batch, hw[0], hw[1], A, RF), dtype=torch.float32, device=dev) for hw in gen.layers_hw)
    hw = (ctypes.c_int32 * 6)(*[d for l in gen.layers_hw for d in l])
    ws = torch.empty((lib.b200_yolo_loss_workspace_bytes(hw, batch, A),), dtype=torch.uint8, device=dev)
    global_batch = batch * world
    in_graph = b.exchange is not None      # peer mailboxes / library NCCL: the exchange is part of the captured step

    def step(heads, boxes, classes, off):
        """One step on this rank's images: target assignment + loss, the 12 terms summed over the ranks."""
        gen.GetTargetsBatch(classes, boxes, off, out=y_true)
        if in_graph or world == 1 or args.exchange in ("local", "peer-idle"):
            return tyu._loss_call(y_true, heads, (image, image), anc, 0.5, "ciou", 0, batch_divisor=global_batch,
                                  workspace=ws, exchange=b.exchange)
        loss, parts = tyu._loss_call(y_true, heads, (image, image), anc, 0.5, "ciou", 0, batch_divisor=global_batch,
                                     return_parts=True, workspace=ws)
        return tyu.combine_loss_parts(parts)

    sampler = ClockSampler(b.local_rank)
    if rank == 0:
        sampler.start()
    raw = lambda: step(heads_d, boxes_d, classes_d, off_d)
    if world > 1:
        raw(); raw()   # communicator / mailbox warm-up outside the timed region, the same number of times on every rank
        b.barrier()
    peer = b.exchange is not None and hasattr(b.exchange, "mailboxes")
    overlapped = False
    unit = 1   # steps per call of dev_step
    if args.no_graph or (world > 1 and not in_graph and args.exchange not in ("local", "peer-idle")):
        dev_step = raw
    elif (world == 1 or (peer and not args.fused_exchange)) and args.graph_steps > 1 and args.steps % args.graph_steps == 0:
        # ONE CUDA graph holds `graph_steps` consecutive steps.  At N > 1 every step's graph section ends with this rank's 12
        # terms (already divided by the global batch); its exchange — one one-warp kernel over the NVLink mailboxes
        # (b200_allreduce_loss_peer: publish + collect) plus the 12-term fold — is a side branch of the graph that runs under
        # the kernels of the following step and joins at the end of the graph.  (Remote stores inside the step's last kernel
        # cost the step ~6 us — the kernel cannot retire before its peer writes are acknowledged; host-side event hand-offs
        # between per-step graphs cost ~4 us; a branch inside the graph costs neither.)
        unit = args.graph_steps
        overlapped = world > 1
        side = torch.cuda.Stream()

        keep = []   # every sub-step's result tensors stay referenced: the side branch still reads them when the next one starts

        def multi_step():
            main = torch.cuda.current_stream()
            loss = None
            del keep[:]
            for _ in range(unit):
                gen.GetTargetsBatch(classes_d, boxes_d, off_d, out=y_true)
                loss, parts = tyu._loss_call(y_true, heads_d, (image, image), anc, 0.5, "ciou", 0, batch_divisor=global_batch,
                                             workspace=ws, return_parts=True)
                keep.append((loss, parts))
                if world > 1:
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        b.exchange.allreduce_(parts)
                        b.lib.b200_yolo_loss_combine(parts.data_ptr(), loss.data_ptr(), side.cuda_stream)
            if world > 1:
                main.wait_stream(side)
            return loss
        dev_step = b.runtime.capture(multi_step)
    else:
        dev_step = b.runtime.capture(raw)
    ms_dev, windows = b.timed(dev_step, args.steps, args.warmup, args.repeats, unit=unit)
    last = b.last
    torch.cuda.synchronize()
    loss_val = float(last.item())
    del b.tail_hooks[:]
    clocks = sampler.stop() if rank == 0 else None
    b.log("headline timed")
    if args.dump_outputs and rank == 0:
        # the last timed step's results as a caller receives them: the loss and GetTargets' dense y_true.  The whole y_true
        # is 495 MB at batch 64, so it is sampled: every layer of a fixed, seeded draw of 8 images (62 MB)
        pick = np.sort(np.random.default_rng(SEED + 9).choice(batch, min(batch, 8), replace=False))
        idx = torch.from_numpy(pick).to(dev)
        outs = {"loss": last.cpu().numpy()}
        for l, t in enumerate(y_true):
            outs["y_true_%d" % l] = t.index_select(0, idx).cpu().numpy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        line["dump"] = {"dir": args.dump_outputs, "files": sorted(n + ".npy" for n in outs), "y_true_images": pick.tolist()}
    n_fill = sum(int(t.numel()) for t in y_true)
    line.update({
        "metric": "images/sec", "value": global_batch / (ms_dev / 1e3), "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "timing": {"windows": len(windows), "steps_per_window": args.steps, "ms_per_step": spread(windows),
                   "what": "each window = exactly --steps steps between barrier + synchronize, CUDA events, max over ranks; "
                           "value / ms_per_step are the median window"},
        "config": {"workload": WHAT["c2"], "image": image, "per_gpu_batch": batch, "global_batch": global_batch,
                   "classes": 80, "anchors_per_cell": 3, "gt_boxes_per_image": "U{1..100} (the same draw on every rank; heads differ per rank)",
                   "parallelism": "dp%d (images sharded; one 12-float all-reduce per step: %s)" % (world, b.exchange_kind),
                   "launch": "launch by launch" if dev_step is raw else (
                       ("one CUDA graph per %d consecutive steps" % unit if unit > 1 else "one CUDA graph per step") + (
                           "; the exchange of step i (a one-warp peer-mailbox kernel) is a side branch of the graph under step i+1" if overlapped
                           else ("; exchange inside the finalize kernel" if world > 1 else ""))),
                   "l2": "inputs larger than L2 (y_pred %.0f MB + y_true %.0f MB per step vs 126 MB L2)" % (n_fill * 4 / 1e6, n_fill * 4 / 1e6)},
        "loss": loss_val, "clocks": clocks,
        "gpu_launches": (5 + (2 if overlapped else 0)) * args.steps * len(windows),
        "gpu_launches_note": "5 kernels per step (fill, scatter, scan + GT prep, ignore-lean + object terms, finalize + exact ignore pass)" + (
            " + exchange and fold kernels on the side branch" if overlapped else ""),
    })
    if b.exchange is not None and hasattr(b.exchange, "status"):
        ep, err = b.exchange.status()
        line["config"]["exchange_status"] = {"exchanges": ep, "timeouts": err}
    if args.only_step:
        return
    # ---- the dominant kernel, timed alone with CUDA events (roofline.achieved / frac) ----
    st = T.stream_ptr()
    tp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in y_true])
    pp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in heads_d])
    anc_h = np.ascontiguousarray(anc.reshape(-1))
    img_h = np.array([image, image], dtype=F)
    parts_t = torch.empty((3, 4), dtype=torch.float32, device=dev)
    loss_t = torch.empty((), dtype=torch.float32, device=dev)

    def ph_fill():
        lib.b200_yolo_assign_targets(boxes_d.data_ptr(), classes_d.data_ptr(), off_d.data_ptr(), batch, 0,
                                     anc_h.ctypes.data_as(ctypes.c_void_p), A, img_h.ctypes.data_as(ctypes.c_void_p), 80, hw, tp, 1, st)

    def ph_scatter():
        lib.b200_yolo_assign_targets(boxes_d.data_ptr(), classes_d.data_ptr(), off_d.data_ptr(), batch, boxes_d.shape[0],
                                     anc_h.ctypes.data_as(ctypes.c_void_p), A, img_h.ctypes.data_as(ctypes.c_void_p), 80, hw, tp, 0, st)

    def ph_loss_stage(mask):
        def run():
            lib.b200_yolo_loss_stages(tp, pp, hw, batch, A, 80, anc_h.ctypes.data_as(ctypes.c_void_p), img_h.ctypes.data_as(ctypes.c_void_p),
                                      0.5, 2, 0, float(global_batch), parts_t.data_ptr(), loss_t.data_ptr(), ws.data_ptr(), ws.numel(), mask, st)
        return run
    ph_fill(); ph_scatter()
    n_rec = n_fill // RF
    phases = []
    for name, fn, nbytes in (
            ("fill_zero_multi_kernel", ph_fill, n_fill * 4),
            ("yolo_scatter_targets_kernel", ph_scatter, int(boxes_d.shape[0]) * (16 + 4 + 340)),
            ("yolo_loss_scan_kernel", ph_loss_stage(3), n_fill * 4),          # its last CTAs prepare the GT lists
            ("yolo_loss_ignore_lean_kernel", ph_loss_stage(4), n_fill * 4),   # stage 4 alone: + the exact pass as its own launch
            ("yolo_loss_finalize_kernel", ph_loss_stage(8), n_rec // 128 * 8)):
        if name == "yolo_loss_finalize_kernel" and world > 1:
            continue   # stage 8 alone would exchange on one rank only; its time is in the step
        ms, _ = b.timed(fn, args.steps, 3, 5)
        phases.append({"kernel": name, "ms": ms, "algorithmic_bytes": nbytes, "gbps": nbytes / ms / 1e6})
        if fn in (ph_fill, ph_scatter):
            ph_fill(); ph_scatter()  # restore valid targets (repeated scatters collide with themselves)
    tab = b.table("c2")
    dom_name = (tab.get("dominant") or {}).get("name")
    dom = next((p for p in phases if dom_name and p["kernel"] in dom_name), None) or max(phases, key=lambda p: p["ms"])
    live = {"kernel": dom["kernel"], "achieved": dom["gbps"], "frac": dom["gbps"] / b.peak, "kernel_ms_live": dom["ms"],
            "dominant_chosen_by": "ncu launch list (profiles/r02_kernels.json)" if dom_name else "live timing (no ncu table found)"}
    roof = b.roofline("c2", batch, ms_dev, live)
    kt = {k["name"].split("(")[0].replace("void ", "").split("<")[0]: k for k in tab.get("kernels", [])}
    if dom["kernel"] in kt and kt[dom["kernel"]].get("dram_bytes"):
        roof["traffic"] = kt[dom["kernel"]]["dram_bytes"]
        roof["achieved_dram_gbps"] = roof["traffic"] / dom["ms"] / 1e6
        roof["frac_kernel_dram"] = roof["achieved_dram_gbps"] / b.peak
    roof["phases"] = phases
    roof["note"] = ("achieved/frac: the dominant kernel's SURVEY 8(d) dense bytes over its live CUDA-event time; the loss kernels are "
                    "sector-sparse (obj*(...) kills the class channels of non-object cells), so dense-equivalent figures can exceed the "
                    "physical peak; frac_dram / traffic use ncu DRAM bytes.  Kernels below ~15 us are launch-interval-bound when timed "
                    "alone from Python; their device durations are in the ncu launch list")
    line["roofline"] = roof
    b.log("phases timed")
    # ---- API extensions measured beside the drop-in step (N == 1) ----
    if world == 1:
        from tfmv_b200.ai_models.datasets.coco_dataset import TargetBuffers
        tbuf = TargetBuffers()

        def pstep():
            yt = gen.GetTargetsBatch(classes_d, boxes_d, off_d, buffers=tbuf)
            return tyu._loss_call(yt, heads_d, (image, image), anc, 0.5, "ciou", 0, batch_divisor=global_batch, workspace=ws)
        pstep()
        pfn = b.wrap(pstep)
        ms_p, _ = b.timed(pfn, args.steps, 3, 5)
        ploss = float(pfn().item())
        line["persistent_targets"] = {"what": "GetTargetsBatch(buffers=TargetBuffers) + GetLoss: y_true reused, only the previous step's records re-zeroed",
                                      "value": global_batch / (ms_p / 1e3), "unit": "images/s", "ms_per_step": ms_p, "loss_equal": ploss == loss_val}
        ws_f = torch.empty((lib.b200_yolo_loss_from_boxes_workspace_bytes(hw, batch, A, int(boxes_d.shape[0])),), dtype=torch.uint8, device=dev)
        fstep = lambda: tyu.GetLossFromBoxes(classes_d, boxes_d, off_d, heads_d, (image, image), anc, 80, 0.5, "ciou",
                                             batch_divisor=global_batch, workspace=ws_f)
        ffn = b.wrap(fstep)
        ms_f, _ = b.timed(ffn, args.steps, 3, 5)
        floss = float(ffn().item())
        line["sparse_target_fusion"] = {"what": "GetLossFromBoxes: assignment + loss from the box lists, no dense y_true (API extension, SURVEY 8f N3)",
                                        "value": global_batch / (ms_f / 1e3), "unit": "images/s", "ms_per_step": ms_f,
                                        "loss_rel_diff": abs(floss - loss_val) / abs(loss_val)}
        # the reference's own execution model: DataGenerator.GetTargets runs in tf.data workers UNDER the previous train step
        # (datasets/coco_dataset.py:328).  Same calls, same fresh dense y_true per batch, two target buffers: GetTargets of batch
        # i + 1 on a side stream while GetLoss of batch i runs (the first GetTargets of every graph is not overlapped)
        gsteps = args.graph_steps if (not args.no_graph and args.steps % args.graph_steps == 0) else 1
        yt2 = [y_true, tuple(torch.empty_like(t) for t in y_true)]
        pside = torch.cuda.Stream()
        pkeep = []

        def pipelined():
            main = torch.cuda.current_stream()
            del pkeep[:]
            gen.GetTargetsBatch(classes_d, boxes_d, off_d, out=yt2[0])
            loss = None
            for i in range(gsteps):
                if i + 1 < gsteps:
                    pside.wait_stream(main)            # loss i - 1 has released the buffer that targets i + 1 overwrite
                    with torch.cuda.stream(pside):
                        gen.GetTargetsBatch(classes_d, boxes_d, off_d, out=yt2[(i + 1) % 2])
                loss = tyu._loss_call(yt2[i % 2], heads_d, (image, image), anc, 0.5, "ciou", 0, batch_divisor=global_batch, workspace=ws)
                pkeep.append(loss)
                main.wait_stream(pside)                # loss i + 1 needs targets i + 1
            return loss
        pipelined()
        torch.cuda.synchronize()
        plfn = b.wrap(pipelined)
        ms_pl, _ = b.timed(plfn, args.steps, 3, 5, unit=gsteps)
        plloss = float(plfn().item())
        line["pipelined_targets"] = {"what": "GetTargets of batch i+1 on a second stream under GetLoss of batch i (what tf.data does for the reference), "
                                             "two dense target buffers, %d consecutive steps per graph" % gsteps,
                                     "value": global_batch / (ms_pl / 1e3), "unit": "images/s", "ms_per_step": ms_pl, "loss_equal": plloss == loss_val}
    # ---- end to end through the public API with HOST buffers ----
    e2e_steps = max(3, min(args.steps, 10))
    call = lambda hp, bx, cl, of: float(step(hp, bx, cl, of).item())
    ms_e2e, _ = b.timed(lambda: call(heads_p, boxes_p, classes_p, off_p), e2e_steps, 2, 3)
    h2d = sum(h.numel() * 4 for h in heads_p) + boxes_p.numel() * 4 + classes_p.numel() * 4 + off_p.numel() * 4
    e2e = {"value": global_batch / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": int(h2d) * world,
           "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e,
           "what": "pinned host y_pred handed to GetLoss and read in place by the loss kernels over PCIe (they need ~6 % of it); boxes / "
                   "classes / offsets copied; loss scalar read back"}

    def copy_step():
        hd = [h.to(dev, non_blocking=True) for h in heads_p]
        return call(hd, boxes_p, classes_p, off_p)
    ms_cp, _ = b.timed(copy_step, e2e_steps, 2, 3)
    e2e["explicit_copy"] = {"value": global_batch / (ms_cp / 1e3), "unit": "images/s", "ms_per_step": ms_cp,
                            "what": "whole y_pred copied host->device from pinned memory first (495 MB per step per GPU, PCIe-bound)"}
    heads_pg = [torch.from_numpy(np.ascontiguousarray(h)) for h in heads_h]   # ordinary (pageable) host arrays

    def pageable_step():
        hd = [h.to(dev) for h in heads_pg]
        return call(hd, boxes_h, classes_h, off_h)
    ms_pg, _ = b.timed(pageable_step, max(2, e2e_steps // 2), 1, 2)
    e2e["pageable_host"] = {"value": global_batch / (ms_pg / 1e3), "unit": "images/s", "ms_per_step": ms_pg,
                            "what": "caller holds plain (pageable) NumPy arrays: staged copy of the whole y_pred, then the same call"}
    e2e["note"] = "the headline e2e needs caller-pinned memory; explicit_copy and pageable_host are what other callers get"
    line["e2e"] = e2e
    # ---- CPU baseline beside it (rank 0, N == 1): median of >= 5 runs after one warm-up ----
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = args.cpu_sample or 16
        cpu_step_images((image, SEED + 6, n))
        runs = [cpu_step_images((image, SEED + 6, n))[0] for _ in range(5)]
        med = statistics.median(runs)
        line["cpu_baseline"] = {"value": n / med, "unit": "images/s", "cores": 1, "kind": "port",
                                "sample": "%d images of the same workload (NumPy oracle GetTargets+GetLoss, single process), median of 5 runs "
                                          "after 1 warm-up, %.2f s per run (min %.2f, max %.2f)" % (n, med, min(runs), max(runs))}
    else:
        line["cpu_baseline"] = None


# ------------------------------------------------------------------------------------------------
def yolo_heads_dev(b, batch, image, gen):
    from tfmv_b200 import synth
    return [b.torch.randn((batch, s, s, 255), device=b.dev, generator=gen) for s in synth.yolo_grids(image)]


def config_c1(b):
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.utils import tf_yolo_utils as tyu
    torch, args = b.torch, b.args
    anc = synth.yolo_anchors().astype(F)
    g = torch.Generator(device=b.dev).manual_seed(SEED + 1)
    out = {"what": WHAT["c1"], "algorithmic_bytes_per_image": BYTES["c1"]}
    if not args.only_step:
        h1 = yolo_heads_dev(b, 1, 416, g)
        f1 = b.wrap(lambda: tyu.GetNMSBoxesBatch(*h1, anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou"))
        ms1, w1 = b.timed(f1, max(args.steps, 50), 10, args.config_repeats)
        out["batch1"] = {"latency_us": ms1 * 1e3, "images_per_s": 1e3 / ms1, "latency_us_spread": spread([x * 1e3 for x in w1]),
                         "note": "3.6 MB input: L2-resident, launch/latency-bound by construction (SURVEY 8d)"}
    B = 256
    hb = yolo_heads_dev(b, B, 416, g)
    fb = b.wrap(lambda: tyu.GetNMSBoxesBatch(*hb, anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou"))
    ms, w = b.timed(fb, args.steps, args.warmup, args.config_repeats)
    out.update({"batch": B, "value": B / ms * 1e3, "unit": "images/s", "ms_per_step": ms, "ms_per_step_spread": spread(w),
                "roofline": b.roofline("c1", B, ms), "gpu_launches_per_step": 3,
                "l2": "inputs larger than L2 (927 MB of heads per step)"})
    return out


def effdet_setup(b, name, batch, seed):
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.efficientnet.utils.anchors import Anchors
    torch = b.torch
    c = synth.EFFDET_CONFIGS[name]
    a = Anchors(c["min_level"], c["max_level"], c["image_size"], c["num_scales"], c["aspect_ratios"], c["anchor_scale"])
    g = torch.Generator(device=b.dev).manual_seed(seed)
    shapes = [tuple(x.shape) for x in a.boxes]
    rel = [torch.randn((batch,) + s, device=b.dev, generator=g) * 0.25 for s in shapes]
    cls = [torch.randn((batch,) + s[:-1] + (81,), device=b.dev, generator=g) for s in shapes]
    return c, a, rel, cls


def config_c3(b):
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.efficientnet.efficientdet_net_train import get_loss
    args, torch = b.args, b.torch
    B = 128
    c, a, rel, cls = effdet_setup(b, "d0", B, SEED + 3)
    rng = np.random.default_rng(SEED + 3)
    boxes, classes, off = synth.gt_batch(rng, B, (c["image_size"][1], c["image_size"][0]), max_boxes=100, order="yxyx")
    d_boxes, d_cls, d_off = to_dev(b, boxes), to_dev(b, (classes + 1).astype(np.int32)), to_dev(b, off)
    tb, tc, tm = a.generate_targets_batch(d_boxes, d_cls, d_off, 81)

    def step():   # efficientdet_net_train.py:135-169 test_step: loss, convert_outputs_boxes, convert_outputs_one per image
        if hasattr(a, "eval_step"):
            return a.eval_step(tb, tc, tm, rel, cls)
        loss = get_loss(tb, tc, tm, rel, cls)
        dec = a.convert_outputs_boxes(rel)
        return loss, a.convert_outputs_batch(dec, cls)
    ms, w = b.timed(b.wrap(step), args.steps, args.warmup, args.config_repeats)
    out = {"what": WHAT["c3"], "batch": B, "value": B / ms * 1e3, "unit": "images/s", "ms_per_step": ms, "ms_per_step_spread": spread(w),
           "algorithmic_bytes_per_image": BYTES["c3"], "roofline": b.roofline("c3", B, ms),
           "fused": bool(hasattr(a, "eval_step")), "l2": "inputs larger than L2 (2 x 2.04 GB class tensors per step)"}
    if not args.only_step:
        ph = {}
        ph["loss"], _ = b.timed(b.wrap(lambda: get_loss(tb, tc, tm, rel, cls)), args.steps, 3, 3)
        ph["decode"], _ = b.timed(b.wrap(lambda: a.convert_outputs_boxes(rel)), args.steps, 3, 3)
        dec = a.convert_outputs_boxes(rel)
        ph["postprocess"], _ = b.timed(b.wrap(lambda: a.convert_outputs_batch(dec, cls)), args.steps, 3, 3)
        ph["generate_targets (not part of the step)"], _ = b.timed(b.wrap(lambda: a.generate_targets_batch(d_boxes, d_cls, d_off, 81)), args.steps, 3, 3)
        out["phase_ms_separate_calls"] = ph
    return out


def config_c4(b):
    args = b.args
    B = 16
    c, a, rel, cls = effdet_setup(b, "d7", B, SEED + 4)

    def step():
        if hasattr(a, "decode_and_postprocess"):
            return a.decode_and_postprocess(rel, cls)
        dec = a.convert_outputs_boxes(rel)
        return a.convert_outputs_batch(dec, cls)
    ms, w = b.timed(b.wrap(step), args.steps, args.warmup, args.config_repeats)
    out = {"what": WHAT["c4"], "batch": B, "value": B / ms * 1e3, "unit": "images/s", "ms_per_step": ms, "ms_per_step_spread": spread(w),
           "algorithmic_bytes_per_image": BYTES["c4"], "roofline": b.roofline("c4", B, ms),
           "fused": bool(hasattr(a, "decode_and_postprocess")), "l2": "inputs larger than L2 (2.3 GB of class logits per step)"}
    if not args.only_step:
        ph = {}
        ph["decode"], _ = b.timed(b.wrap(lambda: a.convert_outputs_boxes(rel)), args.steps, 3, 3)
        dec = a.convert_outputs_boxes(rel)
        ph["postprocess"], _ = b.timed(b.wrap(lambda: a.convert_outputs_batch(dec, cls)), args.steps, 3, 3)
        out["phase_ms_separate_calls"] = ph
    return out


def config_c5(b):
    """BASELINE configs[4]: YOLOv4 608, GLOBAL batch 512 sharded by image over the ranks (strong scaling inside this entry):
    GetLoss(ciou) + decode + per-class NMS(diou) on the same y_pred, the 12 loss terms all-reduced."""
    from tfmv_b200 import synth
    from tfmv_b200.ai_models.datasets.coco_dataset import DataGenerator
    from tfmv_b200.ai_models.utils import tf_yolo_utils as tyu
    args, torch, world, rank = b.args, b.torch, b.world, b.rank
    G, image = args.c5_global_batch, 608
    lo, hi = tyu.shard_range(G, rank, world)
    B = hi - lo
    anc = synth.yolo_anchors().astype(F)
    g = torch.Generator(device=b.dev).manual_seed(SEED + 5 + 1000 * rank)
    heads = yolo_heads_dev(b, B, image, g)
    rng = np.random.default_rng(SEED + 5)
    boxes, classes, off = synth.gt_batch(rng, G, (image, image), max_boxes=100)
    sl = slice(off[lo], off[hi])
    gen = DataGenerator(80, anc, (image, image))
    y_true = gen.GetTargetsBatch(to_dev(b, classes[sl]), to_dev(b, boxes[sl]), to_dev(b, (off[lo:hi + 1] - off[lo]).astype(np.int32)))
    in_graph = b.exchange is not None
    fused = getattr(tyu, "LossAndNMSBoxesBatch", None)

    def step():
        if fused is not None:
            return fused(y_true, heads, (image, image), anc, 80, 0.5, "ciou", 0.5, 0.3, 0.5, "diou", global_batch=G, exchange=b.exchange)
        if in_graph or world == 1:
            loss = tyu._loss_call(y_true, heads, (image, image), anc, 0.5, "ciou", 0, batch_divisor=G, exchange=b.exchange)
        else:
            loss, parts = tyu._loss_call(y_true, heads, (image, image), anc, 0.5, "ciou", 0, batch_divisor=G, return_parts=True)
            loss = tyu.combine_loss_parts(parts)
        return loss, tyu.GetNMSBoxesBatch(*heads, anc, (image, image), 80, 0.5, 0.3, 0.5, "diou")
    if world > 1:
        step()
        b.barrier()
    # several consecutive steps per CUDA graph, as the headline: at N > 1 every step ends in an exchange that couples the
    # ranks, so the host-side launch jitter of ANY rank would otherwise be paid by all of them at every step
    unit = 1
    if args.no_graph or (world > 1 and not in_graph):
        fn = step
    else:
        unit = max(d for d in range(1, 6) if args.steps % d == 0)
        if unit > 1:
            def multi():
                out = None
                for _ in range(unit):
                    out = step()
                return out
            fn = b.runtime.capture(multi)
        else:
            fn = b.runtime.capture(step)
    ms, w = b.timed(fn, args.steps, args.warmup, args.config_repeats, unit=unit)
    loss = float(fn()[0].item())
    out = {"what": WHAT["c5"], "global_batch": G, "per_gpu_batch": B, "n_gpus": world, "value": G / ms * 1e3, "unit": "images/s",
           "ms_per_step": ms, "ms_per_step_spread": spread(w), "scaling": "strong (global batch fixed at %d)" % G, "loss": loss,
           "algorithmic_bytes_per_image": BYTES["c5"], "roofline": b.roofline("c5", B, ms), "fused": fused is not None,
           "exchange": b.exchange_kind, "launch": "launch by launch" if fn is step else "one CUDA graph per %d consecutive steps" % unit,
           "l2": "inputs larger than L2 (%.1f GB of heads + %.1f GB of targets per rank)" % (
               sum(h.numel() for h in heads) * 4 / 1e9, sum(t.numel() for t in y_true) * 4 / 1e9)}
    out["roofline"]["note"] = "fractions are per GPU: this rank's %d images over the step time" % B
    return out


# ------------------------------------------------------------------------------------------------
def run_b200(args):
    b = Bench(args)
    torch = b.torch
    only = [c for c in args.only.split(",") if c]
    want = lambda c: (not only) or (c in only)
    line = {}
    if want("c2"):
        headline_c2(b, line)
    torch.cuda.empty_cache()
    configs = {}
    plan = [("c5", config_c5)] + ([("c1", config_c1), ("c3", config_c3), ("c4", config_c4)] if b.world == 1 else [])
    for name, fn in plan:
        if not want(name):
            continue
        try:
            configs[name] = fn(b)
        except Exception as e:  # noqa: BLE001  (a failing extra config must not lose the headline line)
            import traceback
            configs[name] = {"error": repr(e), "trace": traceback.format_exc()[-1500:]}
            if b.world > 1:
                raise
        b.log("%s done" % name)
        torch.cuda.empty_cache()
    if want("c2") and "value" in line:
        configs["c2"] = {"what": WHAT["c2"], "batch": line["config"]["per_gpu_batch"], "value": line["value"], "unit": "images/s",
                         "ms_per_step": line["ms_per_step"], "algorithmic_bytes_per_image": BYTES["c2"],
                         "roofline": {k: v for k, v in (line.get("roofline") or b.roofline("c2", line["config"]["per_gpu_batch"], line["ms_per_step"])).items() if k != "phases"},
                         "note": "the headline of this line"}
    # ---- one-shot parity of every config's entry points against the committed golden fixtures ----
    if b.rank == 0 and not args.only_step:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            import parity
            res = parity.run_all(b.dev)
            for c, r in res.items():
                if c in configs:
                    configs[c]["parity"] = r
            line["parity"] = {"source": "tests/golden/parity.py: CUDA path vs tests/golden/{yolo_64,effdet_64}.npz", "all_ok": all(r.get("ok") for r in res.values())}
        except Exception as e:  # noqa: BLE001
            line["parity"] = {"error": repr(e)}
    line["configs"] = {k: configs[k] for k in sorted(configs)}
    if "metric" not in line:   # --only without c2: still one well-formed line
        first = next(iter(line["configs"].values()), {})
        line.update({"metric": "images/sec", "value": first.get("value"), "unit": "images/s", "n_gpus": b.world, "steps": args.steps,
                     "warmup": max(args.warmup, 3), "ms_per_step": first.get("ms_per_step"), "higher_is_better": True, "scaling": "weak",
                     "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": first.get("what"), "only": only}})
    if b.rank == 0:
        emit(line)
    if b.exchange is not None:
        b.barrier()
        b.exchange.close()
    if b.world > 1:
        b.dist.destroy_process_group()


def main():
    # stdout carries exactly ONE JSON line: whatever libraries print to file descriptor 1 (NCCL's version banner ...) goes to
    # stderr instead; the line itself is written to a private duplicate of the original stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
