"""GPU parity: the batched serving path (b200_letterbox_batch, b200_unletterbox_boxes_batch; image_helper.letterbox_batch,
object_detection.prepare_images / restore_predictions_batch) against the reference goldens, the oracle and the
single-image calls, slot by slot and bit for bit; the decoded frames -> pixel boxes chain eager and graph-captured."""
import ctypes
import hashlib
import os
import re
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
F = np.float32
CAP = 84  # LB_MAX_IMAGES in csrc/letterbox.cu: frames per launch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from letterbox_inputs import CASES, make_image  # noqa: E402

LB_GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_letterbox.npz"))
_sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _host(t):
    return None if t is None else t.cpu().numpy()


def test_letterbox_batch_reproduces_reference_goldens(lib, cuda):
    """Every golden case that shares a target size and background goes into one batch (1x1 to 4032x3024, bilinear
    fallback frames included); each slot must carry the reference's sha256 and padding."""
    from tfmv_b200.ai_models.utils import image_helper as ih
    groups = {}
    for i, (name, h, w, size, kind) in enumerate(CASES):
        bg = tuple(int(v) for v in LB_GOLD[name + "/bg"])
        groups.setdefault((tuple(size), bg), []).append(i)
    # at least one batch mixes shrinking frames with one that takes the bilinear fallback (416^2 on black:
    # 1920x1080, 4032x3024 and 320x240)
    assert any(len({CASES[i][0].startswith("small_") for i in v}) == 2 and len(v) >= 3 for v in groups.values())
    for (size, bg), idx in groups.items():
        frames = [make_image(i, CASES[i][1], CASES[i][2], CASES[i][4]) for i in idx]
        u8, f32, paddings, resized = ih.letterbox_batch(frames, size, bg, True, True)
        assert tuple(u8.shape) == (len(idx), size[1], size[0], 3) and tuple(f32.shape) == tuple(u8.shape)
        u8, f32 = _host(u8), _host(f32)
        for s, i in enumerate(idx):
            name = CASES[i][0]
            assert tuple(paddings[s]) == tuple(int(v) for v in LB_GOLD[name + "/padding"]), name
            assert _sha(u8[s]) == str(LB_GOLD[name + "/sha_u8"]), name
            assert _sha(f32[s][None]) == str(LB_GOLD[name + "/sha_f32"]), name


def _random_frames(rng, n, tw, th):
    """Sizes drawn like test_gpu_views::test_letterbox_random_sizes_match_oracle: generic, integral block / 2x2 / copy,
    scale 1 on one axis, smaller than the target (bilinear fallback)."""
    from oracle import letterbox as olb
    out = []
    it = 0
    while len(out) < n:
        h, w = int(rng.integers(th // 2, 3 * th)), int(rng.integers(tw // 2, 3 * tw))
        if it % 6 == 1:
            h, w = int(rng.integers(1, 2 * th)), int(rng.integers(1, tw + 1))
        if it % 5 == 0:
            k = int(rng.integers(1, 5)); h, w = th * k, tw * k
        if it % 7 == 0:
            h, w = th + int(rng.integers(0, 2)), tw * 2
        it += 1
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if it % 3 else (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
        if min(olb.proportional_size(w, h, tw, th)) >= 1:   # an empty resize is a refusal, tested below
            out.append(img)
    return out


@pytest.mark.parametrize("target,outputs", [((416, 256), "both"), ((608, 608), "u8"), ((416, 256), "f32"), ((608, 608), "both")])
def test_letterbox_batch_random_mixed_sizes_match_oracle_and_single(lib, cuda, target, outputs):
    import torch
    from oracle import letterbox as olb
    from tfmv_b200.ai_models.utils import image_helper as ih
    tw, th = target
    rng = np.random.default_rng(20261020 + tw + len(outputs))
    imgs = _random_frames(rng, 30, tw, th)
    bg = tuple(int(v) for v in rng.integers(0, 256, 3))
    # device, pinned (read in place) and pageable frames in one list
    frames = [torch.from_numpy(im).to(cuda) if i % 3 == 0 else (torch.from_numpy(im).pin_memory() if i % 3 == 1 else im)
              for i, im in enumerate(imgs)]
    want_u8, want_f32 = outputs in ("u8", "both"), outputs in ("f32", "both")
    u8, f32, paddings, resized = ih.letterbox_batch(frames, (tw, th), bg, want_u8, want_f32)
    assert (u8 is None) != want_u8 and (f32 is None) != want_f32
    assert paddings.dtype == np.int32 and paddings.shape == (30, 4) and resized.dtype == np.int32 and resized.shape == (30, 2)
    u8, f32 = _host(u8), _host(f32)
    modes = set()
    for s, img in enumerate(imgs):
        h, w = img.shape[:2]
        want, pad = olb.proportional_resize(img, (tw, th), bg_color=bg)
        rw, rh = olb.proportional_size(w, h, tw, th)
        modes.add("linear" if rw > w or rh > h else ("block" if w % rw == 0 and h % rh == 0 else "generic"))
        assert tuple(paddings[s]) == tuple(pad) and tuple(resized[s]) == (rw, rh), (s, h, w)
        one_u8, one_f32, one_pad, _ = ih.letterbox(img, (tw, th), bg, True, True)
        assert tuple(one_pad) == tuple(pad)
        if want_u8:
            assert np.array_equal(u8[s], want), (s, h, w)
            assert np.array_equal(u8[s], _host(one_u8))
        if want_f32:
            assert np.array_equal(f32[s], want[..., ::-1].astype(F) / 255), (s, h, w)
            assert np.array_equal(f32[s], _host(one_f32))
    assert modes == {"linear", "block", "generic"}


def test_letterbox_batch_chunking_and_stacked_input(lib, cuda):
    import torch
    from oracle import letterbox as olb
    from tfmv_b200.ai_models.utils import image_helper as ih
    rng = np.random.default_rng(20261021)
    bg = (17, 99, 201)
    # N == 1 is the single-image call
    img = rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    u8, f32, pad, rs = ih.letterbox_batch([img], (416, 416), bg, True, True)
    o8, o32, opad, ors = ih.letterbox(img, (416, 416), bg, True, True)
    assert np.array_equal(_host(u8)[0], _host(o8)) and np.array_equal(_host(f32)[0], _host(o32))
    assert tuple(pad[0]) == opad and tuple(rs[0]) == ors
    # exactly one launch's worth, and one frame more (a second launch); tiny frames of mixed sizes
    for n in (CAP, CAP + 1):
        imgs = []
        while len(imgs) < n:
            h, w = int(rng.integers(1, 40)), int(rng.integers(1, 40))
            if min(olb.proportional_size(w, h, 24, 16)) >= 1:
                imgs.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        frames = [torch.from_numpy(im).to(cuda) for im in imgs]
        u8, f32, pad, _ = ih.letterbox_batch(frames, (24, 16), bg, True, True)
        u8, f32 = _host(u8), _host(f32)
        for s, im in enumerate(imgs):
            want, wpad = olb.proportional_resize(im, (24, 16), bg_color=bg)
            assert np.array_equal(u8[s], want), (n, s, im.shape)
            assert np.array_equal(f32[s], want[..., ::-1].astype(F) / 255), (n, s)
            assert tuple(pad[s]) == wpad
    # a (N,H,W,3) tensor (frame i at base + i*H*W*3) equals the same frames as a list: device and pinned host
    stack = torch.from_numpy(rng.integers(0, 256, (CAP + 3, 45, 70, 3), dtype=np.uint8))
    ref_u8, ref_f32, ref_pad, ref_rs = ih.letterbox_batch([f for f in stack], (64, 48), bg, True, True)
    for src in (stack.to(cuda), stack.pin_memory(), stack.numpy()):
        u8, f32, pad, rs = ih.letterbox_batch(src, (64, 48), bg, True, True)
        assert torch.equal(u8, ref_u8) and torch.equal(f32, ref_f32)
        assert np.array_equal(pad, ref_pad) and np.array_equal(rs, ref_rs)
    want, _ = olb.proportional_resize(stack[CAP + 2].numpy(), (64, 48), bg_color=bg)
    assert np.array_equal(_host(ref_u8)[CAP + 2], want)


def _geometry_of(paddings, sizes):
    return np.concatenate([np.int32(paddings), np.int32(sizes)], 1)


def test_restore_predictions_batch_matches_oracle_and_single(lib, cuda):
    import torch
    from oracle import views as ov
    from tfmv_b200.views.object_detection import prepare_images, restore_predictions, restore_predictions_batch
    rng = np.random.default_rng(20261022)
    B, K, C = 16, 300, 80
    sizes = [(640, 480), (333, 777), (416, 416), (1920, 1080), (100, 80), (4032, 3024), (500, 2000), (1600, 900),
             (417, 416), (37, 91), (1280, 720), (800, 600), (1024, 1024), (720, 1280), (3000, 200), (64, 64)]
    frames = [torch.zeros((h, w, 3), dtype=torch.uint8, device=cuda) for (w, h) in sizes]
    imgs, paddings, olds, geometry = prepare_images(frames, (416, 416))
    assert tuple(imgs.shape) == (B, 416, 416, 3) and str(geometry.dtype) == "torch.int32" and geometry.is_cuda
    assert olds.dtype == np.int32 and olds.tolist() == [list(s) for s in sizes]
    assert np.array_equal(geometry.cpu().numpy(), _geometry_of(paddings, olds))
    counts = rng.integers(1, K, B).astype(np.int32)
    counts[3], counts[7], counts[11] = 0, K, K
    c = rng.uniform(-0.1, 1.1, (B, K, 2))
    wh = np.exp(rng.uniform(np.log(1e-3), np.log(0.8), (B, K, 2)))
    boxes = np.concatenate([c - wh / 2, c + wh / 2], 2).astype(F)
    boxes[:, ::50] = boxes[:, 1::50]
    for b, (w, h) in enumerate(sizes):   # a width right at the 2 px limit (on the original image)
        boxes[b, 5, 2] = boxes[b, 5, 0] + F(2.0 / w)
    nms = {"boxes": torch.from_numpy(boxes).to(cuda), "count": torch.from_numpy(counts).to(cuda),
           "classes_id": torch.from_numpy(rng.integers(0, C, (B, K)).astype(np.int32)).to(cuda),
           "scores": torch.from_numpy(rng.random((B, K)).astype(F)).to(cuda),
           "classes": torch.from_numpy(rng.random((B, K, C)).astype(F)).to(cuda),
           "confidence": torch.from_numpy(rng.random((B, K, 1)).astype(F)).to(cuda)}
    got = restore_predictions_batch(nms, (416, 416), geometry)
    assert tuple(got["boxes"].shape) == (B, K, 4) and str(got["boxes"].dtype) == "torch.int32"
    cnt = got["count"].cpu().numpy()
    keys = ("classes_id", "scores", "classes", "confidence")
    host = {k: nms[k].cpu().numpy() for k in keys}
    for b in range(B):
        n = int(counts[b])
        want = ov.restore_predictions(boxes[b, :n], *[host[k][b, :n] for k in keys], (416, 416), paddings[b], olds[b])
        one = restore_predictions(nms["boxes"][b, :n], *[nms[k][b, :n] for k in keys], np.int32([416, 416]), paddings[b], olds[b])
        k = int(cnt[b])
        assert k == want[0].shape[0], b
        rows = [got["boxes"][b, :k]] + [got[key][b, :k] for key in keys]
        for g, w, o in zip(rows, want, one):
            assert np.array_equal(g.cpu().numpy(), w), b
            assert torch.equal(g, o), b
    assert cnt[3] == 0 and 0 < cnt[7] < K and cnt.min() >= 0
    # without the optional classes the dict has no classes either
    del nms["classes"]
    assert "classes" not in restore_predictions_batch(nms, (416, 416), geometry)


def _standin_backbone(seed, A=3, C=80):
    """A fixed stand-in for the network: sample the 416^2 input on the three YOLOv3 grids (mean of 4 strided taps per
    cell) and apply a seeded per-cell 3 -> A*(5+C) affine map.  Elementwise only, so a frame gives the same heads
    alone or in a batch."""
    import torch
    g = torch.Generator().manual_seed(seed)
    R = A * (5 + C)
    Wm = torch.randn((3, R), generator=g) * 3.0
    bias = torch.randn((R,), generator=g) * 0.5
    params = {}

    def run(x):  # x (N,416,416,3)
        dev = x.device
        if dev not in params:
            params[dev] = (Wm.to(dev), bias.to(dev))
        w, b = params[dev]
        heads = []
        for s in (32, 16, 8):
            q = s // 4
            p = (x[:, q::s, q::s] + x[:, 3 * q::s, q::s] + x[:, q::s, 3 * q::s] + x[:, 3 * q::s, 3 * q::s]) * 0.25
            heads.append(p[..., 0:1] * w[0] + p[..., 1:2] * w[1] + p[..., 2:3] * w[2] + b)
        return [h.contiguous() for h in heads]
    return run


def _frames_mixed(rng, cuda, sizes):
    import torch
    out = []
    for (w, h) in sizes:
        y, x = np.mgrid[0:h, 0:w]
        cx, cy = rng.uniform(0, w), rng.uniform(0, h)
        blob = (np.hypot(x - cx, y - cy) < rng.uniform(0.1, 0.4) * min(w, h))[..., None]
        img = np.where(blob, rng.integers(0, 256, 3), rng.integers(0, 256, (h, w, 3))).astype(np.uint8)
        out.append(torch.from_numpy(img).to(cuda))
    return out


def test_serving_chain_batched_eager_and_graph_match_per_frame(lib, cuda):
    import torch
    from tfmv_b200 import runtime, synth
    from tfmv_b200.ai_models.utils.tf_yolo_utils import GetNMSBoxes, GetNMSBoxesBatch
    from tfmv_b200.views.object_detection import prepare_image, prepare_images, restore_predictions, restore_predictions_batch
    rng = np.random.default_rng(20261023)
    anc = synth.yolo_anchors().astype(F)
    net = _standin_backbone(7)
    sizes = [(640, 480), (1920, 1080), (333, 777), (320, 240), (4032, 3024), (416, 416), (1000, 700), (200, 150)]
    frames = _frames_mixed(rng, cuda, sizes)
    keys = ("classes_id", "scores", "classes", "confidence")

    def chain():
        imgs, _, _, geometry = prepare_images(frames, (416, 416))
        nms = GetNMSBoxesBatch(*net(imgs), anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou")
        return restore_predictions_batch(nms, (416, 416), geometry)

    def per_frame():
        res = []
        for f in frames:
            img, padding, old = prepare_image(f, (416, 416))
            y = GetNMSBoxes(*net(img), anc, (416, 416), 80, 0.5, 0.3, 0.5, "iou")
            res.append(restore_predictions(*y, np.int32([416, 416]), padding, old))
        return res

    def same(batched, singles):
        cnt = batched["count"].cpu().tolist()
        for b, one in enumerate(singles):
            k = cnt[b]
            assert k == one[0].shape[0], (b, k, one[0].shape[0])
            for g, o in zip([batched["boxes"][b, :k]] + [batched[key][b, :k] for key in keys], one):
                assert torch.equal(g, o), b
        return cnt

    eager = chain()
    cnt = same(eager, per_frame())
    assert sum(c > 0 for c in cnt) >= len(sizes) - 1 and max(cnt) > 3, cnt
    # the whole chain as one CUDA graph; refill the frame buffers in place, replay, compare with eager on the new content
    step = runtime.capture(chain)
    for f, new in zip(frames, _frames_mixed(rng, cuda, sizes)):
        f.copy_(new)
    replayed = step()
    torch.cuda.synchronize()
    fresh = chain()
    cnt2 = same(fresh, per_frame())
    assert cnt2 != cnt or any(not torch.equal(eager["boxes"][b, :k], fresh["boxes"][b, :k]) for b, k in enumerate(cnt2))
    assert torch.equal(replayed["count"], fresh["count"])
    for b, k in enumerate(cnt2):
        for key in ("boxes",) + keys:
            assert torch.equal(replayed[key][b, :k], fresh[key][b, :k]), (key, b)


def test_batch_refusals_name_the_frame_and_launch_nothing(lib, cuda):
    import torch
    from tfmv_b200.ai_models.utils import image_helper as ih
    from tfmv_b200.views.object_detection import prepare_images
    ok = torch.zeros((480, 640, 3), dtype=torch.uint8, device=cuda)
    with pytest.raises(ValueError, match=r"image 2: .*empty"):
        ih.letterbox_batch([ok, ok, np.zeros((2, 4000, 3), np.uint8), ok], (416, 416), (0, 0, 0), True, False)
    with pytest.raises(RuntimeError, match=r"image 0: 3-channel"):
        ih.letterbox_batch([np.zeros((50, 50, 4), np.uint8)] * 3, (416, 416), (0, 0, 0), True, False)
    with pytest.raises(ValueError, match="frame 2 has 4 channels"):
        ih.letterbox_batch([ok, ok, np.zeros((50, 50, 4), np.uint8)], (416, 416), (0, 0, 0), True, False)
    with pytest.raises(ValueError, match="frame 1"):
        ih.letterbox_batch([ok, np.zeros((50, 50, 3), np.float32)], (416, 416), (0, 0, 0), True, False)
    # the C ABI directly: an invalid frame leaves the outputs untouched (nothing launched)
    n = 3
    out = torch.full((n, 416, 416, 3), 77, dtype=torch.uint8, device=cuda)
    geo = torch.full((n, 6), -5, dtype=torch.int32, device=cuda)
    bg = (ctypes.c_uint8 * 3)(1, 2, 3)
    pad = (ctypes.c_int32 * (4 * n))()
    for bad_ptr, bad_hw, msg in ((ok.data_ptr(), (2, 4000), "image 1: .*empty"), (0, (480, 640), "image 1: null")):
        imgs = (ctypes.c_void_p * n)(ok.data_ptr(), bad_ptr, ok.data_ptr())
        hw = (ctypes.c_int32 * (2 * n))(480, 640, *bad_hw, 480, 640)
        assert lib.b200_letterbox_batch(n, imgs, hw, 3, 416, 416, bg, out.data_ptr(), None, pad, None, geo.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream) == -1
        assert re.search(msg, lib.b200_last_error().decode())
    torch.cuda.synchronize()
    assert int(out.min()) == 77 and int(out.max()) == 77 and int(geo.min()) == -5 and int(geo.max()) == -5
    # N == 0
    u8, f32, pads, rs = ih.letterbox_batch([], (416, 416), (0, 0, 0), True, True)
    assert tuple(u8.shape) == (0, 416, 416, 3) and tuple(f32.shape) == (0, 416, 416, 3) and pads.shape == (0, 4) and rs.shape == (0, 2)
    imgs, pads, olds, geometry = prepare_images([], (416, 416))
    assert tuple(imgs.shape) == (0, 416, 416, 3) and tuple(geometry.shape) == (0, 6) and olds.shape == (0, 2)
