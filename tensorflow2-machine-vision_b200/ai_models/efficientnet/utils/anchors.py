"""Drop-in for the reference's efficientnet/utils/anchors.py (Anchors :12-274).

Same constructor and method names / argument order / return arity; tensors are torch CUDA tensors (or anything
DLPack / array-like).  Anchor boxes are never read from memory by the kernels: they are rebuilt from a small
per-level table (row/column centres, half extents) computed here with the reference's own Python arithmetic.
"""
import ctypes
import math
from typing import List, Tuple, Union

import numpy as np
import torch

from .... import _lib, _tensors as T
from .get_feat_sizes import get_feat_sizes

EPSILON = 1e-8


def _range_f32(start, limit, delta):
  '''tf.range(start, limit, delta) on float32: ceil((limit-start)/delta) values, accumulated in fp32.'''
  start, limit, delta = np.float32(start), np.float32(limit), np.float32(delta)
  n = int(math.ceil(abs((float(limit) - float(start)) / float(delta))))
  out = np.empty((n,), dtype=np.float32)
  v = start
  for i in range(n):
    out[i] = v
    v = np.float32(v + delta)
  return out


class Anchors(object):
  '''Anchor generation, target assignment, decode and per-image post-processing.'''

  def __init__(self, min_level: int, max_level: int, image_size: Tuple[int, int],
               num_scales: int, aspect_ratios: List[Tuple[float, float]],
               anchor_scale: Union[float, List[float]]):
    '''
    Args:
      image_size: (H, W)
      min_level / max_level: feature levels
      num_scales: octave scales per level
      aspect_ratios: list of (y, x) ratios — aspect[1] scales x and aspect[0] scales y (reference :66-67)
      anchor_scale: scalar or one value per level
    '''
    self.min_level = min_level
    self.max_level = max_level
    self.image_size = image_size
    self.num_scales = num_scales
    self.aspect_ratios = aspect_ratios
    self.anchor_scale = anchor_scale
    if isinstance(anchor_scale, (list, tuple)):
      assert len(anchor_scale) == max_level - min_level + 1
      self.anchor_scales = anchor_scale
    else:
      self.anchor_scales = [anchor_scale] * (max_level - min_level + 1)
    self.feat_sizes = get_feat_sizes(self.image_size, self.max_level)
    self._num_levels = max_level - min_level + 1
    self._A = self.get_anchors_per_location()
    self._level_hw = [self.feat_sizes[l] for l in range(min_level, max_level + 1)]
    self._hw = (ctypes.c_int32 * (2 * self._num_levels))(*[d for hw in self._level_hw for d in hw])
    self._table_host = self._build_table()
    self._table = None   # device copy, created on first use
    self._boxes = None

  # -- host-side table: exactly the reference's Python float arithmetic, then one fp32 rounding -----------
  def _build_table(self):
    fs = self.feat_sizes
    parts = []
    for level in range(self.min_level, self.max_level + 1):
      stride = (fs[0][0] / float(fs[level][0]), fs[0][1] / float(fs[level][1]))
      # centres of the level must tile the level's feature map exactly
      yc = _range_f32(stride[0] / 2, self.image_size[0], stride[0])
      xc = _range_f32(stride[1] / 2, self.image_size[1], stride[1])
      if len(yc) != fs[level][0] or len(xc) != fs[level][1]:
        raise ValueError('image_size %r does not tile level %d (%r centres vs feature size %r)' % (
          self.image_size, level, (len(yc), len(xc)), fs[level]))
      hy, hx = [], []
      for scale_octave in range(self.num_scales):
        for aspect in self.aspect_ratios:
          octave_scale = scale_octave / float(self.num_scales)
          a_scale = self.anchor_scales[level - self.min_level]
          hx.append(a_scale * stride[1] * 2**octave_scale * aspect[1] / 2.0)
          hy.append(a_scale * stride[0] * 2**octave_scale * aspect[0] / 2.0)
      parts += [yc, xc, np.asarray(hy, dtype=np.float32), np.asarray(hx, dtype=np.float32)]
    return np.ascontiguousarray(np.concatenate(parts).astype(np.float32))

  def _dev_table(self):
    if self._table is None:
      self._table = T.to_cuda(self._table_host)
      assert self._table.numel() == _lib.load().b200_effdet_table_floats(self._num_levels, self._hw, self._A)
    return self._table

  @property
  def boxes(self):
    '''List over levels of (H, W, anchors, [y1, x1, y2, x2]) tensors (reference attribute `boxes`).'''
    if self._boxes is None:
      lib = _lib.load()
      tab = self._dev_table()
      out = []
      for l, (h, w) in enumerate(self._level_hw):
        t = torch.empty((h, w, self._A, 4), dtype=torch.float32, device=tab.device)
        _lib.check(lib.b200_effdet_anchors(self._num_levels, self._hw, self._A, T.ptr(tab), l, T.ptr(t),
                                           T.stream_ptr()), 'Anchors._generate_boxes')
        out.append(t)
      self._boxes = out
    return self._boxes

  def _generate_boxes(self):
    return self.boxes

  def get_anchors_per_location(self):
    return self.num_scales * len(self.aspect_ratios)

  # -- targets ------------------------------------------------------------------------------------------
  def generate_targets_batch(self, boxes, classes, offsets, classes_num, iou_threshold=0.5, class_index=False):
    '''Batched generate_targets: boxes [total,4] yxyx, classes [total], offsets [B+1] ->
    (boxes, classes, masks) tuples over levels of (B,H,W,A,4), (B,H,W,A,classes_num), (B,H,W,A,1) bool.
    class_index=True (sparse-target mode, SURVEY §8f N3): classes are (B,H,W,A) int32 class ids instead of the
    one-hot rows (0 for unmatched anchors); efficientdet_net_train.get_loss accepts them directly.'''
    lib = _lib.load()
    tab = self._dev_table()
    gb = T.to_cuda(boxes).reshape(-1, 4)
    gc = T.to_cuda(classes, torch.int32).reshape(-1)
    go = T.to_cuda(offsets, torch.int32).reshape(-1)
    B = go.numel() - 1
    C = int(classes_num)
    dev = tab.device
    ob = [torch.empty((B, h, w, self._A, 4), dtype=torch.float32, device=dev) for h, w in self._level_hw]
    if class_index:
      oc = [torch.empty((B, h, w, self._A), dtype=torch.int32, device=dev) for h, w in self._level_hw]
    else:
      oc = [torch.empty((B, h, w, self._A, C), dtype=torch.float32, device=dev) for h, w in self._level_hw]
    om = [torch.empty((B, h, w, self._A, 1), dtype=torch.bool, device=dev) for h, w in self._level_hw]
    L = self._num_levels
    pb = (ctypes.c_void_p * L)(*[t.data_ptr() for t in ob])
    pc = (ctypes.c_void_p * L)(*[t.data_ptr() for t in oc])
    pm = (ctypes.c_void_p * L)(*[t.data_ptr() for t in om])
    assign = lib.b200_effdet_assign_targets_indexed if class_index else lib.b200_effdet_assign_targets
    _lib.check(assign(L, self._hw, self._A, T.ptr(tab), C, B, T.ptr(gb), T.ptr(gc), T.ptr(go),
                                              float(iou_threshold), pb, pc, pm, T.stream_ptr()), 'generate_targets')
    return tuple(ob), tuple(oc), tuple(om)

  def generate_targets(self, boxes, classes, classes_num, iou_threshold=0.5):
    '''
    One image: boxes [n, 4] yxyx, classes [n] ->
      boxes:   [level, [h, w, anchors, [ty, tx, th, tw]]]
      classes: [level, [h, w, anchors, classes_num]]   (one-hot, unmatched anchors = class 0)
      masks:   [level, [h, w, anchors, 1]] bool
    '''
    n = T.to_cuda(boxes).reshape(-1, 4).shape[0]
    ob, oc, om = self.generate_targets_batch(boxes, classes, np.array([0, n], dtype=np.int32), classes_num, iou_threshold)
    return tuple(t[0] for t in ob), tuple(t[0] for t in oc), tuple(t[0] for t in om)

  # -- decode -------------------------------------------------------------------------------------------
  def convert_outputs_boxes(self, outputs_boxes):
    '''[level, [batch, h, w, anchors, [ty, tx, th, tw]]] -> [level, [batch, h, w, anchors, [y1, x1, y2, x2]]]
    (float32; offsets that are all bfloat16 or all float16 are read in place).'''
    lib = _lib.load()
    tab = self._dev_table()
    rel, rel_dtype = T.to_cuda_heads(outputs_boxes)
    if len(rel) != self._num_levels:
      raise ValueError('expected %d levels, got %d' % (self._num_levels, len(rel)))
    B = rel[0].shape[0]
    for t, (h, w) in zip(rel, self._level_hw):
      if tuple(t.shape) != (B, h, w, self._A, 4):
        raise ValueError('level shape %r != %r' % (tuple(t.shape), (B, h, w, self._A, 4)))
    out = [torch.empty(t.shape, dtype=torch.float32, device=t.device) for t in rel]
    L = self._num_levels
    pr = (ctypes.c_void_p * L)(*[t.data_ptr() for t in rel])
    po = (ctypes.c_void_p * L)(*[t.data_ptr() for t in out])
    _lib.check(lib.b200_effdet_decode_typed(L, self._hw, self._A, T.ptr(tab), B, pr, rel_dtype, po, T.stream_ptr()),
               'convert_outputs_boxes')
    return tuple(out)

  # -- post-processing ----------------------------------------------------------------------------------
  def convert_outputs_batch(self, outputs_boxes, outputs_classes, first_image=0, num_images=None, max_output_size=200,
                            iou_threshold=0.5, score_threshold=0.0001, iou_type='diou', with_indices=False):
    '''convert_outputs_one for a range of images in one launch.  Returns a dict of padded tensors
    [n, max_output_size, ...] (boxes, classes_id int64, scores) and `count` [n].  Boxes or logits that are all bfloat16
    or all float16 are read in place; the results are those of the float32 call on the widened tensors.'''
    assert iou_type in ('iou', 'giou', 'diou', 'ciou')
    lib = _lib.load()
    bx, box_dtype = T.to_cuda_heads(outputs_boxes)
    cl, cls_dtype = T.to_cuda_heads(outputs_classes)
    L = self._num_levels
    if len(bx) != L or len(cl) != L:
      raise ValueError('expected %d levels' % L)
    B = cl[0].shape[0]
    C = cl[0].shape[-1]
    n = B - first_image if num_images is None else int(num_images)
    K = int(max_output_size)
    dev = cl[0].device
    out = {
      'boxes': torch.empty((n, K, 4), dtype=torch.float32, device=dev),
      'classes_id': torch.empty((n, K), dtype=torch.int64, device=dev),
      'scores': torch.empty((n, K), dtype=torch.float32, device=dev),
      'count': torch.empty((n,), dtype=torch.int32, device=dev),   # written for every image by the NMS kernel
    }
    if with_indices:
      out['sel_idx'] = torch.empty((n, K), dtype=torch.int32, device=dev)
      out['sel_anchor'] = torch.empty((n, K), dtype=torch.int32, device=dev)
    ws_bytes = lib.b200_effdet_postprocess_workspace_bytes(L, self._hw, self._A, n, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    pb = (ctypes.c_void_p * L)(*[t.data_ptr() for t in bx])
    pc = (ctypes.c_void_p * L)(*[t.data_ptr() for t in cl])
    _lib.check(lib.b200_effdet_postprocess_typed(L, self._hw, self._A, C, B, int(first_image), n, pb, box_dtype, pc, cls_dtype, K,
                                                 float(iou_threshold), float(score_threshold), _lib.METRIC_EFF[iou_type],
                                                 T.ptr(out['boxes']), T.ptr(out['classes_id']), T.ptr(out['scores']),
                                                 T.ptr(out.get('sel_idx')), T.ptr(out.get('sel_anchor')), T.ptr(out['count']),
                                                 T.ptr(ws), ws_bytes, T.stream_ptr()), 'convert_outputs_one')
    return out

  # -- fused passes (one read of the class logits) -----------------------------------------------------------
  def _post_outputs(self, n, K, dev, with_indices):
    out = {
      'boxes': torch.empty((n, K, 4), dtype=torch.float32, device=dev),
      'classes_id': torch.empty((n, K), dtype=torch.int64, device=dev),
      'scores': torch.empty((n, K), dtype=torch.float32, device=dev),
      'count': torch.empty((n,), dtype=torch.int32, device=dev),   # written for every image by the NMS kernel
    }
    if with_indices:
      out['sel_idx'] = torch.empty((n, K), dtype=torch.int32, device=dev)
      out['sel_anchor'] = torch.empty((n, K), dtype=torch.int32, device=dev)
    return out

  def decode_and_postprocess(self, outputs_boxes, outputs_classes, max_output_size=200, iou_threshold=0.5,
                             score_threshold=0.0001, iou_type='diou', with_indices=False):
    '''convert_outputs_boxes followed by convert_outputs_one for every image of the batch (anchors.py:141-202) in one
    pass over the heads.  Returns (decoded boxes per level (float32), dict as convert_outputs_batch).  Offsets or logits
    that are all bfloat16 or all float16 are read in place; the results are those of the float32 call on the widened tensors.'''
    assert iou_type in ('iou', 'giou', 'diou', 'ciou')
    lib = _lib.load()
    tab = self._dev_table()
    rel, rel_dtype = T.to_cuda_heads(outputs_boxes)
    cl, cls_dtype = T.to_cuda_heads(outputs_classes)
    L = self._num_levels
    if len(rel) != L or len(cl) != L:
      raise ValueError('expected %d levels' % L)
    B, C, K = cl[0].shape[0], cl[0].shape[-1], int(max_output_size)
    for t, c, (h, w) in zip(rel, cl, self._level_hw):
      if tuple(t.shape) != (B, h, w, self._A, 4) or tuple(c.shape) != (B, h, w, self._A, C):
        raise ValueError('level shapes %r / %r do not match (B,%d,%d,%d,4|C)' % (tuple(t.shape), tuple(c.shape), h, w, self._A))
    dev = cl[0].device
    dec = [torch.empty(t.shape, dtype=torch.float32, device=t.device) for t in rel]
    out = self._post_outputs(B, K, dev, with_indices)
    ws_bytes = lib.b200_effdet_eval_workspace_bytes(L, self._hw, self._A, B, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])
    _lib.check(lib.b200_effdet_decode_postprocess_typed(L, self._hw, self._A, T.ptr(tab), C, B, arr(rel), rel_dtype, arr(cl),
                                                        cls_dtype, arr(dec), K, float(iou_threshold), float(score_threshold),
                                                        _lib.METRIC_EFF[iou_type], T.ptr(out['boxes']), T.ptr(out['classes_id']),
                                                        T.ptr(out['scores']), T.ptr(out.get('sel_idx')), T.ptr(out.get('sel_anchor')),
                                                        T.ptr(out['count']), T.ptr(ws), ws_bytes, T.stream_ptr()), 'decode_and_postprocess')
    return tuple(dec), out

  def eval_step(self, y_true_boxes, y_true_classes, y_true_masks, y_pred_boxes, y_pred_classes, alpha=0.25, gamma=1.5,
                delta=0.1, max_output_size=200, iou_threshold=0.5, score_threshold=0.0001, iou_type='diou',
                with_indices=False, exchange=None, return_parts=False):
    '''EfficientDetNetTrain.test_step (efficientdet_net_train.py:135-169) without the backbone and the L2 term: the
    _get_loss value, convert_outputs_boxes and convert_outputs_one for every image, reading the class logits ONCE.
    Returns (loss, decoded boxes per level, dict as convert_outputs_batch).  exchange: runtime.PeerExchange /
    NcclExchange for the data-parallel sum of the 2L+1 loss terms.'''
    assert iou_type in ('iou', 'giou', 'diou', 'ciou')
    lib = _lib.load()
    tab = self._dev_table()
    L = self._num_levels
    tb = [T.to_cuda(t) for t in y_true_boxes]
    tc = [T.to_cuda(t) for t in y_true_classes]
    tm = [T.to_cuda(t, torch.bool) for t in y_true_masks]
    rel = [T.to_cuda(t) for t in y_pred_boxes]
    cl = [T.to_cuda(t) for t in y_pred_classes]
    if not (len(tb) == len(tc) == len(tm) == len(rel) == len(cl) == L):
      raise ValueError('expected %d levels' % L)
    B, C, K = cl[0].shape[0], cl[0].shape[-1], int(max_output_size)
    for l, (h, w) in enumerate(self._level_hw):
      if tuple(rel[l].shape) != (B, h, w, self._A, 4) or tuple(cl[l].shape) != (B, h, w, self._A, C):
        raise ValueError('prediction shapes of level %d do not match (B,%d,%d,%d,4|C)' % (l, h, w, self._A))
      if tb[l].shape != rel[l].shape or tc[l].shape != cl[l].shape or tm[l].numel() != rel[l].numel() // 4:
        raise ValueError('target shapes of level %d differ from the predictions (dense one-hot class targets expected)' % l)
    dev = cl[0].device
    if C > 128:
      # the one-pass stream stages 64-anchor tiles of logits and targets in shared memory (classes_num <= 128): wider heads
      # take the separate calls — same results, the logits are read twice
      from ..efficientdet_net_train import get_loss
      res = get_loss(tb, tc, tm, rel, cl, alpha, gamma, delta, exchange=exchange, return_parts=True)
      dec = self.convert_outputs_boxes(rel)
      out = self.convert_outputs_batch(dec, cl, max_output_size=K, iou_threshold=iou_threshold, score_threshold=score_threshold,
                                       iou_type=iou_type, with_indices=with_indices)
      return (res[0], tuple(dec), out, res[1], res[2]) if return_parts else (res[0], tuple(dec), out)
    dec = [torch.empty_like(t) for t in rel]
    out = self._post_outputs(B, K, dev, with_indices)
    sums = torch.empty((2 * L + 1,), dtype=torch.float64, device=dev)
    ws_bytes = lib.b200_effdet_eval_workspace_bytes(L, self._hw, self._A, B, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])
    _lib.check(lib.b200_effdet_eval_step(L, self._hw, self._A, T.ptr(tab), C, B, arr(tb), arr(tc), arr(tm), arr(rel), arr(cl),
                                         float(alpha), float(gamma), float(delta), 0.0, T.ptr(sums), arr(dec), K,
                                         float(iou_threshold), float(score_threshold), _lib.METRIC_EFF[iou_type],
                                         T.ptr(out['boxes']), T.ptr(out['classes_id']), T.ptr(out['scores']),
                                         T.ptr(out.get('sel_idx')), T.ptr(out.get('sel_anchor')), T.ptr(out['count']),
                                         T.ptr(ws), ws_bytes, T.stream_ptr()), 'eval_step')
    return self._eval_finalize(sums, cl, dec, out, exchange, return_parts, 'eval_step')

  def _eval_finalize(self, sums, cl, dec, out, exchange, return_parts, what):
    '''The tail of the eval steps: the data-parallel sum of the 2L+1 terms and the loss normalisation.'''
    lib = _lib.load()
    L, dev = self._num_levels, sums.device
    scale = 1
    peer = exchange is not None and hasattr(exchange, 'mailboxes')
    if exchange is not None:
      if not peer:
        exchange.allreduce_(sums)
      scale = exchange.world
    nm = (ctypes.c_double * L)(*[float(t.numel()) * scale for t in cl])
    parts = torch.empty((L, 2), dtype=torch.float32, device=dev)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    npos = torch.empty((), dtype=torch.float32, device=dev)
    if peer:
      rank, world, boxes_ = exchange.args()
      _lib.check(lib.b200_focal_box_finalize_dp(L, T.ptr(sums), nm, T.ptr(parts), T.ptr(loss), T.ptr(npos), rank, world, boxes_,
                                                T.stream_ptr()), what + ' (data parallel)')
    else:
      _lib.check(lib.b200_focal_box_finalize(L, T.ptr(sums), nm, T.ptr(parts), T.ptr(loss), T.ptr(npos), T.stream_ptr()), what)
    if return_parts:
      return loss, tuple(dec), out, parts, npos
    return loss, tuple(dec), out

  def eval_step_from_boxes(self, boxes, classes, offsets, y_pred_boxes, y_pred_classes, match_iou_threshold=0.5, alpha=0.25,
                           gamma=1.5, delta=0.1, max_output_size=200, iou_threshold=0.5, score_threshold=0.0001,
                           iou_type='diou', with_indices=False, exchange=None, return_parts=False):
    '''eval_step with the ground truth as box lists instead of the dense targets: boxes [total,4] y1,x1,y2,x2, classes
    [total], offsets [B+1] as generate_targets_batch takes them (match_iou_threshold is its iou_threshold).  Returns what
    eval_step returns on generate_targets_batch's targets, bit for bit, without writing the targets: one call matches
    the anchors to the boxes (one int32 per anchor) and streams the heads once, reading only the logits of the class
    tensor.  The keyword arguments are eval_step's.  No host synchronisation (capturable with runtime.capture).
    classes_num < 4 and > 128 take generate_targets_batch + eval_step.

    The per-image mAP of test_step follows from the returned dict, e.g. with the box lists as ground truth:
    utils.mAP.Get_mAP_padded(boxes, classes, offsets, out, classes_num).'''
    assert iou_type in ('iou', 'giou', 'diou', 'ciou')
    from ..efficientdet_net_train import _from_boxes_args
    gb, gc, go, rel, cl, _, B, C = _from_boxes_args(self, boxes, classes, offsets, y_pred_boxes, y_pred_classes)
    rel, cl = [T.to_cuda(t) for t in rel], [T.to_cuda(t) for t in cl]   # the tiled stream reads fp32 heads
    if C < 4 or C > 128:
      # the one-pass stream rebuilds one-hot rows a float4 at a time (C >= 4) and stages 64-anchor tiles of logits in
      # shared memory (C <= 128): other heads take the dense targets — same results
      tb, tc, tm = self.generate_targets_batch(gb, gc, go, C, match_iou_threshold)
      return self.eval_step(tb, tc, tm, rel, cl, alpha=alpha, gamma=gamma, delta=delta, max_output_size=max_output_size,
                            iou_threshold=iou_threshold, score_threshold=score_threshold, iou_type=iou_type,
                            with_indices=with_indices, exchange=exchange, return_parts=return_parts)
    lib = _lib.load()
    tab = self._dev_table()
    L, K, dev = self._num_levels, int(max_output_size), cl[0].device
    dec = [torch.empty_like(t) for t in rel]
    out = self._post_outputs(B, K, dev, with_indices)
    sums = torch.empty((2 * L + 1,), dtype=torch.float64, device=dev)
    ws_bytes = lib.b200_effdet_eval_step_from_boxes_workspace_bytes(L, self._hw, self._A, B, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])
    _lib.check(lib.b200_effdet_eval_step_from_boxes(L, self._hw, self._A, T.ptr(tab), C, B, T.ptr(gb), T.ptr(gc), T.ptr(go),
                                                    gb.shape[0], float(match_iou_threshold), arr(rel), arr(cl), float(alpha),
                                                    float(gamma), float(delta), 0.0, T.ptr(sums), arr(dec), K,
                                                    float(iou_threshold), float(score_threshold), _lib.METRIC_EFF[iou_type],
                                                    T.ptr(out['boxes']), T.ptr(out['classes_id']), T.ptr(out['scores']),
                                                    T.ptr(out.get('sel_idx')), T.ptr(out.get('sel_anchor')), T.ptr(out['count']),
                                                    T.ptr(ws), ws_bytes, T.stream_ptr()), 'eval_step_from_boxes')
    return self._eval_finalize(sums, cl, dec, out, exchange, return_parts, 'eval_step_from_boxes')

  def convert_outputs_one(self, batch_index, outputs_boxes, outputs_classes):
    '''One image of the batch: (nms_boxes [K,4], nms_classes_id [K] int64, nms_scores [K]); K <= 200.'''
    r = self.convert_outputs_batch(outputs_boxes, outputs_classes, first_image=int(batch_index), num_images=1)
    k = int(r['count'][0].item())
    return r['boxes'][0, :k], r['classes_id'][0, :k], r['scores'][0, :k]
