"""Drop-in for the loss aggregation of the reference's efficientnet/efficientdet_net_train.py
(EfficientDetNetTrain._get_loss :41-52).  The L2-regularisation term (:21-28,42) is over model weights and stays
in the TF graph; add it to the value returned here."""
import ctypes

import numpy as np
import torch

from ... import _lib, _tensors as T
from ..losses.focal_loss import _partial_sums, _pred_heads


def get_loss(y_true_boxes, y_true_classes, y_true_masks, y_pred_boxes, y_pred_classes, alpha=0.25, gamma=1.5,
             delta=0.1, global_batch_scale=1, group=None, return_parts=False, with_grad=False, exchange=None,
             grad_dtype=torch.float32, grad_scale=None):
  '''sum over levels of (50 * box_loss + focal_loss) with num_positives = sum(masks) + 1.

  Data parallel: every rank passes its shard; the 2L+1 fp64 partial sums are all-reduced once before the
  normalisation — inside the finalize kernel over NVLink peer mailboxes (exchange=runtime.PeerExchange), by the
  library's ncclAllReduce (runtime.NcclExchange), or by torch.distributed on `group` (exchange=None).  `global_batch_scale` = world size when the per-level element count of the Keras mean must refer
  to the global batch.

  Mixed precision: box outputs and class logits that are all bf16, or all fp16, are read in place (the sums are
  bit-identical to the call on the widened heads); any other mix is cast to fp32.  grad_dtype / grad_scale (with_grad):
  as get_loss_and_grad.
  '''
  lib = _lib.load()
  if with_grad:
    T.grad_code(grad_dtype)
  pb, pc, pdt = _pred_heads(list(y_pred_boxes), list(y_pred_classes))
  sums, numel = _partial_sums(list(y_true_boxes), list(y_true_classes), list(y_true_masks), pb, pc, alpha, gamma, delta, 0.0)
  import torch.distributed as dist
  peer = exchange is not None and hasattr(exchange, 'mailboxes')
  if exchange is not None:
    # runtime.NcclExchange: ncclAllReduce issued by the library; runtime.PeerExchange: summed inside the finalize kernel
    if not peer:
      exchange.allreduce_(sums)
    global_batch_scale = exchange.world
  elif dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    global_batch_scale = dist.get_world_size(group)
  L = len(numel)
  nm = (ctypes.c_double * L)(*[n * global_batch_scale for n in numel])
  parts = torch.empty((L, 2), dtype=torch.float32, device=sums.device)
  loss = torch.empty((), dtype=torch.float32, device=sums.device)
  npos = torch.empty((), dtype=torch.float32, device=sums.device)
  if peer:
    rank, world, boxes_ = exchange.args()
    _lib.check(lib.b200_focal_box_finalize_dp(L, T.ptr(sums), nm, T.ptr(parts), T.ptr(loss), T.ptr(npos), rank, world, boxes_,
                                              T.stream_ptr()), '_get_loss (data parallel)')
  else:
    _lib.check(lib.b200_focal_box_finalize(L, T.ptr(sums), nm, T.ptr(parts), T.ptr(loss), T.ptr(npos), T.stream_ptr()),
               '_get_loss')
  if with_grad:
    tb = [T.to_cuda(t) for t in y_true_boxes]
    # class targets: one-hot float tensors, or integer class ids (generate_targets_batch(class_index=True)) — the same
    # detection as the forward pass uses
    indexed = any(not torch.is_floating_point(torch.as_tensor(t)) for t in y_true_classes)
    tc = [T.to_cuda(t, torch.int32) if indexed else T.to_cuda(t) for t in y_true_classes]
    grads, gdt, scale = T.grad_out(pb + pc, grad_dtype, grad_scale)
    gb, gc = grads[:L], grads[L:]
    C = pc[0].shape[-1]
    for l in range(L):
      if tc[l].numel() * (C if indexed else 1) != pc[l].numel():
        raise ValueError('class target / output shapes differ at level %d' % l)
    anc = (ctypes.c_ulonglong * L)(*[t.numel() // C for t in pc])
    arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])
    grad = lib.b200_focal_box_grad_indexed_typed if indexed else lib.b200_focal_box_grad_typed
    _lib.check(grad(L, anc, C, arr(tb), arr(tc), arr(pb), arr(pc), pdt, float(alpha), float(gamma), float(delta), 0.0,
                    T.ptr(sums), nm, arr(gb), arr(gc), gdt, T.ptr(scale), T.stream_ptr()),
               '_get_loss backward')
    return loss, tuple(gb), tuple(gc)
  return (loss, parts, npos) if return_parts else loss


def get_loss_and_grad(y_true_boxes, y_true_classes, y_true_masks, y_pred_boxes, y_pred_classes, alpha=0.25, gamma=1.5,
                      delta=0.1, grad_dtype=torch.float32, grad_scale=None):
  '''_get_loss plus (d loss / d y_pred_boxes[l], d loss / d y_pred_classes[l]) for an upstream gradient of 1.

  Mixed precision: heads that are all bf16 or all fp16 are read in place.  grad_dtype (torch.float32, the default,
  torch.bfloat16 or torch.float16) is the type both gradient families are written in, each element rounded once from
  g * grad_scale, where g is the fp32 gradient of the call on the widened heads.  grad_scale: None (no multiply), a
  1-element float32 tensor on the heads' device (e.g. a loss scale that changes between steps: no host
  synchronisation, graph capturable) or a Python float.'''
  return get_loss(y_true_boxes, y_true_classes, y_true_masks, y_pred_boxes, y_pred_classes, alpha, gamma, delta,
                  with_grad=True, grad_dtype=grad_dtype, grad_scale=grad_scale)


def _from_boxes_args(anchors, boxes, classes, offsets, y_pred_boxes, y_pred_classes):
  '''Checks and device placement shared by get_loss_from_boxes, get_loss_from_boxes_and_grad and
  Anchors.eval_step_from_boxes.'''
  L = anchors._num_levels
  pb, pc, pdt = _pred_heads(list(y_pred_boxes), list(y_pred_classes))
  if len(pb) != L or len(pc) != L:
    raise ValueError('expected %d levels, got %d box / %d class outputs' % (L, len(pb), len(pc)))
  gb = T.to_cuda(boxes).reshape(-1, 4)
  if gb.data_ptr() % 16:
    gb = gb.clone()   # the loss pass reads a GT box as one 16-byte load
  gc = T.to_cuda(classes, torch.int32).reshape(-1)
  go = T.to_cuda(offsets, torch.int32).reshape(-1)
  if gc.numel() != gb.shape[0]:
    raise ValueError('%d boxes but %d classes' % (gb.shape[0], gc.numel()))
  B, C = go.numel() - 1, pc[0].shape[-1]
  if B < 0:
    raise ValueError('offsets must hold B + 1 entries')
  for l, (h, w) in enumerate(anchors._level_hw):
    if tuple(pb[l].shape) != (B, h, w, anchors._A, 4) or tuple(pc[l].shape) != (B, h, w, anchors._A, C):
      raise ValueError('prediction shapes of level %d (%r / %r) do not match (%d,%d,%d,%d,4|C)' % (
          l, tuple(pb[l].shape), tuple(pc[l].shape), B, h, w, anchors._A))
  return gb, gc, go, pb, pc, pdt, B, C


def _loss_from_boxes(anchors, boxes, classes, offsets, y_pred_boxes, y_pred_classes, iou_threshold, alpha, gamma, delta,
                     global_batch_scale, group, exchange, return_parts, with_grad, grad_dtype=torch.float32, grad_scale=None):
  if with_grad:
    T.grad_code(grad_dtype)
  gb, gc, go, pb, pc, pdt, B, C = _from_boxes_args(anchors, boxes, classes, offsets, y_pred_boxes, y_pred_classes)
  if C < 4:
    # the one-pass kernel rebuilds one-hot rows a float4 at a time (a float4 may straddle at most two anchors):
    # narrower heads take the dense targets — same results
    tb, tc, tm = anchors.generate_targets_batch(gb, gc, go, C, iou_threshold)
    return get_loss(tb, tc, tm, pb, pc, alpha, gamma, delta, global_batch_scale, group, return_parts, with_grad, exchange,
                    grad_dtype, grad_scale)
  lib = _lib.load()
  import torch.distributed as dist
  allreduce = None
  if exchange is not None:
    allreduce, global_batch_scale = exchange.allreduce_, exchange.world
  elif dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
    allreduce = lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    global_batch_scale = dist.get_world_size(group)
  L, dev = anchors._num_levels, pc[0].device
  tab = anchors._dev_table()
  nm = (ctypes.c_double * L)(*[float(t.numel()) * global_batch_scale for t in pc])
  sums = torch.empty((2 * L + 1,), dtype=torch.float64, device=dev)
  ws_bytes = lib.b200_effdet_loss_from_boxes_workspace_bytes(L, anchors._hw, anchors._A, B)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
  n_boxes = gb.shape[0]
  _lib.check(lib.b200_effdet_loss_from_boxes_match(L, anchors._hw, anchors._A, T.ptr(tab), B, T.ptr(gb), T.ptr(go), n_boxes,
                                                   float(iou_threshold), T.ptr(sums), T.ptr(ws), ws_bytes, T.stream_ptr()),
             'get_loss_from_boxes (match)')
  if allreduce is not None:
    allreduce(sums[2 * L:])   # num_positives over the global batch scales every gradient
  arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])
  grad_b = grad_c = scale = None
  gdt = T.DTYPE_F32
  if with_grad:
    grads, gdt, scale = T.grad_out(pb + pc, grad_dtype, grad_scale)
    grad_b, grad_c = grads[:L], grads[L:]
  _lib.check(lib.b200_effdet_loss_from_boxes_grad_typed(L, anchors._hw, anchors._A, T.ptr(tab), C, B, T.ptr(gb), T.ptr(gc),
                                                        n_boxes, arr(pb), arr(pc), pdt, float(alpha), float(gamma), float(delta),
                                                        0.0, nm, T.ptr(sums), arr(grad_b) if with_grad else None,
                                                        arr(grad_c) if with_grad else None, gdt, T.ptr(scale), T.ptr(ws),
                                                        ws_bytes, T.stream_ptr()),
             'get_loss_from_boxes')
  if allreduce is not None:
    allreduce(sums[:2 * L])
  parts = torch.empty((L, 2), dtype=torch.float32, device=dev)
  loss = torch.empty((), dtype=torch.float32, device=dev)
  npos = torch.empty((), dtype=torch.float32, device=dev)
  # sums[2L] is global already: the plain finalize (the _dp form would add it once per rank)
  _lib.check(lib.b200_focal_box_finalize(L, T.ptr(sums), nm, T.ptr(parts), T.ptr(loss), T.ptr(npos), T.stream_ptr()),
             'get_loss_from_boxes (finalize)')
  if with_grad:
    return loss, tuple(grad_b), tuple(grad_c)
  return (loss, parts, npos) if return_parts else loss


def get_loss_from_boxes(anchors, boxes, classes, offsets, y_pred_boxes, y_pred_classes, iou_threshold=0.5, alpha=0.25,
                        gamma=1.5, delta=0.1, global_batch_scale=1, group=None, exchange=None, return_parts=False):
  '''Anchors.generate_targets_batch + get_loss without materialising the targets (SURVEY §8f N3).

  anchors: utils.anchors.Anchors; boxes [total,4] y1,x1,y2,x2, classes [total], offsets [B+1] (image b owns rows
  offsets[b]:offsets[b+1]).  The loss equals get_loss on the targets generate_targets_batch writes from the same boxes
  (fp64 sums in another order).  Data parallel: every rank passes its own images; the matched-anchor count and then the
  2L loss terms are all-reduced (exchange = runtime.PeerExchange / NcclExchange, or torch.distributed on `group`).  No
  host synchronisation: the call can be captured with runtime.capture.  classes_num < 4 takes generate_targets_batch +
  get_loss.  Box outputs and class logits that are all bf16, or all fp16, are read in place (the loss is bit-identical
  to the call on the widened heads); any other mix is cast to fp32.'''
  return _loss_from_boxes(anchors, boxes, classes, offsets, y_pred_boxes, y_pred_classes, iou_threshold, alpha, gamma, delta,
                          global_batch_scale, group, exchange, return_parts, False)


def get_loss_from_boxes_and_grad(anchors, boxes, classes, offsets, y_pred_boxes, y_pred_classes, iou_threshold=0.5,
                                 alpha=0.25, gamma=1.5, delta=0.1, global_batch_scale=1, group=None, exchange=None,
                                 grad_dtype=torch.float32, grad_scale=None):
  '''get_loss_from_boxes plus (d loss / d y_pred_boxes[l], d loss / d y_pred_classes[l]) for an upstream gradient of 1,
  in one pass over the heads: returns (loss, grad_boxes, grad_classes) as get_loss_and_grad does, with gradients
  bit-identical to generate_targets_batch + get_loss_and_grad on the same boxes.  Mixed precision (bf16 / fp16 heads,
  grad_dtype, grad_scale): as get_loss_and_grad.'''
  return _loss_from_boxes(anchors, boxes, classes, offsets, y_pred_boxes, y_pred_classes, iou_threshold, alpha, gamma, delta,
                          global_batch_scale, group, exchange, False, True, grad_dtype, grad_scale)


class EfficientDetNetTrain(object):
  '''Only the head-loss part of the reference class: `_get_loss` with the reference's argument order.'''

  def __init__(self, alpha=0.25, gamma=1.5, **unused):
    self.alpha = alpha
    self.gamma = gamma

  def _get_loss(self, y_true_boxes, y_true_classes, y_true_masks, y_pred_boxes, y_pred_classes):
    return get_loss(y_true_boxes, y_true_classes, y_true_masks, y_pred_boxes, y_pred_classes, self.alpha, self.gamma)
