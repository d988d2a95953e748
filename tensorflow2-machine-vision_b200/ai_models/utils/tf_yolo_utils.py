"""Drop-in for the reference's utils/tf_yolo_utils.py: GetLoss (:6-127), GetBoxes (:129-167), GetNMSBoxes (:169-269).

Same names, positional order, defaults and NHWC layouts; tensors may be torch CUDA tensors, anything exporting
DLPack (tf.experimental.dlpack.to_dlpack on a TF box), or host arrays (copied).  Results are torch CUDA tensors.
"""
import ctypes

import numpy as np
import torch

from ... import _lib, _tensors as T

NMS_MAX_OUTPUT = 500  # hard-coded in the reference, tf_yolo_utils.py:259


def GetBoxes(y, anchors_wh, classes_num):
  '''Head offsets -> boxes in [0,1].

  Args:
    y: (batch, H, W, anchors_num, 5+classes_num)
    anchors_wh: (anchors_num, 2), already divided by image_wh
  Returns:
    boxes (N,4) x1,y1,x2,y2; confidence (N,1); classes (N,classes_num) — rows with x2<=x1 or y2<=y1 removed,
    batch dimension flattened, row-major order (reference :163-166).
  '''
  lib = _lib.load()
  y = T.to_cuda(y)
  B, H, W, A = y.shape[0], y.shape[1], y.shape[2], y.shape[3]
  C = int(classes_num)
  if y.shape[4] != 5 + C:
    raise ValueError('last dimension %d != 5 + classes_num %d' % (y.shape[4], C))
  anc = T.to_cuda(anchors_wh).reshape(-1)
  if anc.numel() != 2 * A:
    raise ValueError('anchors_wh must be (anchors_num, 2)')
  n = B * H * W * A
  boxes = torch.empty((n, 4), dtype=torch.float32, device=y.device)
  conf = torch.empty((n, 1), dtype=torch.float32, device=y.device)
  classes = torch.empty((n, C), dtype=torch.float32, device=y.device)
  valid = torch.empty((n,), dtype=torch.uint8, device=y.device)
  _lib.check(lib.b200_yolo_decode_dense(T.ptr(y), B, H, W, A, C, T.ptr(anc), T.ptr(boxes), T.ptr(conf),
                                        T.ptr(classes), T.ptr(valid), T.stream_ptr()), 'GetBoxes')
  return _compact_rows(valid, [boxes, conf, classes])


def _compact_rows(flags, arrays):
  '''tf.boolean_mask over rows, order preserved: flags (n,) uint8, arrays of shape (n, k_i).'''
  lib = _lib.load()
  n = flags.numel()
  dev = flags.device
  pos = torch.empty((max(n, 1),), dtype=torch.int32, device=dev)
  total = torch.zeros((1,), dtype=torch.int32, device=dev)
  ws_bytes = lib.b200_row_positions_workspace_bytes(n)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
  _lib.check(lib.b200_row_positions(T.ptr(flags), n, T.ptr(pos), T.ptr(total), T.ptr(ws), ws_bytes, T.stream_ptr()),
             'boolean_mask')
  k = int(total.item())
  out = []
  for a in arrays:
    rf = a.shape[1]
    d = torch.empty((k, rf), dtype=torch.float32, device=dev)
    if k:
      _lib.check(lib.b200_gather_rows(T.ptr(a), rf, T.ptr(flags), T.ptr(pos), n, T.ptr(d), T.stream_ptr()), 'boolean_mask')
    out.append(d)
  return tuple(out)


def GetGroudTruth(y, classes_num=None):
  '''yolo_v4/model.py:380-395: dense target (…, 5+C) -> (n, 5) rows [x1, y1, x2, y2, class] of the records with
  conf != 0, in row-major order (the mAP input).'''
  lib = _lib.load()
  y = T.to_cuda(y)
  C = y.shape[-1] - 5 if classes_num is None else int(classes_num)
  n = y.numel() // (5 + C)
  rows = torch.empty((n, 5), dtype=torch.float32, device=y.device)
  flags = torch.empty((n,), dtype=torch.uint8, device=y.device)
  _lib.check(lib.b200_yolo_ground_truth_rows(T.ptr(y), n, C, T.ptr(rows), T.ptr(flags), T.stream_ptr()), 'GetGroudTruth')
  return _compact_rows(flags, [rows])[0]


def _levels(y1, y2, y3, anchors_wh):
  anc = T.host_floats(anchors_wh)
  if anc.size % 6 != 0:
    raise ValueError('anchors_wh must be (3, anchors_num, 2)')
  A = anc.size // 6
  heads, dtype = T.to_cuda_heads((y1, y2, y3))
  heads = [t.reshape(t.shape[0], t.shape[1], t.shape[2], -1) if t.dim() == 5 else t for t in heads]
  B = heads[0].shape[0]
  ch = heads[0].shape[3]
  if ch % A != 0:
    raise ValueError('channel count %d is not a multiple of anchors_num %d' % (ch, A))
  for t in heads:
    if t.shape[0] != B or t.shape[3] != ch:
      raise ValueError('the three heads disagree on batch or channel size')
  return heads, dtype, anc, A, B, ch // A


def GetNMSBoxesBatch(y1, y2, y3, anchors_wh, image_wh, classes_num,
  confidence_thresh=0.5, scores_thresh=0.3, iou_thresh=0.5, iou_type='iou',
  max_output_size=NMS_MAX_OUTPUT, with_classes=True, with_indices=False):
  '''Batched form of GetNMSBoxes: the reference's B == 1 semantics applied to every image.

  Returns a dict of padded tensors [B, max_output_size, ...] plus `count` [B] (int32):
  boxes, classes_id, scores, classes (optional), confidence, and with_indices -> sel_idx / sel_anchor.
  Heads that are all bfloat16 or all float16 (mixed-precision networks) are read in place; the outputs are fp32 and
  bit-identical to those of the fp32 heads y.float().
  '''
  assert iou_type in ['iou','diou','ciou']
  lib = _lib.load()
  heads, dtype, anc, A, B, RF = _levels(y1, y2, y3, anchors_wh)
  C = int(classes_num)
  if RF != 5 + C:
    raise ValueError('head channels %d != anchors_num*(5+classes_num)' % (RF * A))
  img = T.host_floats(image_wh, 2)
  dev = heads[0].device
  K = int(max_output_size)
  hw = (ctypes.c_int32 * 6)(*[d for t in heads for d in (t.shape[1], t.shape[2])])
  hp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in heads])
  out = {
    'boxes': torch.empty((B, K, 4), dtype=torch.float32, device=dev),
    'classes_id': torch.empty((B, K), dtype=torch.int32, device=dev),
    'scores': torch.empty((B, K), dtype=torch.float32, device=dev),
    'confidence': torch.empty((B, K, 1), dtype=torch.float32, device=dev),
    'count': torch.empty((B,), dtype=torch.int32, device=dev),   # written for every image by the NMS kernel
  }
  if with_classes:
    out['classes'] = torch.empty((B, K, C), dtype=torch.float32, device=dev)
  if with_indices:
    out['sel_idx'] = torch.empty((B, K), dtype=torch.int32, device=dev)
    out['sel_anchor'] = torch.empty((B, K), dtype=torch.int32, device=dev)
  ws_bytes = lib.b200_yolo_decode_nms_workspace_bytes(hw, B, A, K)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
  _lib.check(lib.b200_yolo_decode_nms_typed(
    hp, dtype, hw, B, A, C, anc.ctypes.data_as(ctypes.c_void_p), img.ctypes.data_as(ctypes.c_void_p),
    float(confidence_thresh), float(scores_thresh), float(iou_thresh), _lib.METRIC_YOLO[iou_type], K,
    T.ptr(out['boxes']), T.ptr(out['classes_id']), T.ptr(out['scores']), T.ptr(out.get('classes')),
    T.ptr(out['confidence']), T.ptr(out.get('sel_idx')), T.ptr(out.get('sel_anchor')), T.ptr(out['count']),
    T.ptr(ws), ws_bytes, T.stream_ptr()), 'GetNMSBoxes')
  return out


def GetNMSBoxes(y1, y2, y3, anchors_wh, image_wh, classes_num,
  confidence_thresh=0.5, scores_thresh=0.3, iou_thresh=0.5, iou_type='iou'):
  '''Decode the three heads, threshold, per-class NMS (cap 500), gather.

  Returns (selected_boxes (K,4), selected_classes_id (K,) int32, selected_scores (K,),
  selected_classes (K,classes_num), selected_confidence (K,1)) exactly as the reference for batch size 1.
  For batch size > 1 (where the reference would run one NMS over the flattened batch) the per-image results
  are concatenated in image order; use GetNMSBoxesBatch to keep them apart.
  '''
  r = GetNMSBoxesBatch(y1, y2, y3, anchors_wh, image_wh, classes_num, confidence_thresh, scores_thresh,
                       iou_thresh, iou_type)
  cnt = r['count'].cpu().tolist()
  pick = lambda t: torch.cat([t[b, :cnt[b]] for b in range(len(cnt))], dim=0) if len(cnt) != 1 else t[0, :cnt[0]]
  return pick(r['boxes']), pick(r['classes_id']), pick(r['scores']), pick(r['classes']), pick(r['confidence'])


def _pred_levels(y_pred, with_grad):
  '''y_pred of the loss -> (3 tensors, B200_DTYPE_* code).  All three levels bf16, or all fp16, are read in place in their
  type (the loss, parts, ignore mask and fp32 gradient are bit-identical to the call on y.float()); any other mix is cast
  to fp32.  y_pred in pinned host memory is consumed in place by the forward (unified addressing): the forward kernels
  need only the five box/conf logits of every record and the object records, ~6 % of the tensor, so fetching those
  sectors over PCIe beats copying the whole tensor first (9.2 -> 3.1 ms at 608x608 batch 64).  The backward pass needs
  device tensors.'''
  if len(y_pred) != 3:
    raise ValueError('y_pred must hold 3 levels')
  return T.to_cuda_heads(y_pred, keep_pinned=not with_grad)


def _loss_call(y_true, y_pred, image_wh, anchors_wh, iou_thresh, iou_type, variant, batch_divisor=None,
               return_parts=False, workspace=None, ignore_out=None, with_grad=False, exchange=None, defer_collect=False,
               grad_dtype=torch.float32, grad_scale=None):
  """exchange: a runtime.PeerExchange (the 12 terms are summed over the ranks inside the finalize kernel, NVLink peer
  stores) or a runtime.NcclExchange (b200_allreduce_loss + b200_yolo_loss_combine behind the loss); batch_divisor must
  then be the GLOBAL batch.  Forward only.  defer_collect (PeerExchange only): the call ends with the publish half of the
  exchange and returns this rank's own terms; exchange.collect_yolo(parts, loss) on another stream finishes it.
  y_pred: see _pred_levels; a PeerExchange call reads fp32 only (half levels are cast)."""
  lib = _lib.load()
  if len(y_true) != 3 or len(y_pred) != 3:
    raise ValueError('y_true and y_pred must each hold 3 levels')
  if with_grad:
    T.grad_code(grad_dtype)
  yt = [T.to_cuda(t) for t in y_true]
  yp, pdt = _pred_levels(y_pred, with_grad)
  if pdt != T.DTYPE_F32 and exchange is not None and hasattr(exchange, 'mailboxes'):
    yp, pdt = [T.to_cuda(t) for t in yp], T.DTYPE_F32   # the fused-exchange entries read fp32 heads
  anc = T.host_floats(anchors_wh)
  if anc.size % 6 != 0:
    raise ValueError('anchors_wh must be (3, anchors_num, 2)')
  A = anc.size // 6
  B = yt[0].shape[0]
  RF = yt[0].shape[-1]
  for l in range(3):
    if yt[l].dim() != 5 or yt[l].shape[3] != A:
      raise ValueError('y_true[%d] must be (B,H,W,%d,5+C)' % (l, A))
    if yp[l].numel() != yt[l].numel():
      raise ValueError('y_pred[%d] cannot be reshaped to y_true[%d]' % (l, l))
  img = T.host_floats(image_wh, 2)
  dev = yt[0].device
  hw = (ctypes.c_int32 * 6)(*[d for t in yt for d in (t.shape[1], t.shape[2])])
  tp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in yt])
  pp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in yp])
  parts = torch.empty((3, 4), dtype=torch.float32, device=dev)
  loss = torch.empty((), dtype=torch.float32, device=dev)
  ws_bytes = lib.b200_yolo_loss_workspace_bytes(hw, B, A)
  if workspace is None or workspace.numel() < ws_bytes:
    workspace = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
  div = float(B if batch_divisor is None else batch_divisor)
  if with_grad:
    grads, gdt, scale = T.grad_out(yp, grad_dtype, grad_scale)
    gp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in grads])
    _lib.check(lib.b200_yolo_loss_grad_typed(tp, pp, pdt, hw, B, A, RF - 5, anc.ctypes.data_as(ctypes.c_void_p),
                                             img.ctypes.data_as(ctypes.c_void_p), float(iou_thresh),
                                             _lib.METRIC_YOLO[iou_type], variant, div, T.ptr(parts), T.ptr(loss), gp, gdt,
                                             T.ptr(scale), T.ptr(workspace), ws_bytes, T.stream_ptr()), 'GetLoss')
    return loss, parts, grads
  if exchange is not None and hasattr(exchange, 'mailboxes'):
    rank, world, boxes_ = exchange.args()
    entry = lib.b200_yolo_loss_dp_publish if (defer_collect and world > 1) else lib.b200_yolo_loss_dp
    _lib.check(entry(tp, pp, hw, B, A, RF - 5, anc.ctypes.data_as(ctypes.c_void_p),
                                     img.ctypes.data_as(ctypes.c_void_p), float(iou_thresh), _lib.METRIC_YOLO[iou_type],
                                     variant, div, T.ptr(parts), T.ptr(loss), T.ptr(workspace), ws_bytes, rank, world, boxes_,
                                     T.stream_ptr()), 'GetLoss (data parallel)')
    return (loss, parts) if return_parts else loss
  _lib.check(lib.b200_yolo_loss_typed(tp, pp, pdt, hw, B, A, RF - 5, anc.ctypes.data_as(ctypes.c_void_p),
                                      img.ctypes.data_as(ctypes.c_void_p), float(iou_thresh), _lib.METRIC_YOLO[iou_type],
                                      variant, div, T.ptr(parts), T.ptr(loss), T.ptr(ignore_out), T.ptr(workspace), ws_bytes,
                                      T.stream_ptr()),
             'GetLoss')
  if exchange is not None:  # NCCL transport: all-reduce the 12 terms in place, then the reference's order of additions
    exchange.allreduce_(parts)
    _lib.check(lib.b200_yolo_loss_combine(T.ptr(parts), T.ptr(loss), T.stream_ptr()), 'GetLoss (data parallel)')
  return (loss, parts) if return_parts else loss


def GetLoss(y_true, y_pred, image_wh, anchors_wh, iou_thresh=0.5, iou_type='iou'):
  '''
  YOLO loss (forward value).

  Args:
    y_true: [(batch, 13, 13, 3, 5+num_classes), (batch, 26, 26, 3, ...), (batch, 52, 52, 3, ...)]
    y_pred: same three levels, (batch, H, W, 3*(5+num_classes)) or already split per anchor
    image_wh: (w, h) pixels; anchors_wh: (3, 3, 2) pixels, layer 0 = coarsest head
    iou_type: metric of the ignore mask only ('iou' for YOLOv3, 'ciou' for YOLOv4 call sites)
  Returns:
    scalar fp32 tensor (device)
  '''
  assert iou_type in ['iou','diou','ciou']
  return _loss_call(y_true, y_pred, image_wh, anchors_wh, iou_thresh, iou_type, 0)


def GetLossFromBoxes(classes, boxes, offsets, y_pred, image_wh, anchors_wh, classes_num, iou_thresh=0.5, iou_type='iou',
                     target_anchors=None, batch_divisor=None, return_parts=False, workspace=None, ignore_out=None):
  '''
  Sparse-target fusion (SURVEY §8f N3, an API extension, not a reference signature): DataGenerator.GetTargets
  followed by GetLoss without materialising the dense y_true.  Same value as
  GetLoss(GetTargetsBatch(classes, boxes, offsets), y_pred, ...) up to fp64 summation order.

  Args:
    classes [total] int, boxes [total,4] pixel corners x1,y1,x2,y2, offsets [B+1] (image b owns boxes offsets[b]:offsets[b+1])
    y_pred: three levels (B, H, W, 3*(5+classes_num)) or already split per anchor
    anchors_wh: (3, anchors_num, 2) pixels, as GetLoss takes them
    target_anchors: the anchors DataGenerator was constructed with (default: anchors_wh)
  '''
  assert iou_type in ['iou','diou','ciou']
  loss, parts, _ = _boxes_call(classes, boxes, offsets, y_pred, image_wh, anchors_wh, classes_num, iou_thresh, iou_type,
                               target_anchors, batch_divisor, workspace, ignore_out=ignore_out)
  return (loss, parts) if return_parts else loss


def GetLossFromBoxesAndGrad(classes, boxes, offsets, y_pred, image_wh, anchors_wh, classes_num, iou_thresh=0.5, iou_type='iou',
                            target_anchors=None, batch_divisor=None, return_parts=False, workspace=None,
                            grad_dtype=torch.float32, grad_scale=None):
  '''GetLossFromBoxes plus d loss / d y_pred (list of 3 tensors shaped like y_pred) for an upstream gradient of 1: the
  training step of the sparse-target path.  Gradients bit-identical to
  GetLossAndGrad(DataGenerator(classes_num, target_anchors, image_wh).GetTargetsBatch(classes, boxes, offsets), y_pred, ...).
  Returns (loss, grads), or (loss, parts, grads) with return_parts.

  Data parallel: each rank passes its own images with batch_divisor = the global batch.  The gradients need no exchange;
  the (3,4) parts go through combine_loss_parts (or any all-reduce + b200_yolo_loss_combine) for the global loss.
  Wrap with tf.custom_gradient (INTEGRATION.md §3).

  Mixed precision: y_pred levels that are all bf16 or all fp16 are read in place.  grad_dtype (torch.float32, the
  default, torch.bfloat16 or torch.float16) is the type the gradients are written in, each element rounded once from
  g * grad_scale, where g is the fp32 gradient of the call on y.float().  grad_scale: None (no multiply), a 1-element
  float32 tensor on the device (e.g. a loss scale that changes between steps: no host synchronisation, graph
  capturable) or a Python float.'''
  assert iou_type in ['iou','diou','ciou']
  loss, parts, grads = _boxes_call(classes, boxes, offsets, y_pred, image_wh, anchors_wh, classes_num, iou_thresh, iou_type,
                                   target_anchors, batch_divisor, workspace, with_grad=True, grad_dtype=grad_dtype,
                                   grad_scale=grad_scale)
  return (loss, parts, grads) if return_parts else (loss, grads)


def _boxes_call(classes, boxes, offsets, y_pred, image_wh, anchors_wh, classes_num, iou_thresh, iou_type, target_anchors,
                batch_divisor, workspace, ignore_out=None, with_grad=False, grad_dtype=torch.float32, grad_scale=None):
  '''Argument checks and marshalling of the sparse-target entries.  Returns (loss, parts, grads or None).'''
  lib = _lib.load()
  if with_grad:
    T.grad_code(grad_dtype)
  yp, pdt = _pred_levels(y_pred, with_grad)
  boxes = T.to_cuda(boxes).reshape(-1, 4)
  classes = T.to_cuda(classes, torch.int32).reshape(-1)
  offsets = T.to_cuda(offsets, torch.int32).reshape(-1)
  anc = T.host_floats(anchors_wh)
  if anc.size % 6 != 0:
    raise ValueError('anchors_wh must be (3, anchors_num, 2)')
  tanc = anc if target_anchors is None else T.host_floats(target_anchors)
  if tanc.size != anc.size:
    raise ValueError('target_anchors must have the shape of anchors_wh')
  A = anc.size // 6
  B = offsets.numel() - 1
  RF = 5 + int(classes_num)
  for l in range(3):
    if yp[l].dim() < 3 or yp[l].shape[0] != B or yp[l].numel() != B * yp[l].shape[1] * yp[l].shape[2] * A * RF:
      raise ValueError('y_pred[%d] must be (B,H,W,%d*(5+C)) with B = len(offsets)-1' % (l, A))
  img = T.host_floats(image_wh, 2)
  dev = boxes.device
  hw = (ctypes.c_int32 * 6)(*[d for t in yp for d in (t.shape[1], t.shape[2])])
  pp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in yp])
  parts = torch.empty((3, 4), dtype=torch.float32, device=dev)
  loss = torch.empty((), dtype=torch.float32, device=dev)
  total = int(boxes.shape[0])
  ws_bytes = lib.b200_yolo_loss_from_boxes_workspace_bytes(hw, B, A, total)
  if workspace is None or workspace.numel() < ws_bytes:
    workspace = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
  div = float(B if batch_divisor is None else batch_divisor)
  if with_grad:
    grads, gdt, scale = T.grad_out(yp, grad_dtype, grad_scale)
    gp = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in grads])
    _lib.check(lib.b200_yolo_loss_from_boxes_grad_typed(T.ptr(boxes), T.ptr(classes), T.ptr(offsets), total,
                                                        tanc.ctypes.data_as(ctypes.c_void_p), pp, pdt, hw, B, A, RF - 5,
                                                        anc.ctypes.data_as(ctypes.c_void_p), img.ctypes.data_as(ctypes.c_void_p),
                                                        float(iou_thresh), _lib.METRIC_YOLO[iou_type], 0, div, T.ptr(parts),
                                                        T.ptr(loss), gp, gdt, T.ptr(scale), T.ptr(workspace), workspace.numel(),
                                                        T.stream_ptr()), 'GetLossFromBoxesAndGrad')
    return loss, parts, grads
  _lib.check(lib.b200_yolo_loss_from_boxes_typed(T.ptr(boxes), T.ptr(classes), T.ptr(offsets), total,
                                                 tanc.ctypes.data_as(ctypes.c_void_p), pp, pdt, hw, B, A, RF - 5,
                                                 anc.ctypes.data_as(ctypes.c_void_p), img.ctypes.data_as(ctypes.c_void_p),
                                                 float(iou_thresh), _lib.METRIC_YOLO[iou_type], 0, div, T.ptr(parts), T.ptr(loss),
                                                 T.ptr(ignore_out), T.ptr(workspace), workspace.numel(), T.stream_ptr()),
             'GetLossFromBoxes')
  return loss, parts, None


_SIDE_STREAMS = {}


def _side_stream(dev):
  key = (dev.type, dev.index)
  if key not in _SIDE_STREAMS:
    _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
  return _SIDE_STREAMS[key]


def LossAndNMSBoxesBatch(y_true, y_pred, image_wh, anchors_wh, classes_num, iou_thresh=0.5, iou_type='iou',
                         confidence_thresh=0.5, scores_thresh=0.3, nms_iou_thresh=0.5, nms_iou_type='iou',
                         max_output_size=NMS_MAX_OUTPUT, global_batch=None, exchange=None, with_classes=True,
                         with_indices=False, loss_anchors_wh=None, workspace=None):
  '''
  GetLoss and GetNMSBoxes on the SAME y_pred (an evaluation step that also reports the loss; BASELINE config 5).  The two
  are independent given y_pred, so they run as two concurrent chains: decode filter -> NMS -> class rows on a second
  stream, object scan -> GT preparation -> ignore mask / terms -> finalize (+ the data-parallel exchange) on the
  current one.  The persistent decode filter (one CTA per SM, issue-bound) and the latency-bound loss kernels share the
  SMs, and the per-image NMS CTAs run beside the loss instead of behind it.  CUDA-graph capturable (the fork / join
  become graph branches).  Returns (loss, dict as GetNMSBoxesBatch).

  loss_anchors_wh: the anchors GetLoss takes when they differ in units from the ones GetNMSBoxes takes (default: the same).
  '''
  assert iou_type in ['iou','diou','ciou'] and nms_iou_type in ['iou','diou','ciou']
  heads, _ = T.to_cuda_heads(y_pred)   # bf16 / fp16 heads stay in their type for both branches
  dev = heads[0].device
  main = torch.cuda.current_stream(dev)
  side = _side_stream(dev)
  side.wait_stream(main)
  with torch.cuda.stream(side):
    r = GetNMSBoxesBatch(heads[0], heads[1], heads[2], anchors_wh, image_wh, classes_num, confidence_thresh, scores_thresh,
                         nms_iou_thresh, nms_iou_type, max_output_size, with_classes, with_indices)
  B = heads[0].shape[0]
  loss = _loss_call(y_true, heads, image_wh, anchors_wh if loss_anchors_wh is None else loss_anchors_wh, iou_thresh, iou_type, 0,
                    batch_divisor=B if global_batch is None else global_batch, workspace=workspace, exchange=exchange)
  main.wait_stream(side)
  for t in r.values():
    t.record_stream(main)   # allocated on the side stream, consumed by the caller on the current one
  return loss, r


def GetGroudTruthFromBoxes(classes, boxes, offsets, image_wh, anchors_wh, classes_num):
  '''GetGroudTruth of the three levels DataGenerator(classes_num, anchors_wh, image_wh).GetTargetsBatch(classes, boxes,
  offsets) would write, without the dense targets (an API extension).  classes [total] int, boxes [total,4] pixel corners
  x1,y1,x2,y2, offsets [B+1]; anchors_wh as DataGenerator takes them.  Returns (rows [total,5], count [B] int32): the rows
  of image b are rows[offsets[b] : offsets[b] + count[b]], bit-identical to
  torch.cat([GetGroudTruth(t[b]) for t in GetTargetsBatch(...)]); the rest of its range is zero.  No host
  synchronisation.'''
  lib = _lib.load()
  boxes = T.to_cuda(boxes).reshape(-1, 4)
  if boxes.data_ptr() % 16:
    boxes = boxes.clone()   # one 16-byte load per box
  classes = T.to_cuda(classes, torch.int32).reshape(-1)
  offsets = T.to_cuda(offsets, torch.int32).reshape(-1)
  if classes.numel() != boxes.shape[0]:
    raise ValueError('%d boxes but %d classes' % (boxes.shape[0], classes.numel()))
  anc = T.host_floats(anchors_wh)
  if anc.size % 6 != 0:
    raise ValueError('anchors_wh must be (3, anchors_num, 2)')
  img = T.host_floats(image_wh, 2)
  w, h = int(img[0]), int(img[1])
  hw = (ctypes.c_int32 * 6)(*[d for s in (32, 16, 8) for d in (h // s, w // s)])   # DataGenerator.layers_hw
  B, total, dev = offsets.numel() - 1, int(boxes.shape[0]), boxes.device
  if B < 0:
    raise ValueError('offsets must hold B + 1 entries')
  rows = torch.zeros((total, 5), dtype=torch.float32, device=dev)
  count = torch.empty((B,), dtype=torch.int32, device=dev)
  ws_bytes = lib.b200_yolo_ground_truth_from_boxes_workspace_bytes(hw, B, anc.size // 6, total)
  ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev)
  _lib.check(lib.b200_yolo_ground_truth_from_boxes(T.ptr(boxes), T.ptr(classes), T.ptr(offsets), total, B, hw, anc.size // 6,
                                                   int(classes_num), anc.ctypes.data_as(ctypes.c_void_p),
                                                   img.ctypes.data_as(ctypes.c_void_p), T.ptr(rows), T.ptr(count), T.ptr(ws),
                                                   ws_bytes, T.stream_ptr()), 'GetGroudTruthFromBoxes')
  return rows, count


def EvalStepFromBoxes(classes, boxes, offsets, y_pred, image_wh, anchors_wh, classes_num, iou_thresh=0.5, iou_type='iou',
                      confidence_thresh=0.5, scores_thresh=0.3, nms_iou_thresh=0.5, nms_iou_type='iou',
                      max_output_size=NMS_MAX_OUTPUT, target_anchors=None, batch_divisor=None, map_thresh=0.5,
                      with_classes=True, with_indices=False, return_parts=False, workspace=None):
  '''test_step (yolo_v4/model.py:341-378) from box lists, with no dense y_true and no host synchronisation (an API
  extension): GetLossFromBoxes and GetNMSBoxesBatch on the same y_pred as the two stream branches of LossAndNMSBoxesBatch
  (the loss branch also builds GetGroudTruthFromBoxes' rows), then Get_mAP_padded of the NMS output against those rows.
  Arguments: GetLossFromBoxes' (target_anchors = the anchors DataGenerator takes, default anchors_wh) and
  LossAndNMSBoxesBatch's thresholds.  Returns (loss, dict as GetNMSBoxesBatch, mAP float64 [B]); with return_parts
  (loss, parts, dict, mAP).  Data parallel: as GetLossFromBoxes — batch_divisor = the global batch, parts combined with
  combine_loss_parts; the mAP is per image and needs no exchange.  CUDA-graph capturable.'''
  from .mAP import Get_mAP_padded
  assert iou_type in ['iou','diou','ciou'] and nms_iou_type in ['iou','diou','ciou']
  heads, _ = T.to_cuda_heads(y_pred)   # bf16 / fp16 heads stay in their type for both branches
  dev = heads[0].device
  main = torch.cuda.current_stream(dev)
  side = _side_stream(dev)
  side.wait_stream(main)
  with torch.cuda.stream(side):
    r = GetNMSBoxesBatch(heads[0], heads[1], heads[2], anchors_wh, image_wh, classes_num, confidence_thresh, scores_thresh,
                         nms_iou_thresh, nms_iou_type, max_output_size, with_classes, with_indices)
  loss, parts, _ = _boxes_call(classes, boxes, offsets, heads, image_wh, anchors_wh, classes_num, iou_thresh, iou_type,
                               target_anchors, batch_divisor, workspace)
  rows, count = GetGroudTruthFromBoxes(classes, boxes, offsets, image_wh,
                                       anchors_wh if target_anchors is None else target_anchors, classes_num)
  main.wait_stream(side)
  for t in r.values():
    t.record_stream(main)   # allocated on the side stream, consumed on the current one
  m_ap = Get_mAP_padded(rows[:, :4], rows[:, 4].to(torch.int32), offsets, r, classes_num, map_thresh, gt_count=count)
  return (loss, parts, r, m_ap) if return_parts else (loss, r, m_ap)


def GetLossAndGrad(y_true, y_pred, image_wh, anchors_wh, iou_thresh=0.5, iou_type='iou', grad_dtype=torch.float32,
                   grad_scale=None):
  '''GetLoss plus d loss / d y_pred (list of 3 tensors shaped like y_pred) for an upstream gradient of 1 —
  what tf.GradientTape derives from the reference's GetLoss.  Wrap with tf.custom_gradient (INTEGRATION.md §3).
  Mixed precision (bf16 / fp16 y_pred, grad_dtype, grad_scale): as GetLossFromBoxesAndGrad.'''
  assert iou_type in ['iou','diou','ciou']
  loss, _, grads = _loss_call(y_true, y_pred, image_wh, anchors_wh, iou_thresh, iou_type, 0, with_grad=True,
                              grad_dtype=grad_dtype, grad_scale=grad_scale)
  return loss, grads


def combine_loss_parts(parts, group=None):
  '''The multi-GPU exchange step of GetLoss: `parts` (3,4) = per level {xy, wh, obj, cls} already divided by the
  GLOBAL batch on every rank.  One all-reduce(sum) of the 12 floats, then the reference's order of additions
  (tyu:125).  Works on any torch.distributed backend (NCCL on the GPUs, gloo in the CPU tests).'''
  import torch.distributed as dist
  if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
    dist.all_reduce(parts, op=dist.ReduceOp.SUM, group=group)
  per_level = ((parts[:, 0] + parts[:, 1]) + parts[:, 2]) + parts[:, 3]
  return (per_level[0] + per_level[1]) + per_level[2]


def shard_range(batch, rank, world):
  '''Contiguous image range [lo, hi) of `rank` when `batch` images are sharded over `world` ranks.'''
  base, rem = divmod(int(batch), int(world))
  lo = rank * base + min(rank, rem)
  return lo, lo + base + (1 if rank < rem else 0)


def GetLossSharded(y_true, y_pred, image_wh, anchors_wh, iou_thresh=0.5, iou_type='iou', global_batch=None,
                   group=None, exchange=None):
  '''Data-parallel GetLoss: every rank passes its own images; the 12 per-level terms (already divided by the
  global batch) are summed over the ranks and re-added in the reference's order (tyu:120-125).
  exchange = runtime.PeerExchange: the sum happens inside the loss's finalize kernel over NVLink peer stores (no
  collective launch; CUDA-graph capturable); runtime.NcclExchange: b200_allreduce_loss (ncclAllReduce issued by the
  library on the current stream); None: torch.distributed.all_reduce on `group` (any backend, e.g. gloo in CPU tests).'''
  import torch.distributed as dist
  assert iou_type in ['iou','diou','ciou']
  world = exchange.world if exchange is not None else (dist.get_world_size(group) if dist.is_initialized() else 1)
  if global_batch is None:
    global_batch = T.to_cuda(y_true[0]).shape[0] * world
  if exchange is not None:
    return _loss_call(y_true, y_pred, image_wh, anchors_wh, iou_thresh, iou_type, 0, batch_divisor=global_batch,
                      exchange=exchange)
  loss, parts = _loss_call(y_true, y_pred, image_wh, anchors_wh, iou_thresh, iou_type, 0,
                           batch_divisor=global_batch, return_parts=True)
  if world > 1:
    loss = combine_loss_parts(parts, group)
  return loss
