"""Drop-in for the reference's utils/mAP.py (Get_mAP_one :114-125), the evaluation step right after NMS in
test_step (yolo_v4/model.py:377, efficientnet/efficientdet_net_train.py:166)."""
import numpy as np
import torch

from ... import _lib, _tensors as T


def Get_mAP_batch(groud_truth, gt_offsets, prediction, pred_offsets, class_num, thresh=0.5):
  '''Per-image mAP for a batch: groud_truth [total,5] (x1,y1,x2,y2,class), prediction [total,6]
  (x1,y1,x2,y2,class,score), offsets [B+1].  Returns a float64 tensor [B].'''
  lib = _lib.load()
  gt = T.to_cuda(groud_truth).reshape(-1, 5)
  pr = T.to_cuda(prediction).reshape(-1, 6)
  go = np.asarray(gt_offsets.cpu() if isinstance(gt_offsets, torch.Tensor) else gt_offsets, dtype=np.int32).reshape(-1)
  po = np.asarray(pred_offsets.cpu() if isinstance(pred_offsets, torch.Tensor) else pred_offsets, dtype=np.int32).reshape(-1)
  B = go.size - 1
  out = torch.zeros((B,), dtype=torch.float64, device=gt.device)
  max_g = int(np.max(np.diff(go))) if B else 0
  max_p = int(np.max(np.diff(po))) if B else 0
  dgo, dpo = T.to_cuda(go, torch.int32), T.to_cuda(po, torch.int32)
  _lib.check(lib.b200_map_per_image(T.ptr(gt), T.ptr(dgo), T.ptr(pr), T.ptr(dpo), B, max_g, max_p, int(class_num),
                                    float(thresh), T.ptr(out), T.stream_ptr()), 'Get_mAP_one')
  return out


def Get_mAP_one(groud_truth, prediction, class_num, thresh=0.5):
  '''mAP of one image (float64 scalar tensor): groud_truth (n,5), prediction (m,6).'''
  n = T.to_cuda(groud_truth).reshape(-1, 5).shape[0]
  m = T.to_cuda(prediction).reshape(-1, 6).shape[0]
  return Get_mAP_batch(groud_truth, [0, n], prediction, [0, m], class_num, thresh)[0]


def Get_mAP_padded(gt_boxes, gt_classes, gt_offsets, nms, class_num, thresh=0.5, gt_count=None):
  '''Per-image mAP straight from the padded NMS output, without a host round trip (graph-capturable).

  nms: the dict GetNMSBoxesBatch / Anchors.convert_outputs_batch / Anchors.eval_step return — boxes [B,K,4],
  classes_id [B,K] (int32 or int64), scores [B,K], count [B] on the device.  Ground truth as box lists: gt_boxes
  [total,4] in the corner order of the predicted boxes, gt_classes [total], gt_offsets [B+1]; image b uses rows
  gt_offsets[b] .. gt_offsets[b] + gt_count[b] (gt_count [B], or None for the whole range).  Same arithmetic as
  Get_mAP_batch; returns a float64 tensor [B].'''
  lib = _lib.load()
  boxes, scores = T.to_cuda(nms['boxes']), T.to_cuda(nms['scores'])
  cls = nms['classes_id']
  cls = T.to_cuda(cls, torch.int64 if getattr(cls, 'dtype', None) == torch.int64 else torch.int32)
  count = T.to_cuda(nms['count'], torch.int32).reshape(-1)
  B = count.numel()
  if boxes.dim() != 3 or boxes.shape[0] != B or boxes.shape[2] != 4:
    raise ValueError('nms boxes must be [B,K,4] with B = count.numel() = %d, got %r' % (B, tuple(boxes.shape)))
  K = boxes.shape[1]
  if tuple(cls.shape) != (B, K) or tuple(scores.shape) != (B, K):
    raise ValueError('nms classes_id / scores must be [%d,%d], got %r / %r' % (B, K, tuple(cls.shape), tuple(scores.shape)))
  gb = T.to_cuda(gt_boxes).reshape(-1, 4)
  gc = T.to_cuda(gt_classes, torch.int32).reshape(-1)
  go = T.to_cuda(gt_offsets, torch.int32).reshape(-1)
  if gc.numel() != gb.shape[0]:
    raise ValueError('%d ground-truth boxes but %d classes' % (gb.shape[0], gc.numel()))
  if go.numel() != B + 1:
    raise ValueError('gt_offsets must hold B + 1 = %d entries, got %d' % (B + 1, go.numel()))
  gn = None
  if gt_count is not None:
    gn = T.to_cuda(gt_count, torch.int32).reshape(-1)
    if gn.numel() != B:
      raise ValueError('gt_count must hold B = %d entries, got %d' % (B, gn.numel()))
  out = torch.empty((B,), dtype=torch.float64, device=boxes.device)
  _lib.check(lib.b200_map_padded(T.ptr(boxes), T.ptr(cls), cls.element_size(), T.ptr(scores), T.ptr(count), B, K, T.ptr(gb),
                                 T.ptr(gc), gb.shape[0], T.ptr(go), T.ptr(gn), int(class_num), float(thresh), T.ptr(out), T.stream_ptr()),
             'Get_mAP_padded')
  return out
