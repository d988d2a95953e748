"""The image plumbing of the reference's serving view (views/object_detection.py:46-85, inline code of `predict`) as
two functions around model.Predict:
  prepare_image        letterbox on black (opencvProportionalResize), BGR->RGB, float32 / 255, batch axis (:50-62)
  restore_predictions  map Predict's normalised boxes on the letterboxed input back to pixels of the original image,
                       clip, drop boxes not larger than 2 px, truncate to int32, filter the other outputs alike (:70-85)
and their batched forms for N frames of mixed sizes, each one launch (per 84 frames for the letterbox) whatever N is:
  prepare_images             -> (N,h,w,3) network input + per-frame geometry on the device
  restore_predictions_batch  GetNMSBoxesBatch's padded output -> pixel boxes of every frame, padded alike
Decoded frames -> prepare_images -> backbone -> GetNMSBoxesBatch -> restore_predictions_batch can be captured as one
CUDA graph; a replay then expects frames of the sizes it was captured with (the per-frame plans are kernel arguments).
"""
import ctypes

import numpy as np
import torch

from .. import _lib, _tensors as T
from ..ai_models.utils import image_helper


def prepare_image(img_old, image_size=(416, 416)):
  '''
  Args:
    img_old: HxWx3 uint8 BGR image as cv2 decodes it (numpy / device tensor / pinned host tensor)
    image_size: (w,h) of the network input
  Returns:
    predict_img (1,h,w,3) float32 RGB in [0,1] on the device, padding (top,bottom,left,right), image_size_old int32 (w,h)
  '''
  width, height = image_helper.opencvGetImageSize(img_old)
  _, img, padding, _ = image_helper.letterbox(img_old, image_size, (0, 0, 0), False, True)
  return img[None], padding, np.int32([width, height])


def restore_predictions(y_boxes, y_classes_id, y_scores, y_classes, y_confidence, image_size, padding, image_size_old):
  '''
  Args (one image, as Predict returns them):
    y_boxes (n,4) normalised x1,y1,x2,y2; y_classes_id (n,); y_scores (n,); y_classes (n,C); y_confidence (n,1)
    image_size: (w,h) of the network input; padding: (top,bottom,left,right) from opencvProportionalResize;
    image_size_old: (w,h) of the original image
  Returns:
    y_boxes (k,4) int32 pixels, y_classes_id (k,), y_scores (k,), y_classes (k,C), y_confidence (k,1)
  '''
  lib = _lib.load()
  boxes = T.to_cuda(y_boxes).reshape(-1, 4)
  n = boxes.shape[0]
  dev = boxes.device
  out_boxes = torch.empty((max(n, 1), 4), dtype=torch.int32, device=dev)
  out_index = torch.empty((max(n, 1),), dtype=torch.int32, device=dev)
  out_count = torch.zeros((1,), dtype=torch.int32, device=dev)
  i2 = lambda v, k: (ctypes.c_int32 * k)(*[int(x) for x in np.asarray(v).reshape(-1)[:k]])
  _lib.check(lib.b200_unletterbox_boxes(T.ptr(boxes), None, 1, n, i2(image_size, 2), i2(padding, 4), i2(image_size_old, 2),
                                        T.ptr(out_boxes), T.ptr(out_index), T.ptr(out_count), T.stream_ptr()), 'restore_predictions')
  k = int(out_count.item())
  idx = out_index[:k].long()
  take = lambda t: t if t is None else (t if isinstance(t, torch.Tensor) else torch.as_tensor(np.asarray(t))).to(dev)[idx]
  return out_boxes[:k], take(y_classes_id), take(y_scores), take(y_classes), take(y_confidence)


def prepare_images(frames, image_size=(416, 416)):
  '''
  Batched prepare_image.
  Args:
    frames: list of HxWx3 uint8 BGR images of any sizes (numpy / device / pinned host tensors), or one (N,H,W,3) tensor
    image_size: (w,h) of the network input
  Returns:
    predict_imgs (N,h,w,3) float32 RGB in [0,1] on the device, paddings (N,4) int32 (top,bottom,left,right),
    image_sizes_old (N,2) int32 (w,h), geometry (N,6) int32 on the device (paddings then (w,h): restore_predictions_batch)
  '''
  _, imgs, paddings, _, geometry, hw = image_helper._letterbox_batch(frames, image_size, (0, 0, 0), False, True, True)
  return imgs, paddings, np.ascontiguousarray(hw[:, ::-1]), geometry


def restore_predictions_batch(nms, image_size, geometry):
  '''
  Batched restore_predictions.
  Args:
    nms: the dict GetNMSBoxesBatch returns (boxes [B,K,4], count [B], classes_id, scores, classes (optional), confidence)
    image_size: (w,h) of the network input; geometry: (B,6) int32 device tensor from prepare_images
  Returns:
    dict of padded tensors: boxes [B,K,4] int32 pixels, count [B] int32, classes_id, scores, classes (when given) and
    confidence gathered alike; row b cut to count[b] is restore_predictions of image b.  Rows past count are unspecified.
  '''
  lib = _lib.load()
  boxes = T.to_cuda(nms['boxes'])
  B, K = int(boxes.shape[0]), int(boxes.shape[1])
  dev = boxes.device
  counts = T.to_cuda(nms['count'], torch.int32)
  geometry = T.to_cuda(geometry, torch.int32)
  if tuple(geometry.shape) != (B, 6):
    raise ValueError('restore_predictions_batch: geometry must be (%d, 6), got %s' % (B, tuple(geometry.shape)))
  out_boxes = torch.empty((B, K, 4), dtype=torch.int32, device=dev)
  out_index = torch.zeros((B, K), dtype=torch.int32, device=dev)   # rows past count gather row 0
  out_count = torch.empty((B,), dtype=torch.int32, device=dev)
  size = (ctypes.c_int32 * 2)(*[int(x) for x in np.asarray(image_size).reshape(-1)[:2]])
  _lib.check(lib.b200_unletterbox_boxes_batch(T.ptr(boxes), T.ptr(counts), B, K, size, T.ptr(geometry), T.ptr(out_boxes),
                                              T.ptr(out_index), T.ptr(out_count), T.stream_ptr()), 'restore_predictions_batch')
  idx = out_index.long()
  out = {'boxes': out_boxes, 'count': out_count}
  for key in ('classes_id', 'scores', 'classes', 'confidence'):
    t = nms.get(key)
    if t is not None:
      out[key] = torch.take_along_dim(t, idx.view((B, K) + (1,) * (t.dim() - 2)), dim=1)
  return out
