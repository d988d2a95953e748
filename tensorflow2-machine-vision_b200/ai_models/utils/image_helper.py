"""Mirror of the one function of the reference's ImageHelper that sits on the serving path:
opencvProportionalResize (utils/image_helper.py:293-325) — proportional INTER_AREA resize + constant border — on the
device (csrc/letterbox.cu, OpenCV's 8-bit arithmetic bit for bit).  The augmentation options of the reference
(random background colour, BORDER_REPLICATE) are not part of the serving path and are refused.  letterbox_batch is the
same for many frames of mixed sizes in one launch (the batched serving path)."""
import ctypes

import numpy as np
import torch

from ... import _lib, _tensors as T

BORDER_CONSTANT = 0  # cv2.BORDER_CONSTANT


def opencvGetImageSize(opencv_img):
  '''(width, height) of an HxWxC image (image_helper.py:82-86)'''
  return int(opencv_img.shape[1]), int(opencv_img.shape[0])


def _image_on_device(opencv_img):
  T.require_cuda()
  if isinstance(opencv_img, torch.Tensor):
    t = opencv_img
  else:
    t = torch.from_numpy(np.ascontiguousarray(opencv_img))
  if t.dtype != torch.uint8 or t.dim() != 3:
    raise ValueError('expected an HxWx3 uint8 image, got %s %s' % (tuple(t.shape), t.dtype))
  if not t.is_cuda and not (t.is_pinned() and t.is_contiguous()):
    t = t.cuda()  # pageable host memory: one copy; pinned host memory is read in place by the kernel
  return t.contiguous()


def letterbox(opencv_img, size, bg_color, want_u8, want_f32):
  '''One launch of b200_letterbox_image -> (uint8 image or None, float32 RGB/255 image or None, padding, (rw, rh))'''
  lib = _lib.load()
  img = _image_on_device(opencv_img)
  dev = torch.device('cuda', torch.cuda.current_device()) if not img.is_cuda else img.device
  new_width, new_height = int(size[0]), int(size[1])
  out_u8 = torch.empty((new_height, new_width, 3), dtype=torch.uint8, device=dev) if want_u8 else None
  out_f32 = torch.empty((new_height, new_width, 3), dtype=torch.float32, device=dev) if want_f32 else None
  bg = (ctypes.c_uint8 * 3)(*[int(min(max(round(float(v)), 0), 255)) for v in list(bg_color)[:3]])
  padding = (ctypes.c_int32 * 4)()
  resized = (ctypes.c_int32 * 2)()
  _lib.check(lib.b200_letterbox_image(T.ptr(img), int(img.shape[0]), int(img.shape[1]), int(img.shape[2]), new_width, new_height,
                                      bg, T.ptr(out_u8), T.ptr(out_f32), padding, resized, T.stream_ptr()), 'opencvProportionalResize')
  return out_u8, out_f32, tuple(int(v) for v in padding), (int(resized[0]), int(resized[1]))


def _frames_on_device(frames):
  '''-> (tensors to keep alive, frame pointers, [N,2] height,width, channels, device)'''
  T.require_cuda()
  if isinstance(frames, np.ndarray) and frames.ndim == 4:
    frames = torch.from_numpy(np.ascontiguousarray(frames))
  if isinstance(frames, torch.Tensor):  # (N,H,W,C) as a video decoder writes it: frame i starts at base + i*H*W*C
    if frames.dtype != torch.uint8 or frames.dim() != 4:
      raise ValueError('letterbox_batch: expected an (N,H,W,3) uint8 tensor, got %s %s' % (tuple(frames.shape), frames.dtype))
    t = frames
    if not t.is_cuda and not (t.is_pinned() and t.is_contiguous()):
      t = t.cuda()
    t = t.contiguous()
    n, h, w, c = (int(v) for v in t.shape)
    return [t], [t.data_ptr() + i * h * w * c for i in range(n)], [(h, w)] * n, c, t.device if t.is_cuda else None
  keep = []
  for i, f in enumerate(frames):
    try:
      keep.append(_image_on_device(f))
    except ValueError as e:
      raise ValueError('letterbox_batch: frame %d: %s' % (i, e))
  channels = int(keep[0].shape[2]) if keep else 3
  for i, t in enumerate(keep):
    if int(t.shape[2]) != channels:
      raise ValueError('letterbox_batch: frame %d has %d channels, frame 0 has %d' % (i, int(t.shape[2]), channels))
  devs = {t.device for t in keep if t.is_cuda}
  if len(devs) > 1:
    raise ValueError('letterbox_batch: frames on different devices %s' % sorted(str(d) for d in devs))
  return keep, [t.data_ptr() for t in keep], [(int(t.shape[0]), int(t.shape[1])) for t in keep], channels, \
      (devs.pop() if devs else None)


def letterbox_batch(frames, size, bg_color, want_u8, want_f32):
  '''letterbox() for N frames of any sizes: b200_letterbox_batch, one launch per 84 frames.

  Args:
    frames: a list of HxWx3 uint8 images of any sizes (numpy, device tensors, pinned host tensors read in place; mixed),
      or one (N,H,W,3) uint8 tensor as a video decoder writes it
    size: (new_width, new_height)
  Returns:
    (uint8 (N,h,w,3) or None, float32 RGB/255 (N,h,w,3) or None, paddings int32 (N,4), resized (rw, rh) int32 (N,2))
  '''
  return _letterbox_batch(frames, size, bg_color, want_u8, want_f32, False)[:4]


def _letterbox_batch(frames, size, bg_color, want_u8, want_f32, want_geometry):
  '''letterbox_batch + (geometry (N,6) int32 on the device or None, source sizes int32 (N,2) height,width)'''
  lib = _lib.load()
  keep, ptrs, hw, channels, dev = _frames_on_device(frames)
  n = len(ptrs)
  dev = dev or torch.device('cuda', torch.cuda.current_device())
  new_width, new_height = int(size[0]), int(size[1])
  out_u8 = torch.empty((n, new_height, new_width, 3), dtype=torch.uint8, device=dev) if want_u8 else None
  out_f32 = torch.empty((n, new_height, new_width, 3), dtype=torch.float32, device=dev) if want_f32 else None
  geometry = torch.empty((n, 6), dtype=torch.int32, device=dev) if want_geometry else None  # written by the kernel
  bg = (ctypes.c_uint8 * 3)(*[int(min(max(round(float(v)), 0), 255)) for v in list(bg_color)[:3]])
  paddings = np.zeros((n, 4), np.int32)
  resized = np.zeros((n, 2), np.int32)
  c_ptrs = (ctypes.c_void_p * max(n, 1))(*ptrs)
  c_hw = np.ascontiguousarray(np.int32(hw).reshape(n, 2))
  _lib.check(lib.b200_letterbox_batch(n, c_ptrs, c_hw.ctypes.data_as(ctypes.c_void_p), channels, new_width, new_height, bg,
                                      T.ptr(out_u8), T.ptr(out_f32), paddings.ctypes.data_as(ctypes.c_void_p),
                                      resized.ctypes.data_as(ctypes.c_void_p), T.ptr(geometry), T.stream_ptr()),
             'letterbox_batch')
  return out_u8, out_f32, paddings, resized, geometry, c_hw


def opencvProportionalResize(opencv_img, size, points=None, bg_color=(128, 128, 128), bg_mode=BORDER_CONSTANT):
  '''
  Args:
    opencv_img: HxWx3 uint8 (numpy, or a torch tensor on the device / in pinned host memory); size: (new_width, new_height)
    points: optional [[x, y], ...] on the original image
  Returns:
    result_img (new_height,new_width,3) uint8 on the device, result_points float32 (n,2), padding (top,bottom,left,right)
  '''
  if bg_color is None or bg_mode != BORDER_CONSTANT:
    raise NotImplementedError('opencvProportionalResize: only a given colour with BORDER_CONSTANT (the serving path) is built')
  width, height = opencvGetImageSize(opencv_img)
  result_img, _, padding, (resize_width, resize_height) = letterbox(opencv_img, size, bg_color, True, False)
  result_points = []
  if points is not None:
    for p in points:  # image_helper.py:319-323
      result_points.append([p[0] * resize_width / width + padding[2], p[1] * resize_height / height + padding[0]])
  return result_img, np.float32(result_points), padding
