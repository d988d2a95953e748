"""Drop-in for the reference's losses/focal_loss.py (FocalLoss :3-52)."""
import ctypes

import torch

from ... import _lib, _tensors as T


def _pred_heads(pred_boxes, pred_classes):
  '''Box outputs and class logits of the loss (either list may be None or hold None levels) -> (box levels, class levels,
  B200_DTYPE_* code shared by both).  When every given level is bf16, or every one is fp16, the levels stay in their type
  and the kernels read them in place: sums and gradients are those of the call on the widened heads (y.float()).  Any
  other mix, fp32 logits with bf16 boxes included, is cast to fp32.'''
  pb, pc = list(pred_boxes or []), list(pred_classes or [])
  given = [k for k, t in enumerate(pb + pc) if t is not None]
  heads, code = T.to_cuda_heads([(pb + pc)[k] for k in given])
  out = [None] * (len(pb) + len(pc))
  for k, h in zip(given, heads):
    out[k] = h
  return (out[:len(pb)] if pred_boxes is not None else None), (out[len(pb):] if pred_classes is not None else None), code


def _partial_sums(true_boxes, true_classes, true_masks, pred_boxes, pred_classes, alpha, gamma, delta, label_smoothing):
  '''Levels -> device fp64 sums [2L+1] = focal_l..., huber_l..., positives.  Any of the class / box halves may be None.
  Heads: see _pred_heads.'''
  lib = _lib.load()
  L = len(pred_classes) if pred_classes is not None else len(pred_boxes)
  none = [None] * L
  tb = [T.to_cuda(t) if t is not None else None for t in (true_boxes or none)]
  # class targets: one-hot float tensors shaped like the logits, or (sparse-target mode) integer class ids with one
  # entry per anchor
  indexed = true_classes is not None and any(t is not None and not torch.is_floating_point(torch.as_tensor(t)) for t in true_classes)
  tc = [(T.to_cuda(t, torch.int32) if indexed else T.to_cuda(t)) if t is not None else None for t in (true_classes or none)]
  tm = [T.to_cuda(t, torch.bool) if t is not None else None for t in (true_masks or none)]
  pb, pc, pdt = _pred_heads(pred_boxes, pred_classes)
  pb, pc = pb or none, pc or none
  C = next((t.shape[-1] for t in pc if t is not None), 1)
  anchors, numel = [], []
  for l in range(L):
    if pc[l] is not None:
      if indexed:
        if tc[l].numel() * C != pc[l].numel():
          raise ValueError('class id / output shapes differ at level %d' % l)
      elif tc[l].shape != pc[l].shape:
        raise ValueError('class target / output shapes differ at level %d' % l)
      anchors.append(pc[l].numel() // C)
      numel.append(float(pc[l].numel()))
    else:
      anchors.append(pb[l].numel() // 4)
      numel.append(1.0)
    if pb[l] is not None and (tb[l].shape != pb[l].shape or tm[l].numel() != pb[l].numel() // 4):
      raise ValueError('box target / output / mask shapes differ at level %d' % l)
  dev = next(t.device for t in pc + pb if t is not None)
  anc = (ctypes.c_ulonglong * L)(*anchors)
  arr = lambda ts: (ctypes.c_void_p * L)(*[T.ptr(t) for t in ts])
  sums = torch.empty((2 * L + 1,), dtype=torch.float64, device=dev)
  ws_bytes = max(int(lib.b200_focal_box_workspace_bytes(L, anc, max(C, 4))), 256)
  ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
  fn = lib.b200_focal_box_partial_sums_indexed_typed if indexed else lib.b200_focal_box_partial_sums_typed
  _lib.check(fn(L, anc, C, arr(tb), arr(tc), arr(tm), arr(pb), arr(pc), pdt, float(alpha), float(gamma), float(delta),
                float(label_smoothing), T.ptr(sums), T.ptr(ws), ws_bytes, T.stream_ptr()), 'focal/box loss')
  return sums, numel


class FocalLoss(object):
  """Focal loss between `logits` and the golden `target` values: -(1-pt)^gamma * log(pt)."""

  def __init__(self, alpha=0.25, gamma=1.5, label_smoothing=0.0, **kwargs):
    self.alpha = alpha
    self.gamma = gamma
    self.label_smoothing = label_smoothing

  def call(self, y, y_pred):
    """y: (normalizer, y_true).  Returns the per-element tensor alpha_factor * modulating_factor * ce / normalizer."""
    lib = _lib.load()
    normalizer, y_true = y
    yt = T.to_cuda(y_true)
    yp = T.to_cuda(y_pred)
    out = torch.empty_like(yp)
    _lib.check(lib.b200_focal_elementwise(T.ptr(yt), T.ptr(yp), yp.numel(), float(normalizer), float(self.alpha),
                                          float(self.gamma), float(self.label_smoothing), T.ptr(out), T.stream_ptr()),
               'FocalLoss.call')
    return out

  def __call__(self, y, y_pred):
    """keras.losses.Loss.__call__ with the default reduction: mean over every element of `call`'s result."""
    normalizer, y_true = y
    sums, numel = _partial_sums(None, [y_true], None, None, [y_pred], self.alpha, self.gamma, 0.1, self.label_smoothing)
    return (sums[0] / float(normalizer) / numel[0]).to(torch.float32)
