"""Device-memory plumbing for the shims (torch is used for allocation, streams and DLPack only)."""
import numpy as np
import torch


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("tensorflow2-machine-vision_b200 needs a CUDA device (B200); there is no CPU fallback")


def _as_tensor(x):
    """Anything tensor-like -> torch tensor in its own dtype and place (zero-copy for torch/DLPack inputs)."""
    if isinstance(x, torch.Tensor):
        return x
    if hasattr(x, "__dlpack__") and not isinstance(x, np.ndarray):
        return torch.from_dlpack(x)  # e.g. tf.experimental.dlpack / cupy
    t = torch.from_numpy(np.ascontiguousarray(np.asarray(x)))
    return t.pin_memory() if t.numel() > (1 << 16) else t


def to_cuda(x, dtype=torch.float32):
    """Anything tensor-like -> contiguous CUDA tensor of `dtype` (zero-copy for CUDA/DLPack inputs)."""
    require_cuda()
    t = _as_tensor(x)
    if t.dtype != dtype:
        t = t.to(dtype)
    if not t.is_cuda:
        t = t.cuda(non_blocking=True)
    return t.contiguous()


# element-type codes of the C ABI (B200_DTYPE_*) for the head dtypes the post-processing and the losses read in place
DTYPE_F32 = 0
_HALF_CODES = {torch.bfloat16: 1, torch.float16: 2}
DTYPE_CODES = {torch.float32: DTYPE_F32, **_HALF_CODES}


def to_cuda_heads(xs, keep_pinned=False):
    """The levels of one head family (YOLO heads, EfficientDet box tensors or class logits) -> (contiguous CUDA tensors,
    B200_DTYPE_* code).  A family that is all bf16 or all fp16 stays in its type: the kernels widen each element to fp32
    exactly, so the results are those of the fp32 call on the widened tensors, without a cast pass or an fp32 copy.
    Any other family is cast to fp32 as to_cuda does.  keep_pinned: the caller's torch tensors in page-locked host memory
    (is_pinned_host_f32) that already have the family's type are returned as they are, for kernels that read them in
    place."""
    require_cuda()
    ts = [_as_tensor(x) for x in xs]
    code = _HALF_CODES.get(ts[0].dtype) if ts else None
    if code is None or not all(t.dtype == ts[0].dtype for t in ts):
        code = DTYPE_F32
    dtype = ts[0].dtype if code != DTYPE_F32 else torch.float32
    keep = lambda x, t: keep_pinned and t is x and t.dtype == dtype and is_pinned_host_f32(t)
    return [t if keep(x, t) else to_cuda(t, dtype) for x, t in zip(xs, ts)], code


def grad_code(grad_dtype):
    """B200_DTYPE_* code of the gradient dtype of a loss backward call (checked before anything touches the device)."""
    code = DTYPE_CODES.get(grad_dtype)
    if code is None:
        raise ValueError("grad_dtype must be torch.float32, torch.bfloat16 or torch.float16, not %r" % (grad_dtype,))
    return code


def grad_out(heads, grad_dtype, grad_scale):
    """The gradient tensors of a loss backward call (shaped like `heads`, of grad_dtype), their B200_DTYPE_* code and the
    scale tensor (1-element fp32 on the heads' device, or None; a Python float is put there)."""
    code = grad_code(grad_dtype)
    dev = heads[0].device
    if grad_scale is not None and not isinstance(grad_scale, torch.Tensor):
        grad_scale = torch.full((1,), float(grad_scale), dtype=torch.float32, device=dev)
    if grad_scale is not None and (grad_scale.dtype != torch.float32 or grad_scale.numel() != 1 or grad_scale.device != dev):
        raise ValueError("grad_scale must be a 1-element float32 tensor on %s, or a Python float" % dev)
    grads = [torch.empty(t.shape, dtype=grad_dtype, device=dev) for t in heads]
    return grads, code, grad_scale


def is_pinned_host_f32(x):
    """A contiguous fp32, bf16 or fp16 torch tensor in page-locked host memory: device kernels can read it in place (UVA)."""
    return (isinstance(x, torch.Tensor) and not x.is_cuda and x.dtype in DTYPE_CODES and x.is_contiguous()
            and x.is_pinned() and torch.cuda.is_available())


def ptr(t):
    return 0 if t is None else t.data_ptr()


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def host_floats(x, n=None):
    """Small host-side float32 parameter (anchors, image size) as a flat numpy array."""
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    a = np.ascontiguousarray(np.asarray(x, dtype=np.float32)).reshape(-1)
    if n is not None and a.size != n:
        raise ValueError("expected %d values, got %d" % (n, a.size))
    return a
