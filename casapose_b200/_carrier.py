"""Tensor carriers.  The product is the C-ABI library; PyTorch only carries device memory.

`as_cuda_f32` accepts a torch tensor or ANY object exporting ``__dlpack__`` (TensorFlow eager
tensors, CuPy, JAX, ...) and returns a zero-copy torch view of it.  Layout or dtype mismatches are
errors, not silent copies (SURVEY.md section 8b).  `as_cuda_float` also takes the 16-bit network outputs
the *_typed entry points read natively."""
import torch

# casa_dtype codes (include/casapose_b200.h)
DTYPE_CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def as_cuda(x, dtype, name):
    if not isinstance(x, torch.Tensor):
        if hasattr(x, "__dlpack__"):
            x = torch.from_dlpack(x)
        else:
            raise TypeError("%s: expected a torch tensor or a __dlpack__ exporter, got %r" % (name, type(x)))
    if not x.is_cuda:
        raise ValueError("%s must live on a CUDA device (got %s); use the *_host entry point for host buffers" % (name, x.device))
    if x.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, x.dtype))
    if not x.is_contiguous():
        raise ValueError("%s must be C-contiguous (NHWC, like the reference's tensors)" % name)
    return x


def as_cuda_f32(x, name):
    return as_cuda(x, torch.float32, name)


def as_cuda_float(x, name):
    """Like as_cuda_f32, for a float32, float16 or bfloat16 tensor: returns (tensor, casa_dtype code)."""
    if not isinstance(x, torch.Tensor) and hasattr(x, "__dlpack__"):
        x = torch.from_dlpack(x)
    if isinstance(x, torch.Tensor) and x.dtype in DTYPE_CODES:
        return as_cuda(x, x.dtype, name), DTYPE_CODES[x.dtype]
    if isinstance(x, torch.Tensor) and x.is_cuda:
        raise TypeError("%s must be float32, float16 or bfloat16, got %s" % (name, x.dtype))
    return as_cuda(x, torch.float32, name), 0  # raises: not a tensor, not on a device, or another dtype


def ptr(t):
    return None if t is None else t.data_ptr()


def current_stream_ptr(device):
    return torch.cuda.current_stream(device).cuda_stream
