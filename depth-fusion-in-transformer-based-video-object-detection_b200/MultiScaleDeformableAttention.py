"""Drop-in for the reference's native extension module ``MultiScaleDeformableAttention``.

The reference builds a pybind module of this name exporting exactly two functions
(/root/reference/models/ops/src/vision.cpp:13-16) and imports it as ``MSDA``
(models/ops/functions/ms_deform_attn_func.py:18).  This module exports the same two
functions with the same positional signatures, argument checks and error behaviour
(models/ops/src/ms_deform_attn.h:20-61, cuda/ms_deform_attn_cuda.cu:20-153), and forwards to
the hand-written sm_100a kernels in libmsda_b200.so through the C ABI of
include/msda_b200.h.  torch is used only for device memory and the current stream.

Deviations from the reference, all deliberate (DESIGN.md "Boundary"):
  * bf16 / fp16 ``value`` is accepted (reference: fp32/fp64 only, cu:64); locations and
    attention weights are then taken in fp32;
  * ``sampling_loc`` / ``attn_weight`` shapes are validated against ``spatial_shapes`` -- the
    reference silently mis-indexes on a level-count mismatch (SURVEY.md section 9.1);
  * kernel launch failures raise instead of being printf'ed (cuh:948-952);
  * the batch is processed in one launch; ``im2col_step`` only keeps its divisibility check
    (cu:50-52);
  * under ``torch.use_deterministic_algorithms(True)`` the backward runs ``msda_backward_deterministic``
    (fixed-point accumulation of grad_value, bitwise reproducible; DESIGN.md section 3.15).
"""
import torch

from . import _lib

_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.float64: _lib.DTYPE_F64,
           torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16}

# test hook: route through the shape-generic kernels
_FORCE_GENERIC = False
def _check_inputs(named, im2col_step):
    value = named[0][1]
    if not value.is_cuda:
        raise RuntimeError("Not implemented on the CPU")                      # ms_deform_attn.h:38,60
    for name, t in named:
        if not t.is_contiguous():
            raise RuntimeError(f"{name} tensor has to be contiguous")         # cu:28-32,93-98
    for name, t in named:
        if not t.is_cuda:
            raise RuntimeError(f"{name} must be a CUDA tensor")               # cu:34-38,100-105
        if t.device != value.device:
            raise RuntimeError(f"{name} must be on the same device as value")
    batch = value.size(0)
    step = min(batch, int(im2col_step))
    if batch > 0 and (step <= 0 or batch % step != 0):
        raise RuntimeError(f"batch({batch}) must divide im2col_step({step})")  # cu:50-52


def _geometry(value, spatial_shapes, level_start_index, sampling_loc, attn_weight):
    if value.dim() != 4 or sampling_loc.dim() != 6 or attn_weight.dim() != 5:
        raise RuntimeError("expected value [N,S,M,D], sampling_loc [N,Lq,M,L,P,2], attn_weight [N,Lq,M,L,P]")
    n, s, m, d = value.shape
    nl = spatial_shapes.size(0)
    lq, p = sampling_loc.size(1), sampling_loc.size(4)
    if spatial_shapes.dtype != torch.int64 or level_start_index.dtype != torch.int64:
        raise RuntimeError("spatial_shapes and level_start_index must be int64 (torch.long)")
    if tuple(spatial_shapes.shape) != (nl, 2) or tuple(level_start_index.shape) != (nl,):
        raise RuntimeError("spatial_shapes must be [L,2] and level_start_index [L]")
    if tuple(sampling_loc.shape) != (n, lq, m, nl, p, 2):
        raise RuntimeError(f"sampling_loc shape {tuple(sampling_loc.shape)} does not match "
                           f"(N={n}, Lq={lq}, M={m}, L={nl}, P={p}, 2)")
    if tuple(attn_weight.shape) != (n, lq, m, nl, p):
        raise RuntimeError(f"attn_weight shape {tuple(attn_weight.shape)} does not match "
                           f"(N={n}, Lq={lq}, M={m}, L={nl}, P={p})")
    return n, s, m, d, nl, lq, p


def _side_dtype(value):
    if value.dtype not in _DTYPES:
        raise RuntimeError(f'"ms_deform_attn" not implemented for \'{value.dtype}\'')
    return torch.float64 if value.dtype == torch.float64 else torch.float32


def ms_deform_attn_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step):
    """-> output [N, Lq, M*D].  Mirrors ms_deform_attn_forward (ms_deform_attn.h:20-39)."""
    _check_inputs([("value", value), ("spatial_shapes", spatial_shapes),
                   ("level_start_index", level_start_index), ("sampling_loc", sampling_loc),
                   ("attn_weight", attn_weight)], im2col_step)
    n, s, m, d, nl, lq, p = _geometry(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)
    side = _side_dtype(value)
    if sampling_loc.dtype != side:
        sampling_loc = sampling_loc.to(side)
    if attn_weight.dtype != side:
        attn_weight = attn_weight.to(side)
    lib = _lib.load()
    with torch.cuda.device(value.device):
        output = torch.empty((n, lq, m * d), dtype=value.dtype, device=value.device)
        code = lib.msda_forward(
            _DTYPES[value.dtype], value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
            sampling_loc.data_ptr(), attn_weight.data_ptr(), n, s, m, d, nl, lq, p, output.data_ptr(),
            _lib.FLAG_FORCE_GENERIC if _FORCE_GENERIC else 0, torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "ms_deform_attn_forward")
    return output


def ms_deform_attn_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output,
                            im2col_step):
    """-> [grad_value, grad_sampling_loc, grad_attn_weight].  Mirrors ms_deform_attn_backward
    (ms_deform_attn.h:41-61)."""
    _check_inputs([("value", value), ("spatial_shapes", spatial_shapes),
                   ("level_start_index", level_start_index), ("sampling_loc", sampling_loc),
                   ("attn_weight", attn_weight), ("grad_output", grad_output)], im2col_step)
    n, s, m, d, nl, lq, p = _geometry(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)
    if grad_output.numel() != n * lq * m * d or grad_output.dtype != value.dtype:
        raise RuntimeError("grad_output must be [N, Lq, M*D] with the dtype of value")
    side = _side_dtype(value)
    loc_dtype, attn_dtype = sampling_loc.dtype, attn_weight.dtype
    if loc_dtype != side:
        sampling_loc = sampling_loc.to(side)
    if attn_dtype != side:
        attn_weight = attn_weight.to(side)
    lib = _lib.load()
    with torch.cuda.device(value.device):
        grad_value = torch.empty_like(value)
        grad_loc = torch.empty_like(sampling_loc)
        grad_attn = torch.empty_like(attn_weight)
        args = (_DTYPES[value.dtype], grad_output.data_ptr(), value.data_ptr(), spatial_shapes.data_ptr(),
                level_start_index.data_ptr(), sampling_loc.data_ptr(), attn_weight.data_ptr(),
                n, s, m, d, nl, lq, p, grad_value.data_ptr(), grad_loc.data_ptr(), grad_attn.data_ptr())
        flags = _lib.FLAG_FORCE_GENERIC if _FORCE_GENERIC else 0
        stream = torch.cuda.current_stream().cuda_stream
        if torch.are_deterministic_algorithms_enabled():
            scratch = _lib.deterministic_scratch(value.device, value.numel())
            code = lib.msda_backward_deterministic(*args, None, flags, scratch.data_ptr(), scratch.numel(), stream)
        else:
            accum = None
            if value.dtype in (torch.bfloat16, torch.float16):
                accum = torch.empty(value.shape, dtype=torch.float32, device=value.device)
            code = lib.msda_backward(*args, accum.data_ptr() if accum is not None else None, flags, stream)
    _lib.check(code, "ms_deform_attn_backward")
    if grad_loc.dtype != loc_dtype:
        grad_loc = grad_loc.to(loc_dtype)
    if grad_attn.dtype != attn_dtype:
        grad_attn = grad_attn.to(attn_dtype)
    return [grad_value, grad_loc, grad_attn]
