"""Autograd binding of the FUSED layer op (C ABI msda_fused_forward / msda_fused_backward).

One kernel per direction replaces, inside ``MSDeformAttn.forward``, the reference's chain
    softmax(attention_weights(query))                       ms_deform_attn.py:99-100
    reference_points + sampling_offsets(query) / normaliser :102-110
    MSDeformAttnFunction.apply(...)                         :114
so the sampling locations [N,Lq,M,L,P,2] and attention weights [N,Lq,M,L,P] (and their
gradients) are never written to HBM.  ``raw`` is the output of ONE projection GEMM whose rows are
``[ sampling offsets (M*L*P*2) | attention logits (M*L*P) ]``.
Under ``torch.use_deterministic_algorithms(True)`` the backward runs ``msda_fused_backward_deterministic``
(bitwise reproducible gradients; DESIGN.md section 3.15).
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from ... import _lib
from ... import MultiScaleDeformableAttention as _msda

_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16}


def fused_supported(value, raw, ref_dim, n_levels, n_points):
    """True when the fused kernels cover this call (else use the unfused op)."""
    if not (value.is_cuda and raw.is_cuda) or value.dtype not in _DTYPES or raw.dtype not in _DTYPES:
        return False
    if value.dtype == torch.float32 and raw.dtype != torch.float32:
        return False
    _, s, m, d = value.shape
    return bool(_lib.load().msda_fused_supported(_DTYPES[value.dtype], _DTYPES[raw.dtype], int(ref_dim), int(s),
                                                 int(m), int(d), int(n_levels), int(n_points)))


def _pixel_strided(value):
    """Pixel stride (elements) of a [N,S,M,D] value view whose pixels are dense rows of M*D elements spaced evenly
    -- a column slice of a wider projection output -- or 0 when the view is not of that form."""
    n, s, m, d = value.shape
    ld = value.stride(1)
    if value.stride(3) != 1 or value.stride(2) != d or ld < m * d or (n > 1 and value.stride(0) != s * ld):
        return 0
    vec = 16 // value.element_size()
    if ld % vec != 0 or value.data_ptr() % 16 != 0 or s * ld >= 2 ** 31:
        return 0
    return ld


def _aligned(t, nbytes=16):
    return t if t.data_ptr() % nbytes == 0 else t.clone()


class MSDeformAttnFusedFunction(Function):
    """apply(value[N,S,M,D], spatial_shapes[L,2], level_start_index[L], reference_points[N,Lq,L,2|4],
             raw[N,Lq,3*M*L*P], n_points) -> [N, Lq, M*D]
    Differentiable w.r.t. value, reference_points and raw."""

    @staticmethod
    def forward(ctx, value, spatial_shapes, level_start_index, reference_points, raw, n_points):
        n, s, m, d = value.shape
        nl = spatial_shapes.size(0)
        lq = raw.size(1)
        p = int(n_points)
        mlp = m * nl * p
        if raw.size(-1) != 3 * mlp or raw.size(0) != n:
            raise RuntimeError(f"raw must be [N, Lq, 3*M*L*P={3 * mlp}], got {tuple(raw.shape)}")
        if tuple(reference_points.shape[:3]) != (n, lq, nl) or reference_points.size(-1) not in (2, 4):
            raise RuntimeError(f"reference_points must be [N={n}, Lq={lq}, L={nl}, 2|4], got "
                               f"{tuple(reference_points.shape)}")
        if spatial_shapes.dtype != torch.int64 or level_start_index.dtype != torch.int64:
            raise RuntimeError("spatial_shapes and level_start_index must be int64 (torch.long)")
        # a strided column slice is read in place when no gradient will be asked for (backward needs it dense)
        ld = 0
        if not value.is_contiguous() and not any(ctx.needs_input_grad):
            ld = _pixel_strided(value)
        if ld == 0:
            value = _aligned(value.contiguous())
        raw = _aligned(raw.contiguous())
        ref = _aligned(reference_points.detach().to(torch.float32).contiguous())
        spatial_shapes = spatial_shapes.contiguous()
        level_start_index = level_start_index.contiguous()
        lib = _lib.load()
        with torch.cuda.device(value.device):
            out = torch.empty((n, lq, m * d), dtype=value.dtype, device=value.device)
            esz = raw.element_size()
            common = (spatial_shapes.data_ptr(), level_start_index.data_ptr(), ref.data_ptr(), ref.size(-1),
                      raw.data_ptr(), 3 * mlp, raw.data_ptr() + 2 * mlp * esz, 3 * mlp, n, s, m, d, nl, lq, p,
                      out.data_ptr())
            stream = torch.cuda.current_stream().cuda_stream
            if ld:
                code = lib.msda_fused_forward_strided(_DTYPES[value.dtype], _DTYPES[raw.dtype], value.data_ptr(), ld,
                                                      *common, stream)
            else:
                code = lib.msda_fused_forward(_DTYPES[value.dtype], _DTYPES[raw.dtype], value.data_ptr(),
                                              *common, stream)
        _lib.check(code, "msda_fused_forward")
        ctx.save_for_backward(value, spatial_shapes, level_start_index, ref, raw)
        ctx.n_points = p
        ctx.ref_dtype = reference_points.dtype
        ctx.ref_needs_grad = reference_points.requires_grad
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, spatial_shapes, level_start_index, ref, raw = ctx.saved_tensors
        n, s, m, d = value.shape
        nl = spatial_shapes.size(0)
        lq = raw.size(1)
        p = ctx.n_points
        mlp = m * nl * p
        grad_output = _aligned(grad_output.contiguous())
        if grad_output.dtype != value.dtype:
            grad_output = grad_output.to(value.dtype)
        lib = _lib.load()
        deterministic = torch.are_deterministic_algorithms_enabled()
        with torch.cuda.device(value.device):
            grad_value = torch.empty_like(value)
            grad_raw = torch.empty_like(raw)
            grad_ref = None
            if ctx.ref_needs_grad:
                grad_ref = torch.empty_like(ref) if deterministic else torch.zeros_like(ref)
            esz = raw.element_size()
            args = (_DTYPES[value.dtype], _DTYPES[raw.dtype], grad_output.data_ptr(), value.data_ptr(),
                    spatial_shapes.data_ptr(), level_start_index.data_ptr(), ref.data_ptr(), ref.size(-1),
                    raw.data_ptr(), 3 * mlp, raw.data_ptr() + 2 * mlp * esz, 3 * mlp,
                    n, s, m, d, nl, lq, p, grad_value.data_ptr(), grad_raw.data_ptr(),
                    grad_raw.data_ptr() + 2 * mlp * esz,
                    grad_ref.data_ptr() if grad_ref is not None else None)
            stream = torch.cuda.current_stream().cuda_stream
            if deterministic:
                scratch = _lib.deterministic_scratch(value.device, value.numel(),
                                                     grad_ref.numel() if grad_ref is not None else 0, m)
                code = lib.msda_fused_backward_deterministic(*args, None, scratch.data_ptr(), scratch.numel(), stream)
            else:
                accum = torch.empty(value.shape, dtype=torch.float32, device=value.device) \
                    if value.dtype != torch.float32 else None
                code = lib.msda_fused_backward(*args, accum.data_ptr() if accum is not None else None, stream)
        _lib.check(code, "msda_fused_backward_deterministic" if deterministic else "msda_fused_backward")
        if grad_ref is not None and grad_ref.dtype != ctx.ref_dtype:
            grad_ref = grad_ref.to(ctx.ref_dtype)
        return grad_value, None, None, grad_ref, grad_raw, None


# ------------------------------------------------------------------------------------------------------------------
# Inference with a HEAD-MAJOR value tensor (csrc/value_proj_hm.cu + csrc/msda_forward_hm.cu): the value projection runs
# as an own tcgen05 GEMM whose epilogue adds the bias, zeroes the padding rows and writes [N, M, S, D] -- the layout in
# which the x-neighbours of a bilinear footprint are adjacent (3 instead of 4 L1 lines per sample in the gather).
# No autograd: callers use it only when no gradient is needed.
# ------------------------------------------------------------------------------------------------------------------
def head_major_supported(value_proj, input_flatten, raw, ref_dim, n_heads, n_levels, n_points):
    """bf16 CUDA inference at d_model 256 / 8 heads of 32 with a raw projection the fused kernels accept."""
    w = value_proj.weight
    if not (input_flatten.is_cuda and raw.is_cuda) or input_flatten.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        return False
    if value_proj.bias is None or raw.dtype not in _DTYPES or input_flatten.dim() != 3 or input_flatten.size(0) == 0:
        return False
    lib = _lib.load()
    d_model = w.shape[0]
    if w.shape[1] != d_model or d_model % n_heads != 0:
        return False
    if not lib.msda_layer_value_proj_head_major_supported(_lib.DTYPE_BF16, int(d_model), int(n_heads)):
        return False
    s = input_flatten.size(1)
    return bool(lib.msda_fused_supported(_lib.DTYPE_BF16, _DTYPES[raw.dtype], int(ref_dim), int(s), int(n_heads),
                                         int(d_model // n_heads), int(n_levels), int(n_points)))


def value_proj_head_major(value_proj, input_flatten, padding_mask, n_heads):
    """``value_proj(input_flatten)`` with masked rows zeroed (reference ms_deform_attn.py:94-96) -> [N, M, S, D]."""
    n, s, c = input_flatten.shape
    x = _aligned(input_flatten.contiguous())
    w = _aligned(value_proj.weight.detach().contiguous())
    b = value_proj.bias.detach().contiguous()
    mask8 = None
    if padding_mask is not None:
        mask8 = padding_mask.reshape(-1).contiguous()
        mask8 = mask8.view(torch.uint8) if mask8.dtype == torch.bool else (mask8 != 0).to(torch.uint8)
    with torch.cuda.device(x.device):
        out = torch.empty((n, n_heads, s, c // n_heads), dtype=x.dtype, device=x.device)
        code = _lib.load().msda_layer_value_proj_head_major(
            _lib.DTYPE_BF16, x.data_ptr(), w.data_ptr(), b.data_ptr(), mask8.data_ptr() if mask8 is not None else None,
            n * s, s, c, n_heads, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_value_proj_head_major")
    return out


def fused_forward_head_major(value_hm, spatial_shapes, level_start_index, reference_points, raw, n_points):
    """The fused layer forward (softmax, location arithmetic, gather, head reduction) on a head-major value tensor
    [N, M, S, D] -> [N, Lq, M*D].  Inference only."""
    n, m, s, d = value_hm.shape
    nl = spatial_shapes.size(0)
    lq = raw.size(1)
    p = int(n_points)
    mlp = m * nl * p
    if raw.size(-1) != 3 * mlp or raw.size(0) != n:
        raise RuntimeError(f"raw must be [N, Lq, 3*M*L*P={3 * mlp}], got {tuple(raw.shape)}")
    raw = _aligned(raw.contiguous())
    ref = _aligned(reference_points.detach().to(torch.float32).contiguous())
    with torch.cuda.device(value_hm.device):
        out = torch.empty((n, lq, m * d), dtype=value_hm.dtype, device=value_hm.device)
        esz = raw.element_size()
        code = _lib.load().msda_fused_forward_head_major(
            _DTYPES[value_hm.dtype], _DTYPES[raw.dtype], value_hm.data_ptr(), spatial_shapes.contiguous().data_ptr(),
            level_start_index.contiguous().data_ptr(), ref.data_ptr(), ref.size(-1), raw.data_ptr(), 3 * mlp,
            raw.data_ptr() + 2 * mlp * esz, 3 * mlp, n, s, m, d, nl, lq, p, out.data_ptr(),
            torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_fused_forward_head_major")
    return out
