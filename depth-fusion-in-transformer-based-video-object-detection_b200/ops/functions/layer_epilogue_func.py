"""Autograd bindings of the layer-epilogue kernels (C ABI ``msda_layer_*``, csrc/layer_epilogue.cu).

``add_layer_norm(norm, branch, residual, act, pos)`` is what the reference layer classes spell as
    norm(residual + act(branch))            deformable_transformer_single.py:538-541, :393-400, :452-459
    ... + pos                               :530-531 (query of the next deformable attention)
as ONE kernel per direction.  ``zero_masked_rows_`` is MSDeformAttn's
``value.masked_fill(mask[..., None], 0)`` (models/ops/modules/ms_deform_attn.py:95-96) in place.
``linear_relu`` is ``relu(linear1(x))`` with the activation in the GEMM epilogue (library GEMM).
Both take the layer's ``nn.Dropout`` and then apply it inside the same kernels (``dropout`` for the other sites).
CUDA tensors only; callers keep the PyTorch composition for shapes the kernels do not cover.
"""
import ctypes

import torch
import torch.nn.functional as F
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from ... import _lib

_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16}
ACT_CODES = {None: 0, "none": 0, "relu": 1, "gelu": 2}


def add_layer_norm_supported(x, channels):
    return x.is_cuda and x.dtype in _DTYPES and \
        bool(_lib.load().msda_layer_add_layernorm_supported(_DTYPES[x.dtype], int(channels)))


def _ptr(t):
    return None if t is None else t.data_ptr()


def _dense(t):
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


# Dropout on the package's kernels (DESIGN.md section 3.16): each call draws one int64 key on the device, and the mask of
# element e of the call's [rows, C] output is a function of (key, e) (Philox4x32-10, msda_common.cuh: dropout_keep8).  The
# backward regenerates it from the saved key, so no mask is stored and no separate dropout pass runs: the mask is applied
# inside the add-LayerNorm and ReLU-GEMM kernels.  Taken when the module is exactly nn.Dropout, in training, 0 < p < 1,
# on a CUDA fp32 / bf16 / fp16 tensor; False keeps torch's nn.Dropout between the kernels (the A/B of
# tools/bench_dropout.py).
PACKAGE_DROPOUT = True


def _dropout_key(device):
    """The key of one dropout call: one int64 from torch's CUDA generator, never read back (graph-capturable)."""
    return torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=device)


def _dropout_mode(module, x):
    """"none": no dropout (no module, eval mode or p == 0: no key is drawn); "package": the package's kernels;
    "module": torch's ``module(x)``."""
    if module is None:
        return "none"
    if type(module) is not nn.Dropout:
        return "module"
    if not module.training or module.p == 0:
        return "none"
    if PACKAGE_DROPOUT and 0 < module.p < 1 and x.is_cuda and x.dtype in _DTYPES:
        return "package"
    return "module"


def dropout_rule(p):
    """(threshold, scale) of the keep rule at rate p: an element is kept iff its 16-bit draw is >= threshold."""
    t, scale = ctypes.c_uint32(), ctypes.c_float()
    _lib.check(_lib.load().msda_layer_dropout_rule(float(p), ctypes.byref(t), ctypes.byref(scale)),
               "msda_layer_dropout_rule")
    return t.value, scale.value


def _dropout_into(x, y, p, key):
    """y = x * mask(key) * scale over the contiguous x (y may be x)."""
    with torch.cuda.device(x.device):
        code = _lib.load().msda_layer_dropout(_DTYPES[x.dtype], x.data_ptr(), y.data_ptr(), x.numel(), float(p),
                                              key.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_dropout")
    return y


def relu_dropout_grad(grad, out, p):
    """grad * scale where out > 0, else 0: the backward of dropout(relu(.)) at rate p from its output alone."""
    grad = grad.reshape(out.shape).contiguous()
    if grad.dtype != out.dtype:
        grad = grad.to(out.dtype)
    dx = torch.empty_like(out)
    with torch.cuda.device(out.device):
        code = _lib.load().msda_layer_relu_dropout_grad(_DTYPES[out.dtype], grad.data_ptr(), out.data_ptr(), dx.data_ptr(),
                                                        out.numel(), float(p), torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_relu_dropout_grad")
    return dx


class DropoutFunction(Function):
    """apply(x, p, key) -> x * mask * scale; the backward is the same kernel on the gradient with the same key."""

    @staticmethod
    def forward(ctx, x, p, key):
        xc = x.contiguous()
        y = _dropout_into(xc, torch.empty_like(xc), p, key)
        ctx.save_for_backward(key)
        ctx.p = p
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        (key,) = ctx.saved_tensors
        g = grad.contiguous()
        return _dropout_into(g, torch.empty_like(g), ctx.p, key), None, None


def dropout(module, x):
    """``module(x)`` for the layer's dropout module: the package's kernel when it applies (see PACKAGE_DROPOUT)."""
    mode = _dropout_mode(module, x)
    if mode == "none":
        return x
    if mode == "module":
        return module(x)
    return DropoutFunction.apply(x, float(module.p), _dropout_key(x.device))


class AddLayerNormFunction(Function):
    """apply(branch, residual|None, gamma, beta, eps, act_code, pos|None[, p, key]) -> y  or  (y, y + pos);
    with a key, dropout at rate p on act(branch)."""

    @staticmethod
    def forward(ctx, branch, residual, gamma, beta, eps, act, pos, p=0.0, key=None):
        shape = branch.shape
        c = shape[-1]
        dt = branch.dtype
        branch = _dense(branch)
        residual = None if residual is None else _dense(residual.to(dt))
        pos = None if pos is None else _dense(pos.to(dt).expand(shape))
        gamma_c, beta_c = _dense(gamma.to(dt)), _dense(beta.to(dt))
        rows = branch.numel() // c if c else 0
        needs_grad = any(ctx.needs_input_grad)
        lib = _lib.load()
        with torch.cuda.device(branch.device):
            y = torch.empty_like(branch)
            y_pos = torch.empty_like(branch) if pos is not None else None
            mean = torch.empty(rows, dtype=torch.float32, device=branch.device) if needs_grad else None
            rstd = torch.empty_like(mean) if needs_grad else None
            args = (_DTYPES[dt], act, branch.data_ptr(), _ptr(residual), gamma_c.data_ptr(), beta_c.data_ptr(),
                    _ptr(pos), rows, c, float(eps), y.data_ptr(), _ptr(y_pos), _ptr(mean), _ptr(rstd))
            stream = torch.cuda.current_stream().cuda_stream
            if key is None:
                code = lib.msda_layer_add_layernorm_forward(*args, stream)
            else:
                code = lib.msda_layer_add_layernorm_dropout_forward(*args, float(p), key.data_ptr(), stream)
        _lib.check(code, "msda_layer_add_layernorm_forward")
        if needs_grad:
            ctx.save_for_backward(branch, residual, gamma_c, mean, rstd, key)
            ctx.p = p
            ctx.act = act
            ctx.param_dtypes = (gamma.dtype, beta.dtype)
            ctx.has_pos = pos is not None
        if y_pos is None:
            return y
        return y, y_pos

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y, grad_y_pos=None):
        branch, residual, gamma, mean, rstd, key = ctx.saved_tensors
        c = branch.shape[-1]
        rows = branch.numel() // c
        dt = branch.dtype
        if grad_y is None and grad_y_pos is None:
            return (None,) * 9
        if grad_y is None:            # only the y + pos output was used downstream
            grad_y, grad_y_pos_k = grad_y_pos, None
        else:
            grad_y_pos_k = grad_y_pos
        grad_y = _dense(grad_y.to(dt))
        grad_y_pos_k = None if grad_y_pos_k is None else _dense(grad_y_pos_k.to(dt))
        lib = _lib.load()
        with torch.cuda.device(branch.device):
            d_res = torch.empty_like(branch) if residual is not None else None
            own = ctx.act != 0 or residual is None or key is not None
            d_branch = torch.empty_like(branch) if own else d_res
            d_gamma = torch.empty_like(gamma)
            d_beta = torch.empty_like(gamma)
            blocks = lib.msda_layer_add_layernorm_partial_blocks(rows)
            partial = torch.empty((blocks, 2, c), dtype=torch.float32, device=branch.device)
            args = (_DTYPES[dt], ctx.act, grad_y.data_ptr(), _ptr(grad_y_pos_k), branch.data_ptr(), _ptr(residual),
                    gamma.data_ptr(), mean.data_ptr(), rstd.data_ptr(), rows, c, d_branch.data_ptr(), _ptr(d_res),
                    d_gamma.data_ptr(), d_beta.data_ptr(), partial.data_ptr(), blocks)
            stream = torch.cuda.current_stream().cuda_stream
            if key is None:
                code = lib.msda_layer_add_layernorm_backward(*args, stream)
            else:
                code = lib.msda_layer_add_layernorm_dropout_backward(*args, float(ctx.p), key.data_ptr(), stream)
        _lib.check(code, "msda_layer_add_layernorm_backward")
        d_pos = grad_y_pos if ctx.has_pos else None
        return (d_branch, d_res, d_gamma.to(ctx.param_dtypes[0]), d_beta.to(ctx.param_dtypes[1]), None, None,
                d_pos, None, None)


def add_layer_norm(norm, branch, residual=None, act=None, pos=None, dropout=None):
    """``norm(residual + dropout(act(branch)))`` and, when ``pos`` is given, also ``that + pos``.

    ``norm`` is the layer's ``nn.LayerNorm`` (parameters / eps are read from it, so state_dict keys
    stay the reference's), ``dropout`` the layer's ``nn.Dropout`` or None.  Returns ``y`` or ``(y, y_pos)``."""
    c = branch.shape[-1]
    fusable = (add_layer_norm_supported(branch, c) and norm.elementwise_affine and norm.bias is not None
               and tuple(norm.normalized_shape) == (c,) and act in ACT_CODES
               and (residual is None or residual.shape == branch.shape)
               and (pos is None or pos.shape == branch.shape))
    mode = _dropout_mode(dropout, branch)
    if mode == "package" and fusable and _lib.load().msda_layer_add_layernorm_dropout_supported(_DTYPES[branch.dtype], c):
        return AddLayerNormFunction.apply(branch, residual, norm.weight, norm.bias, norm.eps, ACT_CODES[act], pos,
                                          float(dropout.p), _dropout_key(branch.device))
    if mode != "none":
        h = branch if act in (None, "none") else getattr(F, act)(branch)
        return add_layer_norm(norm, globals()["dropout"](dropout, h), residual, None, pos)
    if fusable:
        return AddLayerNormFunction.apply(branch, residual, norm.weight, norm.bias, norm.eps, ACT_CODES[act], pos)
    # PyTorch composition (shapes the kernel does not cover)
    h = branch if act in (None, "none") else getattr(F, act)(branch)
    y = norm(h if residual is None else residual + h)
    return y if pos is None else (y, y + pos)


def norm_act(norm, x, act=None, inplace=False):
    """``act(norm(x))`` -- normalise, then activate (the order of the TransVOD++ dynamic interaction head,
    /root/reference/models/sparse_roi_head/head.py:156-170; ``add_layer_norm`` activates BEFORE the norm).
    One kernel when no gradient is needed and the row width is covered (64 .. 1024 channels of bf16, 32 .. 512 of
    fp32); ``inplace`` lets it overwrite ``x``.  Otherwise the PyTorch composition."""
    c = x.shape[-1]
    needs_grad = torch.is_grad_enabled() and (x.requires_grad or norm.weight.requires_grad)
    if (not needs_grad and x.is_cuda and x.dtype in _DTYPES and act in ACT_CODES and norm.elementwise_affine
            and norm.bias is not None and tuple(norm.normalized_shape) == (c,)
            and _lib.load().msda_layer_norm_act_supported(_DTYPES[x.dtype], int(c))):
        dense = x.contiguous()
        if dense.data_ptr() % 16 != 0:
            dense = dense.clone()
        y = dense if (inplace and dense is x) or dense is not x else torch.empty_like(dense)
        gamma, beta = _dense(norm.weight.detach().to(x.dtype)), _dense(norm.bias.detach().to(x.dtype))
        with torch.cuda.device(x.device):
            code = _lib.load().msda_layer_norm_act_forward(
                _DTYPES[x.dtype], dense.data_ptr(), gamma.data_ptr(), beta.data_ptr(), dense.numel() // c, int(c),
                float(norm.eps), ACT_CODES[act], y.data_ptr(), torch.cuda.current_stream().cuda_stream)
        _lib.check(code, "msda_layer_norm_act_forward")
        return y
    y = norm(x)
    return y if act in (None, "none") else getattr(F, act)(y)


class ZeroMaskedRowsFunction(Function):
    """In place: rows of ``value`` [N, S, C] whose ``mask`` [N, S] entry is True become zero."""

    @staticmethod
    def forward(ctx, value, mask, exclusive=False):
        ctx.exclusive = bool(exclusive)
        if not value.is_contiguous():
            raise RuntimeError("zero_masked_rows_: value must be contiguous")
        mask8 = mask.contiguous().view(torch.uint8) if mask.dtype == torch.bool else (mask != 0).to(torch.uint8)
        c = value.shape[-1]
        rows = value.numel() // c if c else 0
        if mask8.numel() != rows:
            raise RuntimeError(f"mask has {mask8.numel()} entries for {rows} rows")
        code = _lib.load().msda_layer_zero_masked_rows(
            _DTYPES[value.dtype], value.data_ptr(), mask8.data_ptr(), rows, c,
            torch.cuda.current_stream().cuda_stream)
        _lib.check(code, "msda_layer_zero_masked_rows")
        ctx.mark_dirty(value)
        ctx.save_for_backward(mask8)
        return value

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        (mask8,) = ctx.saved_tensors
        # Autograd forbids mutating an incoming gradient: the same buffer may feed another consumer of `value`, a
        # tensor hook or retain_grad.  So the rows are zeroed in a COPY -- unless the call site vouched that `value`
        # feeds only the deformable-attention op (whose backward allocates this gradient fresh) by passing
        # exclusive=True to zero_masked_rows_: then the 180 MB copy per layer is skipped.
        if not ctx.exclusive or not grad.is_contiguous() or grad.data_ptr() % 16:
            grad = grad.contiguous().clone()
        c = grad.shape[-1]
        code = _lib.load().msda_layer_zero_masked_rows(
            _DTYPES[grad.dtype], grad.data_ptr(), mask8.data_ptr(), grad.numel() // c, c,
            torch.cuda.current_stream().cuda_stream)
        _lib.check(code, "msda_layer_zero_masked_rows")
        return grad, None, None


def zero_masked_rows_(value, mask, exclusive=False):
    """``value.masked_fill(mask[..., None], 0)`` for a freshly produced ``value`` (modified in place).
    ``exclusive=True``: the caller guarantees that the result has exactly one consumer whose backward hands over a
    freshly allocated gradient (the deformable-attention op); the backward then zeroes that gradient in place."""
    c = value.shape[-1]
    if value.is_cuda and value.dtype in _DTYPES and value.is_contiguous() and (c * value.element_size()) % 16 == 0 \
            and value.data_ptr() % 16 == 0:
        with torch.cuda.device(value.device):
            return ZeroMaskedRowsFunction.apply(value, mask, exclusive)
    return value.masked_fill(mask[..., None], float(0))


def column_sum(g2):
    """sum over rows of a contiguous [rows, C] CUDA matrix -> [C] (bias gradient), at HBM rate."""
    rows, c = g2.shape
    lib = _lib.load()
    blocks = lib.msda_layer_colsum_blocks(_DTYPES[g2.dtype], rows, c) if g2.dtype in _DTYPES and g2.is_cuda else 0
    if blocks == 0 or not g2.is_contiguous() or g2.data_ptr() % 16:
        return g2.sum(0)
    with torch.cuda.device(g2.device):
        out = torch.empty(c, dtype=g2.dtype, device=g2.device)
        partial = torch.empty((blocks, c), dtype=torch.float32, device=g2.device)
        code = lib.msda_layer_colsum(_DTYPES[g2.dtype], g2.data_ptr(), rows, c, out.data_ptr(), partial.data_ptr(),
                                     blocks, torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_colsum")
    return out


class LinearFunction(Function):
    """x @ W^T + b as the library GEMM, with a backward that takes the bias gradient from the
    column-sum kernel instead of PyTorch's generic reduction.  bf16 training from BF16_TRAIN_KERNEL_MIN_ROWS rows up:
    the package's own kernels in both directions (_bf16_train_kernels_apply); fp32 training in fp32 train-GEMM mode
    "tf32x3": the three-term TF32 kernels in both directions (_fp32_train_kernels_apply)."""

    @staticmethod
    def forward(ctx, x2, weight, bias):              # x2 [rows, in] -> fresh [rows, out] (never a view)
        # under torch.autocast the GEMM runs in the autocast dtype like F.linear does; the operands are saved as
        # they were used, so that the backward (which runs outside autocast) multiplies matching dtypes
        if torch.is_autocast_enabled():
            adt = torch.get_autocast_gpu_dtype()
            x2, weight_c, bias_c = x2.to(adt), weight.to(adt), bias.to(adt)
        else:
            weight_c, bias_c = weight, bias
        ctx.save_for_backward(x2, weight_c)
        ctx.param_dtypes = (weight.dtype, bias.dtype)
        ctx.kernels = any(ctx.needs_input_grad) and _bf16_train_kernels_apply(x2, weight_c, bias_c)
        ctx.tf32x3 = not ctx.kernels and any(ctx.needs_input_grad) and _fp32_train_kernels_apply(x2, weight_c, bias_c)
        if ctx.kernels:
            return linear_bf16(x2, weight_c, bias_c)
        if ctx.tf32x3:
            return _linear_tf32x3_kernel(x2, *_tf32_weight_split(weight_c, live=True), bias_c)
        return torch.addmm(bias_c, x2, weight_c.t())

    @staticmethod
    @once_differentiable
    def backward(ctx, g2):
        x2, weight = ctx.saved_tensors
        if not g2.is_contiguous():
            g2 = g2.contiguous()
        if g2.dtype != weight.dtype:
            g2 = g2.to(weight.dtype)
        if ctx.kernels:
            return _bf16_linear_backward(ctx.needs_input_grad, g2, x2, weight, ctx.param_dtypes)
        if ctx.tf32x3:
            return _tf32x3_linear_backward(ctx.needs_input_grad, g2, x2, weight)
        dx = g2 @ weight if ctx.needs_input_grad[0] else None
        dw = (g2.t() @ x2).to(ctx.param_dtypes[0]) if ctx.needs_input_grad[1] else None
        db = column_sum(g2).to(ctx.param_dtypes[1]) if ctx.needs_input_grad[2] else None
        return dx, dw, db


# How the fp32 projections of an inference pass are evaluated (the gather kernels are not affected):
#   "tf32x3"   (default) error-compensated split on the tensor cores: x = x_hi + x_lo, W = W_hi + W_lo with the *_hi parts
#              on TF32's 10 mantissa bits, y = x_lo W_hi^T + x_hi W_lo^T + x_hi W_hi^T with fp32 accumulation; the dropped
#              x_lo W_lo^T term and the rounding of the *_lo operands are O(2^-22).  fp32-grade results
#              (tests/test_gpu_layer_epilogue.py: 6.9e-7 normalised against fp64 at K = 256, the IEEE SGEMM 7.2e-7, one TF32
#              GEMM 3e-4; every fp32 golden of tests/test_gpu_modules.py holds its 1e-5 with it) at a third of the TF32
#              tensor rate instead of the SIMT SGEMM rate: 6-layer fp32 encoder 45.7 -> 12.2 ms.  One tcgen05 kernel per
#              layer (csrc/linear_tf32x3.cu: the activation tile is split in shared memory, bias / ReLU in the epilogue);
#              shapes it does not take fall back to the split pass (msda_layer_tf32_split) + one library TF32 GEMM over
#              the concatenated reduction.  Only without gradients and from TF32X3_MIN_ROWS rows up.
#   "library"  whatever torch.backends.cuda.matmul says (IEEE SGEMM unless the caller allowed TF32): the reference's own
#              arithmetic, bit for bit what F.linear gives.
FP32_GEMM_MODE = "tf32x3"
TF32X3_MIN_ROWS = 1024              # below this the SGEMM is as fast


def set_fp32_gemm_mode(mode):
    global FP32_GEMM_MODE
    if mode not in ("library", "tf32x3"):
        raise ValueError(f"unknown fp32 GEMM mode {mode!r}")
    previous, FP32_GEMM_MODE = FP32_GEMM_MODE, mode
    return previous


def _tf32_split(t):
    """t [rows, cols] (fp32) -> [rows, 3 * cols] = [lo | hi | hi]: hi = t rounded to TF32's 10 mantissa bits (nearest, ties
    away), lo = t - hi (exact).  One kernel (C ABI ``msda_layer_tf32_split``) on CUDA; the torch composition otherwise."""
    rows, cols = t.shape
    if t.is_cuda and t.is_contiguous() and cols % 4 == 0 and t.data_ptr() % 16 == 0 and rows > 0:
        out = torch.empty((rows, 3 * cols), dtype=torch.float32, device=t.device)
        with torch.cuda.device(t.device):
            code = _lib.load().msda_layer_tf32_split(t.data_ptr(), rows, cols, out.data_ptr(),
                                                     torch.cuda.current_stream().cuda_stream)
        _lib.check(code, "msda_layer_tf32_split")
        return out
    hi = ((t.contiguous().view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)
    return torch.cat([t - hi, hi, hi], 1)


def _tf32x3_wanted(x, weight):
    # (under torch.autocast an fp32 nn.Linear is the caller's request for a 16-bit GEMM: F.linear honours it)
    return (FP32_GEMM_MODE == "tf32x3" and x.is_cuda and x.dtype == torch.float32 and weight.dtype == torch.float32
            and not torch.is_autocast_enabled()
            and x.numel() // max(x.shape[-1], 1) >= TF32X3_MIN_ROWS
            and not (torch.is_grad_enabled() and (x.requires_grad or weight.requires_grad)))


def _tf32_weight_split(weight, live=False):
    """weight -> (hi, lo): hi = weight rounded to TF32's 10 mantissa bits (nearest, ties away), lo = weight - hi (exact).
    Cached ON the weight tensor (weights are static in inference) together with the version counter it was made from:
    the cache dies with the tensor, and an in-place update (optimizer step, load_state_dict) invalidates it.
    live=True (training): under CUDA-graph capture the split is always made inside the graph, never taken from the cache,
    so that every replay splits the weights as the optimizer left them (its in-place updates happen outside the graph)."""
    hit = getattr(weight, "_dfvod_tf32_split", None)
    capturing = weight.is_cuda and torch.cuda.is_current_stream_capturing()
    if hit is None or hit[0] != weight._version or hit[1].device != weight.device or (live and capturing):
        w = weight.detach().contiguous()
        hi = ((w.view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)
        hit = (weight._version, hi, w - hi)
        # (tensors made during a CUDA-graph capture live in the graph's private pool: never cache those)
        if not capturing:
            try:
                weight._dfvod_tf32_split = hit
            except (AttributeError, RuntimeError):      # a tensor that takes no attributes: split every call
                pass
    return hit[1], hit[2]


def linear_tf32x3_kernel_supported(x, weight):
    """The one-kernel route (csrc/linear_tf32x3.cu): the activation tile is split in shared memory."""
    n, k = weight.shape
    return (x.is_cuda and x.dtype == torch.float32 and weight.dtype == torch.float32 and x.shape[-1] == k
            and bool(_lib.load().msda_layer_linear_tf32x3_supported(n, k)))


def _tf32x3_kernel_wins(n, k):
    """Measured on B200 at 8 x 22223 rows (tools/run_tf32x3.py), one kernel vs split pass + library GEMM: the kernel wins
    at every shape of the model (DESIGN.md section 3.5)."""
    return True


def _linear_tf32x3_kernel(x2, w_hi, w_lo, bias, relu=False, dropout=None):
    """x2 [rows, k] @ (w_hi + w_lo)^T + bias -> a fresh [rows, n] (ReLU) on csrc/linear_tf32x3.cu; (w_hi, w_lo) [n, k]
    contiguous, the TF32 split of a weight (_tf32_weight_split) or of its transpose.  dropout = (p, key): ReLU, then
    dropout in the epilogue."""
    n, k = w_hi.shape
    if not x2.is_contiguous() or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    b = None if bias is None else bias.detach().contiguous()
    y = torch.empty((x2.shape[0], n), dtype=torch.float32, device=x2.device)
    with torch.cuda.device(x2.device):
        stream = torch.cuda.current_stream().cuda_stream
        if dropout is None:
            code = _lib.load().msda_layer_linear_tf32x3(x2.data_ptr(), w_hi.data_ptr(), w_lo.data_ptr(),
                                                        None if b is None else b.data_ptr(), x2.shape[0], n, k,
                                                        1 if relu else 0, y.data_ptr(), stream)
        else:
            code = _lib.load().msda_layer_linear_tf32x3_relu_dropout(
                x2.data_ptr(), w_hi.data_ptr(), w_lo.data_ptr(), None if b is None else b.data_ptr(), x2.shape[0], n, k,
                float(dropout[0]), dropout[1].data_ptr(), y.data_ptr(), stream)
    _lib.check(code, "msda_layer_linear_tf32x3")
    return y


def linear_tf32x3(x, weight, bias, relu=False, route=None):
    """route: None = the faster of the two for the shape, "kernel" / "library" to force one (tests, measurements)."""
    k = x.shape[-1]
    use_kernel = linear_tf32x3_kernel_supported(x, weight) and route != "library" and (
        route == "kernel" or _tf32x3_kernel_wins(weight.shape[0], k))
    if use_kernel:
        y = _linear_tf32x3_kernel(x.reshape(-1, k), *_tf32_weight_split(weight), bias, relu)
        return y.view(*x.shape[:-1], weight.shape[0])
    # shapes the kernel does not take: the same split as ONE library TF32 GEMM over the concatenated reduction
    a = _tf32_split(x.reshape(-1, k).contiguous())                       # [rows, 3k] = [lo | hi | hi]
    w = _tf32_split(weight.detach().contiguous())
    w = torch.cat([w[:, k:2 * k], w[:, :k], w[:, 2 * k:]], 1)            # [n, 3k]    = [hi | lo | hi]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        y = torch.mm(a, w.t()) if bias is None else torch.addmm(bias.detach(), a, w.t())
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    if relu:
        y = torch.relu_(y)
    return y.view(*x.shape[:-1], weight.shape[0])


# bf16 inference: the nn.Linear layers run as one TMA / tcgen05 kernel (csrc/linear_bf16.cu: bias, ReLU and the padding-row
# zeroing of value_proj in the epilogue) from BF16_KERNEL_MIN_ROWS rows up; set to None to keep the library GEMM.  The
# kernel is persistent over 128-row tiles, one CTA per SM: below ~148 tiles it leaves SMs idle and the library's split of a
# small problem is faster (6+6 transformer, 2400 decoder rows: 5.44 ms with the library there, 5.58 ms with the kernel).
BF16_KERNEL_MIN_ROWS = 16384


def _bf16_kernel_wanted(x, weight, bias):
    return (BF16_KERNEL_MIN_ROWS is not None and x.is_cuda and x.dtype == torch.bfloat16 and weight.dtype == torch.bfloat16
            and (bias is None or bias.dtype == torch.bfloat16) and x.shape[-1] == weight.shape[1]
            and x.numel() // max(x.shape[-1], 1) >= BF16_KERNEL_MIN_ROWS
            and not (torch.is_grad_enabled() and (x.requires_grad or weight.requires_grad
                                                  or (bias is not None and bias.requires_grad)))
            and bool(_lib.load().msda_layer_linear_bf16_supported(weight.shape[0], weight.shape[1])))


def linear_bf16(x, weight, bias, relu=False, zero_rows=None):
    """y = x W^T + b (ReLU, rows of ``zero_rows`` [rows] bool zeroed) through csrc/linear_bf16.cu."""
    k = x.shape[-1]
    x2 = x.reshape(-1, k)
    if not x2.is_contiguous() or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    w = weight.detach()
    if not w.is_contiguous() or w.data_ptr() % 16 != 0:
        w = w.contiguous()
    b = None if bias is None else bias.detach().contiguous()
    m = None
    if zero_rows is not None:
        m = zero_rows.reshape(-1)
        m = (m if m.dtype == torch.bool else m != 0).contiguous().view(torch.uint8)
        if m.numel() != x2.shape[0]:
            raise ValueError("zero_rows must have one entry per row")
    y = torch.empty((x2.shape[0], weight.shape[0]), dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device):
        code = _lib.load().msda_layer_linear_bf16(x2.data_ptr(), w.data_ptr(), None if b is None else b.data_ptr(),
                                                  None if m is None else m.data_ptr(), x2.shape[0], weight.shape[0], k,
                                                  1 if relu else 0, y.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_linear_bf16")
    # (a 2-d input gets y itself, not a view of it: LinearFunction hands it to autograd, where it may be modified in place)
    return y if x.dim() == 2 else y.view(*x.shape[:-1], weight.shape[0])


# bf16 training: from BF16_TRAIN_KERNEL_MIN_ROWS rows up, LinearFunction and LinearReLUFunction run their forward on
# csrc/linear_bf16.cu and their backward as dx = g W (the same kernel with W^T as its weight) and one weight-gradient kernel
# that also gives the bias gradient (linear_bf16_wgrad: g is read once for both).  Set to None to keep the library GEMMs.
# The kernels spread 128-row tiles (forward, dx) and row slices (dW) over all SMs; the threshold keeps the decoder-sized
# GEMMs (1200 rows) on the library.  Graphed Encoder-Cross-Fusion training step on one B200 (DESIGN.md section 3.13):
# 22.05 ms with the library GEMMs, 21.53 ms on the kernels (1000 W power limit).
BF16_TRAIN_KERNEL_MIN_ROWS = 16384


def _bf16_train_kernels_win(n, k):
    """Measured on B200 at 88 892 rows (tools/bench_train_linears.py, DESIGN.md section 3.13): dx + dW + db on the kernels
    beat the library's three calls where the layer's input is one column tile wide (256 <- 256, 384 <- 256,
    1024 <- 256: 5-14 % faster) and lose at 256 <- 1024 (linear2 of the feed-forward block: 6 % slower), which keeps
    the library."""
    return k <= 256


def _bf16_train_kernels_apply(x2, weight, bias):
    """Gradients flow (checked by the caller), the operands as multiplied are CUDA bf16, enough rows, a shape where the
    kernels are faster, and the forward, input-gradient and weight-gradient kernels all take it."""
    if BF16_TRAIN_KERNEL_MIN_ROWS is None or not x2.is_cuda or x2.shape[0] < BF16_TRAIN_KERNEL_MIN_ROWS:
        return False
    if x2.dtype != torch.bfloat16 or weight.dtype != torch.bfloat16 or (bias is not None and bias.dtype != torch.bfloat16):
        return False
    n, k = weight.shape
    lib = _lib.load()
    return (x2.shape[1] == k and _bf16_train_kernels_win(n, k) and bool(lib.msda_layer_linear_bf16_supported(n, k))
            and bool(lib.msda_layer_linear_bf16_supported(k, n)) and bool(lib.msda_layer_linear_bf16_wgrad_supported(n, k)))


def linear_bf16_wgrad(g2, x2, with_bias=True):
    """(g2^T x2, g2.sum(0) or None) for bf16 g2 [rows, out], x2 [rows, in] through csrc/linear_bf16.cu: one pass over g2
    gives both; fp32 split-K partials summed in a fixed order (deterministic)."""
    rows, n = g2.shape
    k = x2.shape[1]
    if x2.shape[0] != rows or g2.dtype != torch.bfloat16 or x2.dtype != torch.bfloat16:
        raise ValueError("linear_bf16_wgrad: bf16 g [rows, out] and x [rows, in] expected")
    lib = _lib.load()
    floats = lib.msda_layer_linear_bf16_wgrad_scratch_floats(rows, n, k)
    if floats == 0:
        raise ValueError(f"linear_bf16_wgrad: shape rows={rows}, out={n}, in={k} not supported")
    if not g2.is_contiguous() or g2.data_ptr() % 16 != 0:
        g2 = g2.contiguous()
    if not x2.is_contiguous() or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    dw = torch.empty((n, k), dtype=torch.bfloat16, device=g2.device)
    db = torch.empty(n, dtype=torch.bfloat16, device=g2.device) if with_bias else None
    scratch = torch.empty(floats, dtype=torch.float32, device=g2.device)
    with torch.cuda.device(g2.device):
        code = lib.msda_layer_linear_bf16_wgrad(g2.data_ptr(), x2.data_ptr(), rows, n, k, dw.data_ptr(),
                                                None if db is None else db.data_ptr(), scratch.data_ptr(), floats,
                                                torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_linear_bf16_wgrad")
    return dw, db


def _bf16_linear_backward(needs_input_grad, g2, x2, weight, param_dtypes):
    """(dx, dW, db) of a bf16 linear layer on the package's kernels; g2 [rows, out] contiguous bf16 (after the ReLU mask),
    dW / db cast to the parameters' dtypes (autocast)."""
    # W^T is made from the live weight on every backward (at most 0.5 MB): a cached copy goes stale under .data writes
    dx = linear_bf16(g2, weight.t().contiguous(), None) if needs_input_grad[0] else None
    dw = db = None
    if needs_input_grad[1]:
        dw, db = linear_bf16_wgrad(g2, x2, with_bias=needs_input_grad[2])
    elif needs_input_grad[2]:
        db = column_sum(g2)
    return dx, (None if dw is None else dw.to(param_dtypes[0])), (None if db is None else db.to(param_dtypes[1]))


# fp32 training (the backward, and the forward of a layer whose gradients flow):
#   "library"  (default) torch's GEMMs, IEEE SGEMM unless the caller allowed TF32: the reference's own arithmetic, bit for
#              bit.  fp32 training is compared against it, so it stays the default until an fp32 convergence comparison
#              says otherwise.
#   "tf32x3"   the three-term TF32 kernels of csrc/linear_tf32x3.cu in both directions, from FP32_TRAIN_KERNEL_MIN_ROWS rows
#              up at the shapes where they were measured faster (_fp32_train_kernels_win): forward y = x W^T + b and
#              dx = g W are linear_tf32x3 (with the split of W^T as the weight pair for dx), dW = g^T x and db = sum g
#              one linear_tf32x3_wgrad (both operands split in shared memory, g read once).  fp32-grade, not bit for
#              bit the SGEMM: within 1e-5 of fp64 like the library (tests/test_gpu_linear_tf32x3_train.py).
# A different numerical contract, not a faster route to the same bits: like FP32_GEMM_MODE, the caller chooses.
# FP32_TRAIN_KERNEL_MIN_ROWS: the smallest row count measured (tools/bench_train_fp32.py, DESIGN.md section 3.14); every
# shape of the model was already faster on the kernels there (backward 1.17-1.71x, forward 1.48-2.84x on one B200).
# Graphed fp32 Encoder-Cross-Fusion training step, 4 frames: 106.2 ms in mode "library", 44.1 ms in mode "tf32x3".
FP32_TRAIN_GEMM_MODE = "library"
FP32_TRAIN_KERNEL_MIN_ROWS = 2400


def set_fp32_train_gemm_mode(mode):
    """Selects how fp32 training evaluates the linear layers ("library" or "tf32x3"); returns the previous mode."""
    global FP32_TRAIN_GEMM_MODE
    if mode not in ("library", "tf32x3"):
        raise ValueError(f"unknown fp32 training GEMM mode {mode!r}")
    previous, FP32_TRAIN_GEMM_MODE = FP32_TRAIN_GEMM_MODE, mode
    return previous


def _fp32_train_kernels_win(n, k):
    """Shapes where forward + dx + dW + db on the kernels beat the SGEMM path.  Measured on B200 (tools/bench_train_fp32.py,
    DESIGN.md section 3.14) at 2 400, 88 892 and 177 784 rows: every shape of the model wins (256 <- 256, 384 <- 256,
    1024 <- 256 and 256 <- 1024; backward 1.17-3.60x, forward 1.48-6.19x), so none is excluded."""
    return True


def _fp32_train_kernels_apply(x2, weight, bias):
    """Mode "tf32x3", gradients flow (checked by the caller), the operands as multiplied are CUDA fp32 (not under
    autocast), enough rows, a shape where the kernels are faster, and the forward, input-gradient and weight-gradient
    kernels all take it."""
    if (FP32_TRAIN_GEMM_MODE != "tf32x3" or FP32_TRAIN_KERNEL_MIN_ROWS is None or not x2.is_cuda
            or x2.shape[0] < FP32_TRAIN_KERNEL_MIN_ROWS or torch.is_autocast_enabled()):
        return False
    if x2.dtype != torch.float32 or weight.dtype != torch.float32 or (bias is not None and bias.dtype != torch.float32):
        return False
    n, k = weight.shape
    lib = _lib.load()
    return (x2.shape[1] == k and _fp32_train_kernels_win(n, k) and bool(lib.msda_layer_linear_tf32x3_supported(n, k))
            and bool(lib.msda_layer_linear_tf32x3_supported(k, n))
            and bool(lib.msda_layer_linear_tf32x3_wgrad_supported(n, k)))


def linear_tf32x3_wgrad(g2, x2, with_bias=True):
    """(g2^T x2, g2.sum(0) or None) for fp32 g2 [rows, out], x2 [rows, in] through csrc/linear_tf32x3.cu: the three-term
    TF32 split of both operands, fp32-grade; one pass over g2 gives both; split-K partials summed in a fixed order
    (deterministic)."""
    rows, n = g2.shape
    k = x2.shape[1]
    if x2.shape[0] != rows or g2.dtype != torch.float32 or x2.dtype != torch.float32:
        raise ValueError("linear_tf32x3_wgrad: fp32 g [rows, out] and x [rows, in] expected")
    lib = _lib.load()
    floats = lib.msda_layer_linear_tf32x3_wgrad_scratch_floats(rows, n, k)
    if floats == 0:
        raise ValueError(f"linear_tf32x3_wgrad: shape rows={rows}, out={n}, in={k} not supported")
    if not g2.is_contiguous() or g2.data_ptr() % 16 != 0:
        g2 = g2.contiguous()
    if not x2.is_contiguous() or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    dw = torch.empty((n, k), dtype=torch.float32, device=g2.device)
    db = torch.empty(n, dtype=torch.float32, device=g2.device) if with_bias else None
    scratch = torch.empty(floats, dtype=torch.float32, device=g2.device)
    with torch.cuda.device(g2.device):
        code = lib.msda_layer_linear_tf32x3_wgrad(g2.data_ptr(), x2.data_ptr(), rows, n, k, dw.data_ptr(),
                                                  None if db is None else db.data_ptr(), scratch.data_ptr(), floats,
                                                  torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_linear_tf32x3_wgrad")
    return dw, db


def _tf32x3_linear_backward(needs_input_grad, g2, x2, weight):
    """(dx, dW, db) of an fp32 linear layer on the three-term TF32 kernels; g2 [rows, out] contiguous fp32 (after the ReLU
    mask)."""
    dx = dw = db = None
    if needs_input_grad[0]:
        # the transpose of the split is the split of the transpose: (W_hi^T, W_lo^T) is the weight pair of dx = g W
        w_hi, w_lo = _tf32_weight_split(weight, live=True)
        dx = _linear_tf32x3_kernel(g2, w_hi.t().contiguous(), w_lo.t().contiguous(), None)
    if needs_input_grad[1]:
        dw, db = linear_tf32x3_wgrad(g2, x2, with_bias=needs_input_grad[2])
    elif needs_input_grad[2]:
        db = column_sum(g2)
    return dx, dw, db


def linear_wb(x, weight, bias):
    """``F.linear(x, weight, bias)``: same GEMM; the custom backward only when gradients flow."""
    if _tf32x3_wanted(x, weight):
        return linear_tf32x3(x, weight, bias)
    if _bf16_kernel_wanted(x, weight, bias):
        return linear_bf16(x, weight, bias)
    if x.is_cuda and bias is not None and x.dtype == weight.dtype and x.dtype in _DTYPES \
            and torch.is_grad_enabled() and (x.requires_grad or weight.requires_grad or bias.requires_grad):
        out = LinearFunction.apply(x.reshape(-1, x.shape[-1]), weight, bias)
        return out if x.dim() == 2 else out.view(*x.shape[:-1], weight.shape[0])
    return F.linear(x, weight, bias)


def linear(module, x):
    """``module(x)`` for an ``nn.Linear``."""
    return linear_wb(x, module.weight, module.bias)


def linear_zero_rows(module, x, zero_rows):
    """``module(x).masked_fill(zero_rows[..., None], 0)`` -- value_proj and its padding mask (reference
    models/ops/modules/ms_deform_attn.py:94-96).  x [rows, in_features]; bf16 inference: one kernel (the mask is applied in
    the GEMM epilogue); otherwise the projection followed by the in-place row-zeroing kernel."""
    if zero_rows is not None and _bf16_kernel_wanted(x, module.weight, module.bias):
        return linear_bf16(x, module.weight, module.bias, zero_rows=zero_rows)
    y = linear(module, x)
    if zero_rows is not None:
        # `y` is a fresh tensor consumed by the caller's next op and by nothing else
        y = zero_masked_rows_(y, zero_rows.reshape(-1), exclusive=True)
    return y


class LinearReLUFunction(Function):
    """relu(x @ W^T + b) with bias and ReLU in the GEMM epilogue (cuBLASLt through
    torch._addmm_activation): the pre-activation never reaches HBM.  bf16 training from BF16_TRAIN_KERNEL_MIN_ROWS rows up:
    the package's own kernels in both directions (_bf16_train_kernels_apply); fp32 training in fp32 train-GEMM mode
    "tf32x3": the three-term TF32 kernels in both directions (_fp32_train_kernels_apply)."""

    @staticmethod
    def forward(ctx, x, weight, bias, p=0.0, key=None):
        # with a key: dropout(relu(.)) at rate p; the saved output is the dropped one, and it alone gives the backward
        x2 = x.reshape(-1, x.shape[-1])
        ctx.kernels = any(ctx.needs_input_grad) and _bf16_train_kernels_apply(x2, weight, bias)
        ctx.tf32x3 = not ctx.kernels and any(ctx.needs_input_grad) and _fp32_train_kernels_apply(x2, weight, bias)
        fused = key is not None and _relu_dropout_epilogue_wins(weight.shape[0], weight.shape[1])
        if ctx.kernels:
            out = _linear_bf16_relu_dropout(x2, weight, bias, p, key) if fused else linear_bf16(x2, weight, bias, relu=True)
        elif ctx.tf32x3:
            w_split = _tf32_weight_split(weight, live=True)
            out = _linear_tf32x3_kernel(x2, *w_split, bias, relu=True, dropout=(p, key) if fused else None)
        else:
            out = torch._addmm_activation(bias, x2, weight.t(), use_gelu=False)
            fused = False
        if key is not None and not fused:
            _dropout_into(out, out, p, key)
        ctx.save_for_backward(x2, weight, out)
        ctx.x_shape = x.shape
        ctx.p = p if key is not None else None
        return out.view(*x.shape[:-1], weight.shape[0])

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        x2, weight, out = ctx.saved_tensors
        if ctx.p is None:
            g = torch.ops.aten.threshold_backward(grad.reshape(out.shape), out, 0)
        else:
            g = relu_dropout_grad(grad, out, ctx.p)
        if ctx.kernels:
            dx, dw, db = _bf16_linear_backward(ctx.needs_input_grad, g.contiguous(), x2, weight,
                                               (weight.dtype, weight.dtype))
        elif ctx.tf32x3:
            dx, dw, db = _tf32x3_linear_backward(ctx.needs_input_grad, g.contiguous(), x2, weight)
        else:
            dx = g @ weight if ctx.needs_input_grad[0] else None
            dw = g.t() @ x2 if ctx.needs_input_grad[1] else None
            db = column_sum(g) if ctx.needs_input_grad[2] else None
        return (None if dx is None else dx.view(ctx.x_shape)), dw, db, None, None


def _relu_dropout_epilogue_wins(n, k):
    """Dropout in the GEMM epilogue (bf16 and tf32x3 kernel routes) against the plain ReLU GEMM + the in-place dropout
    kernel.  Measured on one B200 (1000 W) at 88 892 rows, 1024 <- 256, bf16 forward + backward (tools/bench_dropout.py,
    DESIGN.md section 3.16): 0.354 ms in the epilogue, 0.389 ms as GEMM + dropout kernel, so the epilogue is taken."""
    return True


def _linear_bf16_relu_dropout(x2, weight, bias, p, key):
    """dropout(relu(x2 W^T + b)) -> a fresh bf16 [rows, n] on csrc/linear_bf16.cu, the mask applied in the epilogue."""
    n, k = weight.shape
    if not x2.is_contiguous() or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    w = weight.detach()
    if not w.is_contiguous() or w.data_ptr() % 16 != 0:
        w = w.contiguous()
    b = None if bias is None else bias.detach().contiguous()
    y = torch.empty((x2.shape[0], n), dtype=torch.bfloat16, device=x2.device)
    with torch.cuda.device(x2.device):
        code = _lib.load().msda_layer_linear_bf16_relu_dropout(
            x2.data_ptr(), w.data_ptr(), None if b is None else b.data_ptr(), x2.shape[0], n, k, float(p), key.data_ptr(),
            y.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_linear_bf16_relu_dropout")
    return y


def linear_relu(linear, x, dropout=None):
    """``dropout(relu(linear(x)))``; epilogue-fused on CUDA for 16-bit / fp32 dense inputs.  ``dropout`` is the layer's
    ``nn.Dropout`` or None."""
    mode = _dropout_mode(dropout, x)
    if mode == "module":
        return dropout(linear_relu(linear, x))
    if mode == "package":
        if x.dtype == linear.weight.dtype and linear.bias is not None:
            return LinearReLUFunction.apply(x, linear.weight, linear.bias, float(dropout.p), _dropout_key(x.device))
        return globals()["dropout"](dropout, linear_relu(linear, x))
    if _tf32x3_wanted(x, linear.weight):
        return linear_tf32x3(x, linear.weight, linear.bias, relu=True)
    if _bf16_kernel_wanted(x, linear.weight, linear.bias):
        return linear_bf16(x, linear.weight, linear.bias, relu=True)
    if x.is_cuda and linear.bias is not None and x.dtype == linear.weight.dtype and x.dtype in _DTYPES:
        return LinearReLUFunction.apply(x, linear.weight, linear.bias)
    return F.relu(linear(x))


def ffn_layer_norm_supported(x, linear1, linear2, norm):
    """The tcgen05 feed-forward kernel covers bf16 inference at d_model 256 (csrc/ffn_fused.cu)."""
    if not x.is_cuda or x.dtype != torch.bfloat16 or linear1.bias is None or linear2.bias is None:
        return False
    if torch.is_grad_enabled() and (x.requires_grad or linear1.weight.requires_grad or linear2.weight.requires_grad
                                    or norm.weight.requires_grad):
        return False                  # forward only: training keeps the hidden activation for autograd
    if any(t.dtype != torch.bfloat16 for t in (linear1.weight, linear2.weight, norm.weight)):
        return False
    c, f = x.shape[-1], linear1.out_features
    if linear1.in_features != c or linear2.in_features != f or linear2.out_features != c or \
            tuple(norm.normalized_shape) != (c,) or not norm.elementwise_affine or norm.bias is None:
        return False
    return bool(_lib.load().msda_layer_ffn_layernorm_supported(_lib.DTYPE_BF16, int(c), int(f)))


def ffn_layer_norm(linear1, linear2, norm, x, pos=None):
    """``norm(x + linear2(relu(linear1(x))))`` (and ``that + pos``) in ONE tensor-core kernel; call only
    when :func:`ffn_layer_norm_supported`."""
    shape = x.shape
    c = shape[-1]
    x2 = _dense(x.reshape(-1, c))
    rows = x2.shape[0]
    pos2 = None if pos is None else _dense(pos.to(x.dtype).expand(shape).reshape(-1, c))
    w1, b1, w2, b2 = (_dense(t.detach()) for t in (linear1.weight, linear1.bias, linear2.weight, linear2.bias))
    gamma, beta = _dense(norm.weight.detach()), _dense(norm.bias.detach())
    with torch.cuda.device(x.device):
        y = torch.empty_like(x2)
        y_pos = torch.empty_like(x2) if pos2 is not None else None
        code = _lib.load().msda_layer_ffn_layernorm_forward(
            _lib.DTYPE_BF16, x2.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
            gamma.data_ptr(), beta.data_ptr(), _ptr(pos2), rows, c, linear1.out_features, float(norm.eps),
            y.data_ptr(), _ptr(y_pos), torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_ffn_layernorm_forward")
    y = y.view(shape)
    return y if y_pos is None else (y, y_pos.view(shape))


def proj_layer_norm_supported(x, linear, norm):
    """The tcgen05 projection + residual + LayerNorm kernel covers bf16 inference at d_model 256 (csrc/proj_fused.cu)."""
    if not x.is_cuda or x.dtype != torch.bfloat16 or linear.bias is None:
        return False
    if torch.is_grad_enabled() and (x.requires_grad or linear.weight.requires_grad or norm.weight.requires_grad):
        return False
    if linear.weight.dtype != torch.bfloat16 or norm.weight.dtype != torch.bfloat16:
        return False
    c = x.shape[-1]
    if linear.in_features != c or linear.out_features != c or tuple(norm.normalized_shape) != (c,) or \
            not norm.elementwise_affine or norm.bias is None:
        return False
    return bool(_lib.load().msda_layer_proj_layernorm_supported(_lib.DTYPE_BF16, int(c), int(c)))


def proj_layer_norm(linear, norm, x, residual=None, pos=None):
    """``norm(residual + linear(x))`` (and ``that + pos``): the attention's output projection and the layer's
    residual + LayerNorm in ONE tensor-core kernel when :func:`proj_layer_norm_supported`; otherwise the
    GEMM + fused add-LayerNorm composition."""
    # with a `pos` output the one-kernel path (117 us at 8 x 22223 rows) loses to GEMM + fused norm (111 us): the
    # LayerNorm warps have no registers left to prefetch the pos rows.  The C ABI keeps the option; the layers use
    # the composition there.
    if pos is not None or not proj_layer_norm_supported(x, linear, norm) or (residual is not None and (
            residual.shape != x.shape or residual.dtype != x.dtype or
            (torch.is_grad_enabled() and residual.requires_grad))):
        return add_layer_norm(norm, globals()["linear"](linear, x), residual, None, pos)
    shape = x.shape
    c = shape[-1]
    x2 = _dense(x.reshape(-1, c))
    rows = x2.shape[0]
    res2 = None if residual is None else _dense(residual.reshape(-1, c))
    pos2 = None if pos is None else _dense(pos.to(x.dtype).expand(shape).reshape(-1, c))
    w, b = _dense(linear.weight.detach()), _dense(linear.bias.detach())
    gamma, beta = _dense(norm.weight.detach()), _dense(norm.bias.detach())
    with torch.cuda.device(x.device):
        y = torch.empty_like(x2)
        y_pos = torch.empty_like(x2) if pos2 is not None else None
        code = _lib.load().msda_layer_proj_layernorm_forward(
            _lib.DTYPE_BF16, x2.data_ptr(), w.data_ptr(), b.data_ptr(), _ptr(res2), gamma.data_ptr(), beta.data_ptr(),
            _ptr(pos2), rows, c, float(norm.eps), y.data_ptr(), _ptr(y_pos), torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "msda_layer_proj_layernorm_forward")
    y = y.view(shape)
    return y if y_pos is None else (y, y_pos.view(shape))


def flatten_levels(maps, channel_adds=None):
    """[N,C,H_l,W_l] per level -> tokens [N, sum_l H_l*W_l, C] (+ channel_adds[l] per level), one transposing
    kernel per level writing straight into its slice (no per-level transposes, adds and torch.cat).
    Forward only: callers keep the PyTorch composition when gradients are needed."""
    n, c = maps[0].shape[:2]
    dt = maps[0].dtype
    sizes = [m.shape[2] * m.shape[3] for m in maps]
    total = sum(sizes)
    lib = _lib.load()
    with torch.cuda.device(maps[0].device):
        out = torch.empty((n, total, c), dtype=dt, device=maps[0].device)
        start = 0
        stream = torch.cuda.current_stream().cuda_stream
        for lvl, (m, hw) in enumerate(zip(maps, sizes)):
            m = m.contiguous()
            add = None if channel_adds is None else channel_adds[lvl].detach().to(dt).contiguous()
            code = lib.msda_layer_flatten_level(_DTYPES[dt], m.data_ptr(), _ptr(add), n, c, hw, out.data_ptr(), total,
                                                start, stream)
            _lib.check(code, "msda_layer_flatten_level")
            start += hw
    return out


def flatten_levels_supported(maps):
    return all(m.is_cuda and m.dim() == 4 and m.dtype in _DTYPES and m.dtype == maps[0].dtype and
               m.shape[:2] == maps[0].shape[:2] for m in maps) and not (
        torch.is_grad_enabled() and any(m.requires_grad for m in maps))
