"""ctypes binding of libmsda_b200.so (C ABI declared in include/msda_b200.h).

The library is built in-tree by ``make`` in this directory (see ``__graft_entry__.build``).
There is no fallback: if the shared object is missing the import of the op fails loudly.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MSDA_B200_LIB selects another build of the same ABI (A/B kernel experiments); default: in-tree
LIB_PATH = os.environ.get("MSDA_B200_LIB") or os.path.join(_HERE, "libmsda_b200.so")

ABI_VERSION = 25
DTYPE_F32, DTYPE_F64, DTYPE_BF16, DTYPE_F16 = 0, 1, 2, 3
FLAG_FORCE_GENERIC = 1
FLAG_TC = 4
FLAG_VALUE_HEAD_MAJOR = 8

_lib = None


class MSDAError(RuntimeError):
    pass


def load():
    """Load the shared library once and declare the prototypes of include/msda_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MSDAError(
            f"{LIB_PATH} not found: the sm_100a CUDA library has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'` or `make` in the package "
            "directory). There is no CPU or PyTorch fallback for this op.")
    lib = ctypes.CDLL(LIB_PATH)
    c_int, c_vp = ctypes.c_int, ctypes.c_void_p
    lib.msda_abi_version.restype = c_int
    lib.msda_abi_version.argtypes = []
    lib.msda_error_string.restype = ctypes.c_char_p
    lib.msda_error_string.argtypes = [c_int]
    lib.msda_forward.restype = c_int
    lib.msda_forward.argtypes = [c_int, c_vp, c_vp, c_vp, c_vp, c_vp] + [c_int] * 7 + [c_vp, c_int, c_vp]
    lib.msda_backward.restype = c_int
    lib.msda_backward.argtypes = [c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp] + [c_int] * 7 + \
                                 [c_vp, c_vp, c_vp, c_vp, c_int, c_vp]
    c_i64, c_fp = ctypes.c_int64, ctypes.c_void_p
    lib.msda_fused_supported.restype = c_int
    lib.msda_fused_supported.argtypes = [c_int] * 8
    fused_common = [c_vp, c_vp, c_vp, c_fp, c_int, c_vp, c_i64, c_vp, c_i64] + [c_int] * 7
    lib.msda_fused_forward.restype = c_int
    lib.msda_fused_forward.argtypes = [c_int, c_int] + fused_common + [c_vp, c_vp]
    lib.msda_fused_forward_strided.restype = c_int
    lib.msda_fused_forward_strided.argtypes = [c_int, c_int, c_vp, c_i64] + fused_common[1:] + [c_vp, c_vp]
    lib.msda_fused_backward.restype = c_int
    lib.msda_fused_backward.argtypes = [c_int, c_int, c_vp] + fused_common + [c_vp, c_vp, c_vp, c_fp, c_vp, c_vp]
    lib.msda_deterministic_scratch_bytes.restype = c_i64
    lib.msda_deterministic_scratch_bytes.argtypes = [c_i64, c_i64, c_int]
    lib.msda_backward_deterministic.restype = c_int
    lib.msda_backward_deterministic.argtypes = lib.msda_backward.argtypes[:-1] + [c_vp, c_i64, c_vp]
    lib.msda_fused_backward_deterministic.restype = c_int
    lib.msda_fused_backward_deterministic.argtypes = lib.msda_fused_backward.argtypes[:-1] + [c_vp, c_i64, c_vp]
    lib.msda_fused_forward_head_major.restype = c_int
    lib.msda_fused_forward_head_major.argtypes = [c_int, c_int] + fused_common + [c_vp, c_vp]
    lib.msda_layer_value_proj_head_major_supported.restype = c_int
    lib.msda_layer_value_proj_head_major_supported.argtypes = [c_int, c_int, c_int]
    lib.msda_layer_value_proj_head_major.restype = c_int
    lib.msda_layer_value_proj_head_major.argtypes = [c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp]
    c_f = ctypes.c_float
    lib.msda_layer_add_layernorm_supported.restype = c_int
    lib.msda_layer_add_layernorm_supported.argtypes = [c_int, c_int]
    lib.msda_layer_add_layernorm_partial_blocks.restype = c_int
    lib.msda_layer_add_layernorm_partial_blocks.argtypes = [c_i64]
    lib.msda_layer_add_layernorm_forward.restype = c_int
    lib.msda_layer_add_layernorm_forward.argtypes = [c_int, c_int] + [c_vp] * 5 + [c_i64, c_int, c_f] + [c_vp] * 5
    lib.msda_layer_add_layernorm_backward.restype = c_int
    lib.msda_layer_add_layernorm_backward.argtypes = [c_int, c_int] + [c_vp] * 7 + [c_i64, c_int] + [c_vp] * 5 + \
                                                     [c_int, c_vp]
    lib.msda_layer_ffn_layernorm_supported.restype = c_int
    lib.msda_layer_ffn_layernorm_supported.argtypes = [c_int, c_int, c_int]
    lib.msda_layer_ffn_layernorm_forward.restype = c_int
    lib.msda_layer_ffn_layernorm_forward.argtypes = [c_int] + [c_vp] * 8 + [c_i64, c_int, c_int, c_f, c_vp, c_vp, c_vp]
    lib.msda_layer_flatten_level.restype = c_int
    lib.msda_layer_flatten_level.argtypes = [c_int, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_i64, c_i64, c_vp]
    for fn in (lib.msda_roi_align_forward, lib.msda_roi_align_backward):
        fn.restype = c_int
        fn.argtypes = [c_int, c_vp, c_vp] + [c_int] * 7 + [ctypes.c_double, c_int, c_int, c_vp, c_vp]
    lib.msda_roi_align_backward_deterministic.restype = c_int
    lib.msda_roi_align_backward_deterministic.argtypes = lib.msda_roi_align_backward.argtypes[:-1] + [c_vp, c_i64, c_vp]
    lib.msda_layer_proj_layernorm_supported.restype = c_int
    lib.msda_layer_proj_layernorm_supported.argtypes = [c_int, c_int, c_int]
    lib.msda_layer_proj_layernorm_forward.restype = c_int
    lib.msda_layer_proj_layernorm_forward.argtypes = [c_int] + [c_vp] * 7 + [c_i64, c_int, c_f, c_vp, c_vp, c_vp]
    lib.msda_layer_tf32_split.restype = c_int
    lib.msda_layer_tf32_split.argtypes = [c_vp, c_i64, c_int, c_vp, c_vp]
    lib.msda_layer_linear_bf16_supported.restype = c_int
    lib.msda_layer_linear_bf16_supported.argtypes = [c_int, c_int]
    lib.msda_layer_linear_bf16.restype = c_int
    lib.msda_layer_linear_bf16.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp]
    lib.msda_layer_linear_bf16_wgrad_supported.restype = c_int
    lib.msda_layer_linear_bf16_wgrad_supported.argtypes = [c_int, c_int]
    lib.msda_layer_linear_bf16_wgrad_scratch_floats.restype = c_i64
    lib.msda_layer_linear_bf16_wgrad_scratch_floats.argtypes = [c_i64, c_int, c_int]
    lib.msda_layer_linear_bf16_wgrad.restype = c_int
    lib.msda_layer_linear_bf16_wgrad.argtypes = [c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp]
    lib.msda_layer_linear_tf32x3_supported.restype = c_int
    lib.msda_layer_linear_tf32x3_supported.argtypes = [c_int, c_int]
    lib.msda_layer_linear_tf32x3.restype = c_int
    lib.msda_layer_linear_tf32x3.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp]
    lib.msda_layer_linear_tf32x3_wgrad_supported.restype = c_int
    lib.msda_layer_linear_tf32x3_wgrad_supported.argtypes = [c_int, c_int]
    lib.msda_layer_linear_tf32x3_wgrad_scratch_floats.restype = c_i64
    lib.msda_layer_linear_tf32x3_wgrad_scratch_floats.argtypes = [c_i64, c_int, c_int]
    lib.msda_layer_linear_tf32x3_wgrad.restype = c_int
    lib.msda_layer_linear_tf32x3_wgrad.argtypes = [c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp]
    lib.msda_layer_sine_coordinates.restype = c_int
    lib.msda_layer_sine_coordinates.argtypes = [c_vp, c_int, c_int, c_int, c_int, c_f, c_vp, c_vp, c_vp]
    lib.msda_layer_sine_position_tokens.restype = c_int
    lib.msda_layer_sine_position_tokens.argtypes = [c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_int, c_i64, c_vp, c_i64, c_i64,
                                                    c_vp]
    lib.msda_layer_group_norm_tokens_slabs.restype = c_int
    lib.msda_layer_group_norm_tokens_slabs.argtypes = [c_int, c_i64, c_int, c_int]
    lib.msda_layer_group_norm_tokens.restype = c_int
    lib.msda_layer_group_norm_tokens.argtypes = [c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_i64, c_int, c_int, c_f, c_i64,
                                                 c_vp, c_int, c_vp, c_vp]
    lib.msda_layer_norm_act_supported.restype = c_int
    lib.msda_layer_norm_act_supported.argtypes = [c_int, c_int]
    lib.msda_layer_norm_act_forward.restype = c_int
    lib.msda_layer_norm_act_forward.argtypes = [c_int, c_vp, c_vp, c_vp, c_i64, c_int, c_f, c_int, c_vp, c_vp]
    lib.msda_layer_dropout_rule.restype = c_int
    lib.msda_layer_dropout_rule.argtypes = [c_f, ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(c_f)]
    lib.msda_layer_add_layernorm_dropout_supported.restype = c_int
    lib.msda_layer_add_layernorm_dropout_supported.argtypes = [c_int, c_int]
    lib.msda_layer_add_layernorm_dropout_forward.restype = c_int
    lib.msda_layer_add_layernorm_dropout_forward.argtypes = lib.msda_layer_add_layernorm_forward.argtypes[:-1] + \
        [c_f, c_vp, c_vp]
    lib.msda_layer_add_layernorm_dropout_backward.restype = c_int
    lib.msda_layer_add_layernorm_dropout_backward.argtypes = lib.msda_layer_add_layernorm_backward.argtypes[:-1] + \
        [c_f, c_vp, c_vp]
    lib.msda_layer_dropout.restype = c_int
    lib.msda_layer_dropout.argtypes = [c_int, c_vp, c_vp, c_i64, c_f, c_vp, c_vp]
    lib.msda_layer_relu_dropout_grad.restype = c_int
    lib.msda_layer_relu_dropout_grad.argtypes = [c_int, c_vp, c_vp, c_vp, c_i64, c_f, c_vp]
    lib.msda_layer_linear_bf16_relu_dropout.restype = c_int
    lib.msda_layer_linear_bf16_relu_dropout.argtypes = [c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_f, c_vp, c_vp, c_vp]
    lib.msda_layer_linear_tf32x3_relu_dropout.restype = c_int
    lib.msda_layer_linear_tf32x3_relu_dropout.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_f, c_vp, c_vp,
                                                          c_vp]
    lib.msda_layer_colsum_blocks.restype = c_int
    lib.msda_layer_colsum_blocks.argtypes = [c_int, c_i64, c_int]
    lib.msda_layer_colsum.restype = c_int
    lib.msda_layer_colsum.argtypes = [c_int, c_vp, c_i64, c_int, c_vp, c_vp, c_int, c_vp]
    lib.msda_layer_zero_masked_rows.restype = c_int
    lib.msda_layer_zero_masked_rows.argtypes = [c_int, c_vp, c_vp, c_i64, c_int, c_vp]
    lib.msda_linear_assignment_scratch_bytes.restype = c_i64
    lib.msda_linear_assignment_scratch_bytes.argtypes = [c_int, c_int, c_int]
    lib.msda_linear_assignment.restype = c_int
    lib.msda_linear_assignment.argtypes = [c_vp, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_i64,
                                           c_vp]
    if lib.msda_abi_version() != ABI_VERSION:
        raise MSDAError(f"libmsda_b200.so ABI {lib.msda_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def deterministic_scratch(device, grad_elements, grad_reference_elements=0, num_heads=0):
    """Scratch of the *_deterministic calls, from torch's caching allocator."""
    import torch
    nbytes = load().msda_deterministic_scratch_bytes(int(grad_elements), int(grad_reference_elements), int(num_heads))
    if nbytes < 0:
        raise MSDAError(f"msda_deterministic_scratch_bytes({grad_elements}, {grad_reference_elements}) failed")
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def check(code, what):
    if code != 0:
        msg = load().msda_error_string(code).decode()
        raise MSDAError(f"{what} failed: CUDA error {code} ({msg})")
