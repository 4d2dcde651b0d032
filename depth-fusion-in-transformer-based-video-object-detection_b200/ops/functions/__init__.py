from .ms_deform_attn_func import MSDeformAttnFunction
from .ms_deform_attn_fused_func import (MSDeformAttnFusedFunction, fused_supported, head_major_supported,
                                         value_proj_head_major, fused_forward_head_major)
from .layer_epilogue_func import add_layer_norm, norm_act, proj_layer_norm, proj_layer_norm_supported, flatten_levels, flatten_levels_supported, ffn_layer_norm, ffn_layer_norm_supported, column_sum, linear, linear_relu, linear_wb, zero_masked_rows_, set_fp32_gemm_mode, set_fp32_train_gemm_mode, linear_tf32x3, linear_tf32x3_wgrad, linear_bf16, linear_bf16_wgrad, linear_zero_rows, dropout

__all__ = ["MSDeformAttnFunction", "MSDeformAttnFusedFunction", "fused_supported",
           "add_layer_norm", "norm_act", "proj_layer_norm", "proj_layer_norm_supported", "flatten_levels", "flatten_levels_supported", "ffn_layer_norm", "ffn_layer_norm_supported", "column_sum", "linear", "linear_relu", "linear_wb", "zero_masked_rows_", "set_fp32_gemm_mode", "set_fp32_train_gemm_mode", "linear_tf32x3", "linear_tf32x3_wgrad", "linear_bf16", "linear_bf16_wgrad", "linear_zero_rows", "dropout"]
