// C-ABI entry points of libmsda_b200.so (declared in include/msda_b200.h).
#include "../../include/msda_b200.h"
#include "msda_launch.h"

static bool bad_dims(int N, int S, int M, int D, int L, int Lq, int P)
{
    return N < 0 || S < 0 || M < 0 || D < 0 || L < 0 || Lq < 0 || P < 0;
}

extern "C" int msda_abi_version(void) { return 25; }

extern "C" const char* msda_error_string(int code)
{
    return cudaGetErrorString((cudaError_t)code);
}

extern "C" int msda_forward(int dtype, const void* value, const int64_t* spatial_shapes,
                            const int64_t* level_start_index, const void* sampling_loc,
                            const void* attn_weight, int batch, int spatial_size, int num_heads,
                            int channels, int num_levels, int num_query, int num_point, void* output,
                            int flags, void* stream)
{
    if (dtype < 0 || dtype > 3 || bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point))
        return (int)cudaErrorInvalidValue;
    msda::FwdArgs a;
    a.dtype = dtype;
    a.value = value; a.shapes = spatial_shapes; a.lsi = level_start_index;
    a.loc = sampling_loc; a.attn = attn_weight; a.out = output;
    a.N = batch; a.S = spatial_size; a.M = num_heads; a.D = channels;
    a.L = num_levels; a.Lq = num_query; a.P = num_point;
    a.force_generic = (flags & MSDA_FLAG_FORCE_GENERIC) ? 1 : 0;
    a.no_tc = (flags & MSDA_FLAG_TC) ? 0 : 1;
    a.head_major = (flags & MSDA_FLAG_VALUE_HEAD_MAJOR) ? 1 : 0;
    if (num_levels == 0 || num_point == 0) {   // empty sum: output is all zeros
        const size_t esz = dtype == MSDA_DTYPE_F64 ? 8 : (dtype == MSDA_DTYPE_F32 ? 4 : 2);
        return (int)cudaMemsetAsync(output, 0, (size_t)batch * num_query * num_heads * channels * esz,
                                    (cudaStream_t)stream);
    }
    if (a.head_major) return (int)msda::forward_hm(a, (cudaStream_t)stream);
    return (int)msda::forward(a, (cudaStream_t)stream);
}

extern "C" int msda_backward(int dtype, const void* grad_output, const void* value,
                             const int64_t* spatial_shapes, const int64_t* level_start_index,
                             const void* sampling_loc, const void* attn_weight, int batch,
                             int spatial_size, int num_heads, int channels, int num_levels,
                             int num_query, int num_point, void* grad_value, void* grad_sampling_loc,
                             void* grad_attn_weight, void* grad_value_accum_f32, int flags, void* stream)
{
    if (dtype < 0 || dtype > 3 || bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point))
        return (int)cudaErrorInvalidValue;
    msda::BwdArgs a;
    a.dtype = dtype;
    a.grad_out = grad_output; a.value = value; a.shapes = spatial_shapes; a.lsi = level_start_index;
    a.loc = sampling_loc; a.attn = attn_weight;
    a.grad_value = grad_value; a.grad_loc = grad_sampling_loc; a.grad_attn = grad_attn_weight;
    a.grad_value_accum = (float*)grad_value_accum_f32;
    a.N = batch; a.S = spatial_size; a.M = num_heads; a.D = channels;
    a.L = num_levels; a.Lq = num_query; a.P = num_point;
    a.force_generic = (flags & MSDA_FLAG_FORCE_GENERIC) ? 1 : 0;
    a.no_tc = (flags & MSDA_FLAG_TC) ? 0 : 1;
    return (int)msda::backward(a, (cudaStream_t)stream);
}

extern "C" int64_t msda_deterministic_scratch_bytes(int64_t grad_elements, int64_t grad_reference_elements,
                                                   int num_heads)
{
    if (grad_elements < 0 || grad_reference_elements < 0 || num_heads < 0) return -1;
    return (int64_t)msda::det_scratch_bytes((long long)grad_elements, (long long)grad_reference_elements * num_heads);
}

extern "C" int msda_backward_deterministic(int dtype, const void* grad_output, const void* value,
                                           const int64_t* spatial_shapes, const int64_t* level_start_index,
                                           const void* sampling_loc, const void* attn_weight, int batch,
                                           int spatial_size, int num_heads, int channels, int num_levels,
                                           int num_query, int num_point, void* grad_value, void* grad_sampling_loc,
                                           void* grad_attn_weight, void* grad_value_accum_f32, int flags,
                                           void* scratch, int64_t scratch_bytes, void* stream)
{
    (void)grad_value_accum_f32;
    if (dtype < 0 || dtype > 3 || bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point) ||
        (flags & MSDA_FLAG_TC))
        return (int)cudaErrorInvalidValue;
    msda::BwdArgs a;
    a.dtype = dtype;
    a.grad_out = grad_output; a.value = value; a.shapes = spatial_shapes; a.lsi = level_start_index;
    a.loc = sampling_loc; a.attn = attn_weight;
    a.grad_value = grad_value; a.grad_loc = grad_sampling_loc; a.grad_attn = grad_attn_weight;
    a.grad_value_accum = nullptr;
    a.N = batch; a.S = spatial_size; a.M = num_heads; a.D = channels;
    a.L = num_levels; a.Lq = num_query; a.P = num_point;
    a.force_generic = (flags & MSDA_FLAG_FORCE_GENERIC) ? 1 : 0;
    a.no_tc = 1;
    return (int)msda::backward_deterministic(a, scratch, (long long)scratch_bytes, (cudaStream_t)stream);
}

static msda::FusedArgs make_fused(int dtype, int raw_dtype, const void* value, const int64_t* shapes,
                                  const int64_t* lsi, const float* ref, int ref_dim, const void* offsets,
                                  int64_t off_stride, const void* logits, int64_t logit_stride, int N, int S,
                                  int M, int D, int L, int Lq, int P)
{
    msda::FusedArgs a = {};
    a.dtype = dtype; a.raw_dtype = raw_dtype;
    a.value = value; a.shapes = shapes; a.lsi = lsi; a.ref = ref; a.ref_dim = ref_dim;
    a.offsets = offsets; a.off_stride = off_stride; a.logits = logits; a.logit_stride = logit_stride;
    a.N = N; a.S = S; a.M = M; a.D = D; a.L = L; a.Lq = Lq; a.P = P;
    return a;
}

extern "C" int msda_fused_supported(int dtype, int raw_dtype, int ref_dim, int spatial_size, int num_heads,
                                    int channels, int num_levels, int num_point)
{
    msda::FusedArgs a = make_fused(dtype, raw_dtype, nullptr, nullptr, nullptr, nullptr, ref_dim, nullptr, 0,
                                   nullptr, 0, 1, spatial_size, num_heads, channels, num_levels, 1, num_point);
    return msda::fused_supported(a) ? 1 : 0;
}

extern "C" int msda_fused_forward(int dtype, int raw_dtype, const void* value, const int64_t* spatial_shapes,
                                  const int64_t* level_start_index, const float* reference_points, int ref_dim,
                                  const void* sampling_offsets_raw, int64_t offsets_query_stride,
                                  const void* attention_logits_raw, int64_t logits_query_stride, int batch,
                                  int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                  int num_point, void* output, void* stream)
{
    if (bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point))
        return (int)cudaErrorInvalidValue;
    msda::FusedArgs a = make_fused(dtype, raw_dtype, value, spatial_shapes, level_start_index, reference_points,
                                   ref_dim, sampling_offsets_raw, offsets_query_stride, attention_logits_raw,
                                   logits_query_stride, batch, spatial_size, num_heads, channels, num_levels,
                                   num_query, num_point);
    a.out = output;
    return (int)msda::fused_forward(a, (cudaStream_t)stream);
}

extern "C" int msda_fused_forward_strided(int dtype, int raw_dtype, const void* value, int64_t value_pixel_stride,
                                          const int64_t* spatial_shapes, const int64_t* level_start_index,
                                          const float* reference_points, int ref_dim,
                                          const void* sampling_offsets_raw, int64_t offsets_query_stride,
                                          const void* attention_logits_raw, int64_t logits_query_stride, int batch,
                                          int spatial_size, int num_heads, int channels, int num_levels,
                                          int num_query, int num_point, void* output, void* stream)
{
    if (bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point) || value_pixel_stride < 0)
        return (int)cudaErrorInvalidValue;
    msda::FusedArgs a = make_fused(dtype, raw_dtype, value, spatial_shapes, level_start_index, reference_points,
                                   ref_dim, sampling_offsets_raw, offsets_query_stride, attention_logits_raw,
                                   logits_query_stride, batch, spatial_size, num_heads, channels, num_levels,
                                   num_query, num_point);
    a.out = output;
    a.value_ld = (long long)value_pixel_stride;
    return (int)msda::fused_forward(a, (cudaStream_t)stream);
}

extern "C" int msda_fused_backward(int dtype, int raw_dtype, const void* grad_output, const void* value,
                                   const int64_t* spatial_shapes, const int64_t* level_start_index,
                                   const float* reference_points, int ref_dim, const void* sampling_offsets_raw,
                                   int64_t offsets_query_stride, const void* attention_logits_raw,
                                   int64_t logits_query_stride, int batch, int spatial_size, int num_heads,
                                   int channels, int num_levels, int num_query, int num_point, void* grad_value,
                                   void* grad_offsets_raw, void* grad_logits_raw, float* grad_reference_points,
                                   void* grad_value_accum_f32, void* stream)
{
    if (bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point))
        return (int)cudaErrorInvalidValue;
    msda::FusedArgs a = make_fused(dtype, raw_dtype, value, spatial_shapes, level_start_index, reference_points,
                                   ref_dim, sampling_offsets_raw, offsets_query_stride, attention_logits_raw,
                                   logits_query_stride, batch, spatial_size, num_heads, channels, num_levels,
                                   num_query, num_point);
    a.grad_out = grad_output;
    a.grad_value = grad_value; a.grad_offsets = grad_offsets_raw; a.grad_logits = grad_logits_raw;
    a.grad_ref = grad_reference_points; a.grad_value_accum = (float*)grad_value_accum_f32;
    return (int)msda::fused_backward(a, (cudaStream_t)stream);
}

extern "C" int msda_fused_backward_deterministic(int dtype, int raw_dtype, const void* grad_output, const void* value,
                                                 const int64_t* spatial_shapes, const int64_t* level_start_index,
                                                 const float* reference_points, int ref_dim,
                                                 const void* sampling_offsets_raw, int64_t offsets_query_stride,
                                                 const void* attention_logits_raw, int64_t logits_query_stride,
                                                 int batch, int spatial_size, int num_heads, int channels,
                                                 int num_levels, int num_query, int num_point, void* grad_value,
                                                 void* grad_offsets_raw, void* grad_logits_raw,
                                                 float* grad_reference_points, void* grad_value_accum_f32,
                                                 void* scratch, int64_t scratch_bytes, void* stream)
{
    (void)grad_value_accum_f32;
    if (bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point))
        return (int)cudaErrorInvalidValue;
    msda::FusedArgs a = make_fused(dtype, raw_dtype, value, spatial_shapes, level_start_index, reference_points,
                                   ref_dim, sampling_offsets_raw, offsets_query_stride, attention_logits_raw,
                                   logits_query_stride, batch, spatial_size, num_heads, channels, num_levels,
                                   num_query, num_point);
    a.grad_out = grad_output;
    a.grad_value = grad_value; a.grad_offsets = grad_offsets_raw; a.grad_logits = grad_logits_raw;
    a.grad_ref = grad_reference_points;
    return (int)msda::fused_backward_deterministic(a, scratch, (long long)scratch_bytes, (cudaStream_t)stream);
}

// ---- layer epilogues --------------------------------------------------------------------------
extern "C" int msda_layer_add_layernorm_supported(int dtype, int channels)
{
    return msda::add_layernorm_chunks(dtype, channels) > 0 ? 1 : 0;
}

extern "C" int msda_layer_add_layernorm_partial_blocks(int64_t rows)
{
    return msda::add_layernorm_partial_blocks((long long)rows);
}

static int add_layernorm_forward(int dtype, int act, const void* branch, const void* residual, const void* gamma,
                                 const void* beta, const void* pos, int64_t rows, int channels, float eps, void* y,
                                 void* y_pos, float* mean, float* rstd, const uint64_t* drop_key, msda::DropoutRule drop,
                                 void* stream)
{
    if (rows < 0 || msda::add_layernorm_chunks(dtype, channels) == 0 || (y_pos != nullptr) != (pos != nullptr) ||
        (mean != nullptr) != (rstd != nullptr))
        return (int)cudaErrorInvalidValue;
    msda::AddLayerNormArgs a = {};
    a.dtype = dtype; a.act = act; a.rows = rows; a.C = channels; a.eps = eps;
    a.branch = branch; a.residual = residual; a.gamma = gamma; a.beta = beta; a.pos = pos;
    a.y = y; a.y_pos = y_pos; a.mean = mean; a.rstd = rstd;
    a.drop_key = reinterpret_cast<const unsigned long long*>(drop_key); a.drop = drop;
    return (int)msda::add_layernorm(a, false, (cudaStream_t)stream);
}

extern "C" int msda_layer_add_layernorm_forward(int dtype, int act, const void* branch, const void* residual,
                                                const void* gamma, const void* beta, const void* pos,
                                                int64_t rows, int channels, float eps, void* y, void* y_pos,
                                                float* mean, float* rstd, void* stream)
{
    return add_layernorm_forward(dtype, act, branch, residual, gamma, beta, pos, rows, channels, eps, y, y_pos, mean, rstd,
                                 nullptr, msda::DropoutRule{0u, 1.f}, stream);
}

static int add_layernorm_backward(int dtype, int act, const void* grad_y, const void* grad_y_pos, const void* branch,
                                  const void* residual, const void* gamma, const float* mean, const float* rstd,
                                  int64_t rows, int channels, void* grad_branch, void* grad_residual, void* grad_gamma,
                                  void* grad_beta, float* partial_scratch, int partial_blocks, const uint64_t* drop_key,
                                  msda::DropoutRule drop, void* stream)
{
    if (rows < 0 || msda::add_layernorm_chunks(dtype, channels) == 0 || partial_blocks < 1 ||
        partial_blocks > msda::add_layernorm_partial_blocks((long long)rows) ||
        (grad_residual == nullptr) != (residual == nullptr))
        return (int)cudaErrorInvalidValue;
    msda::AddLayerNormArgs a = {};
    a.drop_key = reinterpret_cast<const unsigned long long*>(drop_key); a.drop = drop;
    a.dtype = dtype; a.act = act; a.rows = rows; a.C = channels;
    a.branch = branch; a.residual = residual; a.gamma = gamma;
    a.mean = const_cast<float*>(mean); a.rstd = const_cast<float*>(rstd);
    a.dy = grad_y; a.dy_pos = grad_y_pos; a.d_branch = grad_branch; a.d_residual = grad_residual;
    a.d_gamma = grad_gamma; a.d_beta = grad_beta; a.partial = partial_scratch; a.partial_blocks = partial_blocks;
    if (rows == 0) {     // no rows: parameter gradients are zero
        const size_t esz = dtype == MSDA_DTYPE_F32 ? 4 : 2;
        cudaError_t e = cudaMemsetAsync(grad_gamma, 0, channels * esz, (cudaStream_t)stream);
        if (e != cudaSuccess) return (int)e;
        return (int)cudaMemsetAsync(grad_beta, 0, channels * esz, (cudaStream_t)stream);
    }
    return (int)msda::add_layernorm(a, true, (cudaStream_t)stream);
}

extern "C" int msda_layer_add_layernorm_backward(int dtype, int act, const void* grad_y, const void* grad_y_pos,
                                                 const void* branch, const void* residual, const void* gamma,
                                                 const float* mean, const float* rstd, int64_t rows, int channels,
                                                 void* grad_branch, void* grad_residual, void* grad_gamma,
                                                 void* grad_beta, float* partial_scratch, int partial_blocks,
                                                 void* stream)
{
    return add_layernorm_backward(dtype, act, grad_y, grad_y_pos, branch, residual, gamma, mean, rstd, rows, channels,
                                  grad_branch, grad_residual, grad_gamma, grad_beta, partial_scratch, partial_blocks,
                                  nullptr, msda::DropoutRule{0u, 1.f}, stream);
}

// ---- dropout (DESIGN.md section 3.16) ------------------------------------------------------------
extern "C" int msda_layer_dropout_rule(float p, uint32_t* threshold, float* scale)
{
    msda::DropoutRule r;
    if (!msda::dropout_rule(p, &r) || threshold == nullptr || scale == nullptr) return (int)cudaErrorInvalidValue;
    *threshold = r.thresh;
    *scale = r.scale;
    return 0;
}

extern "C" int msda_layer_add_layernorm_dropout_supported(int dtype, int channels)
{
    return msda::add_layernorm_dropout_supported(dtype, channels) ? 1 : 0;
}

extern "C" int msda_layer_add_layernorm_dropout_forward(int dtype, int act, const void* branch, const void* residual,
                                                        const void* gamma, const void* beta, const void* pos,
                                                        int64_t rows, int channels, float eps, void* y, void* y_pos,
                                                        float* mean, float* rstd, float p, const uint64_t* key,
                                                        void* stream)
{
    msda::DropoutRule r;
    if (!msda::dropout_rule(p, &r) || key == nullptr || !msda::add_layernorm_dropout_supported(dtype, channels))
        return (int)cudaErrorInvalidValue;
    return add_layernorm_forward(dtype, act, branch, residual, gamma, beta, pos, rows, channels, eps, y, y_pos, mean, rstd,
                                 key, r, stream);
}

extern "C" int msda_layer_add_layernorm_dropout_backward(int dtype, int act, const void* grad_y, const void* grad_y_pos,
                                                         const void* branch, const void* residual, const void* gamma,
                                                         const float* mean, const float* rstd, int64_t rows,
                                                         int channels, void* grad_branch, void* grad_residual,
                                                         void* grad_gamma, void* grad_beta, float* partial_scratch,
                                                         int partial_blocks, float p, const uint64_t* key, void* stream)
{
    msda::DropoutRule r;
    if (!msda::dropout_rule(p, &r) || key == nullptr || !msda::add_layernorm_dropout_supported(dtype, channels) ||
        grad_branch == nullptr || grad_branch == grad_residual)
        return (int)cudaErrorInvalidValue;
    return add_layernorm_backward(dtype, act, grad_y, grad_y_pos, branch, residual, gamma, mean, rstd, rows, channels,
                                  grad_branch, grad_residual, grad_gamma, grad_beta, partial_scratch, partial_blocks, key,
                                  r, stream);
}

extern "C" int msda_layer_dropout(int dtype, const void* x, void* y, int64_t n, float p, const uint64_t* key, void* stream)
{
    msda::DropoutRule r;
    if (!msda::dropout_rule(p, &r) || key == nullptr) return (int)cudaErrorInvalidValue;
    return (int)msda::dropout(dtype, x, y, (long long)n, reinterpret_cast<const unsigned long long*>(key), r,
                              (cudaStream_t)stream);
}

extern "C" int msda_layer_relu_dropout_grad(int dtype, const void* grad_y, const void* y, void* grad_x, int64_t n, float p,
                                            void* stream)
{
    msda::DropoutRule r;
    if (!msda::dropout_rule(p, &r)) return (int)cudaErrorInvalidValue;
    return (int)msda::relu_dropout_grad(dtype, grad_y, y, grad_x, (long long)n, r.scale, (cudaStream_t)stream);
}

extern "C" int msda_layer_zero_masked_rows(int dtype, void* data, const uint8_t* mask, int64_t rows, int channels,
                                           void* stream)
{
    if (rows < 0 || channels < 0) return (int)cudaErrorInvalidValue;
    return (int)msda::zero_masked_rows(dtype, data, mask, (long long)rows, channels, (cudaStream_t)stream);
}

extern "C" int msda_layer_colsum_blocks(int dtype, int64_t rows, int channels)
{
    return rows < 0 ? 0 : msda::colsum_blocks(dtype, (long long)rows, channels);
}

extern "C" int msda_layer_colsum(int dtype, const void* x, int64_t rows, int channels, void* out,
                                 float* partial_scratch, int partial_blocks, void* stream)
{
    if (rows < 0) return (int)cudaErrorInvalidValue;
    return (int)msda::colsum(dtype, x, (long long)rows, channels, out, partial_scratch, partial_blocks,
                             (cudaStream_t)stream);
}

// ---- fused feed-forward block (tcgen05) ------------------------------------------------------------
extern "C" int msda_layer_ffn_layernorm_supported(int dtype, int d_model, int d_ffn)
{
    return msda::ffn_layernorm_supported(dtype, d_model, d_ffn) ? 1 : 0;
}

extern "C" int msda_layer_ffn_layernorm_forward(int dtype, const void* x, const void* w1, const void* b1,
                                                const void* w2, const void* b2, const void* gamma,
                                                const void* beta, const void* pos, int64_t rows, int d_model,
                                                int d_ffn, float eps, void* y, void* y_pos, void* stream)
{
    if (rows < 0) return (int)cudaErrorInvalidValue;
    msda::FfnArgs a = {};
    a.dtype = dtype; a.rows = rows; a.C = d_model; a.F = d_ffn; a.eps = eps;
    a.x = x; a.w1 = w1; a.b1 = b1; a.w2 = w2; a.b2 = b2; a.gamma = gamma; a.beta = beta; a.pos = pos;
    a.y = y; a.y_pos = y_pos;
    return (int)msda::ffn_layernorm_forward(a, (cudaStream_t)stream);
}

extern "C" int msda_layer_flatten_level(int dtype, const void* feature_map, const void* channel_add, int batch,
                                        int channels, int height_x_width, void* tokens, int64_t tokens_per_item,
                                        int64_t level_start, void* stream)
{
    if (batch < 0 || channels < 0 || height_x_width < 0 || level_start < 0 ||
        level_start + height_x_width > tokens_per_item)
        return (int)cudaErrorInvalidValue;
    return (int)msda::flatten_level(dtype, feature_map, channel_add, tokens, batch, channels, height_x_width,
                                    (long long)tokens_per_item, (long long)level_start, (cudaStream_t)stream);
}

static bool bad_roi_dims(int batch, int height, int width, int channels, int num_rois, int ph, int pw)
{
    return batch < 0 || height <= 0 || width <= 0 || channels < 0 || num_rois < 0 || ph <= 0 || pw <= 0;
}

extern "C" int msda_roi_align_forward(int dtype, const void* feature_tokens, const void* rois, int batch, int height,
                                      int width, int channels, int num_rois, int pooled_height, int pooled_width,
                                      double spatial_scale, int sampling_ratio, int aligned, void* pooled, void* stream)
{
    if (bad_roi_dims(batch, height, width, channels, num_rois, pooled_height, pooled_width) || sampling_ratio < 0)
        return (int)cudaErrorInvalidValue;
    msda::RoiAlignArgs a{};
    a.dtype = dtype; a.feat = feature_tokens; a.rois = rois; a.out = pooled;
    a.N = batch; a.H = height; a.W = width; a.C = channels; a.K = num_rois; a.PH = pooled_height; a.PW = pooled_width;
    a.scale = spatial_scale; a.sampling_ratio = sampling_ratio; a.aligned = aligned;
    return (int)msda::roi_align_forward(a, (cudaStream_t)stream);
}

extern "C" int msda_roi_align_backward(int dtype, const void* grad_pooled, const void* rois, int batch, int height,
                                       int width, int channels, int num_rois, int pooled_height, int pooled_width,
                                       double spatial_scale, int sampling_ratio, int aligned, void* grad_feature_accum,
                                       void* stream)
{
    if (bad_roi_dims(batch, height, width, channels, num_rois, pooled_height, pooled_width) || sampling_ratio < 0)
        return (int)cudaErrorInvalidValue;
    msda::RoiAlignArgs a{};
    a.dtype = dtype; a.grad_out = grad_pooled; a.rois = rois; a.grad_accum = grad_feature_accum;
    a.N = batch; a.H = height; a.W = width; a.C = channels; a.K = num_rois; a.PH = pooled_height; a.PW = pooled_width;
    a.scale = spatial_scale; a.sampling_ratio = sampling_ratio; a.aligned = aligned;
    return (int)msda::roi_align_backward(a, (cudaStream_t)stream);
}

extern "C" int msda_roi_align_backward_deterministic(int dtype, const void* grad_pooled, const void* rois, int batch,
                                                     int height, int width, int channels, int num_rois,
                                                     int pooled_height, int pooled_width, double spatial_scale,
                                                     int sampling_ratio, int aligned, void* grad_feature,
                                                     void* scratch, int64_t scratch_bytes, void* stream)
{
    if (bad_roi_dims(batch, height, width, channels, num_rois, pooled_height, pooled_width) || sampling_ratio < 0)
        return (int)cudaErrorInvalidValue;
    msda::RoiAlignArgs a{};
    a.dtype = dtype; a.grad_out = grad_pooled; a.rois = rois; a.grad_accum = grad_feature;
    a.N = batch; a.H = height; a.W = width; a.C = channels; a.K = num_rois; a.PH = pooled_height; a.PW = pooled_width;
    a.scale = spatial_scale; a.sampling_ratio = sampling_ratio; a.aligned = aligned;
    return (int)msda::roi_align_backward_deterministic(a, scratch, (long long)scratch_bytes, (cudaStream_t)stream);
}

extern "C" int msda_layer_norm_act_supported(int dtype, int channels)
{
    return msda::norm_act_supported(dtype, channels) ? 1 : 0;
}

extern "C" int msda_layer_norm_act_forward(int dtype, const void* x, const void* gamma, const void* beta, int64_t rows,
                                           int channels, float eps, int act, void* y, void* stream)
{
    if (rows < 0) return (int)cudaErrorInvalidValue;
    return (int)msda::norm_act_forward(dtype, x, gamma, beta, y, (long long)rows, channels, eps, act,
                                       (cudaStream_t)stream);
}

extern "C" int msda_layer_group_norm_tokens_slabs(int dtype, int64_t tokens_per_item, int channels, int groups)
{
    return msda::group_norm_tokens_slabs(dtype, (long long)tokens_per_item, channels, groups);
}

extern "C" int msda_layer_group_norm_tokens(int dtype, const void* x, const void* channel_bias, const void* gamma,
                                            const void* beta, int batch, int64_t tokens_per_item, int channels,
                                            int groups, float eps, int64_t item_stride, float* partial_scratch,
                                            int slabs, void* y, void* stream)
{
    if (batch < 0 || tokens_per_item < 0 || item_stride < 0) return (int)cudaErrorInvalidValue;
    if (tokens_per_item == 0) return 0;
    return (int)msda::group_norm_tokens(dtype, x, channel_bias, gamma, beta, y, partial_scratch, batch,
                                        (long long)tokens_per_item, channels, groups, slabs, eps,
                                        (long long)item_stride, (cudaStream_t)stream);
}

extern "C" int msda_fused_forward_head_major(int dtype, int raw_dtype, const void* value_hm, const int64_t* spatial_shapes,
                                             const int64_t* level_start_index, const float* reference_points, int ref_dim,
                                             const void* sampling_offsets_raw, int64_t offsets_query_stride,
                                             const void* attention_logits_raw, int64_t logits_query_stride, int batch,
                                             int spatial_size, int num_heads, int channels, int num_levels, int num_query,
                                             int num_point, void* output, void* stream)
{
    if (bad_dims(batch, spatial_size, num_heads, channels, num_levels, num_query, num_point))
        return (int)cudaErrorInvalidValue;
    msda::FusedArgs a = make_fused(dtype, raw_dtype, value_hm, spatial_shapes, level_start_index, reference_points,
                                   ref_dim, sampling_offsets_raw, offsets_query_stride, attention_logits_raw,
                                   logits_query_stride, batch, spatial_size, num_heads, channels, num_levels,
                                   num_query, num_point);
    a.out = output;
    return (int)msda::fused_forward_hm(a, (cudaStream_t)stream);
}

extern "C" int msda_layer_value_proj_head_major_supported(int dtype, int d_model, int num_heads)
{
    return msda::value_proj_hm_supported(dtype, d_model, num_heads) ? 1 : 0;
}

extern "C" int msda_layer_value_proj_head_major(int dtype, const void* x, const void* weight, const void* bias,
                                                const unsigned char* padding_mask, int64_t rows, int tokens_per_frame,
                                                int d_model, int num_heads, void* value_hm, void* stream)
{
    if (rows < 0 || !msda::value_proj_hm_supported(dtype, d_model, num_heads)) return (int)cudaErrorInvalidValue;
    return (int)msda::value_proj_hm(dtype, x, weight, bias, padding_mask, value_hm, (long long)rows, tokens_per_frame,
                                    (cudaStream_t)stream);
}

extern "C" int msda_layer_proj_layernorm_supported(int dtype, int d_in, int d_out)
{
    return msda::proj_layernorm_supported(dtype, d_in, d_out) ? 1 : 0;
}

extern "C" int msda_layer_proj_layernorm_forward(int dtype, const void* x, const void* weight, const void* bias,
                                                 const void* residual, const void* gamma, const void* beta,
                                                 const void* pos, int64_t rows, int d_model, float eps, void* y,
                                                 void* y_pos, void* stream)
{
    if (rows < 0) return (int)cudaErrorInvalidValue;
    msda::ProjArgs a{};
    a.dtype = dtype; a.rows = (long long)rows; a.C = d_model; a.eps = eps;
    a.x = x; a.w = weight; a.b = bias; a.residual = residual; a.gamma = gamma; a.beta = beta; a.pos = pos;
    a.y = y; a.y_pos = y_pos;
    return (int)msda::proj_layernorm_forward(a, (cudaStream_t)stream);
}

extern "C" int msda_layer_sine_position_tokens(int dtype, const float* y_embed, const float* x_embed, const float* dim_t,
                                               int num_pos_feats, const void* channel_add, int batch,
                                               int64_t height_x_width, void* tokens, int64_t tokens_per_item,
                                               int64_t level_start, void* stream)
{
    if (batch < 0 || num_pos_feats < 0 || height_x_width < 0 || level_start < 0 ||
        level_start + height_x_width > tokens_per_item)
        return (int)cudaErrorInvalidValue;
    return (int)msda::sine_position_tokens(dtype, y_embed, x_embed, dim_t, channel_add, tokens, batch,
                                           (long long)height_x_width, num_pos_feats, (long long)tokens_per_item,
                                           (long long)level_start, (cudaStream_t)stream);
}

extern "C" int msda_layer_sine_coordinates(const uint8_t* padding_mask, int batch, int height, int width, int normalize,
                                           float scale, float* y_embed, float* x_embed, void* stream)
{
    if (batch < 0 || height < 0 || width < 0) return (int)cudaErrorInvalidValue;
    return (int)msda::sine_coordinates(padding_mask, y_embed, x_embed, batch, height, width, normalize, scale,
                                       (cudaStream_t)stream);
}

extern "C" int msda_layer_tf32_split(const float* x, int64_t rows, int cols, float* out, void* stream)
{
    if (rows < 0 || cols < 0) return (int)cudaErrorInvalidValue;
    return (int)msda::tf32_split(x, out, (long long)rows, cols, (cudaStream_t)stream);
}

extern "C" int msda_layer_linear_bf16_supported(int out_features, int in_features)
{
    return msda::linear_bf16_supported(out_features, in_features) ? 1 : 0;
}

extern "C" int msda_layer_linear_bf16(const void* x, const void* weight, const void* bias, const uint8_t* zero_rows,
                                      int64_t rows, int out_features, int in_features, int relu, void* y, void* stream)
{
    if (rows < 0) return (int)cudaErrorInvalidValue;
    return (int)msda::linear_bf16(x, weight, bias, zero_rows, (long long)rows, out_features, in_features, relu, y,
                                  (cudaStream_t)stream);
}

extern "C" int msda_layer_linear_bf16_relu_dropout(const void* x, const void* weight, const void* bias, int64_t rows,
                                                   int out_features, int in_features, float p, const uint64_t* key, void* y,
                                                   void* stream)
{
    msda::DropoutRule r;
    if (rows < 0 || !msda::dropout_rule(p, &r) || key == nullptr) return (int)cudaErrorInvalidValue;
    return (int)msda::linear_bf16_relu_dropout(x, weight, bias, (long long)rows, out_features, in_features,
                                               reinterpret_cast<const unsigned long long*>(key), r, y, (cudaStream_t)stream);
}

extern "C" int msda_layer_linear_bf16_wgrad_supported(int out_features, int in_features)
{
    return msda::linear_bf16_wgrad_supported(out_features, in_features) ? 1 : 0;
}

extern "C" int64_t msda_layer_linear_bf16_wgrad_scratch_floats(int64_t rows, int out_features, int in_features)
{
    return (int64_t)msda::linear_bf16_wgrad_scratch_floats((long long)rows, out_features, in_features);
}

extern "C" int msda_layer_linear_bf16_wgrad(const void* grad_y, const void* x, int64_t rows, int out_features,
                                            int in_features, void* grad_weight, void* grad_bias, float* scratch,
                                            int64_t scratch_floats, void* stream)
{
    return (int)msda::linear_bf16_wgrad(grad_y, x, (long long)rows, out_features, in_features, grad_weight, grad_bias,
                                        scratch, (long long)scratch_floats, (cudaStream_t)stream);
}

extern "C" int msda_layer_linear_tf32x3_supported(int out_features, int in_features)
{
    return msda::linear_tf32x3_supported(out_features, in_features) ? 1 : 0;
}

extern "C" int msda_layer_linear_tf32x3(const float* x, const float* weight_hi, const float* weight_lo, const float* bias,
                                        int64_t rows, int out_features, int in_features, int relu, float* y, void* stream)
{
    if (rows < 0) return (int)cudaErrorInvalidValue;
    return (int)msda::linear_tf32x3(x, weight_hi, weight_lo, bias, (long long)rows, out_features, in_features, relu, y,
                                    (cudaStream_t)stream);
}

extern "C" int msda_layer_linear_tf32x3_relu_dropout(const float* x, const float* weight_hi, const float* weight_lo,
                                                     const float* bias, int64_t rows, int out_features, int in_features,
                                                     float p, const uint64_t* key, float* y, void* stream)
{
    msda::DropoutRule r;
    if (rows < 0 || !msda::dropout_rule(p, &r) || key == nullptr) return (int)cudaErrorInvalidValue;
    return (int)msda::linear_tf32x3_relu_dropout(x, weight_hi, weight_lo, bias, (long long)rows, out_features, in_features,
                                                 reinterpret_cast<const unsigned long long*>(key), r, y,
                                                 (cudaStream_t)stream);
}

extern "C" int msda_layer_linear_tf32x3_wgrad_supported(int out_features, int in_features)
{
    return msda::linear_tf32x3_wgrad_supported(out_features, in_features) ? 1 : 0;
}

extern "C" int64_t msda_layer_linear_tf32x3_wgrad_scratch_floats(int64_t rows, int out_features, int in_features)
{
    return (int64_t)msda::linear_tf32x3_wgrad_scratch_floats((long long)rows, out_features, in_features);
}

extern "C" int msda_layer_linear_tf32x3_wgrad(const float* grad_y, const float* x, int64_t rows, int out_features,
                                              int in_features, float* grad_weight, float* grad_bias, float* scratch,
                                              int64_t scratch_floats, void* stream)
{
    return (int)msda::linear_tf32x3_wgrad(grad_y, x, (long long)rows, out_features, in_features, grad_weight, grad_bias,
                                          scratch, (long long)scratch_floats, (cudaStream_t)stream);
}

// ---- batched linear assignment (hungarian.cu) ------------------------------------------------------

extern "C" int64_t msda_linear_assignment_scratch_bytes(int num_problems, int num_queries, int max_targets)
{
    return (int64_t)msda::linear_assignment_scratch_bytes(num_problems, num_queries, max_targets);
}

extern "C" int msda_linear_assignment(const float* cost, int64_t problem_stride, int64_t query_stride,
                                      const int64_t* counts, int num_problems, int num_queries, int max_targets,
                                      int32_t* query_of_target, int32_t* target_of_query, int32_t* status,
                                      void* scratch, int64_t scratch_bytes, void* stream)
{
    return (int)msda::linear_assignment(cost, (long long)problem_stride, (long long)query_stride, counts,
                                        num_problems, num_queries, max_targets, query_of_target, target_of_query,
                                        status, scratch, (long long)scratch_bytes, (cudaStream_t)stream);
}
