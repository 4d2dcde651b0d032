/* msda_b200.h - C ABI of libmsda_b200.so: multi-scale deformable attention for NVIDIA B200
 * (sm_100a).
 *
 * This is the drop-in boundary for the reference's native extension
 * `MultiScaleDeformableAttention` (pybind module, /root/reference/models/ops/src/vision.cpp:13-16).
 * Each entry point replaces one reference host launcher; argument order and meaning follow it:
 *
 *   msda_forward    <- ms_deformable_im2col_cuda   (models/ops/src/cuda/ms_deform_im2col_cuda.cuh:923-954)
 *                      as called by ms_deform_attn_cuda_forward (cuda/ms_deform_attn_cuda.cu:61-75)
 *   msda_backward   <- ms_deformable_col2im_cuda   (cuda/ms_deform_im2col_cuda.cuh:956-1327)
 *                      as called by ms_deform_attn_cuda_backward (cuda/ms_deform_attn_cuda.cu:131-148)
 *
 * Conventions (all pointers are DEVICE pointers, contiguous, on the current device):
 *   value        [N, S, M, D]         `dtype`
 *   spatial_shapes [L, 2]  int64 (H, W);  level_start_index [L] int64   (read on the device,
 *                                      exactly as the reference does, cuda/ms_deform_attn_cuda.cu:67-68)
 *   sampling_loc [N, Lq, M, L, P, 2]  (x, y) normalised to [0,1];  fp32, or fp64 when dtype is F64
 *   attn_weight  [N, Lq, M, L, P]     same type as sampling_loc
 *   output / grad_output [N, Lq, M, D] `dtype`
 * For the 16-bit dtypes (new behaviour - the reference op is fp32/fp64 only,
 * cuda/ms_deform_attn_cuda.cu:64) value/output/grad_output/grad_value are 16-bit while
 * locations, attention weights and their gradients stay fp32, and all arithmetic is fp32.
 *
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 * asynchronous, re-entrant, keep no global state and never synchronise.
 * Unlike the reference (which only printf's launch failures, cuh:948-952,1321-1325) every entry
 * point returns the cudaError_t of its launches as an int: 0 on success.
 * There is NO CPU implementation behind these symbols.
 */
#ifndef MSDA_B200_H
#define MSDA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    MSDA_DTYPE_F32 = 0,
    MSDA_DTYPE_F64 = 1,
    MSDA_DTYPE_BF16 = 2,
    MSDA_DTYPE_F16 = 3
} msda_dtype;

/* flags */
#define MSDA_FLAG_FORCE_GENERIC 1   /* route through the shape-generic kernels (testing) */
#define MSDA_FLAG_TC 4              /* msda_forward / msda_backward: run the tensor-core (tcgen05 + TMA) formulation where
                                       it applies (bf16 values, 32 channels per head, <= 4 levels, <= 4 points, at least
                                       2048 queries): csrc/msda_tc_forward.cu computes the output as C . V_window per
                                       128-query tile, csrc/msda_tc_backward.cu accumulates grad_value as C^T . G with one
                                       bulk tensor reduction per window row (grad_sampling_loc / grad_attn_weight stay
                                       with the default kernel).  Exact for any input and parity-tested, but measured
                                       SLOWER than the default lane-group kernels on B200 (DESIGN.md section 3.10):
                                       opt-in, for experiments */

#define MSDA_FLAG_VALUE_HEAD_MAJOR 8 /* msda_forward: `value` is laid out [N, M, S, D] (all pixels of a head contiguous)
                                       instead of the reference's [N, S, M, D].  BF16, D = 32 only (else an error).
                                       The x-neighbours of a bilinear footprint are then adjacent in memory: 3 instead
                                       of 4 L1 lines per sample (csrc/msda_forward_hm.cu) */

/* ABI version of this header (bumped on any signature change). */
int msda_abi_version(void);

/* Human-readable text for a return code of the functions below. */
const char* msda_error_string(int code);

/* out[n,q,m,:] = sum_{l,p} attn[n,q,m,l,p] * bilinear(value_l[n,:,m,:], loc[n,q,m,l,p]).
 * Writes every element of `output` (no zero-fill needed). */
int msda_forward(int dtype,
                 const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                 const void* sampling_loc, const void* attn_weight,
                 int batch, int spatial_size, int num_heads, int channels,
                 int num_levels, int num_query, int num_point,
                 void* output, int flags, void* stream);

/* Gradients of msda_forward.  grad_value is zero-filled by the call and then accumulated
 * into; grad_sampling_loc and grad_attn_weight are fully overwritten (zeros for samples that
 * fall outside the map), so none of the three needs initialising by the caller.
 * grad_value_accum_f32: for 16-bit dtypes an fp32 scratch buffer of batch*spatial_size*
 * num_heads*channels elements the vector atomics accumulate into before the cast to
 * grad_value; ignored (may be NULL) for F32 / F64. */
int msda_backward(int dtype,
                  const void* grad_output,
                  const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                  const void* sampling_loc, const void* attn_weight,
                  int batch, int spatial_size, int num_heads, int channels,
                  int num_levels, int num_query, int num_point,
                  void* grad_value, void* grad_sampling_loc, void* grad_attn_weight,
                  void* grad_value_accum_f32, int flags, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Deterministic backward: the same gradients as msda_backward / msda_fused_backward / msda_roi_align_backward, but
 * two calls on the same inputs give the same bits in any launch order (what a framework's deterministic mode asks
 * of an op).  Every contribution to a grad_value / grad_feature element is rounded to a multiple of 2^-shift and the
 * integers are summed with 64-bit integer reductions, which are associative.  A pre-pass on the device computes a
 * bound B >= |every element| from the inputs and picks shift = 61 - ceil(log2 B), so no partial sum can overflow; the
 * quantum is about B * 2^-61 (finer than fp32 atomics for fp32 and 16-bit gradients, coarser than fp64 atomics for
 * fp64 ones).  B == 0 gives zeros.  When B is not finite (Inf or NaN in grad_output, in the attention weights or in
 * the attention logits) EVERY element of grad_value / grad_feature is NaN, where the non-deterministic calls only
 * poison the elements the bad values reach.  The fused op's grad_reference_points is summed over the heads in a
 * fixed order from per-(query, level, head) partials instead of atomics.
 *   scratch: device memory of at least msda_deterministic_scratch_bytes(grad_elements, grad_reference_elements,
 *            num_heads) bytes, 16-byte aligned, contents ignored and overwritten.  grad_elements = elements of
 *            grad_value (batch*spatial_size*num_heads*channels) or of grad_feature (batch*height*width*channels);
 *            grad_reference_elements = elements of grad_reference_points (batch*num_query*num_levels*ref_dim) when
 *            the fused call is given one, else 0.  Returns -1 for negative arguments.
 * Each call fully writes every gradient it is given (nothing needs zeroing), allocates nothing, never reads back to
 * the host and is stream-ordered on `stream` without synchronising, so it can be captured in a CUDA graph.
 * cudaErrorInvalidValue for a too small or NULL scratch, and from msda_backward_deterministic for MSDA_FLAG_TC (the
 * tensor-core formulation has no deterministic variant).  grad_value_accum_f32 is ignored (may be NULL). */
int64_t msda_deterministic_scratch_bytes(int64_t grad_elements, int64_t grad_reference_elements, int num_heads);
int msda_backward_deterministic(int dtype,
                                const void* grad_output,
                                const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                const void* sampling_loc, const void* attn_weight,
                                int batch, int spatial_size, int num_heads, int channels,
                                int num_levels, int num_query, int num_point,
                                void* grad_value, void* grad_sampling_loc, void* grad_attn_weight,
                                void* grad_value_accum_f32, int flags, void* scratch, int64_t scratch_bytes,
                                void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused layer op (no counterpart symbol in the reference: it replaces the chain
 * softmax -> offset/normaliser arithmetic -> MSDeformAttnFunction of MSDeformAttn.forward,
 * /root/reference/models/ops/modules/ms_deform_attn.py:98-115, with ONE kernel per direction;
 * sampling locations and attention weights never exist in HBM).
 *
 *   reference_points      [N*Lq, L, ref_dim] fp32, ref_dim 2 (points) or 4 (boxes cx,cy,w,h)
 *   sampling_offsets_raw  output of the sampling_offsets projection, element (nq, m, l, p, xy) at
 *                         base[nq*offsets_query_stride + ((m*L + l)*P + p)*2 + xy]
 *   attention_logits_raw  output of the attention_weights projection (pre-softmax), element
 *                         (nq, m, l, p) at base[nq*logits_query_stride + (m*L + l)*P + p]
 *   raw_dtype             F32, or BF16 when dtype is BF16
 * The two raw tensors may be slices of one [N*Lq, 3*M*L*P] GEMM output (both strides 3*M*L*P).
 * Supported: dtype F32 / BF16, channels 16 / 32 / 64, num_levels*num_point <= 16
 * (msda_fused_supported); everything else goes through msda_forward / msda_backward.
 * Backward: grad_offsets_raw / grad_logits_raw use the addressing of their inputs and are fully
 * written; grad_reference_points (may be NULL) is accumulated into with atomics - zero it first.
 */
int msda_fused_supported(int dtype, int raw_dtype, int ref_dim, int spatial_size, int num_heads,
                         int channels, int num_levels, int num_point);

int msda_fused_forward(int dtype, int raw_dtype,
                       const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                       const float* reference_points, int ref_dim,
                       const void* sampling_offsets_raw, int64_t offsets_query_stride,
                       const void* attention_logits_raw, int64_t logits_query_stride,
                       int batch, int spatial_size, int num_heads, int channels,
                       int num_levels, int num_query, int num_point,
                       void* output, void* stream);

/* Head-major variants for inference (round 2).  value_hm is laid out [N, M, S, D]: all pixels of a head contiguous, so
 * the x-neighbours of a bilinear footprint are adjacent in memory (3 instead of 4 L1 lines per sample).  BF16, D = 32.
 * msda_layer_value_proj_head_major computes  value = x @ W^T + b  (reference modules/ms_deform_attn.py:94), zeroes the
 * rows of padding_mask (:95-96; one byte per row, may be NULL) and writes that layout directly from the GEMM epilogue
 * (tcgen05, d_model 256, 8 heads); msda_fused_forward_head_major is msda_fused_forward reading it. */
int msda_fused_forward_head_major(int dtype, int raw_dtype,
                                  const void* value_hm, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                  const float* reference_points, int ref_dim,
                                  const void* sampling_offsets_raw, int64_t offsets_query_stride,
                                  const void* attention_logits_raw, int64_t logits_query_stride,
                                  int batch, int spatial_size, int num_heads, int channels, int num_levels,
                                  int num_query, int num_point, void* output, void* stream);
int msda_layer_value_proj_head_major_supported(int dtype, int d_model, int num_heads);
int msda_layer_value_proj_head_major(int dtype, const void* x, const void* weight, const void* bias,
                                     const unsigned char* padding_mask, int64_t rows, int tokens_per_frame,
                                     int d_model, int num_heads, void* value_hm, void* stream);

/* msda_fused_forward reading `value` with a pixel stride: pixel r of item n starts at
 * value[(n * spatial_size + r) * value_pixel_stride] (elements; >= num_heads * channels, a multiple of the 16-byte
 * vector; 0 = dense).  Lets one GEMM compute the value projections of several layers that attend to the same
 * memory (the six decoder layers each re-project the encoder memory, /root/reference/models/
 * deformable_transformer_single.py:617-628 via ms_deform_attn.py:94) and hand each layer its column slice. */
int msda_fused_forward_strided(int dtype, int raw_dtype,
                               const void* value, int64_t value_pixel_stride,
                               const int64_t* spatial_shapes, const int64_t* level_start_index,
                               const float* reference_points, int ref_dim,
                               const void* sampling_offsets_raw, int64_t offsets_query_stride,
                               const void* attention_logits_raw, int64_t logits_query_stride,
                               int batch, int spatial_size, int num_heads, int channels,
                               int num_levels, int num_query, int num_point,
                               void* output, void* stream);

int msda_fused_backward(int dtype, int raw_dtype,
                        const void* grad_output,
                        const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                        const float* reference_points, int ref_dim,
                        const void* sampling_offsets_raw, int64_t offsets_query_stride,
                        const void* attention_logits_raw, int64_t logits_query_stride,
                        int batch, int spatial_size, int num_heads, int channels,
                        int num_levels, int num_query, int num_point,
                        void* grad_value, void* grad_offsets_raw, void* grad_logits_raw,
                        float* grad_reference_points, void* grad_value_accum_f32, void* stream);
/* msda_fused_backward with the guarantee of msda_backward_deterministic (see there); grad_reference_points (may be
 * NULL) is fully written, not accumulated into. */
int msda_fused_backward_deterministic(int dtype, int raw_dtype,
                                      const void* grad_output,
                                      const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                      const float* reference_points, int ref_dim,
                                      const void* sampling_offsets_raw, int64_t offsets_query_stride,
                                      const void* attention_logits_raw, int64_t logits_query_stride,
                                      int batch, int spatial_size, int num_heads, int channels,
                                      int num_levels, int num_query, int num_point,
                                      void* grad_value, void* grad_offsets_raw, void* grad_logits_raw,
                                      float* grad_reference_points, void* grad_value_accum_f32,
                                      void* scratch, int64_t scratch_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Layer epilogues around the deformable attention (no counterpart symbol in the reference, which
 * runs them as separate PyTorch element-wise kernels).  They replace, in every layer class that owns
 * an MSDeformAttn,
 *     x = norm(residual + dropout(branch))                 /root/reference/models/deformable_transformer_single.py:538-541
 *     x = norm(x + dropout(act(linear1(x))))   (fusion)    :393-400, :452-459  (and :544-548, :617-642)
 *     query = x + pos                                      :530-531, :538
 * with ONE kernel per direction:
 *     v = residual + act(branch);  y = LayerNorm_C(v) * gamma + beta;  y_pos = y + pos (optional)
 * `act`: 0 identity, 1 ReLU, 2 GELU (exact erf form).
 * All tensors are [rows, channels] (gamma / beta [channels]) of `dtype` (F32, BF16 or F16), 16-byte
 * aligned; arithmetic is fp32.  residual / pos / y_pos / mean / rstd may be NULL (pos and y_pos
 * together, mean and rstd together).  mean / rstd [rows] fp32 are the row statistics the backward
 * needs.  Supported channel counts: msda_layer_add_layernorm_supported (a multiple of 128 (F32) or
 * 256 (16-bit) elements with 1, 2 or 4 sixteen-byte chunks per lane, i.e. 128/256/512 or
 * 256/512/1024).
 * Backward: grad_y_pos may be NULL.  grad_residual must be given iff residual was.  With act == 0 and
 * a residual, d branch == d residual and only grad_residual is written (grad_branch is ignored).
 * partial_scratch: fp32 [partial_blocks, 2, channels]; partial_blocks =
 * msda_layer_add_layernorm_partial_blocks(rows).  grad_gamma / grad_beta [channels] are overwritten.
 */
int msda_layer_add_layernorm_supported(int dtype, int channels);
int msda_layer_add_layernorm_partial_blocks(int64_t rows);
int msda_layer_add_layernorm_forward(int dtype, int act,
                                     const void* branch, const void* residual,
                                     const void* gamma, const void* beta, const void* pos,
                                     int64_t rows, int channels, float eps,
                                     void* y, void* y_pos, float* mean, float* rstd, void* stream);
int msda_layer_add_layernorm_backward(int dtype, int act,
                                      const void* grad_y, const void* grad_y_pos,
                                      const void* branch, const void* residual, const void* gamma,
                                      const float* mean, const float* rstd,
                                      int64_t rows, int channels,
                                      void* grad_branch, void* grad_residual,
                                      void* grad_gamma, void* grad_beta,
                                      float* partial_scratch, int partial_blocks, void* stream);

/* Fused feed-forward block of the encoder / decoder layers on the tcgen05 tensor cores (inference):
 *     y = LayerNorm(x + linear2(relu(linear1(x)))) * gamma + beta;   y_pos = y + pos (optional)
 * = forward_ffn + norm2 (+ the next layer's query) of DeformableTransformerEncoderLayer,
 * /root/reference/models/deformable_transformer_single.py:544-548 (:530-531).  The [rows, d_ffn] hidden
 * activation stays in tensor / shared memory.  All tensors BF16, 16-byte aligned; w1 [d_ffn, d_model] and
 * w2 [d_model, d_ffn] in nn.Linear layout.  Supported: BF16, d_model 256, d_ffn a multiple of 64
 * (msda_layer_ffn_layernorm_supported); pos / y_pos may be NULL together. */
int msda_layer_ffn_layernorm_supported(int dtype, int d_model, int d_ffn);
int msda_layer_ffn_layernorm_forward(int dtype,
                                     const void* x, const void* w1, const void* b1,
                                     const void* w2, const void* b2,
                                     const void* gamma, const void* beta, const void* pos,
                                     int64_t rows, int d_model, int d_ffn, float eps,
                                     void* y, void* y_pos, void* stream);

/* y = LayerNorm(residual + (x @ weight^T + bias)) * gamma + beta and, when pos / y_pos are given, y_pos = y + pos:
 * `output_proj` of MSDeformAttn (/root/reference/models/ops/modules/ms_deform_attn.py:116) together with the
 * `norm1(src + dropout1(src2))` of the layer that owns it (models/deformable_transformer_single.py:538-541; the
 * fusion layers' adapt Linear + norm :385-394), as ONE tcgen05 kernel with the weight stationary in tensor memory.
 * All tensors BF16, 16-byte aligned, x / residual / pos / y / y_pos [rows, d_model], weight [d_model, d_model] in
 * nn.Linear layout.  Supported: BF16, d_model 256 (msda_layer_proj_layernorm_supported); residual may be NULL,
 * pos / y_pos NULL together.  Forward only. */
int msda_layer_proj_layernorm_supported(int dtype, int d_in, int d_out);
int msda_layer_proj_layernorm_forward(int dtype, const void* x, const void* weight, const void* bias,
                                      const void* residual, const void* gamma, const void* beta, const void* pos,
                                      int64_t rows, int d_model, float eps, void* y, void* y_pos, void* stream);

/* One pyramid level from NCHW to token-major, written into its slice of the flattened token tensor:
 *     tokens[n, level_start + y*W + x, c] = feature_map[n, c, y, x] (+ channel_add[c])
 * = src.flatten(2).transpose(1, 2) (+ level_embed[l]) and its share of the concatenation in
 * DeformableTransformer.forward, /root/reference/models/deformable_transformer_single.py:190-206.
 * feature_map [batch, channels, H*W] contiguous, tokens [batch, tokens_per_item, channels], channel_add
 * [channels] or NULL; dtype F32 / BF16 / F16. */
int msda_layer_flatten_level(int dtype, const void* feature_map, const void* channel_add, int batch,
                             int channels, int height_x_width, void* tokens, int64_t tokens_per_item,
                             int64_t level_start, void* stream);

/* out[c] = sum over rows of x[row, c]: the bias gradient of the Linear layers around the deformable
 * attention (PyTorch's autograd computes it with a generic reduction; this is the HBM-rate version).
 * x [rows, channels] and out [channels] of `dtype` (F32 / BF16 / F16), fp32 accumulation.
 * partial_scratch: fp32 [partial_blocks, channels], partial_blocks = msda_layer_colsum_blocks(...)
 * (0 = shape not supported: channels*itemsize must be a multiple of 16 and at most 4096 bytes). */
int msda_layer_colsum_blocks(int dtype, int64_t rows, int channels);
int msda_layer_colsum(int dtype, const void* x, int64_t rows, int channels, void* out,
                      float* partial_scratch, int partial_blocks, void* stream);

/* value.masked_fill(padding_mask[..., None], 0) of MSDeformAttn.forward
 * (/root/reference/models/ops/modules/ms_deform_attn.py:95-96), in place: rows of data[rows, channels]
 * whose mask byte is non-zero are overwritten with zeros; only the mask and those rows are touched. */
int msda_layer_zero_masked_rows(int dtype, void* data, const uint8_t* mask, int64_t rows, int channels,
                                void* stream);

/* Left operand of an error-compensated TF32 product: x [rows, cols] FP32 -> out [rows, 3 * cols] = [ lo | hi | hi ] per
 * row, hi = x rounded to TF32 (10 mantissa bits, nearest), lo = x - hi (exact).  With W [n, cols] arranged as
 * [ hi_W | lo_W | hi_W ], out W'^T = lo_x hi_W^T + hi_x lo_W^T + hi_x hi_W^T in ONE TF32 tensor-core GEMM is FP32-grade: it
 * stands in for the IEEE SGEMMs of the reference's FP32 nn.Linear layers
 * (/root/reference/models/ops/modules/ms_deform_attn.py:94-116, deformable_transformer_single.py:544-548) when the caller
 * selects it.  cols % 4 == 0; x and out 16-byte aligned. */
int msda_layer_tf32_split(const float* x, int64_t rows, int cols, float* out, void* stream);

/* The same FP32-grade product as ONE kernel: y [rows, out_features] = x [rows, in_features] weight^T + bias (then ReLU when
 * relu != 0), FP32 in and out -- an nn.Linear of the reference's FP32 model
 * (/root/reference/models/ops/modules/ms_deform_attn.py:94-116, deformable_transformer_single.py:544-548) on the tcgen05
 * tensor cores.  weight_hi [out, in] = weight rounded to TF32 (10 mantissa bits, nearest), weight_lo = weight - weight_hi
 * (the caller splits the static weight once); the activation tile is split in shared memory inside the kernel, so no
 * [lo | hi | hi] copy of x ever reaches HBM.  bias may be NULL.  out_features % 32 == 0, in_features % 32 == 0, 16-byte
 * aligned buffers (..._supported answers for a shape). */
int msda_layer_linear_tf32x3_supported(int out_features, int in_features);

/* BF16 nn.Linear of an inference pass as one TMA / tcgen05 kernel: y [rows, out_features] = x [rows, in_features] weight^T
 * + bias, then ReLU when relu != 0, then rows whose zero_rows byte is non-zero overwritten with zeros -- value_proj with
 * its masked_fill(padding_mask, 0) (/root/reference/models/ops/modules/ms_deform_attn.py:94-96), the
 * [sampling_offsets | attention_weights] projection (:98-100), linear1 + ReLU
 * (deformable_transformer_single.py:544-548).  bias and zero_rows may be NULL.  out_features % 64 == 0,
 * in_features % 64 == 0, 16-byte aligned buffers (..._supported answers for a shape). */
int msda_layer_linear_bf16_supported(int out_features, int in_features);
int msda_layer_linear_bf16(const void* x, const void* weight, const void* bias, const uint8_t* zero_rows,
                           int64_t rows, int out_features, int in_features, int relu, void* y, void* stream);
int msda_layer_linear_tf32x3(const float* x, const float* weight_hi, const float* weight_lo, const float* bias,
                             int64_t rows, int out_features, int in_features, int relu, float* y, void* stream);

/* Weight and bias gradient of that FP32 nn.Linear (training), at the same fp32 grade: grad_weight [out_features,
 * in_features] = grad_y^T x and grad_bias [out_features] = grad_y summed over the rows, from grad_y [rows, out_features]
 * and x [rows, in_features], all FP32 row-major.  Both operands are split into TF32 hi / lo parts in shared memory and
 * the product is g_hi^T x_hi + g_lo^T x_hi + g_hi^T x_lo on the tcgen05 tensor cores; the main accumulator is drained
 * into fp32 registers every 256 rows, so the tensor core's truncating accumulation does not build up over long
 * reductions.  One pass over grad_y gives both outputs.  The rows are split into slices whose fp32 partial sums go to
 * `scratch` (scratch_floats >= msda_layer_linear_tf32x3_wgrad_scratch_floats(rows, ...), 0 = shape not supported), then
 * a second kernel adds them in a fixed order: two calls on the same inputs give the same bits.  grad_bias may be NULL.
 * out_features % 32 == 0, in_features % 32 == 0 (both >= 32), rows >= 1, 16-byte aligned buffers;
 * cudaErrorInvalidValue otherwise.  Stream-ordered on `stream`, no allocation, no synchronisation (can be captured in a
 * CUDA graph).  The input gradient grad_x = grad_y weight is msda_layer_linear_tf32x3 with the split of weight^T
 * [in_features, out_features] as its weight pair. */
int msda_layer_linear_tf32x3_wgrad_supported(int out_features, int in_features);
int64_t msda_layer_linear_tf32x3_wgrad_scratch_floats(int64_t rows, int out_features, int in_features);
int msda_layer_linear_tf32x3_wgrad(const float* grad_y, const float* x, int64_t rows, int out_features, int in_features,
                                   float* grad_weight, float* grad_bias, float* scratch, int64_t scratch_floats,
                                   void* stream);

/* Weight and bias gradient of that BF16 nn.Linear (training): grad_weight [out_features, in_features] = grad_y^T x and
 * grad_bias [out_features] = grad_y summed over the rows, from grad_y [rows, out_features] and x [rows, in_features], all
 * BF16 row-major, fp32 accumulation on the tcgen05 tensor cores.  One pass over grad_y gives both: the bias gradient is
 * not a second read of grad_y.  The rows are split into slices whose fp32 partial sums go to `scratch`
 * (scratch_floats >= msda_layer_linear_bf16_wgrad_scratch_floats(rows, ...), 0 = shape not supported), then a second
 * kernel adds them in a fixed order: two calls on the same inputs give the same bits.  grad_bias may be NULL.
 * out_features % 64 == 0, in_features % 64 == 0, rows >= 1, 16-byte aligned buffers; cudaErrorInvalidValue otherwise.
 * Stream-ordered on `stream`, no allocation, no synchronisation (can be captured in a CUDA graph).  The input gradient
 * grad_x = grad_y weight is msda_layer_linear_bf16 with weight^T [in_features, out_features] as its weight. */
int msda_layer_linear_bf16_wgrad_supported(int out_features, int in_features);
int64_t msda_layer_linear_bf16_wgrad_scratch_floats(int64_t rows, int out_features, int in_features);
int msda_layer_linear_bf16_wgrad(const void* grad_y, const void* x, int64_t rows, int out_features, int in_features,
                                 void* grad_weight, void* grad_bias, float* scratch, int64_t scratch_floats, void* stream);

/* Cumulative coordinates of the sine position embedding (PositionEmbeddingSine.forward,
 * /root/reference/models/position_encoding.py:39-46): padding_mask [batch, height, width] bytes (non-zero = padding),
 * y_embed / x_embed [batch, height, width] FP32 = cumsum of the valid pixels down the rows / along the columns and,
 * when normalize != 0, (c - 0.5) / (last + 1e-6) * scale with the reference's operation order (bit-identical to the
 * reference's tensor ops). */
int msda_layer_sine_coordinates(const uint8_t* padding_mask, int batch, int height, int width, int normalize,
                                float scale, float* y_embed, float* x_embed, void* stream);

/* Sine position embedding of one pyramid level, written into its slice of the flattened token tensor:
 *     tokens[n, level_start + p, c] = T( T( f(coord[n, p] / dim_t[c mod F]) ) + channel_add[c] ),  F = num_pos_feats,
 *     coord = y_embed for c < F, x_embed for c >= F;  f = sin for even c mod F, cos for odd
 * = PositionEmbeddingSine.forward (/root/reference/models/position_encoding.py:35-56), the joiner's cast to the
 * feature dtype, and flatten(2).transpose(1, 2) + level_embed[l] of DeformableTransformer.forward
 * (deformable_transformer_single.py:196-199) in one pass.  y_embed / x_embed [batch, H*W] FP32 are the (normalised)
 * cumulative coordinates the reference computes from the padding mask (:41-46), dim_t [F] FP32 its
 * temperature ** (2 * (k / 2) / F) (:48-49); tokens [batch, tokens_per_item, 2 * F] of `dtype` (F32 / BF16 / F16),
 * channel_add [2 * F] of `dtype` or NULL. */
int msda_layer_sine_position_tokens(int dtype, const float* y_embed, const float* x_embed, const float* dim_t,
                                    int num_pos_feats, const void* channel_add, int batch, int64_t height_x_width,
                                    void* tokens, int64_t tokens_per_item, int64_t level_start, void* stream);

/* GroupNorm on token-major activations x [batch, tokens_per_item, channels] (groups of channels / groups consecutive
 * channels, statistics per (item, group)): the nn.GroupNorm(32, hidden_dim) of the reference's input projections,
 * /root/reference/models/deformable_detr_single.py:101-150, applied to the projection computed token-major so that
 * the flatten / transpose / concatenation of deformable_transformer_single.py:190-206 disappear.  y may be x.
 * channel_bias [channels] or NULL: added to x first (the convolution's bias, so the projection GEMM needs no
 * epilogue); item_stride: elements between consecutive items of x and y (0 = dense; a level's slice of the
 * flattened multi-level token tensor has tokens_of_all_levels * channels).
 * partial_scratch: fp32 [batch, slabs, groups, 2], slabs = msda_layer_group_norm_tokens_slabs(...) (0 = shape not
 * supported: groups <= 64, channels / groups a multiple of the 16-byte vector).  dtype F32 / BF16 / F16.  Forward. */
int msda_layer_group_norm_tokens_slabs(int dtype, int64_t tokens_per_item, int channels, int groups);
int msda_layer_group_norm_tokens(int dtype, const void* x, const void* channel_bias, const void* gamma,
                                 const void* beta, int batch, int64_t tokens_per_item, int channels, int groups,
                                 float eps, int64_t item_stride, float* partial_scratch, int slabs, void* y,
                                 void* stream);

/* y = act(LayerNorm(x) * gamma + beta), act 0 identity / 1 relu / 2 gelu(erf): the normalise-then-activate steps
 * of the TransVOD++ dynamic interaction head, features = relu(norm(bmm(...))),
 * /root/reference/models/sparse_roi_head/head.py:156-170.  x, y [rows, channels] (y may be x), gamma / beta
 * [channels], all `dtype` (F32 / BF16 / F16), 16-byte aligned; channels * itemsize in {128, 256, 512, 1024, 2048}
 * (msda_layer_norm_act_supported).  Forward only. */
int msda_layer_norm_act_supported(int dtype, int channels);
int msda_layer_norm_act_forward(int dtype, const void* x, const void* gamma, const void* beta, int64_t rows,
                                int channels, float eps, int act, void* y, void* stream);

/* RoIAlign of the TransVOD++ temporal query stage: mmcv.ops.RoIAlign(output_size, spatial_scale, sampling_ratio,
 * pool_mode='avg', aligned) as constructed at /root/reference/models/deformable_transformer_multi_plusplus.py:129-132
 * and called at :499 and :514 (mmcv-full 1.7.0, not vendored by the reference; algorithm of its
 * roi_align_cuda_kernel.cuh).  Replaces the mmcv binding roi_align_forward / roi_align_backward for pool_mode 'avg'.
 * Layouts are token-major, i.e. what the encoder produces and what the query head consumes, so the reference's
 * permute to NCHW (:498) and back (sparse_roi_head/head.py:66) disappear:
 *   feature_tokens     [batch, height*width, channels]            dtype
 *   rois               [num_rois, 5] = (batch index, x1, y1, x2, y2) FP32 (FP64 when dtype is F64), image units
 *   pooled/grad_pooled [num_rois, pooled_height*pooled_width, channels] dtype
 *   grad_feature_accum [batch, height*width, channels] FP32 (FP64 when dtype is F64), zero-initialised by the
 *                      caller, accumulated with reductions (cast to dtype by the caller)
 * sampling_ratio 0 = adaptive ceil(roi_size / pooled_size) grid, as in mmcv. */
int msda_roi_align_forward(int dtype, const void* feature_tokens, const void* rois, int batch, int height,
                           int width, int channels, int num_rois, int pooled_height, int pooled_width,
                           double spatial_scale, int sampling_ratio, int aligned, void* pooled, void* stream);
int msda_roi_align_backward(int dtype, const void* grad_pooled, const void* rois, int batch, int height,
                            int width, int channels, int num_rois, int pooled_height, int pooled_width,
                            double spatial_scale, int sampling_ratio, int aligned, void* grad_feature_accum,
                            void* stream);
/* msda_roi_align_backward with the guarantee of msda_backward_deterministic (see there).  grad_feature
 * [batch, height*width, channels] is in `dtype` (not an FP32 accumulator) and fully written; the bound is
 * num_rois * pooled_height * pooled_width * max |grad_pooled| (a bin adds at most |grad_pooled| to any pixel). */
int msda_roi_align_backward_deterministic(int dtype, const void* grad_pooled, const void* rois, int batch, int height,
                                          int width, int channels, int num_rois, int pooled_height, int pooled_width,
                                          double spatial_scale, int sampling_ratio, int aligned, void* grad_feature,
                                          void* scratch, int64_t scratch_bytes, void* stream);

/* Dropout on the package's kernels (DESIGN.md section 3.16).  `key` points to ONE uint64 in device memory
 * (drawn per call by the caller on the device; it is never read on the host, so the calls
 * can be captured in a CUDA graph).  Element e of a call's contiguous [rows, channels] output draws
 *     u(e) = (r[(e & 7) >> 1] >> (16 * (e & 1))) & 0xFFFF,
 *     r = Philox4x32-10(counter (lo32(e >> 3), hi32(e >> 3), 0, 0), key (lo32(key), hi32(key)))
 * and is kept iff u(e) >= threshold = floor(p * 65536 + 0.5); kept values are multiplied by
 * scale = float(1 / (1 - p)).  msda_layer_dropout_rule reports threshold and scale.  Every call returns
 * cudaErrorInvalidValue for p outside (0, 1) or a NULL key.
 *
 * add-LayerNorm with dropout on the branch: v = residual + act(branch) * mask * scale, otherwise as
 * msda_layer_add_layernorm_forward / _backward.  The backward regenerates the mask from the same key and p; it
 * always writes grad_branch (never aliased with grad_residual).  Channel counts:
 * msda_layer_add_layernorm_dropout_supported (1 or 2 sixteen-byte chunks per lane: 128/256 F32, 256/512 16-bit).
 *
 * msda_layer_dropout: y = x * mask * scale over n contiguous elements of dtype; y == x is allowed.  Called on a
 * gradient with the same key and p it is the backward.
 * msda_layer_relu_dropout_grad: grad_x = y > 0 ? grad_y * scale : 0, the backward of dropout(relu(.)) from its
 * output y alone (no key).
 * msda_layer_linear_bf16_relu_dropout / msda_layer_linear_tf32x3_relu_dropout: msda_layer_linear_bf16 /
 * msda_layer_linear_tf32x3 with relu = 1 and dropout applied in the epilogue (element index row * out_features + col). */
int msda_layer_dropout_rule(float p, uint32_t* threshold, float* scale);
int msda_layer_add_layernorm_dropout_supported(int dtype, int channels);
int msda_layer_add_layernorm_dropout_forward(int dtype, int act,
                                             const void* branch, const void* residual,
                                             const void* gamma, const void* beta, const void* pos,
                                             int64_t rows, int channels, float eps,
                                             void* y, void* y_pos, float* mean, float* rstd,
                                             float p, const uint64_t* key, void* stream);
int msda_layer_add_layernorm_dropout_backward(int dtype, int act,
                                              const void* grad_y, const void* grad_y_pos,
                                              const void* branch, const void* residual, const void* gamma,
                                              const float* mean, const float* rstd,
                                              int64_t rows, int channels,
                                              void* grad_branch, void* grad_residual,
                                              void* grad_gamma, void* grad_beta,
                                              float* partial_scratch, int partial_blocks,
                                              float p, const uint64_t* key, void* stream);
int msda_layer_dropout(int dtype, const void* x, void* y, int64_t n, float p, const uint64_t* key, void* stream);
int msda_layer_relu_dropout_grad(int dtype, const void* grad_y, const void* y, void* grad_x, int64_t n, float p,
                                 void* stream);
int msda_layer_linear_bf16_relu_dropout(const void* x, const void* weight, const void* bias, int64_t rows,
                                        int out_features, int in_features, float p, const uint64_t* key, void* y,
                                        void* stream);
int msda_layer_linear_tf32x3_relu_dropout(const float* x, const float* weight_hi, const float* weight_lo,
                                          const float* bias, int64_t rows, int out_features, int in_features,
                                          float p, const uint64_t* key, float* y, void* stream);

/* Batched rectangular linear assignment (csrc/hungarian.cu, DESIGN.md section 3.17): the Hungarian matching of
 * Deformable DETR's set criterion, solved on the device for many (image, output head) problems in one launch.
 *   cost             fp32; problem p's cost of matching query q to target t is
 *                    cost[p * problem_stride + q * query_stride + t]  (t < max_targets, q < num_queries)
 *   counts           [num_problems] int64 target counts T_p, read on the device; 0 <= T_p <= min(max_targets,
 *                    num_queries) is required
 *   query_of_target  [num_problems, max_targets] int32: the query matched to target t, -1 for t >= T_p
 *   target_of_query  [num_problems, num_queries] int32: the target matched to query q, -1 if unmatched
 *   status           [num_problems] int32: 0 solved; 1 a cost of the first T_p targets is NaN or +-Inf;
 *                    2 T_p out of range; 3 no feasible matching.  A non-zero status writes -1 to all of the
 *                    problem's outputs.  The call never traps on bad data.
 * Every target is matched, at the least total cost: the shortest-augmenting-path algorithm of
 * scipy.optimize.linear_sum_assignment on the same fp64-widened costs with fp64 potentials, so costs without
 * ties give scipy's assignment.  Among equal-cost solutions the choice may differ from scipy's.
 * `scratch` of msda_linear_assignment_scratch_bytes bytes (0 for num_queries <= 1024, when the state lives in
 * shared memory); the scratch bytes call returns -1 for negative sizes. */
int64_t msda_linear_assignment_scratch_bytes(int num_problems, int num_queries, int max_targets);
int msda_linear_assignment(const float* cost, int64_t problem_stride, int64_t query_stride, const int64_t* counts,
                           int num_problems, int num_queries, int max_targets, int32_t* query_of_target,
                           int32_t* target_of_query, int32_t* status, void* scratch, int64_t scratch_bytes,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSDA_B200_H */
