// Internal (C++) launch interface between the C-ABI layer (msda_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace msda {

enum DType { kF32 = 0, kF64 = 1, kBF16 = 2, kF16 = 3 };   // == msda_dtype in include/msda_b200.h

struct FwdArgs {
    int dtype;
    const void* value;        // [N,S,M,D] dtype
    const int64_t* shapes;    // [L,2] device
    const int64_t* lsi;       // [L]   device
    const void* loc;          // [N,Lq,M,L,P,2]  fp32 (fp64 when dtype == kF64)
    const void* attn;         // [N,Lq,M,L,P]    same type as loc
    void* out;                // [N,Lq,M,D] dtype
    int N, S, M, D, L, Lq, P;
    int force_generic;        // tests: route through the generic kernel
    int no_tc;                // 0: take the tensor-core formulation (msda_tc_forward.cu) where it applies (opt-in)
    int head_major;           // value is [N, M, S, D] (msda_forward_hm.cu: bf16, D = 32) instead of [N, S, M, D]
};

struct BwdArgs {
    int dtype;
    const void* grad_out;     // [N,Lq,M,D] dtype
    const void* value;
    const int64_t* shapes;
    const int64_t* lsi;
    const void* loc;
    const void* attn;
    void* grad_value;         // [N,S,M,D] dtype, written (zero-initialised by the launcher)
    void* grad_loc;           // like loc, every element written
    void* grad_attn;          // like attn, every element written
    float* grad_value_accum;  // 16-bit dtypes only: fp32 [N,S,M,D] scratch the atomics land in
    int N, S, M, D, L, Lq, P;
    int force_generic;
    int no_tc;
};

// Fused layer op: sampling locations and attention weights are NOT materialised.  The kernels
// read the raw outputs of the sampling_offsets / attention_weights projections and the
// reference points, and do softmax + location arithmetic (modules/ms_deform_attn.py:98-110 of the
// reference) in registers.
struct FusedArgs {
    int dtype;                // value / out / grad_out / grad_value dtype (kF32, kBF16, kF16)
    int raw_dtype;            // offsets / logits dtype (kF32 or kBF16/kF16 matching dtype)
    const void* value;
    const int64_t* shapes;
    const int64_t* lsi;
    const float* ref;         // [N*Lq, L, ref_dim] fp32
    int ref_dim;              // 2 or 4
    const void* offsets;      // element (nq, m, l, p, xy) at offsets[nq*off_stride + ((m*L + l)*P + p)*2 + xy]
    long long off_stride;
    const void* logits;       // element (nq, m, l, p)     at logits[nq*logit_stride + (m*L + l)*P + p]
    long long logit_stride;
    void* out;                // forward: [N,Lq,M,D]
    // backward only
    const void* grad_out;
    void* grad_value;         // [N,S,M,D] dtype
    float* grad_value_accum;  // 16-bit dtypes: fp32 scratch
    void* grad_offsets;       // same addressing as offsets (raw dtype), fully written
    void* grad_logits;        // same addressing as logits, fully written
    float* grad_ref;          // [N*Lq, L, ref_dim] fp32, accumulated with atomics (caller zero-fills); may be null
    int N, S, M, D, L, Lq, P;
    long long value_ld;       // forward only: elements between consecutive pixels of value (0 = dense, M*D)
};

bool fused_supported(const FusedArgs& a);
bool fused_raw_layout_ok(const FusedArgs& a);   // strides / alignment of offsets, grad_offsets
cudaError_t fused_forward(const FusedArgs& a, cudaStream_t stream);
cudaError_t fused_backward(const FusedArgs& a, cudaStream_t stream);

cudaError_t forward(const FwdArgs& a, cudaStream_t stream);
// head-major value layout [N, M, S, 32] (bf16): msda_forward_hm.cu
bool forward_hm_supported(int dtype, int D, int L, int P);
cudaError_t forward_hm(const FwdArgs& a, cudaStream_t stream);
cudaError_t fused_forward_hm(const FusedArgs& a, cudaStream_t stream);
// value_proj on tcgen05 with a head-major epilogue (value_proj_hm.cu): x [rows, 256] bf16 -> out_hm [N, 8, S, 32]
bool value_proj_hm_supported(int dtype, int d_model, int n_heads);
cudaError_t value_proj_hm(int dtype, const void* x, const void* w, const void* b, const unsigned char* mask, void* out_hm,
                          long long rows, int S, cudaStream_t stream);

// Tensor-core formulation (msda_tc_forward.cu / msda_tc_backward.cu): bf16 values, 32 channels per head, <= 4 levels,
// <= 4 points.  forward() / backward() route to it when it applies.
bool tc_forward_supported(const FwdArgs& a);
cudaError_t tc_forward(const FwdArgs& a, cudaStream_t stream);
bool tc_backward_supported(const BwdArgs& a);
// grad_value of every (tile, level) whose window fits -> a.grad_value_accum (zeroed by the caller);
// red_levels[pair] = mask of the levels left to msda_bwd_fast_kernel's reductions
cudaError_t tc_backward_dv(const BwdArgs& a, unsigned char* red_levels, cudaStream_t stream);

cudaError_t backward(const BwdArgs& a, cudaStream_t stream);

// Deterministic backward (deterministic.cu, DESIGN.md section 3.15).  scratch: [256-byte DetHeader | int64
// accumulators, one per gradient element, padded to 256 bytes | fp32 partials of grad_reference_points (fused op)].
struct DetHeader;
long long det_scratch_bytes(long long grad_elements, long long ref_partial_floats);   // -1 = negative sizes
float* det_ref_partials(void* scratch, long long grad_elements);
cudaError_t det_begin(void* scratch, long long grad_elements, cudaStream_t stream);   // zero header + accumulators
cudaError_t det_absmax(int dtype, const void* x, long long rows, int cols, long long ld, unsigned long long* slot,
                       cudaStream_t stream);
cudaError_t det_attn_sum_max(bool f64, const void* attn, long long pairs, int LP, unsigned long long* slot,
                             cudaStream_t stream);
// bound B = count * max|g| * (amax_mode 0: max pair sum |a|; 1: 1, or non-finite when the scanned logits are)
cudaError_t det_finalize(DetHeader* h, double count, int amax_mode, bool f64, cudaStream_t stream);
cudaError_t det_finish(int dtype, const long long* acc, void* out, long long count, const DetHeader* h,
                       cudaStream_t stream);
cudaError_t det_fold_ref(const float* part, float* grad_ref, long long rows, int M, int R, cudaStream_t stream);
// scratch of at least det_scratch_bytes(N*S*M*D, 0) (plain) / (N*S*M*D, grad_ref ? N*Lq*L*M*ref_dim : 0) (fused)
cudaError_t backward_deterministic(const BwdArgs& a, void* scratch, long long scratch_bytes, cudaStream_t stream);
cudaError_t fused_backward_deterministic(const FusedArgs& a, void* scratch, long long scratch_bytes,
                                         cudaStream_t stream);

// Dropout keep rule (DESIGN.md section 3.16): an element is kept iff its 16-bit Philox draw (dropout_keep8 in
// msda_common.cuh) is >= thresh = floor(p * 65536 + 0.5); kept values are multiplied by scale = float(1 / (1 - p)).
// false for p outside (0, 1).
struct DropoutRule {
    unsigned thresh;
    float scale;
};
inline bool dropout_rule(float p, DropoutRule* r)
{
    if (!(p > 0.f && p < 1.f)) return false;
    r->thresh = (unsigned)((double)p * 65536.0 + 0.5);
    r->scale = (float)(1.0 / (1.0 - (double)p));
    return true;
}

// Layer epilogues (layer_epilogue.cu):  y = LayerNorm(residual + act(branch)) * gamma + beta,
// optional y_pos = y + pos; backward of the same.
struct AddLayerNormArgs {
    int dtype;                // kF32 / kBF16 / kF16: type of every tensor below except mean/rstd/partial
    int act;                  // 0 identity, 1 relu, 2 gelu (erf)
    long long rows;
    int C;
    float eps;
    const void* branch;       // [rows, C]
    const void* residual;     // [rows, C] or null
    const void* gamma;        // [C]
    const void* beta;         // [C]   (forward)
    const void* pos;          // [rows, C] or null (forward, with y_pos)
    void* y;                  // forward out
    void* y_pos;              // forward out or null
    float* mean;              // [rows] forward out (may be null) / backward in
    float* rstd;
    // backward
    const void* dy;           // [rows, C]
    const void* dy_pos;       // [rows, C] or null
    void* d_branch;           // written unless (act == 0 and d_residual != null): then d_branch == d_residual
    void* d_residual;         // or null
    void* d_gamma;            // [C]
    void* d_beta;             // [C]
    float* partial;           // [partial_blocks, 2, C] fp32 scratch
    int partial_blocks;       // from add_layernorm_partial_blocks(rows)
    // dropout on act(branch): v = residual + act(branch) * mask * scale; null key = no dropout.  With dropout, d_branch
    // is always written (never aliases d_residual)
    const unsigned long long* drop_key;
    DropoutRule drop;
};
int add_layernorm_chunks(int dtype, int C);            // 0 = unsupported shape
int add_layernorm_partial_blocks(long long rows);
bool add_layernorm_dropout_supported(int dtype, int C);   // the widths the dropout path takes
cudaError_t add_layernorm(const AddLayerNormArgs& a, bool backward, cudaStream_t stream);
// y = x * mask * scale over n contiguous elements (in place allowed); dx = out > 0 ? g * scale : 0 (the backward of
// dropout(relu(.)) from its saved output)
cudaError_t dropout(int dtype, const void* x, void* y, long long n, const unsigned long long* key, DropoutRule rule,
                    cudaStream_t stream);
cudaError_t relu_dropout_grad(int dtype, const void* g, const void* out, void* dx, long long n, float scale,
                              cudaStream_t stream);
// Fused feed-forward block on tcgen05 (ffn_fused.cu): y = LayerNorm(x + W2 relu(W1 x + b1) + b2), y_pos = y + pos
struct FfnArgs {
    int dtype;                // kBF16
    long long rows;
    int C, F;                 // d_model (256), d_ffn (multiple of 64)
    float eps;
    const void* x;            // [rows, C]
    const void* w1;           // [F, C]   (nn.Linear weight layout)
    const void* b1;           // [F]
    const void* w2;           // [C, F]
    const void* b2;           // [C]
    const void* gamma;        // [C]
    const void* beta;         // [C]
    const void* pos;          // [rows, C] or null
    void* y;                  // [rows, C]
    void* y_pos;              // [rows, C] or null
};
bool ffn_layernorm_supported(int dtype, int d_model, int d_ffn);
cudaError_t ffn_layernorm_forward(const FfnArgs& a, cudaStream_t stream);

// Output projection + residual + LayerNorm on tcgen05 (proj_fused.cu): y = LayerNorm(residual + x @ W^T + b), y_pos = y + pos
struct ProjArgs {
    int dtype;                // kBF16
    long long rows;
    int C;                    // d_model (256): W is [C, C] in nn.Linear layout
    float eps;
    const void* x;            // [rows, C]
    const void* w;            // [C, C]
    const void* b;            // [C]
    const void* residual;     // [rows, C] or null
    const void* gamma;        // [C]
    const void* beta;         // [C]
    const void* pos;          // [rows, C] or null
    void* y;                  // [rows, C]
    void* y_pos;              // [rows, C] or null
};
bool proj_layernorm_supported(int dtype, int d_in, int d_out);
cudaError_t proj_layernorm_forward(const ProjArgs& a, cudaStream_t stream);

int group_norm_tokens_slabs(int dtype, long long S, int C, int G);    // 0 = unsupported shape
cudaError_t group_norm_tokens(int dtype, const void* x, const void* pre_bias, const void* gamma, const void* beta,
                              void* y, float* partial, int N, long long S, int C, int G, int slabs, float eps,
                              long long item_stride, cudaStream_t stream);
bool norm_act_supported(int dtype, int C);
cudaError_t norm_act_forward(int dtype, const void* x, const void* gamma, const void* beta, void* y, long long rows,
                             int C, float eps, int act, cudaStream_t stream);
cudaError_t tf32_split(const float* x, float* out, long long rows, int cols, cudaStream_t stream);
// y = x W^T + b (+ ReLU) in fp32 with the three-term TF32 split evaluated inside one tcgen05 kernel (linear_tf32x3.cu)
// y = x W^T + b (+ ReLU, + rows zeroed by a mask) in bf16: TMA / tcgen05 / TMEM kernel of linear_bf16.cu
bool linear_bf16_supported(int n, int k);
cudaError_t linear_bf16(const void* x, const void* w, const void* bias, const unsigned char* row_mask, long long rows, int n,
                        int k, int relu, void* y, cudaStream_t stream);
// y = dropout(relu(x W^T + b)) in the epilogue: mask of element row * n + col from `key` (dropout_keep8)
cudaError_t linear_bf16_relu_dropout(const void* x, const void* w, const void* bias, long long rows, int n, int k,
                                     const unsigned long long* key, DropoutRule rule, void* y, cudaStream_t stream);
// weight / bias gradient of that layer: dW [n, k] = g^T x, db [n] = sum over rows of g (bf16, fp32 split-K partials in
// `scratch`, summed in a fixed order by a second kernel: deterministic)
bool linear_bf16_wgrad_supported(int n, int k);
long long linear_bf16_wgrad_scratch_floats(long long rows, int n, int k);   // 0 = unsupported
cudaError_t linear_bf16_wgrad(const void* g, const void* x, long long rows, int n, int k, void* dw, void* db,
                              float* scratch, long long scratch_floats, cudaStream_t stream);
bool linear_tf32x3_supported(int n, int k);
cudaError_t linear_tf32x3(const float* x, const float* w_hi, const float* w_lo, const float* bias, long long rows, int n,
                          int k, int relu, float* y, cudaStream_t stream);
// y = dropout(relu(x W^T + b)) in the epilogue: mask of element row * n + col from `key` (dropout_keep8)
cudaError_t linear_tf32x3_relu_dropout(const float* x, const float* w_hi, const float* w_lo, const float* bias,
                                       long long rows, int n, int k, const unsigned long long* key, DropoutRule rule,
                                       float* y, cudaStream_t stream);
// weight / bias gradient of that layer: dW [n, k] = g^T x, db [n] = sum over rows of g (fp32, the three-term split with
// both operands split in shared memory; fp32 split-K partials in `scratch`, summed in a fixed order: deterministic)
bool linear_tf32x3_wgrad_supported(int n, int k);
long long linear_tf32x3_wgrad_scratch_floats(long long rows, int n, int k);   // 0 = unsupported
cudaError_t linear_tf32x3_wgrad(const float* g, const float* x, long long rows, int n, int k, float* dw, float* db,
                                float* scratch, long long scratch_floats, cudaStream_t stream);
cudaError_t sine_coordinates(const unsigned char* mask, float* y_embed, float* x_embed, int N, int H, int W,
                             int normalize, float scale, cudaStream_t stream);
cudaError_t sine_position_tokens(int dtype, const float* y_embed, const float* x_embed, const float* dim_t,
                                 const void* add, void* out, int N, long long HW, int F, long long S, long long start,
                                 cudaStream_t stream);
cudaError_t flatten_level(int dtype, const void* x, const void* add, void* out, int N, int C, int HW, long long S,
                          long long start, cudaStream_t stream);
// RoIAlign on token-major maps (roi_align.cu): feat [N, H*W, C], rois [K,5] (batch index, x1, y1, x2, y2) in fp32
// (fp64 when dtype == kF64), out / grad_out [K, PH*PW, C], grad_accum [N, H*W, C] fp32 (fp64) zero-initialised.
struct RoiAlignArgs {
    int dtype;
    const void* feat;
    const void* rois;
    void* out;
    const void* grad_out;
    void* grad_accum;
    int N, H, W, C, K, PH, PW;
    double scale;
    int sampling_ratio, aligned;
};
cudaError_t roi_align_forward(const RoiAlignArgs& a, cudaStream_t stream);
cudaError_t roi_align_backward(const RoiAlignArgs& a, cudaStream_t stream);
// grad_accum is then the dtype gradient, fully written; scratch >= det_scratch_bytes(N*H*W*C, 0)
cudaError_t roi_align_backward_deterministic(const RoiAlignArgs& a, void* scratch, long long scratch_bytes,
                                             cudaStream_t stream);

int colsum_blocks(int dtype, long long rows, int C);   // 0 = unsupported shape
cudaError_t colsum(int dtype, const void* x, long long rows, int C, void* out, float* partial, int blocks,
                   cudaStream_t stream);
cudaError_t zero_masked_rows(int dtype, void* data, const unsigned char* mask, long long rows, int C,
                             cudaStream_t stream);

// Batched rectangular linear assignment (hungarian.cu, DESIGN.md section 3.17)
long long linear_assignment_scratch_bytes(int P, int Q, int Tmax);
cudaError_t linear_assignment(const float* cost, long long problem_stride, long long query_stride,
                              const int64_t* counts, int P, int Q, int Tmax, int* query_of_target,
                              int* target_of_query, int* status, void* scratch, long long scratch_bytes,
                              cudaStream_t stream);

}  // namespace msda
