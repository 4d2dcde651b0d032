// Layer epilogues around the deformable attention (SURVEY 8f rank 1) for sm_100a.
//
// Every layer class of the reference that owns an MSDeformAttn wraps it as
//     x = LayerNorm(residual + dropout(branch))                         (deformable_transformer_single.py:538-541,
//     x = LayerNorm(x + dropout(act(Linear(x))))   (fusion layers)       :393-400, :452-459, :544-548, :617-642)
// and the next deformable attention queries with `x + pos` (:530-531, :538).  In the reference these
// are separate element-wise launches (add, LayerNorm, add) that each re-read and re-write the
// [rows, C] activation; here ONE kernel per direction does
//     v      = residual + act(branch)              act in {identity, relu, gelu(erf)}
//     y      = LayerNorm(v) * gamma + beta
//     y_pos  = y + pos                              (optional second output: the next layer's query)
// with fp32 arithmetic, 16-byte accesses and one warp per row (row statistics by shuffles, no
// shared memory, no block barrier).  The backward kernel produces d branch, d residual and
// per-CTA partial sums of d gamma / d beta that a second tiny kernel folds.
// These kernels are HBM-bound: algorithmic bytes = every operand once.
//
// Also here: zero_masked_rows - `value.masked_fill(padding_mask[..., None], 0)` of
// MSDeformAttn.forward (models/ops/modules/ms_deform_attn.py:95-96) done in place on the fresh
// projection output, touching only the mask bytes and the masked rows.
#include "msda_common.cuh"
#include "msda_launch.h"

namespace msda {

enum Act { kActNone = 0, kActRelu = 1, kActGelu = 2 };

template <int ACT> __device__ __forceinline__ float act_fwd(float x)
{
    if constexpr (ACT == kActRelu) return fmaxf(x, 0.f);
    if constexpr (ACT == kActGelu) return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f));
    return x;
}
template <int ACT> __device__ __forceinline__ float act_bwd(float x)      // d act / d x
{
    if constexpr (ACT == kActRelu) return x > 0.f ? 1.f : 0.f;
    if constexpr (ACT == kActGelu) {
        const float cdf = 0.5f * (1.f + erff(x * 0.70710678118654752440f));
        const float pdf = 0.39894228040143267794f * expf(-0.5f * x * x);
        return cdf + x * pdf;
    }
    return 1.f;
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

template <typename T> struct Vec16 { static constexpr int n = 16 / (int)sizeof(T); };

template <typename T> __device__ __forceinline__ void load16(const T* p, float* f)
{
    const uint4 raw = *reinterpret_cast<const uint4*>(p);
    unpack<T>(raw, f);
}
template <typename T> __device__ __forceinline__ void load16_stream(const T* p, float* f)
{
    unpack<T>(ldg_stream_v4(p), f);
}
template <typename T> __device__ __forceinline__ void store16(T* p, const float* f)
{
    *reinterpret_cast<uint4*>(p) = pack<T>(f);
}
// round-trip through the storage type (y_pos is defined on the ROUNDED y, like the unfused chain)
template <typename T> __device__ __forceinline__ float round_to(float v) { return to_f32<T>(from_f32<T>(v)); }

// keep bits of the V elements from flat index e0 on (e0 % 8 + V <= 8): bit i = element e0 + i kept
__device__ __forceinline__ unsigned keep_bits(long long e0, unsigned long long key, unsigned thresh)
{
    return dropout_keep8((unsigned long long)e0 >> 3, key, thresh) >> (e0 & 7);
}
// a * mask * scale: a dropped element is a * 0, so NaN and Inf propagate as in torch's dropout
__device__ __forceinline__ float drop_mul(unsigned bits, int e, float scale) { return (bits >> e) & 1u ? scale : 0.f; }

constexpr int kLnWarps = 8;

// K = 16-byte chunks per lane: C = K * 32 * (16 / sizeof(T)).
// DROP: v = residual + act(branch) * mask * scale (dropout on the branch, mask of element row * C + c).
template <typename T, int K, int ACT, bool DROP>
__global__ void __launch_bounds__(kLnWarps * 32)
add_layernorm_fwd_kernel(const T* __restrict__ branch, const T* __restrict__ residual,
                         const T* __restrict__ gamma, const T* __restrict__ beta, const T* __restrict__ pos,
                         T* __restrict__ y, T* __restrict__ y_pos, float* __restrict__ mean_out,
                         float* __restrict__ rstd_out, long long rows, float eps,
                         const unsigned long long* __restrict__ drop_key, unsigned drop_thresh, float drop_scale)
{
    constexpr int V = Vec16<T>::n;
    constexpr int C = K * 32 * V;
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * kLnWarps + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * kLnWarps;

    float g[K][V], b[K][V];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        load16<T>(gamma + (k * 32 + lane) * V, g[k]);
        load16<T>(beta + (k * 32 + lane) * V, b[k]);
    }
    unsigned long long key = 0;
    if constexpr (DROP) key = *drop_key;
    for (long long row = warp0; row < rows; row += nwarps) {
        const long long base = row * C;
        float v[K][V];
#pragma unroll
        for (int k = 0; k < K; ++k) load16_stream<T>(branch + base + (k * 32 + lane) * V, v[k]);
        if constexpr (DROP) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const unsigned bits = keep_bits(base + (k * 32 + lane) * V, key, drop_thresh);
#pragma unroll
                for (int e = 0; e < V; ++e) v[k][e] = act_fwd<ACT>(v[k][e]) * drop_mul(bits, e, drop_scale);
            }
        }
        if (residual != nullptr) {
            float r[K][V];
#pragma unroll
            for (int k = 0; k < K; ++k) load16_stream<T>(residual + base + (k * 32 + lane) * V, r[k]);
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int e = 0; e < V; ++e) v[k][e] = r[k][e] + (DROP ? v[k][e] : act_fwd<ACT>(v[k][e]));
        } else if constexpr (!DROP) {
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int e = 0; e < V; ++e) v[k][e] = act_fwd<ACT>(v[k][e]);
        }
        float p[K][V];
        if (y_pos != nullptr) {
#pragma unroll
            for (int k = 0; k < K; ++k) load16_stream<T>(pos + base + (k * 32 + lane) * V, p[k]);
        }
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int e = 0; e < V; ++e) s += v[k][e];
        const float mean = warp_sum(s) * (1.f / C);
        float ss = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int e = 0; e < V; ++e) { const float d = v[k][e] - mean; ss = fmaf(d, d, ss); }
        const float rstd = rsqrtf(warp_sum(ss) * (1.f / C) + eps);
        if (mean_out != nullptr && lane == 0) { mean_out[row] = mean; rstd_out[row] = rstd; }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float o[V];
#pragma unroll
            for (int e = 0; e < V; ++e) o[e] = fmaf((v[k][e] - mean) * rstd, g[k][e], b[k][e]);
            store16<T>(y + base + (k * 32 + lane) * V, o);
            if (y_pos != nullptr) {
#pragma unroll
                for (int e = 0; e < V; ++e) o[e] = round_to<T>(o[e]) + p[k][e];
                store16<T>(y_pos + base + (k * 32 + lane) * V, o);
            }
        }
    }
}

// d_branch = d v * act'(branch), d_residual = d v, with
//   d v = rstd * (gy*gamma - mean_c(gy*gamma) - xhat * mean_c(gy*gamma*xhat)),  gy = dy (+ dy_pos)
// partial[blockIdx][0][c] = sum over this CTA's rows of gy*xhat, partial[blockIdx][1][c] = sum of gy.
// DROP: the forward's mask is regenerated from the key, both for v and for d_branch = d v * mask * scale * act'(branch).
template <typename T, int K, int ACT, bool DROP>
__global__ void __launch_bounds__(kLnWarps * 32, DROP ? 1 : 0)
add_layernorm_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ dy_pos, const T* __restrict__ branch,
                         const T* __restrict__ residual, const T* __restrict__ gamma,
                         const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                         T* __restrict__ d_branch, T* __restrict__ d_residual, float* __restrict__ partial,
                         long long rows, const unsigned long long* __restrict__ drop_key, unsigned drop_thresh,
                         float drop_scale)
{
    constexpr int V = Vec16<T>::n;
    constexpr int C = K * 32 * V;
    __shared__ float s_red[kLnWarps][C];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long warp0 = (long long)blockIdx.x * kLnWarps + warp;
    const long long nwarps = (long long)gridDim.x * kLnWarps;

    float g[K][V], dg[K][V], db[K][V];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        load16<T>(gamma + (k * 32 + lane) * V, g[k]);
#pragma unroll
        for (int e = 0; e < V; ++e) { dg[k][e] = 0.f; db[k][e] = 0.f; }
    }
    unsigned long long key = 0;
    if constexpr (DROP) key = *drop_key;
    for (long long row = warp0; row < rows; row += nwarps) {
        const long long base = row * C;
        float gy[K][V], x[K][V], v[K][V];
        unsigned bits[K];
        if constexpr (DROP) {
#pragma unroll
            for (int k = 0; k < K; ++k) bits[k] = keep_bits(base + (k * 32 + lane) * V, key, drop_thresh);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            load16_stream<T>(dy + base + (k * 32 + lane) * V, gy[k]);
            load16_stream<T>(branch + base + (k * 32 + lane) * V, x[k]);
        }
        if (dy_pos != nullptr) {
            float t[K][V];
#pragma unroll
            for (int k = 0; k < K; ++k) load16_stream<T>(dy_pos + base + (k * 32 + lane) * V, t[k]);
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int e = 0; e < V; ++e) gy[k][e] += t[k][e];
        }
        if (residual != nullptr) {
#pragma unroll
            for (int k = 0; k < K; ++k) load16_stream<T>(residual + base + (k * 32 + lane) * V, v[k]);
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int e = 0; e < V; ++e)
                    v[k][e] += DROP ? act_fwd<ACT>(x[k][e]) * drop_mul(bits[k], e, drop_scale) : act_fwd<ACT>(x[k][e]);
        } else {
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int e = 0; e < V; ++e)
                    v[k][e] = DROP ? act_fwd<ACT>(x[k][e]) * drop_mul(bits[k], e, drop_scale) : act_fwd<ACT>(x[k][e]);
        }
        const float mean = mean_in[row], rstd = rstd_in[row];
        float c1 = 0.f, c2 = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const float xhat = (v[k][e] - mean) * rstd;
                const float gg = gy[k][e] * g[k][e];
                dg[k][e] = fmaf(gy[k][e], xhat, dg[k][e]);
                db[k][e] += gy[k][e];
                v[k][e] = xhat;
                gy[k][e] = gg;
                c1 += gg;
                c2 = fmaf(gg, xhat, c2);
            }
        c1 = warp_sum(c1) * (1.f / C);
        c2 = warp_sum(c2) * (1.f / C);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float dv[V];
#pragma unroll
            for (int e = 0; e < V; ++e) dv[e] = rstd * (gy[k][e] - c1 - v[k][e] * c2);
            if (d_residual != nullptr) store16<T>(d_residual + base + (k * 32 + lane) * V, dv);
            if (DROP) {
#pragma unroll
                for (int e = 0; e < V; ++e) dv[e] *= drop_mul(bits[k], e, drop_scale) * act_bwd<ACT>(x[k][e]);
                store16<T>(d_branch + base + (k * 32 + lane) * V, dv);
            } else if (ACT != kActNone || d_residual == nullptr) {
#pragma unroll
                for (int e = 0; e < V; ++e) dv[e] *= act_bwd<ACT>(x[k][e]);
                store16<T>(d_branch + base + (k * 32 + lane) * V, dv);
            }
        }
    }
    // fold the warps' partial d gamma / d beta through shared memory, one [2, C] row per CTA
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int e = 0; e < V; ++e) s_red[warp][(k * 32 + lane) * V + e] = pass == 0 ? dg[k][e] : db[k][e];
        __syncthreads();
        for (int c = threadIdx.x; c < C; c += kLnWarps * 32) {
            float t = 0.f;
#pragma unroll
            for (int w = 0; w < kLnWarps; ++w) t += s_red[w][c];
            partial[((long long)blockIdx.x * 2 + pass) * C + c] = t;
        }
        __syncthreads();
    }
}

// d_gamma[c] = sum_b partial[b][0][c], d_beta[c] = sum_b partial[b][1][c]
template <typename T>
__global__ void fold_partials_kernel(const float* __restrict__ partial, int nblocks, int C,
                                     T* __restrict__ d_gamma, T* __restrict__ d_beta)
{
    const int col = blockIdx.x * 32 + (threadIdx.x & 31);      // 32 columns per CTA, 8 row-slices
    const int slice = threadIdx.x >> 5;
    __shared__ float s[8][2][33];
    float a = 0.f, b = 0.f;
    if (col < C) {
        for (int r = slice; r < nblocks; r += 8) {
            a += partial[((long long)r * 2 + 0) * C + col];
            b += partial[((long long)r * 2 + 1) * C + col];
        }
    }
    s[slice][0][threadIdx.x & 31] = a;
    s[slice][1][threadIdx.x & 31] = b;
    __syncthreads();
    if (slice == 0 && col < C) {
        float ta = 0.f, tb = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) { ta += s[w][0][threadIdx.x]; tb += s[w][1][threadIdx.x]; }
        d_gamma[col] = from_f32<T>(ta);
        d_beta[col] = from_f32<T>(tb);
    }
}

// rows whose mask byte is non-zero are overwritten with zeros; 32 rows per warp step
template <typename T>
__global__ void __launch_bounds__(256)
zero_masked_rows_kernel(T* __restrict__ data, const unsigned char* __restrict__ mask, long long rows, int C)
{
    constexpr int V = Vec16<T>::n;
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * 8;
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    for (long long r0 = warp0 * 32; r0 < rows; r0 += nwarps * 32) {
        const long long r = r0 + lane;
        unsigned hit = __ballot_sync(0xffffffffu, r < rows && mask[r] != 0);
        while (hit) {
            const int bit = __ffs(hit) - 1;
            hit &= hit - 1;
            T* row = data + (r0 + bit) * C;
            for (int c = lane * V; c < C; c += 32 * V) *reinterpret_cast<uint4*>(row + c) = z;
        }
    }
}

// Column sums of a [rows, C] matrix (bias gradient of a Linear: grad_bias = sum over tokens of
// grad_output).  Thread = one 16-byte column chunk x one row lane; per-CTA partials [gridDim, C] in
// fp32, folded by colsum_fold_kernel.  nch = chunks per row, rl = row lanes per CTA (rl * nch <= 256).
template <typename T>
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const T* __restrict__ x, long long rows, int C, int nch, int rl, float* __restrict__ partial)
{
    constexpr int V = Vec16<T>::n;
    extern __shared__ float s_cs[];                    // [rl][C]
    const int ch = threadIdx.x % nch, lane_r = threadIdx.x / nch;
    const bool worker = lane_r < rl;
    float acc[V];
#pragma unroll
    for (int e = 0; e < V; ++e) acc[e] = 0.f;
    if (worker) {
        const long long step = (long long)gridDim.x * rl;
        long long r = (long long)blockIdx.x * rl + lane_r;
        // two rows in flight per thread
        for (; r + step < rows; r += 2 * step) {
            float a[V], b[V];
            load16_stream<T>(x + r * C + ch * V, a);
            load16_stream<T>(x + (r + step) * C + ch * V, b);
#pragma unroll
            for (int e = 0; e < V; ++e) acc[e] += a[e] + b[e];
        }
        if (r < rows) {
            float a[V];
            load16_stream<T>(x + r * C + ch * V, a);
#pragma unroll
            for (int e = 0; e < V; ++e) acc[e] += a[e];
        }
#pragma unroll
        for (int e = 0; e < V; ++e) s_cs[lane_r * C + ch * V + e] = acc[e];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
        float t = 0.f;
        for (int w = 0; w < rl; ++w) t += s_cs[w * C + c];
        partial[(long long)blockIdx.x * C + c] = t;
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
colsum_fold_kernel(const float* __restrict__ partial, int nblocks, int C, T* __restrict__ out)
{
    const int col = blockIdx.x * 32 + (threadIdx.x & 31);
    const int slice = threadIdx.x >> 5;
    __shared__ float s[8][33];
    float a = 0.f;
    if (col < C)
        for (int r = slice; r < nblocks; r += 8) a += partial[(long long)r * C + col];
    s[slice][threadIdx.x & 31] = a;
    __syncthreads();
    if (slice == 0 && col < C) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += s[w][threadIdx.x];
        out[col] = from_f32<T>(t);
    }
}

// One pyramid level, NCHW -> token-major: out[n, start + p, c] = x[n, c, p] (+ add[c]), p = y*W + x.
// The reference does this with flatten(2).transpose(1,2) per level, a level-embedding add and torch.cat
// (deformable_transformer_single.py:190-206).  32 x 32 tiles through shared memory: reads coalesced along
// the pixels, writes coalesced along the channels.
template <typename T>
__global__ void __launch_bounds__(256)
flatten_level_kernel(const T* __restrict__ x, const T* __restrict__ add, T* __restrict__ out,
                     int C, int HW, long long S, long long start)
{
    __shared__ T tile[32][33];
    const int n = blockIdx.z;
    const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8 threads
    const T* xin = x + (long long)n * C * HW;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + ty + 8 * k, p = p0 + tx;
        if (c < C && p < HW) tile[ty + 8 * k][tx] = xin[(long long)c * HW + p];
    }
    __syncthreads();
    T* o = out + ((long long)n * S + start) * C;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int p = p0 + ty + 8 * k, c = c0 + tx;
        if (c < C && p < HW) {
            float v = to_f32<T>(tile[tx][ty + 8 * k]);
            if (add != nullptr) v = to_f32<T>(from_f32<T>(v + to_f32<T>(add[c])));
            o[(long long)p * C + c] = from_f32<T>(v);
        }
    }
}

// The same transpose for channel counts that are whole 16-byte vectors (every model of the reference: 256 channels):
// 64 pixels x 128 bytes of channels per CTA, 16 independent loads per thread in flight before the tile is written,
// and one 16-byte store per thread per pixel -- 8 consecutive lanes write one pixel's whole 128-byte line.  The 32 x 32
// kernel above issues ~43 instructions per element (ncu: 84 % issue-active at 2.4 TB/s); this one ~6.
template <typename T>
__global__ void __launch_bounds__(256)
flatten_level_vec_kernel(const T* __restrict__ x, const T* __restrict__ add, T* __restrict__ out,
                         int C, int HW, long long S, long long start)
{
    constexpr int VEC = 16 / sizeof(T), CT = 8 * VEC, PT = 64, PITCH = PT + 4 / sizeof(T);
    __shared__ T tile[CT][PITCH];
    const int n = blockIdx.z;
    const int p0 = blockIdx.x * PT, c0 = blockIdx.y * CT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const T* row = x + ((long long)n * C + c0 + warp) * HW + p0 + lane;
    const long long step = 8LL * HW;
    T r[CT / 8][2];
    const bool in0 = p0 + lane < HW, in1 = p0 + lane + 32 < HW;
#pragma unroll
    for (int k = 0; k < CT / 8; ++k, row += step) {
        const bool ok = c0 + warp + 8 * k < C;
        r[k][0] = ok && in0 ? row[0] : T();
        r[k][1] = ok && in1 ? row[32] : T();
    }
#pragma unroll
    for (int k = 0; k < CT / 8; ++k) {
        tile[warp + 8 * k][lane] = r[k][0];
        tile[warp + 8 * k][lane + 32] = r[k][1];
    }
    __syncthreads();
    const int chunk = threadIdx.x & 7;
    const int c = c0 + chunk * VEC;
    if (c >= C) return;                                         // C is a multiple of VEC: chunks are whole or absent
    float addv[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) addv[v] = add != nullptr ? to_f32<T>(add[c + v]) : 0.f;
    T* o = out + ((long long)n * S + start + p0) * C + c;
#pragma unroll
    for (int pp = threadIdx.x >> 3; pp < PT; pp += 32) {
        if (p0 + pp >= HW) break;
        alignas(16) T v16[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const T t = tile[chunk * VEC + v][pp];
            v16[v] = add != nullptr ? from_f32<T>(to_f32<T>(t) + addv[v]) : t;
        }
        *reinterpret_cast<uint4*>(o + (long long)pp * C) = *reinterpret_cast<const uint4*>(v16);
    }
}

template <typename T>
static void launch_flatten(const void* x, const void* add, void* out, int N, int C, int HW, long long S,
                           long long start, cudaStream_t st)
{
    constexpr int VEC = 16 / sizeof(T);
    if (C % VEC == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0) {
        const dim3 grid((HW + 63) / 64, (C + 8 * VEC - 1) / (8 * VEC), N);
        flatten_level_vec_kernel<T><<<grid, 256, 0, st>>>((const T*)x, (const T*)add, (T*)out, C, HW, S, start);
    } else {
        const dim3 grid((HW + 31) / 32, (C + 31) / 32, N);
        flatten_level_kernel<T><<<grid, 256, 0, st>>>((const T*)x, (const T*)add, (T*)out, C, HW, S, start);
    }
}

cudaError_t flatten_level(int dtype, const void* x, const void* add, void* out, int N, int C, int HW, long long S,
                          long long start, cudaStream_t st)
{
    if (N <= 0 || C <= 0 || HW <= 0) return cudaSuccess;
    if (N > 65535) return cudaErrorInvalidValue;
    switch (dtype) {
        case kF32: launch_flatten<float>(x, add, out, N, C, HW, S, start, st); break;
        case kBF16: launch_flatten<__nv_bfloat16>(x, add, out, N, C, HW, S, start, st); break;
        case kF16: launch_flatten<__half>(x, add, out, N, C, HW, S, start, st); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
int colsum_blocks(int dtype, long long rows, int C)
{
    const int V = dtype == kF32 ? 4 : 8;
    if ((dtype != kF32 && dtype != kBF16 && dtype != kF16) || C <= 0 || C % V != 0 || C / V > 256) return 0;
    const int rl = 256 / (C / V);
    long long want = (rows + 4LL * rl - 1) / (4LL * rl);     // >= 4 rows per row lane
    if (want < 1) want = 1;
    return (int)(want < 148 * 4 ? want : 148 * 4);
}

template <typename T>
static cudaError_t launch_colsum(const T* x, long long rows, int C, T* out, float* partial, int blocks, cudaStream_t st)
{
    constexpr int V = Vec16<T>::n;
    const int nch = C / V, rl = 256 / nch;
    colsum_partial_kernel<T><<<blocks, 256, (size_t)rl * C * sizeof(float), st>>>(x, rows, C, nch, rl, partial);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    colsum_fold_kernel<T><<<(C + 31) / 32, 256, 0, st>>>(partial, blocks, C, out);
    return cudaGetLastError();
}

cudaError_t colsum(int dtype, const void* x, long long rows, int C, void* out, float* partial, int blocks,
                   cudaStream_t st)
{
    if (blocks < 1 || blocks > colsum_blocks(dtype, rows, C)) return cudaErrorInvalidValue;
    switch (dtype) {
        case kF32:  return launch_colsum<float>((const float*)x, rows, C, (float*)out, partial, blocks, st);
        case kBF16: return launch_colsum<__nv_bfloat16>((const __nv_bfloat16*)x, rows, C, (__nv_bfloat16*)out, partial, blocks, st);
        case kF16:  return launch_colsum<__half>((const __half*)x, rows, C, (__half*)out, partial, blocks, st);
        default:    return cudaErrorInvalidValue;
    }
}

static int ln_grid(long long rows)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long want = (rows + kLnWarps - 1) / kLnWarps;
    const long long cap = (long long)sms * 8;                  // persistent: 8 CTAs x 8 warps per SM
    return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

int add_layernorm_chunks(int dtype, int C)
{
    const int per = dtype == kF32 ? 128 : 256;                 // elements covered by one 16-byte chunk per lane
    if (dtype != kF32 && dtype != kBF16 && dtype != kF16) return 0;
    if (C <= 0 || C % per != 0) return 0;
    const int k = C / per;
    return (k == 1 || k == 2 || k == 4) ? k : 0;
}

template <typename T, int K, bool DROP>
static cudaError_t launch_ln_fwd(const AddLayerNormArgs& a, cudaStream_t st)
{
    const int grid = ln_grid(a.rows);
#define MSDA_LN_FWD(ACT) \
    add_layernorm_fwd_kernel<T, K, ACT, DROP><<<grid, kLnWarps * 32, 0, st>>>( \
        (const T*)a.branch, (const T*)a.residual, (const T*)a.gamma, (const T*)a.beta, (const T*)a.pos, \
        (T*)a.y, (T*)a.y_pos, a.mean, a.rstd, a.rows, a.eps, a.drop_key, a.drop.thresh, a.drop.scale)
    switch (a.act) {
        case kActNone: MSDA_LN_FWD(kActNone); break;
        case kActRelu: MSDA_LN_FWD(kActRelu); break;
        case kActGelu: MSDA_LN_FWD(kActGelu); break;
        default: return cudaErrorInvalidValue;
    }
#undef MSDA_LN_FWD
    return cudaGetLastError();
}

template <typename T, int K, bool DROP>
static cudaError_t launch_ln_bwd(const AddLayerNormArgs& a, cudaStream_t st)
{
    const int grid = a.partial_blocks;
#define MSDA_LN_BWD(ACT) \
    add_layernorm_bwd_kernel<T, K, ACT, DROP><<<grid, kLnWarps * 32, 0, st>>>( \
        (const T*)a.dy, (const T*)a.dy_pos, (const T*)a.branch, (const T*)a.residual, (const T*)a.gamma, \
        a.mean, a.rstd, (T*)a.d_branch, (T*)a.d_residual, a.partial, a.rows, a.drop_key, a.drop.thresh, a.drop.scale)
    switch (a.act) {
        case kActNone: MSDA_LN_BWD(kActNone); break;
        case kActRelu: MSDA_LN_BWD(kActRelu); break;
        case kActGelu: MSDA_LN_BWD(kActGelu); break;
        default: return cudaErrorInvalidValue;
    }
#undef MSDA_LN_BWD
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    fold_partials_kernel<T><<<(a.C + 31) / 32, 256, 0, st>>>(a.partial, grid, a.C, (T*)a.d_gamma, (T*)a.d_beta);
    return cudaGetLastError();
}

template <typename T, bool DROP>
static cudaError_t dispatch_ln(const AddLayerNormArgs& a, bool backward, cudaStream_t st)
{
    switch (add_layernorm_chunks(a.dtype, a.C)) {
        case 1: return backward ? launch_ln_bwd<T, 1, DROP>(a, st) : launch_ln_fwd<T, 1, DROP>(a, st);
        case 2: return backward ? launch_ln_bwd<T, 2, DROP>(a, st) : launch_ln_fwd<T, 2, DROP>(a, st);
        case 4:
            if constexpr (DROP) return cudaErrorInvalidValue;       // see add_layernorm_dropout_supported
            else return backward ? launch_ln_bwd<T, 4, false>(a, st) : launch_ln_fwd<T, 4, false>(a, st);
        default: return cudaErrorInvalidValue;
    }
}
template <typename T>
static cudaError_t dispatch_ln(const AddLayerNormArgs& a, bool backward, cudaStream_t st)
{
    return a.drop_key != nullptr ? dispatch_ln<T, true>(a, backward, st) : dispatch_ln<T, false>(a, backward, st);
}

int add_layernorm_partial_blocks(long long rows) { return ln_grid(rows); }

// With dropout: one or two 16-byte chunks per lane (up to 512 channels of a 16-bit type, 256 of fp32).  The four-chunk
// GELU backward already spills without dropout; the dropout instantiations stop at two chunks and spill nothing.
bool add_layernorm_dropout_supported(int dtype, int C)
{
    const int k = add_layernorm_chunks(dtype, C);
    return k == 1 || k == 2;
}

cudaError_t add_layernorm(const AddLayerNormArgs& a, bool backward, cudaStream_t st)
{
    if (a.rows == 0) return cudaSuccess;
    switch (a.dtype) {
        case kF32:  return dispatch_ln<float>(a, backward, st);
        case kBF16: return dispatch_ln<__nv_bfloat16>(a, backward, st);
        case kF16:  return dispatch_ln<__half>(a, backward, st);
        default:    return cudaErrorInvalidValue;
    }
}

// y = act(LayerNorm(x) * gamma + beta): the normalise-then-activate steps of the TransVOD++ dynamic interaction
// head (features = relu(norm(bmm(...))), /root/reference/models/sparse_roi_head/head.py:156-170), whose rows are
// narrow (64 channels after the first per-box product).  LANES lanes own a row (32 / LANES rows per warp), K 16-byte
// chunks per lane: C = LANES * K * 16 / sizeof(T).  In place is fine (y == x): a lane reads its elements before it
// writes them.  Forward only -- training keeps the PyTorch composition.
template <typename T, int LANES, int K, int ACT>
__global__ void __launch_bounds__(kLnWarps * 32)
norm_act_fwd_kernel(const T* __restrict__ x, const T* __restrict__ gamma, const T* __restrict__ beta, T* __restrict__ y,
                    long long rows, float eps)
{
    constexpr int V = Vec16<T>::n;
    constexpr int C = LANES * K * V;
    constexpr int RPW = 32 / LANES;
    const int lane = threadIdx.x & 31, sub = lane % LANES, rw = lane / LANES;
    const long long first = ((long long)blockIdx.x * kLnWarps + (threadIdx.x >> 5)) * RPW + rw;
    const long long stride = (long long)gridDim.x * kLnWarps * RPW;
    float g[K][V], b[K][V];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        load16<T>(gamma + (k * LANES + sub) * V, g[k]);
        load16<T>(beta + (k * LANES + sub) * V, b[k]);
    }
    // every lane of a warp runs the same number of iterations (the shuffles are warp-wide); rows past the end are
    // clamped for the loads and skipped for the stores
    const long long iters = (rows + stride - 1) / stride;
    for (long long it = 0; it < iters; ++it) {
        const long long row_raw = first + it * stride;
        const bool live = row_raw < rows;
        const long long base = (live ? row_raw : rows - 1) * C;
        float v[K][V];
#pragma unroll
        for (int k = 0; k < K; ++k) load16_stream<T>(x + base + (k * LANES + sub) * V, v[k]);
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int e = 0; e < V; ++e) s += v[k][e];
#pragma unroll
        for (int off = LANES / 2; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        const float mean = s * (1.f / C);
        float ss = 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int e = 0; e < V; ++e) { const float d = v[k][e] - mean; ss = fmaf(d, d, ss); }
#pragma unroll
        for (int off = LANES / 2; off >= 1; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
        const float rstd = rsqrtf(ss * (1.f / C) + eps);
        if (live) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                float o[V];
#pragma unroll
                for (int e = 0; e < V; ++e) {
                    // the unfused chain rounds the LayerNorm output to T before the activation
                    o[e] = act_fwd<ACT>(round_to<T>(fmaf((v[k][e] - mean) * rstd, g[k][e], b[k][e])));
                }
                store16<T>(y + base + (k * LANES + sub) * V, o);
            }
        }
    }
}

template <typename T, int LANES, int K>
static cudaError_t launch_norm_act(const void* x, const void* gamma, const void* beta, void* y, long long rows,
                                   float eps, int act, cudaStream_t st)
{
    const long long rows_per_cta = (long long)kLnWarps * (32 / LANES);
    const long long want = (rows + rows_per_cta - 1) / rows_per_cta;
    const int grid = (int)(want < 148 * 8 ? want : 148 * 8);
#define MSDA_NA(ACT) norm_act_fwd_kernel<T, LANES, K, ACT><<<grid, kLnWarps * 32, 0, st>>>( \
        (const T*)x, (const T*)gamma, (const T*)beta, (T*)y, rows, eps)
    switch (act) {
        case kActNone: MSDA_NA(kActNone); break;
        case kActRelu: MSDA_NA(kActRelu); break;
        case kActGelu: MSDA_NA(kActGelu); break;
        default: return cudaErrorInvalidValue;
    }
#undef MSDA_NA
    return cudaGetLastError();
}

bool norm_act_supported(int dtype, int C)
{
    const int esz = dtype == kF32 ? 4 : (dtype == kBF16 || dtype == kF16 ? 2 : 0);
    if (esz == 0 || C <= 0) return false;
    const int bytes = C * esz;
    return bytes == 128 || bytes == 256 || bytes == 512 || bytes == 1024 || bytes == 2048;
}

template <typename T>
static cudaError_t dispatch_norm_act(int bytes, const void* x, const void* gamma, const void* beta, void* y,
                                     long long rows, float eps, int act, cudaStream_t st)
{
    switch (bytes) {
        case 128:  return launch_norm_act<T, 8, 1>(x, gamma, beta, y, rows, eps, act, st);
        case 256:  return launch_norm_act<T, 16, 1>(x, gamma, beta, y, rows, eps, act, st);
        case 512:  return launch_norm_act<T, 32, 1>(x, gamma, beta, y, rows, eps, act, st);
        case 1024: return launch_norm_act<T, 32, 2>(x, gamma, beta, y, rows, eps, act, st);
        case 2048: return launch_norm_act<T, 32, 4>(x, gamma, beta, y, rows, eps, act, st);
        default:   return cudaErrorInvalidValue;
    }
}

cudaError_t norm_act_forward(int dtype, const void* x, const void* gamma, const void* beta, void* y, long long rows,
                             int C, float eps, int act, cudaStream_t st)
{
    if (!norm_act_supported(dtype, C)) return cudaErrorInvalidValue;
    if (rows == 0) return cudaSuccess;
    switch (dtype) {
        case kF32:  return dispatch_norm_act<float>(C * 4, x, gamma, beta, y, rows, eps, act, st);
        case kBF16: return dispatch_norm_act<__nv_bfloat16>(C * 2, x, gamma, beta, y, rows, eps, act, st);
        case kF16:  return dispatch_norm_act<__half>(C * 2, x, gamma, beta, y, rows, eps, act, st);
        default:    return cudaErrorInvalidValue;
    }
}

// GroupNorm on TOKEN-MAJOR activations: x [N, S, C], groups of C / G consecutive channels, statistics per (n, group)
// over S * C / G elements.  The reference's input projections are Conv2d(1x1) + GroupNorm(32, 256) on NCHW maps that
// the transformer then flattens and transposes (/root/reference/models/deformable_detr_single.py:101-150, :262-267;
// deformable_transformer_single.py:190-206); with the projection computed as a token-major GEMM the norm runs here and
// the NCHW tensor, its transpose and the concatenation never exist.
//   pass 1: per-CTA partial (sum, sum of squares) of each group over a slab of rows -> partial[n][slab][G][2]
//   pass 2: every CTA folds its sample's partials (fp64), then y = (x - mean) * rstd * gamma + beta, in place.
// A 16-byte vector never straddles two groups (host checks (C / G) % V == 0).
constexpr int kGnWarps = 8;
constexpr int kGnMaxGroups = 64;
constexpr int kGnMaxVecs = 256;         // C * sizeof(T) <= 4096 bytes

template <typename T>
__global__ void __launch_bounds__(kGnWarps * 32)
group_norm_tokens_stats_kernel(const T* __restrict__ x, const T* __restrict__ pre_bias, float* __restrict__ partial,
                               long long S, int C, int G, int slabs, long long item_stride)
{
    constexpr int V = Vec16<T>::n;
    __shared__ float s_part[kGnWarps][kGnMaxVecs][2];        // fixed-order fold below: results are deterministic
    const int n = blockIdx.y, slab = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long rows_per = (S + slabs - 1) / slabs;
    const long long r0 = (long long)slab * rows_per, r1 = r0 + rows_per < S ? r0 + rows_per : S;
    const int vecs = C / V, cpg = C / G;
    const T* base = x + (long long)n * item_stride;
    for (int v = lane; v < vecs; v += 32) {                  // a lane keeps to its own vector columns
        float sum = 0.f, sq = 0.f, pb[V];
#pragma unroll
        for (int e = 0; e < V; ++e) pb[e] = 0.f;
        if (pre_bias != nullptr) load16<T>(pre_bias + v * V, pb);
        for (long long r = r0 + warp; r < r1; r += kGnWarps) {
            float f[V];
            load16_stream<T>(base + r * C + v * V, f);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const float t = pre_bias != nullptr ? round_to<T>(f[e] + pb[e]) : f[e];   // the conv output is a T
                sum += t;
                sq = fmaf(t, t, sq);
            }
        }
        s_part[warp][v][0] = sum;
        s_part[warp][v][1] = sq;
    }
    __syncthreads();
    if (threadIdx.x < G) {
        const int vpg = cpg / V;                             // vector columns per group
        float sum = 0.f, sq = 0.f;
        for (int w = 0; w < kGnWarps; ++w)
            for (int v = threadIdx.x * vpg; v < (threadIdx.x + 1) * vpg; ++v) { sum += s_part[w][v][0]; sq += s_part[w][v][1]; }
        float* out = partial + (((long long)n * slabs + slab) * G + threadIdx.x) * 2;
        out[0] = sum;
        out[1] = sq;
    }
}

template <typename T>
__global__ void __launch_bounds__(kGnWarps * 32)
group_norm_tokens_apply_kernel(const T* __restrict__ x, const T* __restrict__ pre_bias,
                               const float* __restrict__ partial, const T* __restrict__ gamma,
                               const T* __restrict__ beta, T* __restrict__ y, long long S, int C, int G, int slabs,
                               float eps, long long item_stride)
{
    constexpr int V = Vec16<T>::n;
    __shared__ float s_mean[kGnMaxGroups], s_rstd[kGnMaxGroups];
    const int n = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < G) {
        double sum = 0.0, sq = 0.0;
        for (int sl = 0; sl < slabs; ++sl) {
            const float* p = partial + (((long long)n * slabs + sl) * G + threadIdx.x) * 2;
            sum += (double)p[0];
            sq += (double)p[1];
        }
        const double cnt = (double)S * (double)(C / G);
        const double mean = sum / cnt;
        double var = sq / cnt - mean * mean;
        var = var > 0.0 ? var : 0.0;
        s_mean[threadIdx.x] = (float)mean;
        s_rstd[threadIdx.x] = (float)(1.0 / sqrt(var + (double)eps));
    }
    __syncthreads();
    const int vecs = C / V, cpg = C / G;
    const T* xin = x + (long long)n * item_stride;
    T* yout = y + (long long)n * item_stride;
    const long long rows_per = (S + gridDim.x - 1) / gridDim.x;
    const long long r0 = (long long)blockIdx.x * rows_per, r1 = r0 + rows_per < S ? r0 + rows_per : S;
    for (int v = lane; v < vecs; v += 32) {
        float g[V], b[V], pb[V];
        load16<T>(gamma + v * V, g);
        load16<T>(beta + v * V, b);
#pragma unroll
        for (int e = 0; e < V; ++e) pb[e] = 0.f;
        if (pre_bias != nullptr) load16<T>(pre_bias + v * V, pb);
        const int grp = v * V / cpg;
        const float mean = s_mean[grp], rstd = s_rstd[grp];
        for (long long r = r0 + warp; r < r1; r += kGnWarps) {
            float f[V];
            load16_stream<T>(xin + r * C + v * V, f);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const float t = pre_bias != nullptr ? round_to<T>(f[e] + pb[e]) : f[e];
                f[e] = fmaf((t - mean) * rstd, g[e], b[e]);
            }
            store16<T>(yout + r * C + v * V, f);
        }
    }
}

int group_norm_tokens_slabs(int dtype, long long S, int C, int G)
{
    const int esz = dtype == kF32 ? 4 : (dtype == kBF16 || dtype == kF16 ? 2 : 0);
    if (esz == 0 || C <= 0 || G <= 0 || G > kGnMaxGroups || C % G != 0 || S <= 0) return 0;
    const int v = 16 / esz;
    if ((C / G) % v != 0 || C / v > kGnMaxVecs) return 0;
    const long long want = (S + 63) / 64;                    // >= 64 rows per slab
    return (int)(want < 64 ? want : 64);
}

template <typename T>
static cudaError_t launch_group_norm_tokens(const void* x, const void* pre_bias, const void* gamma, const void* beta,
                                            void* y, float* partial, int N, long long S, int C, int G, int slabs,
                                            float eps, long long item_stride, cudaStream_t st)
{
    group_norm_tokens_stats_kernel<T><<<dim3(slabs, N), kGnWarps * 32, 0, st>>>((const T*)x, (const T*)pre_bias, partial,
                                                                               S, C, G, slabs, item_stride);
    const long long want = (S + 31) / 32;
    const int per_sample = (int)(want < 296 ? want : 296);
    const int blocks = per_sample > 0 ? per_sample : 1;
    group_norm_tokens_apply_kernel<T><<<dim3(blocks, N), kGnWarps * 32, 0, st>>>(
        (const T*)x, (const T*)pre_bias, partial, (const T*)gamma, (const T*)beta, (T*)y, S, C, G, slabs, eps, item_stride);
    return cudaGetLastError();
}

cudaError_t group_norm_tokens(int dtype, const void* x, const void* pre_bias, const void* gamma, const void* beta,
                              void* y, float* partial, int N, long long S, int C, int G, int slabs, float eps,
                              long long item_stride, cudaStream_t st)
{
    if (N == 0) return cudaSuccess;
    if (slabs <= 0 || slabs != group_norm_tokens_slabs(dtype, S, C, G) || N > 65535) return cudaErrorInvalidValue;
    if (item_stride == 0) item_stride = S * C;
    const int v = dtype == kF32 ? 4 : 8;
    if (item_stride < S * C || item_stride % v != 0) return cudaErrorInvalidValue;
    switch (dtype) {
        case kF32:  return launch_group_norm_tokens<float>(x, pre_bias, gamma, beta, y, partial, N, S, C, G, slabs, eps, item_stride, st);
        case kBF16: return launch_group_norm_tokens<__nv_bfloat16>(x, pre_bias, gamma, beta, y, partial, N, S, C, G, slabs, eps, item_stride, st);
        case kF16:  return launch_group_norm_tokens<__half>(x, pre_bias, gamma, beta, y, partial, N, S, C, G, slabs, eps, item_stride, st);
        default:    return cudaErrorInvalidValue;
    }
}

// Sine position embedding written TOKEN-MAJOR: the reference's PositionEmbeddingSine
// (/root/reference/models/position_encoding.py:20-56) builds [N, 2F, H, W] in fp32 (divide the cumulative row / column
// coordinate by temperature^(2*(k/2)/F), sin on even k, cos on odd k, y block then x block), the backbone joiner casts it
// to the feature dtype, and DeformableTransformer.forward flattens, transposes and adds level_embed[l]
// (deformable_transformer_single.py:196-199).  Here the (tiny) coordinate maps come from the same torch ops and one
// kernel writes pos[n, start + p, c] = T(T(sin|cos(coord[n, p] / dim_t[c % F])) + add[c]) -- one pass, no NCHW tensor.
template <typename T>
__global__ void __launch_bounds__(256)
sine_position_tokens_kernel(const float* __restrict__ y_embed, const float* __restrict__ x_embed,
                            const float* __restrict__ dim_t, const T* __restrict__ add, T* __restrict__ out, int F,
                            long long HW, long long S, long long start, long long pixels)
{
    const long long pix = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);      // one warp per pixel of one item
    if (pix >= pixels) return;
    const int lane = threadIdx.x & 31;
    const long long n = pix / HW, p = pix - n * HW;
    const float ye = y_embed[pix], xe = x_embed[pix];
    T* o = out + (n * S + start + p) * (2 * F);
    // channels 2j and 2j + 1 share dim_t (temperature ** (2 * (k / 2) / F)) and therefore the argument: one division
    // and one sincosf per pair, no divergence between the sin and the cos lanes, a paired store
    for (int c = 2 * lane; c < 2 * F; c += 64) {
        const int k = c < F ? c : c - F;
        const float arg = __fdiv_rn(c < F ? ye : xe, dim_t[k]);
        float sn, cs;
        sincosf(arg, &sn, &cs);
        float v0 = to_f32<T>(from_f32<T>(sn)), v1 = to_f32<T>(from_f32<T>(cs));
        if (add != nullptr) {
            v0 = v0 + to_f32<T>(add[c]);
            v1 = v1 + to_f32<T>(add[c + 1]);
        }
        struct alignas(2 * sizeof(T)) Pair { T a, b; };             // channel pairs are pair-aligned: 2F and c are even
        Pair pr;
        pr.a = from_f32<T>(v0);
        pr.b = from_f32<T>(v1);
        *reinterpret_cast<Pair*>(o + c) = pr;
    }
}

// The cumulative coordinates of PositionEmbeddingSine (position_encoding.py:39-46): y_embed = cumsum over rows of
// ~mask, x_embed = cumsum over columns, optionally (c - 0.5) / (last + 1e-6) * scale -- the ~10 tiny launches per level
// that otherwise dominate the embedding's time.  Counts are exact integers in fp32 and the normalisation uses the
// reference's operation order with IEEE roundings (no contraction), so the maps equal the torch ops bit for bit.
// x: one warp per row (ballot prefix counts).  y: one CTA per 32 columns of an item, a band of rows per warp, the band
// counts exchanged through shared memory.  Both count first and write the final value once (no read-back).
__device__ __forceinline__ float sine_coordinate(int count, int total, int normalize, float scale)
{
    const float c = (float)count;
    return normalize ? __fmul_rn(__fdiv_rn(__fsub_rn(c, 0.5f), __fadd_rn((float)total, 1e-6f)), scale) : c;
}

__global__ void __launch_bounds__(256)
sine_coordinates_kernel(const unsigned char* __restrict__ mask, float* __restrict__ y_embed,
                        float* __restrict__ x_embed, int N, int H, int W, int normalize, float scale, int row_blocks)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if ((int)blockIdx.x < row_blocks) {
        // x: one warp per row; the row is counted, then re-read (L1) for the running prefix
        const long long row = (long long)blockIdx.x * 8 + warp;
        if (row >= (long long)N * H) return;
        const unsigned char* m = mask + row * W;
        float* x = x_embed + row * W;
        int total = 0;
        for (int j0 = 0; j0 < W; j0 += 32)
            total += __popc(__ballot_sync(0xffffffffu, j0 + lane < W && m[j0 + lane] == 0));
        int carry = 0;
        for (int j0 = 0; j0 < W; j0 += 32) {
            const int j = j0 + lane;
            const unsigned bits = __ballot_sync(0xffffffffu, j < W && m[j] == 0);
            if (j < W)
                x[j] = sine_coordinate(carry + __popc(bits & (0xffffffffu >> (31 - lane))), total, normalize, scale);
            carry += __popc(bits);
        }
        return;
    }
    // y: one CTA per (item, 32 columns); warp w owns a band of rows, band counts meet in shared memory
    __shared__ int band[8][32];
    const int col_groups = (W + 31) / 32;
    const int group = blockIdx.x - row_blocks;
    const int n = group / col_groups;
    const int j = (group - n * col_groups) * 32 + lane;
    const int rows = (H + 7) / 8;
    const int i0 = warp * rows, i1 = min(H, i0 + rows);
    const unsigned char* m = mask + (long long)n * H * W + j;
    int count = 0;
    if (j < W) {
#pragma unroll 4
        for (int i = i0; i < i1; ++i) count += m[(long long)i * W] == 0;
    }
    band[warp][lane] = count;
    __syncthreads();
    if (j >= W) return;
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        const int b = band[w][lane];
        before += w < warp ? b : 0;
        total += b;
    }
    float* y = y_embed + (long long)n * H * W + j;
#pragma unroll 4
    for (int i = i0; i < i1; ++i) {
        before += m[(long long)i * W] == 0;
        y[(long long)i * W] = sine_coordinate(before, total, normalize, scale);
    }
}

cudaError_t sine_coordinates(const unsigned char* mask, float* y_embed, float* x_embed, int N, int H, int W,
                             int normalize, float scale, cudaStream_t st)
{
    if (N == 0 || H == 0 || W == 0) return cudaSuccess;
    const long long row_blocks = ((long long)N * H + 7) / 8;
    const long long blocks = row_blocks + (long long)N * ((W + 31) / 32);
    if (blocks > 0x7fffffffLL) return cudaErrorInvalidValue;
    sine_coordinates_kernel<<<(unsigned)blocks, 256, 0, st>>>(mask, y_embed, x_embed, N, H, W, normalize, scale,
                                                             (int)row_blocks);
    return cudaGetLastError();
}

cudaError_t sine_position_tokens(int dtype, const float* y_embed, const float* x_embed, const float* dim_t,
                                 const void* add, void* out, int N, long long HW, int F, long long S, long long start,
                                 cudaStream_t st)
{
    const long long pixels = (long long)N * HW;
    if (pixels == 0 || F == 0) return cudaSuccess;
    if (F & 1) return cudaErrorInvalidValue;      // the reference's 0::2 / 1::2 interleave needs an even F as well
    const unsigned blocks = (unsigned)((pixels + 7) / 8);
    switch (dtype) {
        case kF32:
            sine_position_tokens_kernel<float><<<blocks, 256, 0, st>>>(y_embed, x_embed, dim_t, (const float*)add,
                                                                      (float*)out, F, HW, S, start, pixels);
            break;
        case kBF16:
            sine_position_tokens_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(
                y_embed, x_embed, dim_t, (const __nv_bfloat16*)add, (__nv_bfloat16*)out, F, HW, S, start, pixels);
            break;
        case kF16:
            sine_position_tokens_kernel<__half><<<blocks, 256, 0, st>>>(y_embed, x_embed, dim_t, (const __half*)add,
                                                                       (__half*)out, F, HW, S, start, pixels);
            break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// x [rows, cols] (fp32) -> out [rows, 3 * cols] = [ lo | hi | hi ] per row, hi = x rounded to TF32's 10 mantissa bits
// (nearest, ties away from zero: add half an ulp to the bit pattern, clear the 13 low bits), lo = x - hi (exact in fp32).
// One pass builds the left operand of the error-compensated TF32 product
//     x W^T ~= [ lo_x | hi_x | hi_x ] [ hi_W | lo_W | hi_W ]^T          (ops/functions/layer_epilogue_func.py: linear_tf32x3)
// so that ONE tensor-core GEMM with a 3x longer reduction replaces the SGEMM.  cols % 4 == 0, 16-byte aligned buffers.
__global__ void __launch_bounds__(256)
tf32_split_kernel(const float* __restrict__ x, float* __restrict__ out, long long rows, int cols)
{
    const int vpr = cols / 4;                                  // float4 per row
    const long long vecs = rows * vpr;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < vecs; i += stride) {
        const long long r = i / vpr;
        const int k = (int)(i - r * vpr);
        const float4 v = __ldcs(reinterpret_cast<const float4*>(x) + i);
        float4 h, l;
        h.x = __int_as_float((__float_as_int(v.x) + 0x1000) & 0xffffe000);
        h.y = __int_as_float((__float_as_int(v.y) + 0x1000) & 0xffffe000);
        h.z = __int_as_float((__float_as_int(v.z) + 0x1000) & 0xffffe000);
        h.w = __int_as_float((__float_as_int(v.w) + 0x1000) & 0xffffe000);
        l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
        float4* o = reinterpret_cast<float4*>(out) + r * 3 * vpr + k;
        o[0] = l;
        o[vpr] = h;
        o[2 * vpr] = h;
    }
}

cudaError_t tf32_split(const float* x, float* out, long long rows, int cols, cudaStream_t st)
{
    if (rows <= 0 || cols <= 0) return cudaSuccess;
    if (cols % 4 != 0 || (reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) % 16 != 0)
        return cudaErrorInvalidValue;
    long long blocks = (rows * (cols / 4) + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    tf32_split_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, out, rows, cols);
    return cudaGetLastError();
}

cudaError_t zero_masked_rows(int dtype, void* data, const unsigned char* mask, long long rows, int C, cudaStream_t st)
{
    if (rows == 0 || C == 0) return cudaSuccess;
    const int esz = dtype == kF32 ? 4 : (dtype == kBF16 || dtype == kF16 ? 2 : 0);
    if (esz == 0 || (C * esz) % 16 != 0) return cudaErrorInvalidValue;
    const long long want = (rows + 255) / 256;
    const int grid = (int)(want < 148 * 8 ? want : 148 * 8);
    if (esz == 4) zero_masked_rows_kernel<float><<<grid, 256, 0, st>>>((float*)data, mask, rows, C);
    else zero_masked_rows_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((__nv_bfloat16*)data, mask, rows, C);
    return cudaGetLastError();
}

// Standalone dropout, y = x * mask * scale (x == y allowed): thread = one group of 8 elements = one Philox call, 16-byte
// accesses when both pointers are 16-byte aligned (`vec`), element by element for the tail group.
template <typename T>
__global__ void __launch_bounds__(256)
dropout_kernel(const T* x, T* y, long long n, const unsigned long long* __restrict__ key_ptr, unsigned thresh,
               float scale, int vec)
{
    constexpr int V = Vec16<T>::n;
    const unsigned long long key = *key_ptr;
    const long long groups = (n + 7) >> 3;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
        const unsigned bits = dropout_keep8((unsigned long long)g, key, thresh);
        const long long e0 = g << 3;
        if (vec && e0 + 8 <= n) {
#pragma unroll
            for (int h = 0; h < 8 / V; ++h) {
                float f[V];
                load16<T>(x + e0 + h * V, f);
#pragma unroll
                for (int e = 0; e < V; ++e) f[e] *= drop_mul(bits, h * V + e, scale);
                store16<T>(y + e0 + h * V, f);
            }
        } else {
            for (int i = 0; i < 8 && e0 + i < n; ++i)
                y[e0 + i] = from_f32<T>(to_f32<T>(x[e0 + i]) * drop_mul(bits, i, scale));
        }
    }
}

// Backward of dropout(relu(.)) from its saved output: dx = out > 0 ? g * scale : 0.  A dropped element and a non-positive
// pre-activation both have out == 0, so neither the mask nor the key is needed.
template <typename T>
__global__ void __launch_bounds__(256)
relu_dropout_grad_kernel(const T* __restrict__ g, const T* __restrict__ out, T* dx, long long n, float scale, int vec)
{
    constexpr int V = Vec16<T>::n;
    const long long chunks = (n + V - 1) / V;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < chunks; c += stride) {
        const long long e0 = c * V;
        if (vec && e0 + V <= n) {
            float fg[V], fo[V];
            load16_stream<T>(g + e0, fg);
            load16_stream<T>(out + e0, fo);
#pragma unroll
            for (int e = 0; e < V; ++e) fg[e] = fo[e] > 0.f ? fg[e] * scale : 0.f;
            store16<T>(dx + e0, fg);
        } else {
            for (long long e = e0; e < n && e < e0 + V; ++e)
                dx[e] = from_f32<T>(to_f32<T>(out[e]) > 0.f ? to_f32<T>(g[e]) * scale : 0.f);
        }
    }
}

static int elementwise_grid(long long items)
{
    const long long want = (items + 255) / 256;
    return (int)(want < 148 * 16 ? (want > 0 ? want : 1) : 148 * 16);
}

cudaError_t dropout(int dtype, const void* x, void* y, long long n, const unsigned long long* key, DropoutRule rule,
                    cudaStream_t st)
{
    if (n < 0 || key == nullptr) return cudaErrorInvalidValue;
    if (n == 0) return cudaSuccess;
    const int vec = (reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) % 16 == 0;
    const int grid = elementwise_grid((n + 7) / 8);
    switch (dtype) {
        case kF32:
            dropout_kernel<float><<<grid, 256, 0, st>>>((const float*)x, (float*)y, n, key, rule.thresh, rule.scale, vec);
            break;
        case kBF16:
            dropout_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, n, key,
                                                                 rule.thresh, rule.scale, vec);
            break;
        case kF16:
            dropout_kernel<__half><<<grid, 256, 0, st>>>((const __half*)x, (__half*)y, n, key, rule.thresh, rule.scale, vec);
            break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t relu_dropout_grad(int dtype, const void* g, const void* out, void* dx, long long n, float scale,
                              cudaStream_t st)
{
    if (n < 0) return cudaErrorInvalidValue;
    if (n == 0) return cudaSuccess;
    const int vec = (reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(dx)) %
                    16 == 0;
    switch (dtype) {
        case kF32:
            relu_dropout_grad_kernel<float><<<elementwise_grid((n + 3) / 4), 256, 0, st>>>(
                (const float*)g, (const float*)out, (float*)dx, n, scale, vec);
            break;
        case kBF16:
            relu_dropout_grad_kernel<__nv_bfloat16><<<elementwise_grid((n + 7) / 8), 256, 0, st>>>(
                (const __nv_bfloat16*)g, (const __nv_bfloat16*)out, (__nv_bfloat16*)dx, n, scale, vec);
            break;
        case kF16:
            relu_dropout_grad_kernel<__half><<<elementwise_grid((n + 7) / 8), 256, 0, st>>>(
                (const __half*)g, (const __half*)out, (__half*)dx, n, scale, vec);
            break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

}  // namespace msda
