// Pre-pass and finishing kernels of the deterministic backward (C ABI *_deterministic, DESIGN.md section 3.15).
//
// The accumulating kernels (msda_backward.cu, roi_align.cu with DET = true) add every contribution c to a gradient
// element as the int64 rint(c * 2^shift).  This file computes `shift` on the device, per launch, from a bound B on
// the magnitude of every gradient element, and turns the int64 sums back into the output dtype.
//
// Why no sum can overflow.  Let B >= sum_i |c_i| for every element (the exact contributions; each op proves its own
// B from its inputs).  shift = 61 - e where B = m 2^e, m in [0.5, 1) (frexp), so 2^shift B <= 2^61.  Each computed
// contribution carries at most a few fp32 roundings (relative 2^-22 together) and its conversion adds at most 1/2, so
// an element with K contributions sums to at most 2^61 (1 + 2^-22) + K / 2 in magnitude, and B itself is computed in
// double from fp32-exact maxima (relative error ~2^-50).  K is below 2^40 for any tensor that fits a GPU, so the sum
// stays below 2^61 + 2^40 < 2^63: no partial sum wraps, in any order.  The shift is clamped to 126 (2^shift must be
// an fp32 normal for the fp32 contributions) and 1000 for fp64; a contribution that small then rounds to zero, which
// is the quantum the format has.
#include <float.h>
#include "msda_common.cuh"
#include "msda_launch.h"

namespace msda {
namespace {

// |x| as the bits of a double: integer order == numeric order for non-negative values, +Inf above every finite value,
// NaN (canonicalised) above +Inf.  An integer max is exact, so the result does not depend on the order of the maxima.
__device__ __forceinline__ unsigned long long det_abs_bits(double x)
{
    return x != x ? 0x7fffffffffffffffull : (unsigned long long)__double_as_longlong(fabs(x));
}

template <typename T> __device__ __forceinline__ double to_f64(T v) { return (double)to_f32<T>(v); }
template <> __device__ __forceinline__ double to_f64<double>(double v) { return v; }

__device__ __forceinline__ void block_max_to(unsigned long long v, unsigned long long* slot)
{
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, off);
        v = o > v ? o : v;
    }
    if ((threadIdx.x & 31) == 0 && v != 0) atomicMax(slot, v);
}

// max |x[r, c]| over rows x cols elements with row stride ld
template <typename T>
__global__ void __launch_bounds__(256)
det_absmax_kernel(const T* __restrict__ x, long long rows, int cols, long long ld, unsigned long long* slot)
{
    const long long total = rows * cols;
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned long long m = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long r = ld == cols ? 0 : i / cols;        // dense: no 64-bit division per element
        const unsigned long long b = det_abs_bits(to_f64<T>(x[i + r * (ld - cols)]));
        m = b > m ? b : m;
    }
    block_max_to(m, slot);
}

// max over pairs of sum_s |attn[pair, s]| (the pair's samples in a fixed order, in double)
template <typename T>
__global__ void __launch_bounds__(256)
det_attn_sum_kernel(const T* __restrict__ attn, long long pairs, int LP, unsigned long long* slot)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned long long m = 0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < pairs; p += stride) {
        double s = 0.0;
        for (int j = 0; j < LP; ++j) s += fabs((double)attn[p * LP + j]);
        const unsigned long long b = det_abs_bits(s);
        m = b > m ? b : m;
    }
    block_max_to(m, slot);
}

// B = count * gmax * amax; amax_mode 1: the attention factor is 1 and amax only tells whether it is finite
__global__ void det_finalize_kernel(DetHeader* h, double count, int amax_mode, int max_shift)
{
    const double g = __longlong_as_double((long long)h->gmax);
    double a = __longlong_as_double((long long)h->amax);
    if (amax_mode == 1) a = a <= DBL_MAX ? 1.0 : a;
    const double B = count * g * a;
    int shift = 0;
    h->poison = 0;
    if (!(B <= DBL_MAX)) {
        h->poison = 1;                 // Inf or NaN somewhere in the inputs of the bound
    } else if (B > 0.0) {
        int e;
        frexp(B, &e);
        shift = 61 - e;
        shift = shift > max_shift ? max_shift : shift;
    }
    h->shift = shift;
    h->scale = ldexp(1.0, shift);
    h->inv_scale = ldexp(1.0, -shift);
    h->scale_f = (float)h->scale;
}

template <typename VT> __device__ __forceinline__ VT from_f64(double v) { return from_f32<VT>((float)v); }
template <> __device__ __forceinline__ double from_f64<double>(double v) { return v; }

template <typename VT>
__global__ void __launch_bounds__(256)
det_finish_kernel(const long long* __restrict__ acc, VT* __restrict__ out, long long count, const DetHeader* h)
{
    const double inv = h->inv_scale;
    const bool poison = h->poison != 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        out[i] = from_f64<VT>(poison ? __longlong_as_double(0x7ff8000000000000ll) : (double)acc[i] * inv);
}

// grad_ref[nq, l, r] = sum over heads m (in order) of part[nq, l, m, r]
__global__ void __launch_bounds__(256)
det_fold_ref_kernel(const float* __restrict__ part, float* __restrict__ grad_ref, long long rows, int M, int R)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < rows * R; i += stride) {
        const long long row = i / R;
        const int r = (int)(i - row * R);
        float s = 0.f;
        for (int m = 0; m < M; ++m) s += part[(row * M + m) * R + r];
        grad_ref[i] = s;
    }
}

unsigned grid_for(long long n)
{
    long long blocks = (n + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 148 * 16) blocks = 148 * 16;
    return (unsigned)blocks;
}

}  // namespace

long long det_scratch_bytes(long long grad_elements, long long ref_partial_floats)
{
    if (grad_elements < 0 || ref_partial_floats < 0) return -1;
    const long long acc = (grad_elements * 8 + 255) / 256 * 256;
    return kDetHeaderBytes + acc + ref_partial_floats * 4;
}

float* det_ref_partials(void* scratch, long long grad_elements)
{
    return reinterpret_cast<float*>(static_cast<char*>(scratch) + kDetHeaderBytes + (grad_elements * 8 + 255) / 256 * 256);
}

cudaError_t det_begin(void* scratch, long long grad_elements, cudaStream_t stream)
{
    return cudaMemsetAsync(scratch, 0, (size_t)(kDetHeaderBytes + grad_elements * 8), stream);
}

cudaError_t det_absmax(int dtype, const void* x, long long rows, int cols, long long ld, unsigned long long* slot,
                       cudaStream_t stream)
{
    const long long n = rows * cols;
    if (n <= 0) return cudaSuccess;
    const unsigned g = grid_for(n);
    switch (dtype) {
        case kF32:  det_absmax_kernel<float><<<g, 256, 0, stream>>>((const float*)x, rows, cols, ld, slot); break;
        case kF64:  det_absmax_kernel<double><<<g, 256, 0, stream>>>((const double*)x, rows, cols, ld, slot); break;
        case kBF16: det_absmax_kernel<__nv_bfloat16><<<g, 256, 0, stream>>>((const __nv_bfloat16*)x, rows, cols, ld, slot); break;
        case kF16:  det_absmax_kernel<__half><<<g, 256, 0, stream>>>((const __half*)x, rows, cols, ld, slot); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t det_attn_sum_max(bool f64, const void* attn, long long pairs, int LP, unsigned long long* slot,
                             cudaStream_t stream)
{
    if (pairs <= 0) return cudaSuccess;
    if (f64) det_attn_sum_kernel<double><<<grid_for(pairs), 256, 0, stream>>>((const double*)attn, pairs, LP, slot);
    else det_attn_sum_kernel<float><<<grid_for(pairs), 256, 0, stream>>>((const float*)attn, pairs, LP, slot);
    return cudaGetLastError();
}

cudaError_t det_finalize(DetHeader* h, double count, int amax_mode, bool f64, cudaStream_t stream)
{
    det_finalize_kernel<<<1, 1, 0, stream>>>(h, count, amax_mode, f64 ? 1000 : 126);
    return cudaGetLastError();
}

cudaError_t det_finish(int dtype, const long long* acc, void* out, long long count, const DetHeader* h,
                       cudaStream_t stream)
{
    if (count <= 0) return cudaSuccess;
    const unsigned g = grid_for(count);
    switch (dtype) {
        case kF32:  det_finish_kernel<float><<<g, 256, 0, stream>>>(acc, (float*)out, count, h); break;
        case kF64:  det_finish_kernel<double><<<g, 256, 0, stream>>>(acc, (double*)out, count, h); break;
        case kBF16: det_finish_kernel<__nv_bfloat16><<<g, 256, 0, stream>>>(acc, (__nv_bfloat16*)out, count, h); break;
        case kF16:  det_finish_kernel<__half><<<g, 256, 0, stream>>>(acc, (__half*)out, count, h); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t det_fold_ref(const float* part, float* grad_ref, long long rows, int M, int R, cudaStream_t stream)
{
    if (rows * R <= 0) return cudaSuccess;
    det_fold_ref_kernel<<<grid_for(rows * R), 256, 0, stream>>>(part, grad_ref, rows, M, R);
    return cudaGetLastError();
}

}  // namespace msda
