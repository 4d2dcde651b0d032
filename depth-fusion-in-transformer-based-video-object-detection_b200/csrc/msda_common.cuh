// Shared device helpers for the sm_100a multi-scale deformable attention kernels.
//
// Data layout in HBM (the reference's, unchanged so the op stays a drop-in):
//   value        [N, S, M, D]        pixel-major, one pixel record = M*D contiguous elements
//   sampling_loc [N, Lq, M, L, P, 2] (x, y) normalised to [0,1]
//   attn_weight  [N, Lq, M, L, P]
//   output       [N, Lq, M, D]
//   spatial_shapes [L,2] (H,W) int64 and level_start_index [L] int64, both ON DEVICE
// A "pair" is one (n, q, m) triple; pairs are numbered flat, pair = (n*Lq + q)*M + m, so that
// the loc / attn / output blocks of consecutive pairs are contiguous in memory.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace msda {

constexpr int kMaxLevelsFast = 32;   // level metadata staged in shared memory by the fast kernels
constexpr int kChunk = 16;           // samples (level x point) processed per pass by the fast kernels

// ----------------------------------------------------------------------------------------
// dtype traits: storage type of value/output, arithmetic type, and the 16-byte vector shape
// ----------------------------------------------------------------------------------------
template <typename VT> struct Traits;
template <> struct Traits<float>         { using acc_t = float;  using loc_t = float;  static constexpr int kEpl = 4; };
template <> struct Traits<double>        { using acc_t = double; using loc_t = double; static constexpr int kEpl = 2; };
template <> struct Traits<__nv_bfloat16> { using acc_t = float;  using loc_t = float;  static constexpr int kEpl = 8; };
template <> struct Traits<__half>        { using acc_t = float;  using loc_t = float;  static constexpr int kEpl = 8; };

template <typename VT> __device__ __forceinline__ float to_f32(VT v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

template <typename VT> __device__ __forceinline__ VT from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

// ----------------------------------------------------------------------------------------
// 128-bit global accesses.  Value rows are re-read by neighbouring queries, so they go through
// the read-only path and are allowed to allocate in L1; loc/attn/grad streams are read once.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_v4(const void* p)
{
    uint4 r;
    asm("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ldg_stream_v4(const void* p)
{
    uint4 r;
    asm("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_v4(void* p, uint4 v)
{
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ float ldg_stream_f32(const float* p)
{
    float r;
    asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ float2 ldg_stream_f32x2(const float* p)
{
    float2 r;
    asm("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
// one 16-byte vector reduction into global memory (sm_90+): REDG.E.ADD.F32x4
__device__ __forceinline__ void red_add_f32x4(float* p, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" :: "l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__device__ __forceinline__ uint2 ldg_v2(const void* p)
{
    uint2 r;
    asm("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg_stream_v2(const void* p)
{
    uint2 r;
    asm("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}

// unpack one 16-byte vector of VT into kEpl floats
template <typename VT> __device__ __forceinline__ void unpack(const uint4& raw, float* f);
template <> __device__ __forceinline__ void unpack<float>(const uint4& raw, float* f)
{
    f[0] = __uint_as_float(raw.x); f[1] = __uint_as_float(raw.y);
    f[2] = __uint_as_float(raw.z); f[3] = __uint_as_float(raw.w);
}
template <> __device__ __forceinline__ void unpack<__nv_bfloat16>(const uint4& raw, float* f)
{
    // bf16 -> f32 is a 16-bit shift
    f[0] = __uint_as_float(raw.x << 16); f[1] = __uint_as_float(raw.x & 0xffff0000u);
    f[2] = __uint_as_float(raw.y << 16); f[3] = __uint_as_float(raw.y & 0xffff0000u);
    f[4] = __uint_as_float(raw.z << 16); f[5] = __uint_as_float(raw.z & 0xffff0000u);
    f[6] = __uint_as_float(raw.w << 16); f[7] = __uint_as_float(raw.w & 0xffff0000u);
}
template <> __device__ __forceinline__ void unpack<__half>(const uint4& raw, float* f)
{
    const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 t = __half22float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}
template <typename VT> __device__ __forceinline__ uint4 pack(const float* f);
template <> __device__ __forceinline__ uint4 pack<float>(const float* f)
{
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
}
template <> __device__ __forceinline__ uint4 pack<__nv_bfloat16>(const float* f)
{
    uint4 r;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    return r;
}
template <> __device__ __forceinline__ uint4 pack<__half>(const float* f)
{
    uint4 r;
    __half2* h = reinterpret_cast<__half2*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
    return r;
}

// A lane's channel slice: EPL consecutive elements of VT, moved with ONE load of EPL*sizeof(VT)
// bytes (16 B, or 8 B for the 16-bit backward where 4 channels per lane keep the fp32 vector
// reductions row-complete).  `zero` slices stand in for out-of-map corners.
template <typename VT, int EPL> struct Slice;
template <typename VT> struct Slice<VT, 16 / (int)sizeof(VT)> {
    using raw_t = uint4;
    static __device__ __forceinline__ raw_t zero() { return make_uint4(0u, 0u, 0u, 0u); }
    static __device__ __forceinline__ raw_t load(const VT* p) { return ldg_v4(p); }
    static __device__ __forceinline__ raw_t load_stream(const VT* p) { return ldg_stream_v4(p); }
    static __device__ __forceinline__ void unpack(const raw_t& r, float* f) { msda::unpack<VT>(r, f); }
};
template <> struct Slice<__nv_bfloat16, 4> {
    using raw_t = uint2;
    static __device__ __forceinline__ raw_t zero() { return make_uint2(0u, 0u); }
    static __device__ __forceinline__ raw_t load(const __nv_bfloat16* p) { return ldg_v2(p); }
    static __device__ __forceinline__ raw_t load_stream(const __nv_bfloat16* p) { return ldg_stream_v2(p); }
    static __device__ __forceinline__ void unpack(const raw_t& r, float* f)
    {
        f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
        f[2] = __uint_as_float(r.y << 16); f[3] = __uint_as_float(r.y & 0xffff0000u);
    }
};
template <> struct Slice<__half, 4> {
    using raw_t = uint2;
    static __device__ __forceinline__ raw_t zero() { return make_uint2(0u, 0u); }
    static __device__ __forceinline__ raw_t load(const __half* p) { return ldg_v2(p); }
    static __device__ __forceinline__ raw_t load_stream(const __half* p) { return ldg_stream_v2(p); }
    static __device__ __forceinline__ void unpack(const raw_t& r, float* f)
    {
        const __half2* h = reinterpret_cast<const __half2*>(&r);
        const float2 a = __half22float2(h[0]), b = __half22float2(h[1]);
        f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y;
    }
};

// ----------------------------------------------------------------------------------------
// Bilinear footprint of one sample (the arithmetic of ms_deform_attn_im2col_bilinear,
// reference cuda/ms_deform_im2col_cuda.cuh:33-84, with the caller's range test :288 folded in).
// ----------------------------------------------------------------------------------------
struct Footprint {
    int   pix00;     // level_start + y0*W + x0 (pixel index inside one batch element; may be
                     // out of range when a corner is invalid -- never dereferenced then)
    int   rowstep;   // W
    unsigned ok;     // bit0..3: corner (y0,x0) (y0,x1) (y1,x0) (y1,x1) lies inside the map
    float lw, lh;    // fractional parts
};

template <typename T>
__device__ __forceinline__ Footprint footprint(T loc_x, T loc_y, int H, int W, int start)
{
    // pixel convention of align_corners=False: x = loc_x * W - 0.5   (cuh:285-286)
    const T w_im = loc_x * (T)W - (T)0.5;
    const T h_im = loc_y * (T)H - (T)0.5;
    Footprint f;
    const bool inside = (h_im > (T)-1) && (w_im > (T)-1) && (h_im < (T)H) && (w_im < (T)W);
    const T hf = floor(h_im), wf = floor(w_im);
    const int y0 = (int)hf, x0 = (int)wf;
    f.lh = (float)(h_im - hf);
    f.lw = (float)(w_im - wf);
    const bool y0ok = y0 >= 0, y1ok = y0 + 1 <= H - 1, x0ok = x0 >= 0, x1ok = x0 + 1 <= W - 1;
    f.ok = inside ? ((y0ok && x0ok ? 1u : 0u) | (y0ok && x1ok ? 2u : 0u) |
                     (y1ok && x0ok ? 4u : 0u) | (y1ok && x1ok ? 8u : 0u)) : 0u;
    f.pix00 = start + y0 * W + x0;
    f.rowstep = W;
    return f;
}

// ----------------------------------------------------------------------------------------
// Where a pair's samples come from.  Plain: materialised sampling_loc / attn_weight (the drop-in
// op).  Fused: raw projection outputs + reference points.
// ----------------------------------------------------------------------------------------
struct SampleSrc {
    const void* loc;          // plain: sampling_loc base ; fused: offsets base
    const void* attn;         // plain: attn_weight base  ; fused: logits base
    const float* ref;         // fused only
    long long loc_stride;     // fused: elements between consecutive queries
    long long attn_stride;
    int ref_dim;              // fused: 2 or 4
};

template <typename RT> __device__ __forceinline__ float2 load_raw2(const RT* p);
template <> __device__ __forceinline__ float2 load_raw2<float>(const float* p) { return ldg_stream_f32x2(p); }
template <> __device__ __forceinline__ float2 load_raw2<__nv_bfloat16>(const __nv_bfloat16* p)
{
    unsigned r;
    asm("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u));
}
template <> __device__ __forceinline__ float2 load_raw2<__half>(const __half* p)
{
    unsigned r;
    asm("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return __half22float2(*reinterpret_cast<const __half2*>(&r));
}
template <typename RT> __device__ __forceinline__ float load_raw1(const RT* p) { return to_f32<RT>(*p); }
template <> __device__ __forceinline__ float load_raw1<float>(const float* p) { return ldg_stream_f32(p); }

template <typename RT> __device__ __forceinline__ void store_raw2(RT* p, float a, float b);
template <> __device__ __forceinline__ void store_raw2<float>(float* p, float a, float b)
{
    *reinterpret_cast<float2*>(p) = make_float2(a, b);
}
template <> __device__ __forceinline__ void store_raw2<__nv_bfloat16>(__nv_bfloat16* p, float a, float b)
{
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}
template <> __device__ __forceinline__ void store_raw2<__half>(__half* p, float a, float b)
{
    *reinterpret_cast<__half2*>(p) = __floats2half2_rn(a, b);
}

template <int G> __device__ __forceinline__ float group_max(float v)
{
#pragma unroll
    for (int off = G / 2; off >= 1; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}
template <int G> __device__ __forceinline__ float group_sum(float v)
{
#pragma unroll
    for (int off = G / 2; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// Sampling location of one sample from its raw offset and reference point
// (reference modules/ms_deform_attn.py:102-110).
// The divisions by W, H and n_points are multiplications by reciprocals the caller computes once per CTA (an IEEE float
// division is ~12 instructions with a slow-path call; phase 1 of the 16-bit fused kernels ran 12 of them per lane): the
// location moves by at most one ulp.
__device__ __forceinline__ float2 fused_location(float2 off, const float* __restrict__ ref_l, int ref_dim,
                                                 float inv_h, float inv_w, float half_inv_p)
{
    if (ref_dim == 2) {
        const float2 r = *reinterpret_cast<const float2*>(ref_l);
        return make_float2(fmaf(off.x, inv_w, r.x), fmaf(off.y, inv_h, r.y));
    }
    const float4 r = *reinterpret_cast<const float4*>(ref_l);
    return make_float2(fmaf(off.x * half_inv_p, r.z, r.x), fmaf(off.y * half_inv_p, r.w, r.y));
}

// exact s / P for 0 <= s < 65536 / P  (magic = ceil(65536 / P), computed on the host)
__device__ __forceinline__ int div_by_points(int s, int magic) { return (s * magic) >> 16; }

// Packed fp32 arithmetic (Blackwell: fma / mul / sub .f32x2 -> FFMA2 / FMUL2 / FADD2).  nvcc emits these only from inline
// PTX; each half is an ordinary IEEE operation.
struct alignas(8) F2 { float x, y; };
__device__ __forceinline__ unsigned long long f2_bits(F2 a) { return *reinterpret_cast<unsigned long long*>(&a); }
__device__ __forceinline__ F2 f2_from(unsigned long long a) { return *reinterpret_cast<F2*>(&a); }
__device__ __forceinline__ F2 f2_dup(float a) { F2 r; r.x = a; r.y = a; return r; }
__device__ __forceinline__ F2 fma2(F2 a, F2 b, F2 c)
{
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)), "l"(f2_bits(c)));
    return f2_from(d);
}
__device__ __forceinline__ F2 mul2(F2 a, F2 b)
{
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return f2_from(d);
}
__device__ __forceinline__ F2 sub2(F2 a, F2 b)
{
    unsigned long long d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return f2_from(d);
}


// An address the compiler cannot re-derive from the kernel parameters (it would otherwise rebuild base + offset with
// 64-bit shifts and carries at every use instead of keeping the pointer in a register pair).
__device__ __forceinline__ unsigned long long opaque_addr(const void* p)
{
    unsigned long long a = reinterpret_cast<unsigned long long>(p);
    asm volatile("" : "+l"(a));
    return a;
}
// red.global.add.v4.f32 of coef * (g01, g23), issued only when coef != 0.  One asm block: the two packed products stay
// outside the predicate, so ptxas emits a predicated REDG instead of a branch around a multiply-and-reduce block.
__device__ __forceinline__ void red_scaled_f32x4_if(float* p, float coef, F2 g01, F2 g23)
{
    asm volatile("{\n\t.reg .pred q;\n\t.reg .b64 c2, lo, hi;\n\t.reg .f32 a, b, c, d;\n\t"
                 "mov.b64 c2, {%1, %1};\n\t"
                 "mul.rn.f32x2 lo, c2, %2;\n\t"
                 "mul.rn.f32x2 hi, c2, %3;\n\t"
                 "mov.b64 {a, b}, lo;\n\t"
                 "mov.b64 {c, d}, hi;\n\t"
                 "setp.neu.f32 q, %1, 0f00000000;\n\t"
                 "@q red.global.add.v4.f32 [%0], {a, b, c, d};\n\t}"
                 :: "l"(p), "f"(coef), "l"(f2_bits(g01)), "l"(f2_bits(g23)) : "memory");
}

// ----------------------------------------------------------------------------------------
// Deterministic backward (C ABI *_deterministic, csrc/deterministic.cu, DESIGN.md section 3.15): every contribution
// to a gradient element is rounded to an integer multiple of 2^-shift and the integers are summed with 64-bit
// reductions.  Integer addition is associative, so the sum does not depend on the order the hardware runs them in.
// The pre-pass writes this header at the start of the caller's scratch; the accumulation kernels read the scale there.
// ----------------------------------------------------------------------------------------
struct DetHeader {
    unsigned long long gmax;   // max |grad_output| as the bits of a double (NaN above +Inf: see det_abs_bits)
    unsigned long long amax;   // max over pairs of sum |attention|, same encoding
    double scale, inv_scale;   // 2^shift, 2^-shift
    float scale_f;             // 2^shift for fp32 contributions
    int shift;
    int poison;                // non-finite bound: the finishing kernel writes NaN everywhere
};
constexpr long long kDetHeaderBytes = 256;   // the int64 accumulators start here

__device__ __forceinline__ void red_fixed(long long* p, float v, float scale)
{
    // v * scale is exact (a power of two); |v * scale| < 2^62 by the choice of shift, so the conversion cannot saturate
    atomicAdd(reinterpret_cast<unsigned long long*>(p), (unsigned long long)__float2ll_rn(v * scale));
}
__device__ __forceinline__ void red_fixed(long long* p, double v, double scale)
{
    atomicAdd(reinterpret_cast<unsigned long long*>(p), (unsigned long long)__double2ll_rn(v * scale));
}

// ----------------------------------------------------------------------------------------
// Dropout mask (DESIGN.md section 3.16).  Element e of a call's contiguous [rows, C] output draws the 16-bit number
//     u(e) = (r[(e & 7) >> 1] >> (16 * (e & 1))) & 0xFFFF,   r = Philox4x32-10(counter (lo32(e >> 3), hi32(e >> 3), 0, 0),
//                                                                               key (lo32(key), hi32(key)))
// and is kept iff u(e) >= thresh (dropout_rule in msda_launch.h).  One Philox call covers the 8 elements of a group.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, unsigned k0, unsigned k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r > 0) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    }
    return c;
}

// keep bits of the elements 8 * group + i, i = 0..7: bit i set = element kept
__device__ __forceinline__ unsigned dropout_keep8(unsigned long long group, unsigned long long key, unsigned thresh)
{
    const uint4 r = philox4x32_10(make_uint4((unsigned)group, (unsigned)(group >> 32), 0u, 0u), (unsigned)key,
                                  (unsigned)(key >> 32));
    const unsigned w[4] = {r.x, r.y, r.z, r.w};
    unsigned m = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        m |= ((w[i] & 0xFFFFu) >= thresh ? 1u : 0u) << (2 * i) | ((w[i] >> 16) >= thresh ? 1u : 0u) << (2 * i + 1);
    return m;
}

}  // namespace msda
