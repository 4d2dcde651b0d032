// RoIAlign for the TransVOD++ temporal query stage (SURVEY.md 8f rank 3): the reference pools a 7x7x256 patch
// per decoder box out of the encoder memory with mmcv.ops.RoIAlign(output_size=7, sampling_ratio=2,
// spatial_scale=1/32, pool_mode='avg', aligned=True)
//     /root/reference/models/deformable_transformer_multi_plusplus.py:129-132 (construction), :499, :514 (calls).
// mmcv-full 1.7.0 is a third-party dependency that is not under /root/reference; the arithmetic restated here
// is its published algorithm (mmcv/ops/csrc/common/cuda/roi_align_cuda_kernel.cuh, the Detectron RoIAlign that
// torchvision.ops.roi_align also implements -- the tests pin this kernel against both an in-repo numpy
// restatement and torchvision's CPU implementation).
//
// It is the same bilinear gather as the deformable attention, so it gets the same treatment: the feature map
// is read TOKEN-MAJOR ([N, H*W, C], what the encoder produces -- the reference first permutes the memory to
// NCHW and the head then permutes the pooled patch back, :498, head.py:66) and the pooled patch is written
// [K, PH*PW, C]; one warp per output bin, lanes across the channels (coalesced rows), fp32 accumulation.
#include "msda_common.cuh"
#include "msda_launch.h"

namespace msda {
namespace {

template <typename CT> struct BinSample {
    int p1, p2, p3, p4;        // pixel indices y*W + x of the four corners
    CT w1, w2, w3, w4;         // bilinear weights; all zero for a sample outside the map
};

// mmcv bilinear_interpolate / bilinear_interpolate_gradient (roi_align_cuda_kernel.cuh): samples more than one
// pixel outside contribute nothing, coordinates are clamped into the map, the last row / column repeats.
template <typename CT>
__device__ __forceinline__ BinSample<CT> bin_sample(CT y, CT x, int H, int W)
{
    BinSample<CT> s;
    if (y < (CT)-1 || y > (CT)H || x < (CT)-1 || x > (CT)W) {
        s.p1 = s.p2 = s.p3 = s.p4 = 0;
        s.w1 = s.w2 = s.w3 = s.w4 = (CT)0;
        return s;
    }
    if (y <= (CT)0) y = (CT)0;
    if (x <= (CT)0) x = (CT)0;
    int y_low = (int)y, x_low = (int)x, y_high, x_high;
    if (y_low >= H - 1) { y_high = y_low = H - 1; y = (CT)y_low; } else y_high = y_low + 1;
    if (x_low >= W - 1) { x_high = x_low = W - 1; x = (CT)x_low; } else x_high = x_low + 1;
    const CT ly = y - (CT)y_low, lx = x - (CT)x_low, hy = (CT)1 - ly, hx = (CT)1 - lx;
    s.p1 = y_low * W + x_low;  s.p2 = y_low * W + x_high;
    s.p3 = y_high * W + x_low; s.p4 = y_high * W + x_high;
    s.w1 = hy * hx; s.w2 = hy * lx; s.w3 = ly * hx; s.w4 = ly * lx;
    return s;
}

template <typename CT> struct RoiGeom {
    int batch, grid_h, grid_w;
    CT y0, x0, bin_h, bin_w, inv_count;
};

template <typename CT>
__device__ __forceinline__ RoiGeom<CT> roi_geom(const CT* __restrict__ roi, CT scale, int sampling_ratio, int aligned,
                                                int PH, int PW)
{
    RoiGeom<CT> g;
    g.batch = (int)roi[0];
    const CT off = aligned ? (CT)0.5 : (CT)0;
    g.x0 = roi[1] * scale - off;
    g.y0 = roi[2] * scale - off;
    CT rw = roi[3] * scale - off - g.x0, rh = roi[4] * scale - off - g.y0;
    if (!aligned) { rw = rw > (CT)1 ? rw : (CT)1; rh = rh > (CT)1 ? rh : (CT)1; }
    g.bin_h = rh / (CT)PH;
    g.bin_w = rw / (CT)PW;
    g.grid_h = sampling_ratio > 0 ? sampling_ratio : (int)ceil(rh / (CT)PH);
    g.grid_w = sampling_ratio > 0 ? sampling_ratio : (int)ceil(rw / (CT)PW);
    const int count = g.grid_h * g.grid_w;
    g.inv_count = (CT)1 / (CT)(count > 1 ? count : 1);
    return g;
}

template <typename T, typename CT> __device__ __forceinline__ CT load_as(const T* p) { return (CT)to_f32<T>(*p); }
template <> __device__ __forceinline__ double load_as<double, double>(const double* p) { return *p; }
template <typename T, typename CT> __device__ __forceinline__ T store_as(CT v) { return from_f32<T>((float)v); }
template <> __device__ __forceinline__ double store_as<double, double>(double v) { return v; }

// scalar path: any channel count, any dtype (the fp64 tests run here)
template <typename T, typename CT>
__global__ void __launch_bounds__(256)
roi_align_fwd_kernel(const T* __restrict__ feat, const CT* __restrict__ rois, T* __restrict__ out, int N, int H, int W,
                     int C, long long bins, int PH, int PW, CT scale, int sampling_ratio, int aligned)
{
    const long long bin = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (bin >= bins) return;
    const int pw = (int)(bin % PW), ph = (int)((bin / PW) % PH);
    const long long k = bin / ((long long)PW * PH);
    const RoiGeom<CT> g = roi_geom<CT>(rois + 5 * k, scale, sampling_ratio, aligned, PH, PW);
    const bool batch_ok = g.batch >= 0 && g.batch < N;
    const T* map = feat + (long long)(batch_ok ? g.batch : 0) * H * W * C;
    for (int c = lane; c < C; c += 32) {
        CT acc = (CT)0;
        for (int iy = 0; iy < g.grid_h; ++iy) {
            const CT y = g.y0 + (CT)ph * g.bin_h + ((CT)iy + (CT)0.5) * g.bin_h / (CT)g.grid_h;
            for (int ix = 0; ix < g.grid_w; ++ix) {
                const CT x = g.x0 + (CT)pw * g.bin_w + ((CT)ix + (CT)0.5) * g.bin_w / (CT)g.grid_w;
                const BinSample<CT> s = bin_sample<CT>(y, x, H, W);
                if (!batch_ok) continue;
                acc += s.w1 * load_as<T, CT>(map + (long long)s.p1 * C + c) + s.w2 * load_as<T, CT>(map + (long long)s.p2 * C + c) +
                       s.w3 * load_as<T, CT>(map + (long long)s.p3 * C + c) + s.w4 * load_as<T, CT>(map + (long long)s.p4 * C + c);
            }
        }
        out[bin * C + c] = store_as<T, CT>(acc * g.inv_count);
    }
}

// vector path (fp32 / bf16 / fp16, C a multiple of the 16-byte vector): one warp per (box, bin ROW) walks the PW bins
// of that row, so the box geometry and the y terms of the row's samples are computed once per PW bins instead of once
// per bin; every corner row is fetched with 16-byte loads, the GRID x GRID samples of a bin (16 loads for the
// reference's sampling_ratio 2) are unrolled so they are all in flight together.  GRID = 0: run-time sampling grid.
template <typename CT> struct AxisTerm { int low, high; CT l, h; bool valid; };

template <typename CT>
__device__ __forceinline__ AxisTerm<CT> axis_term(CT v, int size)       // one coordinate of mmcv's bilinear_interpolate
{
    AxisTerm<CT> t;
    t.valid = !(v < (CT)-1 || v > (CT)size);
    if (v <= (CT)0) v = (CT)0;
    t.low = (int)v;
    if (t.low >= size - 1) { t.high = t.low = size - 1; v = (CT)t.low; } else t.high = t.low + 1;
    t.l = v - (CT)t.low;
    t.h = (CT)1 - t.l;
    return t;
}

template <typename T, int GRID>
__global__ void __launch_bounds__(256)
roi_align_fwd_vec_kernel(const T* __restrict__ feat, const float* __restrict__ rois, T* __restrict__ out, int N, int H,
                         int W, int C, long long bin_rows, int PH, int PW, float scale, int sampling_ratio, int aligned)
{
    constexpr int V = 16 / (int)sizeof(T);
    const long long brow = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (brow >= bin_rows) return;
    const int ph = (int)(brow % PH);
    const long long k = brow / PH;
    const RoiGeom<float> g = roi_geom<float>(rois + 5 * k, scale, sampling_ratio, aligned, PH, PW);
    const bool batch_ok = g.batch >= 0 && g.batch < N;
    const T* map = feat + (long long)(batch_ok ? g.batch : 0) * H * W * C;
    const int gh = GRID > 0 ? GRID : g.grid_h, gw = GRID > 0 ? GRID : g.grid_w;
    for (int c = lane * V; c < C; c += 32 * V) {
        for (int pw = 0; pw < PW; ++pw) {
            float acc[V];
#pragma unroll
            for (int i = 0; i < V; ++i) acc[i] = 0.f;
            if (batch_ok) {
#pragma unroll
                for (int iy = 0; iy < (GRID > 0 ? GRID : 1 << 30); ++iy) {
                    if (iy >= gh) break;
                    const AxisTerm<float> ty =
                        axis_term<float>(g.y0 + (float)ph * g.bin_h + ((float)iy + 0.5f) * g.bin_h / (float)gh, H);
#pragma unroll
                    for (int ix = 0; ix < (GRID > 0 ? GRID : 1 << 30); ++ix) {
                        if (ix >= gw) break;
                        const AxisTerm<float> tx =
                            axis_term<float>(g.x0 + (float)pw * g.bin_w + ((float)ix + 0.5f) * g.bin_w / (float)gw, W);
                        const float live = (ty.valid && tx.valid) ? 1.f : 0.f;       // outside samples contribute 0
                        const float w1 = ty.h * tx.h * live, w2 = ty.h * tx.l * live, w3 = ty.l * tx.h * live,
                                    w4 = ty.l * tx.l * live;
                        float v1[V], v2[V], v3[V], v4[V];
                        unpack<T>(ldg_v4(map + (long long)(ty.low * W + tx.low) * C + c), v1);
                        unpack<T>(ldg_v4(map + (long long)(ty.low * W + tx.high) * C + c), v2);
                        unpack<T>(ldg_v4(map + (long long)(ty.high * W + tx.low) * C + c), v3);
                        unpack<T>(ldg_v4(map + (long long)(ty.high * W + tx.high) * C + c), v4);
#pragma unroll
                        for (int i = 0; i < V; ++i) acc[i] += w1 * v1[i] + w2 * v2[i] + w3 * v3[i] + w4 * v4[i];
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < V; ++i) acc[i] *= g.inv_count;
            *reinterpret_cast<uint4*>(out + ((k * PH + ph) * PW + pw) * C + c) = pack<T>(acc);
        }
    }
}

__device__ __forceinline__ void atomic_add_ct(float* p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void atomic_add_ct(double* p, double v) { atomicAdd(p, v); }

// backward: every corner of every sample receives weight * grad / count (mmcv roi_align_backward_cuda_kernel);
// accumulation in CT (fp32 for the 16-bit dtypes, the caller casts once).  DET: grad_feat is the int64 accumulator of
// the deterministic backward and every contribution is added in fixed point at det's scale (DESIGN.md section 3.15).
template <typename T, typename CT, bool DET = false>
__global__ void __launch_bounds__(256)
roi_align_bwd_kernel(const T* __restrict__ grad_out, const CT* __restrict__ rois, CT* __restrict__ grad_feat, int N,
                     int H, int W, int C, long long bins, int PH, int PW, CT scale, int sampling_ratio, int aligned,
                     const DetHeader* __restrict__ det)
{
    const long long bin = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (bin >= bins) return;
    const int pw = (int)(bin % PW), ph = (int)((bin / PW) % PH);
    const long long k = bin / ((long long)PW * PH);
    const RoiGeom<CT> g = roi_geom<CT>(rois + 5 * k, scale, sampling_ratio, aligned, PH, PW);
    if (g.batch < 0 || g.batch >= N) return;
    CT* map = grad_feat + (long long)g.batch * H * W * C;
    long long* map64 = reinterpret_cast<long long*>(grad_feat) + (long long)g.batch * H * W * C;
    CT det_scale = (CT)0;
    if constexpr (DET) det_scale = sizeof(CT) == 8 ? (CT)det->scale : (CT)det->scale_f;
    const bool vec = !DET && (C % 4 == 0) && sizeof(CT) == 4;
    for (int iy = 0; iy < g.grid_h; ++iy) {
        const CT y = g.y0 + (CT)ph * g.bin_h + ((CT)iy + (CT)0.5) * g.bin_h / (CT)g.grid_h;
        for (int ix = 0; ix < g.grid_w; ++ix) {
            const CT x = g.x0 + (CT)pw * g.bin_w + ((CT)ix + (CT)0.5) * g.bin_w / (CT)g.grid_w;
            const BinSample<CT> s = bin_sample<CT>(y, x, H, W);
            if (s.w1 == (CT)0 && s.w2 == (CT)0 && s.w3 == (CT)0 && s.w4 == (CT)0) continue;
            const CT wk[4] = {s.w1 * g.inv_count, s.w2 * g.inv_count, s.w3 * g.inv_count, s.w4 * g.inv_count};
            const int pk[4] = {s.p1, s.p2, s.p3, s.p4};
            if (vec) {
                if constexpr (sizeof(CT) == 4) {
                    for (int c = lane * 4; c < C; c += 128) {
                        const T* gp = grad_out + bin * C + c;
                        const float g0 = to_f32<T>(gp[0]), g1 = to_f32<T>(gp[1]), g2 = to_f32<T>(gp[2]), g3 = to_f32<T>(gp[3]);
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            red_add_f32x4(reinterpret_cast<float*>(map) + (long long)pk[q] * C + c, (float)wk[q] * g0,
                                          (float)wk[q] * g1, (float)wk[q] * g2, (float)wk[q] * g3);
                    }
                }
            } else {
                for (int c = lane; c < C; c += 32) {
                    const CT gv = load_as<T, CT>(grad_out + bin * C + c);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if constexpr (DET) red_fixed(map64 + (long long)pk[q] * C + c, wk[q] * gv, det_scale);
                        else atomic_add_ct(map + (long long)pk[q] * C + c, wk[q] * gv);
                    }
                }
            }
        }
    }
}

}  // namespace

cudaError_t roi_align_forward(const RoiAlignArgs& a, cudaStream_t st)
{
    const long long bins = (long long)a.K * a.PH * a.PW;
    if (bins == 0 || a.C == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((bins + 7) / 8);
    const bool aligned16 = ((uintptr_t)a.feat % 16 == 0) && ((uintptr_t)a.out % 16 == 0);
    const long long bin_rows = (long long)a.K * a.PH;
    const unsigned row_blocks = (unsigned)((bin_rows + 7) / 8);
#define ROI_VEC_G(T, GRID)                                                                                           \
    roi_align_fwd_vec_kernel<T, GRID><<<row_blocks, 256, 0, st>>>((const T*)a.feat, (const float*)a.rois, (T*)a.out, \
                                                                 a.N, a.H, a.W, a.C, bin_rows, a.PH, a.PW,           \
                                                                 (float)a.scale, a.sampling_ratio, a.aligned)
#define ROI_VEC(T) do { if (a.sampling_ratio == 2) ROI_VEC_G(T, 2); else ROI_VEC_G(T, 0); } while (0)
#define ROI_SCALAR(T, CT)                                                                                          \
    roi_align_fwd_kernel<T, CT><<<blocks, 256, 0, st>>>((const T*)a.feat, (const CT*)a.rois, (T*)a.out, a.N, a.H,   \
                                                        a.W, a.C, bins, a.PH, a.PW, (CT)a.scale, a.sampling_ratio, a.aligned)
    switch (a.dtype) {
        case kF32:  if (a.C % 4 == 0 && aligned16) ROI_VEC(float); else ROI_SCALAR(float, float); break;
        case kBF16: if (a.C % 8 == 0 && aligned16) ROI_VEC(__nv_bfloat16); else ROI_SCALAR(__nv_bfloat16, float); break;
        case kF16:  if (a.C % 8 == 0 && aligned16) ROI_VEC(__half); else ROI_SCALAR(__half, float); break;
        case kF64:  ROI_SCALAR(double, double); break;
        default: return cudaErrorInvalidValue;
    }
#undef ROI_VEC_G
#undef ROI_VEC
#undef ROI_SCALAR
    return cudaGetLastError();
}

cudaError_t roi_align_backward(const RoiAlignArgs& a, cudaStream_t st)
{
    const long long bins = (long long)a.K * a.PH * a.PW;
    if (bins == 0 || a.C == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((bins + 7) / 8);
#define ROI_BWD(T, CT)                                                                                             \
    roi_align_bwd_kernel<T, CT><<<blocks, 256, 0, st>>>((const T*)a.grad_out, (const CT*)a.rois, (CT*)a.grad_accum, \
                                                        a.N, a.H, a.W, a.C, bins, a.PH, a.PW, (CT)a.scale,          \
                                                        a.sampling_ratio, a.aligned, nullptr)
    switch (a.dtype) {
        case kF32:  ROI_BWD(float, float); break;
        case kBF16: ROI_BWD(__nv_bfloat16, float); break;
        case kF16:  ROI_BWD(__half, float); break;
        case kF64:  ROI_BWD(double, double); break;
        default: return cudaErrorInvalidValue;
    }
#undef ROI_BWD
    return cudaGetLastError();
}

cudaError_t roi_align_backward_deterministic(const RoiAlignArgs& a, void* scratch, long long scratch_bytes,
                                             cudaStream_t st)
{
    if (a.dtype < kF32 || a.dtype > kF16) return cudaErrorInvalidValue;
    const long long count = (long long)a.N * a.H * a.W * a.C;
    if (scratch == nullptr || scratch_bytes < det_scratch_bytes(count, 0)) return cudaErrorInvalidValue;
    DetHeader* h = static_cast<DetHeader*>(scratch);
    long long* acc = reinterpret_cast<long long*>(static_cast<char*>(scratch) + kDetHeaderBytes);
    const long long bins = (long long)a.K * a.PH * a.PW;
    cudaError_t err = det_begin(scratch, count, st);
    if (err == cudaSuccess && bins > 0) err = det_absmax(a.dtype, a.grad_out, bins, a.C, a.C, &h->gmax, st);
    // a sample adds weight * g / count to each corner and its four weights sum to 1 (clamped corners coincide, their
    // weights add), and a bin has `count` samples: a bin adds at most |g| to any pixel, |grad| <= K*PH*PW * max|g|
    if (err == cudaSuccess) err = det_finalize(h, (double)bins, 1, a.dtype == kF64, st);
    if (err == cudaSuccess && bins > 0 && a.C > 0) {
        const unsigned blocks = (unsigned)((bins + 7) / 8);
#define ROI_BWD_DET(T, CT)                                                                                         \
    roi_align_bwd_kernel<T, CT, true><<<blocks, 256, 0, st>>>((const T*)a.grad_out, (const CT*)a.rois, (CT*)acc,     \
                                                              a.N, a.H, a.W, a.C, bins, a.PH, a.PW, (CT)a.scale,    \
                                                              a.sampling_ratio, a.aligned, h)
        switch (a.dtype) {
            case kF32:  ROI_BWD_DET(float, float); break;
            case kBF16: ROI_BWD_DET(__nv_bfloat16, float); break;
            case kF16:  ROI_BWD_DET(__half, float); break;
            case kF64:  ROI_BWD_DET(double, double); break;
        }
#undef ROI_BWD_DET
        err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = det_finish(a.dtype, acc, a.grad_accum, count, h, st);
    return err;
}

}  // namespace msda
