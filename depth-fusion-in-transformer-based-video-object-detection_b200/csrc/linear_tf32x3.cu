// fp32-grade linear layer on the 5th-generation tensor cores (sm_100a):
//
//     y = x W^T + b   (optionally ReLU),   x [rows, K], W [N, K], y [rows, N], everything fp32 in HBM.
//
// The reference model is fp32 end to end (every nn.Linear of models/ops/modules/ms_deform_attn.py:94-116 and
// models/deformable_transformer_single.py:544-548 is an IEEE SGEMM there); on B200 the SIMT SGEMM is 40 of the 45 ms of a
// 6-layer fp32 encoder.  This kernel evaluates the product with the error-compensated three-term TF32 split
//
//     x = x_hi + x_lo,  W = W_hi + W_lo      (*_hi = the operand on TF32's 10 mantissa bits, *_lo = the exact rest)
//     x W^T ~= x_lo W_hi^T + x_hi W_lo^T + x_hi W_hi^T          (fp32 accumulation in tensor memory)
//
// whose dropped term and operand roundings are O(2^-22) -- fp32-grade results (tests/test_gpu_layer_epilogue.py) at a
// third of the TF32 tensor rate.  Round 1 ran the same split as one library TF32 GEMM over a 3K-long reduction, which
// needs a separate pass that writes [lo | hi | hi] (3x the activation) to HBM first: 6.6 of its 20.1 ms.  Here the split
// of the activation tile happens in SHARED MEMORY between the TMA load and the MMA; W_hi / W_lo are split once on the
// host side of the C ABI (weights are static during inference).
//
// One CTA per SM, clusters of two, persistent over (row tile, column tile) pairs, 128 x 256 output tile per CTA, K in blocks of 16 fp32
// (64-byte SWIZZLE_64B rows).  Warp roles (14 warps):
//   0-3, 10-13  epilogue   tcgen05.ld of the finished accumulators (lane = output row), + bias, ReLU, staged 32 x 32 and written
//                   with TMA stores
//   4-7  converter  x tile in shared memory -> x_lo (second tile, same swizzled layout: the split is elementwise, so it
//                   never has to know the layout), then fence.proxy.async; x_hi is the x tile as the tensor core reads it
//   8    MMA issuer 2 K-steps x 3 terms of tcgen05.mma kind::tf32 per K block; TWO accumulators in TMEM (see there)
//   9    TMA producer  x tile and this CTA's half of the W_hi / W_lo tiles (multicast to the cluster) per K block, four
//                      stages of 48 KB
#include <cuda.h>

#include <atomic>

#include "msda_common.cuh"
#include "msda_launch.h"
#include "umma.cuh"

namespace msda {

using namespace umma;

constexpr int kLtBM = 128;                 // output rows per tile (TMEM lanes)
constexpr int kLtBN = 256;                 // output columns per tile (TMEM columns of one accumulator)
// K block: 16 fp32 = 64-byte SWIZZLE_64B rows, four stages of 48 KB (default), or 32 fp32 = one 128-byte SWIZZLE_128B row,
// two stages of 96 KB (-DMSDA_TF32_BK=32).  The same bytes in flight in finer grains: measured at 8 x 22 223 rows, BK 32 |
// BK 16, ms: 256 <- 256: 0.122 | 0.116; 384 <- 256: 0.190 | 0.175; 1024 <- 256: 0.412 | 0.417; 256 <- 1024: 0.380 | 0.370.
#ifndef MSDA_TF32_BK
#define MSDA_TF32_BK 16
#endif
constexpr int kLtBK = MSDA_TF32_BK;
constexpr int kLtRowBytes = kLtBK * 4;     // bytes of a K block row = swizzle span
constexpr int kLtKSteps = kLtBK / 8;       // tcgen05.mma kind::tf32 takes K = 8 per instruction
constexpr int kLtStages = kLtBK == 32 ? 2 : 4;
static_assert(kLtBK == 32 || kLtBK == 16, "K block = one SWIZZLE_128B or SWIZZLE_64B row");
constexpr int kLtCluster = 2;              // CTAs that share every W tile (TMA multicast)
constexpr int kLtABytes = kLtBM * kLtRowBytes;     // 16 KB
constexpr int kLtBBytes = kLtBN * kLtRowBytes;     // 32 KB
constexpr int kLtStageBytes = 2 * kLtABytes + 2 * kLtBBytes;      // x_hi | x_lo | W_hi | W_lo = 96 KB
constexpr int kLtEpiThreads = 256, kLtConvThreads = 128;      // epilogue: warps 0-3 and 10-13 (two per TMEM lane quadrant)
constexpr int kLtThreads = kLtEpiThreads + kLtConvThreads + 64;
constexpr int kLtOutBytes = 32 * 128;      // one epilogue warp's staging tile: 32 rows x 32 fp32, SWIZZLE_128B
constexpr int kLtSmem = kLtStages * kLtStageBytes + 8 * kLtOutBytes + kLtBN * 4 + 256;
static_assert(kLtSmem <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");

struct LtBars {
    unsigned long long full[kLtStages], conv[kLtStages], empty[kLtStages], acc_full, acc_free;
    unsigned tmem_base;
};

// instruction descriptor, kind::tf32: D fp32, A / B TF32 (format 2), both K-major, M x N tile
__device__ __forceinline__ unsigned make_idesc_tf32(int m, int n)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(n >> 3) << 17) | ((unsigned)(m >> 4) << 24);
}
// shared-memory matrix descriptor of a K-major operand tile whose rows are one swizzle span (128 or 64 bytes): 8-row groups
// of 8 x span bytes
__device__ __forceinline__ unsigned long long lt_desc(const void* smem_ptr)
{
    if constexpr (kLtBK == 32) return make_desc_sw128(smem_ptr);
    const unsigned addr = smem_u32(smem_ptr);
    unsigned long long d = 0;
    d |= (unsigned long long)((addr & 0x3FFFF) >> 4);            // start address
    d |= (unsigned long long)1 << 16;                            // leading byte offset (unused for swizzled K-major)
    d |= (unsigned long long)(512 >> 4) << 32;                   // stride between 8-row groups: 8 x 64 bytes
    d |= (unsigned long long)1 << 46;                            // descriptor version (sm_100)
    d |= (unsigned long long)4 << 61;                            // layout: SWIZZLE_64B
    return d;
}
__device__ __forceinline__ void mma_tf32(unsigned tmem_d, unsigned long long desc_a, unsigned long long desc_b,
                                         unsigned idesc, bool accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"((unsigned)accumulate) : "memory");
}

// W tiles are what the kernel streams: 64 of the 80 KB a K block brings in, re-read from L2 by every CTA for every tile --
// at full tensor rate 148 CTAs would ask L2 for 14 TB/s, and the single-CTA version of this kernel sat at the ~6-8 TB/s
// the L2 -> SM fabric delivers (ncu: 911 MB in 153 us, tensor pipe 40 % active).  Two CTAs of a cluster therefore work on
// two ROW tiles of the same column tile in lockstep, each loads HALF of every W tile and multicasts it into both CTAs'
// shared memory: 48 KB per K block and CTA.  A stage is released by the MMAs of BOTH CTAs (multicast tcgen05.commit on
// the `empty` barrier of each).
//
// DROP: dropout after the ReLU, mask of element row * N + col (dropout_keep8: one Philox call per two float4 of a lane).
template <bool DROP>
__global__ void __cluster_dims__(kLtCluster, 1, 1) __launch_bounds__(kLtThreads, 1)
linear_tf32x3_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_wh,
                     const __grid_constant__ CUtensorMap tm_wl, const __grid_constant__ CUtensorMap tm_y,
                     const float* __restrict__ bias, long long rows, int N, int K, int relu, int bn,
                     const unsigned long long* __restrict__ drop_key, unsigned drop_thresh, float drop_scale)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* s_out = smem + kLtStages * kLtStageBytes;            // [8 epilogue warps][kLtOutBytes], 1024-byte aligned
    float* s_bias = reinterpret_cast<float*>(s_out + 8 * kLtOutBytes);
    LtBars* bars = reinterpret_cast<LtBars*>(s_out + 8 * kLtOutBytes + kLtBN * 4);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long tiles_m = (rows + kLtBM - 1) / kLtBM;
    // bn: column tile width chosen by the host (<= kLtBN, a multiple of 32 that splits N evenly: 384 -> 2 x 192)
    const int tiles_n = (N + bn - 1) / bn;
    // work unit of a cluster: kLtCluster consecutive row tiles x one column tile; CTA `rank` takes row tile group * C + rank
    // (past the last row tile: TMA reads zeros, the epilogue stores nothing)
    const long long tiles = ((tiles_m + kLtCluster - 1) / kLtCluster) * tiles_n;
    const int kblocks = K / kLtBK;
    const unsigned rank = cluster_ctarank();
    const long long first = blockIdx.x / kLtCluster, stride = gridDim.x / kLtCluster;
    constexpr unsigned short kAll = (unsigned short)((1u << kLtCluster) - 1u);

    if (warp == 0) tmem_alloc(&bars->tmem_base, 512);
    if (tid == 128) {
        for (int i = 0; i < kLtStages; ++i) {
            mbar_init(&bars->full[i], 1);
            mbar_init(&bars->conv[i], kLtConvThreads);
            mbar_init(&bars->empty[i], kLtCluster);
        }
        mbar_init(&bars->acc_full, 1);
        mbar_init(&bars->acc_free, kLtEpiThreads);
        fence_mbar_init();
        tma_prefetch_desc(&tm_x); tma_prefetch_desc(&tm_wh); tma_prefetch_desc(&tm_wl); tma_prefetch_desc(&tm_y);
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                            // every CTA's barriers exist before anything arrives on them
    tcgen05_fence_after();
    const unsigned tmem = bars->tmem_base;

    if (warp == 9) {
        // ======================================= TMA producer =======================================
        if (elect_one()) {
            unsigned kiter = 0;
            const int kSlice = bn / kLtCluster, kSliceBytes = kSlice * kLtRowBytes;
            for (long long t = first; t < tiles; t += stride) {
                const int m0 = (int)((t / tiles_n) * kLtCluster + rank) * kLtBM, n0 = (int)(t % tiles_n) * bn;
                for (int kb = 0; kb < kblocks; ++kb, ++kiter) {
                    const int s = kiter % kLtStages;
                    // both CTAs are done with the stage: my slices land in the peer's shared memory too
                    if (kiter >= kLtStages) mbar_wait(&bars->empty[s], ((kiter / kLtStages) - 1) & 1);
                    unsigned char* st = smem + s * kLtStageBytes;
                    mbar_expect_tx(&bars->full[s], kLtABytes + 2 * bn * kLtRowBytes);   // my x tile + every CTA's W slices
                    tma_load_2d(st, &tm_x, kb * kLtBK, m0, &bars->full[s]);
                    tma_load_2d_multicast(st + 2 * kLtABytes + rank * kSliceBytes, &tm_wh, kb * kLtBK,
                                          n0 + (int)rank * kSlice, &bars->full[s], kAll);
                    tma_load_2d_multicast(st + 2 * kLtABytes + kLtBBytes + rank * kSliceBytes, &tm_wl, kb * kLtBK,
                                          n0 + (int)rank * kSlice, &bars->full[s], kAll);
                }
            }
        }
        __syncwarp();
    } else if (warp == 8) {
        // ======================================= MMA issuer =======================================
        unsigned kiter = 0, it = 0;
        for (long long t = first; t < tiles; t += stride, ++it) {
            const int n0 = (int)(t % tiles_n) * bn;
            const int n_cur = min(bn, N - n0);
            const unsigned idesc = make_idesc_tf32(kLtBM, n_cur);
            // Two accumulators: the hi x hi products and the two correction terms.  The tensor core truncates when it adds
            // into the accumulator, about half an ulp of the RUNNING SUM per instruction and always towards zero; 96
            // instructions into one accumulator measured 2.3e-6 of the output range (K = 256; 8.5e-6 at K = 1024).  The
            // correction terms are 2^-11 of the sum, so in an accumulator of their own their truncations do not matter,
            // and the main accumulator sees K / 8 instructions, like one plain TF32 GEMM.
            const unsigned acc_big = tmem, acc_small = tmem + kLtBN;
            if (it >= 1) mbar_wait(&bars->acc_free, (it - 1) & 1);               // the epilogue has drained the accumulators
            for (int kb = 0; kb < kblocks; ++kb, ++kiter) {
                const int s = kiter % kLtStages;
                unsigned char* st = smem + s * kLtStageBytes;
                const unsigned long long d_xh = lt_desc(st), d_xl = lt_desc(st + kLtABytes);
                const unsigned long long d_wh = lt_desc(st + 2 * kLtABytes), d_wl = lt_desc(st + 2 * kLtABytes + kLtBBytes);
                mbar_wait(&bars->full[s], (kiter / kLtStages) & 1);              // x and W tiles landed
                tcgen05_fence_after();
                // the two terms with x_hi need nothing from the converter: the tensor core reads the top 19 bits of the
                // fp32 words TMA wrote (x_hi = x truncated to TF32), so they go first and cover the converter's latency
                if (elect_one()) {
#pragma unroll
                    for (int j = 0; j < kLtKSteps; ++j) {                        // K = 8 per instruction: 32 bytes of the row
                        mma_tf32(acc_small, desc_advance(d_xh, j * 32), desc_advance(d_wl, j * 32), idesc, (kb | j) != 0);
                        mma_tf32(acc_big, desc_advance(d_xh, j * 32), desc_advance(d_wh, j * 32), idesc, (kb | j) != 0);
                    }
                }
                __syncwarp();
                mbar_wait(&bars->conv[s], (kiter / kLtStages) & 1);              // x_lo written
                tcgen05_fence_after();
                if (elect_one()) {
#pragma unroll
                    for (int j = 0; j < kLtKSteps; ++j)
                        mma_tf32(acc_small, desc_advance(d_xl, j * 32), desc_advance(d_wh, j * 32), idesc, true);
                    mma_commit_multicast(&bars->empty[s], kAll);                 // stage free (here and in the peer) once these MMAs have read it
                    if (kb == kblocks - 1) mma_commit(&bars->acc_full);
                }
                __syncwarp();
            }
        }
    } else if (warp >= 4 && warp < 8) {
        // ======================================= converter warps =======================================
        const int ct = tid - 128;
        unsigned kiter = 0;
        for (long long t = first; t < tiles; t += stride) {
            for (int kb = 0; kb < kblocks; ++kb, ++kiter) {
                const int s = kiter % kLtStages;
                mbar_wait(&bars->full[s], (kiter / kLtStages) & 1);
                const uint4* xh = reinterpret_cast<const uint4*>(smem + s * kLtStageBytes);
                uint4* xl = reinterpret_cast<uint4*>(smem + s * kLtStageBytes + kLtABytes);
                // x_hi is what the tensor core sees of x: the word with its 13 low mantissa bits cleared (the x tile is not
                // rewritten).  x_lo = x - x_hi is exact in fp32 (at most 13 significant bits); it is rounded to nearest on
                // TF32's 10 mantissa bits here, so that the tensor core's own truncation of it is a no-op.
                auto lo = [](unsigned v) -> unsigned {
                    const float l = __uint_as_float(v) - __uint_as_float(v & 0xffffe000u);
                    return (__float_as_uint(l) + 0x1000u) & 0xffffe000u;
                };
#pragma unroll
                for (int i = 0; i < kLtABytes / 16 / kLtConvThreads; ++i) {
                    const int idx = i * kLtConvThreads + ct;                     // consecutive lanes, consecutive chunks
                    const uint4 v = xh[idx];
                    xl[idx] = make_uint4(lo(v.x), lo(v.y), lo(v.z), lo(v.w));
                }
                fence_proxy_async();                 // generic-proxy writes -> tensor-core (async proxy) reads
                mbar_arrive(&bars->conv[s]);
            }
        }
    } else {
        // ======================================= epilogue warps =======================================
        // two warps per TMEM lane quadrant (warp % 4): warps 0-3 take the even 32-column chunks, warps 10-13 the odd ones
        const int quad = warp & 3, half = warp < 4 ? 0 : 1, et = half * 128 + quad * 32 + lane;
        const unsigned lane_base = (unsigned)(quad * 32) << 16;
        unsigned long long key = 0;
        if constexpr (DROP) key = *drop_key;
        unsigned it = 0;
        for (long long t = first; t < tiles; t += stride, ++it) {
            const long long m0 = ((t / tiles_n) * kLtCluster + rank) * kLtBM;
            const int n0 = (int)(t % tiles_n) * bn;
            const int n_cur = min(bn, N - n0);
            // bias slice of the tile (the previous tile's readers are past their last read: barrier below)
            named_bar_sync(1, kLtEpiThreads);
            for (int i = et; i < kLtBN; i += kLtEpiThreads) s_bias[i] = (bias != nullptr && i < n_cur) ? bias[n0 + i] : 0.f;
            named_bar_sync(1, kLtEpiThreads);
            mbar_wait(&bars->acc_full, it & 1);
            tcgen05_fence_after();
            // 32 rows x 32 columns at a time: TMEM -> registers (lane = row) -> this warp's staging tile in the SWIZZLE_128B
            // layout (16-byte chunk c of row r at chunk c ^ (r & 7): conflict-free for lane = row) -> ONE TMA store of
            // the box (full 128-byte lines; rows past the end of y are clipped by the tensor map).  The staging tile is
            // reused once the previous store has read it.
            const int row0 = (int)m0 + quad * 32;
            unsigned char* stage = s_out + (half * 4 + quad) * kLtOutBytes;
            for (int c = half * 32; c < n_cur; c += 64) {
                float v[32], w[32];
                tmem_ld32(tmem + c + lane_base, v);
                tmem_ld32(tmem + kLtBN + c + lane_base, w);
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncwarp();
                unsigned bits = 0;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c + 4 * q);
                    float4 o = make_float4(v[4 * q] + w[4 * q] + b4.x, v[4 * q + 1] + w[4 * q + 1] + b4.y,
                                           v[4 * q + 2] + w[4 * q + 2] + b4.z, v[4 * q + 3] + w[4 * q + 3] + b4.w);
                    if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                    if constexpr (DROP) {
                        if ((q & 1) == 0)
                            bits = dropout_keep8((unsigned long long)((long long)(row0 + lane) * N + n0 + c + 4 * q) >> 3, key,
                                                 drop_thresh);
                        const unsigned b = bits >> (4 * (q & 1));
                        o.x *= b & 1u ? drop_scale : 0.f;
                        o.y *= b & 2u ? drop_scale : 0.f;
                        o.z *= b & 4u ? drop_scale : 0.f;
                        o.w *= b & 8u ? drop_scale : 0.f;
                    }
                    *reinterpret_cast<float4*>(stage + lane * 128 + ((q ^ (lane & 7)) << 4)) = o;
                }
                fence_proxy_async();                 // generic-proxy writes -> TMA (async proxy) read
                __syncwarp();
                if (lane == 0) {
                    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];"
                                 :: "l"(&tm_y), "r"(smem_u32(stage)), "r"(n0 + c), "r"(row0) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
            tcgen05_fence_before();
            mbar_arrive(&bars->acc_free);
        }
    }
    if ((warp < 4 || warp >= 10) && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // my stores have left shared memory
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                            // no CTA leaves while a peer may still write its shared memory / barriers
    if (warp == 0) tmem_free(tmem, 512);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*LtEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static LtEncodeTiledFn lt_encode_tiled_fn()
{
    static LtEncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<LtEncodeTiledFn>(p);
    }
    return fn;
}

// row-major fp32 matrix [n_rows, n_cols]; box = 32 columns (128 bytes, SWIZZLE_128B) x box_rows rows; rows past the end
// read as zeros
static bool lt_make_map(CUtensorMap* map, const void* base, unsigned long long n_rows, unsigned long long n_cols, int box_rows,
                        int box_cols = kLtBK)
{
    LtEncodeTiledFn fn = lt_encode_tiled_fn();
    if (fn == nullptr) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)n_cols, n_rows};
    const cuuint64_t strides[1] = {(cuuint64_t)n_cols * 4};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
              CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool linear_tf32x3_supported(int n, int k)
{
    return n >= 32 && n % 32 == 0 && k >= 32 && k % 32 == 0;
}

template <bool DROP>
static cudaError_t launch_linear_tf32x3(const float* x, const float* w_hi, const float* w_lo, const float* bias,
                                        long long rows, int n, int k, int relu, const unsigned long long* key,
                                        DropoutRule rule, float* y, cudaStream_t stream)
{
    if (!linear_tf32x3_supported(n, k) || rows < 0 || rows >= (1ll << 31) - 1024) return cudaErrorInvalidValue;   // row coordinates are int
    if (rows == 0) return cudaSuccess;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w_hi) | reinterpret_cast<uintptr_t>(w_lo) |
         reinterpret_cast<uintptr_t>(y)) % 16 != 0)
        return cudaErrorInvalidValue;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    static bool configured[64] = {};          // the attribute is per device: one process may drive several GPUs
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(linear_tf32x3_kernel<DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLtSmem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    // column tile width: as few tiles as 256 columns allow, of equal width (a multiple of 32; each CTA of the cluster
    // loads bn / 2 weight rows, a multiple of the 8-row swizzle group)
    const int tiles_n = (n + kLtBN - 1) / kLtBN;
    const int bn = ((n + tiles_n - 1) / tiles_n + 31) / 32 * 32;
    alignas(64) CUtensorMap tm_x, tm_wh, tm_wl, tm_y;
    if (!lt_make_map(&tm_x, x, (unsigned long long)rows, (unsigned long long)k, kLtBM) ||
        !lt_make_map(&tm_wh, w_hi, (unsigned long long)n, (unsigned long long)k, bn / kLtCluster) ||
        !lt_make_map(&tm_wl, w_lo, (unsigned long long)n, (unsigned long long)k, bn / kLtCluster) ||
        !lt_make_map(&tm_y, y, (unsigned long long)rows, (unsigned long long)n, 32, 32))
        return cudaErrorNotSupported;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles_m = (rows + kLtBM - 1) / kLtBM;
    const long long units = ((tiles_m + kLtCluster - 1) / kLtCluster) * ((n + bn - 1) / bn);
    const long long clusters = sms / kLtCluster;
    const int grid = (int)(units < clusters ? units : clusters) * kLtCluster;
    linear_tf32x3_kernel<DROP><<<grid, kLtThreads, kLtSmem, stream>>>(tm_x, tm_wh, tm_wl, tm_y, bias, rows, n, k, relu, bn,
                                                                       key, rule.thresh, rule.scale);
    return cudaGetLastError();
}

cudaError_t linear_tf32x3(const float* x, const float* w_hi, const float* w_lo, const float* bias, long long rows, int n,
                          int k, int relu, float* y, cudaStream_t stream)
{
    return launch_linear_tf32x3<false>(x, w_hi, w_lo, bias, rows, n, k, relu, nullptr, DropoutRule{0u, 1.f}, y, stream);
}

cudaError_t linear_tf32x3_relu_dropout(const float* x, const float* w_hi, const float* w_lo, const float* bias,
                                       long long rows, int n, int k, const unsigned long long* key, DropoutRule rule,
                                       float* y, cudaStream_t stream)
{
    if (key == nullptr) return cudaErrorInvalidValue;
    return launch_linear_tf32x3<true>(x, w_hi, w_lo, bias, rows, n, k, 1, key, rule, y, stream);
}

// ------------------------------------------------------------------------------------------
// weight / bias gradient of the same layer (fp32 training):
//
//     dW [N, K] = g^T x,   db [N] = sum over rows of g,   g [rows, N], x [rows, K], fp32.
//
// The same three-term split, now with BOTH operands activations:  g^T x ~= g_hi^T x_hi + (g_lo^T x_hi + g_hi^T x_lo).
// The reduction runs over `rows`, so as loaded both operands are MN-major: a TMA box {32 columns, 32 rows} with
// SWIZZLE_128B is 32 rows of 128 bytes, 32 features (or inputs) x 32 reduction steps.  kind::tf32 does not take MN-major
// operands: with the transpose bits set it wrote zeros for every descriptor encoding tried, while the same data loaded
// K-major gave the exact product (tools/umma/tf32_mn_probe.cu, profiles/r4_tf32_mn_probe.txt).  So the converter warps
// TRANSPOSE: thread f reads column f of the loaded g tile (feature f, 32 rows; conflict-free, a warp reads one 128-byte
// row per step) and writes row f of the K-major SWIZZLE_128B tiles g_hi^T (the words as loaded; the tensor core truncates
// them to TF32) and g_lo^T, and the same for x.  An output tile is 128 features (four g boxes, M) x up to 128 inputs (four
// x boxes, N); every MMA waits for the converter.
//
// Accumulator truncation: the tensor core truncates towards zero, about half an ulp of the running sum per instruction
// (DESIGN.md section 3.5: 32 instructions into one accumulator 6.9e-7 of the output range, 96 gave 2.3e-6).  A slice of
// ~2 400 rows would be 300 instructions, so (1) the two correction terms go to an accumulator of their own, and (2) the
// main accumulator is drained every kTwChunk K blocks (kTwChunk * 4 instructions): the epilogue warps add (main +
// correction) into fp32 registers with round-to-nearest adds while the MMA issuer fills the other accumulator pair.
// TMEM: pair p = main [256 p, 256 p + 128) | correction [256 p + 128, 256 p + 256) = 512 columns.  Measured on B200
// (DESIGN.md section 3.14): without the drain dW was up to 4.8e-5 of its range off fp64 at 177 784 rows; with a drain
// every 8 K blocks 6-9.5e-7 (the IEEE SGEMM: 4.6e-7-2.1e-6), every 2 K blocks 2.8-5.1e-7.
//
// The bias gradient comes from the converter warps, which read every g element anyway: thread f owns feature f of the
// tile and adds the 32 rows of a K block it transposes (a partial sum per K block, then into the slice sum: fixed order).
// Split-K, scratch layout, the reduce kernel and the determinism argument are those of linear_bf16_wgrad (linear_bf16.cu).
// Warp roles (14 warps): 0-7 epilogue (warp % 4 = TMEM lane quadrant, warp / 4 = which 64 columns), 8-11 converter,
// 12 MMA issuer, 13 TMA producer.
// ------------------------------------------------------------------------------------------
#ifndef MSDA_TF32_WG_CHUNK
#define MSDA_TF32_WG_CHUNK 8
#endif
constexpr int kTwChunk = MSDA_TF32_WG_CHUNK;   // K blocks (of 32 rows) per drain of the main accumulator: 32 instructions
constexpr int kTwBM = 128;                  // output features per tile (TMEM lanes)
constexpr int kTwBN = 128;                  // inputs per tile (TMEM columns of one accumulator)
constexpr int kTwBK = 32;                   // rows per K block
constexpr int kTwBox = 32 * kTwBK * 4;      // one {32 columns, 32 rows} fp32 box: 4 KB
constexpr int kTwOpBytes = 128 * kTwBK * 4;   // one K-major operand tile, 128 rows x 128 bytes: 16 KB
// stage: g as loaded | x as loaded | g_hi^T | g_lo^T | x_hi^T | x_lo^T (converter) = 96 KB
constexpr int kTwStageBytes = 6 * kTwOpBytes;
constexpr int kTwStages = 2;
static_assert(kTwBM == 128 && kTwBN == 128 && kTwBox * 4 == kTwOpBytes, "four 32-wide boxes per operand tile");
constexpr int kTwEpiThreads = 256, kTwConvThreads = 128;
constexpr int kTwThreads = kTwEpiThreads + kTwConvThreads + 64;
constexpr int kTwSmem = kTwStages * kTwStageBytes + 256;       // + barriers
static_assert(kTwSmem <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");
static_assert(kTwChunk >= 1, "at least one K block per accumulator drain");
constexpr int kTwTargetCtas = 148;          // B200 SMs: split count aimed at one CTA per SM, fixed so that the split (and
                                            // so the rounding of the result) does not depend on the device
constexpr int kTwMinKBlocks = 8;            // a split reads at least 256 rows: its partial tile is small against its loads
constexpr long long kTwBlkFloats = (long long)kTwBM * kTwBN + kTwBM;   // partial dW tile + partial db

struct TwBars {
    unsigned long long full[kTwStages], conv[kTwStages], empty[kTwStages], acc_full[2], acc_free[2];
    unsigned tmem_base;
};

// Converter step for one operand: column c (< 128) of the loaded tile (four {32 columns, 32 rows} SWIZZLE_128B boxes) ->
// row c of the K-major SWIZZLE_128B tiles hi (the words as loaded) and lo (x - x_hi on TF32's 10 mantissa bits, rounded
// to nearest, so that the tensor core's own truncation of it is a no-op, as in the forward's converter).  Returns the sum
// of the column (the bias gradient's share of this K block when the operand is g).
__device__ __forceinline__ float tw_transpose_column(const unsigned char* loaded, unsigned char* hi, unsigned char* lo, int c)
{
    const float* box = reinterpret_cast<const float*>(loaded + (c >> 5) * kTwBox);
    const int chunk = (c & 31) >> 2, word = c & 3;
    float v[kTwBK];
#pragma unroll
    for (int r = 0; r < kTwBK; ++r) v[r] = box[r * 32 + ((chunk ^ (r & 7)) << 2) + word];
    float sum = 0.f;
#pragma unroll
    for (int r = 0; r < kTwBK; ++r) sum += v[r];
    auto lo_of = [](float x) -> unsigned {
        const float l = x - __uint_as_float(__float_as_uint(x) & 0xffffe000u);
        return (__float_as_uint(l) + 0x1000u) & 0xffffe000u;
    };
    const unsigned row = (unsigned)((c >> 3) * 1024 + (c & 7) * 128);
#pragma unroll
    for (int q = 0; q < kTwBK / 4; ++q) {
        const unsigned off = row + ((q ^ (c & 7)) << 4);
        *reinterpret_cast<uint4*>(hi + off) = make_uint4(__float_as_uint(v[4 * q]), __float_as_uint(v[4 * q + 1]),
                                                         __float_as_uint(v[4 * q + 2]), __float_as_uint(v[4 * q + 3]));
        *reinterpret_cast<uint4*>(lo + off) = make_uint4(lo_of(v[4 * q]), lo_of(v[4 * q + 1]), lo_of(v[4 * q + 2]),
                                                         lo_of(v[4 * q + 3]));
    }
    return sum;
}

__global__ void __launch_bounds__(kTwThreads, 1)
linear_tf32x3_wgrad_kernel(const __grid_constant__ CUtensorMap tm_g, const __grid_constant__ CUtensorMap tm_x,
                           float* __restrict__ partial, long long rows, int N, int K, int tiles_n, int tiles, int splits,
                           int kb_per_split, int want_db)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    TwBars* bars = reinterpret_cast<TwBars*>(smem + kTwStages * kTwStageBytes);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // CTAs of one split (same rows) are adjacent: the tiles that share a slice of g or x read it from L2
    const int split = blockIdx.x / tiles, t = blockIdx.x % tiles;
    const int m0 = (t / tiles_n) * kTwBM, n0 = (t % tiles_n) * kTwBN;
    const int m_cur = min(kTwBM, N - m0), n_cur = min(kTwBN, K - n0);
    const int g_boxes = m_cur / 32, x_boxes = n_cur / 32;
    const int kblocks = (int)((rows + kTwBK - 1) / kTwBK);
    const int kb0 = split * kb_per_split, kb1 = min(kb0 + kb_per_split, kblocks);
    const int chunks = (kb1 - kb0 + kTwChunk - 1) / kTwChunk;
    const bool with_db = want_db && n0 == 0;
    float* blk = partial + ((long long)t * splits + split) * kTwBlkFloats;

    if (warp == 0) tmem_alloc(&bars->tmem_base, 512);
    if (tid == kTwEpiThreads) {
        for (int i = 0; i < kTwStages; ++i) {
            mbar_init(&bars->full[i], 1);
            mbar_init(&bars->conv[i], kTwConvThreads);
            mbar_init(&bars->empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) { mbar_init(&bars->acc_full[i], 1); mbar_init(&bars->acc_free[i], kTwEpiThreads); }
        fence_mbar_init();
        tma_prefetch_desc(&tm_g); tma_prefetch_desc(&tm_x);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const unsigned tmem = bars->tmem_base;

    if (warp == 13) {
        // ======================================= TMA producer =======================================
        if (elect_one()) {
            // boxes wholly past the last feature / input are not loaded: they only feed accumulator lanes / columns
            // that are never read.  Rows past the end arrive as zeros (TMA out-of-bounds fill).
            const unsigned bytes = (unsigned)(g_boxes + x_boxes) * kTwBox;
            for (int kb = kb0; kb < kb1; ++kb) {
                const int i = kb - kb0, s = i % kTwStages;
                if (i >= kTwStages) mbar_wait(&bars->empty[s], ((i / kTwStages) - 1) & 1);
                unsigned char* st = smem + s * kTwStageBytes;
                mbar_expect_tx(&bars->full[s], bytes);
                for (int c = 0; c < g_boxes; ++c) tma_load_2d(st + c * kTwBox, &tm_g, m0 + 32 * c, kb * kTwBK, &bars->full[s]);
                for (int c = 0; c < x_boxes; ++c)
                    tma_load_2d(st + kTwOpBytes + c * kTwBox, &tm_x, n0 + 32 * c, kb * kTwBK, &bars->full[s]);
            }
        }
        __syncwarp();
    } else if (warp == 12) {
        // ======================================= MMA issuer =======================================
        const unsigned idesc = make_idesc_tf32(kTwBM, n_cur);
        for (int kb = kb0; kb < kb1; ++kb) {
            const int i = kb - kb0, s = i % kTwStages, chunk = i / kTwChunk, p = chunk & 1;
            const bool chunk_first = i % kTwChunk == 0, chunk_last = i % kTwChunk == kTwChunk - 1 || kb == kb1 - 1;
            const unsigned acc_main = tmem + p * 256, acc_corr = acc_main + kTwBN;
            // the epilogue has drained this pair (chunk - 2)
            if (chunk_first && chunk >= 2) mbar_wait(&bars->acc_free[p], ((chunk >> 1) - 1) & 1);
            unsigned char* st = smem + s * kTwStageBytes;
            const unsigned long long d_gh = make_desc_sw128(st + 2 * kTwOpBytes), d_gl = make_desc_sw128(st + 3 * kTwOpBytes);
            const unsigned long long d_xh = make_desc_sw128(st + 4 * kTwOpBytes), d_xl = make_desc_sw128(st + 5 * kTwOpBytes);
            mbar_wait(&bars->conv[s], (i / kTwStages) & 1);                  // K-major hi / lo tiles written
            tcgen05_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < kTwBK / 8; ++j) {                        // K = 8 per instruction: 32 bytes of the row
                    const bool acc = !chunk_first || j != 0;
                    mma_tf32(acc_main, desc_advance(d_gh, j * 32), desc_advance(d_xh, j * 32), idesc, acc);
                    mma_tf32(acc_corr, desc_advance(d_gl, j * 32), desc_advance(d_xh, j * 32), idesc, acc);
                    mma_tf32(acc_corr, desc_advance(d_gh, j * 32), desc_advance(d_xl, j * 32), idesc, true);
                }
                mma_commit(&bars->empty[s]);                                 // stage free once these MMAs are done
                if (chunk_last) mma_commit(&bars->acc_full[p]);
            }
            __syncwarp();
        }
    } else if (warp >= 8) {
        // ======================================= converter warps =======================================
        // thread ct transposes feature ct of the g tile and input ct of the x tile (columns past the loaded boxes are
        // left alone: they only feed accumulator lanes / columns that are never read)
        const int ct = tid - kTwEpiThreads;
        float db = 0.f;
        for (int kb = kb0; kb < kb1; ++kb) {
            const int i = kb - kb0, s = i % kTwStages;
            mbar_wait(&bars->full[s], (i / kTwStages) & 1);
            unsigned char* st = smem + s * kTwStageBytes;
            if (ct < m_cur) db += tw_transpose_column(st, st + 2 * kTwOpBytes, st + 3 * kTwOpBytes, ct);
            if (ct < n_cur) tw_transpose_column(st + kTwOpBytes, st + 4 * kTwOpBytes, st + 5 * kTwOpBytes, ct);
            fence_proxy_async();                     // generic-proxy writes -> tensor-core (async proxy) reads
            mbar_arrive(&bars->conv[s]);
        }
        if (with_db && ct < m_cur) blk[(long long)kTwBM * kTwBN + ct] = db;
    } else {
        // ======================================= epilogue warps =======================================
        // TMEM lane = feature row of the tile; this warp's 64 columns of it summed over the chunks in registers
        const int quad = warp & 3, half = warp >> 2, r = quad * 32 + lane;
        const unsigned lane_base = (unsigned)(quad * 32) << 16;
        float sum[64];
#pragma unroll
        for (int c = 0; c < 64; ++c) sum[c] = 0.f;
        for (int chunk = 0; chunk < chunks; ++chunk) {
            const int p = chunk & 1;
            mbar_wait(&bars->acc_full[p], (chunk >> 1) & 1);
            tcgen05_fence_after();
#pragma unroll
            for (int c = 0; c < 64; c += 16) {
                if (half * 64 + c < n_cur) {
                    float v[16], w[16];
                    tmem_ld16(tmem + p * 256 + half * 64 + c + lane_base, v);
                    tmem_ld16(tmem + p * 256 + kTwBN + half * 64 + c + lane_base, w);
#pragma unroll
                    for (int e = 0; e < 16; ++e) sum[c + e] += v[e] + w[e];
                }
            }
            tcgen05_fence_before();
            mbar_arrive(&bars->acc_free[p]);
        }
        float4* dst = reinterpret_cast<float4*>(blk + (long long)r * kTwBN + half * 64);
#pragma unroll
        for (int q = 0; q < 16; ++q)
            if (half * 64 + 4 * q < n_cur) dst[q] = make_float4(sum[4 * q], sum[4 * q + 1], sum[4 * q + 2], sum[4 * q + 3]);
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 512);
}

// dW / db = sum over the splits of the partial blocks, in split order.  Block (32, 8): x = 4 consecutive outputs, y = every
// 8th split; the 8 sums are added in y order.
__global__ void __launch_bounds__(256)
linear_tf32x3_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, float* __restrict__ db, int N,
                                  int K, int tiles_n, int splits)
{
    __shared__ float4 s_sum[8][32];
    const long long q = (long long)blockIdx.x * 32 + threadIdx.x;        // quad of outputs
    const long long qw = (long long)N * K / 4, qb = db != nullptr ? N / 4 : 0;
    long long base = -1;
    float* dst = nullptr;
    if (q < qw) {
        const long long e = q * 4;
        const int o = (int)(e / K), i = (int)(e % K);
        base = ((long long)((o / kTwBM) * tiles_n + i / kTwBN) * splits) * kTwBlkFloats + (long long)(o % kTwBM) * kTwBN + i % kTwBN;
        dst = dw + e;
    } else if (q < qw + qb) {
        const int o = (int)(q - qw) * 4;
        base = ((long long)((o / kTwBM) * tiles_n) * splits) * kTwBlkFloats + (long long)kTwBM * kTwBN + o % kTwBM;
        dst = db + o;
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (base >= 0)
        for (int s = threadIdx.y; s < splits; s += 8) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(partial + base + (long long)s * kTwBlkFloats));
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
    s_sum[threadIdx.y][threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.y != 0 || base < 0) return;
#pragma unroll
    for (int y = 1; y < 8; ++y) {
        const float4 v = s_sum[y][threadIdx.x];
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    *reinterpret_cast<float4*>(dst) = acc;
}

bool linear_tf32x3_wgrad_supported(int n, int k)
{
    return n >= 32 && n % 32 == 0 && k >= 32 && k % 32 == 0;
}

struct TwPlan {
    int tiles_n, tiles, splits, kb_per_split;
};

static bool tf32x3_wgrad_plan(long long rows, int n, int k, TwPlan* p)
{
    if (!linear_tf32x3_wgrad_supported(n, k) || rows < 1 || rows >= (1ll << 31) - 1024) return false;
    p->tiles_n = (k + kTwBN - 1) / kTwBN;
    p->tiles = ((n + kTwBM - 1) / kTwBM) * p->tiles_n;
    const int kblocks = (int)((rows + kTwBK - 1) / kTwBK);
    const int want = max(1, kTwTargetCtas / p->tiles);
    p->kb_per_split = max(kTwMinKBlocks, (kblocks + want - 1) / want);
    p->splits = (kblocks + p->kb_per_split - 1) / p->kb_per_split;     // every split has at least one K block
    return true;
}

long long linear_tf32x3_wgrad_scratch_floats(long long rows, int n, int k)
{
    TwPlan p;
    return tf32x3_wgrad_plan(rows, n, k, &p) ? (long long)p.tiles * p.splits * kTwBlkFloats : 0;
}

cudaError_t linear_tf32x3_wgrad(const float* g, const float* x, long long rows, int n, int k, float* dw, float* db,
                                float* scratch, long long scratch_floats, cudaStream_t stream)
{
    TwPlan p;
    if (!tf32x3_wgrad_plan(rows, n, k, &p) || scratch_floats < (long long)p.tiles * p.splits * kTwBlkFloats || dw == nullptr)
        return cudaErrorInvalidValue;
    if ((reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dw) |
         reinterpret_cast<uintptr_t>(db) | reinterpret_cast<uintptr_t>(scratch)) % 16 != 0)
        return cudaErrorInvalidValue;
    int dev = 0;
    cudaGetDevice(&dev);
    // the attribute is per device; concurrent first calls may both set it (harmless), none reads a torn flag
    static std::atomic<bool> configured[64];
    if (dev < 0 || dev >= 64 || !configured[dev].load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(linear_tf32x3_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTwSmem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev].store(true, std::memory_order_release);
    }
    alignas(64) CUtensorMap tm_g, tm_x;
    if (!lt_make_map(&tm_g, g, (unsigned long long)rows, (unsigned long long)n, kTwBK, 32) ||
        !lt_make_map(&tm_x, x, (unsigned long long)rows, (unsigned long long)k, kTwBK, 32))
        return cudaErrorNotSupported;
    linear_tf32x3_wgrad_kernel<<<p.tiles * p.splits, kTwThreads, kTwSmem, stream>>>(
        tm_g, tm_x, scratch, rows, n, k, p.tiles_n, p.tiles, p.splits, p.kb_per_split, db != nullptr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const long long quads = (long long)n * k / 4 + (db != nullptr ? n / 4 : 0);
    linear_tf32x3_wgrad_reduce_kernel<<<(unsigned)((quads + 31) / 32), dim3(32, 8), 0, stream>>>(scratch, dw, db, n, k,
                                                                                                p.tiles_n, p.splits);
    return cudaGetLastError();
}

}  // namespace msda
