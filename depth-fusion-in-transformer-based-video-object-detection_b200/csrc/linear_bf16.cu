// bf16 linear layer of an inference pass on the 5th-generation tensor cores (sm_100a):
//
//     y = x W^T + b   (optionally ReLU, optionally rows zeroed by a padding mask),   x [rows, K], W [N, K], y [rows, N], bf16.
//
// `value_proj` of MSDeformAttn with its `masked_fill(padding_mask, 0)` (reference models/ops/modules/ms_deform_attn.py:94-96),
// the [sampling_offsets | attention_weights] projection (:98-100) and every other nn.Linear of a bf16 inference pass.  The
// product is memory-bound (91 MB in, 91-137 MB out at the encoder's 8 x 22 223 rows against 23-35 GFLOP), so the kernel is
// built around the HBM streams: x tiles by TMA through a four-stage ring, the weight tile shared by the two CTAs of a
// cluster (each loads half, TMA multicast), fp32 accumulators double-buffered in tensor memory so that the epilogue of a
// tile -- bias, ReLU, padding rows, bf16, 32 x 64 staging tiles in the SWIZZLE_128B layout, TMA stores of full lines --
// runs under the next tile's loads and MMAs.  Same skeleton as linear_tf32x3.cu without the operand split.
// Warp roles (10 warps): 0-7 epilogue (warp % 4 = TMEM lane quadrant, warp / 4 = which 64-column chunks), 8 MMA issuer,
// 9 TMA producer.
#include <cuda.h>

#include <atomic>

#include "msda_common.cuh"
#include "msda_launch.h"
#include "msda_tc.cuh"
#include "umma.cuh"

namespace msda {

using namespace umma;

constexpr int kLbBM = 128;                 // output rows per tile (TMEM lanes)
constexpr int kLbBN = 256;                 // output columns per tile (TMEM columns of one accumulator)
// K block: 64 bf16 = one 128-byte SWIZZLE_128B row, four stages of 48 KB (default), or 32 bf16 = 64-byte SWIZZLE_64B rows,
// eight stages of 24 KB (-DMSDA_LINEAR_BF16_BK=32: what helped the TF32 kernel is slower here -- 38.2 -> 41.9 us at
// 256 <- 256, 125 -> 131 us at 1024 <- 256)
#ifndef MSDA_LINEAR_BF16_BK
#define MSDA_LINEAR_BF16_BK 64
#endif
constexpr int kLbBK = MSDA_LINEAR_BF16_BK;
constexpr int kLbRowBytes = kLbBK * 2;
constexpr int kLbKSteps = kLbBK / 16;      // tcgen05.mma kind::f16 takes K = 16 per instruction
constexpr int kLbStages = kLbBK == 64 ? 4 : 8;
static_assert(kLbBK == 64 || kLbBK == 32, "K block = one SWIZZLE_128B or SWIZZLE_64B row");
#ifndef MSDA_LINEAR_BF16_CLUSTER
#define MSDA_LINEAR_BF16_CLUSTER 2
#endif
constexpr int kLbCluster = MSDA_LINEAR_BF16_CLUSTER;   // CTAs that share every weight tile (TMA multicast); 1 = none
constexpr int kLbABytes = kLbBM * kLbRowBytes;     // 16 KB
constexpr int kLbBBytes = kLbBN * kLbRowBytes;     // 32 KB
constexpr int kLbStageBytes = kLbABytes + kLbBBytes;
constexpr int kLbEpiThreads = 256;
constexpr int kLbThreads = kLbEpiThreads + 64;
constexpr int kLbOutBytes = 32 * 128;      // one epilogue warp's staging tile: 32 rows x 64 bf16
constexpr int kLbSmem = kLbStages * kLbStageBytes + 8 * kLbOutBytes + kLbBN * 4 + 256;
static_assert(kLbSmem <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");

struct LbBars {
    unsigned long long full[kLbStages], empty[kLbStages], acc_full[2], acc_free[2];
    unsigned tmem_base;
};

// shared-memory matrix descriptor of a K-major operand tile whose rows are one swizzle span (128 or 64 bytes)
__device__ __forceinline__ unsigned long long lb_desc(const void* smem_ptr)
{
    if constexpr (kLbBK == 64) return make_desc_sw128(smem_ptr);
    const unsigned addr = smem_u32(smem_ptr);
    unsigned long long d = 0;
    d |= (unsigned long long)((addr & 0x3FFFF) >> 4);            // start address
    d |= (unsigned long long)1 << 16;                            // leading byte offset (unused for swizzled K-major)
    d |= (unsigned long long)(512 >> 4) << 32;                   // stride between 8-row groups: 8 x 64 bytes
    d |= (unsigned long long)1 << 46;                            // descriptor version (sm_100)
    d |= (unsigned long long)4 << 61;                            // layout: SWIZZLE_64B
    return d;
}

// DROP: dropout after the ReLU, mask of element row * N + col (dropout_keep8: one Philox call per 8 columns a lane packs)
template <bool DROP>
__global__ void __cluster_dims__(kLbCluster, 1, 1) __launch_bounds__(kLbThreads, 1)
linear_bf16_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                   const __grid_constant__ CUtensorMap tm_y, const __nv_bfloat16* __restrict__ bias,
                   const unsigned char* __restrict__ row_mask, long long rows, int N, int K, int relu, int bn,
                   const unsigned long long* __restrict__ drop_key, unsigned drop_thresh, float drop_scale)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* s_out = smem + kLbStages * kLbStageBytes;            // [8 epilogue warps][kLbOutBytes], 1024-byte aligned
    float* s_bias = reinterpret_cast<float*>(s_out + 8 * kLbOutBytes);
    LbBars* bars = reinterpret_cast<LbBars*>(s_out + 8 * kLbOutBytes + kLbBN * 4);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long tiles_m = (rows + kLbBM - 1) / kLbBM;
    // bn: column tile width chosen by the host (<= kLbBN, a multiple of 64 that splits N evenly: 384 -> 2 x 192)
    const int tiles_n = (N + bn - 1) / bn;
    // work unit of a cluster: kLbCluster consecutive row tiles x one column tile; CTA `rank` takes row tile group * C + rank
    // (past the last row tile: TMA reads zeros, the stores are clipped)
    const long long tiles = ((tiles_m + kLbCluster - 1) / kLbCluster) * tiles_n;
    const int kblocks = K / kLbBK;
    const unsigned rank = cluster_ctarank();
    const long long first = blockIdx.x / kLbCluster, stride = gridDim.x / kLbCluster;
    constexpr unsigned short kAll = (unsigned short)((1u << kLbCluster) - 1u);

    if (warp == 0) tmem_alloc(&bars->tmem_base, 512);
    if (tid == kLbEpiThreads) {
        for (int i = 0; i < kLbStages; ++i) {
            mbar_init(&bars->full[i], 1);
            mbar_init(&bars->empty[i], kLbCluster);
        }
        for (int i = 0; i < 2; ++i) { mbar_init(&bars->acc_full[i], 1); mbar_init(&bars->acc_free[i], kLbEpiThreads); }
        fence_mbar_init();
        tma_prefetch_desc(&tm_x); tma_prefetch_desc(&tm_w); tma_prefetch_desc(&tm_y);
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
            const int slice = bn / kLbCluster, slice_bytes = slice * kLbRowBytes;
            for (long long t = first; t < tiles; t += stride) {
                const int m0 = (int)((t / tiles_n) * kLbCluster + rank) * kLbBM, n0 = (int)(t % tiles_n) * bn;
                // (an L2 prefetch of the next unit's x rows was measured: 38.0 -> 40.9 us at 256 <- 256, 96 -> 120 us at
                // 256 <- 1024 -- it only competes with the loads that are needed now)
                for (int kb = 0; kb < kblocks; ++kb, ++kiter) {
                    const int s = kiter % kLbStages;
                    // both CTAs are done with the stage: my slice lands in the peer's shared memory too
                    if (kiter >= kLbStages) mbar_wait(&bars->empty[s], ((kiter / kLbStages) - 1) & 1);
                    unsigned char* st = smem + s * kLbStageBytes;
                    mbar_expect_tx(&bars->full[s], kLbABytes + bn * kLbRowBytes);   // my x tile + every CTA's W slice
                    tma_load_2d(st, &tm_x, kb * kLbBK, m0, &bars->full[s]);
                    tma_load_2d_multicast(st + kLbABytes + rank * slice_bytes, &tm_w, kb * kLbBK, n0 + (int)rank * slice,
                                          &bars->full[s], kAll);
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
            const unsigned idesc = make_idesc_bf16(kLbBM, n_cur);
            const int buf = it & 1;
            const unsigned acc = tmem + buf * kLbBN;
            if (it >= 2) mbar_wait(&bars->acc_free[buf], ((it >> 1) - 1) & 1);     // the epilogue has drained this accumulator
            for (int kb = 0; kb < kblocks; ++kb, ++kiter) {
                const int s = kiter % kLbStages;
                mbar_wait(&bars->full[s], (kiter / kLbStages) & 1);
                tcgen05_fence_after();
                if (elect_one()) {
                    unsigned char* st = smem + s * kLbStageBytes;
                    const unsigned long long d_x = lb_desc(st), d_w = lb_desc(st + kLbABytes);
#pragma unroll
                    for (int j = 0; j < kLbKSteps; ++j)                          // K = 16 per instruction: 32 bytes of the row
                        mma_bf16(acc, desc_advance(d_x, j * 32), desc_advance(d_w, j * 32), idesc, (kb | j) != 0);
                    mma_commit_multicast(&bars->empty[s], kAll);                 // stage free, here and in the peer
                    if (kb == kblocks - 1) mma_commit(&bars->acc_full[buf]);
                }
                __syncwarp();
            }
        }
    } else {
        // ======================================= epilogue warps =======================================
        // two warps per TMEM lane quadrant: warps 0-3 take the even 64-column chunks, warps 4-7 the odd ones
        const int quad = warp & 3, half = warp >> 2;
        const unsigned lane_base = (unsigned)(quad * 32) << 16;
        unsigned long long key = 0;
        if constexpr (DROP) key = *drop_key;
        unsigned it = 0;
        for (long long t = first; t < tiles; t += stride, ++it) {
            const long long m0 = ((t / tiles_n) * kLbCluster + rank) * kLbBM;
            const int n0 = (int)(t % tiles_n) * bn;
            const int n_cur = min(bn, N - n0);
            const int buf = it & 1;
            // bias slice of the tile (the previous tile's readers are past their last read: barrier below)
            named_bar_sync(1, kLbEpiThreads);
            for (int i = tid; i < kLbBN; i += kLbEpiThreads)
                s_bias[i] = (bias != nullptr && i < n_cur) ? __bfloat162float(bias[n0 + i]) : 0.f;
            named_bar_sync(1, kLbEpiThreads);
            const long long row = m0 + quad * 32 + lane;
            const bool dead = row_mask != nullptr && row < rows && row_mask[row] != 0;     // padding row: zeros
            mbar_wait(&bars->acc_full[buf], (it >> 1) & 1);
            tcgen05_fence_after();
            // 32 rows x 64 columns at a time: TMEM -> registers (lane = row) -> this warp's staging tile in the SWIZZLE_128B
            // layout (16-byte chunk c of row r at chunk c ^ (r & 7)) -> one TMA store of the box
            unsigned char* stage = s_out + (half * 4 + quad) * kLbOutBytes;
            for (int c = half * 64; c < n_cur; c += 128) {
                float v[64];
                tmem_ld32(tmem + buf * kLbBN + c + lane_base, v);
                tmem_ld32(tmem + buf * kLbBN + c + 32 + lane_base, v + 32);
                if (lane == 0) tma_store_wait_read();
                __syncwarp();
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    float o[8];
                    unsigned bits = 0;
                    if constexpr (DROP)
                        bits = dropout_keep8((unsigned long long)(row * N + n0 + c + 8 * q) >> 3, key, drop_thresh);
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        o[e] = v[8 * q + e] + s_bias[c + 8 * q + e];
                        if (relu) o[e] = fmaxf(o[e], 0.f);
                        if constexpr (DROP) o[e] *= (bits >> e) & 1u ? drop_scale : 0.f;
                        if (dead) o[e] = 0.f;
                    }
                    *reinterpret_cast<uint4*>(stage + lane * 128 + ((q ^ (lane & 7)) << 4)) = pack<__nv_bfloat16>(o);
                }
                fence_proxy_async();                 // generic-proxy writes -> TMA (async proxy) read
                __syncwarp();
                if (lane == 0) {
                    tma_store_2d(&tm_y, stage, n0 + c, (int)m0 + quad * 32);
                    tma_store_commit();
                }
            }
            tcgen05_fence_before();
            mbar_arrive(&bars->acc_free[buf]);
        }
        if (lane == 0) tma_store_wait_all();         // my stores have left shared memory
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                            // no CTA leaves while a peer may still write its shared memory / barriers
    if (warp == 0) tmem_free(tmem, 512);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*LbEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static LbEncodeTiledFn lb_encode_tiled_fn()
{
    static LbEncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<LbEncodeTiledFn>(p);
    }
    return fn;
}

// row-major bf16 matrix [n_rows, n_cols]; box = 64 columns (128 bytes, SWIZZLE_128B) x box_rows rows
static bool lb_make_map(CUtensorMap* map, const void* base, unsigned long long n_rows, unsigned long long n_cols, int box_rows,
                        int box_cols = kLbBK)
{
    LbEncodeTiledFn fn = lb_encode_tiled_fn();
    if (fn == nullptr) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)n_cols, n_rows};
    const cuuint64_t strides[1] = {(cuuint64_t)n_cols * 2};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
              CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool linear_bf16_supported(int n, int k)
{
    return n >= 64 && n % 64 == 0 && k >= 64 && k % 64 == 0;
}

template <bool DROP>
static cudaError_t launch_linear_bf16(const void* x, const void* w, const void* bias, const unsigned char* row_mask,
                                      long long rows, int n, int k, int relu, const unsigned long long* key,
                                      DropoutRule rule, void* y, cudaStream_t stream)
{
    if (!linear_bf16_supported(n, k) || rows < 0 || rows >= (1ll << 31) - 1024) return cudaErrorInvalidValue;
    if (rows == 0) return cudaSuccess;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(y)) % 16 != 0)
        return cudaErrorInvalidValue;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    static bool configured[64] = {};          // the attribute is per device: one process may drive several GPUs
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(linear_bf16_kernel<DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLbSmem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    // column tile width: as few tiles as 256 columns allow, of equal width (a multiple of 64; each CTA of the cluster
    // loads bn / 2 weight rows, a multiple of the 8-row swizzle group)
    const int tiles_n = (n + kLbBN - 1) / kLbBN;
    const int bn = ((n + tiles_n - 1) / tiles_n + 63) / 64 * 64;
    alignas(64) CUtensorMap tm_x, tm_w, tm_y;
    if (!lb_make_map(&tm_x, x, (unsigned long long)rows, (unsigned long long)k, kLbBM) ||
        !lb_make_map(&tm_w, w, (unsigned long long)n, (unsigned long long)k, bn / kLbCluster) ||
        !lb_make_map(&tm_y, y, (unsigned long long)rows, (unsigned long long)n, 32, 64))
        return cudaErrorNotSupported;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long tiles_m = (rows + kLbBM - 1) / kLbBM;
    const long long units = ((tiles_m + kLbCluster - 1) / kLbCluster) * ((n + bn - 1) / bn);
    const long long clusters = sms / kLbCluster;
    const int grid = (int)(units < clusters ? units : clusters) * kLbCluster;
    linear_bf16_kernel<DROP><<<grid, kLbThreads, kLbSmem, stream>>>(tm_x, tm_w, tm_y, (const __nv_bfloat16*)bias, row_mask, rows,
                                                                     n, k, relu, bn, key, rule.thresh, rule.scale);
    return cudaGetLastError();
}

cudaError_t linear_bf16(const void* x, const void* w, const void* bias, const unsigned char* row_mask, long long rows, int n,
                        int k, int relu, void* y, cudaStream_t stream)
{
    return launch_linear_bf16<false>(x, w, bias, row_mask, rows, n, k, relu, nullptr, DropoutRule{0u, 1.f}, y, stream);
}

cudaError_t linear_bf16_relu_dropout(const void* x, const void* w, const void* bias, long long rows, int n, int k,
                                     const unsigned long long* key, DropoutRule rule, void* y, cudaStream_t stream)
{
    if (key == nullptr) return cudaErrorInvalidValue;
    return launch_linear_bf16<true>(x, w, bias, nullptr, rows, n, k, 1, key, rule, y, stream);
}

// ------------------------------------------------------------------------------------------
// weight / bias gradient of the same layer (training):
//
//     dW [N, K] = g^T x,   db [N] = sum over rows of g,   g [rows, N], x [rows, K], bf16, fp32 accumulation.
//
// The reduction runs over `rows`, so both operands are MN-major: a TMA box {64 columns, 64 rows} with SWIZZLE_128B lands
// as 64 rows of 128 bytes = the MN-major SWIZZLE_128B image of 64 output features (or inputs) x 64 reduction steps.  An
// output tile is 128 features (two g boxes, M) x up to 256 inputs (four x boxes, N).  There are only 2-8 such tiles at
// the model's shapes, so `rows` is split into contiguous slices (split-K), about one CTA per SM: each CTA accumulates its
// slice in TMEM and writes the fp32 partial tile to `scratch`; a second kernel sums the partials in split order (the
// result does not depend on scheduling) and rounds to bf16.  The bias gradient comes from the same g tiles: CTAs of
// column tile 0 issue one more M = 128, N = 16 MMA per K step against a constant all-ones K-major B tile, which puts
// sum_rows g of their 128 features into 16 extra TMEM columns (all equal; column 0 is kept) -- g is read once.
// Warp roles (6 warps): 0-3 epilogue (warp = TMEM lane quadrant), 4 MMA issuer, 5 TMA producer.
// ------------------------------------------------------------------------------------------
constexpr int kWgBM = 128;                  // output features per tile (TMEM lanes)
constexpr int kWgBN = 256;                  // inputs per tile (TMEM columns)
constexpr int kWgBK = 64;                   // rows per K block
constexpr int kWgBox = 64 * kWgBK * 2;      // one {64 columns, 64 rows} bf16 box: 8 KB
constexpr int kWgStageBytes = (kWgBM / 64 + kWgBN / 64) * kWgBox;   // 2 g boxes + 4 x boxes: 48 KB
constexpr int kWgStages = 4;
constexpr int kWgOnesBytes = 16 * 128;      // all-ones B tile of the bias MMA: 16 rows x 64 bf16
constexpr int kWgDbCol = kWgBN;             // TMEM column of the bias accumulator
constexpr int kWgEpiThreads = 128;
constexpr int kWgThreads = kWgEpiThreads + 64;
constexpr int kWgSmem = kWgStages * kWgStageBytes + kWgOnesBytes + 256 + 1024;   // + barriers + alignment slack
static_assert(kWgSmem <= 232448, "exceeds the 227 KB of shared memory a CTA can opt in to");
constexpr int kWgTargetCtas = 148;          // B200 SMs: split count aimed at one CTA per SM, fixed so that the split (and
                                            // so the rounding of the result) does not depend on the device
constexpr int kWgMinKBlocks = 4;            // a split reads at least 256 rows: its partial tile is small against its loads

struct WgBars {
    unsigned long long full[kWgStages], empty[kWgStages], acc_full;
    unsigned tmem_base;
};

__global__ void __launch_bounds__(kWgThreads, 1)
linear_bf16_wgrad_kernel(const __grid_constant__ CUtensorMap tm_g, const __grid_constant__ CUtensorMap tm_x,
                         float* __restrict__ partial, long long rows, int N, int K, int bn, int tiles_n, int tiles,
                         int splits, int kb_per_split, long long blk_floats, int want_db)
{
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* s_ones = smem + kWgStages * kWgStageBytes;          // 1024-byte aligned
    WgBars* bars = reinterpret_cast<WgBars*>(s_ones + kWgOnesBytes);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // CTAs of one split (same rows) are adjacent: the tiles that share a slice of g or x read it from L2
    const int split = blockIdx.x / tiles, t = blockIdx.x % tiles;
    const int m0 = (t / tiles_n) * kWgBM, n0 = (t % tiles_n) * bn;
    const int n_cur = min(bn, K - n0);
    const int kblocks = (int)((rows + kWgBK - 1) / kWgBK);
    const int kb0 = split * kb_per_split, kb1 = min(kb0 + kb_per_split, kblocks);
    const bool with_db = want_db && n0 == 0;

    if (warp == 0) tmem_alloc(&bars->tmem_base, 512);
    for (int i = tid; i < kWgOnesBytes / 16; i += kWgThreads)            // bf16 1.0 = 0x3f80
        reinterpret_cast<uint4*>(s_ones)[i] = make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);
    fence_proxy_async();                                                // generic writes -> tensor-core reads
    if (tid == kWgEpiThreads) {
        for (int i = 0; i < kWgStages; ++i) { mbar_init(&bars->full[i], 1); mbar_init(&bars->empty[i], 1); }
        mbar_init(&bars->acc_full, 1);
        fence_mbar_init();
        tma_prefetch_desc(&tm_g); tma_prefetch_desc(&tm_x);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const unsigned tmem = bars->tmem_base;

    if (warp == 5) {
        // ======================================= TMA producer =======================================
        if (elect_one()) {
            // boxes wholly past the last feature / input are not loaded: they only feed accumulator lanes / columns
            // that are never read.  Rows past the end arrive as zeros (TMA out-of-bounds fill).
            const int g_boxes = min(kWgBM, N - m0) / 64, x_boxes = n_cur / 64;
            const unsigned bytes = (unsigned)(g_boxes + x_boxes) * kWgBox;
            for (int kb = kb0; kb < kb1; ++kb) {
                const int i = kb - kb0, s = i % kWgStages;
                if (i >= kWgStages) mbar_wait(&bars->empty[s], ((i / kWgStages) - 1) & 1);
                unsigned char* st = smem + s * kWgStageBytes;
                mbar_expect_tx(&bars->full[s], bytes);
                for (int c = 0; c < g_boxes; ++c) tma_load_2d(st + c * kWgBox, &tm_g, m0 + 64 * c, kb * kWgBK, &bars->full[s]);
                for (int c = 0; c < x_boxes; ++c)
                    tma_load_2d(st + (kWgBM / 64 + c) * kWgBox, &tm_x, n0 + 64 * c, kb * kWgBK, &bars->full[s]);
            }
        }
        __syncwarp();
    } else if (warp == 4) {
        // ======================================= MMA issuer =======================================
        // A = g^T (M = 128 features, MN-major), B = x (N = inputs, MN-major): leading byte offset = distance between the
        // 64-element boxes along M / N, stride byte offset = 8 rows of 128 bytes; one K = 16 step = 16 rows = 2048 bytes
        const unsigned idesc = tc::make_idesc(kWgBM, n_cur, 1, 1);
        const unsigned idesc_db = tc::make_idesc(kWgBM, 16, 1, 0);
        const unsigned long long d_ones = make_desc_sw128(s_ones);
        for (int kb = kb0; kb < kb1; ++kb) {
            const int i = kb - kb0, s = i % kWgStages;
            mbar_wait(&bars->full[s], (i / kWgStages) & 1);
            tcgen05_fence_after();
            if (elect_one()) {
                unsigned char* st = smem + s * kWgStageBytes;
                const unsigned long long d_g = tc::make_desc(st, kWgBox, 1024, 2);
                const unsigned long long d_x = tc::make_desc(st + (kWgBM / 64) * kWgBox, kWgBox, 1024, 2);
#pragma unroll
                for (int j = 0; j < kWgBK / 16; ++j) {
                    mma_bf16(tmem, desc_advance(d_g, j * 2048), desc_advance(d_x, j * 2048), idesc, (i | j) != 0);
                    if (with_db) mma_bf16(tmem + kWgDbCol, desc_advance(d_g, j * 2048), desc_advance(d_ones, j * 32), idesc_db,
                                          (i | j) != 0);
                }
                mma_commit(&bars->empty[s]);                                 // stage free once these MMAs are done
                if (kb == kb1 - 1) mma_commit(&bars->acc_full);
            }
            __syncwarp();
        }
    } else {
        // ======================================= epilogue warps =======================================
        // TMEM lane = feature row of the tile -> this CTA's fp32 partial block [128][bn] (+ [128] bias partial)
        const unsigned lane_base = (unsigned)(warp * 32) << 16;
        const int r = warp * 32 + lane;
        float* blk = partial + ((long long)t * splits + split) * blk_floats;
        mbar_wait(&bars->acc_full, 0);
        tcgen05_fence_after();
        for (int c = 0; c < n_cur; c += 32) {
            float v[32];
            tmem_ld32(tmem + c + lane_base, v);
            float4* dst = reinterpret_cast<float4*>(blk + (long long)r * bn + c);
#pragma unroll
            for (int q = 0; q < 8; ++q) dst[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
        if (with_db) {
            float v[16];
            tmem_ld16(tmem + kWgDbCol + lane_base, v);
            blk[(long long)kWgBM * bn + r] = v[0];
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 512);
}

// dW / db = sum over the splits of the partial blocks, in split order, rounded to bf16.  Block (32, 8): x = 4 consecutive
// outputs, y = every 8th split; the 8 sums are added in y order.
__global__ void __launch_bounds__(256)
linear_bf16_wgrad_reduce_kernel(const float* __restrict__ partial, __nv_bfloat16* __restrict__ dw, __nv_bfloat16* __restrict__ db,
                                int N, int K, int bn, int tiles_n, int splits, long long blk_floats)
{
    __shared__ float4 s_sum[8][32];
    const long long q = (long long)blockIdx.x * 32 + threadIdx.x;        // quad of outputs
    const long long qw = (long long)N * K / 4, qb = db != nullptr ? N / 4 : 0;
    long long base = -1, dst = 0;
    if (q < qw) {
        const long long e = q * 4;
        const int o = (int)(e / K), i = (int)(e % K);
        base = ((long long)((o / kWgBM) * tiles_n + i / bn) * splits) * blk_floats + (long long)(o % kWgBM) * bn + i % bn;
        dst = e;
    } else if (q < qw + qb) {
        const int o = (int)(q - qw) * 4;
        base = ((long long)((o / kWgBM) * tiles_n) * splits) * blk_floats + (long long)kWgBM * bn + o % kWgBM;
        dst = o;
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (base >= 0)
        for (int s = threadIdx.y; s < splits; s += 8) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(partial + base + (long long)s * blk_floats));
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
    __nv_bfloat162 lo = __floats2bfloat162_rn(acc.x, acc.y), hi = __floats2bfloat162_rn(acc.z, acc.w);
    uint2 packed;
    packed.x = *reinterpret_cast<unsigned*>(&lo);
    packed.y = *reinterpret_cast<unsigned*>(&hi);
    *reinterpret_cast<uint2*>((q < qw ? dw : db) + dst) = packed;
}

bool linear_bf16_wgrad_supported(int n, int k)
{
    return n >= 64 && n % 64 == 0 && k >= 64 && k % 64 == 0;
}

struct WgPlan {
    int bn, tiles_n, tiles, splits, kb_per_split;
    long long blk_floats;
};

static bool wgrad_plan(long long rows, int n, int k, WgPlan* p)
{
    if (!linear_bf16_wgrad_supported(n, k) || rows < 1 || rows >= (1ll << 31) - 1024) return false;
    p->tiles_n = (k + kWgBN - 1) / kWgBN;
    p->bn = ((k + p->tiles_n - 1) / p->tiles_n + 63) / 64 * 64;         // equal column tiles, multiples of 64
    p->tiles = ((n + kWgBM - 1) / kWgBM) * p->tiles_n;
    const int kblocks = (int)((rows + kWgBK - 1) / kWgBK);
    const int want = max(1, kWgTargetCtas / p->tiles);
    p->kb_per_split = max(kWgMinKBlocks, (kblocks + want - 1) / want);
    p->splits = (kblocks + p->kb_per_split - 1) / p->kb_per_split;     // every split has at least one K block
    p->blk_floats = (long long)kWgBM * p->bn + kWgBM;
    return true;
}

long long linear_bf16_wgrad_scratch_floats(long long rows, int n, int k)
{
    WgPlan p;
    return wgrad_plan(rows, n, k, &p) ? (long long)p.tiles * p.splits * p.blk_floats : 0;
}

cudaError_t linear_bf16_wgrad(const void* g, const void* x, long long rows, int n, int k, void* dw, void* db,
                              float* scratch, long long scratch_floats, cudaStream_t stream)
{
    WgPlan p;
    if (!wgrad_plan(rows, n, k, &p) || scratch_floats < (long long)p.tiles * p.splits * p.blk_floats || dw == nullptr)
        return cudaErrorInvalidValue;
    if ((reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dw) |
         reinterpret_cast<uintptr_t>(db) | reinterpret_cast<uintptr_t>(scratch)) % 16 != 0)
        return cudaErrorInvalidValue;
    int dev = 0;
    cudaGetDevice(&dev);
    // the attribute is per device; concurrent first calls may both set it (harmless), none reads a torn flag
    static std::atomic<bool> configured[64];
    if (dev < 0 || dev >= 64 || !configured[dev].load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(linear_bf16_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev].store(true, std::memory_order_release);
    }
    alignas(64) CUtensorMap tm_g, tm_x;
    if (!lb_make_map(&tm_g, g, (unsigned long long)rows, (unsigned long long)n, kWgBK) ||
        !lb_make_map(&tm_x, x, (unsigned long long)rows, (unsigned long long)k, kWgBK))
        return cudaErrorNotSupported;
    linear_bf16_wgrad_kernel<<<p.tiles * p.splits, kWgThreads, kWgSmem, stream>>>(
        tm_g, tm_x, scratch, rows, n, k, p.bn, p.tiles_n, p.tiles, p.splits, p.kb_per_split, p.blk_floats, db != nullptr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const long long quads = (long long)n * k / 4 + (db != nullptr ? n / 4 : 0);
    linear_bf16_wgrad_reduce_kernel<<<(unsigned)((quads + 31) / 32), dim3(32, 8), 0, stream>>>(
        scratch, (__nv_bfloat16*)dw, (__nv_bfloat16*)db, n, k, p.bn, p.tiles_n, p.splits, p.blk_floats);
    return cudaGetLastError();
}

}  // namespace msda
