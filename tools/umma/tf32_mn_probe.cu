// Probe: does tcgen05.mma kind::tf32 take MN-major operands, and with which descriptor encoding?
//
// The fp32 weight-gradient kernel (csrc/linear_tf32x3.cu, linear_tf32x3_wgrad_kernel) multiplies g^T [features, rows] by
// x [rows, inputs] with the reduction over rows, so both operands are MN-major in shared memory: a TMA box {32 fp32
// columns, 32 rows} with SWIZZLE_128B is 32 rows of 128 bytes = 32 features x 32 reduction steps.  This probe loads
// g [32 rows, 128] and x [32 rows, 128] that way (four boxes each, 4 KB apart), issues four K = 8 MMAs (M = 128,
// N = 128, transpose bits set), and compares D with a CPU product of the TF32-truncated inputs for several
// (leading, stride) byte-offset encodings.  A control loads the same operands K-major (transposed on the host: g^T
// [128, 32] and x^T [128, 32], box {32 columns, 128 rows}, the layout of the forward kernel) and issues the MMAs without
// the transpose bits.  Build and run:
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -std=c++17 -I<pkg>/csrc tools/umma/tf32_mn_probe.cu -o probe && ./probe
#include <cuda.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "umma.cuh"

using namespace umma;

constexpr int kRows = 32, kM = 128, kN = 128, kBox = 32 * kRows * 4;

__device__ __forceinline__ unsigned long long desc_mn(const void* p, unsigned lbo, unsigned sbo)
{
    const unsigned addr = smem_u32(p);
    unsigned long long d = 0;
    d |= (unsigned long long)((addr & 0x3FFFF) >> 4);
    d |= (unsigned long long)((lbo >> 4) & 0x3FFF) << 16;
    d |= (unsigned long long)((sbo >> 4) & 0x3FFF) << 32;
    d |= (unsigned long long)1 << 46;
    d |= (unsigned long long)2 << 61;                       // SWIZZLE_128B
    return d;
}

__global__ void probe_kernel(const __grid_constant__ CUtensorMap tm_g, const __grid_constant__ CUtensorMap tm_x, float* d,
                             unsigned lbo, unsigned sbo, unsigned kstep, int kmajor)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(smem + 8 * kBox);
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(smem + 8 * kBox + 64);
    const int warp = threadIdx.x >> 5;
    if (warp == 0) tmem_alloc(tmem_slot, 128);
    if (threadIdx.x == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); fence_mbar_init(); }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const unsigned tmem = *tmem_slot;
    if (threadIdx.x == 0) {
        mbar_expect_tx(&bar[0], 8 * kBox);
        if (kmajor) {                                       // [128 rows, 32 fp32] each: one box of 128 rows
            tma_load_2d(smem, &tm_g, 0, 0, &bar[0]);
            tma_load_2d(smem + 4 * kBox, &tm_x, 0, 0, &bar[0]);
        } else {
            for (int c = 0; c < 4; ++c) {
                tma_load_2d(smem + c * kBox, &tm_g, 32 * c, 0, &bar[0]);
                tma_load_2d(smem + (4 + c) * kBox, &tm_x, 32 * c, 0, &bar[0]);
            }
        }
    }
    if (warp == 0) {
        mbar_wait(&bar[0], 0);
        tcgen05_fence_after();
        if (elect_one()) {
            // kind::tf32 (A / B format 2), D fp32, transpose A and B (MN-major)
            const unsigned transpose = kmajor ? 0u : (1u << 15) | (1u << 16);
            const unsigned idesc = (1u << 4) | (2u << 7) | (2u << 10) | transpose | ((unsigned)(kN >> 3) << 17) |
                                   ((unsigned)(kM >> 4) << 24);
            const unsigned long long da = desc_mn(smem, lbo, sbo), db = desc_mn(smem + 4 * kBox, lbo, sbo);
            for (int j = 0; j < kRows / 8; ++j) {
                const unsigned long long a = desc_advance(da, j * kstep), b = desc_advance(db, j * kstep);
                asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                             "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
                             :: "r"(tmem), "l"(a), "l"(b), "r"(idesc), "r"((unsigned)(j != 0)) : "memory");
            }
            mma_commit(&bar[1]);
        }
        __syncwarp();
    }
    mbar_wait(&bar[1], 0);
    tcgen05_fence_after();
    const int lane_row = (warp & 3) * 32 + (threadIdx.x & 31);
    for (int c = 0; c < kN; c += 32) {
        float v[32];
        tmem_ld32(tmem + c + ((unsigned)((warp & 3) * 32) << 16), v);
        for (int i = 0; i < 32; ++i) d[lane_row * kN + c + i] = v[i];
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) tmem_free(tmem, 128);
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static float tf32_trunc(float v)
{
    unsigned u;
    memcpy(&u, &v, 4);
    u &= 0xffffe000u;
    memcpy(&v, &u, 4);
    return v;
}

int main()
{
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &q) != cudaSuccess) return 1;
    EncodeFn encode = reinterpret_cast<EncodeFn>(fp);
    std::vector<float> g(kRows * kM), x(kRows * kN);
    unsigned s = 12345u;
    auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (float)((s >> 8) & 0xffff) / 32768.f - 1.f; };
    for (auto& v : g) v = rnd();
    for (auto& v : x) v = rnd();
    // reference: D[m][n] = sum_r trunc(g[r][m]) trunc(x[r][n]) in double
    std::vector<double> ref(kM * kN, 0.0);
    double ref_max = 0;
    for (int m = 0; m < kM; ++m)
        for (int n = 0; n < kN; ++n) {
            double acc = 0;
            for (int r = 0; r < kRows; ++r) acc += (double)tf32_trunc(g[r * kM + m]) * (double)tf32_trunc(x[r * kN + n]);
            ref[m * kN + n] = acc;
            ref_max = fmax(ref_max, fabs(acc));
        }
    float *dg, *dx, *dd;
    cudaMalloc(&dg, g.size() * 4);
    cudaMalloc(&dx, x.size() * 4);
    cudaMalloc(&dd, kM * kN * 4);
    cudaMemcpy(dg, g.data(), g.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dx, x.data(), x.size() * 4, cudaMemcpyHostToDevice);
    alignas(64) CUtensorMap tm_g, tm_x;
    const cuuint64_t dims_g[2] = {kM, kRows}, dims_x[2] = {kN, kRows};
    const cuuint64_t str_g[1] = {kM * 4}, str_x[1] = {kN * 4};
    const cuuint32_t box[2] = {32, kRows}, estr[2] = {1, 1};
    CUresult e1 = encode(&tm_g, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dg, dims_g, str_g, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult e2 = encode(&tm_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dx, dims_x, str_x, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    // K-major control: g^T [128, 32] and x^T [128, 32] row-major
    std::vector<float> gt(kM * kRows), xt(kN * kRows);
    for (int r = 0; r < kRows; ++r) {
        for (int m = 0; m < kM; ++m) gt[m * kRows + r] = g[r * kM + m];
        for (int n = 0; n < kN; ++n) xt[n * kRows + r] = x[r * kN + n];
    }
    float *dgt, *dxt;
    cudaMalloc(&dgt, gt.size() * 4);
    cudaMalloc(&dxt, xt.size() * 4);
    cudaMemcpy(dgt, gt.data(), gt.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dxt, xt.data(), xt.size() * 4, cudaMemcpyHostToDevice);
    alignas(64) CUtensorMap tm_gt, tm_xt;
    const cuuint64_t dims_t[2] = {kRows, 128}, str_t[1] = {kRows * 4};
    const cuuint32_t box_t[2] = {32, 128};
    CUresult e3 = encode(&tm_gt, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dgt, dims_t, str_t, box_t, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult e4 = encode(&tm_xt, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dxt, dims_t, str_t, box_t, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    printf("tensor map encode: %d %d %d %d\n", (int)e1, (int)e2, (int)e3, (int)e4);
    const int smem = 8 * kBox + 128;
    cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    struct Variant { unsigned lbo, sbo, kstep; int kmajor; const char* what; };
    const Variant variants[] = {
        {kBox, 1024, 1024, 0, "MN-major, LBO = 4096 (next 32 along M/N), SBO = 1024 (next 8 rows), K step 1024 B"},
        {1024, kBox, 1024, 0, "MN-major, LBO = 1024, SBO = 4096 (swapped)"},
        {16, 1024, 1024, 0, "MN-major, LBO = 16 (unused), SBO = 1024"},
        {16, 1024, 32, 1, "K-major control (host-transposed operands, no transpose bits), SBO = 1024, K step 32 B"},
    };
    std::vector<float> d(kM * kN);
    for (const Variant& v : variants) {
        cudaMemset(dd, 0, kM * kN * 4);
        probe_kernel<<<1, 128, smem>>>(v.kmajor ? tm_gt : tm_g, v.kmajor ? tm_xt : tm_x, dd, v.lbo, v.sbo, v.kstep, v.kmajor);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { printf("%s: %s\n", v.what, cudaGetErrorString(e)); return 1; }
        cudaMemcpy(d.data(), dd, kM * kN * 4, cudaMemcpyDeviceToHost);
        double err = 0, dmax = 0;
        for (int i = 0; i < kM * kN; ++i) {
            const double e = fabs((double)d[i] - ref[i]);
            err = e > err || e != e ? e : err;                      // a NaN counts as an error
            dmax = fmax(dmax, fabs((double)d[i]));
        }
        printf("%s: max|err| %.3e max|ref| %.3e max|D| %.3e -> %s\n", v.what, err, ref_max, dmax,
               err <= 1e-5 * ref_max ? "EXACT" : "mismatch");
    }
    return 0;
}
