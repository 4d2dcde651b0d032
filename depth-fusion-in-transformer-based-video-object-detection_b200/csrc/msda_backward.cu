// Backward multi-scale deformable attention for sm_100a.
//
//   grad_value[n, pix, m, :] += w_corner * A * g            (scatter over the 4 corners)
//   grad_attn [n,q,m,l,p]     = sum_c g_c * bilinear_c
//   grad_loc  [n,q,m,l,p]     = ( W * A * sum_c g_c * d bilinear_c / dx ,
//                                 H * A * sum_c g_c * d bilinear_c / dy )
//
// Replaces the reference's six col2im kernels + switch(channels) (cuda/ms_deform_im2col_cuda.cuh:
// 301-920, 956-1327; helper :87-159).  The production reference kernel for D=32 runs one
// 32-thread block per (n,q,m), issues 4 scalar atomicAdd per channel per sample, and reduces
// grad_loc / grad_attn through shared memory with thread 0 summing serially between two
// __syncthreads per sample (:376-394).
//
// Fast kernel (same lane mapping as the forward: a group of G lanes owns a pair, each lane a
// 16-byte channel slice):
//   * phase 1: one lane per sample computes the footprint ONCE and parks what phase 2 needs in shared memory (48 bytes per
//     sample): the four corner-row byte offsets (corners outside the map clamped to a harmless in-range row), the
//     grad_value coefficient of each row, and (lw, lh, a, corner mask);
//   * phase 2, per sample and lane: 4 unconditional loads, 8 packed FMAs for the corner dot products
//     t_k = <grad_output, value_k>, which give all three gradients of the sample (the sums of cuh:113-158 with the
//     channel sum taken first):
//         grad_attn   = sum_k ca_k t_k      ca = (hh*hw, hh*lw, lh*hw, lh*lw)
//         grad_loc.x ~ a * (hh (t1 - t0) + lh (t3 - t2)),   grad_loc.y ~ a * (hw (t2 - t0) + lw (t3 - t1))
//     then the cross-lane sums (a reduce-scatter over four samples at a time for the plain op) and 4 predicated
//     reductions -- ~100 instructions where the round-1 kernel needed 164 (64-bit address arithmetic per corner,
//     zero-filled predicated loads, branches around every reduction);
//   * grad_value uses ONE 16-byte vector reduction (red.global.add.v4.f32 -> REDG.E.ADD.F32x4)
//     per lane per corner instead of 4 scalar atomics, always into an fp32 buffer.  A lane
//     always owns 4 channels here (16-bit values are read with 8-byte loads) so that the 8 lanes
//     of a group cover one whole 128-byte fp32 row per instruction: measured on B200, the
//     SM->L2 reduction path costs ~5.5 cycles per (instruction, row) whether the row is written
//     whole or in halves (tools/microbench_red.cu), and it is what bounds this kernel;
//   * grad_loc / grad_attn are written for every sample (zeros for samples outside the map),
//     so they need no zero-fill pass; only grad_value is memset.
// Generic kernel: any D / dtype (fp64 for gradcheck): one warp per pair, lanes stride channels.
#include <type_traits>
#include "msda_common.cuh"
#include "msda_launch.h"

namespace msda {

template <int PAIRS> struct BwdWarps { static constexpr int value = PAIRS >= 16 ? 2 : (PAIRS >= 8 ? 4 : 8); };

// resident CTAs per SM the register allocation must allow.  Measured on B200 (tools/ab_variants.sh,
// fp32 / bf16 backward, batch 8): 2 x 8 warps at 128 registers 1.90 / 1.88 ms; 3 x 8 warps at 80
// registers 1.74 / 1.76 ms; 4 x 8 warps at 64 registers (immediate reduction, no spills) 1.70 / 1.75 ms.
#ifndef MSDA_BWD_MINBLOCKS
#define MSDA_BWD_MINBLOCKS 4
#endif
#ifndef MSDA_CTA_PER_HEAD      // see msda_forward.cu
#define MSDA_CTA_PER_HEAD 1
#endif

// Where the per-sample gradients go.  Plain: grad_sampling_loc / grad_attn_weight.  Fused:
// gradients w.r.t. the raw projection outputs (through the location arithmetic and the softmax)
// and, optionally, w.r.t. the reference points.
struct GradDst {
    void* loc;        // plain: grad_loc [pairs,LP,2] fp32 ; fused: grad_offsets (addressing of SampleSrc)
    void* attn;       // plain: grad_attn [pairs,LP] fp32  ; fused: grad_logits
    float* ref;       // fused: grad_ref [N*Lq, L, ref_dim] or nullptr
};

// FUSED: see msda_forward.cu.  Backward of the fused layer op additionally applies
//   d loc / d offset  (1/W, 1/H  or  0.5*wh/P)           reference modules/ms_deform_attn.py:102-110
//   softmax backward   g_logit = a * (g_a - sum_j a_j g_a_j)                      :99-100
// to the finished per-sample gradients in phase 3, so neither the locations / weights nor their
// gradients ever exist in HBM.
// Samples per pass.  8 (instead of the forward's 16) halves the per-lane partial-sum registers
// (3 per sample) and lets a lane keep its own samples' weights in registers between phases: the
// kernel is bound by load latency under RED traffic (ncu: long-scoreboard stalls, 15 resident
// warps at 128 registers), so registers buy resident warps.  3*CH must be divisible by G.
#ifndef MSDA_BWD_CHUNK
#define MSDA_BWD_CHUNK 8
#endif
// 1: before the reductions leave the SM, merge the corner rows that several samples of one (query, head, level)
// share.  Every sample of a pair scatters coefficient * grad_output[pair] -- the SAME row -- so samples that touch the
// same pixel need one reduction of the summed coefficient.  With the encoder's geometry (points a pixel apart along the
// head's direction) 17 % of the corner rows are such duplicates (28 % at initialisation, where the offsets are exact
// integers and half the bilinear weights are exactly zero -- zero-coefficient rows are dropped as well).  The kernel is
// bound by the SM -> L2 reduction path (5.5 cycles per row), so rows saved are time saved; the price is 7 shuffles and
// ~50 ALU instructions per lane, pass and point distance in phase 1.  Only for one sample per lane per pass (head
// width >= 32).  Merging ACROSS queries needs the rows themselves moved between lanes: measured, it costs more L1
// data-pipe wavefronts than the reduction rows it saves (tools/experiments/msda_backward_cta_merge.cu).
#ifndef MSDA_BWD_DEDUP
#define MSDA_BWD_DEDUP 1
#endif

// 1: the fused kernel's passes run as a real loop instead of FCH unrolled copies.  Unrolled, the D = 32 bf16 kernel is
// 4832 instructions (77 KB of SASS) that every warp walks end to end, and ncu shows 14 % of its stall samples waiting for
// instructions (`no_instructions`, profiles/ncu_r1k.json); the per-pass register arrays are then indexed through
// reg_pick / reg_put (selects over a static index) so that they stay in registers.
// 1: phase 1 parks the three coefficient vectors (ca, cx, cy: 48 bytes per sample) that turn the corner dots into the
// sample's gradients; 0: it parks (lw, lh, a, corner mask) -- 16 bytes -- and phase 2 rebuilds the combination (about 15
// more instructions per sample, 2 shared-memory wavefronts fewer: the L1 data pipe is the busier unit, ncu r2c).
#ifndef MSDA_BWD_COEF_RECORDS
#define MSDA_BWD_COEF_RECORDS 0
#endif
// 1 (plain op, 8 lanes per head): the three per-sample sums of FOUR samples are reduced across the group together by a
// reduce-scatter -- 12 shuffles per 4 samples instead of 36 -- which leaves lanes 2s, 2s+1 holding the finished sums of
// sample s of the batch; the even lane stores them.  Shuffles cross the same L1 data pipe as loads and reductions.
#ifndef MSDA_BWD_BATCHED_REDUCE
#define MSDA_BWD_BATCHED_REDUCE 1
#endif
// ... and the same in the fused op, whose lanes then fetch their own samples' sums from the lanes that hold them.  Measured
// (training step, alternating runs): 22.81 ms with it, 22.69 ms without -- the 12 partials cost the 64-register kernel
// spills.  Off.
#ifndef MSDA_BWD_BATCHED_FUSED
#define MSDA_BWD_BATCHED_FUSED 0
#endif
#ifndef MSDA_BWD_FUSED_ROLLED
#define MSDA_BWD_FUSED_ROLLED 1
#endif
template <int K>
__device__ __forceinline__ float reg_pick(const float (&a)[K], int idx)
{
    float r = a[0];
#pragma unroll
    for (int k = 1; k < K; ++k) r = idx == k ? a[k] : r;
    return r;
}
template <int K>
__device__ __forceinline__ void reg_put(float (&a)[K], int idx, float v)
{
#pragma unroll
    for (int k = 0; k < K; ++k) a[k] = idx == k ? v : a[k];
}

// DET (deterministic backward, DESIGN.md section 3.15): gv_accum is the int64 accumulator of the caller's scratch and
// every grad_value contribution is added as a fixed-point integer at the scale of det->scale_f (4 scalar 64-bit
// reductions per lane and corner instead of one red.v4.f32); the fused op's grad_ref goes, without atomics, to
// per-(query, level, head) partials in ref_part, which det_fold_ref sums over the heads.  DET = false compiles to the
// kernel it was before the parameter existed (the two trailing parameters are unused).
template <typename VT, int D, bool FUSED, typename RT, bool DET = false>
__global__ void __launch_bounds__(BwdWarps<32 / (D / 4)>::value * 32, MSDA_BWD_MINBLOCKS)
msda_bwd_fast_kernel(const VT* __restrict__ grad_out, const VT* __restrict__ value,
                     const int64_t* __restrict__ shapes, const int64_t* __restrict__ lsi,
                     const SampleSrc src, float* __restrict__ gv_accum, const GradDst dst,
                     int S, int M, int L, int Lq, int P, int p_magic, long long total_pairs,
                     const unsigned char* __restrict__ red_levels,
                     const DetHeader* __restrict__ det, float* __restrict__ ref_part)
{
    // red_levels (optional): per pair, bit l set = this kernel issues the grad_value reductions of level l; clear =
    // another kernel accumulates that level (msda_tc_backward.cu).  nullptr = every level.
    constexpr int EPL = 4;                       // channels per lane: one red.v4.f32 per corner
    using SliceT = Slice<VT, EPL>;
    constexpr int G = D / EPL;
    constexpr int PAIRS = 32 / G;
    constexpr int WARPS = BwdWarps<PAIRS>::value;
    constexpr int CH = MSDA_BWD_CHUNK > G ? MSDA_BWD_CHUNK : G;   // samples per pass
    constexpr int SPL = CH / G;                  // samples a lane owns per pass: j = sub*SPL + i, in phase 1
                                                 // (footprints) and again after the reduce-scatter (gradients)
    constexpr int FCH = (kChunk + CH - 1) / CH;  // passes of the fused op (host guarantees L*P <= kChunk)
    static_assert(G >= 1 && G <= 32 && (G & (G - 1)) == 0, "fast backward needs 1..32 lanes per head");
    static_assert(CH % G == 0, "pass size must split evenly over the lanes");
    static_assert(!(FUSED && DET) || CH * (MSDA_BWD_COEF_RECORDS ? 5 : 3) + 1 >= kChunk,
                  "the deterministic grad_ref staging reuses a group's records");

    // per-sample records of a pass (+1 record: the groups of a warp start in distinct banks)
    __shared__ int s_meta[3 * kMaxLevelsFast];
    __shared__ float s_inv[FUSED ? 2 * kMaxLevelsFast : 2];       // fused: 1 / H, 1 / W per level
    // record of a sample, 5 x 16 bytes: [0] byte offset (pixel * M*D * sizeof(VT)) of each corner row (corner outside the map -> 0),
    // [1] grad_value coefficient of each row (0 = no reduction), [2..4] corner dots -> grad_attn, grad_loc.x / W,
    // grad_loc.y / H
    constexpr int kRec = MSDA_BWD_COEF_RECORDS ? 5 : 3;
    __shared__ __align__(16) uint4 s_rec[WARPS][PAIRS][CH * kRec + 1];
    constexpr bool BATCHED = MSDA_BWD_BATCHED_REDUCE && (!FUSED || MSDA_BWD_BATCHED_FUSED) && G == 8 && CH == 8 && SPL == 1;
    constexpr bool DEDUP = MSDA_BWD_DEDUP && SPL == 1;

    if (threadIdx.x < L) {
        s_meta[3 * threadIdx.x + 0] = (int)shapes[2 * threadIdx.x];
        s_meta[3 * threadIdx.x + 1] = (int)shapes[2 * threadIdx.x + 1];
        s_meta[3 * threadIdx.x + 2] = (int)lsi[threadIdx.x];
        if constexpr (FUSED) {
            s_inv[2 * threadIdx.x + 0] = 1.f / (float)shapes[2 * threadIdx.x];
            s_inv[2 * threadIdx.x + 1] = 1.f / (float)shapes[2 * threadIdx.x + 1];
        }
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane / G, sub = lane % G;
#if MSDA_CTA_PER_HEAD
    const int m = (int)(blockIdx.x % M);
    const long long nq_total = total_pairs / M;
    const long long nq_raw = ((long long)(blockIdx.x / M) * WARPS + warp) * PAIRS + grp;
    const bool active = nq_raw < nq_total;
    const long long nq = active ? nq_raw : nq_total - 1;
    const long long pair = nq * M + m;
#else
    const long long pair_raw = ((long long)blockIdx.x * WARPS + warp) * PAIRS + grp;
    const bool active = pair_raw < total_pairs;
    const long long pair = active ? pair_raw : total_pairs - 1;
    const int m = (int)(pair % M);
    const long long nq = pair / M;
#endif
    const long long n = nq / Lq;
    const int LP = L * P;
    const int MD = M * D;
    const long long head_off = (n * S * M + m) * (long long)D + sub * EPL;
    // this lane's slice of pixel 0 of its (frame, head), as opaque addresses: a corner address is then one 64-bit add
    // (two instructions) of the 32-bit BYTE offset parked in shared memory -- scaled by 4 / sizeof(VT) for grad_value
    const unsigned long long vaddr = opaque_addr(value + head_off);
    // DET: lane `sub` adds channels sub, sub + G, sub + 2G, sub + 3G of a row, so that each of the four 64-bit reductions
    // of a group covers G consecutive int64 (64 bytes for a 32-channel head): the lane's own 4 consecutive channels
    // would spread every instruction over the whole 256-byte row (measured 12.6 ms for the COCO fp32 backward)
    const unsigned long long gaddr =
        DET ? opaque_addr(reinterpret_cast<long long*>(gv_accum) + (head_off - sub * EPL + sub))
            : opaque_addr(gv_accum + head_off);
    constexpr int kGradShift = DET ? (sizeof(VT) == 4 ? 1 : 2) : (sizeof(VT) == 4 ? 0 : 1);
    float det_scale = 0.f;
    if constexpr (DET) det_scale = det->scale_f;
    const float* lp = nullptr;
    const float* ap = nullptr;
    const RT* op = nullptr;
    const RT* gp = nullptr;
    if constexpr (FUSED) {
        op = static_cast<const RT*>(src.loc) + nq * src.loc_stride + (long long)m * LP * 2;
        gp = static_cast<const RT*>(src.attn) + nq * src.attn_stride + (long long)m * LP;
    } else {
        lp = static_cast<const float*>(src.loc) + pair * LP * 2;
        ap = static_cast<const float*>(src.attn) + pair * LP;
    }

    const unsigned red_mask = red_levels != nullptr ? (unsigned)red_levels[pair] : 0xffffffffu;
    float g[EPL];
    SliceT::unpack(SliceT::load_stream(grad_out + pair * D + sub * EPL), g);
    if (!active) {
#pragma unroll
        for (int c = 0; c < EPL; ++c) g[c] = 0.f;     // clamped duplicate pair contributes nothing
    }
    F2 G01, G23;
    G01.x = g[0]; G01.y = g[1]; G23.x = g[2]; G23.y = g[3];
    float gt[DET ? EPL : 1];                         // DET: grad_output at channels sub + k*G
    if constexpr (DET) {
#pragma unroll
        for (int k = 0; k < EPL; ++k) gt[k] = active ? to_f32<VT>(grad_out[pair * D + k * G + sub]) : 0.f;
    }

    // fused: softmax over the pair's L*P logits; this lane keeps the numerators of its own samples
    float prob[FCH * SPL];
    float inv_sum = 1.f;
    if constexpr (FUSED) {
        float mx = -INFINITY;
#pragma unroll
        for (int c = 0; c < FCH; ++c)
#pragma unroll
            for (int i = 0; i < SPL; ++i) {
                const int s = c * CH + sub * SPL + i;
                prob[c * SPL + i] = s < LP ? load_raw1<RT>(gp + s) : -INFINITY;
                mx = fmaxf(mx, prob[c * SPL + i]);
            }
        mx = group_max<G>(mx);
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < FCH * SPL; ++k) {
            prob[k] = prob[k] == -INFINITY ? 0.f : expf(prob[k] - mx);
            sum += prob[k];
        }
        inv_sum = 1.f / group_sum<G>(sum);            // one division per lane; the samples multiply
    }
    const float half_inv_p = 0.5f / (float)P;
    // fused: finished per-sample gradients of this lane's own samples, kept until the softmax
    // backward can be applied (it needs sum_j a_j * g_a_j over the whole pair)
    float fin_x[FCH * SPL], fin_y[FCH * SPL], fin_a[FCH * SPL], own_a[FCH * SPL];

    const int passes = FUSED ? FCH : (LP + CH - 1) / CH;
#if MSDA_BWD_FUSED_ROLLED
#pragma unroll 1
#else
#pragma unroll
#endif
    for (int c = 0; c < (FUSED ? FCH : 1 << 30); ++c) {
        if (c >= passes) break;
        const int s0 = c * CH;
        if (FUSED && s0 >= LP) break;
        const int cnt = min(CH, LP - s0);
        // ---- phase 1: footprints of this lane's own samples ------------------------------------
        float a_own[SPL];
#pragma unroll
        for (int i = 0; i < SPL; ++i) {
            const int j = sub * SPL + i;
            int4 geo = make_int4(0, 0, 0, 0);
            float4 fr = make_float4(0.f, 0.f, 0.f, 0.f);
            a_own[i] = 0.f;
            if (j < cnt) {
                const int s = s0 + j;
                const int l = div_by_points(s, p_magic);
                float2 xy;
                float a;
                if constexpr (FUSED) {
                    xy = fused_location(load_raw2<RT>(op + 2 * s), src.ref + (nq * L + l) * src.ref_dim, src.ref_dim,
                                        s_inv[2 * l], s_inv[2 * l + 1], half_inv_p);
                    a = reg_pick(prob, c * SPL + i) * inv_sum;
                } else {
                    xy = ldg_stream_f32x2(lp + 2 * s);
                    a = ldg_stream_f32(ap + s);
                }
                const Footprint f = footprint<float>(xy.x, xy.y, s_meta[3 * l], s_meta[3 * l + 1], s_meta[3 * l + 2]);
                geo = make_int4(f.pix00, f.rowstep, (int)f.ok, 0);
                fr = make_float4(f.lw, f.lh, a, 0.f);
                a_own[i] = a;
            }
            // coefficient of each corner row in grad_value: bilinear weight x attention weight (cuh:113-116); every
            // coefficient set is zero for corners outside the map (and for samples past cnt: ok = 0)
            const float lw = fr.x, lh = fr.y, hw = 1.f - fr.x, hh = 1.f - fr.y, a = fr.z;
            const bool k0 = geo.z & 1, k1 = geo.z & 2, k2 = geo.z & 4, k3 = geo.z & 8;
            const float4 ca = make_float4(k0 ? hh * hw : 0.f, k1 ? hh * lw : 0.f, k2 ? lh * hw : 0.f, k3 ? lh * lw : 0.f);
            const int my_level = div_by_points(s0 + j, p_magic);
            float4 ck = make_float4(ca.x * a, ca.y * a, ca.z * a, ca.w * a);
            if constexpr (DEDUP) {
                const float own[4] = {ck.x, ck.y, ck.z, ck.w};
                float merged[4] = {own[0], own[1], own[2], own[3]};
                int dup = 0;
                const int W = geo.y;
                // corner mask / coefficient vector of a neighbour, moved by (dx, dy) pixels into MY corner frame:
                // my corner (cx, cy) is their corner (cx - dx, cy - dy).  Bits / slots: 0 (0,0) 1 (1,0) 2 (0,1) 3 (1,1).
                auto decode = [&](int delta, int& dx, int& dy) -> bool {       // delta = their corner 00 - mine
                    dy = delta > 1 ? 1 : (delta < -1 ? -1 : 0);
                    dx = delta - dy * W;
                    return W > 2 && dx >= -1 && dx <= 1;
                };
                auto shift_mask = [](int m, int dx, int dy) -> int {
                    m = dx == 0 ? m : (dx > 0 ? (m & 5) << 1 : (m & 10) >> 1);
                    return dy == 0 ? m : (dy > 0 ? (m & 3) << 2 : (m & 12) >> 2);
                };
                // Every pair of points of the level is compared: a pixel belongs to the LOWEST sample that touches it.  I
                // collect the coefficients of every higher sample for the pixels we share, and skip the rows whose pixel a
                // lower sample has (it collects mine).
                auto gather = [&](const float (&hc)[4], int dx, int dy) {
                    // x move, then y move, of the neighbour's coefficient vector into my corner frame
                    const float x0 = dx == 0 ? hc[0] : (dx < 0 ? hc[1] : 0.f), x1 = dx == 0 ? hc[1] : (dx > 0 ? hc[0] : 0.f);
                    const float x2 = dx == 0 ? hc[2] : (dx < 0 ? hc[3] : 0.f), x3 = dx == 0 ? hc[3] : (dx > 0 ? hc[2] : 0.f);
                    // only into corners that exist: a slot outside the map must not take anything
                    if (k0) merged[0] += dy == 0 ? x0 : (dy < 0 ? x2 : 0.f);
                    if (k1) merged[1] += dy == 0 ? x1 : (dy < 0 ? x3 : 0.f);
                    if (k2) merged[2] += dy == 0 ? x2 : (dy > 0 ? x0 : 0.f);
                    if (k3) merged[3] += dy == 0 ? x3 : (dy > 0 ? x1 : 0.f);
                };
                const int span = min(P, G);
                for (int d = 1; d < span; ++d) {
                    const int lo_pix = __shfl_up_sync(0xffffffffu, geo.x, d, G);
                    const int lo_ok = __shfl_up_sync(0xffffffffu, geo.z, d, G);
                    const int hi_pix = __shfl_down_sync(0xffffffffu, geo.x, d, G);
                    float hc[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) hc[k] = __shfl_down_sync(0xffffffffu, own[k], d, G);
                    int dx, dy;
                    if (sub >= d && div_by_points(s0 + j - d, p_magic) == my_level && decode(lo_pix - geo.x, dx, dy))
                        dup |= shift_mask(lo_ok, dx, dy);
                    if (sub + d < G && div_by_points(s0 + j + d, p_magic) == my_level && decode(hi_pix - geo.x, dx, dy))
                        gather(hc, dx, dy);
                }
                // a row is mine to issue if the corner lies in the map and no lower sample owns its pixel
                const int mine = geo.z & ~dup;
                ck = make_float4((mine & 1) ? merged[0] : 0.f, (mine & 2) ? merged[1] : 0.f,
                                 (mine & 4) ? merged[2] : 0.f, (mine & 8) ? merged[3] : 0.f);
            }
            if (!((red_mask >> my_level) & 1u)) ck = make_float4(0.f, 0.f, 0.f, 0.f);   // level accumulated elsewhere
            const unsigned MDu = (unsigned)MD * (unsigned)sizeof(VT);   // bytes between neighbouring pixels
            uint4* rec = &s_rec[warp][grp][j * kRec];
            rec[0] = make_uint4(k0 ? (unsigned)geo.x * MDu : 0u, k1 ? (unsigned)(geo.x + 1) * MDu : 0u,
                                k2 ? (unsigned)(geo.x + geo.y) * MDu : 0u, k3 ? (unsigned)(geo.x + geo.y + 1) * MDu : 0u);
            reinterpret_cast<float4*>(rec)[1] = ck;
#if MSDA_BWD_COEF_RECORDS
            const float ahh = a * hh, alh = a * lh, ahw = a * hw, alw = a * lw;
            reinterpret_cast<float4*>(rec)[2] = ca;
            reinterpret_cast<float4*>(rec)[3] = make_float4(k0 ? -ahh : 0.f, k1 ? ahh : 0.f, k2 ? -alh : 0.f, k3 ? alh : 0.f);
            reinterpret_cast<float4*>(rec)[4] = make_float4(k0 ? -ahw : 0.f, k1 ? -alw : 0.f, k2 ? ahw : 0.f, k3 ? alw : 0.f);
#else
            reinterpret_cast<float4*>(rec)[2] = make_float4(lw, lh, a, __int_as_float(geo.z));
#endif
        }
        __syncwarp();

        // ---- phase 2: per-sample gather, corner dots, vector reductions into grad_value ----------
        float part[3 * SPL];
#pragma unroll
        for (int i = 0; i < 3 * SPL; ++i) part[i] = 0.f;
        float acc12[BATCHED ? 12 : 1];                // BATCHED: this lane's partial (px, py, pa) of the batch's 4 samples
#pragma unroll
        for (int i = 0; i < (BATCHED ? 12 : 1); ++i) acc12[i] = 0.f;

#pragma unroll
        for (int j0 = 0; j0 < CH; ++j0) {
            if (j0 < cnt) {
                const uint4* rec = &s_rec[warp][grp][j0 * kRec];
                const uint4 o = rec[0];
                const unsigned ok[4] = {o.x, o.y, o.z, o.w};
                typename SliceT::raw_t raw[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    raw[k] = SliceT::load(reinterpret_cast<const VT*>(vaddr + ok[k]));
                float t[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float v[EPL];
                    SliceT::unpack(raw[k], v);
                    F2 V01, V23;
                    V01.x = v[0]; V01.y = v[1]; V23.x = v[2]; V23.y = v[3];
                    const F2 d = fma2(G23, V23, mul2(G01, V01));      // this lane's 4 channels of <grad_output, value_k>
                    t[k] = d.x + d.y;
                }
                float lx, ly, la;                                     // this lane's share of the sample's three sums
#if MSDA_BWD_COEF_RECORDS
                {
                    const float4 ca = reinterpret_cast<const float4*>(rec)[2], cx = reinterpret_cast<const float4*>(rec)[3],
                                 cy = reinterpret_cast<const float4*>(rec)[4];
                    F2 T01, T23;
                    T01.x = t[0]; T01.y = t[1]; T23.x = t[2]; T23.y = t[3];
                    auto combine = [&](const float4& cf) -> float {
                        F2 C01, C23;
                        C01.x = cf.x; C01.y = cf.y; C23.x = cf.z; C23.y = cf.w;
                        const F2 r = fma2(C23, T23, mul2(C01, T01));
                        return r.x + r.y;
                    };
                    lx = combine(cx); ly = combine(cy); la = combine(ca);
                }
#else
                {
                    const float4 fr = reinterpret_cast<const float4*>(rec)[2];        // lw, lh, a, corner mask
                    const unsigned okm = __float_as_uint(fr.w);
                    const float t0 = (okm & 1u) ? t[0] : 0.f, t1 = (okm & 2u) ? t[1] : 0.f;
                    const float t2 = (okm & 4u) ? t[2] : 0.f, t3 = (okm & 8u) ? t[3] : 0.f;
                    const float lw = fr.x, lh = fr.y, hw = 1.f - fr.x, hh = 1.f - fr.y;
                    lx = fr.z * fmaf(lh, t3 - t2, hh * (t1 - t0));                    // cuh:119-151 (grad_w_weight * top_grad_value)
                    ly = fr.z * fmaf(lw, t3 - t1, hw * (t2 - t0));                    // (grad_h_weight)
                    la = fmaf(lh, fmaf(lw, t3, hw * t2), hh * fmaf(lw, t1, hw * t0)); // cuh:156
                }
#endif
                if constexpr (BATCHED) {
                    acc12[3 * (j0 & 3) + 0] = lx;
                    acc12[3 * (j0 & 3) + 1] = ly;
                    acc12[3 * (j0 & 3) + 2] = la;
                } else {
                    const float px = group_sum<G>(lx), py = group_sum<G>(ly), pa = group_sum<G>(la);
                    if (j0 / SPL == sub) {
                        part[3 * (j0 % SPL) + 0] = px;
                        part[3 * (j0 % SPL) + 1] = py;
                        part[3 * (j0 % SPL) + 2] = pa;
                    }
                }
                const float4 cf = reinterpret_cast<const float4*>(rec)[1];   // 0 = row outside the map / issued by another sample
                const float ck[4] = {cf.x, cf.y, cf.z, cf.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if constexpr (DET) {
                        if (ck[k] != 0.f) {
                            long long* gp64 = reinterpret_cast<long long*>(gaddr + ((unsigned long long)ok[k] << kGradShift));
#pragma unroll
                            for (int c = 0; c < EPL; ++c) red_fixed(gp64 + c * G, ck[k] * gt[c], det_scale);
                        }
                    } else {
                        red_scaled_f32x4_if(reinterpret_cast<float*>(gaddr + ((unsigned long long)ok[k] << kGradShift)), ck[k], G01, G23);
                    }
                }
            }
            if constexpr (BATCHED) {
                if ((j0 & 3) == 3 && j0 - 3 < cnt) {
                    // reduce-scatter of the batch's 12 partial sums over the 8 lanes: after the three steps lanes 2s, 2s+1
                    // hold the finished (px, py, pa) of sample s of the batch in acc12[0..2]
                    {
                        const bool up = (sub & 4) != 0;
#pragma unroll
                        for (int i = 0; i < 6; ++i) {
                            const float send = up ? acc12[i] : acc12[i + 6], keep = up ? acc12[i + 6] : acc12[i];
                            acc12[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                        }
                    }
                    {
                        const bool up = (sub & 2) != 0;
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
                            const float send = up ? acc12[i] : acc12[i + 3], keep = up ? acc12[i + 3] : acc12[i];
                            acc12[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 3; ++i) acc12[i] += __shfl_xor_sync(0xffffffffu, acc12[i], 1);
                    if constexpr (FUSED) {
                        // the fused op finishes a sample in the lane that owns it (softmax backward): lane 4b + s takes
                        // the sums of sample s of batch b from lane 2s
                        const int from = 2 * (sub & 3);
                        const float fx = __shfl_sync(0xffffffffu, acc12[0], from, G);
                        const float fy = __shfl_sync(0xffffffffu, acc12[1], from, G);
                        const float fa = __shfl_sync(0xffffffffu, acc12[2], from, G);
                        if ((sub >> 2) == (j0 >> 2)) { part[0] = fx; part[1] = fy; part[2] = fa; }
                    }
                    const int j = (j0 - 3) + (sub >> 1);               // the sample whose sums this lane pair holds
                    if (!FUSED && active && (sub & 1) == 0 && j < cnt) {
                        const int s = s0 + j;
                        const int l = div_by_points(s, p_magic);
                        const float Hf = (float)s_meta[3 * l], Wf = (float)s_meta[3 * l + 1];
                        float* grad_loc = static_cast<float*>(dst.loc);
                        float* grad_attn = static_cast<float*>(dst.attn);
                        *reinterpret_cast<float2*>(grad_loc + (pair * LP + s) * 2) = make_float2(Wf * acc12[0], Hf * acc12[1]);   // cuh:157-158
                        grad_attn[pair * LP + s] = acc12[2];                                                                   // cuh:156
                    }
#pragma unroll
                    for (int i = 0; i < 12; ++i) acc12[i] = 0.f;
                }
            }
        }
        __syncwarp();

        // ---- phase 3: combine the group's partials; each lane finishes its own SPL samples ----
        if constexpr (BATCHED && !FUSED) {
            // already stored by the lanes that held the sums
        } else if constexpr (!FUSED) {
            float* grad_loc = static_cast<float*>(dst.loc);
            float* grad_attn = static_cast<float*>(dst.attn);
            if (active) {
#pragma unroll
                for (int i = 0; i < SPL; ++i) {
                    const int j = sub * SPL + i;
                    if (j < cnt) {
                        const int s = s0 + j;
                        const int l = div_by_points(s, p_magic);
                        const float Hf = (float)s_meta[3 * l], Wf = (float)s_meta[3 * l + 1];
                        float2 gl = make_float2(Wf * part[3 * i + 0], Hf * part[3 * i + 1]);   // cuh:157-158
                        *reinterpret_cast<float2*>(grad_loc + (pair * LP + s) * 2) = gl;
                        grad_attn[pair * LP + s] = part[3 * i + 2];                            // cuh:156
                    }
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < SPL; ++i) {
                reg_put(fin_x, c * SPL + i, part[3 * i + 0]);
                reg_put(fin_y, c * SPL + i, part[3 * i + 1]);
                reg_put(fin_a, c * SPL + i, part[3 * i + 2]);
                reg_put(own_a, c * SPL + i, a_own[i]);
            }
        }
    }

    if constexpr (FUSED) {
        // softmax backward needs sum_j a_j * g_a_j over the pair's samples
        float dot = 0.f;
#pragma unroll
        for (int k = 0; k < FCH * SPL; ++k) {
            const int s = (k / SPL) * CH + sub * SPL + (k % SPL);
            if (s < LP) dot = fmaf(own_a[k], fin_a[k], dot);
        }
        dot = group_sum<G>(dot);
        if (active) {
            RT* gop = static_cast<RT*>(dst.loc) + nq * src.loc_stride + (long long)m * LP * 2;
            RT* ggp = static_cast<RT*>(dst.attn) + nq * src.attn_stride + (long long)m * LP;
            int run_l = -1;                       // lane-local run of samples on one level -> one grad_ref update
            float rx = 0.f, ry = 0.f, rw = 0.f, rh = 0.f;
            auto flush_ref = [&]() {
                if (!DET && dst.ref != nullptr && run_l >= 0) {
                    float* gr = dst.ref + (nq * L + run_l) * src.ref_dim;
                    atomicAdd(gr, rx);
                    atomicAdd(gr + 1, ry);
                    if (src.ref_dim == 4) { atomicAdd(gr + 2, rw); atomicAdd(gr + 3, rh); }
                }
            };
#pragma unroll
            for (int k = 0; k < FCH * SPL; ++k) {
                const int s = (k / SPL) * CH + sub * SPL + (k % SPL);
                if (s < LP) {
                    const int l = div_by_points(s, p_magic);
                    const float Hf = (float)s_meta[3 * l], Wf = (float)s_meta[3 * l + 1];
                    const float glx = Wf * fin_x[k], gly = Hf * fin_y[k];                     // d/d loc
                    const float a = own_a[k];
                    const float glogit = a * (fin_a[k] - dot);
                    float gox, goy, gwx = 0.f, gwy = 0.f;
                    if (src.ref_dim == 2) {
                        gox = glx * s_inv[2 * l + 1];
                        goy = gly * s_inv[2 * l];
                    } else {
                        const float4 r = *reinterpret_cast<const float4*>(src.ref + (nq * L + l) * 4);
                        gox = glx * (r.z * half_inv_p);
                        goy = gly * (r.w * half_inv_p);
                        if (dst.ref != nullptr) {
                            const float2 off = load_raw2<RT>(op + 2 * s);
                            gwx = glx * (off.x * half_inv_p);
                            gwy = gly * (off.y * half_inv_p);
                        }
                    }
                    store_raw2<RT>(gop + 2 * s, gox, goy);
                    ggp[s] = from_f32<RT>(glogit);
                    if (dst.ref != nullptr) {
                        if constexpr (DET) {
                            reinterpret_cast<float4*>(&s_rec[warp][grp][0])[s] = make_float4(glx, gly, gwx, gwy);
                        } else {
                            if (l != run_l) { flush_ref(); run_l = l; rx = ry = rw = rh = 0.f; }
                            rx += glx; ry += gly; rw += gwx; rh += gwy;
                        }
                    }
                }
            }
            flush_ref();
        }
        if constexpr (DET) {
            // the group's per-sample reference-point gradients are staged in its records (free after the last pass):
            // one lane per level sums the level's points in order into the (query, level, head) partial
            if (dst.ref != nullptr) {
                __syncwarp();
                if (active) {
                    const float4* staged = reinterpret_cast<const float4*>(&s_rec[warp][grp][0]);
                    for (int l = sub; l < L; l += G) {
                        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                        for (int p = 0; p < P; ++p) {
                            const float4 v = staged[l * P + p];
                            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
                        }
                        float* out = ref_part + ((nq * L + l) * M + m) * src.ref_dim;
                        out[0] = acc.x; out[1] = acc.y;
                        if (src.ref_dim == 4) { out[2] = acc.z; out[3] = acc.w; }
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Generic path: one warp per pair, lanes stride the channels, scalar atomics.
// ------------------------------------------------------------------------------------------
template <typename VT> struct ScalarLoad {
    using acc_t = typename Traits<VT>::acc_t;
    static __device__ __forceinline__ acc_t load(const VT* p) { return (acc_t)to_f32<VT>(*p); }
};
template <> struct ScalarLoad<double> {
    using acc_t = double;
    static __device__ __forceinline__ double load(const double* p) { return *p; }
};

// DET: gv_accum is the int64 accumulator of the deterministic backward (see msda_bwd_fast_kernel)
template <typename VT, bool DET = false>
__global__ void __launch_bounds__(256)
msda_bwd_generic_kernel(const VT* __restrict__ grad_out, const VT* __restrict__ value,
                        const int64_t* __restrict__ shapes, const int64_t* __restrict__ lsi,
                        const typename Traits<VT>::loc_t* __restrict__ loc,
                        const typename Traits<VT>::loc_t* __restrict__ attn,
                        typename Traits<VT>::acc_t* __restrict__ gv_accum,
                        typename Traits<VT>::loc_t* __restrict__ grad_loc,
                        typename Traits<VT>::loc_t* __restrict__ grad_attn,
                        int S, int M, int D, int L, int Lq, int P, long long total_pairs,
                        const DetHeader* __restrict__ det)
{
    using acc_t = typename Traits<VT>::acc_t;
    using loc_t = typename Traits<VT>::loc_t;
    acc_t det_scale = 0;
    if constexpr (DET) det_scale = std::is_same<acc_t, double>::value ? (acc_t)det->scale : (acc_t)det->scale_f;
    long long* const gv64 = reinterpret_cast<long long*>(gv_accum);
    auto add = [&](long long i, acc_t v) {
        if constexpr (DET) red_fixed(gv64 + i, v, det_scale);
        else atomicAdd(gv_accum + i, v);
    };
    const int lane = threadIdx.x & 31;
    const long long warps_total = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long MD = (long long)M * D;
    for (long long pair = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; pair < total_pairs;
         pair += warps_total) {
        const int m = (int)(pair % M);
        const long long n = (pair / M) / Lq;
        const long long head_off = (n * S * M + m) * (long long)D;
        const VT* go = grad_out + pair * D;
        const loc_t* lp = loc + pair * L * P * 2;
        const loc_t* ap = attn + pair * L * P;
        for (int l = 0; l < L; ++l) {
            const int H = (int)shapes[2 * l], W = (int)shapes[2 * l + 1], start = (int)lsi[l];
            for (int p = 0; p < P; ++p) {
                const int s = l * P + p;
                const loc_t x = lp[2 * s], y = lp[2 * s + 1];
                const acc_t a = (acc_t)ap[s];
                const Footprint f = footprint<loc_t>(x, y, H, W, start);
                acc_t px = 0, py = 0, pa = 0;
                if (f.ok) {
                    const loc_t w_im = x * (loc_t)W - (loc_t)0.5, h_im = y * (loc_t)H - (loc_t)0.5;
                    const acc_t lw = (acc_t)(w_im - floor(w_im)), lh = (acc_t)(h_im - floor(h_im));
                    const acc_t hw = 1 - lw, hh = 1 - lh;
                    const acc_t w1 = hh * hw, w2 = hh * lw, w3 = lh * hw, w4 = lh * lw;
                    const long long o00 = head_off + (long long)f.pix00 * MD;
                    const long long row = (long long)f.rowstep * MD;
                    for (int c = lane; c < D; c += 32) {
                        const acc_t gc = ScalarLoad<VT>::load(go + c);
                        const acc_t tg = a * gc;
                        acc_t v1 = 0, v2 = 0, v3 = 0, v4 = 0;
                        if (f.ok & 1u) { v1 = ScalarLoad<VT>::load(value + o00 + c);            add(o00 + c, w1 * tg); }
                        if (f.ok & 2u) { v2 = ScalarLoad<VT>::load(value + o00 + MD + c);       add(o00 + MD + c, w2 * tg); }
                        if (f.ok & 4u) { v3 = ScalarLoad<VT>::load(value + o00 + row + c);      add(o00 + row + c, w3 * tg); }
                        if (f.ok & 8u) { v4 = ScalarLoad<VT>::load(value + o00 + row + MD + c); add(o00 + row + MD + c, w4 * tg); }
                        pa += gc * (w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4);
                        px += tg * (hh * (v2 - v1) + lh * (v4 - v3));
                        py += tg * (hw * (v3 - v1) + lw * (v4 - v2));
                    }
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    px += __shfl_xor_sync(0xffffffffu, px, off);
                    py += __shfl_xor_sync(0xffffffffu, py, off);
                    pa += __shfl_xor_sync(0xffffffffu, pa, off);
                }
                if (lane == 0) {
                    grad_loc[(pair * L * P + s) * 2] = (loc_t)((acc_t)W * px);
                    grad_loc[(pair * L * P + s) * 2 + 1] = (loc_t)((acc_t)H * py);
                    grad_attn[pair * L * P + s] = (loc_t)pa;
                }
            }
        }
    }
}

// fp32 accumulation buffer -> 16-bit grad_value
template <typename VT>
__global__ void __launch_bounds__(256)
msda_cast_accum_kernel(const float* __restrict__ src, VT* __restrict__ dst, long long count)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long vec = count / 8;
    for (long long i = i0; i < vec; i += stride) {
        float f[8];
        const uint4 a = ldg_stream_v4(src + i * 8), b = ldg_stream_v4(src + i * 8 + 4);
        unpack<float>(a, f);
        unpack<float>(b, f + 4);
        stg_stream_v4(dst + i * 8, pack<VT>(f));
    }
    for (long long i = vec * 8 + i0; i < count; i += stride) dst[i] = from_f32<VT>(src[i]);
}

// ------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------
template <typename VT, int D, bool DET = false>
static cudaError_t launch_bwd_fast(const BwdArgs& a, float* accum, cudaStream_t stream,
                                   const unsigned char* red_levels = nullptr, const DetHeader* det = nullptr)
{
    constexpr int G = D / 4;
    constexpr int PAIRS = 32 / G;
    constexpr int WARPS = BwdWarps<PAIRS>::value;
    const long long total_pairs = (long long)a.N * a.Lq * a.M;
#if MSDA_CTA_PER_HEAD
    const long long nq_total = (long long)a.N * a.Lq;
    const long long blocks = ((nq_total + WARPS * PAIRS - 1) / (WARPS * PAIRS)) * a.M;
#else
    const long long blocks = (total_pairs + WARPS * PAIRS - 1) / (WARPS * PAIRS);
#endif
    if (blocks > 0x7fffffffll) return cudaErrorInvalidConfiguration;
    const int p_magic = (65536 + a.P - 1) / a.P;
    SampleSrc src;
    src.loc = a.loc; src.attn = a.attn; src.ref = nullptr; src.loc_stride = 0; src.attn_stride = 0; src.ref_dim = 0;
    GradDst dst;
    dst.loc = a.grad_loc; dst.attn = a.grad_attn; dst.ref = nullptr;
    msda_bwd_fast_kernel<VT, D, false, float, DET><<<(unsigned)blocks, WARPS * 32, 0, stream>>>(
        (const VT*)a.grad_out, (const VT*)a.value, a.shapes, a.lsi, src, accum, dst,
        a.S, a.M, a.L, a.Lq, a.P, p_magic, total_pairs, red_levels, det, nullptr);
    return cudaGetLastError();
}

template <typename VT, int D, typename RT, bool DET = false>
static cudaError_t launch_bwd_fused(const FusedArgs& a, float* accum, cudaStream_t stream,
                                    const DetHeader* det = nullptr, float* ref_part = nullptr)
{
    constexpr int G = D / 4;
    constexpr int PAIRS = 32 / G;
    constexpr int WARPS = BwdWarps<PAIRS>::value;
    const long long total_pairs = (long long)a.N * a.Lq * a.M;
#if MSDA_CTA_PER_HEAD
    const long long nq_total = (long long)a.N * a.Lq;
    const long long blocks = ((nq_total + WARPS * PAIRS - 1) / (WARPS * PAIRS)) * a.M;
#else
    const long long blocks = (total_pairs + WARPS * PAIRS - 1) / (WARPS * PAIRS);
#endif
    if (blocks > 0x7fffffffll) return cudaErrorInvalidConfiguration;
    const int p_magic = (65536 + a.P - 1) / a.P;
    SampleSrc src;
    src.loc = a.offsets; src.attn = a.logits; src.ref = a.ref;
    src.loc_stride = a.off_stride; src.attn_stride = a.logit_stride; src.ref_dim = a.ref_dim;
    GradDst dst;
    dst.loc = a.grad_offsets; dst.attn = a.grad_logits; dst.ref = a.grad_ref;
    msda_bwd_fast_kernel<VT, D, true, RT, DET><<<(unsigned)blocks, WARPS * 32, 0, stream>>>(
        (const VT*)a.grad_out, (const VT*)a.value, a.shapes, a.lsi, src, accum, dst,
        a.S, a.M, a.L, a.Lq, a.P, p_magic, total_pairs, nullptr, det, ref_part);
    return cudaGetLastError();
}

template <typename VT, bool DET = false>
static cudaError_t launch_bwd_generic(const BwdArgs& a, typename Traits<VT>::acc_t* accum, cudaStream_t stream,
                                      const DetHeader* det = nullptr)
{
    using loc_t = typename Traits<VT>::loc_t;
    const long long total_pairs = (long long)a.N * a.Lq * a.M;
    long long blocks = (total_pairs + 7) / 8;
    if (blocks > (1ll << 30)) blocks = 1ll << 30;
    msda_bwd_generic_kernel<VT, DET><<<(unsigned)blocks, 256, 0, stream>>>(
        (const VT*)a.grad_out, (const VT*)a.value, a.shapes, a.lsi, (const loc_t*)a.loc, (const loc_t*)a.attn,
        accum, (loc_t*)a.grad_loc, (loc_t*)a.grad_attn, a.S, a.M, a.D, a.L, a.Lq, a.P, total_pairs, det);
    return cudaGetLastError();
}

static bool fast_shape_ok(const BwdArgs& a)
{
    return !a.force_generic && a.L <= kMaxLevelsFast && a.P <= 64 && (long long)a.L * a.P * a.P < 65536 &&
           (long long)a.S * a.M * a.D < (1ll << 30);      // 32-bit byte offsets inside one frame
}

template <typename VT>
static cudaError_t run_bwd_16or32(const BwdArgs& a, cudaStream_t stream)
{
    constexpr bool k16 = sizeof(VT) == 2;
    const size_t count = (size_t)a.N * a.S * a.M * a.D;
    float* accum = k16 ? a.grad_value_accum : (float*)a.grad_value;
    if (k16 && accum == nullptr) return cudaErrorInvalidValue;
    cudaError_t err = cudaMemsetAsync(accum, 0, count * sizeof(float), stream);
    if (err != cudaSuccess) return err;
    const long long total_pairs = (long long)a.N * a.Lq * a.M;
    if constexpr (std::is_same<VT, __nv_bfloat16>::value) {
        if (!a.no_tc && total_pairs > 0 && fast_shape_ok(a) && tc_backward_supported(a)) {
            // opt-in: grad_value of every (tile, level) whose window fits is accumulated on the tensor cores
            // (msda_tc_backward.cu); the lane-group kernel keeps grad_loc / grad_attn and the levels left over
            unsigned char* red_levels = nullptr;
            err = cudaMallocAsync((void**)&red_levels, (size_t)total_pairs, stream);
            if (err != cudaSuccess) return err;
            err = tc_backward_dv(a, red_levels, stream);
            if (err == cudaSuccess) err = launch_bwd_fast<VT, 32>(a, accum, stream, red_levels);
            const cudaError_t e2 = cudaFreeAsync(red_levels, stream);
            if (err != cudaSuccess) return err;
            if (e2 != cudaSuccess) return e2;
            long long blocks = (long long)((count / 8 + 255) / 256);
            if (blocks < 1) blocks = 1;
            if (blocks > 148 * 16) blocks = 148 * 16;
            msda_cast_accum_kernel<VT><<<(unsigned)blocks, 256, 0, stream>>>(accum, (VT*)a.grad_value, (long long)count);
            return cudaGetLastError();
        }
    }
    if (total_pairs > 0 && a.D > 0) {
        bool done = false;
        if (fast_shape_ok(a)) {
            done = true;
            switch (a.D) {   // G = D/4 lanes per head must be a power of two <= 32
                case 4:   err = launch_bwd_fast<VT, 4>(a, accum, stream); break;
                case 8:   err = launch_bwd_fast<VT, 8>(a, accum, stream); break;
                case 16:  err = launch_bwd_fast<VT, 16>(a, accum, stream); break;
                case 32:  err = launch_bwd_fast<VT, 32>(a, accum, stream); break;
                case 64:  err = launch_bwd_fast<VT, 64>(a, accum, stream); break;
                case 128: err = launch_bwd_fast<VT, 128>(a, accum, stream); break;     // one (query, head) per warp
                default: done = false;
            }
        }
        if (!done) err = launch_bwd_generic<VT>(a, accum, stream);
        if (err != cudaSuccess) return err;
    }
    if (k16 && count > 0) {
        long long blocks = (long long)((count / 8 + 255) / 256);
        if (blocks < 1) blocks = 1;
        if (blocks > 148 * 16) blocks = 148 * 16;
        msda_cast_accum_kernel<VT><<<(unsigned)blocks, 256, 0, stream>>>(accum, (VT*)a.grad_value, (long long)count);
        err = cudaGetLastError();
    }
    return err;
}

template <typename VT, typename RT>
static cudaError_t run_bwd_fused(const FusedArgs& a, cudaStream_t stream)
{
    constexpr bool k16 = sizeof(VT) == 2;
    const size_t count = (size_t)a.N * a.S * a.M * a.D;
    float* accum = k16 ? a.grad_value_accum : (float*)a.grad_value;
    if (k16 && accum == nullptr) return cudaErrorInvalidValue;
    cudaError_t err = cudaMemsetAsync(accum, 0, count * sizeof(float), stream);
    if (err != cudaSuccess) return err;
    if ((long long)a.N * a.Lq * a.M > 0) {
        switch (a.D) {
            case 16: err = launch_bwd_fused<VT, 16, RT>(a, accum, stream); break;
            case 32: err = launch_bwd_fused<VT, 32, RT>(a, accum, stream); break;
            case 64: err = launch_bwd_fused<VT, 64, RT>(a, accum, stream); break;
            default: err = cudaErrorInvalidValue;
        }
        if (err != cudaSuccess) return err;
    }
    if (k16 && count > 0) {
        long long blocks = (long long)((count / 8 + 255) / 256);
        if (blocks < 1) blocks = 1;
        if (blocks > 148 * 16) blocks = 148 * 16;
        msda_cast_accum_kernel<VT><<<(unsigned)blocks, 256, 0, stream>>>(accum, (VT*)a.grad_value, (long long)count);
        err = cudaGetLastError();
    }
    return err;
}

cudaError_t fused_backward(const FusedArgs& a, cudaStream_t stream)
{
    if (!fused_supported(a) || !fused_raw_layout_ok(a)) return cudaErrorInvalidValue;
    if (a.dtype == kF32) return run_bwd_fused<float, float>(a, stream);
    if (a.raw_dtype == kF32) return run_bwd_fused<__nv_bfloat16, float>(a, stream);
    return run_bwd_fused<__nv_bfloat16, __nv_bfloat16>(a, stream);
}

cudaError_t backward(const BwdArgs& a, cudaStream_t stream)
{
    if (a.L == 0 || a.P == 0) {
        // empty sum (the forward writes zeros, msda_forward): grad_value is all zeros, grad_loc / grad_attn have no
        // elements.  Also keeps P = 0 away from the launchers' 65536 / P.
        if (a.dtype < kF32 || a.dtype > kF16) return cudaErrorInvalidValue;
        const size_t esz = a.dtype == kF64 ? 8 : (a.dtype == kF32 ? 4 : 2);
        return cudaMemsetAsync(a.grad_value, 0, (size_t)a.N * a.S * a.M * a.D * esz, stream);
    }
    switch (a.dtype) {
        case kF32:  return run_bwd_16or32<float>(a, stream);
        case kBF16: return run_bwd_16or32<__nv_bfloat16>(a, stream);
        case kF16:  return run_bwd_16or32<__half>(a, stream);
        case kF64: {
            const size_t count = (size_t)a.N * a.S * a.M * a.D;
            cudaError_t err = cudaMemsetAsync(a.grad_value, 0, count * sizeof(double), stream);
            if (err != cudaSuccess) return err;
            if ((long long)a.N * a.Lq * a.M == 0 || a.D == 0) return cudaSuccess;
            return launch_bwd_generic<double>(a, (double*)a.grad_value, stream);
        }
    }
    return cudaErrorInvalidValue;
}

// ------------------------------------------------------------------------------------------
// deterministic backward (DESIGN.md section 3.15): zero the accumulators, bound the gradient, accumulate in fixed
// point, convert.  Same kernels as above with DET = true; stream-ordered, no allocation, no host read-back.
// ------------------------------------------------------------------------------------------
template <typename VT>
static cudaError_t run_bwd_det(const BwdArgs& a, long long* acc, const DetHeader* det, cudaStream_t stream)
{
    float* acc_f = reinterpret_cast<float*>(acc);
    if (fast_shape_ok(a)) {
        switch (a.D) {
            case 4:   return launch_bwd_fast<VT, 4, true>(a, acc_f, stream, nullptr, det);
            case 8:   return launch_bwd_fast<VT, 8, true>(a, acc_f, stream, nullptr, det);
            case 16:  return launch_bwd_fast<VT, 16, true>(a, acc_f, stream, nullptr, det);
            case 32:  return launch_bwd_fast<VT, 32, true>(a, acc_f, stream, nullptr, det);
            case 64:  return launch_bwd_fast<VT, 64, true>(a, acc_f, stream, nullptr, det);
            case 128: return launch_bwd_fast<VT, 128, true>(a, acc_f, stream, nullptr, det);
            default: break;
        }
    }
    return launch_bwd_generic<VT, true>(a, reinterpret_cast<typename Traits<VT>::acc_t*>(acc), stream, det);
}

cudaError_t backward_deterministic(const BwdArgs& a, void* scratch, long long scratch_bytes, cudaStream_t stream)
{
    if (a.dtype < kF32 || a.dtype > kF16 || !a.no_tc) return cudaErrorInvalidValue;   // no tensor-core variant
    const long long count = (long long)a.N * a.S * a.M * a.D;
    if (scratch == nullptr || scratch_bytes < det_scratch_bytes(count, 0)) return cudaErrorInvalidValue;
    if (a.L == 0 || a.P == 0) return backward(a, stream);         // grad_value = 0, nothing is accumulated
    DetHeader* h = static_cast<DetHeader*>(scratch);
    long long* acc = reinterpret_cast<long long*>(static_cast<char*>(scratch) + kDetHeaderBytes);
    cudaError_t err = det_begin(scratch, count, stream);
    const long long pairs = (long long)a.N * a.Lq * a.M;
    if (err == cudaSuccess) err = det_absmax(a.dtype, a.grad_out, pairs, a.D, a.D, &h->gmax, stream);
    if (err == cudaSuccess) err = det_attn_sum_max(a.dtype == kF64, a.attn, pairs, a.L * a.P, &h->amax, stream);
    // a pixel of one (frame, head) receives, per query, at most |a| |g| from each sample (the bilinear weights of a
    // sample are at most 1 at any one pixel):  |grad_value| <= Lq * max|g| * max_pair sum |a|
    if (err == cudaSuccess) err = det_finalize(h, (double)a.Lq, 0, a.dtype == kF64, stream);
    if (err == cudaSuccess && pairs > 0 && a.D > 0) {
        switch (a.dtype) {
            case kF32:  err = run_bwd_det<float>(a, acc, h, stream); break;
            case kBF16: err = run_bwd_det<__nv_bfloat16>(a, acc, h, stream); break;
            case kF16:  err = run_bwd_det<__half>(a, acc, h, stream); break;
            case kF64:  err = launch_bwd_generic<double, true>(a, reinterpret_cast<double*>(acc), stream, h); break;
        }
    }
    if (err == cudaSuccess) err = det_finish(a.dtype, acc, a.grad_value, count, h, stream);
    return err;
}

template <typename VT, typename RT>
static cudaError_t run_bwd_fused_det(const FusedArgs& a, long long* acc, const DetHeader* det, float* ref_part,
                                     cudaStream_t stream)
{
    float* acc_f = reinterpret_cast<float*>(acc);
    switch (a.D) {
        case 16: return launch_bwd_fused<VT, 16, RT, true>(a, acc_f, stream, det, ref_part);
        case 32: return launch_bwd_fused<VT, 32, RT, true>(a, acc_f, stream, det, ref_part);
        case 64: return launch_bwd_fused<VT, 64, RT, true>(a, acc_f, stream, det, ref_part);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t fused_backward_deterministic(const FusedArgs& a, void* scratch, long long scratch_bytes,
                                         cudaStream_t stream)
{
    if (!fused_supported(a) || !fused_raw_layout_ok(a)) return cudaErrorInvalidValue;
    const long long count = (long long)a.N * a.S * a.M * a.D;
    const long long rows = (long long)a.N * a.Lq * a.L;     // grad_ref rows (query, level)
    const long long part = a.grad_ref != nullptr ? rows * a.M * a.ref_dim : 0;
    if (scratch == nullptr || scratch_bytes < det_scratch_bytes(count, part)) return cudaErrorInvalidValue;
    DetHeader* h = static_cast<DetHeader*>(scratch);
    long long* acc = reinterpret_cast<long long*>(static_cast<char*>(scratch) + kDetHeaderBytes);
    float* ref_part = det_ref_partials(scratch, count);
    const long long pairs = (long long)a.N * a.Lq * a.M;
    const long long nq = (long long)a.N * a.Lq;
    const int mlp = a.M * a.L * a.P;
    cudaError_t err = det_begin(scratch, count, stream);
    if (err == cudaSuccess) err = det_absmax(a.dtype, a.grad_out, pairs, a.D, a.D, &h->gmax, stream);
    // the attention weights are a softmax (sum |a| = 1 per pair): the logits are scanned only for Inf / NaN
    if (err == cudaSuccess) err = det_absmax(a.raw_dtype, a.logits, nq, mlp, a.logit_stride, &h->amax, stream);
    if (err == cudaSuccess) err = det_finalize(h, (double)a.Lq, 1, false, stream);
    if (err == cudaSuccess && pairs > 0) {
        if (a.dtype == kF32) err = run_bwd_fused_det<float, float>(a, acc, h, ref_part, stream);
        else if (a.raw_dtype == kF32) err = run_bwd_fused_det<__nv_bfloat16, float>(a, acc, h, ref_part, stream);
        else err = run_bwd_fused_det<__nv_bfloat16, __nv_bfloat16>(a, acc, h, ref_part, stream);
    }
    if (err == cudaSuccess) err = det_finish(a.dtype, acc, a.grad_value, count, h, stream);
    if (err == cudaSuccess && a.grad_ref != nullptr) err = det_fold_ref(ref_part, a.grad_ref, rows, a.M, a.ref_dim, stream);
    return err;
}

}  // namespace msda
