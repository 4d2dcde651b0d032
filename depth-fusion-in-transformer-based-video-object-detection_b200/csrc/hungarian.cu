// Batched rectangular linear assignment (C ABI msda_linear_assignment, DESIGN.md section 3.17).
//
// One CTA solves one problem: the cost C[q, t] of matching query q to target t, T <= Q targets, every target
// matched.  The targets are the rows that get augmented, the queries are the columns, so a problem costs
// O(T^2 Q) instead of the O(Q^3) of a square solve.  The algorithm is the shortest-augmenting-path method of
// Jonker-Volgenant in Crouse's form (scipy.optimize.linear_sum_assignment), with the same fp64 arithmetic on
// the same fp64-widened costs:  reduced cost r = minVal + C - u[i] - v[j], the same dual updates and the same
// augmentation.  Only the order in which tied columns are considered differs: a Dijkstra step takes the
// column of least distance, among those an unassigned one (scipy's rule), among those the lowest index.
//
// Column j is owned by thread j % kThreads: only its owner touches its distance, path and scanned flag during
// a search, so a Dijkstra step needs one block-wide arg-min and nothing else.  The variant is picked from Q:
// a one-warp CTA with the state in shared memory (Q <= kLapWarpMaxQ: the decoder heads, Q = 300), or a
// 1024-thread CTA with the state in a global scratch slab per problem (the two-stage encoder proposals,
// Q = S, up to tens of thousands of columns).
#include <math.h>
#include <stddef.h>
#include "msda_launch.h"

namespace msda {
namespace {

constexpr int kLapWarpMaxQ = 1024;        // 25 Q + 13 T bytes of state: <= 38.9 KB, under the 48 KB default
constexpr int kLapCtaThreads = 1024;
constexpr int kAssignedBit = 1 << 30;     // tie key: unassigned columns first, then the lower index

constexpr int kStatusNonFinite = 1;
constexpr int kStatusBadCount = 2;
constexpr int kStatusInfeasible = 3;

__host__ __device__ inline size_t lap_state_bytes(int Q, int R)
{
    return (size_t)8 * (2 * (size_t)Q + R) + (size_t)4 * (2 * (size_t)Q + R) + (size_t)Q + R;
}

__host__ inline size_t lap_scratch_per_problem(int Q, int R) { return (lap_state_bytes(Q, R) + 255) & ~(size_t)255; }

struct LapState {
    double* v;            // [Q] column potentials
    double* dist;         // [Q] shortest-path distance of the current search
    double* u;            // [R] row potentials
    int* path;            // [Q] predecessor row
    int* row4col;         // [Q] row assigned to the column, -1 if none
    int* col4row;         // [R] column assigned to the row, -1 if none
    unsigned char* sc;    // [Q] column scanned in the current search
    unsigned char* sr;    // [R] row reached in the current search
};

__device__ inline LapState carve(char* base, int Q, int R)
{
    LapState s;
    s.v = reinterpret_cast<double*>(base);
    s.dist = s.v + Q;
    s.u = s.dist + Q;
    s.path = reinterpret_cast<int*>(s.u + R);
    s.row4col = s.path + Q;
    s.col4row = s.row4col + Q;
    s.sc = reinterpret_cast<unsigned char*>(s.col4row + R);
    s.sr = s.sc + Q;
    return s;
}

__device__ __forceinline__ bool key_less(double a, int ka, double b, int kb)
{
    return a < b || (a == b && ka < kb);
}

// Arg-min of (val, key) over the CTA; every thread returns the winner.  `buf` alternates between calls, so one
// barrier per call suffices: a warp can only overwrite a buffer after every warp has passed the next call's barrier.
template <int kThreads>
__device__ __forceinline__ void block_argmin(double& val, int& key, double (*red_val)[kThreads / 32],
                                             int (*red_key)[kThreads / 32], int buf)
{
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, val, off);
        const int ok = __shfl_xor_sync(0xffffffffu, key, off);
        if (key_less(ov, ok, val, key)) { val = ov; key = ok; }
    }
    if constexpr (kThreads > 32) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) { red_val[buf][warp] = val; red_key[buf][warp] = key; }
        __syncthreads();
        val = lane < kThreads / 32 ? red_val[buf][lane] : INFINITY;
        key = lane < kThreads / 32 ? red_key[buf][lane] : 0x7fffffff;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, val, off);
            const int ok = __shfl_xor_sync(0xffffffffu, key, off);
            if (key_less(ov, ok, val, key)) { val = ov; key = ok; }
        }
    }
}

template <int kThreads, bool kShared>
__global__ void __launch_bounds__(kThreads) linear_assignment_kernel(
    const float* __restrict__ cost, long long problem_stride, long long query_stride, const int64_t* __restrict__ counts,
    int Q, int Tmax, int* __restrict__ query_of_target, int* __restrict__ target_of_query, int* __restrict__ status,
    char* scratch, size_t scratch_per_problem)
{
    extern __shared__ __align__(16) char lap_smem[];
    __shared__ double red_val[2][kThreads / 32];
    __shared__ int red_key[2][kThreads / 32];

    const int p = blockIdx.x, tid = threadIdx.x;
    const int R = Tmax < Q ? Tmax : Q;
    const float* C = cost + (long long)p * problem_stride;
    int* qot = query_of_target + (long long)p * Tmax;
    int* toq = target_of_query + (long long)p * Q;

    const long long count = counts[p];
    const bool bad_count = count < 0 || count > R;
    const int T = bad_count ? 0 : (int)count;
    int nonfinite = 0;
    for (int q = tid; q < Q; q += kThreads)
        for (int t = 0; t < T; ++t)
            nonfinite |= !isfinite(C[q * query_stride + t]);
    nonfinite = __syncthreads_or(nonfinite);

    int st = bad_count ? kStatusBadCount : nonfinite ? kStatusNonFinite : 0;
    LapState s = carve(kShared ? lap_smem : scratch + (size_t)p * scratch_per_problem, Q, R);
    if (st == 0 && T > 0) {
        for (int j = tid; j < Q; j += kThreads) { s.v[j] = 0.0; s.row4col[j] = -1; }
        for (int i = tid; i < T; i += kThreads) { s.u[i] = 0.0; s.col4row[i] = -1; }
        int buf = 0;
        for (int cur = 0; cur < T && st == 0; ++cur) {
            for (int j = tid; j < Q; j += kThreads) { s.dist[j] = INFINITY; s.sc[j] = 0; }
            for (int i = tid; i < T; i += kThreads) s.sr[i] = 0;
            __syncthreads();
            // Dijkstra from row `cur` over the reduced costs; row4col and the potentials are read-only here
            double min_val = 0.0;
            int i = cur, sink = -1;
            while (sink < 0) {
                if (tid == 0) s.sr[i] = 1;
                const double ui = s.u[i];
                double best = INFINITY;
                int best_key = 0x7fffffff;
                for (int j = tid; j < Q; j += kThreads) {
                    if (s.sc[j]) continue;
                    const double r = min_val + (double)C[j * query_stride + i] - ui - s.v[j];
                    double d = s.dist[j];
                    if (r < d) { s.path[j] = i; s.dist[j] = r; d = r; }
                    const int key = (s.row4col[j] < 0 ? 0 : kAssignedBit) | j;
                    if (key_less(d, key, best, best_key)) { best = d; best_key = key; }
                }
                block_argmin<kThreads>(best, best_key, red_val, red_key, buf);
                buf ^= 1;
                if (best == INFINITY) { st = kStatusInfeasible; break; }
                min_val = best;
                const int j = best_key & (kAssignedBit - 1);
                if (j % kThreads == tid) s.sc[j] = 1;
                const int owner = s.row4col[j];
                if (owner < 0) sink = j; else i = owner;
            }
            __syncthreads();
            if (st != 0) break;
            // dual update, as scipy: the reached rows and scanned columns move by min_val - dist
            for (int r = tid; r < T; r += kThreads)
                if (r == cur) s.u[r] += min_val;
                else if (s.sr[r]) s.u[r] += min_val - s.dist[s.col4row[r]];
            for (int j = tid; j < Q; j += kThreads)
                if (s.sc[j]) s.v[j] -= min_val - s.dist[j];
            __syncthreads();
            if (tid == 0) {
                int j = sink;
                for (;;) {
                    const int r = s.path[j];
                    s.row4col[j] = r;
                    const int prev = s.col4row[r];
                    s.col4row[r] = j;
                    j = prev;
                    if (r == cur) break;
                }
            }
            __syncthreads();
        }
    }
    const bool ok = st == 0;
    for (int t = tid; t < Tmax; t += kThreads) qot[t] = ok && t < T ? s.col4row[t] : -1;
    for (int q = tid; q < Q; q += kThreads) toq[q] = ok && T > 0 ? s.row4col[q] : -1;
    if (tid == 0) status[p] = st;
}

}  // namespace

long long linear_assignment_scratch_bytes(int P, int Q, int Tmax)
{
    if (P < 0 || Q < 0 || Tmax < 0) return -1;
    if (Q <= kLapWarpMaxQ) return 0;
    return (long long)P * (long long)lap_scratch_per_problem(Q, Tmax < Q ? Tmax : Q);
}

cudaError_t linear_assignment(const float* cost, long long problem_stride, long long query_stride,
                              const int64_t* counts, int P, int Q, int Tmax, int* query_of_target,
                              int* target_of_query, int* status, void* scratch, long long scratch_bytes,
                              cudaStream_t stream)
{
    if (P < 0 || Q < 0 || Tmax < 0 || problem_stride < 0 || query_stride < 0) return cudaErrorInvalidValue;
    if (P == 0) return cudaSuccess;
    if (!cost || !counts || !query_of_target || !status || (Q > 0 && !target_of_query)) return cudaErrorInvalidValue;
    const int R = Tmax < Q ? Tmax : Q;
    if (Q <= kLapWarpMaxQ) {
        linear_assignment_kernel<32, true><<<P, 32, lap_state_bytes(Q, R), stream>>>(
            cost, problem_stride, query_stride, counts, Q, Tmax, query_of_target, target_of_query, status, nullptr, 0);
    } else {
        if (!scratch || scratch_bytes < linear_assignment_scratch_bytes(P, Q, Tmax)) return cudaErrorInvalidValue;
        linear_assignment_kernel<kLapCtaThreads, false><<<P, kLapCtaThreads, 0, stream>>>(
            cost, problem_stride, query_stride, counts, Q, Tmax, query_of_target, target_of_query, status,
            static_cast<char*>(scratch), lap_scratch_per_problem(Q, R));
    }
    return cudaGetLastError();
}

}  // namespace msda
