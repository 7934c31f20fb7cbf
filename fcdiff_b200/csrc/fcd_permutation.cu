// Westfall-Young step-down max-T counts of a permutation test (no reference counterpart: the reference has no
// permutation driver; fcdiff_b200/sweep.py collects the statistics).
//
// T [R1][pitch]: row 0 holds the observed statistics, rows 1.. those of relabelled data.  One family is the
// column range [k0, k1); `order` lists its columns ascending by (T[0][k], k) (sigma, sorted on the host).
// With G[r][j] = T[r][sigma(j)]:
//   count_unc[sigma(j) - k0] = #{r : G[r][j] >= G[0][j]}
//   count_sd[j]              = #{r : max_{i <= j} G[r][i] >= G[0][j]}
// Three passes over the family's R1 x Kf values:
//   1. maxt_gather_kernel: G in sigma order (the gathered reads of a row come from L2: a block's neighbours work
//      on the same row) and the maximum of every (row, chunk) of kMtChunk positions;
//   2. maxt_carry_kernel: exclusive prefix maxima of the chunk maxima, per row (R1 x Kf / kMtChunk values);
//   3. maxt_count_kernel: one CTA per (chunk, slice of replicas), one warp per replica: the carry-in, a warp
//      prefix max over 32 positions at a time, both comparisons with the sorted observed row, counts in
//      registers, then shared memory, then one integer atomic per (CTA, position) into global memory.
// The counts are integers: the result does not depend on the launch shape or the order of the atomics.
#include "fcdiff_b200.h"
#include "fcd_common.cuh"

namespace fcd {

constexpr int     kMtChunk   = 512;                   // sorted positions per chunk
constexpr int     kMtThreads = 256;
constexpr int     kMtWarps   = kMtThreads / 32;
constexpr int     kMtSeg     = kMtChunk / 32;         // 32-wide segments of a chunk (a lane's counters)
constexpr int64_t kMtMaxRows = (int64_t)1 << 20;
constexpr int64_t kMtMaxCols = (int64_t)1 << 24;

// G[r][j] = T[r][order[j]] for j < Kf; cm[r][b] = max of chunk b of row r.  Block = (row, chunk), row major.
__global__ void __launch_bounds__(kMtThreads)
maxt_gather_kernel(const double* __restrict__ T, int64_t pitch, const int64_t* __restrict__ order, int64_t Kf,
                   int64_t nchunks, double* __restrict__ G, double* __restrict__ cm) {
    __shared__ double red[kMtWarps];
    const int64_t r = blockIdx.x / nchunks, b = blockIdx.x - r * nchunks;
    const int64_t j0 = b * kMtChunk;
    const int64_t j1 = j0 + kMtChunk < Kf ? j0 + kMtChunk : Kf;
    const double* row = T + r * pitch;
    double* g = G + r * Kf;
    double m = -INFINITY;
    for (int64_t j = j0 + threadIdx.x; j < j1; j += kMtThreads) {
        const double v = __ldg(row + __ldg(order + j));
        g[j] = v;
        m = fmax(m, v);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, d));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        double x = red[0];
#pragma unroll
        for (int w = 1; w < kMtWarps; ++w) x = fmax(x, red[w]);
        cm[r * nchunks + b] = x;
    }
}

// cm[r][b] <- max_{b' < b} cm[r][b'] (-inf for b = 0), in place.  One warp per row.
__global__ void __launch_bounds__(kMtThreads)
maxt_carry_kernel(double* __restrict__ cm, int64_t R1, int64_t nchunks) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (blockIdx.x * (int64_t)kMtThreads + threadIdx.x) >> 5;
    if (r >= R1) return;
    double* c = cm + r * nchunks;
    double carry = -INFINITY;
    for (int64_t b0 = 0; b0 < nchunks; b0 += 32) {
        const int64_t b = b0 + lane;
        const double v = b < nchunks ? c[b] : -INFINITY;
        double incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl = fmax(incl, t);
        }
        double excl = __shfl_up_sync(0xffffffffu, incl, 1);
        excl = lane == 0 ? carry : fmax(excl, carry);
        if (b < nchunks) c[b] = excl;
        carry = fmax(carry, __shfl_sync(0xffffffffu, incl, 31));
    }
}

// Counts of chunk blockIdx.x over the replicas r = blockIdx.y * kMtWarps + warp (+ gridDim.y * kMtWarps ...).
// Lane l keeps the counts of positions s * 32 + l of the chunk in registers.
__global__ void __launch_bounds__(kMtThreads)
maxt_count_kernel(const double* __restrict__ G, int64_t Kf, int64_t R1, int64_t nchunks, const double* __restrict__ cm,
                  const int64_t* __restrict__ order, int64_t k0, unsigned long long* __restrict__ count_unc,
                  unsigned long long* __restrict__ count_sd) {
    __shared__ double obs[kMtChunk];
    __shared__ int cu_s[kMtChunk], cs_s[kMtChunk];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t b = blockIdx.x;
    const int64_t j0 = b * kMtChunk;
    const int len = (int)(j0 + kMtChunk < Kf ? kMtChunk : Kf - j0);
    for (int j = threadIdx.x; j < kMtChunk; j += kMtThreads) {
        obs[j] = j < len ? G[j0 + j] : INFINITY;        // row 0 in sigma order; no count past the end
        cu_s[j] = 0;
        cs_s[j] = 0;
    }
    __syncthreads();
    int cu[kMtSeg], cs[kMtSeg];
#pragma unroll
    for (int s = 0; s < kMtSeg; ++s) cu[s] = cs[s] = 0;
    const int64_t stride = (int64_t)gridDim.y * kMtWarps;
    for (int64_t r = (int64_t)blockIdx.y * kMtWarps + warp; r < R1; r += stride) {
        const double* g = G + r * Kf + j0;
        double v[kMtSeg];
#pragma unroll
        for (int s = 0; s < kMtSeg; ++s) v[s] = s * 32 + lane < len ? g[s * 32 + lane] : -INFINITY;
        double carry = cm[r * nchunks + b];
#pragma unroll
        for (int s = 0; s < kMtSeg; ++s) {
            double m = v[s];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, m, d);
                if (lane >= d) m = fmax(m, t);
            }
            m = fmax(m, carry);
            const double o = obs[s * 32 + lane];
            cu[s] += v[s] >= o;
            cs[s] += m >= o;
            carry = __shfl_sync(0xffffffffu, m, 31);
        }
    }
#pragma unroll
    for (int s = 0; s < kMtSeg; ++s) {
        if (cu[s]) atomicAdd(&cu_s[s * 32 + lane], cu[s]);
        if (cs[s]) atomicAdd(&cs_s[s * 32 + lane], cs[s]);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < len; j += kMtThreads) {
        if (cu_s[j]) atomicAdd(count_unc + (__ldg(order + j0 + j) - k0), (unsigned long long)cu_s[j]);
        if (cs_s[j]) atomicAdd(count_sd + j0 + j, (unsigned long long)cs_s[j]);
    }
}

int64_t maxt_chunks(int64_t K) { return (K + kMtChunk - 1) / kMtChunk; }

}  // namespace fcd

using namespace fcd;

extern "C" {

int64_t fcd_maxt_ws_bytes(int64_t R1, int64_t K) {
    if (R1 < 1 || K < 1 || R1 > kMtMaxRows || K > kMtMaxCols) return 0;
    return R1 * (K + maxt_chunks(K)) * (int64_t)sizeof(double);
}

int fcd_maxt_counts(const double* T, int64_t R1, int64_t K, int64_t pitch, const int64_t* order, int64_t k0,
                    int64_t k1, int64_t* count_unc, int64_t* count_sd, double* ws, void* stream) {
    FCD_REQUIRE(T != nullptr && order != nullptr && count_unc != nullptr && count_sd != nullptr && ws != nullptr,
                "fcd_maxt_counts: NULL argument");
    FCD_REQUIRE(R1 >= 1 && R1 <= kMtMaxRows, "fcd_maxt_counts: R1=%lld rows (1..%lld)", (long long)R1,
                (long long)kMtMaxRows);
    FCD_REQUIRE(K >= 1 && K <= kMtMaxCols, "fcd_maxt_counts: K=%lld columns (1..%lld)", (long long)K,
                (long long)kMtMaxCols);
    FCD_REQUIRE(pitch >= K && 0 <= k0 && k0 < k1 && k1 <= K, "fcd_maxt_counts: bad shape or family [%lld, %lld)",
                (long long)k0, (long long)k1);
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(T) | reinterpret_cast<uintptr_t>(order) |
                  reinterpret_cast<uintptr_t>(count_unc) | reinterpret_cast<uintptr_t>(count_sd) |
                  reinterpret_cast<uintptr_t>(ws)) & 7) == 0, "fcd_maxt_counts: arrays must be 8-byte aligned");
    const int64_t Kf = k1 - k0;
    const int64_t nchunks = maxt_chunks(Kf);
    FCD_REQUIRE(R1 * nchunks < ((int64_t)1 << 31), "fcd_maxt_counts: %lld x %lld is too large for one launch",
                (long long)R1, (long long)Kf);
    cudaStream_t st = (cudaStream_t)stream;
    double* G = ws;
    double* cm = ws + R1 * Kf;
    cudaError_t err = cudaMemsetAsync(count_unc, 0, Kf * sizeof(int64_t), st);
    if (err == cudaSuccess) err = cudaMemsetAsync(count_sd, 0, Kf * sizeof(int64_t), st);
    FCD_REQUIRE(err == cudaSuccess, "fcd_maxt_counts: %s", cudaGetErrorString(err));
    maxt_gather_kernel<<<(unsigned)(R1 * nchunks), kMtThreads, 0, st>>>(T, pitch, order, Kf, nchunks, G, cm);
    int rc = check_launch("fcd_maxt_counts(gather)");
    if (rc != 0) return rc;
    maxt_carry_kernel<<<(unsigned)((R1 + kMtWarps - 1) / kMtWarps), kMtThreads, 0, st>>>(cm, R1, nchunks);
    rc = check_launch("fcd_maxt_counts(carry)");
    if (rc != 0) return rc;
    // enough CTAs to fill the GPU several times over, each with at least a warp's worth of replicas
    const int64_t slices_max = (R1 + kMtWarps - 1) / kMtWarps;
    int64_t slices = ((int64_t)sm_count() * 8 + nchunks - 1) / nchunks;
    slices = slices < slices_max ? slices : slices_max;
    slices = slices < 65535 ? slices : 65535;
    maxt_count_kernel<<<dim3((unsigned)nchunks, (unsigned)slices), kMtThreads, 0, st>>>(
        G, Kf, R1, nchunks, cm, order, k0, reinterpret_cast<unsigned long long*>(count_unc),
        reinterpret_cast<unsigned long long*>(count_sd));
    return check_launch("fcd_maxt_counts(count)");
}

}  // extern "C"
