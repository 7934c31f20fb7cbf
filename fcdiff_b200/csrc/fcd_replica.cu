// Replica sweeps (BASELINE.json configs[4]: group-label permutations / restarts of one data set).
//
// A relabelling changes WHICH columns of the (C, S) correlation matrix are controls and which are
// patients -- nothing else.  The responsibility planes p_k(x), L(x) (fcd_common.cuh) depend on the
// correlation value and (mu, sigma) only, so they are built ONCE for all S subjects
// (fcd_resp_cache over every column), and a replica's inputs are selections from them:
//   * healthy sufficient statistics of the replica's control columns (fcdiff/fit.py:111-114, 171
//     reduce to S1, S2): fcd_healthy_stats_cols;
//   * edge-major planes of its patient columns: fcd_gather_columns (all planes in one launch).
// Pure data movement (+ one masked sum): no exponential is taken again.
#include "fcdiff_b200.h"
#include "fcd_common.cuh"

namespace fcd {

// S1[c] = sum_h X[c][cols[h]], S2[c] = sum_h X[c][cols[h]]^2: one warp per edge row; the row (S doubles,
// contiguous) is read through L1, the lanes walk the column list.  MASKED: NaN entries are left out and
// S0[c] counts the observed ones (healthy_stats_kernel).
template <bool MASKED>
__global__ void __launch_bounds__(256)
healthy_stats_cols_kernel(const double* __restrict__ X, int64_t C, int64_t pitchS, const int32_t* __restrict__ cols,
                          int H, double* __restrict__ S1, double* __restrict__ S2, double* __restrict__ S0) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = warp0; c < C; c += nwarps) {
        const double* row = X + c * pitchS;
        double s1 = 0.0, s2 = 0.0, s0 = 0.0;
        for (int h = lane; h < H; h += 32) {
            const double x = __ldg(row + __ldg(cols + h));
            if (MASKED && isnan(x)) continue;
            s1 += x;
            s2 = fma(x, x, s2);
            if (MASKED) s0 += 1.0;
        }
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        if (MASKED) s0 = warp_sum(s0);
        if (lane == 0) {
            S1[c] = s1;
            S2[c] = s2;
            if (MASKED) S0[c] = s0;
        }
    }
}

// dst[p][c][j] = src[p][c][cols[j]] for j < U; columns [U, pitchD) are written as zeros.  One warp per
// (plane, row); writes coalesced, reads gathered inside one row (the row is read once either way).
__global__ void __launch_bounds__(256)
gather_columns_kernel(const double* __restrict__ src, int64_t planeStrideS, int64_t pitchS, int nplanes, int64_t C,
                      const int32_t* __restrict__ cols, int U, double* __restrict__ dst, int64_t planeStrideD,
                      int64_t pitchD) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rows = (int64_t)nplanes * C;
    for (int64_t r = warp0; r < rows; r += nwarps) {
        const int64_t p = r / C, c = r - p * C;
        const double* s = src + p * planeStrideS + c * pitchS;
        double* d = dst + p * planeStrideD + c * pitchD;
        for (int j = lane; j < pitchD; j += 32) d[j] = j < U ? __ldg(s + __ldg(cols + j)) : 0.0;
    }
}

}  // namespace fcd

using namespace fcd;

extern "C" {

// S0 == NULL: every control is observed (the unmasked kernel); otherwise NaN entries are left out and S0 counts
// the observed controls of each edge.
int fcd_healthy_stats_cols(const double* X, int64_t C, int64_t pitchS, const int32_t* cols, int32_t H, double* S1,
                           double* S2, double* S0, void* stream) {
    FCD_REQUIRE(X != nullptr && cols != nullptr && S1 != nullptr && S2 != nullptr, "fcd_healthy_stats_cols: NULL argument");
    FCD_REQUIRE(C >= 0 && H >= 1 && pitchS >= 1, "fcd_healthy_stats_cols: bad shape");
    if (C == 0) return 0;
    int64_t grid = (C + 7) / 8;
    if (grid > (int64_t)sm_count() * 16) grid = (int64_t)sm_count() * 16;
    if (S0 == nullptr)
        healthy_stats_cols_kernel<false><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(X, C, pitchS, cols, H, S1, S2,
                                                                                             nullptr);
    else
        healthy_stats_cols_kernel<true><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(X, C, pitchS, cols, H, S1, S2, S0);
    return check_launch("fcd_healthy_stats_cols");
}

int fcd_gather_columns(const double* src, int64_t planeStrideS, int64_t pitchS, int32_t nplanes, int64_t C,
                       const int32_t* cols, int32_t U, double* dst, int64_t planeStrideD, int64_t pitchD, void* stream) {
    FCD_REQUIRE(src != nullptr && cols != nullptr && dst != nullptr, "fcd_gather_columns: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && pitchD >= U && nplanes >= 1 && pitchS >= 1, "fcd_gather_columns: bad shape");
    if (C == 0) return 0;
    int64_t grid = ((int64_t)nplanes * C + 7) / 8;
    if (grid > (int64_t)sm_count() * 16) grid = (int64_t)sm_count() * 16;
    gather_columns_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(src, planeStrideS, pitchS, nplanes, C, cols, U,
                                                                            dst, planeStrideD, pitchD);
    return check_launch("fcd_gather_columns");
}

}  // extern "C"
