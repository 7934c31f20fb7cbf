// K1 -- region time series -> Pearson correlations -> Fisher z, written in the
// edge-major (C, S) layout the EM kernels consume.  No reference counterpart
// (SURVEY 8 a11): the oracle is numpy.corrcoef + numpy.arctanh.
//
// Stage 1 (standardise): each row x[s,n,:] is centred and scaled to unit
//   Euclidean norm in fp64 and stored as fp32 Z[s][n][Tp] (Tp = T rounded up to
//   kKChunk, zero padded), so that R = Z Z^T directly.
// Stage 2 (Gram): R tiles; this file holds the SIMT implementation with fp64
//   accumulation (`gram_simt_kernel`), used for odd shapes and as the numerical
//   yard-stick of the tensor-core implementation (fcd_corr_tc.cu).
// Stage 3 (epilogue, fused into stage 2): clip to [-1, 1], atanh, scatter of the
//   strict lower triangle to out[c][s0 + s], c = n(n-1)/2 + m.
#include "fcd_common.cuh"
#include "fcd_corr.cuh"

#include <cstdlib>

namespace fcd {

// One warp per (subject, region) row.  SPLIT: write the TF32 hi / lo parts
// (both exactly representable in TF32) for the tensor-core path.
// MASK (fcd_corr_fisherz_clean without confounds): only the frames t with keep[s][t] != 0 (every frame
// when keep is NULL) are read; the others are written as zeros.  The sums are those of the unmasked form
// in the same order, divided by the number of kept frames, so an all-kept mask gives the same bits.  A
// row with a non-finite kept sample or of zero variance is written as zeros, and status[r] = 1 marks it.
// OutT = double (fcd_corr_partial, MASK only): the fp64 rows are stored as they are computed.
template <bool SPLIT, bool MASK = false, typename OutT = float>
__global__ void __launch_bounds__(256)
standardise_kernel(const float* __restrict__ ts, int64_t rows, int T, int Tp, OutT* __restrict__ Z,
                   float* __restrict__ Zlo, const uint8_t* __restrict__ keep = nullptr, int N = 0,
                   uint8_t* __restrict__ status = nullptr) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < rows; r += nwarps) {
        const float* x = ts + r * T;
        const uint8_t* kp = MASK && keep != nullptr ? keep + (r / N) * T : nullptr;
        double s = 0.0;
        int cnt = 0;
        for (int t = lane; t < T; t += 32) {
            if (MASK && kp != nullptr && !kp[t]) continue;
            s += (double)x[t];
            if (MASK) ++cnt;
        }
        const double mean = warp_sum(s) / (double)(MASK ? __reduce_add_sync(0xffffffffu, cnt) : T);
        double ss = 0.0;
        for (int t = lane; t < T; t += 32) {
            if (MASK && kp != nullptr && !kp[t]) continue;
            const double d = (double)x[t] - mean;
            ss = fma(d, d, ss);
        }
        ss = warp_sum(ss);
        const double inv = ss > 0.0 ? rsqrt(ss) : 0.0;
        if (MASK && lane == 0) status[r] = ss > 0.0 ? 0 : 1;
        for (int t = lane; t < Tp; t += 32) {
            const bool use = t < T && (!MASK || (ss > 0.0 && (kp == nullptr || kp[t])));
            const OutT z = use ? (OutT)(((double)x[t] - mean) * inv) : (OutT)0;
            if constexpr (SPLIT) {
                uint32_t hb, lb;
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(z));
                const float zh = __uint_as_float(hb);
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(z - zh));
                Z[r * Tp + t] = zh;
                Zlo[r * Tp + t] = __uint_as_float(lb);
            } else {
                Z[r * Tp + t] = z;
            }
        }
    }
}

// 32x32 output tile per CTA (lower-triangular tiles only), 256 threads, each
// thread a 2x2 micro-tile, fp64 accumulation of fp32 products.
__global__ void __launch_bounds__(256)
gram_simt_kernel(const float* __restrict__ Z, int N, int Tp, int ntile,
                 double* __restrict__ out, int64_t pitch, int s0, int fisher) {
    __shared__ float sa[32][33];
    __shared__ float sb[32][33];
    // linear lower-triangular tile index -> (ti >= tj)
    int ti, tj;
    c_to_nm((int64_t)blockIdx.x + 0, ti, tj);      // reuse: (ti-1, tj) enumerates ti-1 >= tj
    ti -= 1;
    (void)ntile;
    const int s = blockIdx.y;
    const float* Zs = Z + (int64_t)s * N * Tp;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // 16 x 16
    double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
    for (int k0 = 0; k0 < Tp; k0 += 32) {
        for (int i = threadIdx.x; i < 32 * 32; i += 256) {
            const int r = i >> 5, k = i & 31;
            const int na = ti * 32 + r, nb = tj * 32 + r;
            sa[r][k] = na < N ? Zs[(int64_t)na * Tp + k0 + k] : 0.0f;
            sb[r][k] = nb < N ? Zs[(int64_t)nb * Tp + k0 + k] : 0.0f;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < 32; ++k) {
            const double a0 = sa[ty][k], a1 = sa[ty + 16][k];
            const double b0 = sb[tx][k], b1 = sb[tx + 16][k];
            acc[0][0] = fma(a0, b0, acc[0][0]);
            acc[0][1] = fma(a0, b1, acc[0][1]);
            acc[1][0] = fma(a1, b0, acc[1][0]);
            acc[1][1] = fma(a1, b1, acc[1][1]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int n = ti * 32 + ty + 16 * i, m = tj * 32 + tx + 16 * j;
            if (n < N && m < n) {
                const int64_t c = (int64_t)n * (n - 1) / 2 + m;
                out[c * pitch + s0 + s] = corr_epilogue(acc[i][j], fisher);
            }
        }
}

// Rows without a usable time series: one warp per (subject, region) row, the sums of standardise_kernel in
// the same order.  A row with a non-finite sample, or of zero variance, gets NaN (not observed) on every
// one of its N - 1 edges in column s0 + s.  (standardise_kernel cannot tell such a row from a real
// zero correlation: it writes zeros, and a NaN sample ends up as the negative clip.)
__global__ void __launch_bounds__(256)
mark_missing_kernel(const float* __restrict__ ts, int S, int N, int T, double* __restrict__ out, int64_t pitch,
                    int s0) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rows = (int64_t)S * N;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    for (int64_t r = warp0; r < rows; r += nwarps) {
        const float* x = ts + r * T;
        double s = 0.0;
        for (int t = lane; t < T; t += 32) s += (double)x[t];
        const double mean = warp_sum(s) / (double)T;
        double ss = 0.0;
        for (int t = lane; t < T; t += 32) {
            const double d = (double)x[t] - mean;
            ss = fma(d, d, ss);
        }
        ss = warp_sum(ss);
        if (ss > 0.0) continue;                               // also false for NaN: an inf or NaN sample
        const int subj = (int)(r / N), n = (int)(r - (int64_t)subj * N);
        for (int m = lane; m < N; m += 32) {
            if (m == n) continue;
            const int64_t c = n > m ? (int64_t)n * (n - 1) / 2 + m : (int64_t)m * (m - 1) / 2 + n;
            out[c * pitch + s0 + subj] = nan;
        }
    }
}

// Rows flagged by the cleaning stage (status[s][n] != 0): NaN on their N - 1 edges of column s0 + s, one
// warp per row; every other entry is left as it is.
__global__ void __launch_bounds__(256)
mark_status_kernel(const uint8_t* __restrict__ status, int S, int N, double* __restrict__ out, int64_t pitch,
                   int s0) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rows = (int64_t)S * N;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    for (int64_t r = warp0; r < rows; r += nwarps) {
        if (!status[r]) continue;
        const int subj = (int)(r / N), n = (int)(r - (int64_t)subj * N);
        for (int m = lane; m < N; m += 32) {
            if (m == n) continue;
            const int64_t c = n > m ? (int64_t)n * (n - 1) / 2 + m : (int64_t)m * (m - 1) / 2 + n;
            out[c * pitch + s0 + subj] = nan;
        }
    }
}

static int row_grid(int64_t rows) {
    const int64_t g = (rows + 7) / 8;
    const int64_t cap = (int64_t)sm_count() * 8;
    return (int)(g < cap ? g : cap);
}

bool corr_use_tc(int N) { return corr_tc_supported(N) && getenv("FCD_CORR_SIMT") == nullptr; }

int corr_gram(bool tc, const float* Z, const float* Zlo, int S, int N, int Tp, double* out, int64_t pitch, int s0,
              int fisher, cudaStream_t st) {
    if (tc) return corr_gram_tc(Z, Zlo, S, N, Tp, out, pitch, s0, fisher, st);
    FCD_REQUIRE(S <= 65535, "fcd_corr_fisherz: S=%d too large for the SIMT Gram kernel", S);
    const int nt = (N + 31) / 32;
    dim3 grid((unsigned)(nt * (nt + 1) / 2), (unsigned)S);
    gram_simt_kernel<<<grid, 256, 0, st>>>(Z, N, Tp, nt, out, pitch, s0, fisher);
    return check_launch("fcd_corr_fisherz(gram_simt)");
}

int corr_standardise_masked(bool tc, const float* ts, const uint8_t* keep, int S, int N, int T, int Tp, float* Z,
                            float* Zlo, uint8_t* status, cudaStream_t st) {
    const int64_t rows = (int64_t)S * N;
    if (tc) standardise_kernel<true, true><<<row_grid(rows), 256, 0, st>>>(ts, rows, T, Tp, Z, Zlo, keep, N, status);
    else standardise_kernel<false, true><<<row_grid(rows), 256, 0, st>>>(ts, rows, T, Tp, Z, nullptr, keep, N, status);
    return check_launch("fcd_corr_fisherz_clean(standardise)");
}

int corr_standardise_masked_f64(const float* ts, const uint8_t* keep, int S, int N, int T, int Tp, double* Z,
                                uint8_t* status, cudaStream_t st) {
    const int64_t rows = (int64_t)S * N;
    standardise_kernel<false, true, double><<<row_grid(rows), 256, 0, st>>>(ts, rows, T, Tp, Z, nullptr, keep, N,
                                                                            status);
    return check_launch("fcd_corr_partial(standardise)");
}

int corr_mark_status(const uint8_t* status, int S, int N, double* out, int64_t pitch, int s0, cudaStream_t st) {
    mark_status_kernel<<<row_grid((int64_t)S * N), 256, 0, st>>>(status, S, N, out, pitch, s0);
    return check_launch("fcd_corr_fisherz_clean(mark)");
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int64_t fcd_corr_workspace_bytes(int32_t S, int32_t N, int32_t T) {
    if (S < 0 || N < 0 || T < 0) return -1;
    return 2 * ((int64_t)S * N * corr_padded_T(T) * (int64_t)sizeof(float) + 1024) + 1024;
}

int fcd_corr_fisherz(const float* ts, int32_t S, int32_t N, int32_t T,
                     double* out, int64_t pitch, int32_t s0, int32_t fisher,
                     void* zws, void* stream) {
    FCD_REQUIRE(ts != nullptr && out != nullptr && zws != nullptr, "fcd_corr_fisherz: NULL argument");
    FCD_REQUIRE(S >= 0 && N >= 2 && T >= 2 && s0 >= 0 && pitch >= (int64_t)s0 + S && S <= 65535 * 4,
                "fcd_corr_fisherz: bad shape S=%d N=%d T=%d s0=%d pitch=%lld", S, N, T, s0, (long long)pitch);
    if (S == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int Tp = corr_padded_T(T);
    // 1024-byte aligned scratch planes (TMA / UMMA operand tiles need it)
    const int64_t plane = (((int64_t)S * N * Tp * (int64_t)sizeof(float)) + 1023) & ~(int64_t)1023;
    float* Z = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(zws) + 1023) & ~(uintptr_t)1023);
    float* Zlo = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(Z) + plane);
    const int64_t rows = (int64_t)S * N;
    int64_t g = (rows + 7) / 8;
    const int64_t cap = (int64_t)sm_count() * 8;
    const int grid1 = (int)(g < cap ? g : cap);
    const bool tc = corr_tc_supported(N) && getenv("FCD_CORR_SIMT") == nullptr;
    if (tc) standardise_kernel<true><<<grid1, 256, 0, st>>>(ts, rows, T, Tp, Z, Zlo);
    else standardise_kernel<false><<<grid1, 256, 0, st>>>(ts, rows, T, Tp, Z, nullptr);
    int rc = check_launch("fcd_corr_fisherz(standardise)");
    if (rc) return rc;
    return corr_gram(tc, Z, Zlo, S, N, Tp, out, pitch, s0, fisher, st);
}

int fcd_corr_mark_missing(const float* ts, int32_t S, int32_t N, int32_t T, double* out, int64_t pitch, int32_t s0,
                          void* stream) {
    FCD_REQUIRE(ts != nullptr && out != nullptr, "fcd_corr_mark_missing: NULL argument");
    FCD_REQUIRE(S >= 0 && N >= 2 && T >= 2 && s0 >= 0 && pitch >= (int64_t)s0 + S,
                "fcd_corr_mark_missing: bad shape S=%d N=%d T=%d s0=%d pitch=%lld", S, N, T, s0, (long long)pitch);
    if (S == 0) return 0;
    const int64_t rows = (int64_t)S * N;
    int64_t g = (rows + 7) / 8;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (g > cap) g = cap;
    mark_missing_kernel<<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(ts, S, N, T, out, pitch, s0);
    return check_launch("fcd_corr_mark_missing");
}

}  // extern "C"
