// K1 cleaning stage: correlations from censored, ragged and confound-regressed time series
// (fcd_corr_fisherz_clean).  No reference counterpart; oracle: oracle/clean.py (lstsq on [1, G] over the
// kept frames, numpy.corrcoef of the residuals, numpy.arctanh).
//
// For subject s, keep[s][t] selects the frames that enter the correlations (a padded or censored frame
// has keep = 0) and G_s = confounds[s][kept t][0..K) the nuisance regressors.  Every region row x is
//   1. centred over the kept frames,                         x_c = x - mean_kept(x);
//   2. cleared of the confounds,                             e = x_c - Q_s Q_s^T x_c,
//      Q_s an orthonormal basis of the centred G_s over the kept frames (confound_basis_kernel);
//   3. scaled to unit norm,                                  z = e / |e|, zero on every frame not kept,
// and R = Z Z^T is the Gram stage of fcd_corr_fisherz, unchanged (a frame not kept is a zero column of Z).
// r_nm is then the partial correlation of regions n and m given the confounds and a constant.  A sample
// of a frame that is not kept is never read into arithmetic (selected, never multiplied by 0), so NaN or
// inf there has no effect.  Without confounds the standardisation is standardise_kernel<SPLIT, true>
// (fcd_corr.cu); this file holds the K >= 1 form.
#include "fcd_corr.cuh"

namespace fcd {

constexpr int kMaxConfounds = 64;
constexpr int kCleanChunk = 64;             // frames of Q staged in shared memory per step
constexpr double kRankTol = 1e-10;          // drop a confound whose residual norm is <= kRankTol * its raw norm
constexpr int kBasisThreads = 256;

// One CTA per subject.  Q[s][j][0..Tp) is column j of the confounds over the kept frames, centred, then
// orthonormalised by modified Gram-Schmidt (right-looking: once column j is final, it is projected out of
// every later column, one warp per column), run twice; the second pass restores orthogonality to fp64
// rounding.  A column whose norm after projection is <= kRankTol times its raw norm over the kept frames
// (pass 1) or <= kRankTol (pass 2, unit columns) is dropped: written as zeros.  This covers exact
// duplicates, constant columns and columns that are zero on the kept frames.  rank[s] = the columns kept.
// Every sum runs over t in a fixed thread / lane order in which frames that are not kept contribute exact
// zeros, so padding a subject with censored frames changes no bit.
__global__ void __launch_bounds__(kBasisThreads)
confound_basis_kernel(const double* __restrict__ confounds, const uint8_t* __restrict__ keep, int T, int Tp, int K,
                      double* __restrict__ Q, int32_t* __restrict__ rank) {
    __shared__ double sh_ref[kMaxConfounds];
    __shared__ double sh_scale;
    __shared__ int sh_cnt[kBasisThreads / 32];
    const int s = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = kBasisThreads / 32;
    const uint8_t* kp = keep != nullptr ? keep + (int64_t)s * T : nullptr;
    const double* g = confounds + (int64_t)s * T * K;
    double* q = Q + (int64_t)s * K * Tp;
    // transpose to frame-contiguous columns, selecting the kept frames
    for (int t = 0; t < Tp; t += kBasisThreads / K) {          // K <= 64 < kBasisThreads: whole frames per step
        const int tt = t + (int)threadIdx.x / K, j = (int)threadIdx.x % K;
        if (tt >= Tp || (int)threadIdx.x >= kBasisThreads / K * K) continue;
        const bool kept = tt < T && (kp == nullptr || kp[tt]);
        q[(int64_t)j * Tp + tt] = kept ? g[(int64_t)tt * K + j] : 0.0;
    }
    int cnt = 0;
    for (int t = threadIdx.x; t < T; t += kBasisThreads) cnt += (kp == nullptr || kp[t]) ? 1 : 0;
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) sh_cnt[warp] = cnt;
    __syncthreads();
    int n_s = 0;
    for (int w = 0; w < nw; ++w) n_s += sh_cnt[w];
    // centre each column over the kept frames (one warp per column); its raw norm is the drop reference
    for (int j = warp; j < K; j += nw) {
        double* c = q + (int64_t)j * Tp;
        double sum = 0.0, sq = 0.0;
        for (int t = lane; t < Tp; t += 32) {
            sum += c[t];
            sq = fma(c[t], c[t], sq);
        }
        const double mean = warp_sum(sum) / (double)n_s;
        sq = warp_sum(sq);
        for (int t = lane; t < Tp; t += 32) {
            const bool kept = t < T && (kp == nullptr || kp[t]);
            c[t] = kept ? c[t] - mean : 0.0;
        }
        if (lane == 0) sh_ref[j] = sqrt(sq);
    }
    __syncthreads();
    int kept_cols = 0;
    for (int pass = 0; pass < 2; ++pass) {
        kept_cols = 0;
        for (int j = 0; j < K; ++j) {
            double* cj = q + (int64_t)j * Tp;
            if (warp == 0) {
                double sq = 0.0;
                for (int t = lane; t < Tp; t += 32) sq = fma(cj[t], cj[t], sq);
                const double nrm = sqrt(warp_sum(sq));
                const double ref = pass == 0 ? sh_ref[j] : 1.0;
                if (lane == 0) sh_scale = nrm > kRankTol * ref ? 1.0 / nrm : 0.0;
            }
            __syncthreads();
            const double scale = sh_scale;
            kept_cols += scale > 0.0 ? 1 : 0;
            for (int t = threadIdx.x; t < Tp; t += kBasisThreads) cj[t] = scale > 0.0 ? cj[t] * scale : 0.0;
            __syncthreads();
            if (scale > 0.0) {
                for (int i = j + 1 + warp; i < K; i += nw) {
                    double* ci = q + (int64_t)i * Tp;
                    double d = 0.0;
                    for (int t = lane; t < Tp; t += 32) d = fma(cj[t], ci[t], d);
                    d = warp_sum(d);
                    for (int t = lane; t < Tp; t += 32) ci[t] = fma(-d, cj[t], ci[t]);
                }
            }
            __syncthreads();
        }
    }
    if (rank != nullptr && threadIdx.x == 0) rank[s] = kept_cols;
}

// One CTA of W warps per (block of W regions, subject); warp w cleans row n = blockIdx.x * W + w.  The row
// is read from global memory once into shared memory (fp64, W * Tp doubles) and stays there through the
// mean, projection and norm passes.  The subject's Q is staged kCleanChunk frames at a time into shared
// memory and read there by all W warps.  Per lane: t = lane + 32 i, so each lane's partial sums run over
// increasing t and frames beyond the kept ones add exact zeros (padding changes no bit).  The K dot
// products accumulate in registers (KMAX >= K, unrolled) and are reduced once per row.
// A row is unusable when a kept sample is non-finite or its residual sum of squares is at most 2^-40 of
// its centred sum of squares (the region is explained by the confounds to the rounding of its fp32
// input): it is written as zeros and status = 1.  OutT = double (fcd_corr_partial): the fp64 rows are stored.
template <bool SPLIT, int KMAX, typename OutT = float>
__global__ void __launch_bounds__(256)
clean_kernel(const float* __restrict__ ts, const uint8_t* __restrict__ keep, const double* __restrict__ Q, int N,
             int T, int Tp, int K, OutT* __restrict__ Z, float* __restrict__ Zlo, uint8_t* __restrict__ status) {
    extern __shared__ double smem_d[];
    const int W = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int s = blockIdx.y, n = blockIdx.x * W + warp;
    const bool live = n < N;
    double* qs = smem_d;                                        // [K][kCleanChunk]
    double* buf = smem_d + (size_t)K * kCleanChunk + (size_t)warp * Tp;
    const uint8_t* kp = keep != nullptr ? keep + (int64_t)s * T : nullptr;
    const double* qg = Q + (int64_t)s * K * Tp;
    const int64_t r = (int64_t)s * N + n;

    double mean = 0.0, ssc = 0.0;
    if (live) {
        const float* x = ts + r * T;
        double sum = 0.0;
        int cnt = 0;
        for (int t = lane; t < Tp; t += 32) {
            const bool kept = t < T && (kp == nullptr || kp[t]);
            const double v = kept ? (double)x[t] : 0.0;
            buf[t] = v;
            if (kept) {
                sum += v;
                ++cnt;
            }
        }
        mean = warp_sum(sum) / (double)__reduce_add_sync(0xffffffffu, cnt);
        for (int t = lane; t < Tp; t += 32) {
            const bool kept = t < T && (kp == nullptr || kp[t]);
            const double d = kept ? buf[t] - mean : 0.0;
            buf[t] = d;
            ssc = fma(d, d, ssc);
        }
        ssc = warp_sum(ssc);
    }
    // c_k = q_k . x_c
    double c[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) c[k] = 0.0;
    for (int t0 = 0; t0 < Tp; t0 += kCleanChunk) {
        __syncthreads();
        for (int i = threadIdx.x; i < K * kCleanChunk; i += blockDim.x) {
            const int k = i / kCleanChunk, t = t0 + (i - k * kCleanChunk);
            qs[i] = t < Tp ? qg[(int64_t)k * Tp + t] : 0.0;
        }
        __syncthreads();
        if (live) {
#pragma unroll
            for (int h = 0; h < kCleanChunk / 32; ++h) {
                const int t = t0 + h * 32 + lane;
                const double d = t < Tp ? buf[t] : 0.0;
#pragma unroll
                for (int k = 0; k < KMAX; ++k)
                    if (k < K) c[k] = fma(qs[k * kCleanChunk + h * 32 + lane], d, c[k]);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
        if (k < K) c[k] = warp_sum(c[k]);
    // e = x_c - sum_k c_k q_k, in place
    double sse = 0.0;
    for (int t0 = 0; t0 < Tp; t0 += kCleanChunk) {
        __syncthreads();
        for (int i = threadIdx.x; i < K * kCleanChunk; i += blockDim.x) {
            const int k = i / kCleanChunk, t = t0 + (i - k * kCleanChunk);
            qs[i] = t < Tp ? qg[(int64_t)k * Tp + t] : 0.0;
        }
        __syncthreads();
        if (live) {
#pragma unroll
            for (int h = 0; h < kCleanChunk / 32; ++h) {
                const int t = t0 + h * 32 + lane;
                if (t < Tp) {
                    double e = buf[t];
#pragma unroll
                    for (int k = 0; k < KMAX; ++k)
                        if (k < K) e = fma(-c[k], qs[k * kCleanChunk + h * 32 + lane], e);
                    buf[t] = e;
                    sse = fma(e, e, sse);
                }
            }
        }
    }
    if (!live) return;
    sse = warp_sum(sse);
    const bool usable = sse > ldexp(ssc, -40);                  // false for NaN; with sse >= 0 also for ssc = 0
    const double inv = usable ? rsqrt(sse) : 0.0;
    if (lane == 0) status[r] = usable ? 0 : 1;
    for (int t = lane; t < Tp; t += 32) {
        const bool kept = t < T && (kp == nullptr || kp[t]);
        const OutT z = usable && kept ? (OutT)(buf[t] * inv) : (OutT)0;
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

// Warps per CTA of clean_kernel: up to 8 rows, as many as the rows' buffers and the Q chunk leave room for.
static int clean_warps(int Tp, int K) {
    const int64_t free_bytes = (int64_t)kSmemBudget - (int64_t)K * kCleanChunk * 8;
    const int64_t w = free_bytes / ((int64_t)Tp * 8);
    return (int)(w < 8 ? w : 8);
}

template <bool SPLIT, int KMAX, typename OutT>
static int launch_clean(const float* ts, const uint8_t* keep, const double* Q, int S, int N, int T, int Tp, int K,
                        OutT* Z, float* Zlo, uint8_t* status, cudaStream_t st) {
    const int W = clean_warps(Tp, K);
    const size_t smem = ((size_t)K * kCleanChunk + (size_t)W * Tp) * sizeof(double);
    FCD_ALLOW_BIG_SMEM(clean_kernel<SPLIT, KMAX, OutT>);
    dim3 grid((unsigned)((N + W - 1) / W), (unsigned)S);
    clean_kernel<SPLIT, KMAX, OutT><<<grid, 32 * W, smem, st>>>(ts, keep, Q, N, T, Tp, K, Z, Zlo, status);
    return check_launch("fcd_corr_fisherz_clean(clean)");
}

template <bool SPLIT, typename OutT = float>
static int launch_clean_k(const float* ts, const uint8_t* keep, const double* Q, int S, int N, int T, int Tp, int K,
                          OutT* Z, float* Zlo, uint8_t* status, cudaStream_t st) {
    if (K <= 8) return launch_clean<SPLIT, 8>(ts, keep, Q, S, N, T, Tp, K, Z, Zlo, status, st);
    if (K <= 16) return launch_clean<SPLIT, 16>(ts, keep, Q, S, N, T, Tp, K, Z, Zlo, status, st);
    if (K <= 32) return launch_clean<SPLIT, 32>(ts, keep, Q, S, N, T, Tp, K, Z, Zlo, status, st);
    return launch_clean<SPLIT, 64>(ts, keep, Q, S, N, T, Tp, K, Z, Zlo, status, st);
}

int corr_clean_f64(const float* ts, const uint8_t* keep, const double* confounds, int S, int N, int T, int Tp, int K,
                   double* Q, double* Z, uint8_t* status, int32_t* rank, cudaStream_t st) {
    FCD_REQUIRE(clean_warps(Tp, K) >= 1, "fcd_corr_partial: T=%d too long for K=%d confounds", T, K);
    confound_basis_kernel<<<S, kBasisThreads, 0, st>>>(confounds, keep, T, Tp, K, Q, rank);
    const int rc = check_launch("fcd_corr_partial(basis)");
    if (rc) return rc;
    return launch_clean_k<false>(ts, keep, Q, S, N, T, Tp, K, Z, nullptr, status, st);
}

// Workspace layout: Z and Zlo planes (as fcd_corr_fisherz), the status bytes [S][N], Q [S][K][Tp].
struct CleanWs {
    float* Z;
    float* Zlo;
    uint8_t* status;
    double* Q;
};

static int64_t align1k(int64_t b) { return (b + 1023) & ~(int64_t)1023; }

static CleanWs clean_ws(void* zws, int S, int N, int Tp) {
    CleanWs w;
    const int64_t plane = align1k((int64_t)S * N * Tp * (int64_t)sizeof(float));
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(zws) + 1023) & ~(uintptr_t)1023);
    w.Z = reinterpret_cast<float*>(base);
    w.Zlo = reinterpret_cast<float*>(base + plane);
    w.status = base + 2 * plane;
    w.Q = reinterpret_cast<double*>(base + 2 * plane + align1k((int64_t)S * N));
    return w;
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int64_t fcd_corr_clean_workspace_bytes(int32_t S, int32_t N, int32_t T, int32_t K) {
    if (S < 0 || N < 0 || T < 0 || K < 0 || K > kMaxConfounds) return -1;
    const int64_t Tp = corr_padded_T(T);
    return 1024 + 2 * align1k((int64_t)S * N * Tp * (int64_t)sizeof(float)) + align1k((int64_t)S * N) +
           (int64_t)S * K * Tp * (int64_t)sizeof(double);
}

int fcd_corr_fisherz_clean(const float* ts, int32_t S, int32_t N, int32_t T, const uint8_t* keep,
                           const double* confounds, int32_t K, double* out, int64_t pitch, int32_t s0, int32_t fisher,
                           int32_t mark_missing, int32_t* rank, void* zws, void* stream) {
    FCD_REQUIRE(ts != nullptr && out != nullptr && zws != nullptr, "fcd_corr_fisherz_clean: NULL argument");
    FCD_REQUIRE(S >= 0 && N >= 2 && T >= 2 && s0 >= 0 && pitch >= (int64_t)s0 + S && S <= 65535,
                "fcd_corr_fisherz_clean: bad shape S=%d N=%d T=%d s0=%d pitch=%lld", S, N, T, s0, (long long)pitch);
    FCD_REQUIRE(K >= 0 && K <= kMaxConfounds && (K == 0) == (confounds == nullptr),
                "fcd_corr_fisherz_clean: K=%d needs 0 <= K <= %d and confounds NULL iff K == 0", K, kMaxConfounds);
    if (S == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int Tp = corr_padded_T(T);
    const CleanWs w = clean_ws(zws, S, N, Tp);
    const bool tc = corr_use_tc(N);
    int rc;
    if (K == 0) {
        rc = corr_standardise_masked(tc, ts, keep, S, N, T, Tp, w.Z, tc ? w.Zlo : nullptr, w.status, st);
        if (rc) return rc;
        if (rank != nullptr) {
            FCD_REQUIRE(cudaMemsetAsync(rank, 0, (size_t)S * sizeof(int32_t), st) == cudaSuccess,
                        "fcd_corr_fisherz_clean: cudaMemsetAsync(rank) failed");
        }
    } else {
        FCD_REQUIRE(clean_warps(Tp, K) >= 1, "fcd_corr_fisherz_clean: T=%d too long for K=%d confounds", T, K);
        confound_basis_kernel<<<S, kBasisThreads, 0, st>>>(confounds, keep, T, Tp, K, w.Q, rank);
        rc = check_launch("fcd_corr_fisherz_clean(basis)");
        if (rc) return rc;
        rc = tc ? launch_clean_k<true>(ts, keep, w.Q, S, N, T, Tp, K, w.Z, w.Zlo, w.status, st)
                : launch_clean_k<false>(ts, keep, w.Q, S, N, T, Tp, K, w.Z, nullptr, w.status, st);
        if (rc) return rc;
    }
    rc = corr_gram(tc, w.Z, w.Zlo, S, N, Tp, out, pitch, s0, fisher, st);
    if (rc || !mark_missing) return rc;
    return corr_mark_status(w.status, S, N, out, pitch, s0, st);
}

}  // extern "C"
