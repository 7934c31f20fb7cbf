// K1 partial correlations (fcd_corr_partial): Ledoit-Wolf shrunk covariance and one fp64 SPD inverse per
// subject.  No reference counterpart; oracle: oracle/partial.py (sklearn's ledoit_wolf restated,
// numpy.linalg.inv).
//
// Per subject s with n_s kept frames, in batches of subjects that bound the workspace:
//   1. standardise / clean to fp64 rows z_n (unit norm over the kept frames, zero elsewhere): the rows
//      fcd_corr_fisherz_clean forms, without the rounding to fp32 (corr_standardise_masked_f64,
//      corr_clean_f64);
//   2. R = Z Z^T (= X^T X / n_s for the unit-variance rows X = sqrt(n_s) Z^T), lower triangle, fp64 SIMT
//      (partial_gram_kernel), and the per-frame w_t = sum_n z_nt^2 (frame_sq_kernel);
//   3. Ledoit-Wolf over the N_s usable regions (partial_shrink_kernel): mu = tr R / N_s,
//      d2 = |R - mu I|_F^2 / N_s, b2 = min(d2, (n_s sum_t w_t^2 - |R|_F^2) / (n_s N_s)) (sum_t |x_t|^4 / n_s
//      = n_s sum_t w_t^2), delta = b2 / d2 (0 unless b2 > 0), or the fixed shrinkage; Sigma =
//      (1 - delta) R + delta mu I, and the row and column of an unusable region set to e_n;
//   4. -P = -Sigma^-1 in place by the blocked symmetric sweep (partial_invert_kernel);
//   5. r_nm = -P_nm / sqrt(P_nn P_mm), the clip / atanh of corr_epilogue, and the NaN marks of the
//      unusable regions (partial_epilogue_kernel, corr_mark_status).
// Every sum runs in an order fixed by the shapes N and the thread layout, in which frames that are not
// kept add exact zeros: a subject's column has the same bits alone, in a batch, padded or censored further.
// The Gram is fp64 on purpose: Sigma's condition number reaches ~4e3 at 400 regions, which turns the
// ~1e-6 of the split-TF32 Gram (or the 1e-8 of rows rounded to fp32) into visible errors of partial r.
// B200's fp64 rate is the same on DMMA and DFMA, so the register-blocked DFMA tile needs no tensor cores.
#include "fcd_corr.cuh"

#include <cstdlib>

namespace fcd {

constexpr int kPT = 64;                     // output tile edge (Gram, sweep update), 256 threads x 4 x 4
constexpr int kPLd = kPT + 1;               // padded shared-memory row of a tile operand
constexpr int kPKc = 16;                    // frames per Gram step
constexpr int kPNb = 64;                    // pivots per sweep block
constexpr double kPivotTol = 9.094947017729282e-13;    // 2^-40: a pivot <= this (Sigma's diagonal is ~1) fails
constexpr int64_t kPartialWsBudget = (int64_t)4 << 30; // bytes of batch workspace the call aims for
constexpr int kMaxConfoundsPartial = 64;

// acc[i][j] (+/-)= sum_k a[k][ty + 16 i] * b[k][tx + 16 j], operands [k][kPLd] in shared memory.
template <bool SUB>
__device__ __forceinline__ void tile_fma(const double* a, const double* b, int kb, int ty, int tx,
                                         double (&acc)[4][4]) {
#pragma unroll 4
    for (int k = 0; k < kb; ++k) {
        double av[4], bv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            av[i] = a[k * kPLd + ty + 16 * i];
            bv[i] = b[k * kPLd + tx + 16 * i];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fma(SUB ? -av[i] : av[i], bv[j], acc[i][j]);
    }
}

// Deterministic CTA sum (256 threads): warp sums, then warp 0 over the 8 partials in order.
__device__ __forceinline__ double block_sum256(double v, double* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double t = lane < 8 ? sh[lane] : 0.0;
    t = warp_sum(t);
    return t;                                  // valid in every warp (each reduces the same 8 values)
}

// Entry (i, j) of the symmetric matrix from its lower triangle.
__device__ __forceinline__ int64_t sym_at(int N, int i, int j) {
    return i >= j ? (int64_t)i * N + j : (int64_t)j * N + i;
}

// R[s] = Z_s Z_s^T, lower-triangular 64 x 64 tiles (ti >= tj), entries n >= m written.
__global__ void __launch_bounds__(256)
partial_gram_kernel(const double* __restrict__ Z, int N, int Tp, double* __restrict__ A) {
    __shared__ double sa[kPKc * kPLd];
    __shared__ double sb[kPKc * kPLd];
    int ti, tj;
    c_to_nm((int64_t)blockIdx.x, ti, tj);
    ti -= 1;
    const int s = blockIdx.y;
    const double* Zs = Z + (int64_t)s * N * Tp;
    double* As = A + (int64_t)s * N * N;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    double acc[4][4] = {};
    for (int k0 = 0; k0 < Tp; k0 += kPKc) {                  // Tp is a multiple of kPKc
        for (int i = threadIdx.x; i < kPT * kPKc; i += 256) {
            const int r = i / kPKc, k = i - r * kPKc;
            const int na = ti * kPT + r, nb = tj * kPT + r;
            sa[k * kPLd + r] = na < N ? Zs[(int64_t)na * Tp + k0 + k] : 0.0;
            sb[k * kPLd + r] = nb < N ? Zs[(int64_t)nb * Tp + k0 + k] : 0.0;
        }
        __syncthreads();
        tile_fma<false>(sa, sb, kPKc, ty, tx, acc);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = ti * kPT + ty + 16 * i, m = tj * kPT + tx + 16 * j;
            if (n < N && m <= n) As[(int64_t)n * N + m] = acc[i][j];
        }
}

// w[s][t] = sum_n z_nt^2 in increasing n (zero on frames that are not kept).
__global__ void __launch_bounds__(128)
frame_sq_kernel(const double* __restrict__ Z, int N, int Tp, double* __restrict__ w) {
    const int s = blockIdx.y, t = blockIdx.x * 128 + threadIdx.x;
    if (t >= Tp) return;
    const double* z = Z + (int64_t)s * N * Tp + t;
    double acc = 0.0;
    for (int n = 0; n < N; ++n) acc = fma(z[(int64_t)n * Tp], z[(int64_t)n * Tp], acc);
    w[(int64_t)s * Tp + t] = acc;
}

// One CTA per subject: Ledoit-Wolf (shrinkage < 0) or the fixed shrinkage, then Sigma in place over A's
// lower triangle; an unusable region (status != 0) gets the row and column of e_n.  delta -> dout[s].
__global__ void __launch_bounds__(256)
partial_shrink_kernel(double* __restrict__ A, const double* __restrict__ w, const uint8_t* __restrict__ status,
                      const uint8_t* __restrict__ keep, int N, int T, int Tp, double shrinkage,
                      double* __restrict__ dout) {
    __shared__ double sh[8];
    const int s = blockIdx.x;
    double* As = A + (int64_t)s * N * N;
    const uint8_t* st = status + (int64_t)s * N;
    const int64_t L = (int64_t)N * (N + 1) / 2;                // lower triangle, diagonal included
    double ns = 0.0, nu = 0.0, tr = 0.0, rf = 0.0, sw = 0.0;
    for (int t = threadIdx.x; t < T; t += 256) ns += (keep == nullptr || keep[(int64_t)s * T + t]) ? 1.0 : 0.0;
    for (int t = threadIdx.x; t < Tp; t += 256) {
        const double v = w[(int64_t)s * Tp + t];
        sw = fma(v, v, sw);
    }
    for (int n = threadIdx.x; n < N; n += 256)
        if (!st[n]) {
            nu += 1.0;
            tr += As[(int64_t)n * N + n];
        }
    for (int64_t c = threadIdx.x; c < L; c += 256) {
        int n, m;
        c_to_nm(c, n, m);                                      // n > m, (n - 1, m) enumerates n - 1 >= m
        n -= 1;
        if (st[n] || st[m]) continue;
        const double v = As[(int64_t)n * N + m];
        rf = fma(n == m ? v : 2.0 * v, v, rf);
    }
    ns = block_sum256(ns, sh);
    nu = block_sum256(nu, sh);
    tr = block_sum256(tr, sh);
    rf = block_sum256(rf, sh);
    sw = block_sum256(sw, sh);
    const double mu = nu > 0.0 ? tr / nu : 1.0;
    double delta = shrinkage;
    if (shrinkage < 0.0) {
        double f = 0.0;
        for (int64_t c = threadIdx.x; c < L; c += 256) {
            int n, m;
            c_to_nm(c, n, m);
            n -= 1;
            if (st[n] || st[m]) continue;
            const double v = n == m ? As[(int64_t)n * N + m] - mu : As[(int64_t)n * N + m];
            f = fma(n == m ? v : 2.0 * v, v, f);
        }
        f = block_sum256(f, sh);
        const double d2 = nu > 0.0 ? f / nu : 0.0;
        const double b2 = fmin(d2, (ns * sw - rf) / (ns * nu));
        delta = b2 > 0.0 ? b2 / d2 : 0.0;
    }
    const double keep_r = 1.0 - delta, dmu = delta * mu;
    for (int64_t c = threadIdx.x; c < L; c += 256) {
        int n, m;
        c_to_nm(c, n, m);
        n -= 1;
        double* a = As + (int64_t)n * N + m;
        if (st[n] || st[m]) *a = n == m ? 1.0 : 0.0;
        else *a = n == m ? fma(keep_r, *a, dmu) : keep_r * *a;
    }
    if (threadIdx.x == 0 && dout != nullptr) dout[s] = delta;
}

// One CTA per subject: A_s <- -A_s^-1 by the symmetric sweep operator, kPNb pivots K at a time, over the
// lower triangle only.  Sweeping block K: D = A_KK is swept pivot by pivot in shared memory to Dm = -D^-1
// (the pivots are those of a Cholesky factorisation, squared: a pivot <= kPivotTol fails the subject:
// fail[s] = 1 and A_s is left unfinished); W = A_IK D^-1 = -A_IK Dm (I: the other rows); A_II -= W A_KI;
// then A_IK <- W, A_KK <- Dm.  After the last block A_s = -P.  (N^3 / 2 FMAs, as Cholesky, triangular
// inverse and L^-T L^-1 together.)  Wg: [kPNb] doubles per row of scratch for W.
__global__ void __launch_bounds__(256)
partial_invert_kernel(double* __restrict__ A, double* __restrict__ Wg, int N, int32_t* __restrict__ fail) {
    extern __shared__ double smem_d[];
    double* Dm = smem_d;                        // [kPNb][kPLd]
    double* Wt = Dm + kPNb * kPLd;              // [kPNb][kPLd]: W (update) or B (panel) rows, k-major
    double* Bt = Wt + kPNb * kPLd;              // [kPNb][kPLd]
    __shared__ int sh_fail;
    const int s = blockIdx.x;
    double* As = A + (int64_t)s * N * N;
    double* Ws = Wg + (int64_t)s * N * kPNb;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int nt = (N + kPT - 1) / kPT;
    if (threadIdx.x == 0) sh_fail = 0;
    for (int k0 = 0; k0 < N; k0 += kPNb) {
        const int kb = N - k0 < kPNb ? N - k0 : kPNb;
        const int k1 = k0 + kb;
        for (int e = threadIdx.x; e < kb * kb; e += 256) {
            const int i = e / kb, j = e - i * kb;
            Dm[i * kPLd + j] = As[sym_at(N, k0 + i, k0 + j)];
        }
        __syncthreads();
        // sweep D in place: <= 16 entries per thread
        for (int p = 0; p < kb; ++p) {
            const double d = Dm[p * kPLd + p];
            if (!(d > kPivotTol)) {                             // uniform: every thread reads the same d
                if (threadIdx.x == 0) sh_fail = 1;
                break;
            }
            const double id = 1.0 / d;
            double nv[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int e = threadIdx.x + 256 * q;
                if (e < kb * kb) {
                    const int i = e / kb, j = e - i * kb;
                    const double v = Dm[i * kPLd + j];
                    nv[q] = (i == p && j == p) ? -id
                            : (i == p || j == p) ? v * id
                                                 : fma(-Dm[i * kPLd + p] * id, Dm[p * kPLd + j], v);
                }
            }
            __syncthreads();
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int e = threadIdx.x + 256 * q;
                if (e < kb * kb) Dm[(e / kb) * kPLd + e % kb] = nv[q];
            }
            __syncthreads();
        }
        __syncthreads();
        if (sh_fail) break;
        // W = -B Dm, 64 rows at a time (B: the rows of the panel A_IK, zero for rows in K)
        for (int ti = 0; ti < nt; ++ti) {
            for (int e = threadIdx.x; e < kPT * kPNb; e += 256) {
                const int r = e / kPNb, q = e - r * kPNb, n = ti * kPT + r;
                Wt[q * kPLd + r] = (q < kb && n < N && (n < k0 || n >= k1)) ? As[sym_at(N, n, k0 + q)] : 0.0;
            }
            __syncthreads();
            double acc[4][4] = {};
            tile_fma<true>(Wt, Dm, kb, ty, tx, acc);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int n = ti * kPT + ty + 16 * i, l = tx + 16 * j;
                    if (n < N && l < kb) Ws[(int64_t)n * kPNb + l] = acc[i][j];
                }
            __syncthreads();
        }
        // A_II -= W B^T over the lower tiles; entries in K's rows or columns are left for the panel write
        for (int ti = 0; ti < nt; ++ti)
            for (int tj = 0; tj <= ti; ++tj) {
                for (int e = threadIdx.x; e < kPT * kPNb; e += 256) {
                    const int r = e / kPNb, q = e - r * kPNb;
                    const int n = ti * kPT + r, m = tj * kPT + r;
                    const bool okn = q < kb && n < N && (n < k0 || n >= k1);
                    const bool okm = q < kb && m < N && (m < k0 || m >= k1);
                    Wt[q * kPLd + r] = okn ? Ws[(int64_t)n * kPNb + q] : 0.0;
                    Bt[q * kPLd + r] = okm ? As[sym_at(N, m, k0 + q)] : 0.0;
                }
                __syncthreads();
                double acc[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int n = ti * kPT + ty + 16 * i, m = tj * kPT + tx + 16 * j;
                        acc[i][j] = (n < N && m <= n) ? As[(int64_t)n * N + m] : 0.0;
                    }
                tile_fma<true>(Wt, Bt, kb, ty, tx, acc);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int n = ti * kPT + ty + 16 * i, m = tj * kPT + tx + 16 * j;
                        if (n < N && m <= n && (n < k0 || n >= k1) && (m < k0 || m >= k1))
                            As[(int64_t)n * N + m] = acc[i][j];
                    }
                __syncthreads();
            }
        // panel and diagonal block
        for (int e = threadIdx.x; e < N * kb; e += 256) {
            const int n = e / kb, q = e - n * kb;
            if (n < k0 || n >= k1) As[sym_at(N, n, k0 + q)] = Ws[(int64_t)n * kPNb + q];
            else if (n - k0 >= q) As[(int64_t)n * N + k0 + q] = Dm[(n - k0) * kPLd + q];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) fail[s] = sh_fail;
}

// r_nm = -P_nm / sqrt(P_nn P_mm) from A = -P, corr_epilogue, out[c][s0 + s]; NaN for a failed subject.
__global__ void __launch_bounds__(256)
partial_epilogue_kernel(const double* __restrict__ A, const int32_t* __restrict__ fail, int N, double* __restrict__ out,
                        int64_t pitch, int s0, int fisher) {
    const int s = blockIdx.y;
    const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (c >= (int64_t)N * (N - 1) / 2) return;
    int n, m;
    c_to_nm(c, n, m);
    const double* As = A + (int64_t)s * N * N;
    const double r = As[(int64_t)n * N + m] / sqrt(As[(int64_t)n * N + n] * As[(int64_t)m * N + m]);
    out[c * pitch + s0 + s] = fail[s] ? __longlong_as_double(0x7ff8000000000000ll) : corr_epilogue(r, fisher);
}

// Batch workspace: Z [B][N][Tp], A [B][N][N], W [B][N][kPNb], Q [B][K][Tp], w [B][Tp], delta [B],
// status [B][N], each 1024-byte aligned.
struct PartialWs {
    double* Z;
    double* A;
    double* W;
    double* Q;
    double* w;
    double* delta;
    uint8_t* status;
};

static int64_t pal(int64_t b) { return (b + 1023) & ~(int64_t)1023; }

static int64_t partial_ws_for(int64_t B, int N, int Tp, int K) {
    return 1024 + pal(B * N * Tp * 8) + pal(B * N * N * 8) + pal(B * N * kPNb * 8) + pal(B * K * Tp * 8) +
           pal(B * Tp * 8) + pal(B * 8) + pal(B * N);
}

// Subjects per batch: as many as kPartialWsBudget holds (at least one, at most S).
static int partial_batch(int S, int N, int Tp, int K) {
    const int64_t per = partial_ws_for(1, N, Tp, K);
    int64_t b = kPartialWsBudget / per;
    if (b < 1) b = 1;
    if (b > S) b = S;
    return (int)b;
}

static PartialWs partial_ws(void* zws, int B, int N, int Tp, int K) {
    PartialWs w;
    uint8_t* p = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(zws) + 1023) & ~(uintptr_t)1023);
    w.Z = reinterpret_cast<double*>(p);
    p += pal((int64_t)B * N * Tp * 8);
    w.A = reinterpret_cast<double*>(p);
    p += pal((int64_t)B * N * N * 8);
    w.W = reinterpret_cast<double*>(p);
    p += pal((int64_t)B * N * kPNb * 8);
    w.Q = reinterpret_cast<double*>(p);
    p += pal((int64_t)B * K * Tp * 8);
    w.w = reinterpret_cast<double*>(p);
    p += pal((int64_t)B * Tp * 8);
    w.delta = reinterpret_cast<double*>(p);
    p += pal((int64_t)B * 8);
    w.status = p;
    return w;
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int64_t fcd_corr_partial_workspace_bytes(int32_t S, int32_t N, int32_t T, int32_t K) {
    if (S < 0 || N < 0 || T < 0 || K < 0 || K > kMaxConfoundsPartial) return -1;
    if (S == 0) return 1024;
    const int Tp = corr_padded_T(T);
    return partial_ws_for(partial_batch(S, N, Tp, K), N, Tp, K);
}

int fcd_corr_partial(const float* ts, int32_t S, int32_t N, int32_t T, const uint8_t* keep, const double* confounds,
                     int32_t K, double shrinkage, double* out, int64_t pitch, int32_t s0, int32_t fisher,
                     int32_t mark_missing, int32_t* rank, double* shrinkage_out, int32_t* status, void* zws,
                     void* stream) {
    FCD_REQUIRE(ts != nullptr && out != nullptr && status != nullptr && zws != nullptr,
                "fcd_corr_partial: NULL argument");
    FCD_REQUIRE(S >= 0 && N >= 2 && T >= 2 && s0 >= 0 && pitch >= (int64_t)s0 + S && S <= 65535,
                "fcd_corr_partial: bad shape S=%d N=%d T=%d s0=%d pitch=%lld", S, N, T, s0, (long long)pitch);
    FCD_REQUIRE(K >= 0 && K <= kMaxConfoundsPartial && (K == 0) == (confounds == nullptr),
                "fcd_corr_partial: K=%d needs 0 <= K <= %d and confounds NULL iff K == 0", K, kMaxConfoundsPartial);
    FCD_REQUIRE(shrinkage < 0.0 || shrinkage <= 1.0, "fcd_corr_partial: shrinkage %g outside [0, 1]", shrinkage);
    if (S == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int Tp = corr_padded_T(T);
    int B = partial_batch(S, N, Tp, K);
    if (const char* e = getenv("FCD_CORR_PARTIAL_BATCH")) {      // smaller batches (tests: batch boundaries)
        const int b = atoi(e);
        if (b >= 1 && b < B) B = b;
    }
    const PartialWs w = partial_ws(zws, B, N, Tp, K);
    const size_t inv_smem = (size_t)3 * kPNb * kPLd * sizeof(double);
    FCD_ALLOW_BIG_SMEM(partial_invert_kernel);
    const int nt = (N + kPT - 1) / kPT;
    const int64_t C = (int64_t)N * (N - 1) / 2;
    for (int b0 = 0; b0 < S; b0 += B) {
        const int nb = S - b0 < B ? S - b0 : B;
        const float* tsb = ts + (int64_t)b0 * N * T;
        const uint8_t* kb = keep != nullptr ? keep + (int64_t)b0 * T : nullptr;
        int rc;
        if (K == 0) {
            rc = corr_standardise_masked_f64(tsb, kb, nb, N, T, Tp, w.Z, w.status, st);
            if (!rc && rank != nullptr)
                FCD_REQUIRE(cudaMemsetAsync(rank + b0, 0, (size_t)nb * sizeof(int32_t), st) == cudaSuccess,
                            "fcd_corr_partial: cudaMemsetAsync(rank) failed");
        } else {
            rc = corr_clean_f64(tsb, kb, confounds + (int64_t)b0 * T * K, nb, N, T, Tp, K, w.Q, w.Z, w.status,
                                rank != nullptr ? rank + b0 : nullptr, st);
        }
        if (rc) return rc;
        frame_sq_kernel<<<dim3((unsigned)((Tp + 127) / 128), (unsigned)nb), 128, 0, st>>>(w.Z, N, Tp, w.w);
        if ((rc = check_launch("fcd_corr_partial(frame_sq)"))) return rc;
        partial_gram_kernel<<<dim3((unsigned)(nt * (nt + 1) / 2), (unsigned)nb), 256, 0, st>>>(w.Z, N, Tp, w.A);
        if ((rc = check_launch("fcd_corr_partial(gram)"))) return rc;
        partial_shrink_kernel<<<nb, 256, 0, st>>>(w.A, w.w, w.status, kb, N, T, Tp, shrinkage < 0.0 ? -1.0 : shrinkage,
                                                  shrinkage_out != nullptr ? shrinkage_out + b0 : w.delta);
        if ((rc = check_launch("fcd_corr_partial(shrink)"))) return rc;
        partial_invert_kernel<<<nb, 256, inv_smem, st>>>(w.A, w.W, N, status + b0);
        if ((rc = check_launch("fcd_corr_partial(invert)"))) return rc;
        partial_epilogue_kernel<<<dim3((unsigned)((C + 255) / 256), (unsigned)nb), 256, 0, st>>>(
            w.A, status + b0, N, out, pitch, s0 + b0, fisher);
        if ((rc = check_launch("fcd_corr_partial(epilogue)"))) return rc;
        if (mark_missing && (rc = corr_mark_status(w.status, nb, N, out, pitch, s0 + b0, st))) return rc;
    }
    return 0;
}

}  // extern "C"
