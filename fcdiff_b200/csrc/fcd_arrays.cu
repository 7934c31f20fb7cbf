// "Materialised" API-parity kernels: the reference caches (C,H,3), (C,U,3) and
// (C,U,3,3) arrays (fcdiff/fit.py:40-54) and its unit tests assign and read them
// directly.  These kernels run the same steps from such arrays on the GPU; the
// fused hot path (fcd_estep.cu / fcd_mstep.cu) never materialises them.
#include "fcd_common.cuh"

namespace fcd {

constexpr int kArrThreads = 256;

static inline int arr_grid(int64_t items, int per_block) {
    int64_t need = (items + per_block - 1) / per_block;
    int64_t cap = (int64_t)sm_count() * 8;
    if (cap > kMaxReduceBlocks) cap = kMaxReduceBlocks;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

// scipy.stats.norm op order, no FMA contraction (fcdiff/fit.py:114-115):
//   y = (x - loc) / scale
//   logpdf = (-(y*y) / 2 - log(sqrt(2 pi))) - log(scale)
//   pdf    = (exp(-(y*y) / 2) / sqrt(2 pi)) / scale
__device__ __forceinline__ double sp_y(double x, double mu, double sigma) {
    return __ddiv_rn(__dsub_rn(x, mu), sigma);
}
__device__ __forceinline__ double sp_logpdf(double y, double log_sigma) {
    const double h = __ddiv_rn(-__dmul_rn(y, y), 2.0);
    return __dsub_rn(__dsub_rn(h, kHalfLog2Pi), log_sigma);
}
__device__ __forceinline__ double sp_pdf(double y, double sigma) {
    const double h = __ddiv_rn(-__dmul_rn(y, y), 2.0);
    return __ddiv_rn(__ddiv_rn(exp(h), 2.5066282746310002 /* sqrt(2 pi) */), sigma);
}
// fcdiff/fit.py:427-430: eps * N[k] + (1 - eps) * 0.5 * (N[j] + N[j'])
__device__ __forceinline__ double ref_M(double pk, double pj, double pjj, double eps) {
    const double sum_N = __dadd_rn(pj, pjj);
    return __dadd_rn(__dmul_rn(eps, pk), __dmul_rn(__dmul_rn(__dsub_rn(1.0, eps), 0.5), sum_N));
}

struct LpsParams {
    double mu[3], sigma[3], log_sigma[3], epsl[3];
};

// MASKED: a NaN entry is not observed; its caches hold the marginalised values
//   lp_B_g_F = 0 (density factor 1), p_Bt_g_Ft = (1, 1, 1) and lM = 0 (M_kl = eps_l + (1 - eps_l) = 1).
template <bool MASKED>
__global__ void __launch_bounds__(kArrThreads)
materialize_b_kernel(const double* __restrict__ b, int64_t n, const __grid_constant__ LpsParams p,
                     double* __restrict__ lpB) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const double x = b[i];
        if (MASKED && isnan(x)) {
            lpB[i * 3] = lpB[i * 3 + 1] = lpB[i * 3 + 2] = 0.0;
            continue;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) lpB[i * 3 + k] = sp_logpdf(sp_y(x, p.mu[k], p.sigma[k]), p.log_sigma[k]);
    }
}

template <bool MASKED>
__global__ void __launch_bounds__(kArrThreads)
materialize_bt_kernel(const double* __restrict__ bt, int64_t n, const __grid_constant__ LpsParams p,
                      double* __restrict__ pBt, double* __restrict__ lM) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const double x = bt[i];
        if (MASKED && isnan(x)) {
            pBt[i * 3] = pBt[i * 3 + 1] = pBt[i * 3 + 2] = 1.0;
#pragma unroll
            for (int j = 0; j < 9; ++j) lM[i * 9 + j] = 0.0;
            continue;
        }
        double pk[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            pk[k] = sp_pdf(sp_y(x, p.mu[k], p.sigma[k]), p.sigma[k]);
            pBt[i * 3 + k] = pk[k];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double pj = pk[k == 0 ? 1 : 0], pjj = pk[k == 2 ? 1 : 2];
#pragma unroll
            for (int l = 0; l < 3; ++l) lM[i * 9 + k * 3 + l] = log(ref_M(pk[k], pj, pjj, p.epsl[l]));
        }
    }
}

__global__ void __launch_bounds__(kArrThreads)
eval_M_kernel(const double* __restrict__ p, int64_t n, double eps, int k, double* __restrict__ M) {
    const int j = (k == 0) ? 1 : 0, jj = (k == 2) ? 1 : 2;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x)
        M[i] = ref_M(p[i * 3 + k], p[i * 3 + j], p[i * 3 + jj], eps);
}

// `_update_lq_F` from arrays: one warp per edge (fcdiff/fit.py:165-174).
__global__ void __launch_bounds__(kArrThreads)
lqF_from_arrays_kernel(const double* __restrict__ lpB, const double* __restrict__ lM,
                       int64_t C, int H, int U, const double* __restrict__ qR, int N,
                       double lg0, double lg1, double lg2, double* __restrict__ lqF) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    for (int64_t c = warp0; c < C; c += nwarps) {
        int n, m;
        c_to_nm(c, n, m);
        double acc[3] = {0.0, 0.0, 0.0};
        const double* lp = lpB + c * H * 3;
        for (int i = lane; i < H * 3; i += 32) {
            const double v = lp[i];
            const int k = i % 3;
            if (k == 0) acc[0] += v; else if (k == 1) acc[1] += v; else acc[2] += v;
        }
        const double* lm = lM + c * (int64_t)U * 9;
        for (int u = lane; u < U; u += 32) {
            double w[3];
            pair_weights(qR2[(int64_t)n * U + u], qR2[(int64_t)m * U + u], w);
#pragma unroll
            for (int k = 0; k < 3; ++k)
#pragma unroll
                for (int l = 0; l < 3; ++l) acc[k] = fma(w[l], lm[u * 9 + k * 3 + l], acc[k]);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] = warp_sum(acc[k]);
        if (lane == 0) {
            double l[3] = {lg0 + acc[0], lg1 + acc[1], lg2 + acc[2]};
            const double mx = fmax(l[0], fmax(l[1], l[2]));
            const double lse = mx + log(exp(l[0] - mx) + exp(l[1] - mx) + exp(l[2] - mx));
#pragma unroll
            for (int k = 0; k < 3; ++k) lqF[c * 3 + k] = l[k] - lse;
        }
    }
}

// W_l = sum_k qF[c,k] lM[c,u,k,l]  (fcdiff/fit.py:187-194, q_R-independent part);
// WT[u][c] = {W_0 - W_2, W_2 - W_1}: what survives the normalisation of fit.py:196 (fcd_estep.cu, K2b/W)
__global__ void __launch_bounds__(kArrThreads)
region_weights_from_lM_kernel(const double* __restrict__ lM, int64_t C, int U,
                              const double* __restrict__ qF, double* __restrict__ WT) {
    const int64_t total = C * U;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = i / U;
        const int u = (int)(i - c * U);
        const double* lm = lM + i * 9;
        const double q0 = qF[c * 3], q1 = qF[c * 3 + 1], q2 = qF[c * 3 + 2];
        double w[3];
#pragma unroll
        for (int l = 0; l < 3; ++l) w[l] = fma(q2, lm[6 + l], fma(q1, lm[3 + l], q0 * lm[l]));
        reinterpret_cast<double2*>(WT)[(int64_t)u * C + c] = make_double2(w[0] - w[2], w[2] - w[1]);
    }
}

// `_eval_E_lM` from arrays (fcdiff/fit.py:489-511) and, with MODE 1, the
// analytic derivatives `_eval_dE_dh` / `_eval_dE_de` (fit.py:600-697) from the
// `norm` / `mix` arrays the reference's tests pass.
template <int MODE>
__global__ void __launch_bounds__(kArrThreads)
arrays_reduce_kernel(const double* __restrict__ qF, const double* __restrict__ qR,
                     const double* __restrict__ A /* lM or mix [C][U][3][3] */,
                     const double* __restrict__ norm /* [C][U][3], MODE 1 */,
                     int64_t C, int N, int U, double eta, double epsilon,
                     double* __restrict__ out, double* __restrict__ ws) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    double acc[2] = {0.0, 0.0};
    for (int64_t c = warp0; c < C; c += nwarps) {
        int n, m;
        c_to_nm(c, n, m);
        const double qf[3] = {qF[c * 3], qF[c * 3 + 1], qF[c * 3 + 2]};
        for (int u = lane; u < U; u += 32) {
            double w[3];
            pair_weights(qR2[(int64_t)n * U + u], qR2[(int64_t)m * U + u], w);
            const double* a = A + (c * U + u) * 9;
            if (MODE == 0) {
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    double s = 0.0;
#pragma unroll
                    for (int l = 0; l < 3; ++l) s = fma(w[l], a[k * 3 + l], s);
                    acc[0] = fma(qf[k], s, acc[0]);
                }
            } else {
                const double* nr = norm + (c * U + u) * 3;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double oth = nr[k == 0 ? 1 : 0] + nr[k == 2 ? 1 : 2];
                    const double num = nr[k] - 0.5 * oth;
                    const double g0 = num / a[k * 3], g1 = num / a[k * 3 + 1], g2 = num / a[k * 3 + 2];
                    acc[0] -= qf[k] * w[2] * (2.0 * epsilon - 1.0) * g2;                       // fit.py:609-614
                    acc[1] -= qf[k] * (w[1] * g1 - w[0] * g0 + w[2] * (2.0 * eta - 1.0) * g2); // fit.py:653-663
                }
            }
        }
    }
    grid_reduce_store<2, kArrThreads>(acc, ws, out);
}

// out = sum_i a[(i / a_outer) * a_inner + i % a_inner] * x[i % x_len]
__global__ void __launch_bounds__(kArrThreads)
dot_broadcast_kernel(const double* __restrict__ a, int64_t a_outer, int64_t a_inner,
                     const double* __restrict__ x, int64_t x_len, int64_t n,
                     double* __restrict__ out, double* __restrict__ ws) {
    double v[1] = {0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ia = (i / a_outer) * a_inner + i % a_inner;
        v[0] = fma(a[ia], x[i % x_len], v[0]);
    }
    grid_reduce_store<1, kArrThreads>(v, ws, out);
}

// `_eval_dlM_dh` / `_eval_dlM_de` (fcdiff/fit.py:618-641, 667-697):
// (eps * norm_k - 0.5 * eps * (norm_j + norm_j')) / mix, elementwise.
__global__ void __launch_bounds__(kArrThreads)
dlM_kernel(const double* __restrict__ norm, const double* __restrict__ mix, int64_t n, double eps, int k,
           double* __restrict__ out) {
    const int j = (k == 0) ? 1 : 0, jj = (k == 2) ? 1 : 2;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const double sum_ls = __dadd_rn(norm[i * 3 + j], norm[i * 3 + jj]);
        const double num = __dsub_rn(__dmul_rn(eps, norm[i * 3 + k]), __dmul_rn(__dmul_rn(0.5, eps), sum_ls));
        out[i] = __ddiv_rn(num, mix[i]);
    }
}

// `_eval_q_R_w` (fcdiff/fit.py:382-406): out[u][0..2] for one region pair.
__global__ void __launch_bounds__(kArrThreads)
pair_weights_kernel(const double* __restrict__ qR, int U, int n, int m, double* __restrict__ out) {
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    for (int u = blockIdx.x * blockDim.x + threadIdx.x; u < U; u += gridDim.x * blockDim.x) {
        const double2 a = qR2[(int64_t)n * U + u], b = qR2[(int64_t)m * U + u];
        out[u * 3] = __dmul_rn(a.x, b.x);
        out[u * 3 + 1] = __dmul_rn(a.y, b.y);
        out[u * 3 + 2] = __dadd_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x));
    }
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int fcd_materialize_lps(const double* b, const double* bt, int64_t C, int32_t H, int32_t U,
                        const fcd_theta* theta_host, double* lpB, double* pBt, double* lM, int32_t missing,
                        void* stream) {
    FCD_REQUIRE(theta_host != nullptr, "fcd_materialize_lps: theta is NULL");
    FCD_REQUIRE(C >= 0 && H >= 0 && U >= 0, "fcd_materialize_lps: bad shape");
    FCD_REQUIRE(missing == 0 || missing == 1, "fcd_materialize_lps: missing must be 0 or 1, got %d", missing);
    LpsParams p;
    for (int k = 0; k < 3; ++k) {
        p.mu[k] = theta_host->mu[k];
        p.sigma[k] = theta_host->sigma[k];
        p.log_sigma[k] = log(theta_host->sigma[k]);
    }
    p.epsl[0] = 1.0 - theta_host->epsilon;
    p.epsl[1] = theta_host->epsilon;
    p.epsl[2] = theta_host->eta * theta_host->epsilon;
    p.epsl[2] += (1.0 - theta_host->eta) * (1.0 - theta_host->epsilon);      // fit.py:442-443
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
    if (b != nullptr && lpB != nullptr && C * H > 0) {
        if (missing) materialize_b_kernel<true><<<arr_grid(C * H, kArrThreads), kArrThreads, 0, st>>>(b, C * H, p, lpB);
        else materialize_b_kernel<false><<<arr_grid(C * H, kArrThreads), kArrThreads, 0, st>>>(b, C * H, p, lpB);
        rc = check_launch("fcd_materialize_lps(b)");
        if (rc) return rc;
    }
    if (bt != nullptr && pBt != nullptr && lM != nullptr && C * U > 0) {
        if (missing)
            materialize_bt_kernel<true><<<arr_grid(C * U, kArrThreads), kArrThreads, 0, st>>>(bt, C * U, p, pBt, lM);
        else
            materialize_bt_kernel<false><<<arr_grid(C * U, kArrThreads), kArrThreads, 0, st>>>(bt, C * U, p, pBt, lM);
        rc = check_launch("fcd_materialize_lps(bt)");
    }
    return rc;
}

int fcd_eval_M(const double* p, int64_t n, double eta, double epsilon, int32_t k, int32_t l,
               double* M, void* stream) {
    FCD_REQUIRE(k >= 0 && k < 3 && l >= 0 && l < 3 && n >= 0, "fcd_eval_M: bad (k, l) = (%d, %d)", k, l);
    if (n == 0) return 0;
    double eps;
    if (l == 0) eps = 1.0 - epsilon;
    else if (l == 1) eps = epsilon;
    else { eps = eta * epsilon; eps += (1.0 - eta) * (1.0 - epsilon); }
    eval_M_kernel<<<arr_grid(n, kArrThreads), kArrThreads, 0, (cudaStream_t)stream>>>(p, n, eps, k, M);
    return check_launch("fcd_eval_M");
}

int fcd_lqF_from_arrays(const double* lpB, const double* lM, int64_t C, int32_t H, int32_t U,
                        const double* qR, int32_t N, const double* log_gamma_host,
                        double* lqF, void* stream) {
    FCD_REQUIRE(log_gamma_host != nullptr, "fcd_lqF_from_arrays: log_gamma is NULL");
    FCD_REQUIRE(C >= 0 && H >= 0 && U >= 0 && N >= 2 && C <= (int64_t)N * (N - 1) / 2,
                "fcd_lqF_from_arrays: bad shape");
    if (C == 0) return 0;
    lqF_from_arrays_kernel<<<arr_grid(C, kArrThreads / 32), kArrThreads, 0, (cudaStream_t)stream>>>(
        lpB, lM, C, H, U, qR, N, log_gamma_host[0], log_gamma_host[1], log_gamma_host[2], lqF);
    return check_launch("fcd_lqF_from_arrays");
}

int fcd_region_weights_from_lM(const double* lM, int64_t C, int32_t U, const double* qF,
                               double* WT, void* stream) {
    FCD_REQUIRE(C >= 0 && U >= 0, "fcd_region_weights_from_lM: bad shape");
    if (C * U == 0) return 0;
    region_weights_from_lM_kernel<<<arr_grid(C * U, kArrThreads), kArrThreads, 0, (cudaStream_t)stream>>>(
        lM, C, U, qF, WT);
    return check_launch("fcd_region_weights_from_lM");
}

int fcd_ElM_from_arrays(const double* qF, const double* qR, const double* lM,
                        int64_t C, int32_t N, int32_t U, double* out1, double* ws, void* stream) {
    FCD_REQUIRE(ws != nullptr && C >= 0 && N >= 2 && U >= 0 && C <= (int64_t)N * (N - 1) / 2,
                "fcd_ElM_from_arrays: bad arguments");
    // out has room for one double; the reduction writes two -> go through scratch.
    arrays_reduce_kernel<0><<<arr_grid(C, kArrThreads / 32), kArrThreads, 0, (cudaStream_t)stream>>>(
        qF, qR, lM, nullptr, C, N, U, 0.0, 0.0, ws + kWsScratch, ws);
    int rc = check_launch("fcd_ElM_from_arrays");
    if (rc) return rc;
    cudaError_t e = cudaMemcpyAsync(out1, ws + kWsScratch, sizeof(double), cudaMemcpyDeviceToDevice,
                                    (cudaStream_t)stream);
    FCD_REQUIRE(e == cudaSuccess, "fcd_ElM_from_arrays: %s", cudaGetErrorString(e));
    return 0;
}

int fcd_dE_from_arrays(const double* qR, const double* qF, const double* norm, const double* mix,
                       int64_t C, int32_t N, int32_t U, double eta, double epsilon,
                       double* out2, double* ws, void* stream) {
    FCD_REQUIRE(ws != nullptr && C >= 0 && N >= 2 && U >= 0 && C <= (int64_t)N * (N - 1) / 2,
                "fcd_dE_from_arrays: bad arguments");
    arrays_reduce_kernel<1><<<arr_grid(C, kArrThreads / 32), kArrThreads, 0, (cudaStream_t)stream>>>(
        qF, qR, mix, norm, C, N, U, eta, epsilon, out2, ws);
    return check_launch("fcd_dE_from_arrays");
}

int fcd_dot_broadcast(const double* a, int64_t a_outer, int64_t a_inner,
                      const double* x, int64_t x_len, int64_t n,
                      double* out1, double* ws, void* stream) {
    FCD_REQUIRE(ws != nullptr && n >= 0 && a_outer >= 1 && a_inner >= 1 && a_inner <= a_outer && x_len >= 1,
                "fcd_dot_broadcast: bad arguments");
    dot_broadcast_kernel<<<arr_grid(n, kArrThreads), kArrThreads, 0, (cudaStream_t)stream>>>(
        a, a_outer, a_inner, x, x_len, n, out1, ws);
    return check_launch("fcd_dot_broadcast");
}

int fcd_dlM(const double* norm, const double* mix, int64_t n, double eps, int32_t k,
            double* out, void* stream) {
    FCD_REQUIRE(n >= 0 && k >= 0 && k < 3, "fcd_dlM: bad arguments");
    if (n == 0) return 0;
    dlM_kernel<<<arr_grid(n, kArrThreads), kArrThreads, 0, (cudaStream_t)stream>>>(norm, mix, n, eps, k, out);
    return check_launch("fcd_dlM");
}

int fcd_pair_weights(const double* qR, int32_t N, int32_t U, int32_t n, int32_t m,
                     double* out, void* stream) {
    FCD_REQUIRE(N >= 1 && U >= 1 && n >= 0 && n < N && m >= 0 && m < N, "fcd_pair_weights: bad (n, m) = (%d, %d)", n, m);
    pair_weights_kernel<<<arr_grid(U, kArrThreads), kArrThreads, 0, (cudaStream_t)stream>>>(qR, U, n, m, out);
    return check_launch("fcd_pair_weights");
}

}  // extern "C"
