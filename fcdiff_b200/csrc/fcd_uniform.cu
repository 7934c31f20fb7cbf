// The uniform start (fcdiff/fit.py:84-102): q_F = 1/3 and q_R = 1/2 everywhere.  Every element then has
// the SAME pair weights w = (q0^2, q1^2, 2 q0 q1) (fit.py:382-406), so the weighted sums of logarithms
// of fit.py:165-173 and fit.py:489-511 factor:
//     sum_u sum_l w_l log M_kl(c,u)  =  sum_l w_l  S_kl[c]  (+ the theta-free part),
//     S_kl[c] = sum_u log(a_l + b_l p_k(c,u)) = log prod_u (a_l + b_l p_k(c,u)).
// The general kernels take nine logarithms per element in this state (no posterior is decided: tier T3
// of fcd_common.cuh); here the nine row sums are nine running PRODUCTS (fcd_math.cuh "Sum of logs as the
// log of a product"): 9 FMA + 9 MUL per element, nine logarithms per row.  ONE pass over the two streamed
// planes serves the initial free energy (fit.py:74) and the first E-step (fit.py:76), which run at the same
// theta and the same constant q_R:
//   fcd_row_logsums          S[c][k*3 + l], warp per row, TMA ring as in estep_qF_coded_kernel;
//   fcd_estep_qF_rowsums     lq_F from S and the constant pair weights (fit.py:165-174);
//   fcd_elm_rowsums          sum_c sum_k qF[c,k] sum_l w_l S[c][k][l]  (theta-dependent part of E_lM).
// Valid for any CONSTANT q_R; q_F may be arbitrary in fcd_elm_rowsums.
#include "fcd_common.cuh"

namespace fcd {

constexpr int kRsSeg = 128;
constexpr int kRsStage = 2 * kRsSeg * 8;                     // bytes: p_0, p_1
constexpr int kRsMaxDepth = 5;
constexpr size_t rs_ring_bytes(int depth) { return (size_t)kStreamWarps * depth * (kRsStage + 8); }
constexpr int kRsProdMax = 24;                               // factors per running product between two logarithms

template <bool FAST>
__global__ void __launch_bounds__(kStreamThreads, 1)
row_logsums_kernel(const double* __restrict__ P, int64_t planeStride, int64_t C, int U, int64_t pitchU,
                   const __grid_constant__ ThetaDev th, const __grid_constant__ LogTabWindow tab, int depth,
                   double* __restrict__ S) {
    extern __shared__ __align__(128) double s_dyn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* ring0 = reinterpret_cast<unsigned char*>(s_dyn + (FAST ? ((tab.n + 15) & ~15) : 0));
    unsigned char* ring = ring0 + (size_t)warp * depth * kRsStage;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring0 + (size_t)kStreamWarps * depth * kRsStage) + warp * depth;
    if (lane < depth) mbar_init(bars + lane, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    const int nseg = (int)((pitchU + kRsSeg - 1) / kRsSeg);
    const int64_t W = (int64_t)gridDim.x * kStreamWarps;
    const int64_t c_first = (int64_t)blockIdx.x * kStreamWarps + warp;
    const uint32_t ring_s = smem_u32(ring), bars_s = smem_u32(bars);
    int64_t pc = c_first;
    int ps = 0, pd = 0;
    auto issue = [&]() {
        if (pc >= C) return;
        if (lane == 0) {
            const int u0 = ps * kRsSeg;
            const uint32_t np = (uint32_t)(pitchU - u0 < kRsSeg ? pitchU - u0 : kRsSeg);        // even
            const uint32_t st = ring_s + pd * kRsStage, bar = bars_s + pd * 8;
            const double* src = P + pc * pitchU + u0;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(2 * np * 8) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(st), "l"(src), "r"(np * 8), "r"(bar) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(st + kRsSeg * 8), "l"(src + planeStride), "r"(np * 8), "r"(bar) : "memory");
        }
        if (++pd == depth) pd = 0;
        if (++ps == nseg) {
            ps = 0;
            pc += W;
        }
    };
#pragma unroll 1
    for (int i = 0; i < depth; ++i) issue();
    const double* s_tab = load_log_table<FAST>(tab, s_dyn);

    const double al[3] = {th.al[0], th.al[1], th.al[2]}, bl[3] = {th.bl[0], th.bl[1], th.bl[2]};
    double acc[9], pr[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        acc[i] = 0.0;
        pr[i] = 1.0;
    }
    int nf = 0;
    auto flush = [&]() {
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            if (FAST) acc[i] += log_pos<FAST>(pr[i], s_tab);
            pr[i] = 1.0;
        }
        nf = 0;
    };
    int d = 0;
    uint32_t phase = 0;
    for (int64_t c = c_first; c < C; c += W) {
        for (int s = 0; s < nseg; ++s) {
            mbar_wait(bars + d, phase);
            const unsigned char* st = ring + d * kRsStage;
#pragma unroll
            for (int j = 0; j < kRsSeg / 32; ++j) {
                const int u = s * kRsSeg + 32 * j + lane;
                if (s * kRsSeg + 32 * j < U) {               // warp-uniform
                    const bool in = u < U;
                    // lanes beyond the row multiply by exactly 1 (p = 0 would give a_l)
                    const double p0 = *reinterpret_cast<const double*>(st + (32 * j + lane) * 8);
                    const double p1 = *reinterpret_cast<const double*>(st + kRsSeg * 8 + (32 * j + lane) * 8);
                    const double p3[3] = {p0, p1, (1.0 - p0) - p1};
#pragma unroll
                    for (int k = 0; k < 3; ++k)
#pragma unroll
                        for (int l = 0; l < 3; ++l) {
                            const double y = fma(bl[l], p3[k], al[l]);
                            if (FAST) pr[k * 3 + l] *= in ? y : 1.0;
                            else if (in) acc[k * 3 + l] += log(y);
                        }
                    if (++nf == kRsProdMax) flush();
                }
            }
            __syncwarp();
            issue();
            if (++d == depth) {
                d = 0;
                phase ^= 1;
            }
        }
        flush();
#pragma unroll
        for (int i = 0; i < 9; ++i) acc[i] = warp_sum(acc[i]);
        if (lane < 9) {
            double v = acc[0];
#pragma unroll
            for (int i = 1; i < 9; ++i) v = lane == i ? acc[i] : v;
            S[c * 9 + lane] = v;
        }
#pragma unroll
        for (int i = 0; i < 9; ++i) acc[i] = 0.0;
    }
}

// lqF[c,k] = log gamma_k + healthy_k(S1, S2) + sum_l w_l S[c][k][l] - logsumexp_k   (fit.py:165-174; the
// theta-free term L sum_l w_l is common to the three states and cancels, as in estep_qF_kernel)
template <bool MASKED>
__global__ void __launch_bounds__(256)
estep_qF_rowsums_kernel(const double* __restrict__ S1, const double* __restrict__ S2, const double* __restrict__ S0,
                        const double* __restrict__ S,
                        int64_t C, double w0, double w1, double w2, const __grid_constant__ ThetaDev th,
                        double* __restrict__ lqF, double* __restrict__ qF) {
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < C; c += (int64_t)gridDim.x * blockDim.x) {
        double l[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double a = fma(w0, S[c * 9 + k * 3], fma(w1, S[c * 9 + k * 3 + 1], w2 * S[c * 9 + k * 3 + 2]));
            l[k] = th.log_gamma[k] + healthy_term<MASKED>(th, k, S1[c], S2[c], MASKED ? S0[c] : 0.0) + a;
        }
        const double mx = fmax(l[0], fmax(l[1], l[2]));
        const double lse = mx + log(exp(l[0] - mx) + exp(l[1] - mx) + exp(l[2] - mx));
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double v = l[k] - lse;
            lqF[c * 3 + k] = v;
            if (qF) qF[c * 3 + k] = exp(v);
        }
    }
}

// out[0] = sum_c sum_k qF[c,k] sum_l w_l S[c][k][l]
__global__ void __launch_bounds__(256)
elm_rowsums_kernel(const double* __restrict__ S, const double* __restrict__ qF, int64_t C, double w0, double w1,
                   double w2, double* __restrict__ out, double* __restrict__ ws) {
    double v[1] = {0.0};
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < C; c += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int k = 0; k < 3; ++k)
            v[0] = fma(qF[c * 3 + k], fma(w0, S[c * 9 + k * 3], fma(w1, S[c * 9 + k * 3 + 1], w2 * S[c * 9 + k * 3 + 2])), v[0]);
    }
    grid_reduce_store<1, 256>(v, ws, out);
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int fcd_row_logsums(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                    const fcd_theta* theta_host, double* S9, void* stream) {
    FCD_REQUIRE(P != nullptr && theta_host != nullptr && S9 != nullptr, "fcd_row_logsums: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && U < 65536 && pitchU >= U && pitchU % 2 == 0 && planeStride % 2 == 0 &&
                (reinterpret_cast<uintptr_t>(P) & 15) == 0,
                "fcd_row_logsums: planes must be 16-byte aligned with even pitches");
    if (C == 0) return 0;
    const ThetaDev th = make_theta_dev(*theta_host, 0);
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(th.epsl, th.al, st, tab, true), "fcd_row_logsums: log table initialisation failed");
    const bool fast = log_table_covers(th.epsl, th.al);
    const size_t tbytes = fast ? (size_t)((tab.n + 15) & ~15) * sizeof(double) : 0;
    int depth = kRsMaxDepth;
    while (depth > 2 && tbytes + rs_ring_bytes(depth) > kSmemBudget) --depth;
    FCD_REQUIRE(tbytes + rs_ring_bytes(depth) <= kSmemBudget, "fcd_row_logsums: shared memory budget exceeded");
    const size_t smem = tbytes + rs_ring_bytes(depth);
    int64_t grid = (C + kStreamWarps - 1) / kStreamWarps;
    if (grid > sm_count()) grid = sm_count();
    if (fast) {
        FCD_ALLOW_BIG_SMEM(row_logsums_kernel<true>);
        row_logsums_kernel<true><<<(unsigned)grid, kStreamThreads, smem, st>>>(P, planeStride, C, U, pitchU, th, tab, depth, S9);
    } else {
        FCD_ALLOW_BIG_SMEM(row_logsums_kernel<false>);
        row_logsums_kernel<false><<<(unsigned)grid, kStreamThreads, smem, st>>>(P, planeStride, C, U, pitchU, th, tab, depth, S9);
    }
    return check_launch("fcd_row_logsums");
}

// S0 == NULL: every edge has all H controls (the unmasked kernel).
int fcd_estep_qF_rowsums(const double* S1, const double* S2, const double* S0, int32_t H, const double* S9,
                         int64_t C, const double* w3_host, const fcd_theta* theta_host, double* lqF, double* qF,
                         void* stream) {
    FCD_REQUIRE(S1 != nullptr && S2 != nullptr && S9 != nullptr && w3_host != nullptr && theta_host != nullptr &&
                lqF != nullptr && C >= 0 && H >= 1, "fcd_estep_qF_rowsums: bad argument");
    if (C == 0) return 0;
    const ThetaDev th = make_theta_dev(*theta_host, H);
    int64_t grid = (C + 255) / 256;
    if (grid > (int64_t)sm_count() * 8) grid = (int64_t)sm_count() * 8;
    if (S0 != nullptr)
        estep_qF_rowsums_kernel<true><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
            S1, S2, S0, S9, C, w3_host[0], w3_host[1], w3_host[2], th, lqF, qF);
    else
        estep_qF_rowsums_kernel<false><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
            S1, S2, nullptr, S9, C, w3_host[0], w3_host[1], w3_host[2], th, lqF, qF);
    return check_launch("fcd_estep_qF_rowsums");
}

int fcd_elm_rowsums(const double* S9, const double* qF, int64_t C, const double* w3_host, double* out1, double* ws,
                    void* stream) {
    FCD_REQUIRE(S9 != nullptr && qF != nullptr && w3_host != nullptr && out1 != nullptr && ws != nullptr && C >= 0,
                "fcd_elm_rowsums: bad argument");
    int64_t grid = (C + 255) / 256;
    if (grid > (int64_t)sm_count() * 4) grid = (int64_t)sm_count() * 4;
    if (grid < 1) grid = 1;
    elm_rowsums_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(S9, qF, C, w3_host[0], w3_host[1], w3_host[2],
                                                                        out1, ws);
    return check_launch("fcd_elm_rowsums");
}

}  // extern "C"
