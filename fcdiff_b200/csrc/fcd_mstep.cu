// M-step and free-energy kernels: K3a (pi / gamma sums), K3b (objective and
// analytic gradient of the (eta, epsilon) sub-problem), K4 (energy terms).
// All reductions accumulate in fp64: warp shuffle -> block -> deterministic
// last-CTA grid reduction.
#include <cstring>

#include "fcd_common.cuh"
#include "fcd_solver.cuh"

namespace fcd {

constexpr int kRedThreads = 256;

// ------------------------------------------------------------------- K3a
// out[0..2] = sum_c exp(lqF[c,k]) (fcdiff/fit.py:219-220),
// out[3]    = sum_{n,u} exp(lqR[n,u,1]) (fit.py:212-213).
__global__ void __launch_bounds__(kRedThreads)
mstep_stats_kernel(const double* __restrict__ lqF, int64_t C,
                   const double* __restrict__ lqR, int64_t NU,
                   double* __restrict__ out, double* __restrict__ ws) {
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t nth = (int64_t)gridDim.x * blockDim.x;
    for (int64_t c = tid; c < C; c += nth) {
        v[0] += exp(lqF[c * 3]);
        v[1] += exp(lqF[c * 3 + 1]);
        v[2] += exp(lqF[c * 3 + 2]);
    }
    for (int64_t i = tid; i < NU; i += nth) v[3] += exp(lqR[i * 2 + 1]);
    grid_reduce_store<4, kRedThreads>(v, ws, out);
}

// ------------------------------------------------------------------- K3b
// Objective and analytic gradient of the (eta, epsilon) sub-problem from the
// responsibility planes of the local edge rows (fit.py:489-511 for the
// objective, fit.py:600-697 for the gradient; the total density cancels in the
// ratio num / M):
//   out[0] = sum_c sum_k qF_k sum_u sum_l w_l log(a_l + b_l p_k)   (theta-dependent part of E_lM;
//            E_lM = out[0] + the theta-free sum of elm_const_kernel)
//   out[1] = dE/d eta = -(2 eps - 1) sum qF_k w_2 num_k / (a_2 + b_2 p_k)
//   out[2] = dE/d eps = -sum qF_k s_l w_l num_k / (a_l + b_l p_k),  s = (-1, 1, 2 eta - 1)
// with num_k = (3 p_k - 1)/2.  Tiers T1 / T2 / T3 as described in fcd_common.cuh.
struct ElmAcc {
    double obj, ge, gh;       // objective, sum s_l w_l d_l, sum w_2 d_2
};

constexpr int kElmSeg = 256;

// SOLVE: evaluation point from the solver state, the series model's moments (fcd_solver.cuh), optimiser
// step in the last CTA
// (see elm_coded_kernel, fcd_streams.cu).
template <bool GRAD, bool FAST, bool SOLVE>
__global__ void __launch_bounds__(kStreamThreads, 1)
elm_kernel(const double* __restrict__ P, int64_t planeStride, int64_t C, int U, int64_t pitchU,
           const double* __restrict__ qF, const uint8_t* __restrict__ fstate,
           const double* __restrict__ qR, const uint8_t* __restrict__ rstate, int64_t pitchS,
           const int32_t* __restrict__ nm, const __grid_constant__ ThetaDev th,
           const __grid_constant__ LogTabWindow tab, int depth,
           double* __restrict__ out, double* __restrict__ ws,
           SolverState* __restrict__ state, const double* __restrict__ konst_dev,
           const __grid_constant__ CommPeers peers, int rank, int world, SolverPublished* pub,
           unsigned long long seq) {
    static_assert(!SOLVE || GRAD, "the solver needs the gradient sums");
    extern __shared__ __align__(128) double s_dyn[];
    __shared__ double s_sums[kSolverVals];
    if (SOLVE && solver_finished(state, pub, seq)) return;
    SubTheta T;
    if (SOLVE) {
        T = sub_theta(state->x[0], state->x[1]);
    } else {
        T.eta = th.eta;
        T.epsilon = th.epsilon;
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            T.al[l] = th.al[l];
            T.bl[l] = th.bl[l];
        }
    }
    const double* s_tab = load_log_table<FAST>(tab, s_dyn);
    unsigned char* s_stream = reinterpret_cast<unsigned char*>(s_dyn + (FAST ? ((tab.n + 1) & ~1) : 0));
    const double al[3] = {T.al[0], T.al[1], T.al[2]}, bl[3] = {T.bl[0], T.bl[1], T.bl[2]};
    const double sl[3] = {-1.0, 1.0, 2.0 * T.eta - 1.0};
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    ElmAcc acc = {0.0, 0.0, 0.0}, acc1 = {0.0, 0.0, 0.0};
    SolverMoments mo;
#pragma unroll
    for (int k = 0; k < kSolverK - 1; ++k) mo.a[k] = mo.b[k] = 0.0;
    // per-l constants of the T1 body {a_l, b_l, s_l, [l == 2]} (+ [l < 2] s_l for the moments); row 3 is
    // the neutral element for deferred / padding slots: log(1 + 0 p) = 0 exactly, zero gradient weight
    __shared__ double4 s_lc[4];
    __shared__ double s_lq[4];
    if (threadIdx.x < 4) {
        const int l = threadIdx.x;
        s_lc[l] = l < 3 ? make_double4(sel3(l, al), sel3(l, bl), sel3(l, sl), l == 2 ? 1.0 : 0.0) : make_double4(1.0, 0.0, 0.0, 0.0);
        s_lq[l] = l < 2 ? sel3(l, sl) : 0.0;
    }
    __syncthreads();

    // FAST: the T1 logs have weight exactly 1 -- running products, one logarithm per 2 x kProdMax factors
    // (fcd_math.cuh "Sum of logs as the log of a product"); the gradient takes 1 / M from rcp_newton
    double pr0 = 1.0, pr1 = 1.0;
    int nf = 0;
    auto flush = [&]() {
        if (FAST) acc.obj += log_pos<FAST>(pr0 * pr1, s_tab);
        pr0 = pr1 = 1.0;
        nf = 0;
    };
    auto live = [&](const double (&pv)[1], int lp, int e) {
        ElmAcc& a = e ? acc1 : acc;
        const double4 k = s_lc[lp];
        const double M = fma(k.y, pv[0], k.x);
        double rcp = 0.0;
        if (FAST) {
            (e ? pr1 : pr0) *= M;
            if (GRAD) rcp = rcp_newton(M);
        } else if (GRAD) {
            a.obj += fast_log_rcp<FAST>(M, s_tab, rcp);
        } else {
            a.obj += fast_log<FAST>(M, s_tab);
        }
        if (GRAD) {
            const double d = mix_num(pv[0]) * rcp;
            a.ge = fma(k.z, d, a.ge);
            a.gh = fma(k.w, d, a.gh);
            if (SOLVE) {
                add_powers1(mo.a, s_lq[lp] * d);
                add_powers1(mo.b, k.w * d);
            }
        }
        if (e == 1 && ++nf == kProdMax) flush();              // warp-uniform
    };
    struct Ops {
        double p;
        double2 qn, qm;
    };
    auto dload = [&](int64_t c, int u, int n, int m, int k, bool ok) {
        Ops o;
        o.p = 0.0;
        o.qn = o.qm = make_double2(0.0, 0.0);
        if (ok) {
            o.p = ldg_stream1(P + k * planeStride + c * pitchU + u);
            o.qn = __ldg(qR2 + (int64_t)n * U + u);
            o.qm = __ldg(qR2 + (int64_t)m * U + u);
        }
        return o;
    };
    // one element with the weights qw[l]: three logs, gradient and (SOLVE) Hessian sums
    auto weighted3 = [&](double p, const double (&qw)[3]) {
        const double num = mix_num(p);
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            const double M = fma(bl[l], p, al[l]);
            if (GRAD) {
                double rcp;
                acc.obj = fma(qw[l], fast_log_rcp<FAST>(M, s_tab, rcp), acc.obj);
                const double g = num * rcp;
                const double d = qw[l] * g;
                acc.ge = fma(sl[l], d, acc.ge);
                if (l == 2) acc.gh += d;
                if (SOLVE) {
                    if (l == 2) add_powers(mo.b, qw[l], g);
                    else add_powers(mo.a, qw[l], sl[l] * g);
                }
            } else {
                acc.obj = fma(qw[l], fast_log<FAST>(M, s_tab), acc.obj);
            }
        }
    };
    auto dcompute = [&](const Ops& o) {
        double w[3];
        pair_weights(o.qn, o.qm, w);
        weighted3(o.p, w);
    };
    auto full = [&](int64_t c, int n, int m, int u0, int u1) {
        const double qf[3] = {__ldg(qF + c * 3), __ldg(qF + c * 3 + 1), __ldg(qF + c * 3 + 2)};
        for (int u = u0 + (threadIdx.x & 31); u < u1; u += 32) {
            double w[3];
            pair_weights(__ldg(qR2 + (int64_t)n * U + u), __ldg(qR2 + (int64_t)m * U + u), w);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double p = ldg_stream1(P + k * planeStride + c * pitchU + u);
                const double qw[3] = {qf[k] * w[0], qf[k] * w[1], qf[k] * w[2]};
                weighted3(p, qw);
            }
        }
    };
    stream_tiered<1, kElmSeg, kStreamWarps, false, true>(P, planeStride, C, U, pitchU, fstate, rstate, pitchS, nm,
                                                         s_stream, depth, live, dload, dcompute, full,
                                                         [](int64_t) {});
    flush();
    if (SOLVE) {
        double v[kSolverVals];
        solver_sums(acc.obj + acc1.obj, acc.ge + acc1.ge, acc.gh + acc1.gh, mo, v);
        if (grid_reduce_last<kSolverVals, kStreamThreads>(v, ws, s_sums))
            solver_epilogue(s_sums, state, konst_dev, peers, rank, world, pub, seq);
    } else {
        double v[3] = {acc.obj + acc1.obj, -(2.0 * T.epsilon - 1.0) * (acc.gh + acc1.gh), -(acc.ge + acc1.ge)};
        grid_reduce_store<3, kStreamThreads>(v, ws, out);
    }
}

// Theta-free part of E_lM: out[0] = sum_c (sum_k qF_k) sum_u (sum_l w_l) L[c,u]
// (sum_l w_l = (q_n0 + q_n1)(q_m0 + q_m1), fit.py:382-406).  One read of the L plane.
__global__ void __launch_bounds__(kStreamThreads, 1)
elm_const_kernel(const double* __restrict__ L, int64_t C, int U, int64_t pitchU,
                 const double* __restrict__ qF, const uint8_t* __restrict__ fstate,
                 const double* __restrict__ qR, const uint8_t* __restrict__ rstate, int64_t pitchS,
                 const int32_t* __restrict__ nm, int depth, double* __restrict__ out, double* __restrict__ ws) {
    extern __shared__ __align__(128) double s_dyn[];
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    double acc = 0.0;
    auto wsum = [&](int n, int m, int u) {
        const double2 qn = __ldg(qR2 + (int64_t)n * U + u), qm = __ldg(qR2 + (int64_t)m * U + u);
        return (qn.x + qn.y) * (qm.x + qm.y);
    };
    double acc1 = 0.0;
    auto live = [&](const double (&pv)[1], int lp, int e) { (e ? acc1 : acc) += lp < 3 ? pv[0] : 0.0; };
    struct Ops {
        double w, L;
    };
    auto dload = [&](int64_t c, int u, int n, int m, int, bool ok) {
        Ops o;
        o.w = o.L = 0.0;
        if (ok) {
            o.w = wsum(n, m, u);
            o.L = ldg_stream1(L + c * pitchU + u);
        }
        return o;
    };
    auto dcompute = [&](const Ops& o) { acc = fma(o.w, o.L, acc); };
    auto full = [&](int64_t c, int n, int m, int u0, int u1) {
        const double qs = __ldg(qF + c * 3) + __ldg(qF + c * 3 + 1) + __ldg(qF + c * 3 + 2);
        for (int u = u0 + (threadIdx.x & 31); u < u1; u += 32)
            acc = fma(qs * wsum(n, m, u), ldg_stream1(L + c * pitchU + u), acc);
    };
    stream_tiered<1, kElmSeg, kStreamWarps, false, true>(L, 0, C, U, pitchU, fstate, rstate, pitchS, nm,
                                                         reinterpret_cast<unsigned char*>(s_dyn), depth,
                                                         live, dload, dcompute, full, [](int64_t) {});
    double v[1] = {acc + acc1};
    grid_reduce_store<1, kStreamThreads>(v, ws, out);
}

// ------------------------------------------------------------------- K3c
// Per-state sufficient statistics of the correlations (north_star subsystem 3;
// SURVEY 8f item 1 -- the reference ships only disabled pieces of a mu / sigma
// update, fcdiff/fit.py:232-237, 542-597, 709-733).  For the patients, the
// posterior weight that edge (c,u) is in state j, given q_F, q_R and theta, is
//   R_j = p_j sum_k qF_k sum_l w_l kappa_jkl / (a_l + b_l p_k),   kappa_jkl = eps_l (j == k) or a_l (j != k)
//       = p_j ( sum_l a_l Q_l + qF_j sum_l b_l T_jl ),  T_kl = w_l / (a_l + b_l p_k),  Q_l = sum_k qF_k T_kl
// (sum_j R_j = sum_k qF_k sum_l w_l).  out[0..2] = sum R_j, out[3..5] = sum R_j x,
// out[6..8] = sum R_j x^2: the weighted Gaussian statistics whose pooled maximiser
// is the EM (lower-bound) update of mu_j, sigma_j.  Runs once per iteration at
// most; all nine reciprocals for every element (no tiers).
template <bool FAST>
__global__ void __launch_bounds__(kRedThreads, 2)
patient_moments_kernel(const double* __restrict__ P, int64_t planeStride, const double* __restrict__ bt,
                       int64_t C, int U, int64_t pitchU,
                       const double* __restrict__ qF, const double* __restrict__ qR,
                       const int32_t* __restrict__ nm, const __grid_constant__ ThetaDev th,
                       double* __restrict__ out, double* __restrict__ ws) {
    double acc[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    for (int64_t c = warp0; c < C; c += nwarps) {
        const int v = __ldg(nm + c);
        const double2* qn = qR2 + (int64_t)(v & 0xffff) * U;
        const double2* qm = qR2 + (int64_t)((v >> 16) & 0xffff) * U;
        const double qf[3] = {__ldg(qF + c * 3), __ldg(qF + c * 3 + 1), __ldg(qF + c * 3 + 2)};
        for (int u = lane; u < U; u += 32) {
            const int64_t i = c * pitchU + u;
            const double x = ldg_stream1(bt + i);
            const double p[3] = {ldg_stream1(P + i), ldg_stream1(P + planeStride + i),
                                 ldg_stream1(P + 2 * planeStride + i)};
            double w[3];
            pair_weights(__ldg(qn + u), __ldg(qm + u), w);
            double T[3][3], Q[3];
#pragma unroll
            for (int l = 0; l < 3; ++l) {
#pragma unroll
                for (int k = 0; k < 3; ++k) T[k][l] = w[l] * fast_rcp<FAST>(mix_rel(th, l, p[k]));
                Q[l] = fma(qf[0], T[0][l], fma(qf[1], T[1][l], qf[2] * T[2][l]));
            }
            const double T0 = fma(th.al[0], Q[0], fma(th.al[1], Q[1], th.al[2] * Q[2]));
            const double x2 = x * x;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const double Tj = qf[j] * fma(th.bl[0], T[j][0], fma(th.bl[1], T[j][1], th.bl[2] * T[j][2]));
                const double R = p[j] * (T0 + Tj);
                acc[j] += R;
                acc[3 + j] = fma(R, x, acc[3 + j]);
                acc[6 + j] = fma(R, x2, acc[6 + j]);
            }
        }
    }
    grid_reduce_store<9, kRedThreads>(acc, ws, out);
}

// Controls: out[0..2] = H sum_c qF[c,j], out[3..5] = sum_c qF[c,j] S1[c], out[6..8] = sum_c qF[c,j] S2[c].
__global__ void __launch_bounds__(kRedThreads)
control_moments_kernel(const double* __restrict__ S1, const double* __restrict__ S2, double H,
                       const double* __restrict__ qF, int64_t C, double* __restrict__ out,
                       double* __restrict__ ws) {
    double acc[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < C;
         c += (int64_t)gridDim.x * blockDim.x) {
        const double s1 = S1[c], s2 = S2[c];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double q = qF[c * 3 + j];
            acc[j] = fma(H, q, acc[j]);
            acc[3 + j] = fma(q, s1, acc[3 + j]);
            acc[6 + j] = fma(q, s2, acc[6 + j]);
        }
    }
    grid_reduce_store<9, kRedThreads>(acc, ws, out);
}

// ------------------------------------------------------------------- K4
// The six terms of fcdiff/fit.py:142-155.  E_lM (v[3]) of the local shard comes
// from the K3b passes (fcd_elm_obj_grad + fcd_elm_const) and is passed in.
//  v[0] E_lp_F = sum qF log gamma (fit.py:458)   v[1] E_lp_B_g_F (fit.py:472, via S1,S2)
//  v[2] E_lp_R = sum qR log[1-pi, pi] (fit.py:486)
//  v[4] E_lq_F = sum qF lqF (fit.py:525)         v[5] E_lq_R = sum qR lqR (fit.py:539)
// MASKED: S0[c] observed controls of edge c (healthy_term).
template <bool MASKED>
__global__ void __launch_bounds__(kRedThreads)
energy_small_kernel(const double* __restrict__ S1, const double* __restrict__ S2, const double* __restrict__ S0,
                    const double* __restrict__ lqF, const double* __restrict__ qF, int64_t C,
                    const double* __restrict__ lqR, const double* __restrict__ qR, int64_t NU,
                    const __grid_constant__ ThetaDev th, double elm_value, const SolverState* __restrict__ solved,
                    double* __restrict__ out6, double* __restrict__ ws) {
    double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t nth = (int64_t)gridDim.x * blockDim.x;
    // E_lM: given by the host, or taken from the state of the device-resident (eta, epsilon) solve that
    // finished just before this launch on the same stream (f = -E_lM at the solution; NaN if it has not)
    if (tid == 0) v[3] = solved != nullptr ? (solved->done ? -solved->f : __longlong_as_double(0x7ff8000000000000ll)) : elm_value;
    for (int64_t c = tid; c < C; c += nth) {
        const double s1 = S1[c], s2 = S2[c], s0 = MASKED ? S0[c] : 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const double l = lqF[c * 3 + k];
            const double q = qF[c * 3 + k];
            v[0] = fma(q, th.log_gamma[k], v[0]);
            v[1] = fma(q, healthy_term<MASKED>(th, k, s1, s2, s0), v[1]);
            v[4] = fma(q, l, v[4]);
        }
    }
    for (int64_t i = tid; i < NU; i += nth) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const double l = lqR[i * 2 + j];
            const double q = qR[i * 2 + j];
            v[2] = fma(q, th.log_pi2[j], v[2]);
            v[5] = fma(q, l, v[5]);
        }
    }
    grid_reduce_store<6, kRedThreads>(v, ws, out6);
}

static inline int red_grid(int64_t work_items, int items_per_block) {
    int64_t need = (work_items + items_per_block - 1) / items_per_block;
    int64_t cap = (int64_t)sm_count() * 8;
    if (cap > kMaxReduceBlocks) cap = kMaxReduceBlocks;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

static inline int stream_grid(int64_t C) {
    int64_t need = (C + kStreamWarps - 1) / kStreamWarps;      // < 65536 rows per warp: C < 2^20 * grid
    if (need < 1) need = 1;
    return (int)(need < sm_count() ? need : sm_count());          // one persistent CTA per SM
}

static inline bool planes_ok(const void* a, const void* b, int64_t pitchU, int64_t planeStride, int64_t pitchS) {
    const uintptr_t al = reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b);
    return (al & 15) == 0 && pitchU % 2 == 0 && planeStride % 2 == 0 && pitchS % 256 == 0;
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int fcd_mstep_stats(const double* lqF, int64_t C, const double* lqR, int64_t NU,
                    double* out4, double* ws, void* stream) {
    FCD_REQUIRE(C >= 0 && NU >= 0 && ws != nullptr, "fcd_mstep_stats: bad arguments");
    const int64_t work = C > NU ? C : NU;
    mstep_stats_kernel<<<red_grid(work, kRedThreads), kRedThreads, 0, (cudaStream_t)stream>>>(
        lqF, C, lqR, NU, out4, ws);
    return check_launch("fcd_mstep_stats");
}

int fcd_elm_obj_grad(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                     const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate,
                     int64_t pitchS, int32_t N, const int32_t* nm,
                     const fcd_theta* theta_host, int32_t want_grad,
                     double* out3, double* ws, void* stream) {
    FCD_REQUIRE(theta_host != nullptr && ws != nullptr && P != nullptr && qF != nullptr && fstate != nullptr &&
                qR != nullptr && rstate != nullptr && nm != nullptr && out3 != nullptr,
                "fcd_elm_obj_grad: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && U < 65536 && pitchU >= U && pitchS >= U && N >= 2 && N < 65536,
                "fcd_elm_obj_grad: bad shape");
    FCD_REQUIRE(planes_ok(P, nullptr, pitchU, planeStride, pitchS),
                "fcd_elm_obj_grad: planes must be 16-byte aligned with even pitches (pitchS % 256 == 0)");
    const ThetaDev th = make_theta_dev(*theta_host, 0);
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(th.epsl, th.al, st, tab, true), "fcd_elm_obj_grad: log table initialisation failed");
    const bool fast = log_table_covers(th.epsl, th.al);
    const size_t tbytes = fast ? (size_t)((tab.n + 1) & ~1) * sizeof(double) : 0;
    const int depth = stream_depth<1, kElmSeg>(tbytes);
    FCD_REQUIRE(depth >= 2, "fcd_elm_obj_grad: shared memory budget exceeded");
    const size_t smem = tbytes + StreamGeom<1, kElmSeg>::bytes(kStreamWarps, depth);
    const int grid = stream_grid(C);
    CommPeers nopeers;
    comm_peers_from_host(nullptr, 1, nopeers);
#define FCD_ELM(G, F)                                                                                  \
    do {                                                                                               \
        FCD_ALLOW_BIG_SMEM(elm_kernel<G, F, false>);                                                   \
        elm_kernel<G, F, false><<<grid, kStreamThreads, smem, st>>>(P, planeStride, C, U, pitchU, qF, fstate, qR, \
                                                                    rstate, pitchS, nm, th, tab, depth, out3, ws, \
                                                                    nullptr, nullptr, nopeers, 0, 1, nullptr, 0ull); \
    } while (0)
    if (want_grad) { if (fast) FCD_ELM(true, true); else FCD_ELM(true, false); }
    else           { if (fast) FCD_ELM(false, true); else FCD_ELM(false, false); }
#undef FCD_ELM
    return check_launch("fcd_elm_obj_grad");
}

int fcd_elm_tiered_solve(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                         const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate,
                         int64_t pitchS, int32_t N, const int32_t* nm, double eps_lo, double eps_hi, void* state,
                         const double* konst, void* const* windows_host, int32_t rank, int32_t world,
                         void* published_host, uint64_t seq0, int32_t n_launches, double* ws, void* stream) {
    FCD_REQUIRE(state != nullptr && ws != nullptr && P != nullptr && qF != nullptr && fstate != nullptr &&
                qR != nullptr && rstate != nullptr && nm != nullptr, "fcd_elm_tiered_solve: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && U < 65536 && pitchU >= U && pitchS >= U && N >= 2 && N < 65536,
                "fcd_elm_tiered_solve: bad shape");
    FCD_REQUIRE(planes_ok(P, nullptr, pitchU, planeStride, pitchS),
                "fcd_elm_tiered_solve: planes must be 16-byte aligned with even pitches (pitchS % 256 == 0)");
    FCD_REQUIRE(n_launches >= 1 && n_launches <= 64 && world >= 1 && world <= kCommMaxWorld && rank >= 0 && rank < world &&
                eps_lo > 0.0 && eps_lo <= eps_hi && eps_hi < 1.0, "fcd_elm_tiered_solve: bad launch / box arguments");
    CommPeers peers;
    FCD_REQUIRE(comm_peers_from_host(windows_host, world, peers), "fcd_elm_tiered_solve: NULL window");
    SolverPublished* pub = nullptr;
    if (published_host != nullptr) {
        cudaError_t e = cudaHostGetDevicePointer((void**)&pub, published_host, 0);
        FCD_REQUIRE(e == cudaSuccess, "fcd_elm_tiered_solve: cudaHostGetDevicePointer: %s", cudaGetErrorString(e));
    }
    const double m = eps_lo < 1.0 - eps_hi ? eps_lo : 1.0 - eps_hi;
    const double epsl[3] = {m, m, m}, al[3] = {0.5 * m, 0.5 * m, 0.5 * m};
    ThetaDev th;
    memset(&th, 0, sizeof(th));
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(epsl, al, st, tab, true), "fcd_elm_tiered_solve: log table initialisation failed");
    const bool fast = log_table_covers(epsl, al);
    const size_t tbytes = fast ? (size_t)((tab.n + 1) & ~1) * sizeof(double) : 0;
    const int depth = stream_depth<1, kElmSeg>(tbytes);
    FCD_REQUIRE(depth >= 2, "fcd_elm_tiered_solve: shared memory budget exceeded");
    const size_t smem = tbytes + StreamGeom<1, kElmSeg>::bytes(kStreamWarps, depth);
    const int grid = stream_grid(C);
    if (fast) FCD_ALLOW_BIG_SMEM(elm_kernel<true, true, true>);
    else FCD_ALLOW_BIG_SMEM(elm_kernel<true, false, true>);
    for (int i = 0; i < n_launches; ++i) {
        const unsigned long long seq = (unsigned long long)seq0 + (unsigned long long)i;
        if (fast)
            elm_kernel<true, true, true><<<grid, kStreamThreads, smem, st>>>(
                P, planeStride, C, U, pitchU, qF, fstate, qR, rstate, pitchS, nm, th, tab, depth, nullptr, ws,
                static_cast<SolverState*>(state), konst, peers, rank, world, pub, seq);
        else
            elm_kernel<true, false, true><<<grid, kStreamThreads, smem, st>>>(
                P, planeStride, C, U, pitchU, qF, fstate, qR, rstate, pitchS, nm, th, tab, depth, nullptr, ws,
                static_cast<SolverState*>(state), konst, peers, rank, world, pub, seq);
        int rc = check_launch("fcd_elm_tiered_solve");
        if (rc) return rc;
    }
    return 0;
}

int fcd_elm_const(const double* L, int64_t C, int32_t U, int64_t pitchU,
                  const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate,
                  int64_t pitchS, int32_t N, const int32_t* nm, double* out1, double* ws, void* stream) {
    FCD_REQUIRE(ws != nullptr && L != nullptr && qF != nullptr && fstate != nullptr && qR != nullptr &&
                rstate != nullptr && nm != nullptr && out1 != nullptr, "fcd_elm_const: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && U < 65536 && pitchU >= U && pitchS >= U && N >= 2 && N < 65536,
                "fcd_elm_const: bad shape");
    FCD_REQUIRE(planes_ok(L, nullptr, pitchU, 0, pitchS), "fcd_elm_const: plane must be 16-byte aligned with even pitches");
    const int depth = stream_depth<1, kElmSeg>(0);
    const size_t smem = StreamGeom<1, kElmSeg>::bytes(kStreamWarps, depth);
    cudaFuncSetAttribute(elm_const_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget);
    elm_const_kernel<<<stream_grid(C), kStreamThreads, smem, (cudaStream_t)stream>>>(
        L, C, U, pitchU, qF, fstate, qR, rstate, pitchS, nm, depth, out1, ws);
    return check_launch("fcd_elm_const");
}

// S0 == NULL: every edge has all H controls (the unmasked kernel).
int fcd_energy_terms(const double* S1, const double* S2, const double* S0, int32_t H,
                     const double* lqF, const double* qF, int64_t C,
                     const double* lqR, const double* qR, int32_t N, int32_t U,
                     const fcd_theta* theta_host, double elm, const void* solver_state,
                     double* out6, double* ws, void* stream) {
    FCD_REQUIRE(theta_host != nullptr && ws != nullptr && out6 != nullptr, "fcd_energy_terms: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && N >= 2 && H >= 1, "fcd_energy_terms: bad shape");
    const ThetaDev th = make_theta_dev(*theta_host, H);
    const int64_t NU = (int64_t)N * U;
    const int64_t work = C > NU ? C : NU;
    const SolverState* solved = static_cast<const SolverState*>(solver_state);
    if (S0 != nullptr)
        energy_small_kernel<true><<<red_grid(work, kRedThreads), kRedThreads, 0, (cudaStream_t)stream>>>(
            S1, S2, S0, lqF, qF, C, lqR, qR, NU, th, elm, solved, out6, ws);
    else
        energy_small_kernel<false><<<red_grid(work, kRedThreads), kRedThreads, 0, (cudaStream_t)stream>>>(
            S1, S2, nullptr, lqF, qF, C, lqR, qR, NU, th, elm, solved, out6, ws);
    return check_launch("fcd_energy_terms");
}

int fcd_state_moments(const double* S1, const double* S2, int32_t H,
                      const double* bt, const double* P, int64_t planeStride,
                      int64_t C, int32_t U, int64_t pitchU,
                      const double* qF, const double* qR, int32_t N, const int32_t* nm,
                      const fcd_theta* theta_host, double* out18, double* ws, void* stream) {
    FCD_REQUIRE(theta_host != nullptr && ws != nullptr && out18 != nullptr && nm != nullptr,
                "fcd_state_moments: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && pitchU >= U && N >= 2 && N < 65536 && H >= 1, "fcd_state_moments: bad shape");
    const ThetaDev th = make_theta_dev(*theta_host, H);
    cudaStream_t st = (cudaStream_t)stream;
    control_moments_kernel<<<red_grid(C, kRedThreads), kRedThreads, 0, st>>>(S1, S2, (double)H, qF, C, out18, ws);
    int rc = check_launch("fcd_state_moments(controls)");
    if (rc) return rc;
    int grid = red_grid(C, kRedThreads / 32);
    if (grid > sm_count() * 2) grid = sm_count() * 2;
    if (log_table_covers(th.epsl, th.al))
        patient_moments_kernel<true><<<grid, kRedThreads, 0, st>>>(P, planeStride, bt, C, U, pitchU, qF, qR, nm, th,
                                                                   out18 + 9, ws);
    else
        patient_moments_kernel<false><<<grid, kRedThreads, 0, st>>>(P, planeStride, bt, C, U, pitchU, qF, qR, nm, th,
                                                                    out18 + 9, ws);
    return check_launch("fcd_state_moments(patients)");
}

}  // extern "C"
