// Scoring subjects a fitted model was not trained on (UnsharedRegionFit.score_patients): per-patient shares
// of the free energy (fcdiff/fit.py:142-155, 475-539) and the change of q_R between two region sweeps
// (fcdiff/fit.py:176-198).  With theta and q_F fixed the free energy is a sum over patient columns, so every
// term here is kept per patient instead of being reduced to one scalar as K3b / K4 do.
//
//   patient_terms_rows_kernel   per (row block, patient) cell: the E_lM share and sum_k q_F log M_k0 over the
//                               rows of the block, in row order, into part[b][u][2];
//   patient_terms_finish_kernel per patient: the row-block partials in block order, and the two q_R-only sums
//                               (E_lp_R, E_lq_R) over the regions in region order.
// The row blocks are a partition of [0, C) that depends on C alone and a cell is evaluated by ONE thread from
// start to end, so a patient's four sums do not depend on U, on which other patients are scored with it, or on
// how cells are mapped onto lanes.  Lanes run along the patient dimension (coalesced plane and q_R reads); when
// fewer than 32 patients are scored a warp takes several row blocks side by side instead of idling lanes.
//
// Tiers as in fcd_common.cuh: an edge whose q_F is peaked (fstate < 3) reads its k* plane and L only (16 bytes
// per edge-patient); where both regions of the edge are peaked as well the weight is exactly 1 and the factor
// a_l + b_l p enters a running product (one logarithm per kProdMax factors, fcd_math.cuh), otherwise each
// weighted term takes its own logarithm.  Unpeaked edges read all three planes.
//
// Posteriors of the anomalous connections T and the patients' connection states F~
// (UnsharedRegionFit.connection_posteriors), for fitted and held-out patients alike.  Given the template state
// F = k of edge c and the pair state l of its regions (0 both typical, 1 both anomalous, 2 mixed), the
// generative model (fcdiff/model.py:141-188) gives, with the plane values p of b~[c,u] and a_l, b_l, eps_l of
// fcd_common.cuh, the exact conditionals
//   P(F~ = j | k, l, b~) = eps_l p_k / (a_l + b_l p_k)   (j = k),   a_l p_j / (a_l + b_l p_k)   (j != k)
//   P(T = 1  | k, l, b~) = 0 (l = 0),  1 (l = 1),  eta (eps p_k + a_1 (1 - p_k)) / (a_2 + b_2 p_k)   (l = 2)
// and the read-outs are their expectations under q_F[c,k] w_l[c,u], the pair weights of the edge's own regions
// (as fit.py:489-511; the sweep's edge lookup plays no part).
//   connection_rows_kernel      per (row block, patient) cell, the row partition and lane mapping of
//                               patient_terms_rows_kernel: q_T[c][u] (and q_F~[c][u][0..2] when MAPS), and the
//                               cell's sum of q_T over its rows, in row order, into part[b][u];
//   connection_finish_kernel    expected[u]: the row-block partials in block order; rate[c]: row c of q_T summed
//                               in a fixed lane order, over U.
// Tiers: a peaked edge with both regions peaked is one (k*, l*) term (one division); a peaked edge with an
// undecided region takes the three l terms; an unpeaked edge all nine with q_F weights.  Weights <= 2^-60 are
// dropped.  Without maps a peaked edge reads its k* plane only, and only for a mixed pair term.  No logarithm is
// taken, so there is no log table and no SAFE variant; q_T is formed by the same instructions in both variants,
// so the reductions do not depend on whether the maps are written.
//
// Per-subject control log-likelihoods (UnsharedRegionFit.score_controls / classify_subjects): one control's
// share of E_lp_B_g_F (fcdiff/fit.py:461-472) for a new column x, sum_c sum_k q_F[c,k] log N(x_c; mu_k, sigma_k)
// with the log density of fit.py:111-114.
//   control_terms_rows_kernel   per (row block, subject) cell, the row partition and lane mapping of
//                               patient_terms_rows_kernel: the cell's sum over its rows, in row order, into
//                               part[b][s];
//   connection_finish_kernel    (its `expected` blocks only) the row-block partials of each subject in block order.
// All three weighted terms are evaluated on every element: no tiers, no peak states, no logarithm.
#include "fcd_common.cuh"

namespace fcd {

constexpr int kPtThreads = 256;
constexpr int kPtMinRows = 16;            // rows per block at least ...
constexpr int64_t kPtMaxBlocks = 2048;    // ... and at most this many blocks: the partials stay <= 32 KB per patient
constexpr int kChThreads = 1024;

inline int64_t pt_row_blocks(int64_t C) {
    int64_t nb = (C + kPtMinRows - 1) / kPtMinRows;
    if (nb > kPtMaxBlocks) nb = kPtMaxBlocks;
    return nb < 1 ? 1 : nb;
}

// 0 / 1: q_R pair peaked on that state (as peak_states_R), 2: anything else
__device__ __forceinline__ int peak_state2(double2 q) {
    if (q.x == 1.0 && q.y <= kPeakTau) return 0;
    if (q.y == 1.0 && q.x <= kPeakTau) return 1;
    return 2;
}

template <bool FAST>
__global__ void __launch_bounds__(kPtThreads)
patient_terms_rows_kernel(const double* __restrict__ P, int64_t planeStride, const double* __restrict__ L, int64_t C,
                          int U, int64_t pitchU, const double* __restrict__ qF, const uint8_t* __restrict__ fstate,
                          const double* __restrict__ qR, const __grid_constant__ ThetaDev th,
                          const __grid_constant__ LogTabWindow tab, int64_t nb, int64_t rows, int lanesP,
                          double* __restrict__ part) {
    extern __shared__ __align__(16) double s_dyn[];
    const double* s_tab = load_log_table<FAST>(tab, s_dyn);
    const int lane = threadIdx.x & 31;
    // 32-bit index arithmetic (the host bounds the warp count): a 64-bit division is a called routine
    const unsigned gw = (blockIdx.x * kPtThreads + threadIdx.x) >> 5;
    const unsigned tiles = (unsigned)(U + lanesP - 1) / (unsigned)lanesP;
    const int64_t rb = (int64_t)(gw / tiles) * (32 / lanesP) + lane / lanesP;
    const int u = (int)(gw % tiles) * lanesP + (lane & (lanesP - 1));
    if (rb >= nb || u >= U) return;
    const int64_t c0 = rb * rows;
    const int64_t c1 = c0 + rows < C ? c0 + rows : C;
    int n, m;
    c_to_nm(c0, n, m);
    const double2* q2 = reinterpret_cast<const double2*>(qR);
    double accM = 0.0, acc0 = 0.0, sumL = 0.0, sumL0 = 0.0;   // E_lM share; sum_k q_F log M_k0
    double prM = 1.0, pr0 = 1.0;                               // running products of weight-1 factors (FAST)
    int nf = 0;
    for (int64_t c = c0; c < c1; ++c) {
        const int k = __ldg(fstate + c);
        const double Lv = __ldg(L + c * pitchU + u);
        const double2 qn = __ldg(q2 + (int64_t)n * U + u), qm = __ldg(q2 + (int64_t)m * U + u);
        const int sn = peak_state2(qn), sm = peak_state2(qm);
        const bool peakR = sn < 2 && sm < 2;
        const int ls = (sn ^ sm) ? 2 : sn;                     // l* of a peaked pair (fit.py:382-406)
        if (k < 3) {
            const double p = __ldg(P + k * planeStride + c * pitchU + u);
            const double y0 = mix_rel(th, 0, p);
            sumL0 += Lv;
            if (FAST) pr0 *= y0;
            else acc0 += log(y0);
            if (peakR) {
                const double y = mix_rel(th, ls, p);
                if (FAST) prM *= y;
                else accM += log(y);
                sumL += Lv;
            } else {
                double w[3];
                pair_weights(qn, qm, w);
                accM += w[0] * fast_log<FAST>(y0, s_tab) + w[1] * fast_log<FAST>(mix_rel(th, 1, p), s_tab) +
                        w[2] * fast_log<FAST>(mix_rel(th, 2, p), s_tab);
                sumL += (w[0] + w[1] + w[2]) * Lv;
            }
            if (FAST && ++nf == kProdMax) {
                accM += log_pos<FAST>(prM, s_tab);
                acc0 += log_pos<FAST>(pr0, s_tab);
                prM = pr0 = 1.0;
                nf = 0;
            }
        } else {
            const double f[3] = {__ldg(qF + c * 3), __ldg(qF + c * 3 + 1), __ldg(qF + c * 3 + 2)};
            const double fs = f[0] + f[1] + f[2];
            double w[3];
            if (peakR) {
                w[0] = ls == 0 ? 1.0 : 0.0;
                w[1] = ls == 1 ? 1.0 : 0.0;
                w[2] = ls == 2 ? 1.0 : 0.0;
            } else {
                pair_weights(qn, qm, w);
            }
#pragma unroll
            for (int kk = 0; kk < 3; ++kk) {
                const double p = __ldg(P + kk * planeStride + c * pitchU + u);
                const double g0 = fast_log<FAST>(mix_rel(th, 0, p), s_tab);
                acc0 += f[kk] * g0;
                double s = w[0] * g0;
                if (w[1] != 0.0) s += w[1] * fast_log<FAST>(mix_rel(th, 1, p), s_tab);
                if (w[2] != 0.0) s += w[2] * fast_log<FAST>(mix_rel(th, 2, p), s_tab);
                accM += f[kk] * s;
            }
            sumL0 += fs * Lv;
            sumL += fs * (w[0] + w[1] + w[2]) * Lv;
        }
        if (++m == n) {
            ++n;
            m = 0;
        }
    }
    if (FAST) {
        accM += log_pos<FAST>(prM, s_tab);
        acc0 += log_pos<FAST>(pr0, s_tab);
    }
    reinterpret_cast<double2*>(part)[rb * U + u] = make_double2(accM + sumL, acc0 + sumL0);
}

// out4[u] = {E_lM, E_lp_R, E_lq_R, sum_k q_F log M_k0}: warps take the row blocks and regions round robin, the
// eight warp sums are added in warp order
__global__ void __launch_bounds__(kPtThreads)
patient_terms_finish_kernel(const double* __restrict__ part, int64_t nb, const double* __restrict__ qR,
                            const double* __restrict__ lqR, int N, int U, double lp0, double lp1,
                            double* __restrict__ out4) {
    __shared__ double s[kPtThreads / 32][32][4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int u = blockIdx.x * 32 + lane;
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    if (u < U) {
        const double2* p2 = reinterpret_cast<const double2*>(part);
        for (int64_t b = warp; b < nb; b += kPtThreads / 32) {
            const double2 x = p2[b * U + u];
            v[0] += x.x;
            v[3] += x.y;
        }
        const double2* q2 = reinterpret_cast<const double2*>(qR);
        const double2* l2 = reinterpret_cast<const double2*>(lqR);
        for (int n = warp; n < N; n += kPtThreads / 32) {
            const double2 q = q2[(int64_t)n * U + u], l = l2[(int64_t)n * U + u];
            v[1] += q.x * lp0 + q.y * lp1;                            // fit.py:475-486
            v[2] += q.x * l.x + q.y * l.y;                            // fit.py:528-539
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) s[warp][lane][i] = v[i];
    __syncthreads();
    if (warp == 0 && u < U) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double t = s[0][lane][i];
            for (int w = 1; w < kPtThreads / 32; ++w) t += s[w][lane][i];
            out4[(int64_t)u * 4 + i] = t;
        }
    }
}

// per patient: max over regions and both states of |qb - qa|; the block's maximum joins out1 by atomicMax on the
// bit pattern (non-negative doubles order like their bits; a NaN is kept)
__global__ void __launch_bounds__(kChThreads)
qR_change_kernel(const double* __restrict__ qa, const double* __restrict__ qb, int N, int U,
                 double* __restrict__ maxU, double* __restrict__ out1) {
    __shared__ double s[kChThreads / 32][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int u = blockIdx.x * 32 + lane;
    double mx = 0.0;
    if (u < U) {
        const double2* a2 = reinterpret_cast<const double2*>(qa);
        const double2* b2 = reinterpret_cast<const double2*>(qb);
#pragma unroll 4
        for (int n = warp; n < N; n += kChThreads / 32) {
            const double2 a = __ldg(a2 + (int64_t)n * U + u), b = __ldg(b2 + (int64_t)n * U + u);
            const double d0 = fabs(b.x - a.x), d1 = fabs(b.y - a.y);
            mx = (d0 > mx || d0 != d0) ? d0 : mx;
            mx = (d1 > mx || d1 != d1) ? d1 : mx;
        }
    }
    s[warp][lane] = mx;
    __syncthreads();
    if (warp == 0) {
        double t = s[0][lane];
        for (int w = 1; w < kChThreads / 32; ++w) t = (s[w][lane] > t || s[w][lane] != s[w][lane]) ? s[w][lane] : t;
        if (u < U && maxU != nullptr) maxU[u] = t;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double x = __shfl_xor_sync(0xffffffffu, t, o);
            t = (x > t || x != x) ? x : t;
        }
        if (lane == 0)
            atomicMax(reinterpret_cast<unsigned long long*>(out1), (unsigned long long)__double_as_longlong(t));
    }
}

// one (k, l) term of weight wt: P(T = 1 | k, l) into t and, when MAPS, P(F~ = . | k, l) into g.  pk = p_k;
// p: all three planes (read only when MAPS).  The q_T arithmetic is spelled with rounding intrinsics: the
// compiler may not contract it differently in the two variants (whose other uses of wt and inv differ)
template <bool MAPS>
__device__ __forceinline__ void connection_term(const ThetaDev& th, int k, int l, double wt, double pk,
                                                const double (&p)[3], double& t, double (&g)[3]) {
    if (l == 1) t = __dadd_rn(t, wt);
    if (MAPS || l == 2) {
        const double inv = __ddiv_rn(1.0, mix_rel(th, l, pk));
        if (l == 2) {
            const double num = __fma_rn(th.epsilon, pk, __dmul_rn(th.al[1], __dsub_rn(1.0, pk)));
            t = __fma_rn(wt, __dmul_rn(__dmul_rn(th.eta, num), inv), t);
        }
        if (MAPS) {
            const double s = wt * inv, sa = s * th.al[l], se = s * th.epsl[l];
#pragma unroll
            for (int j = 0; j < 3; ++j) g[j] = fma(j == k ? se : sa, p[j], g[j]);
        }
    }
}

template <bool MAPS>
__global__ void __launch_bounds__(kPtThreads)
connection_rows_kernel(const double* __restrict__ P, int64_t planeStride, int64_t C, int U, int64_t pitchU,
                       const double* __restrict__ qF, const uint8_t* __restrict__ fstate,
                       const double* __restrict__ qR, const __grid_constant__ ThetaDev th, int64_t nb, int64_t rows,
                       int lanesP, double* __restrict__ qT, double* __restrict__ qFt, double* __restrict__ part) {
    const int lane = threadIdx.x & 31;
    const unsigned gw = (blockIdx.x * kPtThreads + threadIdx.x) >> 5;
    const unsigned tiles = (unsigned)(U + lanesP - 1) / (unsigned)lanesP;
    const int64_t rb = (int64_t)(gw / tiles) * (32 / lanesP) + lane / lanesP;
    const int u = (int)(gw % tiles) * lanesP + (lane & (lanesP - 1));
    if (rb >= nb || u >= U) return;
    const int64_t c0 = rb * rows;
    const int64_t c1 = c0 + rows < C ? c0 + rows : C;
    int n, m;
    c_to_nm(c0, n, m);
    const double2* q2 = reinterpret_cast<const double2*>(qR);
    double acc = 0.0;
    for (int64_t c = c0; c < c1; ++c) {
        const int k = __ldg(fstate + c);
        const double2 qn = __ldg(q2 + (int64_t)n * U + u), qm = __ldg(q2 + (int64_t)m * U + u);
        const int sn = peak_state2(qn), sm = peak_state2(qm);
        double w[3];
        if (sn < 2 && sm < 2) {
            const int ls = (sn ^ sm) ? 2 : sn;                     // l* of a peaked pair (fit.py:382-406)
            w[0] = ls == 0 ? 1.0 : 0.0;
            w[1] = ls == 1 ? 1.0 : 0.0;
            w[2] = ls == 2 ? 1.0 : 0.0;
        } else {
            w[0] = __dmul_rn(qn.x, qm.x);                          // pair_weights, not contracted
            w[1] = __dmul_rn(qn.y, qm.y);
            w[2] = __fma_rn(qn.y, qm.x, __dmul_rn(qn.x, qm.y));
        }
        const double* pc = P + c * pitchU + u;
        double p[3] = {0.0, 0.0, 0.0};
        if (MAPS || (k == 3 && w[2] > kPeakTau)) {
#pragma unroll
            for (int j = 0; j < 3; ++j) p[j] = __ldg(pc + j * planeStride);
        }
        double t = 0.0, g[3] = {0.0, 0.0, 0.0};
        if (k < 3) {
            const double pk = MAPS ? sel3(k, p) : (w[2] > kPeakTau ? __ldg(pc + k * planeStride) : 0.0);
#pragma unroll
            for (int l = 0; l < 3; ++l)
                if (w[l] > kPeakTau) connection_term<MAPS>(th, k, l, w[l], pk, p, t, g);
        } else {
            const double f[3] = {__ldg(qF + c * 3), __ldg(qF + c * 3 + 1), __ldg(qF + c * 3 + 2)};
#pragma unroll
            for (int kk = 0; kk < 3; ++kk) {
                if (f[kk] <= kPeakTau) continue;
#pragma unroll
                for (int l = 0; l < 3; ++l)
                    if (w[l] > kPeakTau) connection_term<MAPS>(th, kk, l, __dmul_rn(f[kk], w[l]), p[kk], p, t, g);
            }
        }
        qT[c * U + u] = t;
        if (MAPS) {
            double* o = qFt + (c * U + u) * 3;
            o[0] = g[0];
            o[1] = g[1];
            o[2] = g[2];
        }
        acc = __dadd_rn(acc, t);
        if (++m == n) {
            ++n;
            m = 0;
        }
    }
    part[rb * U + u] = acc;
}

// blocks [0, bU): expected[u] for 32 patients each, warps take the row blocks round robin and the eight warp sums
// are added in warp order; blocks [bU, ...): rate[c] for 8 rows each, one warp per row, lanes stride the patients
// and the lane sums are added by a fixed butterfly
__global__ void __launch_bounds__(kPtThreads)
connection_finish_kernel(const double* __restrict__ part, int64_t nb, const double* __restrict__ qT, int64_t C,
                         int U, int bU, double* __restrict__ expected, double* __restrict__ rate) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if ((int)blockIdx.x < bU) {
        __shared__ double s[kPtThreads / 32][32];
        const int u = blockIdx.x * 32 + lane;
        double v = 0.0;
        if (u < U)
            for (int64_t b = warp; b < nb; b += kPtThreads / 32) v += part[b * U + u];
        s[warp][lane] = v;
        __syncthreads();
        if (warp == 0 && u < U) {
            double t = s[0][lane];
            for (int w = 1; w < kPtThreads / 32; ++w) t += s[w][lane];
            expected[u] = t;
        }
        return;
    }
    const int64_t c = (int64_t)(blockIdx.x - bU) * (kPtThreads / 32) + warp;
    if (c >= C) return;
    const double* row = qT + c * U;
    double v = 0.0;
    for (int u = lane; u < U; u += 32) v += row[u];
    v = warp_sum(v);
    if (lane == 0) rate[c] = v / U;
}

// per-state constants of log N(x; mu_k, sigma_k) = -((x - mu_k) / sigma_k)^2 / 2 - nc_k, formed once per launch
struct ControlConsts {
    double mu[3];
    double isig[3];     // 1 / sigma_k
    double nc[3];       // log sigma_k + log sqrt(2 pi)
};

constexpr int kCtRows = 8;                  // rows whose loads a thread has in flight at once

// MASKED: a NaN entry is not observed and enters like a row past the block's end (weight 0, value 0).
template <bool MASKED>
__global__ void __launch_bounds__(kPtThreads)
control_terms_rows_kernel(const double* __restrict__ X, int64_t C, int S, int64_t pitchS, const double* __restrict__ qF,
                          const __grid_constant__ ControlConsts cc, int64_t nb, int64_t rows, int lanesP,
                          double* __restrict__ part) {
    const int lane = threadIdx.x & 31;
    const unsigned gw = (blockIdx.x * kPtThreads + threadIdx.x) >> 5;
    const unsigned tiles = (unsigned)(S + lanesP - 1) / (unsigned)lanesP;
    const int64_t rb = (int64_t)(gw / tiles) * (32 / lanesP) + lane / lanesP;
    const int s = (int)(gw % tiles) * lanesP + (lane & (lanesP - 1));
    if (rb >= nb || s >= S) return;
    const int64_t c0 = rb * rows;
    const int64_t c1 = c0 + rows < C ? c0 + rows : C;
    double acc = 0.0;
    for (int64_t cb = c0; cb < c1; cb += kCtRows) {
        // the column loads of kCtRows rows are issued before any of them is used (bytes in flight, not one row at
        // a time); a row past the block's end repeats its last row with weight 0 and adds exactly +0.0
        double x[kCtRows];
#pragma unroll
        for (int j = 0; j < kCtRows; ++j) x[j] = ldg_stream1(X + (cb + j < c1 ? cb + j : c1 - 1) * pitchS + s);
#pragma unroll
        for (int j = 0; j < kCtRows; ++j) {
            const bool obs = !MASKED || !isnan(x[j]);
            const bool in = cb + j < c1 && obs;
            const double xj = obs ? x[j] : 0.0;
            const double* q = qF + (cb + j < c1 ? cb + j : c1 - 1) * 3;
            const double g0 = __ldg(q), g1 = __ldg(q + 1), g2 = __ldg(q + 2);   // straight-line code: no branch
            const double f0 = in ? g0 : 0.0, f1 = in ? g1 : 0.0, f2 = in ? g2 : 0.0;
            const double z0 = (xj - cc.mu[0]) * cc.isig[0], z1 = (xj - cc.mu[1]) * cc.isig[1],
                         z2 = (xj - cc.mu[2]) * cc.isig[2];
            const double l0 = fma(-0.5 * z0, z0, -cc.nc[0]), l1 = fma(-0.5 * z1, z1, -cc.nc[1]),
                         l2 = fma(-0.5 * z2, z2, -cc.nc[2]);
            acc += fma(f0, l0, fma(f1, l1, f2 * l2));
        }
    }
    part[rb * S + s] = acc;
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int64_t fcd_patient_terms_ws_bytes(int64_t C, int32_t U) {
    if (C < 0 || U < 0) return 0;
    return pt_row_blocks(C) * (int64_t)U * 2 * (int64_t)sizeof(double);
}

int fcd_patient_terms(const double* P, int64_t planeStride, const double* L, int64_t C, int32_t U, int64_t pitchU,
                      const double* qF, const uint8_t* fstate, const double* qR, const double* lqR, int32_t N,
                      const fcd_theta* theta_host, double* out4, double* ws, void* stream) {
    FCD_REQUIRE(P != nullptr && L != nullptr && qF != nullptr && fstate != nullptr && qR != nullptr && lqR != nullptr &&
                theta_host != nullptr && out4 != nullptr && ws != nullptr, "fcd_patient_terms: NULL argument");
    FCD_REQUIRE(N >= 2 && N < 65536 && C == (int64_t)N * (N - 1) / 2, "fcd_patient_terms: C=%lld is not N(N-1)/2 for N=%d",
                (long long)C, N);
    FCD_REQUIRE(U >= 1 && pitchU >= U && planeStride >= C * pitchU, "fcd_patient_terms: bad shape");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(qR) | reinterpret_cast<uintptr_t>(lqR) | reinterpret_cast<uintptr_t>(ws)) &
                 15) == 0, "fcd_patient_terms: qR, lqR and ws must be 16-byte aligned");
    const ThetaDev th = make_theta_dev(*theta_host, 0);
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(th.epsl, th.al, st, tab, true), "fcd_patient_terms: log table initialisation failed");
    const bool fast = log_table_covers(th.epsl, th.al);
    const int64_t nb = pt_row_blocks(C);
    const int64_t rows = (C + nb - 1) / nb;
    int lanesP = 1;
    while (lanesP < 32 && lanesP < U) lanesP *= 2;
    const int64_t warps = ((nb + 32 / lanesP - 1) / (32 / lanesP)) * ((U + lanesP - 1) / lanesP);
    const int64_t grid = (warps * 32 + kPtThreads - 1) / kPtThreads;
    FCD_REQUIRE(warps < ((int64_t)1 << 26), "fcd_patient_terms: %lld patients are too many for one launch", (long long)U);
    const size_t smem = fast ? tab.bytes() : 0;
    if (fast) {
        FCD_ALLOW_BIG_SMEM(patient_terms_rows_kernel<true>);
        patient_terms_rows_kernel<true><<<(unsigned)grid, kPtThreads, smem, st>>>(
            P, planeStride, L, C, U, pitchU, qF, fstate, qR, th, tab, nb, rows, lanesP, ws);
    } else {
        patient_terms_rows_kernel<false><<<(unsigned)grid, kPtThreads, 0, st>>>(
            P, planeStride, L, C, U, pitchU, qF, fstate, qR, th, tab, nb, rows, lanesP, ws);
    }
    int rc = check_launch("fcd_patient_terms(rows)");
    if (rc != 0) return rc;
    patient_terms_finish_kernel<<<(unsigned)((U + 31) / 32), kPtThreads, 0, st>>>(ws, nb, qR, lqR, N, U, th.log_pi2[0],
                                                                                th.log_pi2[1], out4);
    return check_launch("fcd_patient_terms(finish)");
}

int64_t fcd_connection_ws_bytes(int64_t C, int32_t U) {
    if (C < 0 || U < 0) return 0;
    return pt_row_blocks(C) * (int64_t)U * (int64_t)sizeof(double);
}

int fcd_connection_posteriors(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                              const double* qF, const uint8_t* fstate, const double* qR, int32_t N,
                              const fcd_theta* theta_host, double* qT, double* qFt, double* expected, double* rate,
                              double* ws, void* stream) {
    FCD_REQUIRE(P != nullptr && qF != nullptr && fstate != nullptr && qR != nullptr && theta_host != nullptr &&
                qT != nullptr && expected != nullptr && rate != nullptr && ws != nullptr,
                "fcd_connection_posteriors: NULL argument");
    FCD_REQUIRE(N >= 2 && N < 65536 && C == (int64_t)N * (N - 1) / 2,
                "fcd_connection_posteriors: C=%lld is not N(N-1)/2 for N=%d", (long long)C, N);
    FCD_REQUIRE(U >= 1 && pitchU >= U && planeStride >= C * pitchU, "fcd_connection_posteriors: bad shape");
    FCD_REQUIRE((reinterpret_cast<uintptr_t>(qR) & 15) == 0, "fcd_connection_posteriors: qR must be 16-byte aligned");
    const ThetaDev th = make_theta_dev(*theta_host, 0);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nb = pt_row_blocks(C);
    const int64_t rows = (C + nb - 1) / nb;
    int lanesP = 1;
    while (lanesP < 32 && lanesP < U) lanesP *= 2;
    const int64_t warps = ((nb + 32 / lanesP - 1) / (32 / lanesP)) * ((U + lanesP - 1) / lanesP);
    const int64_t grid = (warps * 32 + kPtThreads - 1) / kPtThreads;
    FCD_REQUIRE(warps < ((int64_t)1 << 26), "fcd_connection_posteriors: %lld patients are too many for one launch",
                (long long)U);
    if (qFt != nullptr)
        connection_rows_kernel<true><<<(unsigned)grid, kPtThreads, 0, st>>>(P, planeStride, C, U, pitchU, qF, fstate,
                                                                            qR, th, nb, rows, lanesP, qT, qFt, ws);
    else
        connection_rows_kernel<false><<<(unsigned)grid, kPtThreads, 0, st>>>(P, planeStride, C, U, pitchU, qF, fstate,
                                                                             qR, th, nb, rows, lanesP, qT, qFt, ws);
    int rc = check_launch("fcd_connection_posteriors(rows)");
    if (rc != 0) return rc;
    const int64_t bU = (U + 31) / 32, bC = (C + kPtThreads / 32 - 1) / (kPtThreads / 32);
    FCD_REQUIRE(bU + bC < ((int64_t)1 << 31), "fcd_connection_posteriors: too many edges for one launch");
    connection_finish_kernel<<<(unsigned)(bU + bC), kPtThreads, 0, st>>>(ws, nb, qT, C, U, (int)bU, expected, rate);
    return check_launch("fcd_connection_posteriors(finish)");
}

int64_t fcd_control_terms_ws_bytes(int64_t C, int32_t S) {
    if (C < 0 || S < 0) return 0;
    return pt_row_blocks(C) * (int64_t)S * (int64_t)sizeof(double);
}

int fcd_control_terms(const double* X, int64_t C, int32_t S, int64_t pitchS, const double* qF,
                      const fcd_theta* theta_host, double* out, double* ws, int32_t missing, void* stream) {
    FCD_REQUIRE(X != nullptr && qF != nullptr && theta_host != nullptr && out != nullptr && ws != nullptr,
                "fcd_control_terms: NULL argument");
    FCD_REQUIRE(missing == 0 || missing == 1, "fcd_control_terms: missing must be 0 or 1, got %d", missing);
    const int64_t N = (int64_t)((sqrt(8.0 * (double)C + 1.0) + 1.0) * 0.5);
    FCD_REQUIRE(C >= 1 && N * (N - 1) / 2 == C, "fcd_control_terms: C=%lld is not N(N-1)/2", (long long)C);
    FCD_REQUIRE(S >= 1 && pitchS >= S, "fcd_control_terms: bad shape");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(qF) | reinterpret_cast<uintptr_t>(out) |
                  reinterpret_cast<uintptr_t>(ws)) & 7) == 0,
                "fcd_control_terms: X, qF, out and ws must be 8-byte aligned");
    ControlConsts cc;
    for (int k = 0; k < 3; ++k) {
        cc.mu[k] = theta_host->mu[k];
        cc.isig[k] = 1.0 / theta_host->sigma[k];
        cc.nc[k] = log(theta_host->sigma[k]) + kHalfLog2Pi;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nb = pt_row_blocks(C);
    const int64_t rows = (C + nb - 1) / nb;
    int lanesP = 1;
    while (lanesP < 32 && lanesP < S) lanesP *= 2;
    const int64_t warps = ((nb + 32 / lanesP - 1) / (32 / lanesP)) * ((S + lanesP - 1) / lanesP);
    const int64_t grid = (warps * 32 + kPtThreads - 1) / kPtThreads;
    FCD_REQUIRE(warps < ((int64_t)1 << 26), "fcd_control_terms: %lld subjects are too many for one launch",
                (long long)S);
    if (missing)
        control_terms_rows_kernel<true><<<(unsigned)grid, kPtThreads, 0, st>>>(X, C, S, pitchS, qF, cc, nb, rows, lanesP,
                                                                               ws);
    else
        control_terms_rows_kernel<false><<<(unsigned)grid, kPtThreads, 0, st>>>(X, C, S, pitchS, qF, cc, nb, rows, lanesP,
                                                                                ws);
    int rc = check_launch("fcd_control_terms(rows)");
    if (rc != 0) return rc;
    connection_finish_kernel<<<(unsigned)((S + 31) / 32), kPtThreads, 0, st>>>(ws, nb, nullptr, C, S,
                                                                              (int)((S + 31) / 32), out, nullptr);
    return check_launch("fcd_control_terms(finish)");
}

int fcd_qR_change(const double* qR_old, const double* qR_new, int32_t N, int32_t U, double* maxU, double* out1,
                  void* stream) {
    FCD_REQUIRE(qR_old != nullptr && qR_new != nullptr && out1 != nullptr, "fcd_qR_change: NULL argument");
    FCD_REQUIRE(N >= 1 && U >= 1, "fcd_qR_change: bad shape");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(qR_old) | reinterpret_cast<uintptr_t>(qR_new)) & 15) == 0 &&
                (reinterpret_cast<uintptr_t>(out1) & 7) == 0, "fcd_qR_change: qR arrays must be 16-byte aligned");
    qR_change_kernel<<<(unsigned)((U + 31) / 32), kChThreads, 0, (cudaStream_t)stream>>>(qR_old, qR_new, N, U, maxU, out1);
    return check_launch("fcd_qR_change");
}

}  // extern "C"
