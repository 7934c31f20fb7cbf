// E-step kernels: healthy sufficient statistics, responsibility planes, peak
// states, K2 (template posterior q_F), K2b (region-weight tensor W and the
// Gauss-Seidel sweep for q_R).
#include <cstring>

#include <type_traits>

#include "fcd_common.cuh"
#include "fcd_solver.cuh"

namespace fcd {

constexpr int kEdgeThreads = 256;       // 8 warps, one edge row per warp at a time

// ------------------------------------------------------------------ c_to_nm
__global__ void c_to_nm_kernel(int64_t c0, int64_t C, int32_t* n_out, int32_t* m_out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < C;
         i += (int64_t)gridDim.x * blockDim.x) {
        int n, m;
        c_to_nm(c0 + i, n, m);
        n_out[i] = n;
        m_out[i] = m;
    }
}

__global__ void edge_table_kernel(int64_t c0, int64_t C, int32_t* __restrict__ nm) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < C;
         i += (int64_t)gridDim.x * blockDim.x) {
        int n, m;
        c_to_nm(c0 + i, n, m);
        nm[i] = n | (m << 16);
    }
}

// ------------------------------------------------------------ healthy stats
// S1[c] = sum_h b[c,h], S2[c] = sum_h b[c,h]^2.  One warp per edge row,
// coalesced 64-bit loads along the subject axis.  MASKED: NaN entries are not
// observed and left out; S0[c] counts the observed ones (same sums, same order
// as the unmasked form when nothing is missing).
template <bool MASKED>
__global__ void __launch_bounds__(kEdgeThreads)
healthy_stats_kernel(const double* __restrict__ b, int64_t C, int H, int64_t pitchH,
                     double* __restrict__ S1, double* __restrict__ S2, double* __restrict__ S0) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = warp0; c < C; c += nwarps) {
        const double* row = b + c * pitchH;
        double s1 = 0.0, s2 = 0.0, s0 = 0.0;
        for (int h = lane; h < H; h += 32) {
            double x = ldg_stream1(row + h);
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

// ------------------------------------------------------ responsibility planes
// P0 / P1 / P2 / L planes (see fcd_common.cuh) from the patient correlations; the
// only place where exponentials of the data are taken.  Elementwise over the
// padded [C][pitchU] rows (padding columns are written as zeros).
// MASKED: a NaN entry is not observed and gets p_k = 1/3, L = log 3, so that
// log M_kl = L + log(a_l + b_l / 3) = 0 for every (k, l) and theta: the element
// drops out of every later pass, which read it through the planes only.
template <bool MASKED>
__global__ void __launch_bounds__(256)
resp_cache_kernel(const double* __restrict__ bt, int64_t C, int U, int64_t pitchU,
                  const __grid_constant__ ThetaDev th,
                  double* __restrict__ P, int64_t planeStride, double* __restrict__ L) {
    const int64_t total = C * pitchU;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int u = (int)(i % pitchU);
        Resp r;
        r.p[0] = r.p[1] = r.p[2] = r.L = 0.0;
        if (u < U) {
            const double x = ldg_stream1(bt + i);
            if (MASKED && isnan(x)) {
                r.p[0] = r.p[1] = r.p[2] = 1.0 / 3.0;
                r.L = 1.0986122886681098;                    // log 3
            } else {
                r = resp_eval(x, th);
            }
        }
        P[i] = r.p[0];
        P[planeStride + i] = r.p[1];
        P[2 * planeStride + i] = r.p[2];
        if (L) L[i] = r.L;
    }
}

// ------------------------------------------------------------- peak states
// fstate[c] / rstate[n][u] of fcd_common.cuh from the probabilities.
__global__ void __launch_bounds__(256)
peak_states_F_kernel(const double* __restrict__ qF, int64_t C, uint8_t* __restrict__ fstate) {
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < C;
         c += (int64_t)gridDim.x * blockDim.x) {
        const double q0 = qF[c * 3], q1 = qF[c * 3 + 1], q2 = qF[c * 3 + 2];
        int s = kStateMixedF;
        if (q0 == 1.0 && q1 <= kPeakTau && q2 <= kPeakTau) s = 0;
        else if (q1 == 1.0 && q0 <= kPeakTau && q2 <= kPeakTau) s = 1;
        else if (q2 == 1.0 && q0 <= kPeakTau && q1 <= kPeakTau) s = 2;
        fstate[c] = (uint8_t)s;
    }
}

__global__ void __launch_bounds__(256)
peak_states_R_kernel(const double* __restrict__ qR, int N, int U, int64_t pitchS, uint8_t* __restrict__ rstate) {
    const int64_t total = (int64_t)N * pitchS;
    const double2* q2 = reinterpret_cast<const double2*>(qR);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = i / pitchS;
        const int u = (int)(i - n * pitchS);
        int s = kStateDead;
        if (u < U) {
            const double2 q = q2[n * U + u];
            // mixed; "loose" if the pair is not normalised (the one-weight form of a half record needs q_0 + q_1 = 1)
            s = fabs((q.x + q.y) - 1.0) <= 8.881784197001252e-16 ? kStateMixedR : kStateLooseR;
            if (q.x == 1.0 && q.y <= kPeakTau) s = 0;
            else if (q.y == 1.0 && q.x <= kPeakTau) s = 1;
        }
        rstate[i] = (uint8_t)s;
    }
}

// ---------------------------------------------------------------- MAP labels
// labels[i] = argmax_k lq[i][k] (first maximum on ties, like numpy.argmax): the MAP
// template state of an edge (width 3) or the MAP anomaly flag of a (region,
// patient) pair (width 2) -- what the cited evaluation reads off the posteriors
// (doc/methods.rst:241-246).
__global__ void __launch_bounds__(256)
map_labels_kernel(const double* __restrict__ lq, int64_t n, int width, uint8_t* __restrict__ labels) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double* v = lq + i * width;
        int best = 0;
        double bv = v[0];
        for (int k = 1; k < width; ++k)
            if (v[k] > bv) {
                bv = v[k];
                best = k;
            }
        labels[i] = (uint8_t)best;
    }
}

// ------------------------------------------------------------------- K2
// lqF[c,k] = log gamma_k + healthy_k(S1,S2) + sum_u sum_l w_l log M_kl(bt[c,u])
//            - logsumexp_k                                 (fcdiff/fit.py:157-174)
// The per-(c,u) term L * sum_l w_l is common to the three states k and cancels in
// the normalisation, so it is never formed.  T1: both regions of the element
// peaked -> the three logs of l*; deferred: all nine with the real pair weights.

constexpr int kK2Seg = 128;

template <bool FAST, bool MASKED>
__global__ void __launch_bounds__(kStreamThreads, 1)
estep_qF_kernel(const double* __restrict__ S1, const double* __restrict__ S2, const double* __restrict__ S0,
                const double* __restrict__ P, int64_t planeStride,
                int64_t C, int U, int64_t pitchU,
                const double* __restrict__ qR, const uint8_t* __restrict__ rstate, int64_t pitchS,
                const int32_t* __restrict__ nm,
                const __grid_constant__ ThetaDev th, const __grid_constant__ LogTabWindow tab, int depth,
                double* __restrict__ lqF, double* __restrict__ qF) {
    extern __shared__ __align__(128) double s_dyn[];
    const double* s_tab = load_log_table<FAST>(tab, s_dyn);
    unsigned char* s_stream = reinterpret_cast<unsigned char*>(s_dyn + (FAST ? ((tab.n + 1) & ~1) : 0));
    const int lane = threadIdx.x & 31;
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    double acc[3] = {0.0, 0.0, 0.0};
    // per-l constants {a_l, b_l} of the T1 body; row 3 is neutral: log(1 + 0 p) = 0 exactly
    __shared__ double2 s_lc[4];
    if (threadIdx.x < 4) s_lc[threadIdx.x] = threadIdx.x < 3 ? make_double2(th.al[threadIdx.x], th.bl[threadIdx.x])
                                                             : make_double2(1.0, 0.0);
    __syncthreads();
    double acc1[3] = {0.0, 0.0, 0.0};
    // FAST: the T1 logs have weight exactly 1, so each lane keeps running PRODUCTS of the mixture
    // weights (two sets of three, fcd_math.cuh "Sum of logs as the log of a product") and takes
    // three logarithms per row (or per kProdMax chunks of a long row) instead of three per element.
    double pr[2][3] = {{1.0, 1.0, 1.0}, {1.0, 1.0, 1.0}};
    int nf = 0;
    auto flush = [&]() {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            acc[i] += log_pos<FAST>(pr[0][i] * pr[1][i], s_tab);
            pr[0][i] = pr[1][i] = 1.0;
        }
        nf = 0;
    };
    // planes 0 and 1 are streamed; p_2 = 1 - p_0 - p_1 (absolute error 1e-16 on an argument
    // a_l + b_l p >= min(a_l, eps_l): below the rounding of the log)
    auto live = [&](const double (&pv)[2], int lp, int e) {
        const double2 k = s_lc[lp];
        const double p3[3] = {pv[0], pv[1], (1.0 - pv[0]) - pv[1]};
        if (FAST) {
#pragma unroll
            for (int i = 0; i < 3; ++i) pr[e][i] *= fma(k.y, p3[i], k.x);
            if (e == 1 && ++nf == kProdMax) flush();              // warp-uniform
        } else {
#pragma unroll
            for (int i = 0; i < 3; ++i) (e ? acc1 : acc)[i] += fast_log<FAST>(fma(k.y, p3[i], k.x), s_tab);
        }
    };
    struct Ops {
        double p[3];
        double2 qn, qm;
    };
    auto dload = [&](int64_t c, int u, int n, int m, int, bool ok) {
        Ops o;
        o.p[0] = o.p[1] = o.p[2] = 0.0;
        o.qn = o.qm = make_double2(0.0, 0.0);
        if (ok) {
            o.qn = __ldg(qR2 + (int64_t)n * U + u);
            o.qm = __ldg(qR2 + (int64_t)m * U + u);
            o.p[0] = ldg_stream1(P + c * pitchU + u);
            o.p[1] = ldg_stream1(P + planeStride + c * pitchU + u);
            o.p[2] = (1.0 - o.p[0]) - o.p[1];
        }
        return o;
    };
    auto dcompute = [&](const Ops& o) {
        double w[3];
        pair_weights(o.qn, o.qm, w);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double a = acc[k];
#pragma unroll
            for (int l = 0; l < 3; ++l) a = fma(w[l], fast_log<FAST>(mix_rel(th, l, o.p[k]), s_tab), a);
            acc[k] = a;
        }
    };
    // Row ends: the warp sums are parked in the registers of lane (row mod 32); every 32 rows (and
    // after the last one) all lanes finish their own row at once -- the normalisation's exp / log
    // would otherwise occupy the warp's issue slots for ONE active lane per row.
    double keep[3] = {0.0, 0.0, 0.0};
    int64_t keep_c = -1;
    int rows_done = 0;
    auto finish_rows = [&]() {
        if (keep_c >= 0)
            k2_finish<MASKED>(keep_c, keep, __ldg(S1 + keep_c), __ldg(S2 + keep_c), MASKED ? __ldg(S0 + keep_c) : 0.0,
                              th, lqF, qF);
        keep_c = -1;
    };
    auto row_end = [&](int64_t c) {
        if (FAST && nf > 0) flush();
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] = warp_sum(acc[k] + acc1[k]);
        if (lane == (rows_done & 31)) {
            keep[0] = acc[0];
            keep[1] = acc[1];
            keep[2] = acc[2];
            keep_c = c;
        }
        if ((++rows_done & 31) == 0) finish_rows();
        acc[0] = acc[1] = acc[2] = 0.0;
        acc1[0] = acc1[1] = acc1[2] = 0.0;
    };
    stream_tiered<2, kK2Seg, kStreamWarps, true, false>(P, planeStride, C, U, pitchU, nullptr, rstate, pitchS, nm,
                                                        s_stream, depth, live, dload, dcompute,
                                                        [](int64_t, int, int, int, int) {}, row_end);
    finish_rows();
}

// ------------------------------------------------------------------- K2 (coded)
// The same E-step from the code plane the previous M-step left behind (fcd_streams.cu): between
// that code pass and this E-step q_R has not changed, so code[c][u] still says which pair state l*
// a peaked element has (one byte -> the constants of a running product, no peak-state decoding, no
// queue) and the row's key list names the elements with a mixed region (evaluated densely after
// the row, nine logs each with the real pair weights).  One persistent CTA of 16 warps per SM, warp
// per row; per 128-patient segment three bulk copies (p_0, p_1, codes) into the warp's private ring.
constexpr int kK2cSeg = 256;
constexpr int kK2cStage = 2 * kK2cSeg * 8 + kK2cSeg;          // bytes: p_0, p_1, codes
constexpr int kK2cMaxDepth = 5;
constexpr size_t k2c_ring_bytes(int depth, int nw) { return (size_t)nw * depth * (kK2cStage + 8); }

template <bool FAST, int NW, bool MASKED>
__global__ void __launch_bounds__(NW * 32, 1)
estep_qF_coded_kernel(const double* __restrict__ S1, const double* __restrict__ S2, const double* __restrict__ S0,
                      const double* __restrict__ P, int64_t planeStride, int64_t C, int U, int64_t pitchU,
                      const double* __restrict__ qR, const int32_t* __restrict__ nm,
                      const uint8_t* __restrict__ code, int64_t pitchQ, const int2* __restrict__ counts,
                      const unsigned long long* __restrict__ keysF, const unsigned long long* __restrict__ keysH,
                      const longlong2* __restrict__ rowoff, const double2* __restrict__ Hh,
                      const __grid_constant__ ThetaDev th, const SolverState* __restrict__ solved,
                      const __grid_constant__ LogTabWindow tab, int depth,
                      double* __restrict__ lqF, double* __restrict__ qF) {
    extern __shared__ __align__(128) double s_dyn[];
    __shared__ double2 s_lc[8];
    __shared__ uint64_t s_tabbar;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // the logarithm table first: one bulk copy at the head of this SM's queue (loaded by every thread
    // after the ring fills, it waited behind ~200 KB of them: 5 % of the kernel's stall samples)
    if (threadIdx.x == 0) {
        mbar_init(&s_tabbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        issue_log_table<FAST>(tab, s_dyn, &s_tabbar);
    }
    unsigned char* ring0 = reinterpret_cast<unsigned char*>(s_dyn + (FAST ? ((tab.n + 15) & ~15) : 0));
    unsigned char* ring = ring0 + (size_t)warp * depth * kK2cStage;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring0 + (size_t)NW * depth * kK2cStage) + warp * depth;
    // the ring starts zeroed: lanes beyond the copied bytes of a short segment read stale but finite
    // responsibilities (their code is forced to 3)
    for (int i = lane; i < depth * kK2cStage / 16; i += 32) reinterpret_cast<int4*>(ring)[i] = make_int4(0, 0, 0, 0);
    if (lane < depth) mbar_init(bars + lane, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    // per-code constants {a_l, b_l}; code 3 is neutral: the factor 1 + 0 p = 1 exactly; the codes 4, 5
    // (one undecided region) count as l = 2 here, their correction comes from the half records
    // `solved` != NULL: (eta, epsilon) are the ones the device-resident solve enqueued before this launch
    // left in its state block (the host does not know them yet: the E-step of the NEXT iteration runs
    // while the host waits for that solve, fcdiff_b200/fit.py: _speculative_estep)
    if (threadIdx.x < 8) {
        const int l = threadIdx.x >= 4 ? 2 : threadIdx.x;
        double2 ab = make_double2(1.0, 0.0);
        if (l < 3) {
            if (solved != nullptr) {
                // make_theta_dev's arithmetic (fcd_runtime.cu) operation by operation, no contraction: the
                // launch is bit-identical to the one the host would make after reading the solution
                const double eta = solved->x[0], eps = solved->x[1];
                const double e = l == 0 ? __dadd_rn(1.0, -eps)
                               : l == 1 ? eps
                               : __dadd_rn(__dmul_rn(eta, eps), __dmul_rn(__dadd_rn(1.0, -eta), __dadd_rn(1.0, -eps)));
                const double a = __dmul_rn(__dadd_rn(1.0, -e), 0.5);
                ab = make_double2(a, __dadd_rn(e, -a));
            } else {
                ab = make_double2(th.al[l], th.bl[l]);
            }
        }
        s_lc[threadIdx.x] = ab;
    }
    __syncwarp();

    const int nseg = (int)((pitchU + kK2cSeg - 1) / kK2cSeg);
    const int64_t W = (int64_t)gridDim.x * NW;
    // consecutive rows go to different SMs: the rows of one region are consecutive, and a region that is
    // undecided for many patients makes ALL its rows expensive (half records); at config 3 the launch
    // times are the same as with 16 consecutive rows per CTA
    const int64_t c_first = (int64_t)warp * gridDim.x + blockIdx.x;
    const uint32_t ring_s = smem_u32(ring), bars_s = smem_u32(bars);
    // Issue side: running global pointers (lane 0), segment sizes known in advance -- a segment is a
    // full 128 patients except the row's last one.
    const uint32_t np_last = (uint32_t)(pitchU - (int64_t)(nseg - 1) * kK2cSeg);        // even, 2 .. 128
    const uint32_t cb_last = (np_last + 15) & ~15u;                                      // pitchQ % 16 == 0
    const int64_t skipP = W * pitchU - (int64_t)(nseg - 1) * kK2cSeg, skipC = W * pitchQ - (int64_t)(nseg - 1) * kK2cSeg;
    const double* gp = P + c_first * pitchU;                 // next segment of plane 0 (meaningful in lane 0)
    const uint8_t* gc = code + c_first * pitchQ;
    int rows_to_issue = c_first < C ? (int)((C - c_first + W - 1) / W) : 0;
    int ps = 0, pd = 0;
    auto issue = [&]() {
        if (rows_to_issue <= 0) return;
        const bool last = ps == nseg - 1;
        if (lane == 0) {
            const uint32_t np = last ? np_last : (uint32_t)kK2cSeg, cb = last ? cb_last : (uint32_t)kK2cSeg;
            const uint32_t st = ring_s + pd * kK2cStage, bar = bars_s + pd * 8;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(16 * np + cb) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(st), "l"(gp), "r"(np * 8), "r"(bar) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(st + kK2cSeg * 8), "l"(gp + planeStride), "r"(np * 8), "r"(bar) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(st + 2 * kK2cSeg * 8), "l"(gc), "r"(cb), "r"(bar) : "memory");
            gp += last ? skipP : (int64_t)kK2cSeg;
            gc += last ? skipC : (int64_t)kK2cSeg;
        }
        pd = pd + 1 == depth ? 0 : pd + 1;
        if (last) {
            ps = 0;
            --rows_to_issue;
        } else {
            ++ps;
        }
    };
#pragma unroll 1
    for (int i = 0; i < depth; ++i) issue();
    const double* s_tab = s_dyn - tab.lo;
    __syncthreads();                                         // s_tabbar initialised
    if (FAST) mbar_wait(&s_tabbar, 0);

    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    double acc[3] = {0.0, 0.0, 0.0};
    double pr[2][3] = {{1.0, 1.0, 1.0}, {1.0, 1.0, 1.0}};
    int nf = 0;
    auto flush = [&]() {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            if (FAST) acc[i] += log_pos<FAST>(pr[0][i] * pr[1][i], s_tab);
            pr[0][i] = pr[1][i] = 1.0;
        }
        nf = 0;
    };
    // an element with real pair weights: nine logs (fit.py:165-171 with fit.py:382-406)
    auto weighted = [&](int64_t c, int u, int n, int m) {
        const double2 qn = __ldg(qR2 + (int64_t)n * U + u), qm = __ldg(qR2 + (int64_t)m * U + u);
        const double p0 = __ldg(P + c * pitchU + u), p1 = __ldg(P + planeStride + c * pitchU + u);
        const double p3[3] = {p0, p1, (1.0 - p0) - p1};
        double w[3];
        pair_weights(qn, qm, w);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double a = acc[k];
#pragma unroll
            for (int l = 0; l < 3; ++l) a = fma(w[l], fast_log<FAST>(fma(s_lc[l].y, p3[k], s_lc[l].x), s_tab), a);
            acc[k] = a;
        }
    };
    // an element with one undecided region: q (log M_s - log M_2) per template state (half record {p*, +-q})
    auto half_p = [&](double p0, double p1, bool sx, double q) {
        const double p3[3] = {p0, p1, (1.0 - p0) - p1};
        const double2 x = s_lc[sx ? 1 : 0], z = s_lc[2];
#pragma unroll
        for (int k = 0; k < 3; ++k)
            acc[k] = fma(q, fast_log<FAST>(fma(x.y, p3[k], x.x), s_tab) - fast_log<FAST>(fma(z.y, p3[k], z.x), s_tab), acc[k]);
    };
    auto half = [&](int64_t c, int u, bool sx, double q) {
        half_p(__ldg(P + c * pitchU + u), __ldg(P + planeStride + c * pitchU + u), sx, q);
    };
    double keep[3] = {0.0, 0.0, 0.0};                        // row ends: see estep_qF_kernel
    int64_t keep_c = -1;
    int rows_done = 0;
    auto finish_rows = [&]() {
        if (keep_c >= 0)
            k2_finish<MASKED>(keep_c, keep, __ldg(S1 + keep_c), __ldg(S2 + keep_c), MASKED ? __ldg(S0 + keep_c) : 0.0,
                              th, lqF, qF);
        keep_c = -1;
    };
    // The half records of a row are taken off the critical path (they used to be a chain of dependent
    // gathers after the row's stream: counts -> rowoff -> key -> p_0, p_1): the row's counts / offsets
    // are requested one row ahead; at the start of a row every lane requests the key and the weight of
    // the row's half records lane and lane + 32 (the common case: ~50 per row of 500 patients); while the
    // segments stream through the ring, a lane whose record lies in the resident segment copies its
    // p_0, p_1 from the STAGE (shared memory: no gather at all); after the row the 2 x 32 records are
    // evaluated densely.  Records beyond 64 per row and full records (rare) keep the gather path.
    int2 nxt_cnt = make_int2(0, 0);
    longlong2 nxt_ro = make_longlong2(0, 0);
    if (c_first < C) {
        nxt_cnt = __ldg(counts + c_first);
        if (nxt_cnt.x != 3 * U && (nxt_cnt.x > 0 || nxt_cnt.y > 0)) nxt_ro = __ldg(rowoff + c_first);
    }
    int d = 0;
    uint32_t phase = 0;
    for (int64_t c = c_first; c < C; c += W) {
        const int2 cnt = nxt_cnt;
        const longlong2 ro = nxt_ro;
        const bool listed = cnt.x != 3 * U && (cnt.x > 0 || cnt.y > 0);
        // (the key is not touched before the first segment has been consumed: its latency hides there)
        bool hv[2];
        uint32_t hkey[2] = {0u, 0u};
        double hq[2] = {0.0, 0.0}, hp0[2] = {0.0, 0.0}, hp1[2] = {0.0, 0.0};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int i = lane + 32 * k;
            hv[k] = listed && i < cnt.y;
            if (hv[k]) {
                hkey[k] = __ldg(reinterpret_cast<const uint32_t*>(keysH + ro.y + i));      // low word: u in bits 0-15
                hq[k] = __ldg(Hh + ro.y + i).y;
            }
        }
        if (c + W < C) {                                     // the next row's counts / offsets: in flight during this row
            nxt_cnt = __ldg(counts + c + W);
            nxt_ro = __ldg(rowoff + c + W);                  // (garbage for rows without records: not used then)
        }
        // two elements of the stage per lane: running products of the three template states' factors
        auto pair = [&](const unsigned char* st, int j, uint32_t c2) {
            const double2 a0 = *reinterpret_cast<const double2*>(st + (64 * j + 2 * lane) * 8);
            const double2 a1 = *reinterpret_cast<const double2*>(st + kK2cSeg * 8 + (64 * j + 2 * lane) * 8);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const double2 k = s_lc[(c2 >> (8 * e)) & 0xff];
                const double p0 = e ? a0.y : a0.x, p1 = e ? a1.y : a1.x;
                const double p3[3] = {p0, p1, (1.0 - p0) - p1};
                if (FAST) {
#pragma unroll
                    for (int i = 0; i < 3; ++i) pr[e][i] *= fma(k.y, p3[i], k.x);
                } else {
#pragma unroll
                    for (int i = 0; i < 3; ++i) acc[i] += log(fma(k.y, p3[i], k.x));
                }
            }
        };
        for (int s = 0; s < nseg; ++s) {
            mbar_wait(bars + d, phase);
            const unsigned char* st = ring + d * kK2cStage;
            const unsigned short* cs = reinterpret_cast<const unsigned short*>(st + 2 * kK2cSeg * 8) + lane;
            if (s < nseg - 1 || np_last > (uint32_t)(kK2cSeg - 64)) {
                // every pair of the stage has elements (warp-uniform): one straight-line block, no flush
                // inside; beyond the row's end the stage holds stale (finite) responsibilities and the code
                // is forced to 3 (the row's last segment used to take the bounded path below, a branch and
                // a flush test per pair: half of all segments at 500 patients)
                const int lim = s < nseg - 1 ? kK2cSeg : (int)np_last;
                if (nf + kK2cSeg / 64 > kProdMax) flush();
#pragma unroll
                for (int j = 0; j < kK2cSeg / 64; ++j)
                    pair(st, j, 64 * j + 2 * lane < lim ? (uint32_t)cs[32 * j] : 0x0303u);
                nf += kK2cSeg / 64;
            } else {
#pragma unroll
                for (int j = 0; j < kK2cSeg / 64; ++j) {
                    if (64 * j < (int)np_last) {                        // warp-uniform
                        // beyond pitchU the stage holds stale (finite) responsibilities: force their code to 3
                        pair(st, j, 64 * j + 2 * lane < (int)np_last ? (uint32_t)cs[32 * j] : 0x0303u);
                        if (++nf == kProdMax) flush();
                    }
                }
            }
            // my half records that lie in this segment: p_0, p_1 straight from the stage
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                if (hv[k]) {
                    const uint32_t o = (hkey[k] & 0xffffu) - (uint32_t)(s * kK2cSeg);
                    if (o < (uint32_t)kK2cSeg) {
                        hp0[k] = *reinterpret_cast<const double*>(st + o * 8);
                        hp1[k] = *reinterpret_cast<const double*>(st + kK2cSeg * 8 + o * 8);
                    }
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
        // the row's elements with real weights
        if (cnt.x == 3 * U) {                                // the edge was unpeaked at the code pass: every element
            const int v = __ldg(nm + c);
            const int n = v & 0xffff, m = (v >> 16) & 0xffff;
            for (int u = lane; u < U; u += 32) weighted(c, u, n, m);
        } else if (listed) {
            if (cnt.x > 0) {
                const int v = __ldg(nm + c);
                const int n = v & 0xffff, m = (v >> 16) & 0xffff;
                const unsigned long long* kf = keysF + ro.x;
                for (int i = lane; i < cnt.x; i += 32) weighted(c, (int)(__ldg(kf + i) & 0xffffull), n, m);
            }
#pragma unroll
            for (int k = 0; k < 2; ++k)
                if (32 * k < cnt.y && hv[k])                 // first condition warp-uniform
                    half_p(hp0[k], hp1[k], __double2hiint(hq[k]) < 0, fabs(hq[k]));
            const unsigned long long* kh = keysH + ro.y;
            const double2* hr = Hh + ro.y;
            for (int i = 64 + lane; i < cnt.y; i += 32) {
                const double qs = __ldg(hr + i).y;
                half(c, (int)(__ldg(kh + i) & 0xffffull), __double2hiint(qs) < 0, fabs(qs));
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) acc[k] = warp_sum(acc[k]);
        if (lane == (rows_done & 31)) {
            keep[0] = acc[0];
            keep[1] = acc[1];
            keep[2] = acc[2];
            keep_c = c;
        }
        if ((++rows_done & 31) == 0) finish_rows();
        acc[0] = acc[1] = acc[2] = 0.0;
    }
    finish_rows();
}

// ------------------------------------------------------------------- K2b/P*
// PsT[u][c] = Pe[k*(c)][c][u0 + u]: the patient-major plane of each edge's dominant state, gathered straight from
// the E-step's EDGE-major planes by one transposing pass over the dominant-state rows.  q_F settles after the first
// iteration, so the plane is gathered once and afterwards only the columns of edges whose state changed are
// refreshed (kcache[c] = the state PsT[.][c] was gathered for; 255 = never).  The column of an unpeaked edge is
// marked with a negative "responsibility": region_weights_kernel reads nothing but this plane per element and takes
// the three-plane path for it.  One CTA per 32 edges: it leaves at once when none of its columns changed state (the
// usual launch), otherwise walks the patients in 32 x 32 tiles through padded shared memory -- reads coalesced
// along u, writes along c; columns that did not change are neither read nor written.
__global__ void __launch_bounds__(256)
pstar_refresh_em_kernel(const double* __restrict__ Pe, int64_t planeStride, int64_t pitchU, int u0, int Ul, int64_t C,
                        int64_t pitchC, const uint8_t* __restrict__ fstate, const uint8_t* __restrict__ kcache,
                        double* __restrict__ PsT) {
    __shared__ double tile[32][33];
    __shared__ int s_k[32];
    __shared__ int s_any;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // 32 x 8
    const int64_t cb = (int64_t)blockIdx.x * 32;
    if (threadIdx.x == 0) s_any = 0;
    __syncthreads();
    if (threadIdx.x < 32) {
        const int64_t c = cb + threadIdx.x;
        int k = -1;                                               // -1: unchanged or beyond C
        if (c < C) {
            const int f = fstate[c];
            const int kk = f >= 3 ? 3 : f;
            if (kk != kcache[c]) k = kk;
        }
        s_k[threadIdx.x] = k;
        if (k >= 0) s_any = 1;
    }
    __syncthreads();
    if (!s_any) return;
    for (int ub = 0; ub < Ul; ub += 32) {
#pragma unroll
        for (int j = 0; j < 32; j += 8) {                         // tile[c][u]: coalesced along u
            const int k = s_k[ty + j];
            const int u = ub + tx;
            double v = -1.0;                                      // unpeaked edge: the negative mark
            if (k >= 0 && k < 3 && u < Ul) v = ldg_stream1(Pe + (int64_t)k * planeStride + (cb + ty + j) * pitchU + u0 + u);
            tile[ty + j][tx] = v;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
            const int u = ub + ty + j;
            if (s_k[tx] >= 0 && u < Ul) PsT[(int64_t)u * pitchC + cb + tx] = tile[tx][ty + j];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
pstar_commit_kernel(const uint8_t* __restrict__ fstate, int64_t C, uint8_t* __restrict__ kcache) {
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c < C) kcache[c] = fstate[c] < 3 ? fstate[c] : 3;
}

// ------------------------------------------------------------------- K2b/W
// W_l[c,u] = sum_k qF[c,k] log(a_l + b_l p_k(c,u)) from the responsibility
// planes (see fcd_region_weights_em for the strides).  The omitted per-(c,u) constant L sum_k qF[c,k]
// is the same for l = 0, 1, 2 and enters both states of fcdiff/fit.py:190,194
// multiplied by (q_R[m,u,0] + q_R[m,u,1]), so it cancels at fit.py:196.
// Only the DIFFERENCE of the two region states' sums survives the normalisation of
// fit.py:196-197 (lq = l - logsumexp(l) is a function of l_0 - l_1), and
//   l_0 - l_1 = log(pi_0 / pi_1) + sum_m q_R[m,0] (W_0 - W_2) + q_R[m,1] (W_2 - W_1),
// so the tensor holds two numbers per edge-patient: WT[u][c] = {W_0 - W_2, W_2 - W_1}
// (16 bytes written here and read by the sweep instead of 24).
// Edges whose q_F is peaked (fstate < 3) need the plane of k* only: 3 logs.
template <bool FAST>
__global__ void __launch_bounds__(256)
region_weights_kernel(const double* __restrict__ PT, int64_t planeStride, int64_t strideU, int64_t strideC,
                      int Ul, int64_t C, int64_t pitchC,
                      const double* __restrict__ qF, const uint8_t* __restrict__ fstate,
                      const double* __restrict__ PsT,
                      const __grid_constant__ ThetaDev th, const __grid_constant__ LogTabWindow tab,
                      double* __restrict__ WT) {
    extern __shared__ __align__(16) double s_dyn[];
    const double* s_tab = load_log_table<FAST>(tab, s_dyn);
    // persistent CTAs over (patient, 1024-edge tile) work items: no wave tail, one table load per
    // CTA.  The kernel is bound by load latency, so (a) with the dominant-state plane ONE load per element
    // says everything: the responsibility of a peaked edge, or the negative mark of an unpeaked one
    // (pstar_refresh_em_kernel) -- no state byte is fetched; and (b) the loads of the CTA's next tile are in
    // flight while the logs of the current one are taken.  Tile indices are 32-bit (the host checks the
    // count): no 64-bit division per tile.
    const unsigned tiles_per_row = (unsigned)((C + 1023) / 1024);
    const unsigned ntiles = tiles_per_row * (unsigned)Ul;
    struct Tile {
        double pk[4];
        int ks[4];
    };
    auto load = [&](unsigned t) {
        Tile tl;
        const unsigned u = t / tiles_per_row;
        const int64_t cbase = (int64_t)(t - u * tiles_per_row) * 1024;
        const double* row = PT + (int64_t)u * strideU;        // element (k, u, c): PT[k planeStride + u strideU + c strideC]
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t c = cbase + threadIdx.x + 256 * j;
            tl.pk[j] = 0.0;
            tl.ks[j] = -1;
            if (t < ntiles && c < C) {
                if (PsT) {
                    tl.pk[j] = ldg_stream1(PsT + (int64_t)u * pitchC + c);
                    tl.ks[j] = 0;                             // (peaked or not: read off pk when it is used)
                } else {
                    tl.ks[j] = __ldg(fstate + c);
                    if (tl.ks[j] < 3) tl.pk[j] = ldg_stream1(row + tl.ks[j] * planeStride + c * strideC);
                }
            }
        }
        return tl;
    };
    // two tiles ahead: a thread has the loads of eight elements in flight while it takes the logs of four
    // (three ahead was measured: registers spill, 0.240 ms against 0.223)
    Tile cur = load(blockIdx.x), nxt = load(blockIdx.x + gridDim.x);
    for (unsigned t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const Tile nxt2 = load(t + 2 * gridDim.x);
        const unsigned u = t / tiles_per_row;
        const int64_t cbase = (int64_t)(t - u * tiles_per_row) * 1024;
        const double* row = PT + (int64_t)u * strideU;
        double2* out = reinterpret_cast<double2*>(WT) + (int64_t)u * C;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t c = cbase + threadIdx.x + 256 * j;
            if (cur.ks[j] < 0) continue;
            double w[3];
            if (PsT ? cur.pk[j] >= 0.0 : cur.ks[j] < 3) {
#pragma unroll
                for (int l = 0; l < 3; ++l) w[l] = fast_log<FAST>(mix_rel(th, l, cur.pk[j]), s_tab);
            } else {
                const double q[3] = {__ldg(qF + c * 3), __ldg(qF + c * 3 + 1), __ldg(qF + c * 3 + 2)};
                w[0] = w[1] = w[2] = 0.0;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double p = ldg_stream1(row + k * planeStride + c * strideC);
#pragma unroll
                    for (int l = 0; l < 3; ++l) w[l] = fma(q[k], fast_log<FAST>(mix_rel(th, l, p), s_tab), w[l]);
                }
            }
            out[c] = make_double2(w[0] - w[2], w[2] - w[1]);
        }
        cur = nxt;
        nxt = nxt2;
    }
}

// --------------------------------------------------------------- K2b/sweep
// Gauss-Seidel sweep of fcdiff/fit.py:184-197.  One CTA per patient; thread t
// owns the regions m = t, t+T, ... and keeps their q_R in registers.  Step n:
// every thread forms its partial sums over its m != n from the WT window that
// was prefetched during step n-1 (the loads do not depend on q_R), one warp
// shuffle reduction, ONE block barrier; then only the owner of region n
// finishes the reduction, normalises (fit.py:196) and updates its register
// copy of q_R[n] (fit.py:197) while the other threads already run step n+1.
// The two-slot s_red buffer makes the single barrier per step sufficient.
template <int T, int MPT, int LOOKUP>
__global__ void __launch_bounds__(T)
sweep_kernel(const double* __restrict__ WT, int64_t C, int N, int U, int u0,
             double lp0, double lp1,
             double* __restrict__ qR, double* __restrict__ lqR) {
    constexpr int NW = T / 32;
    __shared__ double s_red[2][NW];
    const int ul = blockIdx.x;
    const int u = u0 + ul;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double2* Wu = reinterpret_cast<const double2*>(WT) + (int64_t)ul * C;     // {W_0 - W_2, W_2 - W_1}
    double q0[MPT], q1[MPT];
#pragma unroll
    for (int j = 0; j < MPT; ++j) {
        const int m = tid + j * T;
        q0[j] = q1[j] = 0.0;
        if (m < N) {
            q0[j] = qR[((int64_t)m * U + u) * 2];
            q1[j] = qR[((int64_t)m * U + u) * 2 + 1];
        }
    }
    // reference lookup: the window of step n starts at edge n(n-1)/2 and moves by n edges per
    // step (fit.py:185-186): one running pointer, no index arithmetic per edge
    const double2* win = Wu + tid;                    // window of the next load_w call (n_next), thread's first edge
    int n_next = 0;
    auto load_w = [&](int n, double2 (&dst)[MPT]) {
        if (LOOKUP == FCD_LOOKUP_REFERENCE) {         // load_w is called with n = 0, 1, 2, ... in order
#pragma unroll
            for (int j = 0; j < MPT; ++j) {
                const int m = tid + j * T;
                dst[j] = make_double2(0.0, 0.0);
                if (m < N && m != n && n < N) dst[j] = __ldg(win + j * T);
            }
            win += n_next;                            // base(n + 1) - base(n) = n
            ++n_next;
        } else {
            const int64_t base = (int64_t)n * (n - 1) / 2;
#pragma unroll
            for (int j = 0; j < MPT; ++j) {
                const int m = tid + j * T;
                dst[j] = make_double2(0.0, 0.0);
                if (m < N && m != n && n < N) {
                    const int64_t c = m < n ? base + m : (int64_t)m * (m - 1) / 2 + n;
                    dst[j] = __ldg(Wu + c);
                }
            }
        }
    };
    const double dlp = lp0 - lp1;
    // One Gauss-Seidel step with the window `w`; the window of step n + 2 is requested
    // into `far` first (the loads do not depend on q_R), so that every window has two
    // steps to arrive.  The three register sets take turns (steps are unrolled by
    // three): no set is ever copied, a copy would wait for its loads.
    auto step = [&](int n, const double2 (&w)[MPT], double2 (&far)[MPT]) {
        load_w(n + 2, far);
        double sd = 0.0;
#pragma unroll
        for (int j = 0; j < MPT; ++j)                 // zero weights for m == n / m >= N
            sd += fma(q0[j], w[j].x, q1[j] * w[j].y);          // (fit.py:188-190) - (fit.py:192-194)
        sd = warp_sum(sd);
        if (lane == 0) s_red[n & 1][warp] = sd;
        __syncthreads();
        if (tid == n % T) {                           // owner of region n
            double a = 0.0;
#pragma unroll
            for (int i = 0; i < NW; ++i) a += s_red[n & 1][i];
            // lq = l - logsumexp(l), q = exp(lq) (fit.py:196-197) with one exponential:
            // with D = l_0 - l_1, d = -|D| and t = exp(d):  lse = max + log1p(t),
            // q_max = 1 / (1 + t), q_min = t / (1 + t).
            const double D = dlp + a;
            const bool first = D >= 0.0;
            const double d = first ? -D : D;
            const double t = exp_nonpos(d);
            // most regions are decided: below 2^-54, log1p(t) = t and 1/(1+t) = 1 to rounding
            // (skips the two long dependent chains of the step's critical path)
            double lg = t, inv = 1.0;
            if (t >= 5.551115123125783e-17) {
                lg = log1p(t);
                inv = 1.0 / (1.0 + t);
            }
            const double lmax = -lg, lmin = d - lg;
            const double qmax = inv, qmin = t * inv;
            const double l0 = first ? lmax : lmin, l1 = first ? lmin : lmax;
            const double p0 = first ? qmax : qmin, p1 = first ? qmin : qmax;
            const int slot = n / T;
#pragma unroll
            for (int j = 0; j < MPT; ++j)
                if (j == slot) {
                    q0[j] = p0;
                    q1[j] = p1;
                }
            const int64_t o = ((int64_t)n * U + u) * 2;
            *reinterpret_cast<double2*>(lqR + o) = make_double2(l0, l1);
            *reinterpret_cast<double2*>(qR + o) = make_double2(p0, p1);
        }
    };
    double2 wa[MPT], wb[MPT], wc[MPT];
    load_w(0, wa);
    load_w(1, wb);
    for (int n = 0; n < N; n += 3) {
        step(n, wa, wc);
        if (n + 1 < N) step(n + 1, wb, wa);
        if (n + 2 < N) step(n + 2, wc, wb);
    }
}

// --------------------------------------------------------------- K2b/sweep, blocked
// The same Gauss-Seidel sweep with the N dependent steps taken in blocks of B = 16 or 32 regions (blocked
// forward substitution), software-pipelined inside the CTA.  sweep_kernel pays, per region, one CTA-wide
// reduction + barrier + normalisation on the critical path (~0.6 us: the launch lasts N of them whatever the
// GPU could do in parallel).  Here one CTA per patient, q_R of all regions in shared memory, and per block b
// of regions [n0, n0 + B) two roles that run CONCURRENTLY, one barrier per block:
//   prepare(b + 1), warps 1..: everything of block b + 1 that does not depend on block b's new q_R --
//          (i)   the two B x B weight tiles the solver will need (rows of block b + 1 x columns of block b:
//                "near"; rows x columns of block b + 1: "in-block"), by 16-byte cp.async straight into shared
//                memory, transposed ([column][row]), no registers held while they fly;
//          (ii)  the rows of block b + 2 are requested into L2 (bulk prefetch): the far loads are latency-
//                bound, an L2 hit returns in a third of the time of an HBM access;
//          (iii) "far": every thread accumulates, for 16 rows at once, the terms of the regions outside
//                blocks b and b + 1 (already updated before, not yet updated after: fit.py:185-194 with the
//                q_R of the moment) and of the regions of block b + 1 AFTER each row (old q_R, masked) -- 16
//                independent accumulators and loads in flight per thread; one warp transpose-reduction per
//                16 rows;
//   solve(b), warp 0: lane i holds D_i = l_0 - l_1 of region n0 + i: far sums + the near tile times the
//          q_R block b - 1 just received, then B right-looking steps: step r broadcasts D_r (final: every
//          earlier region of the block has been added), ALL lanes form q_R[n0 + r] from it (warp-uniform: no
//          divergence, no second broadcast) and add its term to their own D_i; weights from the in-block
//          tile, requested one step ahead.  The chain of a step is one shuffle, the logistic function
//          (exponential in Estrin form, reciprocal by MUFU + one cubic correction) and two FMAs -- for a
//          decided region (|D| >= 37.5: exp(-|D|) < 2^-54) a shuffle, an integer compare and one addition.
//          No reduction, no barrier, no logarithm on the chain;
//   outputs(b - 1), last helper warp: lq_R = l - logsumexp(l), q_R = exp(lq_R) (fit.py:196-197) of the block
//          solved in the previous phase, from its D values, one lane per region -- sweep_kernel's formulas.
// Same arithmetic per term as sweep_kernel (the order of the additions differs; the q_R a later step of the
// sweep uses comes from the chain's reciprocal and is exactly (1, 0) for a decided region, where the stored
// output is the correctly rounded quotient and (1, exp(-|D|) < 5.2e-17): |dD| < 1e-15).
constexpr int kSwRH = 16;                                                  // rows per far pass

template <int LOOKUP>
__device__ __forceinline__ int64_t sweep_edge(int n, int m, int64_t base_n) {
    if (LOOKUP == FCD_LOOKUP_REFERENCE) return base_n + m;                 // nm_to_c(n, m) even for m > n (fit.py:185-186)
    return m < n ? base_n + m : (int64_t)m * (m - 1) / 2 + n;
}

// q_R [Npad] | tiles [2 buffers][near, in-block][B x (B + 1)] | far sums [2][helper warps][B] | D [2][B]
__host__ __device__ constexpr size_t sweep_blocked_smem(int N, int T, int B, int cs = 1) {
    return (size_t)((N + 31) & ~31) * 16 + (size_t)4 * B * (B + 1) * 16 + (size_t)2 * cs * (T / 32 - 1) * B * 8 +
           (size_t)2 * B * 8;
}

// Thread-block cluster helpers (CS > 1 form of the blocked sweep: the CTAs of a cluster share one patient).
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t dsmem_addr(const void* local, uint32_t rank) {
    uint32_t a;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"((uint32_t)__cvta_generic_to_shared(local)), "r"(rank));
    return a;
}
__device__ __forceinline__ void dsmem_store(uint32_t addr, double v) {
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ void dsmem_store2(uint32_t addr, double2 v) {
    asm volatile("st.shared::cluster.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(v.x), "d"(v.y) : "memory");
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;"
                 ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}

// CS > 1 (few patients on this GPU -- sharded fits: 63 patients on 148 SMs): the CS CTAs of a thread-block cluster
// share ONE patient.  The launch lasts a patient's chain of blocks and a block lasts what its far sums take one SM to
// pull from L2; the cluster splits the far columns over its CTAs, CTA r > 0 stores its warps' partial sums into CTA
// 0's shared memory (DSMEM), CTA 0 alone holds the tiles, solves and writes the outputs, and sends every solved
// block's q_R to the others' copies of s_q; the per-block barrier becomes a cluster barrier.
template <int T, int B, int LOOKUP, int CS = 1>
__global__ void __launch_bounds__(T, 512 / T)
sweep_blocked_kernel(const double* __restrict__ WT, int64_t C, int N, int U, int u0, double lp0, double lp1,
                     double* __restrict__ qR, double* __restrict__ lqR) {
    constexpr int NWH = T / 32 - 1, H = T - 32, Bp = B + 1, RH = kSwRH, TILE = B * Bp, NWP = CS * NWH;
    constexpr int LB = B == 32 ? 5 : 4;
    static_assert(B == 16 || B == 32, "block of 16 or 32 regions");
    extern __shared__ __align__(16) double s_sweep[];
    double2* s_q = reinterpret_cast<double2*>(s_sweep);                    // [Npad] q_R of the moment
    const int Npad = (N + 31) & ~31;
    double2* s_tiles = s_q + Npad;                                         // [2][2][B][Bp], [column][row]
    double* s_part = reinterpret_cast<double*>(s_tiles + 4 * TILE);       // [2][CS NWH][B] per-warp far sums
    double* s_D = s_part + 2 * NWP * B;                                    // [2][B] l_0 - l_1 of a solved block
    const int crank = CS > 1 ? (int)cluster_ctarank() : 0;
    const int ul = CS > 1 ? blockIdx.x / CS : blockIdx.x, u = u0 + ul;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double2* Wu = reinterpret_cast<const double2*>(WT) + (int64_t)ul * C;   // {W_0 - W_2, W_2 - W_1}
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    for (int m = tid; m < Npad; m += T) s_q[m] = m < N ? qR2[(int64_t)m * U + u] : make_double2(0.0, 0.0);
    if (CS > 1) cluster_sync_all(); else __syncthreads();
    const double dlp = lp0 - lp1;
    const int nblocks = (N + B - 1) / B;

    // ---- prepare(b): helper warps only
    auto prepare = [&](int b) {
        const int ht = tid - 32, hw = warp - 1;
        const int n0 = b * B;
        const int nb = N - n0 < B ? N - n0 : B;
        double2* tiles = s_tiles + (b & 1) * 2 * TILE;
        // (i) tiles: element e -> tile t (0 near, 1 in-block), row i, column j; lanes walk a row's columns
        // (contiguous edges: both tiles have m < n, where the two lookups agree)
        if (crank == 0)
            for (int e = ht; e < 2 * B * B; e += H) {
                const int t = e >> (2 * LB), i = (e >> LB) & (B - 1), j = e & (B - 1);
                double2* dst = tiles + t * TILE + j * Bp + i;
                const int n = n0 + i;
                const bool live = i < nb && (t == 0 ? b > 0 : j < i);
                if (live) cp_async16(dst, Wu + (int64_t)n * (n - 1) / 2 + (n0 - (t == 0 ? B : 0)) + j);
                else *dst = make_double2(0.0, 0.0);
            }
        // (ii) the rows of block b + 1 (what the NEXT prepare will read, one phase from now) into L2
        if (b + 1 < nblocks && lane == 0 && crank == 0) {                  // (the instruction takes warp-uniform operands)
            const int n1 = n0 + B, nl = n1 + B - 1 < N - 1 ? n1 + B - 1 : N - 1;
            const int64_t e0 = (int64_t)n1 * (n1 - 1) / 2;
            int64_t e1 = (int64_t)nl * (nl - 1) / 2 + (LOOKUP == FCD_LOOKUP_REFERENCE ? N : nl);
            if (e1 > C) e1 = C;
            const char* g0 = reinterpret_cast<const char*>(Wu + e0);
            const int64_t bytes = ((e1 - e0) * (int64_t)sizeof(double2)) & ~(int64_t)15;
            for (int64_t off = (int64_t)hw * 8192; off < bytes; off += (int64_t)NWH * 8192) {
                const uint32_t sz = (uint32_t)(bytes - off < 8192 ? bytes - off : 8192);
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(g0 + off), "r"(sz) : "memory");
            }
        }
        // (iii) far sums.  Row n0 + r of column m is the edge base(n0 + r) + m (reference lookup, and the
        // symmetric one for m < n0): base(n0 + r) = base(n0) + r n0 + r (r - 1) / 2 -- one pointer per column,
        // one 32-bit offset per row; for m > n (symmetric) the edges base(m) + n0 + r.  The rows are taken
        // RH = 16 at a time: 16 accumulators leave the registers for 16 loads in flight per thread.
        const int64_t base0 = (int64_t)n0 * (n0 - 1) / 2;
        using yes = std::integral_constant<bool, true>;
        using no = std::integral_constant<bool, false>;
#pragma unroll 1
        for (int h = 0; h < B; h += RH) {
            double acc[RH];
#pragma unroll
            for (int r = 0; r < RH; ++r) acc[r] = 0.0;
            // `masked` = false is the common case (a whole block of rows, a column outside the block): no
            // predicate per row -- a per-row predicate would cap the loads in flight at the 7 predicate registers
            auto rows = [&](const double2* p, int stride, auto tri, auto masked, int lim, double2 q) {
                p += h * stride + (decltype(tri)::value ? h * (h - 1) / 2 : 0);
                // base(n0 + h + r) - base(n0 + h) = r (n0 + h) + r (r - 1) / 2
                auto off = [&](int r) {
                    return r * (stride + (decltype(tri)::value ? h : 0)) + (decltype(tri)::value ? r * (r - 1) / 2 : 0);
                };
#pragma unroll
                for (int r = 0; r < RH; ++r) {
                    if (!decltype(masked)::value || h + r < lim) {
                        const double2 w = __ldg(p + off(r));
                        acc[r] = fma(q.x, w.x, fma(q.y, w.y, acc[r]));    // (fit.py:188-190) - (fit.py:192-194)
                    }
                }
            };
            for (int m = ht + crank * H; m < N; m += CS * H) {
                const int mb = m >> LB;
                if (mb == b - 1) continue;                                 // near: the solver's (new q_R of block b - 1)
                const double2 q = s_q[m];
                const bool tri = LOOKUP == FCD_LOOKUP_REFERENCE || m < n0;
                const double2* p = tri ? Wu + base0 + m : Wu + (int64_t)m * (m - 1) / 2 + n0;
                if (mb != b && nb == B) {
                    if (tri) rows(p, n0, yes(), no(), B, q);
                    else rows(p, 1, no(), no(), B, q);
                } else {
                    // in-block column: only the rows before the column; last block: only the rows that exist
                    const int lim = mb == b ? m - n0 : nb;
                    if (tri) rows(p, n0, yes(), yes(), lim, q);
                    else rows(p, 1, no(), yes(), lim, q);
                }
            }
            // warp transpose-reduction: 16 sums over 32 lanes, lane r (and r + 16) ends with row h + r
#pragma unroll
            for (int i = 0; i < RH; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 16);
#pragma unroll
            for (int off = RH / 2; off >= 1; off >>= 1) {
                const bool up = (lane & off) != 0;
#pragma unroll
                for (int i = 0; i < off; ++i) {
                    const double send = up ? acc[i] : acc[i + off];
                    const double keep = up ? acc[i + off] : acc[i];
                    acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                }
            }
            if (lane < RH) {
                double* dst = s_part + ((b & 1) * NWP + crank * NWH + hw) * B + h + lane;
                if (CS == 1 || crank == 0) *dst = acc[0];
                else dsmem_store(dsmem_addr(dst, 0), acc[0]);              // into CTA 0's copy
            }
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
    };

    // ---- solve(b): warp 0 only (B = 16: lanes 16.. mirror lanes 0..15)
    auto solve = [&](int b) {
        const int n0 = b * B, li = lane & (B - 1);
        const int nb = N - n0 < B ? N - n0 : B;
        const double2* near = s_tiles + (b & 1) * 2 * TILE;
        const double2* wb = near + TILE;
        double Da = dlp, Db = 0.0;
#pragma unroll
        for (int w = 0; w < NWP; w += 2) {
            Da += s_part[((b & 1) * NWP + w) * B + li];
            if (w + 1 < NWP) Db += s_part[((b & 1) * NWP + w + 1) * B + li];
        }
        double D = Da + Db;
        if (b > 0) {                                                       // near tile x the block solved last
            double d4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int j = 0; j < B; ++j) {
                const double2 qj = s_q[n0 - B + j];                        // broadcast
                const double2 w = near[j * Bp + li];
                d4[j & 3] = fma(qj.x, w.x, fma(qj.y, w.y, d4[j & 3]));
            }
            D += (d4[0] + d4[1]) + (d4[2] + d4[3]);
        }
        double Dmine = 0.0;
        double2 qmine = make_double2(0.0, 0.0);
        double2 wn = wb[li];
        for (int r = 0; r < nb; ++r) {
            const double2 w = wn;
            wn = wb[((r + 1) & (B - 1)) * Bp + li];                       // next step's weights: off the chain
            const double Dr = __shfl_sync(0xffffffffu, D, r);
            // q = exp(lq), lq = l - logsumexp(l) (fit.py:196-197): q_max = 1 / (1 + t), q_min = t / (1 + t),
            // t = exp(-|D|); warp-uniform.  |D| >= 37.5 (an integer compare of the high word): t < 2^-54.
            const int hi = __double2hiint(Dr);
            const bool first = hi >= 0;
            double q0, q1;
            if ((hi & 0x7fffffff) >= 0x4042c000) {
                q0 = first ? 1.0 : 0.0;
                q1 = first ? 0.0 : 1.0;
                D += first ? w.x : w.y;
            } else {
                const double t = exp_nonpos_short(-fabs(Dr));
                const double qmax = rcp_newton(1.0 + t), qmin = t * qmax;
                q0 = first ? qmax : qmin;
                q1 = first ? qmin : qmax;
                D = fma(q0, w.x, fma(q1, w.y, D));                         // rows <= r: zero weight (tile holds j < i only)
            }
            if (lane == r) {
                Dmine = Dr;
                qmine = make_double2(q0, q1);
            }
        }
        if (lane < nb) {
            s_q[n0 + lane] = qmine;
            s_D[(b & 1) * B + lane] = Dmine;
            if constexpr (CS > 1) {                                        // the other CTAs' far sums read their own s_q
#pragma unroll
                for (int r = 1; r < CS; ++r) dsmem_store2(dsmem_addr(s_q + n0 + lane, r), qmine);
            }
        }
    };

    // ---- outputs(b): one warp, a lane per region of a solved block; one exponential (see sweep_kernel)
    auto outputs = [&](int b) {
        const int n0 = b * B;
        const int nb = N - n0 < B ? N - n0 : B;
        if (lane < nb) {
            const double Dm = s_D[(b & 1) * B + lane];
            const bool first = Dm >= 0.0;
            const double d = first ? -Dm : Dm;
            const double e = exp_nonpos(d);
            double lg = e, inv = 1.0;
            if (e >= 5.551115123125783e-17) {
                lg = log1p(e);
                inv = 1.0 / (1.0 + e);
            }
            const double lmax = -lg, lmin = d - lg;
            const double qmax = inv, qmin = e * inv;
            const int64_t o = ((int64_t)(n0 + lane) * U + u) * 2;
            *reinterpret_cast<double2*>(lqR + o) = first ? make_double2(lmax, lmin) : make_double2(lmin, lmax);
            *reinterpret_cast<double2*>(qR + o) = first ? make_double2(qmax, qmin) : make_double2(qmin, qmax);
        }
    };

    if (warp > 0) prepare(0);
    if (CS > 1) cluster_sync_all(); else __syncthreads();
    for (int b = 0; b < nblocks; ++b) {
        if (warp == 0) {
            if (crank == 0) solve(b);
        } else {
            if (warp == NWH && b >= 1 && crank == 0) outputs(b - 1);
            if (b + 1 < nblocks) prepare(b + 1);
        }
        if (CS > 1) cluster_sync_all(); else __syncthreads();     // (the last one also keeps every CTA alive while
    }                                                             //  CTA 0 may still store into its shared memory)
    if (warp == NWH && crank == 0) outputs(nblocks - 1);
}

static inline int grid_for_rows(int64_t rows, int rows_per_block, int waves) {
    int64_t need = (rows + rows_per_block - 1) / rows_per_block;
    int64_t cap = (int64_t)sm_count() * waves;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int fcd_c_to_nm(int64_t c0, int64_t C, int32_t* n_out, int32_t* m_out, void* stream) {
    FCD_REQUIRE(C >= 0 && c0 >= 0, "fcd_c_to_nm: bad range");
    if (C == 0) return 0;
    c_to_nm_kernel<<<grid_for_rows(C, 256, 8), 256, 0, (cudaStream_t)stream>>>(c0, C, n_out, m_out);
    return check_launch("fcd_c_to_nm");
}

int fcd_edge_table(int64_t c0, int64_t C, int32_t* nm, void* stream) {
    FCD_REQUIRE(C >= 0 && c0 >= 0 && (C == 0 || nm != nullptr), "fcd_edge_table: bad arguments");
    FCD_REQUIRE(c0 + C <= (int64_t)65535 * 65534 / 2, "fcd_edge_table: more than 65535 regions");
    if (C == 0) return 0;
    edge_table_kernel<<<grid_for_rows(C, 256, 8), 256, 0, (cudaStream_t)stream>>>(c0, C, nm);
    return check_launch("fcd_edge_table");
}

// S0 == NULL: every control is observed (the unmasked kernel); otherwise NaN entries are left out and S0 counts
// the observed controls of each edge.
int fcd_healthy_stats(const double* b, int64_t C, int32_t H, int64_t pitchH,
                      double* S1, double* S2, double* S0, void* stream) {
    FCD_REQUIRE(C >= 0 && H >= 1 && pitchH >= H, "fcd_healthy_stats: bad shape C=%lld H=%d pitch=%lld",
                (long long)C, H, (long long)pitchH);
    FCD_REQUIRE(S0 == nullptr || C == 0 || (b != nullptr && S1 != nullptr && S2 != nullptr),
                "fcd_healthy_stats: NULL argument");
    if (C == 0) return 0;
    if (S0 == nullptr)
        healthy_stats_kernel<false><<<grid_for_rows(C, kEdgeThreads / 32, 8), kEdgeThreads, 0, (cudaStream_t)stream>>>(
            b, C, H, pitchH, S1, S2, nullptr);
    else
        healthy_stats_kernel<true><<<grid_for_rows(C, kEdgeThreads / 32, 8), kEdgeThreads, 0, (cudaStream_t)stream>>>(
            b, C, H, pitchH, S1, S2, S0);
    return check_launch("fcd_healthy_stats");
}

int fcd_resp_cache(const double* bt, int64_t C, int32_t U, int64_t pitchU,
                   const fcd_theta* theta_host, double* P, int64_t planeStride, double* L, int32_t missing,
                   void* stream) {
    FCD_REQUIRE(theta_host != nullptr && bt != nullptr && P != nullptr, "fcd_resp_cache: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && pitchU >= U && planeStride >= C * pitchU, "fcd_resp_cache: bad shape");
    FCD_REQUIRE(missing == 0 || missing == 1, "fcd_resp_cache: missing must be 0 or 1, got %d", missing);
    if (C == 0) return 0;
    const ThetaDev th = make_theta_dev(*theta_host, 0);
    if (missing)
        resp_cache_kernel<true><<<grid_for_rows(C * pitchU, 256, 16), 256, 0, (cudaStream_t)stream>>>(
            bt, C, U, pitchU, th, P, planeStride, L);
    else
        resp_cache_kernel<false><<<grid_for_rows(C * pitchU, 256, 16), 256, 0, (cudaStream_t)stream>>>(
            bt, C, U, pitchU, th, P, planeStride, L);
    return check_launch("fcd_resp_cache");
}

int fcd_map_labels(const double* lq, int64_t n, int32_t width, uint8_t* labels, void* stream) {
    FCD_REQUIRE(n >= 0 && width >= 1 && (n == 0 || (lq != nullptr && labels != nullptr)), "fcd_map_labels: bad arguments");
    if (n == 0) return 0;
    map_labels_kernel<<<grid_for_rows(n, 256, 8), 256, 0, (cudaStream_t)stream>>>(lq, n, width, labels);
    return check_launch("fcd_map_labels");
}

int fcd_peak_states_F(const double* qF, int64_t C, uint8_t* fstate, void* stream) {
    FCD_REQUIRE(C >= 0 && (C == 0 || (qF != nullptr && fstate != nullptr)), "fcd_peak_states_F: bad arguments");
    if (C == 0) return 0;
    peak_states_F_kernel<<<grid_for_rows(C, 256, 8), 256, 0, (cudaStream_t)stream>>>(qF, C, fstate);
    return check_launch("fcd_peak_states_F");
}

int fcd_peak_states_R(const double* qR, int32_t N, int32_t U, int64_t pitchS, uint8_t* rstate, void* stream) {
    FCD_REQUIRE(N >= 1 && U >= 1 && pitchS >= U && qR != nullptr && rstate != nullptr,
                "fcd_peak_states_R: bad arguments");
    peak_states_R_kernel<<<grid_for_rows((int64_t)N * pitchS, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        qR, N, U, pitchS, rstate);
    return check_launch("fcd_peak_states_R");
}

// S0 == NULL: every edge has all H controls (the unmasked kernel).
int fcd_estep_qF(const double* S1, const double* S2, const double* S0, int32_t H,
                 const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                 const double* qR, const uint8_t* rstate, int64_t pitchS, int32_t N, const int32_t* nm,
                 const fcd_theta* theta_host, double* lqF, double* qF, void* stream) {
    FCD_REQUIRE(theta_host != nullptr && P != nullptr && qR != nullptr && rstate != nullptr && nm != nullptr &&
                lqF != nullptr, "fcd_estep_qF: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && U < 65536 && pitchU >= U && pitchS >= U && N >= 2 && N < 65536,
                "fcd_estep_qF: bad shape");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(P) & 15) == 0) && pitchU % 2 == 0 && planeStride % 2 == 0 &&
                pitchS % 256 == 0, "fcd_estep_qF: planes must be 16-byte aligned with even pitches (pitchS % 256 == 0)");
    if (C == 0) return 0;
    const ThetaDev th = make_theta_dev(*theta_host, H);
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(th.epsl, th.al, st, tab, true), "fcd_estep_qF: log table initialisation failed");
    const bool fast = log_table_covers(th.epsl, th.al);
    const size_t tbytes = fast ? (size_t)((tab.n + 1) & ~1) * sizeof(double) : 0;
    const int depth = stream_depth<2, kK2Seg>(tbytes);
    FCD_REQUIRE(depth >= 2, "fcd_estep_qF: shared memory budget exceeded");
    const size_t smem = tbytes + StreamGeom<2, kK2Seg>::bytes(kStreamWarps, depth);
    int64_t grid = (C + kStreamWarps - 1) / kStreamWarps;
    if (grid > sm_count()) grid = sm_count();                       // one persistent CTA per SM
#define K2_LAUNCH(F, M)                                                                               \
    do {                                                                                              \
        cudaFuncSetAttribute(estep_qF_kernel<F, M>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                             (int)kSmemBudget);                                                       \
        estep_qF_kernel<F, M><<<(unsigned)grid, kStreamThreads, smem, st>>>(                          \
            S1, S2, S0, P, planeStride, C, U, pitchU, qR, rstate, pitchS, nm, th, tab, depth, lqF, qF); \
    } while (0)
    if (S0 != nullptr) {
        if (fast) K2_LAUNCH(true, true); else K2_LAUNCH(false, true);
    } else {
        if (fast) K2_LAUNCH(true, false); else K2_LAUNCH(false, false);
    }
#undef K2_LAUNCH
    return check_launch("fcd_estep_qF");
}

// S0 == NULL: every edge has all H controls (the unmasked kernel).  solver_state == NULL: (eta, epsilon) of
// theta_host; otherwise the solver state block a device-resident solve enqueued BEFORE this launch leaves its
// solution in, with [eps_lo, eps_hi] the box of that solve (it sizes the logarithm table like
// fcd_elm_coded_solve does).
int fcd_estep_qF_coded(const double* S1, const double* S2, const double* S0, int32_t H,
                       const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                       const double* qR, int32_t N, const int32_t* nm,
                       const uint8_t* code, int64_t pitchQ, const int32_t* counts, const uint64_t* keysF,
                       const uint64_t* keysH, const int64_t* rowoff, const double* Hh,
                       const fcd_theta* theta_host, const void* solver_state, double eps_lo, double eps_hi,
                       double* lqF, double* qF, void* stream) {
    FCD_REQUIRE(theta_host != nullptr && S1 != nullptr && S2 != nullptr && P != nullptr && qR != nullptr &&
                nm != nullptr && code != nullptr && counts != nullptr && keysF != nullptr && keysH != nullptr &&
                rowoff != nullptr && Hh != nullptr && lqF != nullptr, "fcd_estep_qF_coded: NULL argument");
    FCD_REQUIRE(C >= 0 && U >= 1 && U < 65536 && pitchU >= U && N >= 2 && N < 65536, "fcd_estep_qF_coded: bad shape");
    FCD_REQUIRE((reinterpret_cast<uintptr_t>(solver_state) & 7) == 0,
                "fcd_estep_qF_coded: solver state must be a device pointer (fcd_solver_init)");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(P) | reinterpret_cast<uintptr_t>(code) | reinterpret_cast<uintptr_t>(rowoff) |
                  reinterpret_cast<uintptr_t>(Hh)) & 15) == 0 && (reinterpret_cast<uintptr_t>(counts) & 7) == 0 &&
                pitchU % 2 == 0 && planeStride % 2 == 0 && pitchQ >= pitchU && pitchQ % 16 == 0,
                "fcd_estep_qF_coded: planes / code / rowoff / half records must be 16-byte aligned (even pitchU, pitchQ % 16 == 0)");
    if (C == 0) return 0;
    const SolverState* solved = static_cast<const SolverState*>(solver_state);
    const ThetaDev th = make_theta_dev(*theta_host, H);
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    double w_eps[3] = {th.epsl[0], th.epsl[1], th.epsl[2]}, w_al[3] = {th.al[0], th.al[1], th.al[2]};
    if (solved != nullptr) {
        // every mixture weight the solve can have ended at lies in [m / 2, 1], m = min(eps_lo, 1 - eps_hi)
        FCD_REQUIRE(eps_lo > 0.0 && eps_lo <= eps_hi && eps_hi < 1.0, "fcd_estep_qF_coded: bad box");
        const double m = eps_lo < 1.0 - eps_hi ? eps_lo : 1.0 - eps_hi;
        for (int l = 0; l < 3; ++l) {
            w_eps[l] = m;
            w_al[l] = 0.5 * m;
        }
    }
    FCD_REQUIRE(log_table_window(w_eps, w_al, st, tab, true), "fcd_estep_qF_coded: log table initialisation failed");
    const bool fast = log_table_covers(w_eps, w_al);
    const size_t tbytes = fast ? (size_t)((tab.n + 15) & ~15) * sizeof(double) : 0;
    // 16 warps per SM (127 registers each).  24 warps (80 registers, three ring stages per warp) were measured no
    // faster (0.199 vs 0.193 ms at config 3): the kernel is bound by the instructions of its row-level work, not by
    // the warps available to hide latency.
    constexpr int NW = 16;
    int depth = kK2cMaxDepth;
    while (depth > 2 && tbytes + k2c_ring_bytes(depth, NW) > kSmemBudget) --depth;
    FCD_REQUIRE(tbytes + k2c_ring_bytes(depth, NW) <= kSmemBudget, "fcd_estep_qF_coded: shared memory budget exceeded");
    const size_t smem = tbytes + k2c_ring_bytes(depth, NW);
    int64_t grid = (C + NW - 1) / NW;
    if (grid > sm_count()) grid = sm_count();                       // one persistent CTA per SM
#define K2C_LAUNCH(F, M)                                                                              \
    do {                                                                                              \
        FCD_ALLOW_BIG_SMEM(estep_qF_coded_kernel<F, NW, M>);                                          \
        estep_qF_coded_kernel<F, NW, M><<<(unsigned)grid, NW * 32, smem, st>>>(                       \
            S1, S2, S0, P, planeStride, C, U, pitchU, qR, nm, code, pitchQ, reinterpret_cast<const int2*>(counts), \
            reinterpret_cast<const unsigned long long*>(keysF), reinterpret_cast<const unsigned long long*>(keysH), \
            reinterpret_cast<const longlong2*>(rowoff), reinterpret_cast<const double2*>(Hh), th, solved, tab, depth, lqF, qF); \
    } while (0)
    if (S0 != nullptr) {
        if (fast) K2C_LAUNCH(true, true); else K2C_LAUNCH(false, true);
    } else {
        if (fast) K2C_LAUNCH(true, false); else K2C_LAUNCH(false, false);
    }
#undef K2C_LAUNCH
    return check_launch("fcd_estep_qF_coded");
}

int fcd_pstar_refresh_em(const double* Pe, int64_t planeStride, int64_t pitchU, int32_t u0, int32_t Ul, int64_t C,
                         int64_t pitchC, const uint8_t* fstate, double* PsT, uint8_t* kcache, void* stream) {
    FCD_REQUIRE(Pe != nullptr && fstate != nullptr && PsT != nullptr && kcache != nullptr,
                "fcd_pstar_refresh_em: NULL argument");
    FCD_REQUIRE(C >= 0 && Ul >= 0 && u0 >= 0 && pitchU >= (int64_t)u0 + Ul && pitchC >= C, "fcd_pstar_refresh_em: bad shape");
    if (C == 0 || Ul == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    pstar_refresh_em_kernel<<<(unsigned)((C + 31) / 32), 256, 0, st>>>(Pe, planeStride, pitchU, u0, Ul, C, pitchC, fstate,
                                                                        kcache, PsT);
    int rc = check_launch("fcd_pstar_refresh_em");
    if (rc) return rc;
    pstar_commit_kernel<<<(unsigned)((C + 255) / 256), 256, 0, st>>>(fstate, C, kcache);
    return check_launch("fcd_pstar_refresh_em(commit)");
}

int fcd_region_weights_em(const double* Pe, int64_t planeStride, int64_t pitchU, int32_t u0, int32_t Ul, int64_t C,
                          int64_t pitchC, const double* qF, const uint8_t* fstate, double* PsT, uint8_t* kcache,
                          const fcd_theta* theta_host, double* WT, void* stream) {
    FCD_REQUIRE(theta_host != nullptr && fstate != nullptr && Pe != nullptr && PsT != nullptr && kcache != nullptr,
                "fcd_region_weights_em: NULL argument");
    FCD_REQUIRE(C >= 0 && Ul >= 0 && u0 >= 0 && pitchU >= (int64_t)u0 + Ul && pitchC >= C, "fcd_region_weights_em: bad shape");
    if (C == 0 || Ul == 0) return 0;
    int rc = fcd_pstar_refresh_em(Pe, planeStride, pitchU, u0, Ul, C, pitchC, fstate, PsT, kcache, stream);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const ThetaDev th = make_theta_dev(*theta_host, 0);
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(th.epsl, th.al, st, tab), "fcd_region_weights_em: log table initialisation failed");
    int64_t ntiles = ((C + 1023) / 1024) * (int64_t)Ul;
    FCD_REQUIRE(ntiles < ((int64_t)1 << 31) - 8 * sm_count(), "fcd_region_weights_em: %lld tiles exceed the 32-bit tile index",
                (long long)ntiles);
    // the edge-major planes [3][C][pitchU] from patient u0 on: element (k, u, c) at Pe + u0 + k planeStride + u + c pitchU
    if (log_table_covers(th.epsl, th.al)) {
        int per_sm = (int)((200 * 1024) / (tab.bytes() + 1024));
        if (per_sm > 8) per_sm = 8;
        if (per_sm < 1) per_sm = 1;
        int64_t grid = (int64_t)sm_count() * per_sm;
        if (grid > ntiles) grid = ntiles;
        cudaFuncSetAttribute(region_weights_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)kLogTabBytes);
        region_weights_kernel<true><<<(unsigned)grid, 256, tab.bytes(), st>>>(
            Pe + u0, planeStride, 1, pitchU, Ul, C, pitchC, qF, fstate, PsT, th, tab, WT);
    } else {
        int64_t grid = (int64_t)sm_count() * 4;
        if (grid > ntiles) grid = ntiles;
        region_weights_kernel<false><<<(unsigned)grid, 256, 0, st>>>(
            Pe + u0, planeStride, 1, pitchU, Ul, C, pitchC, qF, fstate, PsT, th, tab, WT);
    }
    return check_launch("fcd_region_weights_em");
}

int fcd_estep_qR(const double* WT, int64_t C, int32_t N, int32_t U, int32_t u0, int32_t Ul,
                 const double* log_pi2_host, int32_t edge_lookup,
                 double* qR, double* lqR, void* stream) {
    FCD_REQUIRE(log_pi2_host != nullptr, "fcd_estep_qR: log_pi2 is NULL");
    FCD_REQUIRE(N >= 2 && C == (int64_t)N * (N - 1) / 2, "fcd_estep_qR: C=%lld is not N(N-1)/2 for N=%d",
                (long long)C, N);
    FCD_REQUIRE(edge_lookup == FCD_LOOKUP_REFERENCE || edge_lookup == FCD_LOOKUP_SYMMETRIC,
                "fcd_estep_qR: unknown edge_lookup %d", edge_lookup);
    FCD_REQUIRE(!(edge_lookup == FCD_LOOKUP_REFERENCE && N < 3),
                "fcd_estep_qR: edge_lookup='reference' indexes out of bounds for N < 3 (fit.py:186)");
    FCD_REQUIRE(u0 >= 0 && Ul >= 0 && u0 + Ul <= U, "fcd_estep_qR: bad patient range");
    if (Ul == 0) return 0;
    FCD_REQUIRE(N <= 8192, "fcd_estep_qR: N=%d exceeds the 8192 regions the sweep kernel supports", N);
    cudaStream_t st = (cudaStream_t)stream;
    const double lp0 = log_pi2_host[0], lp1 = log_pi2_host[1];
    // blocked forward substitution (sweep_blocked_kernel) from 64 regions on
    if (N >= 64) {
        // launch shape (scripts/sweep_bench.py, profiles/r02_sweep_shapes.txt): blocks of B = 16 regions
        // everywhere (32 was measured, never faster).  Threads: 3 helper warps and FOUR CTAs per SM (25 KB of
        // shared memory at N = 400) when the GPU has patients to fill them with -- every patient of the bench
        // problem resident at once; 7 helper warps for mid-sized atlases or fewer patients; 15 (one CTA per SM)
        // from ~700 regions on, where a patient's chain of blocks is what the launch lasts.
        constexpr int B = 16;
        int T = N >= 700 ? 512 : ((N <= 512 && Ul > 2 * sm_count()) ? 128 : 256);
        while (T < 512 && sweep_blocked_smem(N, T, B) > (size_t)(T == 128 ? 54 : 110) * 1024) T *= 2;
        // Cluster form: two CTAs per patient when that still fits one wave (sharded fits: 63 patients on 148 SMs).
        // Measured (scripts/sweep_bench.py, us, one CTA -> cluster of two): 1131 regions x 63 patients 310 -> 294
        // (undecided regime) / 290 -> 252 (decided); 400 x 63: 86 -> 91 / 74 -> 74; 800 x 125 (does not fit one
        // wave): 204 -> 407.  At 63 patients the launch already moves the patients' 644 MB of weights at ~4 TB/s --
        // it is closer to the memory system's limit than to a single SM's, so the second SM buys little: used from
        // ~700 regions on (512 threads), where it does gain.
        const int cs = (T == 512 && 2 * (int64_t)Ul <= (int64_t)sm_count()) ? 2 : 1;
        const size_t smem = sweep_blocked_smem(N, T, B, cs);
        FCD_REQUIRE(smem <= kSmemBudget, "fcd_estep_qR: N=%d needs %zu bytes of shared memory", N, smem);
        if (cs == 2) {
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.gridDim = dim3((unsigned)(2 * Ul));
            cfg.blockDim = dim3((unsigned)T);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = st;
            cudaLaunchAttribute attr;
            attr.id = cudaLaunchAttributeClusterDimension;
            attr.val.clusterDim.x = 2;
            attr.val.clusterDim.y = 1;
            attr.val.clusterDim.z = 1;
            cfg.attrs = &attr;
            cfg.numAttrs = 1;
            cudaError_t e = cudaSuccess;
#define FCD_SWC(L_)                                                                                           \
            do {                                                                                              \
                FCD_ALLOW_BIG_SMEM((sweep_blocked_kernel<512, B, L_, 2>));                                    \
                e = cudaLaunchKernelEx(&cfg, sweep_blocked_kernel<512, B, L_, 2>, WT, C, N, U, u0, lp0, lp1, qR, lqR); \
            } while (0)
            if (edge_lookup == FCD_LOOKUP_REFERENCE) FCD_SWC(FCD_LOOKUP_REFERENCE);
            else FCD_SWC(FCD_LOOKUP_SYMMETRIC);
#undef FCD_SWC
            FCD_REQUIRE(e == cudaSuccess, "fcd_estep_qR(cluster): %s", cudaGetErrorString(e));
            return check_launch("fcd_estep_qR(blocked, cluster)");
        }
#define FCD_SWB(T_)                                                                                          \
        do {                                                                                                 \
            if (edge_lookup == FCD_LOOKUP_REFERENCE) {                                                       \
                FCD_ALLOW_BIG_SMEM(sweep_blocked_kernel<T_, B, FCD_LOOKUP_REFERENCE>);                       \
                sweep_blocked_kernel<T_, B, FCD_LOOKUP_REFERENCE><<<Ul, T_, smem, st>>>(WT, C, N, U, u0, lp0, lp1, qR, lqR); \
            } else {                                                                                         \
                FCD_ALLOW_BIG_SMEM(sweep_blocked_kernel<T_, B, FCD_LOOKUP_SYMMETRIC>);                       \
                sweep_blocked_kernel<T_, B, FCD_LOOKUP_SYMMETRIC><<<Ul, T_, smem, st>>>(WT, C, N, U, u0, lp0, lp1, qR, lqR); \
            }                                                                                                \
        } while (0)
        if (T == 512) FCD_SWB(512);
        else if (T == 256) FCD_SWB(256);
        else FCD_SWB(128);
#undef FCD_SWB
        return check_launch("fcd_estep_qR(blocked)");
    }
#define SWEEP_LAUNCH(M)                                                                            \
    do {                                                                                           \
        if (edge_lookup == FCD_LOOKUP_REFERENCE)                                                   \
            sweep_kernel<32, M, FCD_LOOKUP_REFERENCE><<<Ul, 32, 0, st>>>(WT, C, N, U, u0, lp0, lp1, qR, lqR); \
        else                                                                                       \
            sweep_kernel<32, M, FCD_LOOKUP_SYMMETRIC><<<Ul, 32, 0, st>>>(WT, C, N, U, u0, lp0, lp1, qR, lqR); \
    } while (0)
    if (N <= 32) SWEEP_LAUNCH(1);
    else SWEEP_LAUNCH(2);
#undef SWEEP_LAUNCH
    return check_launch("fcd_estep_qR");
}

}  // extern "C"
