// Device-side bounded Newton solve of the (eta, epsilon) sub-problem.
//
// The reference minimises -E_lM(eta, epsilon) on [1e-5, 1 - 1e-5]^2 with scipy.optimize.minimize
// (fcdiff/fit.py:228-241): a host optimiser that needs the objective back on the CPU after every
// evaluation.  Each evaluation is one reduction kernel over the patient data (K3b); between two
// of them the GPU waits for a launch -> mapped-memory spin -> Python -> launch round trip, and
// with edge shards for one more exchange kernel.  Here the optimiser's step runs in the LAST CTA
// of the evaluation kernel itself: the partial sums are reduced (and exchanged over the peer
// windows when the edges are sharded), one thread takes a safeguarded projected Newton step on
// the two parameters and stores the next iterate in device memory, where the next evaluation --
// already enqueued behind this one -- reads it.  The host enqueues a batch of evaluations, waits
// once, and reads the state; launches after convergence exit at once.
//
// With y_l = A + eps_l D, A = (1 - p)/2, D = (3 p - 1)/2 the mixture weight relative to the
// total density (fit.py:427-430) and eps_0 = 1 - eps, eps_1 = eps, eps_2 = eta eps + (1 - eta)(1 - eps)
// (fit.py:433-444), every term of E_lM is w_l log y_l and, with g_l = D / y_l,
//     G_l = sum w_l g_l,   Q_l = sum w_l g_l^2
// give the gradient (the reference's fit.py:600-697) AND the Hessian of f = -E_lM:
//     df/d eta = -(2 eps - 1) G_2                     df/d eps = G_0 - G_1 - (2 eta - 1) G_2
//     d2f/d eta2 = (2 eps - 1)^2 Q_2                  d2f/d eps2 = Q_0 + Q_1 + (2 eta - 1)^2 Q_2
//     d2f/d eta d eps = (2 eps - 1)(2 eta - 1) Q_2 - 2 G_2
// An evaluation delivers {obj, ge, gh, qa, qb} = {sum w_l log y_l, sum s_l w_l g_l with
// s = (-1, 1, 2 eta - 1), G_2, Q_0 + Q_1, Q_2} and the higher moments sum w (s_l g_l)^k of the
// series model below (k = 3..kSolverK), from which one evaluation models the objective exactly up
// to the truncation of two one-dimensional series: the solve usually ends on the model of the first
// evaluation.  f is convex along each parameter (a sum of -log of affine functions), not jointly
// (eps_2 is bilinear): a step falls back to the diagonal when the 2 x 2 Hessian is not safely
// positive definite, never moves a parameter more than 3/4 of the way to 0 or 1 (the scale on which
// -log(A + eps D) changes), projects onto the box, and is halved back towards the last accepted
// iterate whenever the objective went up.
#pragma once

#include "fcd_comm.cuh"

namespace fcd {

struct SolverState {
    double x[2];          // (eta, epsilon) the NEXT evaluation is made at; the solution when done
    double xprev[2];      // last accepted iterate
    double fprev;         // objective there
    double f;             // objective at the last accepted iterate (when done on the series model: the model's
                          //   value at x)
    double g[2];          // gradient at the last evaluated point
    double lo[2], hi[2];  // box
    double tol;           // the solve ends on the series model when its remainder bound puts the model's minimiser
                          //   within tol^2 of the objective's, relative to min(x_i, 1 - x_i)
    double step;          // max |dx| of the last step
    int32_t have_prev;    // an accepted iterate exists
    int32_t nfev;         // evaluations consumed
    int32_t nback;        // consecutive halvings
    int32_t done;         // 1: converged; 2: stopped (backtracking exhausted / evaluation budget); 3: exchange timeout
    int32_t max_evals;
    int32_t pad_;
};

// Mapped host copy of the state, written after every evaluation: the state followed by the flag
// the host spins on (= the launch's sequence number).
struct SolverPublished {
    SolverState st;
    unsigned long long seq;
};

// Moments per series the evaluation kernels accumulate (A_k, B_k for k <= kSolverK) and the sums an
// evaluation delivers: obj, ge, gh, qa, qb, the theta-free part of E_lM, then A_3..A_K and B_3..B_K.
constexpr int kSolverK = 4;
constexpr int solver_vals(int K) { return 6 + 2 * (K - 2); }
constexpr int kSolverVals = solver_vals(kSolverK);
// Trust region of the series model: |d eps| G_01 <= rho and |d eps_2| G_2 <= rho (G_l bounds |g_l|)
constexpr double kSolverRho = 0.25;

#ifdef __CUDACC__
#define FCD_HD __host__ __device__
#else
#define FCD_HD
#endif

FCD_HD inline double solver_eps2(double eta, double eps) {
    double e2 = eta * eps;
    e2 += (1.0 - eta) * (1.0 - eps);                          // as sub_theta forms it
    return e2;
}

// The objective as a function of the three mixture scalars.  Every term is w log(A + eps_l D), and
// moving eps_l by d multiplies y_l by 1 + d g_l (g_l = D / y_l at the evaluated point), so with
// d eps_0 = -d eps_1 = -delta, d eps_2 = delta_2 (bilinear in eta, eps: no cross terms in the series)
//     f(eta', eps') = f - sum_k (-1)^(k+1) / k (delta^k A_k + delta_2^k B_k),
//     A_k = sum_{l < 2} w (s_l g_l)^k (s = -1, +1),   B_k = sum_{l = 2} w g_2^k,
// exactly but for the truncation of two one-dimensional series after K terms.  |g_l| <= G_l =
// max(1 / eps_l, 1 / (1 - eps_l)) (g is a Moebius function of p in [0, 1]) and for even K the net
// weights are non-negative (half records: the plane's l = 2 entry and the record's -q_s add up to
// 1 - q_s), so |A_k| <= G^(k-K) A_K and, with r = |delta| G < 1, the remainder of the value is at
// most |delta|^(K+1) G A_K / ((K+1)(1 - r)) and that of the slope |delta|^K G A_K / (1 - r).
template <int K>
struct SeriesModel {
    double a[K + 1], b[K + 1];                                // A_k, B_k (index 0 unused)
    double f, eps, e2, G01, G2;                               // at the evaluated point
};

template <int K>
FCD_HD inline SeriesModel<K> series_model(const double* sums, double eta, double eps, double f) {
    SeriesModel<K> m;
    const double th = 2.0 * eta - 1.0;
    m.a[0] = m.b[0] = 0.0;
    m.a[1] = sums[1] - th * sums[2];                          // ge carries the l = 2 part as (2 eta - 1) gh
    m.b[1] = sums[2];
    m.a[2] = sums[3];
    m.b[2] = sums[4];
    for (int k = 3; k <= K; ++k) {
        m.a[k] = sums[6 + (k - 3)];
        m.b[k] = sums[6 + (K - 2) + (k - 3)];
    }
    m.f = f;
    m.eps = eps;
    m.e2 = solver_eps2(eta, eps);
    m.G01 = fmax(1.0 / eps, 1.0 / (1.0 - eps));
    m.G2 = fmax(1.0 / m.e2, 1.0 / (1.0 - m.e2));
    return m;
}

// sum_{k <= K} (-1)^(k+1) d^k m_k / k and its first two derivatives in d
template <int K>
FCD_HD inline void series_sum(const double* mk, double d, double& v, double& d1, double& d2) {
    v = d1 = d2 = 0.0;
    double pk = 1.0;                                          // d^(k-1)
    double pk2 = 0.0;                                         // d^(k-2)
    for (int k = 1; k <= K; ++k) {
        const double c = (k & 1) ? mk[k] : -mk[k];
        d1 = fma(c, pk, d1);
        d2 = fma((double)(k - 1) * c, pk2, d2);
        v = fma(c * pk, d / (double)k, v);
        pk2 = pk;
        pk *= d;
    }
}

// the model's value, gradient and Hessian {H00, H01, H11} at z = (eta', eps')
template <int K>
FCD_HD inline double model_eval(const SeriesModel<K>& m, const double z[2], double g[2], double H[3]) {
    const double dA = z[1] - m.eps, dB = solver_eps2(z[0], z[1]) - m.e2;
    double va, a1, a2, vb, b1, b2;
    series_sum<K>(m.a, dA, va, a1, a2);
    series_sum<K>(m.b, dB, vb, b1, b2);
    const double te = 2.0 * z[1] - 1.0, th = 2.0 * z[0] - 1.0;   // d delta_2 / d eta', d delta_2 / d eps'
    g[0] = -b1 * te;
    g[1] = -(a1 + b1 * th);
    H[0] = -b2 * te * te;
    H[1] = -(b2 * te * th + 2.0 * b1);
    H[2] = -(a2 + b2 * th * th);
    return m.f - va - vb;
}

template <int K>
FCD_HD inline double model_radius(const SeriesModel<K>& m, const double z[2]) {
    return fmax(fabs(z[1] - m.eps) * m.G01, fabs(solver_eps2(z[0], z[1]) - m.e2) * m.G2);
}

// Remainder bounds at z: the largest relative error of the position the model's slope implies (the
// slope's remainder over the curvature, |delta|^K G^2 M_K (1 + r)^2 / ((1 - r) M_2), relative to
// 1 / G = min(eps_l, 1 - eps_l)), and the absolute error of the model's value.
template <int K>
FCD_HD inline void model_bounds(const SeriesModel<K>& m, const double z[2], double& pos, double& val) {
    const double d[2] = {fabs(z[1] - m.eps), fabs(solver_eps2(z[0], z[1]) - m.e2)};
    const double G[2] = {m.G01, m.G2}, M2[2] = {m.a[2], m.b[2]}, MK[2] = {fabs(m.a[K]), fabs(m.b[K])};
    pos = val = 0.0;
    for (int i = 0; i < 2; ++i) {
        const double r = d[i] * G[i];
        if (!(r < 1.0)) {
            pos = val = 1.7976931348623157e308;
            return;
        }
        double dk = 1.0;
        for (int k = 0; k < K; ++k) dk *= d[i];
        if (M2[i] > 0.0) pos = fmax(pos, dk * G[i] * G[i] * MK[i] * (1.0 + r) * (1.0 + r) / ((1.0 - r) * M2[i]));
        val += dk * d[i] * G[i] * MK[i] / ((K + 1) * (1.0 - r));
    }
}

// Safeguarded projected Newton point from x (gradient g, Hessian {H00, H01, H11}): active set at the
// box, the diagonal when the 2 x 2 Hessian is not safely positive definite, never more than 3/4 of
// the way to 0 or 1 (one common factor: the direction is kept), projection onto the box.
FCD_HD inline void newton_point(const SolverState& st, const double x[2], const double g[2], const double H[3],
                                double xn[2]) {
    const double H00 = H[0], H01 = H[1], H11 = H[2], Hd[2] = {H00, H11};
    bool fr[2];
    const double flat = 1e-14 * (H00 + H11);                  // a parameter the objective does not depend on stays put
    for (int i = 0; i < 2; ++i)                               // active set: at a bound with the gradient pointing out
        fr[i] = !((x[i] <= st.lo[i] && g[i] > 0.0) || (x[i] >= st.hi[i] && g[i] < 0.0)) && Hd[i] > flat;
    double d[2] = {0.0, 0.0};
    const double det = H00 * H11 - H01 * H01;
    if (fr[0] && fr[1] && det > 1e-8 * H00 * H11) {
        d[0] = -(H11 * g[0] - H01 * g[1]) / det;
        d[1] = -(H00 * g[1] - H01 * g[0]) / det;
    } else {
        for (int i = 0; i < 2; ++i)
            if (fr[i]) d[i] = -g[i] / Hd[i];
    }
    double a = 1.0;
    for (int i = 0; i < 2; ++i) {
        const double room = d[i] < 0.0 ? 0.75 * x[i] : 0.75 * (1.0 - x[i]);
        if (fabs(d[i]) > room) a = fmin(a, room / fabs(d[i]));
    }
    for (int i = 0; i < 2; ++i) xn[i] = fmin(st.hi[i], fmax(st.lo[i], x[i] + a * d[i]));
}

// One optimiser transition from the GLOBAL sums (layout of kSolverVals with K moments per series) of
// the evaluation made at st.x.  One thread.  (Plain C++: also compiled for the host, where the CPU
// tests drive it with NumPy-made sums; K = 2 is the quadratic model of the gradient and Hessian sums.)
//
// The first Newton step from the evaluated point is the step of the quadratic model.  If it leaves the
// trust region the model is not used: the step is taken as it is and evaluated.  Otherwise projected
// Newton runs on the series model to its minimiser; if the iteration leaves the region it stops on the
// boundary, and that point is evaluated next.  A minimiser strictly inside the region is the solution,
// without another evaluation, when the remainder bounds put it within tol^2 (relative) of the
// objective's and its value within 1e-12 of |f|.
template <int K>
FCD_HD inline void solver_step(SolverState& st, const double* sums) {
    const double eta = st.x[0], eps = st.x[1];
    const double obj = sums[0], ge = sums[1], G2 = sums[2], QA = sums[3], Q2 = sums[4], konst = sums[5];
    const double f = -(obj + konst);
    const double te = 2.0 * eps - 1.0;
    const double g0 = -te * G2, g1 = -ge;
    st.nfev += 1;
    st.g[0] = g0;
    st.g[1] = g1;
    if (!(fabs(f) <= 1.7976931348623157e308) || !(fabs(g0) + fabs(g1) + fabs(QA) + fabs(Q2) <= 1.7976931348623157e308)) {
        st.f = f;                                             // NaN / inf sums (non-finite inputs): nothing to iterate on
        st.done = 2;
        return;
    }
    if (st.have_prev && f > st.fprev + 1e-12 * fabs(st.fprev)) {
        // the objective went up: halve the step back towards the last accepted iterate
        if (++st.nback > 12 || st.nfev >= st.max_evals) {
            st.x[0] = st.xprev[0];
            st.x[1] = st.xprev[1];
            st.f = st.fprev;
            st.done = 2;
            return;
        }
        st.x[0] = st.xprev[0] + 0.5 * (st.x[0] - st.xprev[0]);
        st.x[1] = st.xprev[1] + 0.5 * (st.x[1] - st.xprev[1]);
        return;
    }
    st.nback = 0;
    const SeriesModel<K> m = series_model<K>(sums, eta, eps, f);
    const double x[2] = {eta, eps};
    double z[2] = {eta, eps}, gz[2] = {g0, g1}, Hz[3], fz = f;
    {
        double gx[2];
        model_eval<K>(m, z, gx, Hz);                          // the Hessian at x; the gradient as delivered
    }
    bool conv = false;
    for (int it = 0; it < 24; ++it) {
        double zn[2];
        newton_point(st, z, gz, Hz, zn);
        if (model_radius<K>(m, zn) > kSolverRho) {
            if (it == 0) {                                    // beyond the model's region: the quadratic model's step
                z[0] = zn[0];
                z[1] = zn[1];
                break;
            }
            double in = 0.0, out = 1.0;                       // stop on the boundary
            for (int j = 0; j < 24; ++j) {
                const double a = 0.5 * (in + out);
                const double za[2] = {z[0] + a * (zn[0] - z[0]), z[1] + a * (zn[1] - z[1])};
                if (model_radius<K>(m, za) > kSolverRho) out = a;
                else in = a;
            }
            z[0] += in * (zn[0] - z[0]);
            z[1] += in * (zn[1] - z[1]);
            break;
        }
        double gn[2], Hn[3];
        double fn = model_eval<K>(m, zn, gn, Hn);
        for (int j = 0; j < 30 && fn > fz + 1e-14 * fabs(fz); ++j) {   // the model went up: halve the step
            zn[0] = 0.5 * (z[0] + zn[0]);
            zn[1] = 0.5 * (z[1] + zn[1]);
            fn = model_eval<K>(m, zn, gn, Hn);
        }
        double srel = 0.0;
        for (int i = 0; i < 2; ++i) srel = fmax(srel, fabs(zn[i] - z[i]) / fmin(z[i], 1.0 - z[i]));
        z[0] = zn[0];
        z[1] = zn[1];
        fz = fn;
        gz[0] = gn[0];
        gz[1] = gn[1];
        Hz[0] = Hn[0];
        Hz[1] = Hn[1];
        Hz[2] = Hn[2];
        if (srel <= 1e-12) {                                  // Newton converges quadratically: z is the minimiser
            conv = true;
            break;
        }
    }
    st.step = fmax(fabs(z[0] - x[0]), fabs(z[1] - x[1]));
    st.xprev[0] = x[0];
    st.xprev[1] = x[1];
    st.fprev = f;
    st.have_prev = 1;
    st.x[0] = z[0];
    st.x[1] = z[1];
    if (conv) {
        double pos, val;
        model_bounds<K>(m, z, pos, val);
        if (pos <= st.tol * st.tol && val <= 1e-12 * fabs(fz)) {
            st.f = fz;
            st.done = 1;
            return;
        }
    }
    st.f = f;
    if (st.nfev >= st.max_evals) {                            // budget: stay at the evaluated point
        st.x[0] = x[0];
        st.x[1] = x[1];
        st.done = 2;
    }
}

#ifdef __CUDACC__
// theta_sub-dependent constants of an evaluation, formed by every thread from the iterate
struct SubTheta {
    double eta, epsilon;
    double al[3], bl[3];
};
__device__ __forceinline__ SubTheta sub_theta(double eta, double epsilon) {
    SubTheta t;
    t.eta = eta;
    t.epsilon = epsilon;
    double e2 = eta * epsilon;
    e2 += (1.0 - eta) * (1.0 - epsilon);                      // fit.py:442-443
    const double epsl[3] = {1.0 - epsilon, epsilon, e2};
#pragma unroll
    for (int l = 0; l < 3; ++l) {
        t.al[l] = (1.0 - epsl[l]) * 0.5;
        t.bl[l] = epsl[l] - t.al[l];
    }
    return t;
}

// Moments of the series model an evaluation accumulates: a[k - 2] = A_k, b[k - 2] = B_k, k = 2..K
struct SolverMoments {
    double a[kSolverK - 1], b[kSolverK - 1];
};
static_assert(kSolverK >= 2 && kSolverK <= 8 && kSolverK % 2 == 0, "the remainder bound needs an even K");

// m[k - 2] += x^k, k = 2..K (elements of weight 1: a power tree, one instruction per moment)
__device__ __forceinline__ void add_powers1(double* m, double x) {
    const double x2 = x * x, x3 = x2 * x;
    m[0] += x2;
    if (kSolverK >= 3) m[1] += x3;
    if (kSolverK >= 4) m[2] = fma(x2, x2, m[2]);
    if (kSolverK >= 5) m[3] = fma(x3, x2, m[3]);
    if (kSolverK >= 6) m[4] = fma(x3, x3, m[4]);
    if (kSolverK >= 7) {
        const double x4 = x2 * x2;
        m[5] = fma(x4, x3, m[5]);
        m[6] = fma(x4, x4, m[6]);
    }
}

// m[k - 2] += w x^k, k = 2..K
__device__ __forceinline__ void add_powers(double* m, double w, double x) {
    double pw = w * x;
#pragma unroll
    for (int k = 2; k <= kSolverK; ++k) {
        pw *= x;
        m[k - 2] += pw;
    }
}

// The values the last CTA reduces: {obj, ge, gh, A_2, B_2, (slot of the theta-free part), A_3.., B_3..}
__device__ __forceinline__ void solver_sums(double obj, double ge, double gh, const SolverMoments& mo,
                                            double (&v)[kSolverVals]) {
    v[0] = obj;
    v[1] = ge;
    v[2] = gh;
    v[3] = mo.a[0];
    v[4] = mo.b[0];
    v[5] = 0.0;
#pragma unroll
    for (int k = 3; k <= kSolverK; ++k) {
        v[6 + (k - 3)] = mo.a[k - 2];
        v[6 + (kSolverK - 2) + (k - 3)] = mo.b[k - 2];
    }
}

__device__ __forceinline__ void solver_publish(const SolverState& st, SolverPublished* pub, unsigned long long seq) {
    if (pub == nullptr) return;
    const double* src = reinterpret_cast<const double*>(&st);
    double* dst = reinterpret_cast<double*>(&pub->st);
    static_assert(sizeof(SolverState) % 8 == 0, "SolverState is copied as doubles");
#pragma unroll
    for (int i = 0; i < (int)(sizeof(SolverState) / 8); ++i) st_relaxed_sys(dst + i, src[i]);
    __threadfence_system();
    st_release_sys(&pub->seq, seq);
}

// Epilogue of an evaluation kernel, run by ALL threads of the CTA that arrived last: s_sums holds
// this rank's sums (shared memory, kSolverVals slots, slot 5 free); the theta-free part of E_lM is
// read from konst_dev (this rank's share) into slot 5; exchange, step, publication.
__device__ __forceinline__ void solver_epilogue(double* s_sums, SolverState* state, const double* konst_dev,
                                                const CommPeers& peers, int rank, int world,
                                                SolverPublished* pub, unsigned long long seq) {
    if (threadIdx.x == 0) s_sums[5] = konst_dev ? *konst_dev : 0.0;
    __syncthreads();
    const bool ok = comm_exchange_cta(s_sums, kSolverVals, peers, rank, world, kCommSpinCycles);
    if (threadIdx.x == 0) {
        SolverState st = *state;
        if (ok) solver_step<kSolverK>(st, s_sums);
        else st.done = 3;
        *state = st;
        __threadfence();
        solver_publish(st, pub, seq);
    }
}

// A launch made after the solve has finished: publishes the (unchanged) state and exits.
__device__ __forceinline__ bool solver_finished(const SolverState* state, SolverPublished* pub, unsigned long long seq) {
    const int done = *reinterpret_cast<const volatile int32_t*>(&state->done);
    if (done && blockIdx.x == 0 && threadIdx.x == 0) solver_publish(*state, pub, seq);
    return done != 0;
}
#endif  // __CUDACC__

}  // namespace fcd
