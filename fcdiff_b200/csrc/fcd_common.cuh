// Shared device/host helpers for the fcdiff_b200 kernels (sm_100a).
//
// Reference formulas are cited as fcdiff/<file>:<line> (reference tree).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "fcdiff_b200.h"
#include "fcd_math.cuh"

namespace fcd {

// ---------------------------------------------------------------- host side
void set_error(const char* fmt, ...);
int  check_launch(const char* what);          // counts the launch, maps cudaGetLastError
int  sm_count();

#define FCD_REQUIRE(cond, ...)                                                   \
    do {                                                                         \
        if (!(cond)) {                                                           \
            ::fcd::set_error(__VA_ARGS__);                                       \
            return -1;                                                           \
        }                                                                        \
    } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel: the opt-in is made
// once per (call site, device), so a process that drives several GPUs gets it on each of them.
#define FCD_ALLOW_BIG_SMEM(...)                                                                          \
    do {                                                                                                 \
        static bool done_[64] = {false};                                                                 \
        int dev_ = -1;                                                                                   \
        if (cudaGetDevice(&dev_) != cudaSuccess || dev_ < 0 || dev_ >= 64 || !done_[dev_]) {             \
            cudaFuncSetAttribute(__VA_ARGS__, cudaFuncAttributeMaxDynamicSharedMemorySize,               \
                                 (int)::fcd::kSmemBudget);                                               \
            if (dev_ >= 0 && dev_ < 64) done_[dev_] = true;                                              \
        }                                                                                                \
    } while (0)

constexpr double kHalfLog2Pi = 0.91893853320467274178032973640562;   // log(sqrt(2 pi))

// Workspace layout (doubles): [0, kWsPartials) per-CTA partial sums,
// then one 64-bit slot holding the arrival ticket, then 16 scratch doubles.
constexpr int     kMaxReduceBlocks = 2048;
constexpr int     kMaxReduceVals   = 16;
constexpr int64_t kWsPartials      = (int64_t)kMaxReduceBlocks * kMaxReduceVals;
constexpr int64_t kWsScratch       = kWsPartials + 2;      // 16 doubles of scratch for chained reductions
constexpr int64_t kWsDoubles       = kWsScratch + 16;

// Derived per-theta constants, passed by value to kernels (__grid_constant__).
struct ThetaDev {
    double mu[3];
    double isig[3];      // 1 / sigma_k
    double lc[3];        // -log(sigma_k)            (the -log sqrt(2 pi) is added where needed)
    double epsl[3];      // eps_l of fcdiff/fit.py:433-444
    double al[3];        // (1 - eps_l) / 2
    double bl[3];        // eps_l - a_l
    double log_gamma[3];
    double hq_a[3];      // healthy quadratic: sum_h logN_k(b) = hq_a*S2 + hq_b*S1 + hq_c
    double hq_b[3];
    double hq_c[3];
    double eta;
    double epsilon;
    double log_pi2[2];
    double hq_c1[3];     // hq_c of one control: the masked form takes H_c * hq_c1 with H_c = S0[c] observed controls
};

ThetaDev make_theta_dev(const fcd_theta& th, int H);

// ---------------------------------------------------------------- device side
#ifdef __CUDACC__

// util.c_to_nm (fcdiff/util.py:82-84) with an exact integer correction of the
// floating-point square root.
__host__ __device__ inline void c_to_nm(int64_t c, int& n, int& m) {
    int64_t nn = (int64_t)((sqrt((double)(8 * c + 1)) - 1.0) * 0.5) + 1;
    while (nn * (nn - 1) / 2 > c) --nn;
    while ((nn + 1) * nn / 2 <= c) ++nn;
    n = (int)nn;
    m = (int)(c - nn * (nn - 1) / 2);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// 128-bit streaming load of two doubles (read-only path, no L1 allocation).
__device__ __forceinline__ double2 ldg_stream2(const double* p) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];"
                 : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ double ldg_stream1(const double* p) {
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
    return r;
}

// Per-element core shared by K2 / K2b / K3 / K4: the *responsibility planes*.
//
// For x = bt[c,u]:   N_k = N(x; mu_k, sigma_k)                      (fit.py:115)
//                    p_k = N_k / (N_0 + N_1 + N_2),   L = log(N_0 + N_1 + N_2).
// Then, with a_l = (1 - eps_l)/2 and b_l = eps_l - a_l,
//     M_kl = eps_l N_k + a_l sum_{j != k} N_j = (a_l + b_l p_k) exp(L)   (fit.py:427-430)
//     log M_kl = L + log(a_l + b_l p_k)                                  (fit.py:117-122)
// exactly, without the underflow of the reference's pdf in the far tails.
// p_k and L depend on (x, mu, sigma) only and the reference never re-estimates
// mu, sigma (fit.py:232-237): resp_cache_kernel takes the exponentials ONCE per
// fit and stores the planes P0, P1, P2 and L ([C][pitchU] each); every later
// pass reads planes.  All dependence on (eta, epsilon) is in (a_l, b_l), and the
// theta-free term sum w L is summed separately (elm_const_kernel).
//
// Tiers.  The posteriors of this model are sharply peaked: q_F[c,:] is one-hot to
// rounding for (practically) every edge and q_R[n,u,:] for ~95 % of the
// (region, patient) pairs.  A weight below kPeakTau = 2^-60 multiplies a log of
// magnitude <= 14: dropping the term changes a sum of O(1) terms by less than
// its own rounding error.  The peak-state bytes (peak_states_*_kernel)
//   fstate[c]   = k* if q_F[c,k*] == 1.0 exactly and the others <= 2^-60, else 3
//   rstate[n,u] = s  if q_R[n,u,s] == 1.0 exactly and the other  <= 2^-60, else 2 (3 if the pair
//                 does not sum to 1 within 2^-50: user-assigned, unnormalised), 4 in the padding column
// let the kernels take, per element,
//   T1: edge and both regions peaked -> ONE plane (k*), ONE log (l* from 2 bytes);
//   T2: edge peaked, a region not    -> k* plane, 3 logs, real pair weights;
//   T3: edge not peaked              -> 3 planes, 9 logs (the reference's form).
// T1 runs for all lanes of a warp; T2 elements are compacted into a per-warp
// queue in shared memory and evaluated 32 at a time, so that the rare expensive
// elements do not drag whole warps into the slow path.
constexpr double kPeakTau = 8.673617379884035e-19;        // 2^-60
constexpr int kStateMixedR = 2, kStateLooseR = 3, kStateDead = 4, kStateMixedF = 3;

struct Resp {
    double p[3];
    double L;
};

__device__ __forceinline__ Resp resp_eval(double x, const ThetaDev& th) {
    double t[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double z = (x - th.mu[k]) * th.isig[k];
        t[k] = fma(-0.5 * z, z, th.lc[k]);
    }
    const double tmax = fmax(t[0], fmax(t[1], t[2]));
    double e[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) e[k] = (t[k] == tmax) ? 1.0 : exp_nonpos(t[k] - tmax);
    const double S = e[0] + e[1] + e[2];
    const double inv = 1.0 / S;
    Resp r;
#pragma unroll
    for (int k = 0; k < 3; ++k) r.p[k] = e[k] * inv;
    r.L = (tmax - kHalfLog2Pi) + log(S);
    return r;
}

// a_l + b_l p: the mixture weight relative to the total density
__device__ __forceinline__ double mix_rel(const ThetaDev& th, int l, double p) { return fma(th.bl[l], p, th.al[l]); }

// numerator of d log M_kl / d eps_l relative to the total density (fit.py:618-697)
__device__ __forceinline__ double mix_num(double p) { return fma(1.5, p, -0.5); }

// q_R pair weights of fcdiff/fit.py:382-406.
__device__ __forceinline__ void pair_weights(double2 qn, double2 qm, double (&w)[3]) {
    w[0] = qn.x * qm.x;
    w[1] = qn.y * qm.y;
    w[2] = fma(qn.y, qm.x, qn.x * qm.y);
}

__device__ __forceinline__ double sel3(int l, const double (&v)[3]) { return l == 0 ? v[0] : (l == 1 ? v[1] : v[2]); }

// ---------------------------------------------------------------- K2 row end
// Healthy term of edge c, sum_h log N_k(b[c,h]) = hq_a S2 + hq_b S1 + hq_c (fit.py:111-114, 171).  MASKED: the
// sums run over the S0 = H_c observed controls of the edge and the constant is H_c hq_c1; hq_c1 = hq_c / (-H) up to
// the sign only (make_theta_dev), so S0 = H gives the bits of the unmasked form.
template <bool MASKED>
__device__ __forceinline__ double healthy_term(const ThetaDev& th, int k, double s1, double s2, double s0) {
    return fma(th.hq_a[k], s2, fma(th.hq_b[k], s1, MASKED ? __dmul_rn(s0, th.hq_c1[k]) : th.hq_c[k]));
}

// lane 0 of the warp that owns edge c: log gamma + healthy quadratic + A, then
// scipy.special.logsumexp: a_max + log(sum exp(a - a_max))           (fit.py:165-174)
template <bool MASKED = false>
__device__ __forceinline__ void k2_finish(int64_t c, const double (&A)[3], double s1, double s2, double s0,
                                          const ThetaDev& th, double* __restrict__ lqF,
                                          double* __restrict__ qF) {
    double l[3];
#pragma unroll
    for (int k = 0; k < 3; ++k)
        l[k] = th.log_gamma[k] + healthy_term<MASKED>(th, k, s1, s2, s0) + A[k];
    const double mx = fmax(l[0], fmax(l[1], l[2]));
    const double lse = mx + log(exp(l[0] - mx) + exp(l[1] - mx) + exp(l[2] - mx));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double v = l[k] - lse;
        lqF[c * 3 + k] = v;
        if (qF) qF[c * 3 + k] = exp(v);
    }
}


// ---------------------------------------------------------------- mbarrier / TMA helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// 1-D bulk copy global -> shared through the TMA unit (dst, src 16-byte aligned,
// bytes a multiple of 16); completion is signalled on `bar` (complete_tx).
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------- tiered streaming walker
// The plane kernels are HBM-streaming with a few fp64 instructions per element,
// so the bytes in flight must not be limited by registers: the rows are staged
// through shared memory by the TMA unit.  One persistent CTA of NCW warps per
// SM.  Warp g (grid-wide index) owns the edge rows c = g, g + G, ...; a row is cut
// into segments of SEG patients.  Every warp runs its own ring of D stages: lane
// 0 issues, per segment, one 1-D bulk copy per plane (NPL planes starting at
// plane fstate[c] when USE_K) and one for each of the two regions' peak-state
// rows, all completing on the stage's mbarrier, and stores {k, n | m << 16} beside
// them; after a stage has been consumed (by the same warp: no "empty" barrier is
// needed) the segment D steps ahead is issued into it.
//   live(pv, lp, e)              T1 body for element e (0 / 1) of a 64-patient chunk, all lanes,
//                                branch-free: lp = l* in 0..2, or 3 for deferred / padding
//                                slots (the kernels map 3 to constants that contribute 0);
//                                e selects one of two independent accumulator sets (ILP);
//   dload(c, u, n, m, k, ok)     loads the operands of one queued element (T2) and returns
//   dcompute(ops)                them; evaluation of up to 4 x 32 queued elements at a time,
//                                all loads issued before the first evaluation;
//   full(c, n, m, u0, u1)        rows with fstate == 3 (T3), patients [u0, u1), from global;
//   row_end(c)                   after the last segment of a row (its deferred elements
//                                have been evaluated when ROW_DRAIN).
// Requirements: planes 16-byte aligned with even pitchU and planeStride, pitchS a
// multiple of 256 with rstate == 4 in [U, pitchS), U < 65536, fewer than 65536 rows
// per warp.
template <int NPL, int SEG>
struct StreamGeom {
    static constexpr int kStageBytes = NPL * SEG * 8 + 2 * SEG;
    static constexpr int kDrainAt = 96;                      // queued elements that trigger an evaluation (<= 4 x 32)
    static constexpr int kQueueSlots = SEG + kDrainAt <= 256 ? 256 : 512;    // >= kDrainAt - 1 + SEG entries (4 B each)
    static_assert(SEG % 64 == 0 && SEG + kDrainAt - 1 <= kQueueSlots, "bad segment");
    // bytes of dynamic shared memory after the log table, for ncw warps and d stages
    static constexpr size_t bytes(int ncw, int d) {
        return (size_t)ncw * ((size_t)kQueueSlots * 4 + (size_t)d * (kStageBytes + 16 + 16));
    }
};

constexpr int kStreamWarps = 16;
constexpr int kStreamThreads = kStreamWarps * 32;
// dynamic shared memory of one CTA (1 CTA / SM): the 227 KB opt-in limit minus 2 KB for the kernels' static
// shared memory (tables, reduction scratch: up to ~1.2 KB) -- the opt-in is refused if static + dynamic exceed it
constexpr size_t kSmemBudget = 225 * 1024;

// Ring depth that fits next to `other` bytes (log table) in the CTA's shared memory; 0 if none does.
template <int NPL, int SEG>
inline int stream_depth(size_t other) {
    using G = StreamGeom<NPL, SEG>;
    for (int d = 8; d >= 2; --d)
        if (other + G::bytes(kStreamWarps, d) <= kSmemBudget) return d;
    return 0;
}

template <int NPL, int SEG, int NCW, bool ROW_DRAIN, bool USE_K, class LiveFn, class DLoadFn, class DComputeFn,
          class FullFn, class RowEndFn>
__device__ __forceinline__ void stream_tiered(const double* __restrict__ P, int64_t planeStride,
                                              int64_t C, int U, int64_t pitchU,
                                              const uint8_t* __restrict__ fstate,
                                              const uint8_t* __restrict__ rstate, int64_t pitchS,
                                              const int32_t* __restrict__ nm, unsigned char* smem, int D,
                                              LiveFn&& live, DLoadFn&& dload, DComputeFn&& dcompute,
                                              FullFn&& full, RowEndFn&& row_end) {
    using G = StreamGeom<NPL, SEG>;
    static_assert(256 % SEG == 0, "state rows are padded to a multiple of 256");
    constexpr int QS = G::kQueueSlots;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* queue = reinterpret_cast<uint32_t*>(smem) + warp * QS;
    unsigned char* ring = smem + (size_t)NCW * QS * 4 + (size_t)warp * D * G::kStageBytes;
    int4* descs = reinterpret_cast<int4*>(smem + (size_t)NCW * QS * 4 + (size_t)NCW * D * G::kStageBytes) + warp * D;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)NCW * QS * 4 +
                                                 (size_t)NCW * D * (G::kStageBytes + 16)) + warp * D;
    // the rings start zeroed: lanes beyond the copied bytes of a short segment read
    // stale but valid responsibilities (their contribution is masked)
    for (int i = lane; i < D * G::kStageBytes / 16; i += 32) reinterpret_cast<int4*>(ring)[i] = make_int4(0, 0, 0, 0);
    if (lane < D) mbar_init(bars + lane, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();

    const int nseg = (U + SEG - 1) / SEG;
    const int64_t nW = (int64_t)gridDim.x * NCW;
    const int64_t c_first = (int64_t)blockIdx.x * NCW + warp;

    // ---- issue side (warp-uniform state; lane 0 talks to the TMA unit)
    int64_t pc = c_first;
    int ps = 0, pd = 0;                                      // next segment / ring slot to issue
    int cur_nm = 0, cur_k = 0, nxt_nm = 0, nxt_k = 0;
    if (pc < C) {
        cur_nm = __ldg(nm + pc);
        cur_k = USE_K ? (int)__ldg(fstate + pc) : 0;
        if (pc + nW < C) {
            nxt_nm = __ldg(nm + pc + nW);
            nxt_k = USE_K ? (int)__ldg(fstate + pc + nW) : 0;
        }
    }
    auto issue = [&]() {
        if (pc >= C) return;
        const int d = pd;
        if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // the warp's reads of this slot are done
            descs[d] = make_int4(cur_k, cur_nm, 0, 0);
            const int u0 = ps * SEG;
            const int np = (int)(pitchU - u0 < SEG ? pitchU - u0 : SEG);
            constexpr int ns = SEG;                                   // pitchS is a multiple of SEG
            const bool planes = cur_k < 3;
            mbar_expect_tx(bars + d, (uint32_t)(2 * ns + (planes ? NPL * np * 8 : 0)));
            unsigned char* st = ring + (size_t)d * G::kStageBytes;
            if (planes) {
                const double* src = P + (int64_t)cur_k * planeStride + pc * pitchU + u0;
#pragma unroll
                for (int i = 0; i < NPL; ++i)
                    tma_load_1d(st + i * SEG * 8, src + i * planeStride, (uint32_t)(np * 8), bars + d);
            }
            tma_load_1d(st + NPL * SEG * 8, rstate + (int64_t)(cur_nm & 0xffff) * pitchS + u0, (uint32_t)ns, bars + d);
            tma_load_1d(st + NPL * SEG * 8 + SEG, rstate + (int64_t)((cur_nm >> 16) & 0xffff) * pitchS + u0,
                        (uint32_t)ns, bars + d);
        }
        if (++pd == D) pd = 0;
        if (++ps == nseg) {
            ps = 0;
            pc += nW;
            cur_nm = nxt_nm;
            cur_k = nxt_k;
            if (pc + nW < C) {
                nxt_nm = __ldg(nm + pc + nW);
                nxt_k = USE_K ? (int)__ldg(fstate + pc + nW) : 0;
            }
        }
    };
    for (int i = 0; i < D; ++i) issue();

    // ---- consume side
    const unsigned lt = (1u << lane) - 1u;
    int qhead = 0, qtail = 0, row = 0, d = 0;
    uint32_t phase = 0;
    for (int64_t c = c_first; c < C; c += nW, ++row) {
        for (int s = 0; s < nseg; ++s) {
            mbar_wait(bars + d, phase);
            const int4 ds = descs[d];
            const int k = ds.x, n = ds.y & 0xffff, m = (ds.y >> 16) & 0xffff;
            const unsigned char* st = ring + (size_t)d * G::kStageBytes;
            if (USE_K && k == 3) {
                const int u1 = (s + 1) * SEG < U ? (s + 1) * SEG : U;
                full(c, n, m, s * SEG, u1);
            } else {
#pragma unroll
                for (int j = 0; j < SEG / 64; ++j) {
                    const int u0 = s * SEG + 64 * j;
                    if (u0 < U) {                                     // warp-uniform
                        double2 p2[NPL];
#pragma unroll
                        for (int i = 0; i < NPL; ++i)
                            p2[i] = *reinterpret_cast<const double2*>(st + i * SEG * 8 + (64 * j + 2 * lane) * 8);
                        const uint32_t sn2 = *reinterpret_cast<const unsigned short*>(st + NPL * SEG * 8 + 64 * j + 2 * lane);
                        const uint32_t sm2 =
                            *reinterpret_cast<const unsigned short*>(st + NPL * SEG * 8 + SEG + 64 * j + 2 * lane);
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int sn = (sn2 >> (8 * e)) & 0xff;
                            const int sm = (sm2 >> (8 * e)) & 0xff;
                            const int o = sn | sm;                    // 0/1 peaked pair, 2/3 mixed, >= 4 padding
                            const int lp = o < 2 ? (((sn ^ sm) << 1) + (sn & sm)) : 3;
                            const bool mixed = (o & 6) == 2;
                            double pv[NPL];
#pragma unroll
                            for (int i = 0; i < NPL; ++i) pv[i] = e ? p2[i].y : p2[i].x;
                            live(pv, lp, e);
                            const unsigned bal = __ballot_sync(0xffffffffu, mixed);       // branch-free push
                            if (mixed)
                                queue[(qtail + __popc(bal & lt)) & (QS - 1)] =
                                    ((uint32_t)row << 16) | (uint32_t)(u0 + 2 * lane + e);
                            qtail += __popc(bal);
                        }
                    }
                }
            }
            __syncwarp();
            issue();                                                  // refill this stage D segments ahead
            const bool row_done = s == nseg - 1;
            const int at_least = (row_done && (ROW_DRAIN || c + nW >= C)) ? 1 : G::kDrainAt;
            while (qtail - qhead >= at_least) {                       // the one deferred call site
                const int cnt = qtail - qhead < 128 ? qtail - qhead : 128;
                decltype(dload((int64_t)0, 0, 0, 0, 0, false)) ops[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    if (b * 32 < cnt) {                               // warp-uniform
                        const int idx = qhead + b * 32 + lane;
                        const bool ok = idx < qtail;
                        uint32_t e = 0;
                        if (ok) e = queue[idx & (QS - 1)];
                        const int64_t ce = c_first + (int64_t)(e >> 16) * nW;
                        int v = 0, ke = 0;
                        if (ok) {
                            v = __ldg(nm + ce);
                            if (USE_K) ke = __ldg(fstate + ce);
                        }
                        ops[b] = dload(ce, (int)(e & 0xffff), v & 0xffff, (v >> 16) & 0xffff, ke, ok);
                    }
                }
#pragma unroll
                for (int b = 0; b < 4; ++b)
                    if (b * 32 < cnt) dcompute(ops[b]);
                qhead += cnt;
                __syncwarp();
            }
            if (row_done) row_end(c);
            if (++d == D) {
                d = 0;
                phase ^= 1;
            }
        }
    }
}

// Deterministic grid reduction: every CTA reduces NV values, writes its partial
// to ws[blockIdx.x*NV + i]; the CTA that arrives last sums the partials in a
// fixed order and writes out[0..NV).  The ticket (ws[kWsPartials]) is restored
// to zero.  Must be called by all threads of the block.
template <int NV, int THREADS>
__device__ __forceinline__ void grid_reduce_store(double (&v)[NV], double* ws, double* out) {
    static_assert(NV <= kMaxReduceVals, "too many values");
    __shared__ double s_part[NV][THREADS / 32];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        double x = warp_sum(v[i]);
        if (lane == 0) s_part[i][warp] = x;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            double x = (lane < THREADS / 32) ? s_part[i][lane] : 0.0;
            x = warp_sum(x);
            if (lane == 0) ws[(int64_t)blockIdx.x * NV + i] = x;
        }
    }
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(ws + kWsPartials);
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned long long t = atomicAdd(ticket, 1ull);
        s_last = (t == (unsigned long long)gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double acc[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += THREADS) {
#pragma unroll
        for (int i = 0; i < NV; ++i) acc[i] += __ldcg(ws + (int64_t)b * NV + i);
    }
    __syncthreads();      // s_part reuse
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        double x = warp_sum(acc[i]);
        if (lane == 0) s_part[i][warp] = x;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            double x = (lane < THREADS / 32) ? s_part[i][lane] : 0.0;
            x = warp_sum(x);
            if (lane == 0) out[i] = x;
        }
        if (lane == 0) *ticket = 0ull;
    }
}

// Same reduction, but the sums stay in the CTA that arrived last: returns true there (for all of
// its threads, with s_out[0..NV) valid in shared memory after the internal barrier) and false in
// every other CTA.  For kernels whose last CTA continues with an epilogue (fcd_solver.cuh).
// The warp partials go through shared memory in rounds of at most 8 values: the static shared memory
// stays inside the 2 KB that kSmemBudget leaves for it whatever NV is.
template <int NV, int THREADS>
__device__ __forceinline__ void cta_sum_rounds(const double (&v)[NV], double (*s_part)[THREADS / 32], double* dst) {
    constexpr int R = NV < 8 ? NV : 8;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int r0 = 0; r0 < NV; r0 += R) {
#pragma unroll
        for (int i = r0; i < r0 + R && i < NV; ++i) {
            double x = warp_sum(v[i]);
            if (lane == 0) s_part[i - r0][warp] = x;
        }
        __syncthreads();
        if (warp == 0) {
#pragma unroll
            for (int i = r0; i < r0 + R && i < NV; ++i) {
                double x = (lane < THREADS / 32) ? s_part[i - r0][lane] : 0.0;
                x = warp_sum(x);
                if (lane == 0) dst[i] = x;
            }
        }
        if (r0 + R < NV) __syncthreads();          // s_part reuse
    }
}

template <int NV, int THREADS>
__device__ __forceinline__ bool grid_reduce_last(double (&v)[NV], double* ws, double* s_out) {
    static_assert(NV <= kMaxReduceVals, "too many values");
    __shared__ double s_part[NV < 8 ? NV : 8][THREADS / 32];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    cta_sum_rounds<NV, THREADS>(v, s_part, ws + (int64_t)blockIdx.x * NV);
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(ws + kWsPartials);
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned long long t = atomicAdd(ticket, 1ull);
        s_last = (t == (unsigned long long)gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return false;
    __threadfence();
    double acc[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += THREADS) {
#pragma unroll
        for (int i = 0; i < NV; ++i) acc[i] += __ldcg(ws + (int64_t)b * NV + i);
    }
    __syncthreads();      // s_part reuse
    cta_sum_rounds<NV, THREADS>(acc, s_part, s_out);
    if (warp == 0 && lane == 0) *ticket = 0ull;
    __syncthreads();
    return true;
}

#endif  // __CUDACC__

}  // namespace fcd
