// K2 (coded), row-group form: the E-step q_F of fcdiff/fit.py:157-174 from the code plane of the previous
// M-step, like estep_qF_coded_kernel (fcd_estep.cu) -- same inputs, same arithmetic per element -- with the
// rows mapped onto the warp differently.
//
// estep_qF_coded_kernel gives a warp ONE row at a time: 500 patients are 16 elements per lane, and every row
// pays the row-level work on top -- four TMA issues, three warp reductions, a flush of the running products,
// the row's half records by two lanes each: ~990 warp-instructions per row of which a third is the element
// loop (profiles/r02b_estep_qF_coded_lines.txt).  Here a warp takes a GROUP of eight consecutive rows, four
// lanes per row:
//   * one 2-D TMA tile per plane (eight rows x 32 patients of p_0, p_1 and the code bytes: three
//     cp.async.bulk.tensor.2d per stage of 4352 bytes) instead of three 1-D copies per row and segment;
//   * a lane walks its row's patients two at a time (one 16-byte read per plane); the row's three running
//     products stay in the lane's registers for the whole row;
//   * the four lanes of a row are combined by two shuffle rounds once per ROW GROUP; 32 rows (four groups)
//     are normalised at once, one lane per row (the exp / log of fit.py:174);
//   * the half records and the records of a row are taken by the row's four lanes after the group.
// One persistent CTA of eight warps per SM, per-warp ring of stages, mbarrier per stage.
#include <cuda.h>

#include <cstdlib>

#include "fcd_estep_rows.cuh"

namespace fcd {

constexpr int kRwRows = 8;                                   // rows per warp group
constexpr int kRwSeg = 32;                                   // patients per stage
constexpr int kRwPlane = kRwRows * kRwSeg * 8;               // 2048 bytes of one plane's tile
constexpr int kRwStage = 2 * kRwPlane + kRwRows * kRwSeg;    // p_0, p_1, codes: 4352 bytes (a multiple of 128)
constexpr int kRwMaxDepth = 6;
constexpr size_t rw_ring_bytes(int depth, int nw) { return (size_t)nw * depth * (kRwStage + 8) + 128; }

__device__ __forceinline__ void rw_tma_2d(uint32_t dst, const CUtensorMap* map, int x, int y, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(bar) : "memory");
}

template <bool FAST, int NW, bool MASKED>
__global__ void __launch_bounds__(NW * 32, 1)
estep_qF_rows_kernel(const __grid_constant__ CUtensorMap map_p0, const __grid_constant__ CUtensorMap map_p1,
                     const __grid_constant__ CUtensorMap map_code,
                     const double* __restrict__ S1, const double* __restrict__ S2, const double* __restrict__ S0,
                     const double* __restrict__ P, int64_t planeStride, int64_t C, int U, int64_t pitchU,
                     const double* __restrict__ qR, const int32_t* __restrict__ nm,
                     const int2* __restrict__ counts, const unsigned long long* __restrict__ keysF,
                     const unsigned long long* __restrict__ keysH, const longlong2* __restrict__ rowoff,
                     const double2* __restrict__ Hh,
                     const __grid_constant__ ThetaDev th, const __grid_constant__ LogTabWindow tab, int depth,
                     double* __restrict__ lqF, double* __restrict__ qF) {
    extern __shared__ __align__(128) double s_dyn[];
    __shared__ double2 s_lc[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // table first, then the rings (128-byte aligned: TMA tile destinations)
    const size_t toff = FAST ? (((size_t)tab.n * 8 + 127) & ~(size_t)127) : 0;
    unsigned char* ring0 = reinterpret_cast<unsigned char*>(s_dyn) + toff;
    unsigned char* ring = ring0 + (size_t)warp * depth * kRwStage;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring0 + (size_t)NW * depth * kRwStage) + warp * depth;
    if (lane < depth) mbar_init(bars + lane, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // per-code constants {a_l, b_l}; code 3 is neutral: the factor 1 + 0 p = 1 exactly; the codes 4, 5
    // (one undecided region) count as l = 2 here, their correction comes from the half records
    if (threadIdx.x < 8) {
        const int l = threadIdx.x >= 4 ? 2 : threadIdx.x;
        s_lc[threadIdx.x] = l < 3 ? make_double2(th.al[l], th.bl[l]) : make_double2(1.0, 0.0);
    }
    __syncwarp();

    const int nseg = (U + kRwSeg - 1) / kRwSeg;
    const int64_t ngroups = (C + kRwRows - 1) / kRwRows;
    const int64_t W = (int64_t)gridDim.x * NW;
    const int64_t g_first = (int64_t)blockIdx.x * NW + warp;
    const uint32_t ring_s = smem_u32(ring), bars_s = smem_u32(bars);
    int64_t pg = g_first;                                    // next (group, segment) to issue
    int ps = 0, pd = 0;
    auto issue = [&]() {
        if (pg >= ngroups) return;
        if (lane == 0) {
            const uint32_t st = ring_s + pd * kRwStage, bar = bars_s + pd * 8;
            const int x = ps * kRwSeg, y = (int)(pg * kRwRows);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(kRwStage) : "memory");
            rw_tma_2d(st, &map_p0, x, y, bar);               // rows / patients beyond the planes arrive as zeros
            rw_tma_2d(st + kRwPlane, &map_p1, x, y, bar);
            rw_tma_2d(st + 2 * kRwPlane, &map_code, x, y, bar);
        }
        pd = pd + 1 == depth ? 0 : pd + 1;
        if (++ps == nseg) {
            ps = 0;
            pg += W;
        }
    };
#pragma unroll 1
    for (int i = 0; i < depth; ++i) issue();
    const double* s_tab = load_log_table<FAST>(tab, s_dyn);  // staged while the first tiles are in flight

    const int r = lane >> 2, sub = lane & 3;                 // row of the group, lane of the row
    // this lane's four 16-byte chunks of a row's 32 patients: sub, sub + 4, sub + 8, sub + 12, in this order for
    // every row -- a row's result does not depend on where in a group (or in an edge shard) the row lies.  (The
    // two rows of a quarter warp then share banks: a two-way conflict on the plane reads; rotating the order
    // per row would remove it and make the last bits of a row depend on its position.)
    int choff[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) choff[j] = sub + 4 * j;
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
            for (int l = 0; l < 3; ++l) a = fma(w[l], fast_log<FAST>(mix_rel(th, l, p3[k]), s_tab), a);
            acc[k] = a;
        }
    };
    // an element with one undecided region: q (log M_s - log M_2) per template state (half record {p*, +-q})
    auto half_p = [&](double p0, double p1, bool sx, double q) {
        const double p3[3] = {p0, p1, (1.0 - p0) - p1};
        const double ax = sx ? th.al[1] : th.al[0], bx = sx ? th.bl[1] : th.bl[0];
#pragma unroll
        for (int k = 0; k < 3; ++k)
            acc[k] = fma(q, fast_log<FAST>(fma(bx, p3[k], ax), s_tab) - fast_log<FAST>(mix_rel(th, 2, p3[k]), s_tab), acc[k]);
    };
    double keep[3] = {0.0, 0.0, 0.0};                        // row ends: 32 rows are finished at once (k2_finish)
    int64_t keep_c = -1;
    int groups_done = 0;
    auto finish_rows = [&]() {
        if (keep_c >= 0)
            k2_finish<MASKED>(keep_c, keep, __ldg(S1 + keep_c), __ldg(S2 + keep_c), MASKED ? __ldg(S0 + keep_c) : 0.0,
                              th, lqF, qF);
        keep_c = -1;
    };

    int d = 0;
    uint32_t phase = 0;
    for (int64_t g = g_first; g < ngroups; g += W) {
        const int64_t c = g * kRwRows + r;                   // this lane's row
        const bool live = c < C;
        // the row's record lists: requested now, used after the tiles
        int2 cnt = make_int2(0, 0);
        longlong2 ro = make_longlong2(0, 0);
        int v = 0;
        if (live) {
            cnt = __ldg(counts + c);
            if (cnt.x > 0 || cnt.y > 0) {
                v = __ldg(nm + c);
                if (cnt.x != 3 * U) ro = __ldg(rowoff + c);
            }
        }
        // Half records of the row (sorted by patient): no gather -- each of the row's four lanes holds its next
        // two records (patient, signed weight) in registers and takes p_0, p_1 from the TILE when the record's
        // patient streams by; the next record is requested as soon as one is consumed.
        const bool listed = live && cnt.x != 3 * U;
        const int nh = listed ? cnt.y : 0;
        const unsigned long long* kh = keysH + ro.y;
        const double2* hr = Hh + ro.y;
        int hidx = sub, hu = 0x7fffffff, hu2 = 0x7fffffff;
        double hq = 0.0, hq2 = 0.0;
        if (hidx < nh) {
            hu = (int)(__ldg(kh + hidx) & 0xffffull);
            hq = __ldg(hr + hidx).y;
        }
        if (hidx + 4 < nh) {
            hu2 = (int)(__ldg(kh + hidx + 4) & 0xffffull);
            hq2 = __ldg(hr + hidx + 4).y;
        }
        for (int s = 0; s < nseg; ++s) {
            mbar_wait(bars + d, phase);
            const unsigned char* st = ring + d * kRwStage;
            const unsigned char* row0 = st + r * (kRwSeg * 8);
            const unsigned char* rowc = st + 2 * kRwPlane + r * kRwSeg;
            if (nf + 4 > kProdMax) flush();
            const bool tail = s == nseg - 1 && (U & (kRwSeg - 1)) != 0;      // warp-uniform: patients beyond U in this tile
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int ch = choff[j];
                const double2 a0 = *reinterpret_cast<const double2*>(row0 + ch * 16);
                const double2 a1 = *reinterpret_cast<const double2*>(row0 + kRwPlane + ch * 16);
                uint32_t c2 = *reinterpret_cast<const unsigned short*>(rowc + ch * 2);
                if (tail) {                                  // (the tile's zero fill would read as code 0)
                    const int u = s * kRwSeg + 2 * ch;
                    if (u >= U) c2 = 0x0303u;
                    else if (u + 1 >= U) c2 = (c2 & 0xffu) | 0x0300u;
                }
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
            }
            nf += 4;
            while (hu < (s + 1) * kRwSeg) {                  // my records whose patient lies in this tile
                const int o = hu - s * kRwSeg;
                half_p(reinterpret_cast<const double*>(row0)[o], reinterpret_cast<const double*>(row0 + kRwPlane)[o],
                       __double2hiint(hq) < 0, fabs(hq));
                hu = hu2;
                hq = hq2;
                hidx += 4;
                hu2 = 0x7fffffff;
                if (hidx + 4 < nh) {
                    hu2 = (int)(__ldg(kh + hidx + 4) & 0xffffull);
                    hq2 = __ldg(hr + hidx + 4).y;
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
        // the row's elements with real weights, four lanes per row
        if (live && (cnt.x > 0 || cnt.y > 0)) {
            const int n = v & 0xffff, m = (v >> 16) & 0xffff;
            if (cnt.x == 3 * U) {                            // the edge was unpeaked at the code pass: every element
                for (int u = sub; u < U; u += 4) weighted(c, u, n, m);
            } else {
                const unsigned long long* kf = keysF + ro.x;
                for (int i = sub; i < cnt.x; i += 4) weighted(c, (int)(__ldg(kf + i) & 0xffffull), n, m);
            }
        }
        __syncwarp();
        // the four lanes of a row -> one sum per row; the group's eight rows are parked in lanes
        // 8 (groups_done mod 4) + row, and every fourth group all 32 lanes finish their rows
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double a = acc[k];
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            const double got = __shfl_sync(0xffffffffu, a, (lane & 7) * 4);
            if ((lane >> 3) == (groups_done & 3)) keep[k] = got;
            acc[k] = 0.0;
        }
        if ((lane >> 3) == (groups_done & 3)) {
            const int64_t cr = g * kRwRows + (lane & 7);
            keep_c = cr < C ? cr : -1;
        }
        if ((++groups_done & 3) == 0) finish_rows();
    }
    finish_rows();
}

// ------------------------------------------------------------------ host side
typedef CUresult (*RwEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static RwEncodeFn rw_encode_fn() {
    static RwEncodeFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<RwEncodeFn>(p);
    }
    return fn;
}

// 2-D map over a [rows][cols] array with the given row pitch (bytes); tiles of kRwRows x kRwSeg elements
static bool rw_make_map(CUtensorMap* map, CUtensorMapDataType dt, int esize, const void* base, int64_t rows, int cols,
                        int64_t pitch_bytes) {
    RwEncodeFn fn = rw_encode_fn();
    if (fn == nullptr) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)pitch_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)kRwSeg, (cuuint32_t)kRwRows};
    const cuuint32_t estr[2] = {1, 1};
    (void)esize;
    return fn(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool estep_rows_supported(int U, int64_t pitchU, int64_t pitchQ) {
    // tensor maps: row pitches must be multiples of 16 bytes (pitchU even, pitchQ % 16 == 0: checked by the caller)
    return U >= 1 && pitchU % 2 == 0 && pitchQ % 16 == 0 && rw_encode_fn() != nullptr;
}

int estep_rows_launch(const double* S1, const double* S2, const double* S0, const double* P, int64_t planeStride,
                      int64_t C, int U, int64_t pitchU, const double* qR, const int32_t* nm, const uint8_t* code,
                      int64_t pitchQ, const int32_t* counts, const uint64_t* keysF, const uint64_t* keysH, const int64_t* rowoff,
                      const double* Hh, const ThetaDev& th, const LogTabWindow& tab, bool fast, double* lqF, double* qF,
                      cudaStream_t st) {
    alignas(64) CUtensorMap map_p0, map_p1, map_code;
    if (!rw_make_map(&map_p0, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 8, P, C, U, pitchU * 8) ||
        !rw_make_map(&map_p1, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 8, P + planeStride, C, U, pitchU * 8) ||
        !rw_make_map(&map_code, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, code, C, U, pitchQ)) {
        set_error("fcd_estep_qF_coded: cuTensorMapEncodeTiled failed");
        return -2;
    }
    const size_t tbytes = fast ? (((size_t)tab.n * 8 + 127) & ~(size_t)127) : 0;
    static const int forced_nw = [] {                         // FCD_K2R_WARPS=8|12|16: experiments
        const char* e = getenv("FCD_K2R_WARPS");
        return e != nullptr ? atoi(e) : 0;
    }();
    int nw = 16;
    if (S0 == nullptr && (forced_nw == 8 || forced_nw == 12 || forced_nw == 16)) nw = forced_nw;
    int depth = kRwMaxDepth;
    while (depth > 2 && tbytes + rw_ring_bytes(depth, nw) > kSmemBudget) --depth;
    FCD_REQUIRE(tbytes + rw_ring_bytes(depth, nw) <= kSmemBudget, "fcd_estep_qF_coded: shared memory budget exceeded");
    const size_t smem = tbytes + rw_ring_bytes(depth, nw);
    const int64_t ngroups = (C + kRwRows - 1) / kRwRows;
    int64_t grid = (ngroups + nw - 1) / nw;
    if (grid > sm_count()) grid = sm_count();                       // one persistent CTA per SM
#define FCD_K2R_(F, NW_, M)                                                                           \
    do {                                                                                              \
        FCD_ALLOW_BIG_SMEM(estep_qF_rows_kernel<F, NW_, M>);                                          \
        estep_qF_rows_kernel<F, NW_, M><<<(unsigned)grid, NW_ * 32, smem, st>>>(                      \
            map_p0, map_p1, map_code, S1, S2, S0, P, planeStride, C, U, pitchU, qR, nm,               \
            reinterpret_cast<const int2*>(counts), reinterpret_cast<const unsigned long long*>(keysF), \
            reinterpret_cast<const unsigned long long*>(keysH), reinterpret_cast<const longlong2*>(rowoff), \
            reinterpret_cast<const double2*>(Hh), th, tab, depth, lqF, qF);                           \
    } while (0)
#define FCD_K2R(F)                                                                                    \
    do {                                                                                              \
        if (nw == 16) FCD_K2R_(F, 16, false);                                                         \
        else if (nw == 12) FCD_K2R_(F, 12, false);                                                    \
        else FCD_K2R_(F, 8, false);                                                                   \
    } while (0)
    // the masked form is built for the default 16 warps only (the other widths are experiments)
    if (S0 != nullptr) {
        if (fast) FCD_K2R_(true, 16, true); else FCD_K2R_(false, 16, true);
    } else {
        if (fast) FCD_K2R(true); else FCD_K2R(false);
    }
#undef FCD_K2R
#undef FCD_K2R_
    return check_launch("fcd_estep_qF_coded(rows)");
}

}  // namespace fcd
