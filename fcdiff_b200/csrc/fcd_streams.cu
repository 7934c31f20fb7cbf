// K3b over the *coded dominant-state plane*.  Within one EM iteration the
// (eta, epsilon) optimiser evaluates E_lM(eta, epsilon) 6-16 times with q_F, q_R
// and the responsibility planes fixed (fcdiff/fit.py:228-241, 270-286).
// Everything of an evaluation that does not depend on (eta, epsilon) is hoisted
// into ONE cheap pass per iteration, the *code pass*:
//   * PsE[c][u] = p_{k*(c)}(c,u): the responsibility of every edge's dominant state,
//     edge-major; a row is re-gathered from the planes only when the edge's state
//     changed (q_F settles after the first iterations);
//   * code[c][u] (one byte): l* in 0..2 when the edge and both regions are peaked
//     (fcd_common.cuh, "Tiers": the element contributes log(a_l + b_l p) for ONE
//     (k*, l*) pair with weight exactly 1), 3 otherwise (nothing to add here);
//   * an element with ONE undecided region (normalised posterior (q_0, q_1), the other region in
//     state s) has the weights (q_s at l = s, 1 - q_s at l = 2): it stays in the plane with code
//     4 + s, where it counts as l = 2 with weight 1, and adds a 16-byte *half record* {p, +-q_s}
//     for the correction q_s (log M_s - log M_2) (sign bit = s);
//   * every other element is expanded into records {p_k, w_0, w_1, w_2} with
//     w_l = q_F[c,k] * pair weight_l (one record if the edge is peaked, three if not);
//   * the theta-free part sum w L of E_lM: (total of the L plane, once per cache)
//     corrected by the record elements.
// An evaluation is then a flat reduction: 9 bytes per edge-patient (p and its code)
// through per-warp TMA rings, the per-l constants from a four-row shared table, the
// logs as the log of a running product -- no row structure, no weights, no
// peak-state decoding, no partition of the elements (an earlier form sorted the p
// into three streams by l*: the sort cost as much per iteration as four evaluations).
// Record order is fixed by per-row counts and an exclusive scan: results are deterministic.
#include <cstring>

#include "fcd_common.cuh"
#include "fcd_solver.cuh"

namespace fcd {

constexpr int kBucketThreads = 256;

// code of element (c,u) from the two regions' peak states: 0..2 = l* (both regions peaked),
// 4 + s = one region mixed and normalised, the other in state s (half record), 3 = any other mixed
// pair (full record), 6 = padding (written as 3, not counted)
__device__ __forceinline__ int pair_code(int sn, int sm) {
    const int o = sn | sm;
    if (o < 2) return ((sn ^ sm) << 1) + (sn & sm);
    if (o & 4) return 6;
    if (sn == kStateMixedR && sm < 2) return 4 + sm;
    if (sm == kStateMixedR && sn < 2) return 4 + sn;
    return 3;
}

// Rows are handled in blocks of kRowBlock consecutive rows per CTA (one warp per
// row, kRowBlock / 8 rows per warp), so that the position of a row's records is
// (offset of its block) + (prefix inside the block): the block totals are scanned by
// one small kernel, the in-block prefix is recomputed in shared memory by the fill
// kernel -- no pass over per-row arrays by a single CTA.
constexpr int kRowBlock = 16;

// Codes of TWO patients at once: a 4096-entry table indexed by the four 3-bit states (sn_a | sm_a << 3 |
// sn_b << 6 | sm_b << 9), entry = the two code bytes; padding (a state above 4, or a dead state) is stored as
// 3 | 8: bit 3 = "do not count".  Built once per device, staged in shared memory per CTA (8 KB).
__device__ unsigned short g_pair_lut[4096];

__global__ void build_pair_lut_kernel() {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 4096) return;
    auto enc = [](int sn, int sm) {
        const int c = (sn > 4 || sm > 4) ? 6 : pair_code(sn, sm);
        return c == 6 ? 0x0b : c;
    };
    g_pair_lut[idx] = (unsigned short)(enc(idx & 7, (idx >> 3) & 7) | (enc((idx >> 6) & 7, (idx >> 9) & 7) << 8));
}

static bool ensure_pair_lut(cudaStream_t st) {
    static bool done[64] = {false};
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return false;
    if (!done[dev]) {
        build_pair_lut_kernel<<<16, 256, 0, st>>>();
        if (cudaGetLastError() != cudaSuccess) return false;
        done[dev] = true;
    }
    return true;
}

// code[c][u] for u in [0, pitchQ) and counts[c] = {full records, half records} of row c; blocktot[b]
// = their sums over the rows of block b.  On the way: PsE[c][:] = P[k*(c)][c][:] for the rows whose dominant
// state changed since the last call (kcache).
template <bool WIDE>
__global__ void __launch_bounds__(kBucketThreads)
code_plane_kernel(const double* __restrict__ P, int64_t planeStride, double* __restrict__ PsE,
                  uint8_t* __restrict__ kcache,
                  const uint8_t* __restrict__ fstate, const uint8_t* __restrict__ rstate, int64_t pitchS,
                  const int32_t* __restrict__ nm, int64_t C, int U, int64_t pitchU, int64_t pitchQ,
                  uint8_t* __restrict__ code, int2* __restrict__ counts, longlong2* __restrict__ blocktot) {
    __shared__ int2 s_cnt[kRowBlock];
    __shared__ uint8_t s_lut[64];                            // pair_code by (sn << 3 | sm): one LDS per element
    __shared__ __align__(16) unsigned short s_lut2[WIDE ? 4096 : 8];   // two elements per read (g_pair_lut)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 64) {
        const int sn = threadIdx.x >> 3, sm = threadIdx.x & 7;
        s_lut[threadIdx.x] = (uint8_t)((sn > 4 || sm > 4) ? 6 : pair_code(sn, sm));
    }
    if (WIDE)
        for (int i = threadIdx.x; i < 4096 / 8; i += kBucketThreads)
            reinterpret_cast<uint4*>(s_lut2)[i] = reinterpret_cast<const uint4*>(g_pair_lut)[i];
    __syncthreads();
    const int64_t cb = (int64_t)blockIdx.x * kRowBlock;
    for (int r = warp; r < kRowBlock; r += kBucketThreads / 32) {
        const int64_t c = cb + r;
        int cnt = 0, cnh = 0;
        if (c < C) {
            const int k = fstate[c];
            unsigned short* crow = reinterpret_cast<unsigned short*>(code + c * pitchQ);      // pitchQ % 16 == 0
            if (k == kStateMixedF) {
                for (int u = 2 * lane; u < pitchQ; u += 64) crow[u >> 1] = 0x0303;
                cnt = 3 * U;
                if (kcache[c] == 255) {                      // never gathered: the plane's row is uninitialised memory,
                    double* dst = PsE + c * pitchQ;          // and the neutral code's factor 1 + 0 p needs a finite p
                    for (int64_t u = 2 * lane; u < pitchU; u += 64) *reinterpret_cast<double2*>(dst + u) = make_double2(0.0, 0.0);
                    __syncwarp();
                    if (lane == 0) kcache[c] = 254;
                }
            } else {
                const int v = __ldg(nm + c);
                if (k != kcache[c]) {                        // warp-uniform; rare once q_F has settled
                    const double* src = P + (int64_t)k * planeStride + c * pitchU;
                    double* dst = PsE + c * pitchQ;
                    for (int64_t u = 2 * lane; u < pitchU; u += 64)
                        *reinterpret_cast<double2*>(dst + u) = ldg_stream2(src + u);
                    __syncwarp();
                    if (lane == 0) kcache[c] = (uint8_t)k;
                }
                const uint8_t* rn = rstate + (int64_t)(v & 0xffff) * pitchS;
                const uint8_t* rm = rstate + (int64_t)((v >> 16) & 0xffff) * pitchS;
                if (WIDE) {
                    // four patients per lane and pass: two table reads give four codes; the record flags of the
                    // four bytes (code == 3: bit0 & bit1 & ~bit2; code >= 4: bit2; bit 3 = padding) are counted
                    // with popc.  The state rows are padded with 4 up to pitchS >= pitchQ.
                    uint32_t* crow4 = reinterpret_cast<uint32_t*>(crow);
                    for (int u = 4 * lane; u < pitchQ; u += 128) {
                        const uint32_t sn4 = __ldg(reinterpret_cast<const uint32_t*>(rn + u));
                        const uint32_t sm4 = __ldg(reinterpret_cast<const uint32_t*>(rm + u));
                        const uint32_t ia = (sn4 & 7u) | ((sm4 & 7u) << 3) | ((sn4 >> 2) & 0x1c0u) | ((sm4 << 1) & 0xe00u);
                        const uint32_t sh = sn4 >> 16, th2 = sm4 >> 16;
                        const uint32_t ib = (sh & 7u) | ((th2 & 7u) << 3) | ((sh >> 2) & 0x1c0u) | ((th2 << 1) & 0xe00u);
                        const uint32_t x = (uint32_t)s_lut2[ia] | ((uint32_t)s_lut2[ib] << 16);
                        const uint32_t live = ~(x >> 3) & 0x01010101u;
                        cnt += __popc(x & (x >> 1) & ~(x >> 2) & live);
                        cnh += __popc((x >> 2) & live);
                        crow4[u >> 2] = x & 0x07070707u;
                    }
                } else
                // two patients per lane; the state rows are padded with 4 up to pitchS >= pitchQ
                for (int u = 2 * lane; u < pitchQ; u += 64) {
                    const uint32_t sn2 = __ldg(reinterpret_cast<const unsigned short*>(rn + u));
                    const uint32_t sm2 = __ldg(reinterpret_cast<const unsigned short*>(rm + u));
                    const int c0 = s_lut[((sn2 & 7) << 3) | (sm2 & 7)], c1 = s_lut[((sn2 >> 5) & 0x38) | ((sm2 >> 8) & 7)];
                    cnt += (c0 == 3) + (c1 == 3);
                    cnh += ((c0 & 6) == 4) + ((c1 & 6) == 4);
                    crow[u >> 1] = (unsigned short)((c0 == 6 ? 3 : c0) | ((c1 == 6 ? 3 : c1) << 8));
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
                    cnh += __shfl_xor_sync(0xffffffffu, cnh, o);
                }
            }
            if (lane == 0) counts[c] = make_int2(cnt, cnh);
        }
        if (lane == 0) s_cnt[r] = make_int2(cnt, cnh);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        longlong2 t = make_longlong2(0, 0);
        for (int r = 0; r < kRowBlock; ++r) {
            t.x += s_cnt[r].x;
            t.y += s_cnt[r].y;
        }
        blocktot[blockIdx.x] = t;
    }
}

// blockoff[b] = exclusive prefix sums of blocktot, total[0..1] the sums (as doubles: < 2^53).  One CTA: every
// thread takes a run of consecutive blocks (serial sums), the runs are scanned by warp shuffles and the 32 warp
// totals by the first warp -- three barriers in all (the first form, a Hillis-Steele scan of 1024 entries per pass
// with two barriers per step, took 17 us on the wait the host makes for the record counts).
__global__ void __launch_bounds__(1024)
record_scan_kernel(const longlong2* __restrict__ blocktot, int64_t nblocks, longlong2* __restrict__ blockoff,
                   double* __restrict__ total) {
    __shared__ long long s_warp[2][32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int64_t per = (nblocks + 1023) / 1024;
    const int64_t b0 = (int64_t)t * per, b1 = b0 + per < nblocks ? b0 + per : nblocks;
    long long run[2] = {0, 0};
    for (int64_t b = b0; b < b1; ++b) {
        const longlong2 v = blocktot[b];
        run[0] += v.x;
        run[1] += v.y;
    }
    long long inc[2] = {run[0], run[1]};                      // inclusive scan of the runs inside the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long w0 = __shfl_up_sync(0xffffffffu, inc[0], d), w1 = __shfl_up_sync(0xffffffffu, inc[1], d);
        if (lane >= d) {
            inc[0] += w0;
            inc[1] += w1;
        }
    }
    if (lane == 31) {
        s_warp[0][warp] = inc[0];
        s_warp[1][warp] = inc[1];
    }
    __syncthreads();
    if (warp == 0) {                                          // exclusive scan of the 32 warp totals
        long long w[2] = {s_warp[0][lane], s_warp[1][lane]};
        const long long mine[2] = {w[0], w[1]};
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long v0 = __shfl_up_sync(0xffffffffu, w[0], d), v1 = __shfl_up_sync(0xffffffffu, w[1], d);
            if (lane >= d) {
                w[0] += v0;
                w[1] += v1;
            }
        }
        s_warp[0][lane] = w[0] - mine[0];
        s_warp[1][lane] = w[1] - mine[1];
        if (lane == 31) {
            total[0] = (double)w[0];
            total[1] = (double)w[1];
        }
    }
    __syncthreads();
    long long off[2] = {s_warp[0][warp] + inc[0] - run[0], s_warp[1][warp] + inc[1] - run[1]};
    for (int64_t b = b0; b < b1; ++b) {
        const longlong2 v = blocktot[b];
        blockoff[b] = make_longlong2(off[0], off[1]);
        off[0] += v.x;
        off[1] += v.y;
    }
}

struct Record {
    double p, w0, w1, w2;
};

// out[0] = sum of the [C][U] plane (pitch pitchU): the L plane's total, once per cache.
__global__ void __launch_bounds__(kBucketThreads)
plane_sum_kernel(const double* __restrict__ X, int64_t C, int U, int64_t pitchU, double* __restrict__ out,
                 double* __restrict__ ws) {
    const int lane = threadIdx.x & 31;
    const int64_t nw = (int64_t)gridDim.x * (kBucketThreads / 32);
    double s0 = 0.0, s1 = 0.0;
    for (int64_t c = (int64_t)blockIdx.x * (kBucketThreads / 32) + (threadIdx.x >> 5); c < C; c += nw) {
        const double* row = X + c * pitchU;
        for (int u = 2 * lane; u < U; u += 64) {             // pitchU even: u + 1 < pitchU
            const double2 v = ldg_stream2(row + u);
            s0 += v.x;
            s1 += u + 1 < U ? v.y : 0.0;
        }
    }
    double vv[1] = {s0 + s1};
    grid_reduce_store<1, kBucketThreads>(vv, ws, out);
}

// Keys of the elements that need a record: (tag << 48) | (c << 16) | u.  Full records (keysF): tag 0 =
// element of a peaked edge whose regions are both undecided or not normalised, tag 1 + k = state k
// of an unpeaked edge (three records per element).  Half records (keysH): tag = s, the state of the
// decided region (code 4 + s).  Same row blocks as code_plane_kernel; rowoff[c] = first key of row c
// in either list (kept for the next E-step).  Only the code plane is read: the operands of a record
// are gathered by the record kernels, one thread per record.
__global__ void __launch_bounds__(kBucketThreads, 4)
record_keys_kernel(const uint8_t* __restrict__ code, const uint8_t* __restrict__ fstate,
                   int64_t C, int U, int64_t pitchQ, const int2* __restrict__ counts,
                   const longlong2* __restrict__ blockoff, unsigned long long* __restrict__ keysF,
                   unsigned long long* __restrict__ keysH, longlong2* __restrict__ rowoff) {
    __shared__ longlong2 s_off[kRowBlock];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t blk = blockIdx.x; blk * kRowBlock < C; blk += gridDim.x) {
        const int64_t cb = blk * kRowBlock;
        __syncthreads();
        if (threadIdx.x < 32) {                              // in-block exclusive prefix of the row counts (one warp scan)
            const int r = threadIdx.x;
            const int2 cv = (r < kRowBlock && cb + r < C) ? counts[cb + r] : make_int2(0, 0);
            long long v0 = cv.x, v1 = cv.y;
#pragma unroll
            for (int o = 1; o < kRowBlock; o <<= 1) {
                const long long w0 = __shfl_up_sync(0xffffffffu, v0, o), w1 = __shfl_up_sync(0xffffffffu, v1, o);
                if (r >= o) {
                    v0 += w0;
                    v1 += w1;
                }
            }
            if (r < kRowBlock) {
                const longlong2 bo = blockoff[blk];
                s_off[r] = make_longlong2(bo.x + v0 - cv.x, bo.y + v1 - cv.y);
                if (cb + r < C) rowoff[cb + r] = s_off[r];
            }
        }
        __syncthreads();
        for (int r = warp; r < kRowBlock; r += kBucketThreads / 32) {
            const int64_t c = cb + r;
            if (c >= C) break;
            const int2 cv = counts[c];
            if (cv.x == 0 && cv.y == 0) continue;            // warp-uniform
            const int k = fstate[c];
            unsigned long long* const dF = keysF + s_off[r].x;
            unsigned long long* const dH = keysH + s_off[r].y;
            const unsigned long long ckey = (unsigned long long)c << 16;
            if (k == kStateMixedF) {                         // three records per element, tagged with their state
                for (int u = lane; u < U; u += 32) {
#pragma unroll
                    for (int kk = 0; kk < 3; ++kk)
                        dF[3 * (int64_t)u + kk] = ((unsigned long long)(1 + kk) << 48) | ckey | (unsigned long long)u;
                }
                continue;
            }
            // a lane owns 16 consecutive patients per pass (one 128-bit load of their codes): it counts
            // its keys, one warp scan of the packed counts gives its offsets, then it stores its keys in
            // order -- no vote per element
            const uint8_t* crow = code + c * pitchQ;
            uint32_t offF = 0, offH = 0;
            for (int ub = 0; ub < U; ub += 512) {
                const int u0 = ub + 16 * lane;
                uint4 cw = make_uint4(0, 0, 0, 0);
                if (u0 < U) cw = __ldg(reinterpret_cast<const uint4*>(crow + u0));           // pitchQ % 16 == 0
                const uint32_t w4[4] = {cw.x, cw.y, cw.z, cw.w};
                // four codes per 32-bit word, all below 8: code == 3 <=> bit0 & bit1 & ~bit2, code >= 4 <=> bit2 --
                // one flag bit per byte, counted with popc (no loop over the 16 codes)
                const int nvalid = U - u0;                   // codes of this lane that exist (<= 0: none, >= 16: all)
                uint32_t mF[4], mH[4], nF = 0, nH = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int v = nvalid - 4 * k;
                    const uint32_t bm = v >= 4 ? 0x01010101u : (v <= 0 ? 0u : (0x01010101u >> (8 * (4 - v))));
                    const uint32_t x = w4[k];
                    mF[k] = x & (x >> 1) & ~(x >> 2) & bm;
                    mH[k] = (x >> 2) & bm;
                    nF += __popc(mF[k]);
                    nH += __popc(mH[k]);
                }
                uint32_t pk = nF | (nH << 16), incl = pk;                                    // both < 2^16
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
                uint32_t pF = offF + ((incl - pk) & 0xffff), pH = offH + ((incl - pk) >> 16);
                if (nF | nH) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        uint32_t m = mF[k] | mH[k];          // ascending patients: bit 8 i of word k = patient u0 + 4 k + i
                        while (m) {
                            const int b = __ffs(m) - 1;
                            m &= m - 1;
                            const unsigned long long u = (unsigned long long)(u0 + 4 * k + (b >> 3));
                            if ((mF[k] >> b) & 1u) dF[pF++] = ckey | u;
                            else dH[pH++] = ((unsigned long long)(((w4[k] >> b) & 0xffu) - 4) << 48) | ckey | u;
                        }
                    }
                }
                offF += tot & 0xffff;
                offH += tot >> 16;
            }
        }
    }
}

// Half records, one thread per key: {p, +-q_s} with p the dominant-state responsibility, q_s the
// undecided region's posterior of state s (the other region's state) and the sign bit = s.
__global__ void __launch_bounds__(kBucketThreads)
record_half_kernel(const unsigned long long* __restrict__ keys, long long nh, const double* __restrict__ PsE,
                   int64_t pitchQ, const double* __restrict__ qR, int U, const uint8_t* __restrict__ rstate,
                   int64_t pitchS, const int32_t* __restrict__ nm, double2* __restrict__ Hh) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nh;
         i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long key = keys[i];
        const int u = (int)(key & 0xffffull), sx = (int)(key >> 48);
        const int64_t c = (int64_t)((key >> 16) & 0xffffffffull);
        const int v = __ldg(nm + c);
        const int n = v & 0xffff, m = (v >> 16) & 0xffff;
        const int who = __ldg(rstate + (int64_t)n * pitchS + u) == kStateMixedR ? n : m;     // the undecided region
        const double q = __ldg(qR + ((int64_t)who * U + u) * 2 + sx);
        const double p = __ldg(PsE + c * pitchQ + u);
        Hh[i] = make_double2(p, sx ? -q : q);
    }
}

// Second half of the record pass, one thread per record: gathers the responsibility (dominant-state
// plane, or plane k of an unpeaked edge), the two regions' posteriors and the element's L, writes
// {p, w_0, w_1, w_2} and accumulates
//   out[0] = Lsum - sum_{record elements} L + sum_records (sum_l w_l) L
// (Lsum = sum of L over all local elements, fcd_plane_sum: the coded elements have weight exactly 1).
__global__ void __launch_bounds__(kBucketThreads)
record_weights_kernel(const unsigned long long* __restrict__ keys, long long nd, const double* __restrict__ P,
                      int64_t planeStride, const double* __restrict__ PsE, int64_t pitchQ,
                      const double* __restrict__ L, int64_t pitchU, const double* __restrict__ Lsum,
                      const double* __restrict__ qF,
                      const double* __restrict__ qR, int U, const int32_t* __restrict__ nm,
                      Record* __restrict__ D, double* __restrict__ out, double* __restrict__ ws) {
    const double2* qR2 = reinterpret_cast<const double2*>(qR);
    double cs = 0.0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nd;
         i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long key = keys[i];
        const int u = (int)(key & 0xffffull), tag = (int)(key >> 48);
        const int64_t c = (int64_t)((key >> 16) & 0xffffffffull);
        const int64_t e = c * pitchU + u;
        const int v = __ldg(nm + c);
        Record rec;
        rec.p = tag == 0 ? __ldg(PsE + c * pitchQ + u) : ldg_stream1(P + (int64_t)(tag - 1) * planeStride + e);
        double w[3];
        pair_weights(__ldg(qR2 + (int64_t)(v & 0xffff) * U + u), __ldg(qR2 + (int64_t)((v >> 16) & 0xffff) * U + u), w);
        double scale = 1.0, cscale = 1.0;
        if (tag > 0) {
            const double qf[3] = {__ldg(qF + c * 3), __ldg(qF + c * 3 + 1), __ldg(qF + c * 3 + 2)};
            scale = qf[tag - 1];
            cscale = tag == 1 ? qf[0] + qf[1] + qf[2] : 0.0;  // the element's theta-free term is counted once
        }
        // the element's theta-free term is counted once (tag <= 1), and it leaves the weight-1 sum.  For
        // normalised posteriors the coefficient is a rounding residue: below 2^-50 the product with
        // L is below the rounding of the sum and L is not fetched (a 64-byte DRAM access per record)
        const double coef = cscale * (w[0] + w[1] + w[2]) - (tag <= 1 ? 1.0 : 0.0);
        if (fabs(coef) > 8.881784197001252e-16) cs = fma(coef, __ldg(L + e), cs);
        rec.w0 = scale * w[0];
        rec.w1 = scale * w[1];
        rec.w2 = scale * w[2];
        D[i] = rec;
    }
    double vv[1] = {cs + ((blockIdx.x == 0 && threadIdx.x == 0) ? Lsum[0] : 0.0)};
    grid_reduce_store<1, kBucketThreads>(vv, ws, out);
}

// One evaluation:
//   out[0] = sum_{code != 3} log(a_l + b_l p) + sum_records sum_l w_l log(a_l + b_l p)
//            + sum_half q (log(a_s + b_s p) - log(a_2 + b_2 p)),          l = code (2 for the codes 4, 5)
//   out[1] = dE/d eta, out[2] = dE/d eps as in elm_kernel (fcd_mstep.cu).
// FAST: the coded elements have weight exactly 1, so the objective is the log of a running product
// (fcd_math.cuh "Sum of logs as the log of a product") and the gradient needs 1 / M only
// (MUFU.RCP64H + Newton): ~11 fp64 instructions and two table reads per element.
// One persistent CTA of 16 warps per SM; the plane is cut into chunks of kEvChunk elements (2 KB of
// p + 256 code bytes, two bulk copies on one mbarrier), followed by the records as chunks of 64 and
// the half records as chunks of 128;
// warp g takes the chunks g, g + G, ...; every warp runs a private ring of kEvDepth stages and
// refills a stage as soon as it has consumed it: the bytes in flight do not depend on registers.
constexpr int kEvChunk = 512;
constexpr int kEvMaxDepth = 4;                                // stages per warp ring (fewer when the log table window is large)
constexpr int kEvWarps = 16;
constexpr int kEvThreads = kEvWarps * 32;
constexpr int kEvStage = kEvChunk * 8 + kEvChunk;            // bytes: p, then codes
constexpr size_t ev_ring_bytes(int depth) { return (size_t)kEvWarps * depth * (kEvStage + 8); }

struct CodedAcc {
    double obj, ge, gh, prod;
};

// HESS: also the moments of the solver's series model (fcd_solver.cuh), one set for both accumulators:
// sum t^k (A_k, l < 2) and sum v^k (B_k, l = 2), k = 2..K.
// The gradient weights are formed from the code in the ALU (it has the headroom; the shared-memory pipe,
// with one 16-byte table read per element for {a_l, b_l} already, does not): sgn = -1, +1 for l = 0, 1 and
// y = [l = 2] (codes 2, 4, 5).  acc.ge collects sum sgn d only: the l = 2
// part of sum s_l d is (2 eta - 1) acc.gh and is added once, after the plane.
template <bool GRAD, bool FAST, bool HESS>
__device__ __forceinline__ void coded_elem(double p, int code, const double2* s_ab, const double* s_tab, CodedAcc& acc,
                                           SolverMoments& mo) {
    const double2 ab = s_ab[code];
    const double M = fma(ab.y, p, ab.x);
    double rcp = 0.0;
    if (FAST) {
        acc.prod *= M;
        if (GRAD) rcp = rcp_newton(M);
    } else if (GRAD) {
        acc.obj += fast_log_rcp<FAST>(M, s_tab, rcp);
    } else {
        acc.obj += fast_log<FAST>(M, s_tab);
    }
    if (GRAD) {
        // the weights as +-2.0 / 0 -- one nibble per code, shifted into the top of the high word (2.0 =
        // 0x4000..., -2.0 = 0xC000...) -- against HALF the derivative factor: exact, three ALU
        // instructions per weight
        const double dh = fma(0.75, p, -0.25) * rcp;                      // mix_num(p) / 2 * rcp
        const int sh = code << 2;
        const double sgn2 = __hiloint2double((int)(((0x4cu >> sh) & 0xfu) << 28), 0);          // l = 0: -2, l = 1: +2
        const double y2 = __hiloint2double((int)(((0x440400u >> sh) & 0xfu) << 28), 0);        // codes 2, 4, 5: 2
        const double t = sgn2 * dh, v = y2 * dh;
        acc.ge += t;
        acc.gh += v;
        if (HESS) {
            add_powers1(mo.a, t);
            add_powers1(mo.b, v);
        }
    }
}

// SOLVE: the evaluation point (eta, epsilon) is read from the solver state in device memory, the
// kernel also accumulates the Hessian sums, and the CTA that arrives last exchanges the sums with
// the other edge shards, takes the optimiser's step and publishes the state (fcd_solver.cuh); a
// launch that finds the solve finished exits at once.
template <bool GRAD, bool FAST, bool SOLVE>
__global__ void __launch_bounds__(kEvThreads, 1)
elm_coded_kernel(const double* __restrict__ PsE, const uint8_t* __restrict__ code, long long nE,
                 const Record* __restrict__ D, long long nd, const double2* __restrict__ Hh, long long nh,
                 const __grid_constant__ ThetaDev th, const __grid_constant__ LogTabWindow tab, int depth,
                 double* __restrict__ out, double* __restrict__ ws,
                 SolverState* __restrict__ state, const double* __restrict__ konst_dev,
                 const __grid_constant__ CommPeers peers, int rank, int world, SolverPublished* pub,
                 unsigned long long seq) {
    static_assert(!SOLVE || GRAD, "the solver needs the gradient sums");
    extern __shared__ __align__(128) double s_dyn[];
    __shared__ double2 s_ab[8];
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
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* ring0 = reinterpret_cast<unsigned char*>(s_dyn + (FAST ? ((tab.n + 15) & ~15) : 0));
    unsigned char* ring = ring0 + (size_t)warp * depth * kEvStage;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring0 + (size_t)kEvWarps * depth * kEvStage) + warp * depth;
    if (lane < depth) mbar_init(bars + lane, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (threadIdx.x < 8) {
        // per-code constants {a_l, b_l}; code 3 is neutral: log(1 + 0 p) = 0 exactly (and zero gradient
        // weight, coded_elem); the codes 4, 5 count as l = 2
        const int code = threadIdx.x;
        const int l = code >= 4 ? 2 : code;
        s_ab[code] = l < 3 ? make_double2(sel3(l, T.al), sel3(l, T.bl)) : make_double2(1.0, 0.0);
    }
    __syncwarp();

    // Chunks are numbered across the two streams: the coded plane (nqf full chunks, then one partial
    // chunk if nE is not a multiple of the chunk), then the records (4 doubles each).  Full plane
    // chunks -- all but a handful -- take the short path: constant sizes, 32-bit shared addresses.
    const long long n3 = nd * 4, n4 = nh * 2;
    const long long nqf = nE / kEvChunk;
    const long long nq0 = (nE + kEvChunk - 1) / kEvChunk, nq1 = (n3 + kEvChunk - 1) / kEvChunk;
    const long long nq01 = nq0 + nq1;
    const long long nq = nq01 + (n4 + kEvChunk - 1) / kEvChunk;
    const double* const Dd = reinterpret_cast<const double*>(D);
    const double* const Hd = reinterpret_cast<const double*>(Hh);
    const long long W = (long long)gridDim.x * kEvWarps;
    const uint32_t ring_s = smem_u32(ring), bars_s = smem_u32(bars);
    long long ip = (long long)blockIdx.x * kEvWarps + warp;  // next chunk to issue
    int pd = 0;
    auto issue = [&]() {
        if (ip >= nq) return;
        if (lane == 0) {
            const uint32_t st = ring_s + pd * kEvStage, bar = bars_s + pd * 8;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            if (ip < nqf) {
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(kEvStage) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(st), "l"(PsE + ip * kEvChunk), "r"(kEvChunk * 8), "r"(bar) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(st + kEvChunk * 8), "l"(code + ip * kEvChunk), "r"(kEvChunk), "r"(bar) : "memory");
            } else if (ip < nq0) {
                const uint32_t cnt = (uint32_t)(nE - ip * kEvChunk);
                const uint32_t pbytes = ((cnt + 1) & ~1u) * 8, cbytes = (cnt + 15) & ~15u;
                mbar_expect_tx(bars + pd, pbytes + cbytes);
                tma_load_1d(ring + pd * kEvStage, PsE + ip * kEvChunk, pbytes, bars + pd);
                tma_load_1d(ring + pd * kEvStage + kEvChunk * 8, code + ip * kEvChunk, cbytes, bars + pd);
            } else {
                const bool half = ip >= nq01;
                const long long i = ip - (half ? nq01 : nq0);
                const long long left = (half ? n4 : n3) - i * kEvChunk;
                const uint32_t bytes = (uint32_t)(left < kEvChunk ? left : kEvChunk) * 8;
                mbar_expect_tx(bars + pd, bytes);
                tma_load_1d(ring + pd * kEvStage, (half ? Hd : Dd) + i * kEvChunk, bytes, bars + pd);
            }
        }
        ip += W;
        if (++pd == depth) pd = 0;
    };
#pragma unroll 1
    for (int i = 0; i < depth; ++i) issue();
    // the table and the constants are staged while the first chunks are in flight
    const double* s_tab = load_log_table<FAST>(tab, s_dyn);

    CodedAcc a0 = {0.0, 0.0, 0.0, 1.0}, a1 = {0.0, 0.0, 0.0, 1.0};
    SolverMoments mo;
#pragma unroll
    for (int k = 0; k < kSolverK - 1; ++k) mo.a[k] = mo.b[k] = 0.0;
    int nf = 0;                                              // factors in each running product
    int d = 0;
    uint32_t phase = 0;
    long long cp = (long long)blockIdx.x * kEvWarps + warp;
    auto advance = [&]() {
        __syncwarp();
        issue();
        if (++d == depth) {
            d = 0;
            phase ^= 1;
        }
        cp += W;
    };
    auto flush = [&]() {
        if (FAST) {
            a0.obj += log_pos<FAST>(a0.prod * a1.prod, s_tab);
            a0.prod = a1.prod = 1.0;
        }
        nf = 0;
    };
    for (; cp < nqf; advance()) {                            // full chunks of the coded plane
        mbar_wait(bars + d, phase);
        const unsigned char* st = ring + d * kEvStage;
#pragma unroll
        for (int j = 0; j < kEvChunk / 64; ++j) {
            const double2 v = *reinterpret_cast<const double2*>(st + (64 * j + 2 * lane) * 8);
            const uint32_t c2 = *reinterpret_cast<const unsigned short*>(st + kEvChunk * 8 + 64 * j + 2 * lane);
            coded_elem<GRAD, FAST, SOLVE>(v.x, c2 & 0xff, s_ab, s_tab, a0, mo);
            coded_elem<GRAD, FAST, SOLVE>(v.y, c2 >> 8, s_ab, s_tab, a1, mo);
        }
        nf += kEvChunk / 64;
        if (nf + kEvChunk / 64 > kProdMax) flush();
    }
    for (; cp < nq0; advance()) {                            // the partial chunk, if any
        const int left = (int)(nE - cp * kEvChunk);
        mbar_wait(bars + d, phase);
        const unsigned char* st = ring + d * kEvStage;
        flush();
        for (int e = lane; e < left; e += 32)
            coded_elem<GRAD, FAST, SOLVE>(reinterpret_cast<const double*>(st)[e], st[kEvChunk * 8 + e], s_ab, s_tab, a0,
                                          mo);
    }
    flush();
    const double al[3] = {T.al[0], T.al[1], T.al[2]}, bl[3] = {T.bl[0], T.bl[1], T.bl[2]};
    const double sl[3] = {-1.0, 1.0, 2.0 * T.eta - 1.0};
    double obj = a0.obj + a1.obj, gh = a0.gh + a1.gh;
    double ge = fma(sl[2], gh, a0.ge + a1.ge);               // sum s_l d over the plane: l < 2 signed, l = 2 through gh
    for (; cp < nq01; advance()) {                           // records {p, w_0, w_1, w_2}: real weights, three logs each
        const long long left = (n3 - (cp - nq0) * kEvChunk) >> 2;
        const int cnt = (int)(left < kEvChunk / 4 ? left : kEvChunk / 4);
        mbar_wait(bars + d, phase);
        const double4* st = reinterpret_cast<const double4*>(ring + d * kEvStage);
#pragma unroll
        for (int j = 0; j < kEvChunk / 128; ++j) {
            const int e = 32 * j + lane;
            if (e < cnt) {
                const double4 r = st[e];
                const double w[3] = {r.y, r.z, r.w};
                const double num = mix_num(r.x);
#pragma unroll
                for (int l = 0; l < 3; ++l) {
                    const double M = fma(bl[l], r.x, al[l]);
                    if (GRAD) {
                        double rcp;
                        obj = fma(w[l], fast_log_rcp<FAST>(M, s_tab, rcp), obj);
                        const double g = num * rcp;
                        const double dd = w[l] * g;
                        ge = fma(sl[l], dd, ge);
                        if (l == 2) gh += dd;
                        if (SOLVE) {
                            if (l == 2) add_powers(mo.b, w[l], g);
                            else add_powers(mo.a, w[l], sl[l] * g);
                        }
                    } else {
                        obj = fma(w[l], fast_log<FAST>(M, s_tab), obj);
                    }
                }
            }
        }
    }
    for (; cp < nq; advance()) {                             // half records {p, +-q}: q (log M_s - log M_2), sign bit = s
        const long long left = (n4 - (cp - nq01) * kEvChunk) >> 1;
        const int cnt = (int)(left < kEvChunk / 2 ? left : kEvChunk / 2);
        mbar_wait(bars + d, phase);
        const double2* st = reinterpret_cast<const double2*>(ring + d * kEvStage);
#pragma unroll
        for (int j = 0; j < kEvChunk / 64; ++j) {
            const int e = 32 * j + lane;
            if (e < cnt) {
                const double2 r = st[e];
                const bool sx = __double2hiint(r.y) < 0;
                const double q = fabs(r.y);
                const double Mx = fma(sx ? bl[1] : bl[0], r.x, sx ? al[1] : al[0]), M2 = fma(bl[2], r.x, al[2]);
                if (GRAD) {
                    double rx, r2;
                    const double lx = fast_log_rcp<FAST>(Mx, s_tab, rx), l2 = fast_log_rcp<FAST>(M2, s_tab, r2);
                    obj = fma(q, lx - l2, obj);
                    const double num = mix_num(r.x);
                    const double gx = num * rx, g2 = num * r2;
                    const double dx = q * gx, d2 = q * g2;
                    ge += fma(sx ? 1.0 : -1.0, dx, -sl[2] * d2);
                    gh -= d2;
                    if (SOLVE) {
                        add_powers(mo.a, q, sx ? gx : -gx);
                        add_powers(mo.b, -q, g2);
                    }
                } else {
                    obj = fma(q, fast_log<FAST>(Mx, s_tab) - fast_log<FAST>(M2, s_tab), obj);
                }
            }
        }
    }
    if (SOLVE) {
        double v[kSolverVals];
        solver_sums(obj, ge, gh, mo, v);
        if (grid_reduce_last<kSolverVals, kEvThreads>(v, ws, s_sums))
            solver_epilogue(s_sums, state, konst_dev, peers, rank, world, pub, seq);
    } else {
        // dE/d eta = -(2 eps - 1) sum_{l = 2} d;  dE/d eps = -sum s_l d                 (fit.py:600-697)
        double v[3] = {obj, -(2.0 * T.epsilon - 1.0) * gh, -ge};
        grid_reduce_store<3, kEvThreads>(v, ws, out);
    }
}

static inline int rows_grid(int64_t rows, int rows_per_block, int waves) {
    int64_t need = (rows + rows_per_block - 1) / rows_per_block;
    int64_t cap = (int64_t)sm_count() * waves;
    if (cap > kMaxReduceBlocks) cap = kMaxReduceBlocks;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int64_t fcd_bucket_blocks(int64_t C) { return (C + kRowBlock - 1) / kRowBlock; }

int fcd_plane_sum(const double* X, int64_t C, int32_t U, int64_t pitchU, double* out1, double* ws, void* stream) {
    FCD_REQUIRE(X != nullptr && out1 != nullptr && ws != nullptr, "fcd_plane_sum: NULL argument");
    FCD_REQUIRE(C >= 1 && U >= 1 && pitchU >= U && pitchU % 2 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0,
                "fcd_plane_sum: bad shape (even pitch, 16-byte aligned)");
    plane_sum_kernel<<<rows_grid(C, kBucketThreads / 32, 8), kBucketThreads, 0, (cudaStream_t)stream>>>(
        X, C, U, pitchU, out1, ws);
    return check_launch("fcd_plane_sum");
}

int64_t fcd_code_pitch(int32_t U) { return ((int64_t)U + 15) & ~(int64_t)15; }

int fcd_code_plane(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                   const uint8_t* fstate, const uint8_t* rstate, int64_t pitchS, const int32_t* nm,
                   double* PsE, uint8_t* kcache, uint8_t* code, int64_t pitchQ, int32_t* counts, int64_t* blockoff,
                   double* total2, void* stream) {
    FCD_REQUIRE(P != nullptr && fstate != nullptr && rstate != nullptr && nm != nullptr && PsE != nullptr &&
                kcache != nullptr && code != nullptr && counts != nullptr && blockoff != nullptr && total2 != nullptr,
                "fcd_code_plane: NULL argument");
    FCD_REQUIRE(C >= 1 && U >= 1 && pitchU >= U && pitchU % 2 == 0 && planeStride % 2 == 0 && pitchQ >= pitchU &&
                pitchQ % 16 == 0 && pitchS >= pitchQ && pitchS % 2 == 0,
                "fcd_code_plane: bad shape (even pitches, pitchQ % 16 == 0, pitchS >= pitchQ >= pitchU)");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(P) | reinterpret_cast<uintptr_t>(PsE) | reinterpret_cast<uintptr_t>(code) |
                  reinterpret_cast<uintptr_t>(blockoff)) & 15) == 0 &&
                (reinterpret_cast<uintptr_t>(rstate) & 1) == 0 && (reinterpret_cast<uintptr_t>(counts) & 7) == 0,
                "fcd_code_plane: planes / code / blockoff must be 16-byte aligned, counts 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nblocks = (C + kRowBlock - 1) / kRowBlock;
    // blockoff doubles as the block totals' storage: [nblocks] totals followed by [nblocks] offsets (pairs)
    longlong2* bt = reinterpret_cast<longlong2*>(blockoff);
    const bool wide = pitchS % 4 == 0 && (reinterpret_cast<uintptr_t>(rstate) & 3) == 0 && ensure_pair_lut(st);
    (wide ? code_plane_kernel<true> : code_plane_kernel<false>)<<<(unsigned)nblocks, kBucketThreads, 0, st>>>(
                                                                    P, planeStride, PsE, kcache, fstate, rstate, pitchS,
                                                                    nm, C, U, pitchU, pitchQ, code,
                                                                    reinterpret_cast<int2*>(counts), bt);
    int rc = check_launch("fcd_code_plane");
    if (rc) return rc;
    record_scan_kernel<<<1, 1024, 0, st>>>(bt, nblocks, bt + nblocks, total2);
    return check_launch("fcd_code_plane(scan)");
}

int fcd_code_records(const double* P, int64_t planeStride, const double* PsE, const uint8_t* code, int64_t pitchQ,
                     const double* L, const double* Lsum, int64_t C, int32_t U, int64_t pitchU,
                     const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate, int64_t pitchS,
                     int32_t N, const int32_t* nm, const int32_t* counts, const int64_t* blockoff,
                     uint64_t* keysF, uint64_t* keysH, int64_t* rowoff, double* D, int64_t nd, double* Hh, int64_t nh,
                     double* out1, double* ws, void* stream) {
    FCD_REQUIRE(P != nullptr && PsE != nullptr && code != nullptr && L != nullptr && Lsum != nullptr && qF != nullptr &&
                fstate != nullptr && qR != nullptr && rstate != nullptr && nm != nullptr && counts != nullptr &&
                blockoff != nullptr && keysF != nullptr && keysH != nullptr && rowoff != nullptr && D != nullptr &&
                Hh != nullptr && out1 != nullptr && ws != nullptr, "fcd_code_records: NULL argument");
    FCD_REQUIRE(C >= 1 && C < (1ll << 32) && U >= 1 && U < 65536 && pitchU >= U && pitchU % 2 == 0 &&
                pitchQ >= pitchU && pitchQ % 16 == 0 && pitchS >= U && N >= 2 && N < 65536 && nd >= 0 && nh >= 0,
                "fcd_code_records: bad shape");
    FCD_REQUIRE((reinterpret_cast<uintptr_t>(D) & 31) == 0 &&
                ((reinterpret_cast<uintptr_t>(Hh) | reinterpret_cast<uintptr_t>(rowoff) | reinterpret_cast<uintptr_t>(blockoff)) & 15) == 0 &&
                ((reinterpret_cast<uintptr_t>(keysF) | reinterpret_cast<uintptr_t>(keysH) | reinterpret_cast<uintptr_t>(counts)) & 7) == 0,
                "fcd_code_records: records must be 32-byte, half records / rowoff 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nblocks = (C + kRowBlock - 1) / kRowBlock;
    int rc = 0;
    if (nd + nh > 0) {
        int64_t grid = nblocks;                              // persistent: the resident CTAs share the row blocks
        if (grid > (int64_t)sm_count() * 4) grid = (int64_t)sm_count() * 4;
        record_keys_kernel<<<(unsigned)grid, kBucketThreads, 0, st>>>(
            code, fstate, C, U, pitchQ, reinterpret_cast<const int2*>(counts),
            reinterpret_cast<const longlong2*>(blockoff) + nblocks, reinterpret_cast<unsigned long long*>(keysF),
            reinterpret_cast<unsigned long long*>(keysH), reinterpret_cast<longlong2*>(rowoff));
        rc = check_launch("fcd_code_records(keys)");
        if (rc) return rc;
    }
    if (nh > 0) {
        int64_t hgrid = (nh + kBucketThreads - 1) / kBucketThreads;
        if (hgrid > (int64_t)sm_count() * 8) hgrid = (int64_t)sm_count() * 8;
        record_half_kernel<<<(unsigned)hgrid, kBucketThreads, 0, st>>>(
            reinterpret_cast<const unsigned long long*>(keysH), nh, PsE, pitchQ, qR, U, rstate, pitchS, nm,
            reinterpret_cast<double2*>(Hh));
        rc = check_launch("fcd_code_records(half)");
        if (rc) return rc;
    }
    int64_t rgrid = (nd + kBucketThreads - 1) / kBucketThreads;       // nd == 0: one CTA writes out1[0] = Lsum
    if (rgrid > (int64_t)sm_count() * 8) rgrid = (int64_t)sm_count() * 8;
    if (rgrid < 1) rgrid = 1;
    record_weights_kernel<<<(unsigned)rgrid, kBucketThreads, 0, st>>>(
        reinterpret_cast<const unsigned long long*>(keysF), nd, P, planeStride, PsE, pitchQ, L, pitchU, Lsum, qF, qR, U, nm,
        reinterpret_cast<Record*>(D), out1, ws);
    return check_launch("fcd_code_records");
}

int fcd_elm_coded(const double* PsE, const uint8_t* code, int64_t nE, const double* D, int64_t nd,
                  const double* Hh, int64_t nh, const fcd_theta* theta_host, int32_t want_grad, double* out3, double* ws,
                  void* stream) {
    FCD_REQUIRE(PsE != nullptr && code != nullptr && theta_host != nullptr && out3 != nullptr && ws != nullptr &&
                (nd == 0 || D != nullptr) && (nh == 0 || Hh != nullptr) && nE >= 1 && nd >= 0 && nh >= 0,
                "fcd_elm_coded: bad argument");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(PsE) | reinterpret_cast<uintptr_t>(code) | reinterpret_cast<uintptr_t>(Hh)) & 15) == 0 &&
                (reinterpret_cast<uintptr_t>(D) & 31) == 0,
                "fcd_elm_coded: plane / code / half records must be 16-byte aligned, records 32-byte aligned");
    const ThetaDev th = make_theta_dev(*theta_host, 0);
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(th.epsl, th.al, st, tab, true), "fcd_elm_coded: log table initialisation failed");
    const bool fast = log_table_covers(th.epsl, th.al);
    const size_t tbytes = fast ? (size_t)((tab.n + 15) & ~15) * sizeof(double) : 0;
    int depth = kEvMaxDepth;
    while (depth > 2 && tbytes + ev_ring_bytes(depth) > kSmemBudget) --depth;
    FCD_REQUIRE(tbytes + ev_ring_bytes(depth) <= kSmemBudget, "fcd_elm_coded: shared memory budget exceeded");
    const size_t smem = tbytes + ev_ring_bytes(depth);
    const long long chunks = (nE + kEvChunk - 1) / kEvChunk + (nd * 4 + kEvChunk - 1) / kEvChunk +
                             (nh * 2 + kEvChunk - 1) / kEvChunk;
    long long grid = (chunks + kEvWarps - 1) / kEvWarps;
    if (grid > sm_count()) grid = sm_count();                // one persistent CTA per SM
    if (grid < 1) grid = 1;
    CommPeers nopeers;
    comm_peers_from_host(nullptr, 1, nopeers);
#define FCD_EC(G_, F_)                                                                                   \
    do {                                                                                                 \
        FCD_ALLOW_BIG_SMEM(elm_coded_kernel<G_, F_, false>);                                             \
        elm_coded_kernel<G_, F_, false><<<(unsigned)grid, kEvThreads, smem, st>>>(                       \
            PsE, code, nE, reinterpret_cast<const Record*>(D), nd, reinterpret_cast<const double2*>(Hh), nh, th, \
            tab, depth, out3, ws, nullptr, nullptr, nopeers, 0, 1, nullptr, 0ull);                       \
    } while (0)
    if (want_grad) { if (fast) FCD_EC(true, true); else FCD_EC(true, false); }
    else           { if (fast) FCD_EC(false, true); else FCD_EC(false, false); }
#undef FCD_EC
    return check_launch("fcd_elm_coded");
}

int fcd_elm_coded_solve(const double* PsE, const uint8_t* code, int64_t nE, const double* D, int64_t nd,
                        const double* Hh, int64_t nh, double eps_lo, double eps_hi, void* state, const double* konst,
                        void* const* windows_host, int32_t rank, int32_t world, void* published_host, uint64_t seq0,
                        int32_t n_launches, double* ws, void* stream) {
    FCD_REQUIRE(PsE != nullptr && code != nullptr && state != nullptr && ws != nullptr &&
                (nd == 0 || D != nullptr) && (nh == 0 || Hh != nullptr) && nE >= 1 && nd >= 0 && nh >= 0,
                "fcd_elm_coded_solve: bad argument");
    FCD_REQUIRE(((reinterpret_cast<uintptr_t>(PsE) | reinterpret_cast<uintptr_t>(code) | reinterpret_cast<uintptr_t>(Hh)) & 15) == 0 &&
                (reinterpret_cast<uintptr_t>(D) & 31) == 0 && (reinterpret_cast<uintptr_t>(state) & 7) == 0,
                "fcd_elm_coded_solve: plane / code / half records must be 16-byte aligned, records 32-byte aligned");
    FCD_REQUIRE(n_launches >= 1 && n_launches <= 64 && world >= 1 && world <= kCommMaxWorld && rank >= 0 && rank < world &&
                eps_lo > 0.0 && eps_lo <= eps_hi && eps_hi < 1.0, "fcd_elm_coded_solve: bad launch / box arguments");
    CommPeers peers;
    FCD_REQUIRE(comm_peers_from_host(windows_host, world, peers), "fcd_elm_coded_solve: NULL window");
    SolverPublished* pub = nullptr;
    if (published_host != nullptr) {
        cudaError_t e = cudaHostGetDevicePointer((void**)&pub, published_host, 0);
        FCD_REQUIRE(e == cudaSuccess, "fcd_elm_coded_solve: cudaHostGetDevicePointer: %s", cudaGetErrorString(e));
    }
    // every mixture weight the solve can form inside the box lies in [m / 2, 1], m = min(eps_lo, 1 - eps_hi)
    const double m = eps_lo < 1.0 - eps_hi ? eps_lo : 1.0 - eps_hi;
    const double epsl[3] = {m, m, m}, al[3] = {0.5 * m, 0.5 * m, 0.5 * m};
    ThetaDev th;
    memset(&th, 0, sizeof(th));
    cudaStream_t st = (cudaStream_t)stream;
    LogTabWindow tab;
    FCD_REQUIRE(log_table_window(epsl, al, st, tab, true), "fcd_elm_coded_solve: log table initialisation failed");
    const bool fast = log_table_covers(epsl, al);
    const size_t tbytes = fast ? (size_t)((tab.n + 15) & ~15) * sizeof(double) : 0;
    int depth = kEvMaxDepth;
    while (depth > 2 && tbytes + ev_ring_bytes(depth) > kSmemBudget) --depth;
    FCD_REQUIRE(tbytes + ev_ring_bytes(depth) <= kSmemBudget, "fcd_elm_coded_solve: shared memory budget exceeded");
    const size_t smem = tbytes + ev_ring_bytes(depth);
    const long long chunks = (nE + kEvChunk - 1) / kEvChunk + (nd * 4 + kEvChunk - 1) / kEvChunk +
                             (nh * 2 + kEvChunk - 1) / kEvChunk;
    long long grid = (chunks + kEvWarps - 1) / kEvWarps;
    if (grid > sm_count()) grid = sm_count();                // one persistent CTA per SM
    if (grid < 1) grid = 1;
    if (fast) FCD_ALLOW_BIG_SMEM(elm_coded_kernel<true, true, true>);
    else FCD_ALLOW_BIG_SMEM(elm_coded_kernel<true, false, true>);
    for (int i = 0; i < n_launches; ++i) {
        const unsigned long long seq = (unsigned long long)seq0 + (unsigned long long)i;
        if (fast)
            elm_coded_kernel<true, true, true><<<(unsigned)grid, kEvThreads, smem, st>>>(
                PsE, code, nE, reinterpret_cast<const Record*>(D), nd, reinterpret_cast<const double2*>(Hh), nh, th, tab,
                depth, nullptr, ws, static_cast<SolverState*>(state), konst, peers, rank, world, pub, seq);
        else
            elm_coded_kernel<true, false, true><<<(unsigned)grid, kEvThreads, smem, st>>>(
                PsE, code, nE, reinterpret_cast<const Record*>(D), nd, reinterpret_cast<const double2*>(Hh), nh, th, tab,
                depth, nullptr, ws, static_cast<SolverState*>(state), konst, peers, rank, world, pub, seq);
        int rc = check_launch("fcd_elm_coded_solve");
        if (rc) return rc;
    }
    return 0;
}

}  // extern "C"
