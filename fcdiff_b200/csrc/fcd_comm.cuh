// Peer-memory exchange of a few doubles (see fcd_comm.cu) as a device function, so that a reduction
// kernel's last CTA can run the exchange itself (no separate launch): used by allreduce_small_kernel and by
// the epilogue of the (eta, epsilon) solver evaluations (fcd_solver.cuh).
#pragma once

#include "fcd_common.cuh"

namespace fcd {

constexpr int kCommMaxWorld = 16;
constexpr int kCommMaxVals = 16;

struct CommWindow {
    double slot[2][kCommMaxWorld][kCommMaxVals];
    unsigned long long flag[2][kCommMaxWorld];
    // Number of exchanges this rank has taken part in.  Kept in the rank's OWN window and advanced by
    // the exchanging CTA itself: host-launched exchanges (fcd_allreduce_small) and exchanges run from
    // a kernel epilogue share one sequence, and the slot-set parity alternates over the exchanges that
    // were actually executed (launches that exit early, e.g. after the solver has converged, take none).
    unsigned long long counter;
};

struct CommPeers {
    CommWindow* w[kCommMaxWorld];
};

constexpr unsigned long long kCommTimeoutBit = 1ull << 63;
constexpr long long kCommSpinCycles = 20000000000ll;          // ~10 s at 2 GHz: a lost peer must not hang the GPU

#ifdef __CUDACC__
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys(double* p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_sys(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

// All-reduce (sum) of s_vals[0..n) over the ranks, run by ALL threads of one CTA (blockDim.x >=
// world * n; s_vals in shared memory).  On return every rank holds the sums formed in rank order
// (bit-identical everywhere).  Returns false if a peer did not arrive within spin_cycles: s_vals
// is then left as it was.  world == 1 is a no-op.
__device__ __forceinline__ bool comm_exchange_cta(double* s_vals, int n, const CommPeers& peers, int rank, int world,
                                                  long long spin_cycles) {
    if (world <= 1) return true;
    __shared__ int s_timeout;
    __shared__ unsigned long long s_seq;
    const int t = threadIdx.x;
    if (t == 0) {
        s_timeout = 0;
        CommWindow* own = peers.w[rank];
        const unsigned long long k = own->counter + 1;        // only this rank's kernels touch it, in stream order
        own->counter = k;
        s_seq = k;
    }
    __syncthreads();
    const unsigned long long seq = s_seq;
    const int par = (int)(seq & 1ull);
    if (t < world * n) {                                      // 1. my partial sums into every rank's window
        const int p = t / n, i = t - p * n;
        st_relaxed_sys(&peers.w[p]->slot[par][rank][i], s_vals[i]);
        __threadfence_system();
    }
    __syncthreads();
    if (t < world) {
        st_release_sys(&peers.w[t]->flag[par][rank], seq);
        const unsigned long long* f = &peers.w[rank]->flag[par][t];           // 2. everybody's flag in my window
        const long long t0 = clock64();
        while (ld_acquire_sys(f) != seq) {
            if (clock64() - t0 > spin_cycles) {
                s_timeout = 1;
                break;
            }
        }
    }
    __syncthreads();
    double s = 0.0;
    if (t < n)                                                // 3. sum in rank order
        for (int r = 0; r < world; ++r) s += ld_relaxed_sys(&peers.w[rank]->slot[par][r][t]);
    const bool ok = s_timeout == 0;
    if (t < n && ok) s_vals[t] = s;
    __syncthreads();
    return ok;
}
#endif  // __CUDACC__

// Host: fills `peers` from the list of windows in this process' address space.
inline bool comm_peers_from_host(void* const* windows_host, int world, CommPeers& peers) {
    for (int r = 0; r < kCommMaxWorld; ++r) peers.w[r] = nullptr;
    if (world <= 1) return true;
    if (windows_host == nullptr || world > kCommMaxWorld) return false;
    for (int r = 0; r < world; ++r) {
        if (windows_host[r] == nullptr) return false;
        peers.w[r] = static_cast<CommWindow*>(windows_host[r]);
    }
    return true;
}

}  // namespace fcd
