// Test-only device harness for the fp64 routines of fcdiff_b200/csrc/fcd_math.cuh (tests/test_gpu_math.py).
// Not part of the library: built with fcd_runtime.cu (the real log_table / log_table_window / log_table_covers /
// make_theta_dev) into a throw-away shared object and driven through ctypes on torch-owned buffers.
//
// Every launcher evaluates one routine elementwise, exactly as the kernels inline it.  The routines that read
// the -log r8 table get the window the library would stage for the given mixture-weight bounds, staged with
// load_log_table<true> into a FULL-size shared array that is first filled with NaN: a table slot outside the
// window reads NaN instead of whatever the shared memory held, and the slot index itself is returned as well.
#include <cmath>
#include <cstring>

#include "fcd_common.cuh"
#include "fcd_math.cuh"

using namespace fcd;

namespace {

constexpr int kThreads = 256;

unsigned grid_for(int64_t n) {
    int64_t g = (n + kThreads - 1) / kThreads;
    if (g > 4 * (int64_t)sm_count()) g = 4 * (int64_t)sm_count();
    return (unsigned)(g < 1 ? 1 : g);
}

// NaN-filled full table, then the window [w.lo, w.lo + w.n) staged at its own slots; returns the slot-indexed table
__device__ const double* stage_window(const LogTabWindow& w, double* s_full) {
    for (int i = threadIdx.x; i < kLogTabSize; i += blockDim.x) s_full[i] = __longlong_as_double(0x7ff8000000000000LL);
    __syncthreads();
    return load_log_table<true>(w, s_full + w.lo);
}

// a slot outside the table itself is reported by its index; it is not read
__device__ __forceinline__ double tab_at(const double* s_tab, int idx) {
    return idx >= 0 && idx < kLogTabSize ? s_tab[idx] : __longlong_as_double(0x7ff8000000000000LL);
}

__global__ void fast_log_kernel(const double* __restrict__ y, int64_t n, const __grid_constant__ LogTabWindow w,
                                double* __restrict__ out, int* __restrict__ slot) {
    extern __shared__ __align__(16) double s_full[];
    const double* s_tab = stage_window(w, s_full);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const LogParts p = log_reduce(y[i]);
        slot[i] = p.idx;
        out[i] = p.idx >= 0 && p.idx < kLogTabSize ? fast_log<true>(y[i], s_tab) : tab_at(s_tab, p.idx);
    }
}

__global__ void fast_log_rcp_kernel(const double* __restrict__ y, int64_t n, const __grid_constant__ LogTabWindow w,
                                    double* __restrict__ lg, double* __restrict__ rcp) {
    extern __shared__ __align__(16) double s_full[];
    const double* s_tab = stage_window(w, s_full);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int idx = log_reduce(y[i]).idx;
        double r = 0.0;
        lg[i] = idx >= 0 && idx < kLogTabSize ? fast_log_rcp<true>(y[i], s_tab, r) : tab_at(s_tab, idx);
        rcp[i] = r;
    }
}

__global__ void log_pos_kernel(const double* __restrict__ x, int64_t n, const __grid_constant__ LogTabWindow w,
                               double* __restrict__ out) {
    extern __shared__ __align__(16) double s_full[];
    const double* s_tab = stage_window(w, s_full);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double m = __hiloint2double((__double2hiint(x[i]) & 0x000fffff) | (1023 << 20), __double2loint(x[i]));
        const int idx = log_reduce(m).idx;
        out[i] = idx >= 0 && idx < kLogTabSize ? log_pos<true>(x[i], s_tab) : tab_at(s_tab, idx);
    }
}

// the mixture weights y_kl = fma(b_l, p, a_l) of the kernels (fcd_uniform.cu, fcd_mstep.cu), their slots and
// their table logarithms; out[3 i + l]
__global__ void mix_slots_kernel(const double* __restrict__ p, int64_t n, const __grid_constant__ ThetaDev th,
                                 const __grid_constant__ LogTabWindow w, double* __restrict__ y_out,
                                 int* __restrict__ slot, double* __restrict__ lg) {
    extern __shared__ __align__(16) double s_full[];
    const double* s_tab = stage_window(w, s_full);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            const double y = fma(th.bl[l], p[i], th.al[l]);
            const int idx = log_reduce(y).idx;
            y_out[3 * i + l] = y;
            slot[3 * i + l] = idx;
            lg[3 * i + l] = idx >= 0 && idx < kLogTabSize ? fast_log<true>(y, s_tab) : tab_at(s_tab, idx);
        }
    }
}

enum Plain { kFastRcp = 0, kRcpNewton = 1, kExpNonpos = 2, kExpNonposShort = 3 };

template <int F>
__global__ void plain_kernel(const double* __restrict__ x, int64_t n, double* __restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double v = x[i];
        out[i] = F == kFastRcp ? fast_rcp<true>(v) : F == kRcpNewton ? rcp_newton(v)
               : F == kExpNonpos ? exp_nonpos(v) : exp_nonpos_short(v);
    }
}

template <class K>
int full_table_smem(K kernel) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLogTabBytes) == cudaSuccess
               ? 0 : -2;
}

bool window_for(const double* epsl, const double* al, int with_mantissa, cudaStream_t st, LogTabWindow& w) {
    return log_table_window(epsl, al, st, w, with_mantissa != 0);
}

}  // namespace

extern "C" {

// the library is built with hidden visibility; only these entry points leave the shared object
#define PROBE_API __attribute__((visibility("default")))

PROBE_API const char* probe_last_error(void) { return fcd_last_error(); }

// {lo, n, covers} of the window the library stages for these weight bounds
PROBE_API int probe_window(const double* epsl3, const double* al3, int with_mantissa, int* lo_n_covers, void* stream) {
    LogTabWindow w;
    if (!window_for(epsl3, al3, with_mantissa, (cudaStream_t)stream, w)) return -2;
    lo_n_covers[0] = w.lo;
    lo_n_covers[1] = w.n;
    lo_n_covers[2] = log_table_covers(epsl3, al3) ? 1 : 0;
    return 0;
}

// the whole device table g_log_tab (kLogTabSize doubles) into dst (device)
PROBE_API int probe_copy_table(double* dst, void* stream) {
    const double* g = log_table((cudaStream_t)stream);
    if (g == nullptr) return -2;
    return cudaMemcpyAsync(dst, g, kLogTabBytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream) == cudaSuccess ? 0 : -2;
}

PROBE_API int probe_table_size(void) { return kLogTabSize; }

PROBE_API int probe_fast_log(const double* y, int64_t n, const double* epsl3, const double* al3, int with_mantissa, double* out,
                   int* slot, void* stream) {
    LogTabWindow w;
    if (!window_for(epsl3, al3, with_mantissa, (cudaStream_t)stream, w) || full_table_smem(fast_log_kernel)) return -2;
    fast_log_kernel<<<grid_for(n), kThreads, kLogTabBytes, (cudaStream_t)stream>>>(y, n, w, out, slot);
    return check_launch("probe_fast_log");
}

PROBE_API int probe_fast_log_rcp(const double* y, int64_t n, const double* epsl3, const double* al3, int with_mantissa,
                       double* lg, double* rcp, void* stream) {
    LogTabWindow w;
    if (!window_for(epsl3, al3, with_mantissa, (cudaStream_t)stream, w) || full_table_smem(fast_log_rcp_kernel)) return -2;
    fast_log_rcp_kernel<<<grid_for(n), kThreads, kLogTabBytes, (cudaStream_t)stream>>>(y, n, w, lg, rcp);
    return check_launch("probe_fast_log_rcp");
}

PROBE_API int probe_log_pos(const double* x, int64_t n, const double* epsl3, const double* al3, double* out, void* stream) {
    LogTabWindow w;
    if (!window_for(epsl3, al3, 1, (cudaStream_t)stream, w) || full_table_smem(log_pos_kernel)) return -2;
    log_pos_kernel<<<grid_for(n), kThreads, kLogTabBytes, (cudaStream_t)stream>>>(x, n, w, out);
    return check_launch("probe_log_pos");
}

// weights of theta (eta, epsilon) as make_theta_dev forms them; the window from (w_epsl3, w_al3) -- the weights'
// own bounds, or the box bounds of the solved evaluations
PROBE_API int probe_mix_slots(const double* p, int64_t n, double eta, double epsilon, const double* w_epsl3, const double* w_al3,
                    int with_mantissa, double* y, int* slot, double* lg, void* stream) {
    fcd_theta t;
    memset(&t, 0, sizeof(t));
    t.pi = 0.5;
    t.eta = eta;
    t.epsilon = epsilon;
    for (int k = 0; k < 3; ++k) {
        t.gamma[k] = 1.0 / 3.0;
        t.sigma[k] = 1.0;
    }
    const ThetaDev th = make_theta_dev(t, 1);
    LogTabWindow w;
    if (!window_for(w_epsl3, w_al3, with_mantissa, (cudaStream_t)stream, w) || full_table_smem(mix_slots_kernel)) return -2;
    mix_slots_kernel<<<grid_for(n), kThreads, kLogTabBytes, (cudaStream_t)stream>>>(p, n, th, w, y, slot, lg);
    return check_launch("probe_mix_slots");
}

// which: 0 fast_rcp, 1 rcp_newton, 2 exp_nonpos, 3 exp_nonpos_short
PROBE_API int probe_plain(int which, const double* x, int64_t n, double* out, void* stream) {
    const unsigned g = grid_for(n);
    cudaStream_t st = (cudaStream_t)stream;
    switch (which) {
        case kFastRcp: plain_kernel<kFastRcp><<<g, kThreads, 0, st>>>(x, n, out); break;
        case kRcpNewton: plain_kernel<kRcpNewton><<<g, kThreads, 0, st>>>(x, n, out); break;
        case kExpNonpos: plain_kernel<kExpNonpos><<<g, kThreads, 0, st>>>(x, n, out); break;
        case kExpNonposShort: plain_kernel<kExpNonposShort><<<g, kThreads, 0, st>>>(x, n, out); break;
        default: return -1;
    }
    return check_launch("probe_plain");
}

}  // extern "C"
