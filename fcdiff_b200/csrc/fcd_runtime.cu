// Runtime glue of libfcdiff_b200: error reporting, launch accounting, theta
// constants.  No device memory is allocated anywhere in this library.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include <nvtx3/nvToolsExt.h>

#include "fcd_common.cuh"
#include "fcd_math.cuh"

namespace fcd {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return -2;
    }
    return 0;
}

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// -log(r8) table of fast_log (fcd_math.cuh): theta-independent, built once per
// device in static device memory (no runtime allocation).
__device__ __align__(128) double g_log_tab[kLogTabSize];

__global__ void build_log_table_kernel() {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kLogTabSize; i += gridDim.x * blockDim.x)
        g_log_tab[i] = -log(log_table_r8(i));
}

const double* log_table(cudaStream_t st) {
    static double* addr[64] = {nullptr};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (addr[dev] == nullptr) {
        double* p = nullptr;
        if (cudaGetSymbolAddress((void**)&p, g_log_tab) != cudaSuccess) return nullptr;
        build_log_table_kernel<<<42, 256, 0, st>>>();
        if (check_launch("build_log_table") != 0) return nullptr;
        if (cudaStreamSynchronize(st) != cudaSuccess) return nullptr;
        addr[dev] = p;
    }
    return addr[dev];
}

bool log_table_covers(const double epsl[3], const double al[3]) {
    for (int l = 0; l < 3; ++l) {
        const double lo = epsl[l] < al[l] ? epsl[l] : al[l];
        if (!(lo > 1.9073486328125e-06) || !(epsl[l] <= 1.0)) return false;      // 2^-19
    }
    return true;
}

bool log_table_window(const double epsl[3], const double al[3], cudaStream_t st, LogTabWindow& w,
                      bool with_mantissa) {
    w.g = log_table(st);
    w.lo = 0;
    w.n = kLogTabSize;
    if (w.g == nullptr) return false;
    if (!log_table_covers(epsl, al)) return true;          // SAFE kernels: table unused
    // up to y = 1: the neutral element of the branch-free T1 bodies is log(1 + 0 p) = 0
    double ymin = 1.0;
    const double ymax = 1.0;
    for (int l = 0; l < 3; ++l) {
        const double lo = epsl[l] < al[l] ? epsl[l] : al[l];
        if (lo < ymin) ymin = lo;
    }
    auto slot = [](double y) {                              // mirrors log_reduce (fcd_math.cuh)
        const double r = 1.0 / y;
        uint64_t bits;
        memcpy(&bits, &r, sizeof(bits));
        const int hi = ((int)(bits >> 32) + (1 << (19 - kLogTabBits))) & ~((1 << (20 - kLogTabBits)) - 1);
        return (hi >> (20 - kLogTabBits)) - kLogTabBase;
    };
    int lo = slot(ymax) - 4, hi = slot(ymin) + 4;           // slack: MUFU.RCP64H error, FMA rounding
    if (lo < 0 || with_mantissa) lo = 0;
    if (hi > kLogTabSize - 1) hi = kLogTabSize - 1;
    lo &= ~1;                                               // 16-byte granules: the window can be staged by one bulk copy
    w.lo = lo;
    w.n = (hi - lo + 2) & ~1;                               // kLogTabSize is even: lo + n stays inside the table
    return true;
}

ThetaDev make_theta_dev(const fcd_theta& th, int H) {
    ThetaDev d;
    memset(&d, 0, sizeof(d));
    for (int k = 0; k < 3; ++k) {
        d.mu[k] = th.mu[k];
        d.isig[k] = 1.0 / th.sigma[k];
        d.lc[k] = -log(th.sigma[k]);
        d.log_gamma[k] = log(th.gamma[k]);
        // sum_h logN_k(b_h) = -(S2 - 2 mu S1 + H mu^2) / (2 sigma^2) - H (log sigma + log sqrt(2 pi))
        // (scipy.stats.norm.logpdf, fcdiff/fit.py:114, summed at fit.py:171)
        const double i2 = 0.5 * d.isig[k] * d.isig[k];
        d.hq_a[k] = -i2;
        d.hq_b[k] = 2.0 * th.mu[k] * i2;
        const double c1 = th.mu[k] * th.mu[k] * i2 + log(th.sigma[k]) + kHalfLog2Pi;
        d.hq_c[k] = -(double)H * c1;
        d.hq_c1[k] = -c1;                                   // H * hq_c1 == hq_c exactly: only the sign moves
    }
    // fcdiff/fit.py:433-444
    d.epsl[0] = 1.0 - th.epsilon;
    d.epsl[1] = th.epsilon;
    d.epsl[2] = th.eta * th.epsilon + (1.0 - th.eta) * (1.0 - th.epsilon);
    for (int l = 0; l < 3; ++l) {
        d.al[l] = (1.0 - d.epsl[l]) * 0.5;
        d.bl[l] = d.epsl[l] - d.al[l];
    }
    d.eta = th.eta;
    d.epsilon = th.epsilon;
    d.log_pi2[0] = log(1.0 - th.pi);
    d.log_pi2[1] = log(th.pi);
    return d;
}

}  // namespace fcd

extern "C" {

int fcd_version(void) { return FCD_VERSION; }

const char* fcd_last_error(void) { return fcd::g_err; }

int fcd_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        fcd::set_error("cudaGetDevice: %s", cudaGetErrorString(e));
        return -2;
    }
    int sm = 0, major = 0, minor = 0;
    cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    if (sm_count_host) *sm_count_host = sm;
    if (cc_major_host) *cc_major_host = major;
    if (cc_minor_host) *cc_minor_host = minor;
    return 0;
}

int64_t fcd_workspace_bytes(void) { return fcd::kWsDoubles * (int64_t)sizeof(double); }

int fcd_download(void* dst_host, const void* src, int64_t bytes, void* stream) {
    if (bytes <= 0) return 0;
    cudaError_t e = cudaMemcpyAsync(dst_host, src, (size_t)bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
    if (e != cudaSuccess) {
        fcd::set_error("fcd_download: %s", cudaGetErrorString(e));
        return -2;
    }
    return 0;
}

void fcd_nvtx_push(const char* name_host) { nvtxRangePushA(name_host ? name_host : "fcd"); }

void fcd_nvtx_pop(void) { nvtxRangePop(); }

int64_t fcd_launch_count(void) { return fcd::g_launches.load(); }

void fcd_launch_count_reset(void) { fcd::g_launches.store(0); }

}  // extern "C"
