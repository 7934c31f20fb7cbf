// Host side of the device-resident (eta, epsilon) solver (fcd_solver.cuh): state set-up, the
// mapped publication block, and the wait for a batch of evaluations.
#include <chrono>
#include <cmath>
#include <cstring>

#include "fcd_solver.cuh"

namespace fcd {

__global__ void solver_init_kernel(SolverState* st, double eta, double eps, double lo0, double lo1, double hi0,
                                   double hi1, double tol, int max_evals) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    SolverState s;
    memset(&s, 0, sizeof(s));
    s.lo[0] = lo0;
    s.lo[1] = lo1;
    s.hi[0] = hi0;
    s.hi[1] = hi1;
    s.x[0] = fmin(hi0, fmax(lo0, eta));
    s.x[1] = fmin(hi1, fmax(lo1, eps));
    s.xprev[0] = s.x[0];
    s.xprev[1] = s.x[1];
    s.tol = tol;
    s.max_evals = max_evals;
    *st = s;
}

template <int K>
static void step_host(SolverState& s, const double* sums) {
    solver_step<K>(s, sums);
}

template <int K>
static void model_host(const double* sums, double eta0, double eps0, const double* z, double* out4) {
    const SeriesModel<K> m = series_model<K>(sums, eta0, eps0, -(sums[0] + sums[5]));
    double g[2], H[3];
    out4[0] = model_eval<K>(m, z, g, H);
    model_bounds<K>(m, z, out4[1], out4[2]);
    out4[3] = model_radius<K>(m, z);
}

}  // namespace fcd

using namespace fcd;

extern "C" {

int64_t fcd_solver_moments(void) { return kSolverK; }

int64_t fcd_solver_state_bytes(void) { return (int64_t)sizeof(SolverState); }
int64_t fcd_solver_published_bytes(void) { return (int64_t)sizeof(SolverPublished); }

int fcd_host_mapped_alloc(int64_t bytes, void** out_host) {
    FCD_REQUIRE(out_host != nullptr && bytes > 0, "fcd_host_mapped_alloc: bad argument");
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocMapped | cudaHostAllocPortable);
    FCD_REQUIRE(e == cudaSuccess, "fcd_host_mapped_alloc: %s", cudaGetErrorString(e));
    memset(p, 0, (size_t)bytes);
    *out_host = p;
    return 0;
}

int fcd_host_mapped_free(void* p_host) {
    if (p_host != nullptr) {
        cudaError_t e = cudaFreeHost(p_host);
        FCD_REQUIRE(e == cudaSuccess, "fcd_host_mapped_free: %s", cudaGetErrorString(e));
    }
    return 0;
}

int fcd_solver_init(void* state, double eta0, double eps0, const double* lo2_host, const double* hi2_host, double tol,
                    int32_t max_evals, void* stream) {
    FCD_REQUIRE(state != nullptr && lo2_host != nullptr && hi2_host != nullptr, "fcd_solver_init: NULL argument");
    FCD_REQUIRE(lo2_host[0] > 0.0 && lo2_host[1] > 0.0 && hi2_host[0] < 1.0 && hi2_host[1] < 1.0 &&
                lo2_host[0] <= hi2_host[0] && lo2_host[1] <= hi2_host[1] && tol >= 0.0 && max_evals >= 1,
                "fcd_solver_init: the box must lie inside (0, 1)^2");
    solver_init_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(static_cast<SolverState*>(state), eta0, eps0, lo2_host[0],
                                                           lo2_host[1], hi2_host[0], hi2_host[1], tol, max_evals);
    return check_launch("fcd_solver_init");
}

/* One optimiser transition on the HOST (the same code the evaluation kernels' last CTA runs): lets the
 * CPU tests drive the state machine with NumPy-made sums.  state_host: an fcd_solver_state initialised by
 * fcd_solver_init_host.  fcd_solver_step_host takes the six sums {obj, ge, G_2, Q_0 + Q_1, Q_2, theta-free
 * part} (the quadratic model), fcd_solver_step_host_moments the layout of kSolverVals with K moments per
 * series; fcd_solver_model_host evaluates the series model of such sums made at (eta0, eps0) at z2:
 * {value, position bound, value bound, radius}. */
int fcd_solver_init_host(void* state_host, double eta0, double eps0, const double* lo2_host, const double* hi2_host,
                         double tol, int32_t max_evals) {
    FCD_REQUIRE(state_host != nullptr && lo2_host != nullptr && hi2_host != nullptr, "fcd_solver_init_host: NULL argument");
    SolverState s;
    memset(&s, 0, sizeof(s));
    for (int i = 0; i < 2; ++i) {
        s.lo[i] = lo2_host[i];
        s.hi[i] = hi2_host[i];
    }
    s.x[0] = fmin(s.hi[0], fmax(s.lo[0], eta0));
    s.x[1] = fmin(s.hi[1], fmax(s.lo[1], eps0));
    s.xprev[0] = s.x[0];
    s.xprev[1] = s.x[1];
    s.tol = tol;
    s.max_evals = max_evals;
    memcpy(state_host, &s, sizeof(s));
    return 0;
}

int fcd_solver_step_host_moments(void* state_host, const double* sums_host, int32_t K) {
    FCD_REQUIRE(state_host != nullptr && sums_host != nullptr, "fcd_solver_step_host_moments: NULL argument");
    FCD_REQUIRE(K == 2 || K == 4 || K == 6 || K == 8, "fcd_solver_step_host_moments: K must be 2, 4, 6 or 8");
    SolverState s;
    memcpy(&s, state_host, sizeof(s));
    if (!s.done) (K == 2 ? step_host<2> : K == 4 ? step_host<4> : K == 6 ? step_host<6> : step_host<8>)(s, sums_host);
    memcpy(state_host, &s, sizeof(s));
    return 0;
}

int fcd_solver_model_host(const double* sums_host, int32_t K, double eta0, double eps0, const double* z2_host,
                          double* out4_host) {
    FCD_REQUIRE(sums_host != nullptr && z2_host != nullptr && out4_host != nullptr, "fcd_solver_model_host: NULL argument");
    FCD_REQUIRE(K == 2 || K == 4 || K == 6 || K == 8, "fcd_solver_model_host: K must be 2, 4, 6 or 8");
    (K == 2 ? model_host<2> : K == 4 ? model_host<4> : K == 6 ? model_host<6> : model_host<8>)(sums_host, eta0, eps0,
                                                                                            z2_host, out4_host);
    return 0;
}

int fcd_solver_step_host(void* state_host, const double* sums6_host) {
    return fcd_solver_step_host_moments(state_host, sums6_host, 2);
}

/* Spins until the launch `seq` of a solver batch has published; copies the state to state_out_host. */
int fcd_solver_wait(const void* published_host, uint64_t seq, void* state_out_host, int32_t timeout_ms) {
    FCD_REQUIRE(published_host != nullptr && state_out_host != nullptr, "fcd_solver_wait: NULL argument");
    const SolverPublished* pub = static_cast<const SolverPublished*>(published_host);
    const volatile unsigned long long* flag = &pub->seq;
    const auto t0 = std::chrono::steady_clock::now();
    long long spins = 0;
    while (*flag != seq) {
        if ((++spins & 0xfff) == 0) {
            const auto dt = std::chrono::steady_clock::now() - t0;
            if (std::chrono::duration_cast<std::chrono::milliseconds>(dt).count() > timeout_ms) {
                cudaError_t e = cudaGetLastError();
                set_error("fcd_solver_wait: launch %llu has not published after %d ms (%s)", (unsigned long long)seq,
                          timeout_ms, cudaGetErrorString(e));
                return -3;
            }
        }
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    const volatile double* src = reinterpret_cast<const volatile double*>(&pub->st);
    double* dst = static_cast<double*>(state_out_host);
    for (size_t i = 0; i < sizeof(SolverState) / 8; ++i) dst[i] = src[i];
    return 0;
}

}  // extern "C"
