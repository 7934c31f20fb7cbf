// Shared pieces of the correlation stage (K1).
#pragma once
#include "fcd_common.cuh"

namespace fcd {

constexpr int kKChunk = 32;     // fp32 elements per K step = 128 bytes = one SWIZZLE_128B row

inline int corr_padded_T(int T) { return (T + kKChunk - 1) / kKChunk * kKChunk; }

#ifdef __CUDACC__
// clip to [-1, 1]; Fisher z = atanh(r) when requested.  Collinear or duplicated regions give |r| = 1
// (and rounding can push a near-collinear pair there): z is taken at the largest magnitude below 1
// (1 - 2^-53 -> |z| = 18.7; 1 - 2^-24 -> 8.7 on the fp32 path), so that no +-inf reaches the fit, where
// it would turn the free energy and the (eta, epsilon) objective into NaN.  A row of zero variance is
// standardised to zeros (standardise_kernel): r = 0 against every other region.
__device__ __forceinline__ double corr_epilogue(double r, int fisher) {
    r = fmin(1.0, fmax(-1.0, r));
    if (!fisher) return r;
    const double lim = 0.99999999999999988897769753748;     // 1 - 2^-53
    return atanh(fmin(lim, fmax(-lim, r)));
}
// Same for an fp32 accumulator of the tensor-core path: the Gram entry carries
// ~1e-6 of TF32 accumulation error, so fp32 transcendental precision (rel. 1e-7)
// loses nothing; atanh(r) = (log1p(r) - log1p(-r)) / 2 is accurate for small |r|.
__device__ __forceinline__ double corr_epilogue_f32(float r, int fisher) {
    r = fminf(1.0f, fmaxf(-1.0f, r));
    if (!fisher) return (double)r;
    const float lim = 0.99999994f;                           // 1 - 2^-24, the largest float below 1
    r = fminf(lim, fmaxf(-lim, r));
    return (double)(0.5f * (log1pf(r) - log1pf(-r)));
}
#endif

// Tensor-core Gram + epilogue (fcd_corr_tc.cu): Zh / Zl are the TF32 hi / lo
// parts of the standardised rows, [S*N][Tp] fp32 each, 1024-byte aligned.
bool corr_tc_supported(int N);
int corr_gram_tc(const float* Zh, const float* Zl, int S, int N, int Tp, double* out, int64_t pitch, int s0,
                 int fisher, cudaStream_t st);

// fcd_corr.cu: the Gram + epilogue of fcd_corr_fisherz on the tensor-core (tc) or SIMT path; corr_use_tc
// is the path fcd_corr_fisherz takes for N (FCD_CORR_SIMT forces SIMT).  The masked standardisation
// (standardise_kernel<SPLIT, true>) and the NaN marking of the rows it flags, for fcd_corr_fisherz_clean.
bool corr_use_tc(int N);
int corr_gram(bool tc, const float* Z, const float* Zlo, int S, int N, int Tp, double* out, int64_t pitch, int s0,
              int fisher, cudaStream_t st);
int corr_standardise_masked(bool tc, const float* ts, const uint8_t* keep, int S, int N, int T, int Tp, float* Z,
                            float* Zlo, uint8_t* status, cudaStream_t st);
int corr_mark_status(const uint8_t* status, int S, int N, double* out, int64_t pitch, int s0, cudaStream_t st);

// fp64 forms of the two standardisations for fcd_corr_partial: the same rows as fcd_corr_fisherz_clean forms
// (K == 0: standardise_kernel<false, true>; K >= 1: confound_basis_kernel into Q [S][K][Tp], then
// clean_kernel), stored as fp64 Z [S][N][Tp] without the rounding to fp32.
int corr_standardise_masked_f64(const float* ts, const uint8_t* keep, int S, int N, int T, int Tp, double* Z,
                                uint8_t* status, cudaStream_t st);
int corr_clean_f64(const float* ts, const uint8_t* keep, const double* confounds, int S, int N, int T, int Tp, int K,
                   double* Q, double* Z, uint8_t* status, int32_t* rank, cudaStream_t st);

}  // namespace fcd
