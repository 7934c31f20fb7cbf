/*
 * fcdiff_b200 -- C-ABI of the B200-native hot path of andy-sweet/fcdiff
 * (variational EM for the individual-anomalous-region model).
 *
 * The reference is pure Python and has no FFI of its own (SURVEY.md 8b): the
 * drop-in boundary is its Python surface (fcdiff.fit / fcdiff.model /
 * fcdiff.util), re-implemented in the package `fcdiff_b200` (alias `fcdiff`)
 * which binds THIS library with ctypes.  Each entry point below cites the
 * reference function (path:line under the reference tree) it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - arrays are float64, C-contiguous, row pitch given in ELEMENTS;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *   - every call returns 0 on success, <0 on error; fcd_last_error() gives the
 *     text of the last error raised on the calling thread;
 *   - no entry point allocates device memory: scratch comes from `ws`
 *     (a device buffer of at least fcd_workspace_bytes() bytes, zero-filled
 *     once by the caller before first use; calls restore it to zero);
 *   - edge order is the reference's lower-triangular row-major order
 *     c = n(n-1)/2 + m, m < n (fcdiff/util.py:40-84);
 *   - an edge shard is the contiguous range [c0, c0 + C) of the global edge
 *     list; `N` is always the global number of regions.
 */
#ifndef FCDIFF_B200_H
#define FCDIFF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FCD_VERSION 123

#if defined(__GNUC__)
#define FCD_API __attribute__((visibility("default")))
#else
#define FCD_API
#endif

/* Model parameters theta (fcdiff/model.py:31-38). */
typedef struct fcd_theta {
    double pi;        /* P(region anomalous)                                   */
    double eta;       /* P(edge anomalous | exactly one end-point anomalous)   */
    double epsilon;   /* P(typical edge differs from the template)             */
    double gamma[3];  /* template state prior (negative, none, positive)       */
    double mu[3];     /* Gaussian means per state                              */
    double sigma[3];  /* Gaussian standard deviations per state                */
} fcd_theta;

enum { FCD_LOOKUP_REFERENCE = 0, FCD_LOOKUP_SYMMETRIC = 1 };

/* ------------------------------------------------------------------ runtime */
FCD_API int fcd_version(void);
FCD_API const char* fcd_last_error(void);
/* SM count and compute capability of the current device. */
FCD_API int fcd_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host);
FCD_API int64_t fcd_workspace_bytes(void);
/* Copies `bytes` from device memory to (pinned) host memory on `stream` and
 * waits for the stream: how the few doubles a reduction kernel leaves behind
 * reach the host-side optimiser / convergence test. */
FCD_API int fcd_download(void* dst_host, const void* src, int64_t bytes, void* stream);
/* Number of kernels this library has launched in this process (bench.py's
 * `gpu_launches`), and reset. */
FCD_API int64_t fcd_launch_count(void);
FCD_API void fcd_launch_count_reset(void);
/* NVTX range around a kernel family (profiling aid, SURVEY 5 "tracing / profiling": the reference has
 * none).  `name_host` is copied by the tools; ranges nest per thread.  No-ops without a profiler. */
FCD_API void fcd_nvtx_push(const char* name_host);
FCD_API void fcd_nvtx_pop(void);

/* ------------------------------------------------------- small exchanges    */
/* One-shot all-reduce (sum) of n <= fcd_comm_max_vals() doubles over NVLink peer
 * memory, result delivered to the host without a copy or a stream synchronisation
 * (csrc/fcd_comm.cu).  Replaces, for the edge-sharded fit, the NCCL all-reduce +
 * download after every reduction kernel: the M-step sums (fcdiff/fit.py:208-220),
 * the objective / gradient partial sums of every (eta, epsilon) evaluation
 * (fit.py:270-286) and the energy terms (fit.py:142-155).
 *   window: fcd_comm_window_bytes() of device memory per rank, created here (the one
 *     explicit allocation of this library), exported / opened as a CUDA IPC handle of
 *     fcd_comm_handle_bytes() bytes; windows_host[world] lists every rank's window in
 *     THIS process' address space (own window at [rank]);
 *   result_host: mapped pinned memory from fcd_host_result_alloc;
 *   seq: 1, 2, 3, ... -- the same on every rank for the same exchange;
 *   fcd_allreduce_small launches one kernel on `stream`: vec (device, in place) and
 *     result_host receive the sums, formed in rank order (bit-identical on all ranks);
 *     world == 1 publishes vec to the host only;
 *   fcd_wait_result spins until exchange seq has been published, copies n doubles. */
FCD_API int64_t fcd_comm_window_bytes(void);
FCD_API int32_t fcd_comm_handle_bytes(void);
FCD_API int32_t fcd_comm_max_world(void);
FCD_API int32_t fcd_comm_max_vals(void);
FCD_API int fcd_comm_window_create(void** window_out_host);
FCD_API int fcd_comm_window_destroy(void* window);
FCD_API int fcd_comm_window_export(void* window, void* handle_host);
FCD_API int fcd_comm_window_open(const void* handle_host, void** peer_window_out_host);
FCD_API int fcd_comm_window_close(void* peer_window);
FCD_API int fcd_host_result_alloc(void** result_out_host);
FCD_API int fcd_host_result_free(void* result_host);
FCD_API int fcd_allreduce_small(double* vec, int32_t n, void* const* windows_host, int32_t rank, int32_t world,
                        uint64_t seq, double* result_host, void* stream);
/* The same exchange; behind the n sums, result_host also receives this rank's OWN values
 * vec[keep0 .. keep0 + nkeep) as they were before the sum (n + nkeep <= fcd_comm_max_vals()): one wait
 * serves the M-step sums of fit.py:208-220, the record counts of all ranks (total: which form the
 * (eta, epsilon) evaluations take, identical on every rank) and of this rank (the size of its lists). */
FCD_API int fcd_allreduce_small_keep(double* vec, int32_t n, int32_t keep0, int32_t nkeep, void* const* windows_host,
                             int32_t rank, int32_t world, uint64_t seq, double* result_host, void* stream);
FCD_API int fcd_wait_result(const double* result_host, int32_t n, uint64_t seq, double* out_host, int32_t timeout_ms);
/* Staging of the all-gather of the region posteriors `_lq_R` / exp(_lq_R) ((N, U, 2), fcdiff/fit.py:176-198)
 * when patients are sharded: pack this rank's columns [u0, u0+Ul) of both arrays into one
 * contiguous block [2][N][ch][2] (ch columns per rank, zero padded); unpack the gathered
 * [world][2][N][ch][2] into the two full arrays. */
FCD_API int fcd_pack_patients(const double* lqR, const double* qR, int32_t N, int32_t U, int32_t u0, int32_t Ul,
                      int32_t ch, double* out, void* stream);
FCD_API int fcd_unpack_patients(const double* gathered, int32_t world, int32_t N, int32_t U, int32_t ch, double* lqR,
                        double* qR, void* stream);

/* ------------------------------------------------------- index arithmetic   */
/* fcdiff/util.py:62-84 c_to_nm for c in [c0, c0+C): n_out[i], m_out[i] int32. */
FCD_API int fcd_c_to_nm(int64_t c0, int64_t C, int32_t* n_out, int32_t* m_out, void* stream);

/* ------------------------------------------------------- fused hot path     */
/* Healthy-subject sufficient statistics, computed once per fit:
 *   S1[c] = sum_h b[c,h],  S2[c] = sum_h b[c,h]^2.
 * They replace the (C,H,3) cache `_lp_B_g_F` of fcdiff/fit.py:111-114: the
 * healthy log-density sum of fit.py:171 is a quadratic in (S1, S2).
 * S0 == NULL: every b[c,h] is taken as observed.  S0 != NULL, for missing entries (fit.missing =
 * "marginalize"): a NaN b[c,h] is not observed and is left out of S1, S2; S0[c] = H_c, the number of observed
 * controls of edge c (a double).  The healthy sum of fit.py:171 over the observed entries is
 * hq_a S2 + hq_b S1 + H_c hq_c1: the constant scales with H_c, so it cannot be folded into S1, S2.  With no NaN,
 * S1 and S2 have the bits of the S0 == NULL form and S0 = H.  The kernels below that take S0 read it the same
 * way: NULL means every edge has all H controls, and S0 = H gives the bits of the NULL form. */
FCD_API int fcd_healthy_stats(const double* b, int64_t C, int32_t H, int64_t pitchH,
                      double* S1, double* S2, double* S0, void* stream);

/* Edge table of the local shard: nm[i] = n | m << 16 for the edge c0 + i
 * (fcdiff/util.py:62-84 c_to_nm; at most 65535 regions).  Built once per fit. */
FCD_API int fcd_edge_table(int64_t c0, int64_t C, int32_t* nm, void* stream);

/* Responsibility planes, built once per fit (the reference never re-estimates
 * mu, sigma, fcdiff/fit.py:232-237): for every patient correlation x = bt[c,u]
 * with N_k = N(x; mu_k, sigma_k) (fit.py:115),
 *   P[k][c][u] = N_k / (N_0 + N_1 + N_2)   (three planes, `planeStride` elements apart)
 *   L[c][u]    = log(N_0 + N_1 + N_2)      (may be NULL)
 * each with the shape and pitch of bt.  Then (fit.py:117-122, 409-444)
 *   log M_kl = L + log(a_l + b_l p_k),  a_l = (1 - eps_l)/2,  b_l = eps_l - a_l,
 * exactly and without underflow; the kernels below read these planes, not bt.
 * missing = 1 for patient correlations with missing entries: a NaN bt[c,u] is not observed and is stored as
 * p_0 = p_1 = p_2 = 1/3, L = log 3.  Then a_l + b_l / 3 = 1/3 for every l and theta, log M_kl = 0 for all
 * (k, l) (fit.py:117-122): the element's density factor is 1 in every kernel that reads the planes.  Finite
 * entries get the bits of missing = 0.  Any other value of `missing` is rejected. */
FCD_API int fcd_resp_cache(const double* bt, int64_t C, int32_t U, int64_t pitchU,
                   const fcd_theta* theta_host, double* P, int64_t planeStride, double* L, int32_t missing,
                   void* stream);

/* Peak states of the posteriors (tier selection, DESIGN.md "Tiers"):
 *   fstate[c]   = k if qF[c,k] == 1.0 and the other two <= 2^-60, else 3;
 *   rstate[n][u] = s if qR[n,u,s] == 1.0 and the other <= 2^-60, else 2;
 *                  4 in the padding columns u >= U (row pitch pitchS, a multiple of 256).
 * A term whose weight is <= 2^-60 is below the rounding error of the sums it
 * would enter and is skipped by the kernels below. */
FCD_API int fcd_peak_states_F(const double* qF, int64_t C, uint8_t* fstate, void* stream);
FCD_API int fcd_peak_states_R(const double* qR, int32_t N, int32_t U, int64_t pitchS, uint8_t* rstate, void* stream);

/* MAP labels of a log-posterior array lq [n][width]: labels[i] = argmax_k lq[i][k]
 * (first maximum on ties).  width 3: template state of an edge (q_F of
 * fit.py:157-174); width 2: anomaly flag of a (region, patient) pair (q_R of
 * fit.py:176-198). */
FCD_API int fcd_map_labels(const double* lq, int64_t n, int32_t width, uint8_t* labels, void* stream);

/* K2 -- E-step for the template posterior; replaces `_update_lq_F`
 * (fcdiff/fit.py:157-174) + `_eval_q_R_w` (fit.py:382-406) + the patient half
 * of `_update_lps` (fit.py:115-122) + `_eval_M` (fit.py:409-444).
 *   lqF[c,k] = log gamma_k + sum_h logN_k(b[c,h])
 *            + sum_u sum_l w_l(n,m,u) log M_kl(bt[c,u]),  minus logsumexp_k.
 * P: planes of the local edge rows; qR [N][U][2] probabilities, rstate their peak
 * states; nm the shard's edge table.  Outputs lqF [C][3] and qF=exp(lqF) [C][3].
 * S0 (may be NULL) of fcd_healthy_stats: the healthy sum of fit.py:171 over the observed controls. */
FCD_API int fcd_estep_qF(const double* S1, const double* S2, const double* S0, int32_t H,
                 const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                 const double* qR, const uint8_t* rstate, int64_t pitchS, int32_t N, const int32_t* nm,
                 const fcd_theta* theta_host, double* lqF, double* qF, void* stream);

/* The same E-step driven by the code pass of the previous M-step (fcd_code_plane / fcd_code_records:
 * valid while q_R has not changed since): the coded elements need no peak-state decoding and no
 * queue -- one code byte selects the constants of a running product -- and the elements with a
 * mixed region are taken from the row's key lists (half records: three differences of logs with
 * one weight; full records: nine logs).  code / counts / keysF / keysH / rowoff / Hh as written by
 * the code pass for the same local rows; rows whose edge was unpeaked then (counts[c][0] == 3 U)
 * are evaluated in full.  S0 (may be NULL) of fcd_healthy_stats (fit.py:157-174 over the observed controls).
 * solver_state == NULL: eta and epsilon come from theta_host, and eps_lo / eps_hi are ignored.
 * solver_state != NULL (device, fcd_solver_init, 8-byte aligned): the E-step of the NEXT iteration, enqueued
 * behind a device-resident (eta, epsilon) solve (fcd_elm_coded_solve / fcd_elm_tiered_solve,
 * fcdiff/fit.py:228-241) whose result the host has not read yet: eta and epsilon are taken from `solver_state` on
 * the device when the kernel starts (theta_host supplies gamma, mu, sigma; its eta / epsilon are ignored);
 * [eps_lo, eps_hi] (0 < eps_lo <= eps_hi < 1) is the epsilon box of that solve and sizes the logarithm table.
 * The reference runs these steps one after the other (fit.py:73-79); here the E-step fills the GPU while the
 * host waits for the solve and the free energy.  The caller discards lqF / qF when the solve had not finished in
 * the launches enqueued before (state.done == 0), ended pinned at the box, or the fit stops. */
FCD_API int fcd_estep_qF_coded(const double* S1, const double* S2, const double* S0, int32_t H,
                       const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                       const double* qR, int32_t N, const int32_t* nm,
                       const uint8_t* code, int64_t pitchQ, const int32_t* counts, const uint64_t* keysF,
                       const uint64_t* keysH, const int64_t* rowoff, const double* Hh,
                       const fcd_theta* theta_host, const void* solver_state, double eps_lo, double eps_hi,
                       double* lqF, double* qF, void* stream);

/* The uniform start (fcdiff/fit.py:84-102: lq_R = -ln 2, lq_F = -ln 3 everywhere).  With a CONSTANT q_R every
 * element has the same pair weights w (fit.py:382-406), and the sums of fit.py:165-173 / 489-511 factor through
 *   S9[c][k*3 + l] = sum_u log(a_l + b_l p_k(c,u))       (a_l, b_l: fit.py:427-444 relative to the total density)
 * -- nine running products per row instead of nine logarithms per element (csrc/fcd_uniform.cu):
 *   fcd_row_logsums: S9 [C][9] from the planes P_0, P_1 ([C][pitchU], 16-byte aligned rows);
 *   fcd_estep_qF_rowsums: `_update_lq_F` (fit.py:157-174) from S9 and w3_host = {q0^2, q1^2, 2 q0 q1}, with S0
 *     (may be NULL) of fcd_healthy_stats (the healthy sum over the observed controls);
 *   fcd_elm_rowsums: out1[0] = sum_c sum_k qF[c,k] sum_l w_l S9[c][k][l], the theta-dependent part of E_lM
 *     (fit.py:489-511); the theta-free part is (sum_l w_l) sum_c (sum_k qF[c,k]) sum_u L[c,u]. */
FCD_API int fcd_row_logsums(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                    const fcd_theta* theta_host, double* S9, void* stream);
FCD_API int fcd_estep_qF_rowsums(const double* S1, const double* S2, const double* S0, int32_t H,
                         const double* S9, int64_t C, const double* w3_host, const fcd_theta* theta_host,
                         double* lqF, double* qF, void* stream);
FCD_API int fcd_elm_rowsums(const double* S9, const double* qF, int64_t C, const double* w3_host, double* out1,
                    double* ws, void* stream);

/* Replica sweeps (BASELINE.json configs[4]; no reference counterpart -- the reference stops at one
 * fit, fcdiff/fit.py:56-82): the responsibility planes of ALL S subjects are built once
 * (fcd_resp_cache on every column of the (C, S) correlation matrix), and a relabelling selects from
 * them (csrc/fcd_replica.cu):
 *   fcd_healthy_stats_cols: S1 / S2 (and S0, may be NULL) of fcd_healthy_stats over the columns cols[0..H) of
 *     X [C][pitchS]; with S0 != NULL only the observed (non-NaN) entries are summed;
 *   fcd_gather_columns: dst[p][c][j] = src[p][c][cols[j]], j < U (columns U..pitchD-1 zero), p < nplanes.
 * cols: int32 device array. */
FCD_API int fcd_healthy_stats_cols(const double* X, int64_t C, int64_t pitchS, const int32_t* cols, int32_t H,
                           double* S1, double* S2, double* S0, void* stream);
FCD_API int fcd_gather_columns(const double* src, int64_t planeStrideS, int64_t pitchS, int32_t nplanes, int64_t C,
                       const int32_t* cols, int32_t U, double* dst, int64_t planeStrideD, int64_t pitchD,
                       void* stream);

/* K2b part 1 -- q_R-independent half of `_update_lq_R` (fcdiff/fit.py:187-194) for the patients [u0, u0 + Ul),
 * from the E-step's edge-major responsibility planes Pe [3][C][pitchU] (fcd_resp_cache):
 *   W_l[c,u] = sum_k qF[c,k] * log M_kl(bt[c][u])
 * up to an additive per-(c,u) constant common to all l, which cancels in the
 * normalisation of fit.py:196 (see DESIGN.md).  Only l_0 - l_1 survives that
 * normalisation, so the tensor holds two numbers per edge-patient (16 bytes):
 *   WT[u][c] = { W_0 - W_2, W_2 - W_1 }     ([Ul][C][2], patient-major)
 * qF / fstate cover ALL edges.
 * PsT / kcache: caller-kept [Ul][pitchC] plane of each edge's dominant-state
 * responsibility and the [C] states it was gathered for (255 = never; set by the
 * caller once).  The call first refreshes the columns of edges whose state changed
 * (fcd_pstar_refresh_em: one transposing pass over those edges' rows of Pe, all of
 * them the first time) and then reads one coalesced plane instead of three; the
 * three-plane path of an unpeaked edge reads Pe with a stride. */
FCD_API int fcd_region_weights_em(const double* Pe, int64_t planeStride, int64_t pitchU, int32_t u0, int32_t Ul, int64_t C,
                          int64_t pitchC, const double* qF, const uint8_t* fstate, double* PsT, uint8_t* kcache,
                          const fcd_theta* theta_host, double* WT, void* stream);
/* The refresh of PsT / kcache alone (see fcd_region_weights_em) for the current peak
 * states, without computing region weights. */
FCD_API int fcd_pstar_refresh_em(const double* Pe, int64_t planeStride, int64_t pitchU, int32_t u0, int32_t Ul, int64_t C,
                         int64_t pitchC, const uint8_t* fstate, double* PsT, uint8_t* kcache, void* stream);

/* K2b part 2 -- Gauss-Seidel sweep of `_update_lq_R` (fcdiff/fit.py:176-198)
 * for the patients [u0, u0+Ul) from WT [Ul][C][2] (fcd_region_weights_em).  qR/lqR are the full [N][U][2] arrays; only
 * the [u0, u0+Ul) columns are read and written.  log_pi2_host = {log(1-pi),
 * log(pi)} (the 2-vector convention of test_fcdiff/test_fit.py:477-487).
 * edge_lookup: FCD_LOOKUP_REFERENCE reproduces nm_to_c(n, m) for all m != n
 * (fit.py:185-186, SURVEY 0.3), FCD_LOOKUP_SYMMETRIC the unordered pair. */
FCD_API int fcd_estep_qR(const double* WT, int64_t C, int32_t N, int32_t U, int32_t u0, int32_t Ul,
                 const double* log_pi2_host, int32_t edge_lookup,
                 double* qR, double* lqR, void* stream);

/* K3a -- M-step sums; replaces `_update_pi` / `_update_gamma`
 * (fcdiff/fit.py:208-220).  out[0..2] = sum_c exp(lqF[c,k]),
 * out[3] = sum_{n,u} exp(lqR[n,u,1]).  The caller divides by counts (after an
 * all-reduce of out[0..2] when edges are sharded). */
FCD_API int fcd_mstep_stats(const double* lqF, int64_t C, const double* lqR, int64_t NU,
                    double* out4, double* ws, void* stream);

/* K3b -- objective and analytic gradient of the (eta, epsilon) sub-problem;
 * replaces `_opt_fun` (fcdiff/fit.py:270-286) = `_update_lps` + `_eval_E_lM`
 * (fit.py:489-511) and `_eval_dE_dh` / `_eval_dE_de` / `_eval_dlM_dh` /
 * `_eval_dlM_de` (fit.py:600-697) in ONE pass over the responsibility planes
 * (one plane, 8 bytes per edge-patient, wherever the posteriors are peaked).
 *   out[0] = sum_c sum_k qF[c,k] sum_u sum_l w_l log(a_l + b_l p_k)
 *            E_lM = out[0] + fcd_elm_const (the part independent of eta, epsilon)
 *   out[1] = dE/d eta, out[2] = dE/d epsilon   (of E = -E_lM; only if want_grad) */
FCD_API int fcd_elm_obj_grad(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                     const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate,
                     int64_t pitchS, int32_t N, const int32_t* nm,
                     const fcd_theta* theta_host, int32_t want_grad,
                     double* out3, double* ws, void* stream);

/* out1[0] = sum_c (sum_k qF[c,k]) sum_u (sum_l w_l) L[c,u]: the part of E_lM
 * (fit.py:489-511) that does not depend on (eta, epsilon). */
FCD_API int fcd_elm_const(const double* L, int64_t C, int32_t U, int64_t pitchU,
                  const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate,
                  int64_t pitchS, int32_t N, const int32_t* nm, double* out1, double* ws, void* stream);

/* K3b over the coded dominant-state plane (DESIGN.md "Coded plane").  Between two
 * E-steps the optimiser evaluates E_lM(eta, epsilon) many times with q_F, q_R fixed
 * (fit.py:228-241): the code pass turns the planes into what an evaluation needs
 * and nothing else --
 *   PsE  [C][pitchQ] f64: responsibility of each edge's dominant state (rows re-gathered
 *        from P only when kcache[c] != fstate[c]; kcache starts at 255, PsE zero-filled);
 *        pitchQ = fcd_code_pitch(U): U rounded up to 16, so that code rows are 16-byte aligned;
 *   code [C][pitchQ] u8 (+ 16 bytes of slack): l* in 0..2 for elements whose edge and
 *        regions are peaked (weight exactly 1, one log); 4 + s for an element with ONE undecided,
 *        normalised region and the other in state s -- it counts as l = 2 with weight 1 and
 *        adds a half record; 3 for all others;
 *   half records {p, +-q_s} (16 bytes, sign bit = s), nh of them: the correction
 *        q_s (log M_s - log M_2) of the elements coded 4 + s (fit.py:382-406 with q_0 + q_1 = 1);
 *   records {p, w_0, w_1, w_2} (32 bytes) for all other elements, nd of them
 * -- and fcd_elm_coded reduces them: 9 bytes per edge-patient per evaluation, no row
 * structure, no partition of the elements.
 *   fcd_plane_sum: out1[0] = sum of a [C][U] plane -- the total of the L plane, once per cache;
 *   fcd_code_plane: refreshes PsE, writes code, counts[c] = {records, half records} of row c
 *     (int32 x 2), blockoff: scratch of 4 * fcd_bucket_blocks(C) int64 (totals and exclusive
 *     prefix sums of blocks of 16 rows), total2 = {nd, nh} (as doubles);
 *   fcd_code_records: D receives the nd records, Hh the nh half records; keysF [nd] / keysH [nh]
 *     uint64 = (tag << 48 | c << 16 | u) of every record / half record and rowoff [C][2] int64 =
 *     first key of each row in either list are kept for fcd_estep_qF_coded (not written when
 *     nd + nh == 0); out1[0] = the theta-free part of E_lM
 *     (same value as fcd_elm_const), formed as Lsum[0] (device, from fcd_plane_sum)
 *     corrected by the record elements only;
 *   fcd_elm_coded: nE = C * pitchQ elements of PsE / code; out3 as fcd_elm_obj_grad. */
FCD_API int64_t fcd_bucket_blocks(int64_t C);
FCD_API int64_t fcd_code_pitch(int32_t U);
FCD_API int fcd_plane_sum(const double* X, int64_t C, int32_t U, int64_t pitchU, double* out1, double* ws,
                  void* stream);
FCD_API int fcd_code_plane(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                   const uint8_t* fstate, const uint8_t* rstate, int64_t pitchS, const int32_t* nm,
                   double* PsE, uint8_t* kcache, uint8_t* code, int64_t pitchQ, int32_t* counts, int64_t* blockoff,
                   double* total2, void* stream);
FCD_API int fcd_code_records(const double* P, int64_t planeStride, const double* PsE, const uint8_t* code,
                     int64_t pitchQ, const double* L, const double* Lsum, int64_t C, int32_t U, int64_t pitchU,
                     const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate, int64_t pitchS,
                     int32_t N, const int32_t* nm, const int32_t* counts, const int64_t* blockoff,
                     uint64_t* keysF, uint64_t* keysH, int64_t* rowoff, double* D, int64_t nd, double* Hh, int64_t nh,
                     double* out1, double* ws, void* stream);
FCD_API int fcd_elm_coded(const double* PsE, const uint8_t* code, int64_t nE, const double* D, int64_t nd,
                  const double* Hh, int64_t nh, const fcd_theta* theta_host, int32_t want_grad, double* out3,
                  double* ws, void* stream);

/* ------------------------------------------- device-resident (eta, epsilon) solver */
/* Replaces the host optimiser of fcdiff/fit.py:228-241 (scipy.optimize.minimize on
 * [1e-5, 1 - 1e-5]^2, objective fit.py:270-286 = -E_lM, gradient fit.py:600-697): a safeguarded
 * projected Newton iteration whose step is taken by the LAST CTA of every evaluation kernel
 * (csrc/fcd_solver.cuh) -- the evaluations of one solve are enqueued back to back and read the
 * iterate from device memory; nothing returns to the host between them.  With edge shards the
 * same CTA first exchanges the six partial sums over the peer windows (fcd_comm_window_*), in rank
 * order, so every rank takes bit-identical steps.
 *   state: fcd_solver_state_bytes() of device memory, set by fcd_solver_init (box lo/hi per
 *     parameter, start point, `tol`: a step with |dx_i| <= tol * min(x_i, 1 - x_i) for both parameters is
 *     taken without another evaluation and ends the solve -- it leaves a relative error ~ tol^2 behind;
 *     max_evals bounds the evaluations);
 *   fcd_elm_coded_solve / fcd_elm_tiered_solve: n_launches evaluations of the coded-plane /
 *     tiered form (arguments as fcd_elm_coded / fcd_elm_obj_grad) at the state's iterate; launches
 *     after the solve has finished exit at once.  [eps_lo, eps_hi] must contain the box of epsilon
 *     (it sizes the shared-memory logarithm table).  konst (device, may be NULL): this rank's
 *     theta-free part of E_lM (fcd_code_records / fcd_elm_const), added to the objective.
 *     published_host: fcd_host_mapped_alloc(fcd_solver_published_bytes()) -- every launch stores
 *     the state there followed by its sequence number seq0 + i;
 *   fcd_solver_wait spins (host) until launch `seq` has published and copies the state
 *     (fcd_solver_state_bytes(), layout `fcd_solver_state` below) to state_out_host. */
typedef struct fcd_solver_state {
    double x[2];         /* (eta, epsilon): next evaluation point; the solution when done */
    double xprev[2];
    double fprev;
    double f;            /* -E_lM at x when done (incl. the theta-free part) */
    double g[2];         /* gradient at the last evaluated point */
    double lo[2], hi[2];
    double tol;
    double step;
    int32_t have_prev, nfev, nback;
    int32_t done;        /* 0 running; 1 converged; 2 stopped (budget / no descent / non-finite); 3 peer time-out */
    int32_t max_evals, pad_;
} fcd_solver_state;
FCD_API int64_t fcd_solver_state_bytes(void);
FCD_API int64_t fcd_solver_published_bytes(void);
FCD_API int fcd_host_mapped_alloc(int64_t bytes, void** out_host);
FCD_API int fcd_host_mapped_free(void* p_host);
FCD_API int fcd_solver_init(void* state, double eta0, double eps0, const double* lo2_host, const double* hi2_host,
                    double tol, int32_t max_evals, void* stream);
FCD_API int fcd_elm_coded_solve(const double* PsE, const uint8_t* code, int64_t nE, const double* D, int64_t nd,
                        const double* Hh, int64_t nh, double eps_lo, double eps_hi, void* state, const double* konst,
                        void* const* windows_host, int32_t rank, int32_t world, void* published_host, uint64_t seq0,
                        int32_t n_launches, double* ws, void* stream);
FCD_API int fcd_elm_tiered_solve(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                         const double* qF, const uint8_t* fstate, const double* qR, const uint8_t* rstate,
                         int64_t pitchS, int32_t N, const int32_t* nm, double eps_lo, double eps_hi, void* state,
                         const double* konst, void* const* windows_host, int32_t rank, int32_t world,
                         void* published_host, uint64_t seq0, int32_t n_launches, double* ws, void* stream);
/* Host-side twins of fcd_solver_init and of the optimiser transition the kernels' last CTA runs (same code):
 * sums6_host = {obj, ge, G_2, Q_0 + Q_1, Q_2, theta-free part} at state.x (csrc/fcd_solver.cuh). */
FCD_API int fcd_solver_init_host(void* state_host, double eta0, double eps0, const double* lo2_host,
                         const double* hi2_host, double tol, int32_t max_evals);
FCD_API int fcd_solver_step_host(void* state_host, const double* sums6_host);
/* The same with K moments per series (K = 2, 4, 6, 8): sums = the six above, then A_3..A_K, B_3..B_K
 * (csrc/fcd_solver.cuh, series model); the evaluation kernels deliver fcd_solver_moments() of them.
 * fcd_solver_model_host: the series model of such sums made at (eta0, eps0), at z2 = (eta, eps):
 * out4 = {model value, position bound, value bound, trust-region radius}. */
FCD_API int64_t fcd_solver_moments(void);
FCD_API int fcd_solver_step_host_moments(void* state_host, const double* sums_host, int32_t K);
FCD_API int fcd_solver_model_host(const double* sums_host, int32_t K, double eta0, double eps0, const double* z2_host,
                                  double* out4_host);
FCD_API int fcd_solver_wait(const void* published_host, uint64_t seq, void* state_out_host, int32_t timeout_ms);

/* K4 -- free-energy terms; replaces `_eval_energy` and `_eval_E_*`
 * (fcdiff/fit.py:142-155, 447-539).  out[0..5] = E_lp_F, E_lp_B_g_F, E_lp_R,
 * E_lM, E_lq_F, E_lq_R over the local edge shard (terms 2 and 5 involve q_R
 * only and are complete on every rank).  qF = exp(lqF), qR = exp(lqR) as left
 * by fcd_estep_qF / fcd_estep_qR (fit.py:146-147); lqF / qF / S1 / S2 are the
 * shard's C rows.  `elm` = E_lM of the shard (fcd_elm_obj_grad + fcd_elm_const
 * at the same q_F, q_R, theta); or, with `solver_state` != NULL (device, fcd_solver_init): the E_lM
 * of the device-resident (eta, epsilon) solve enqueued before this call on the same stream (the
 * GLOBAL value: pass it on one rank only) -- NaN if that solve has not finished.  S0 (may be NULL) of
 * fcd_healthy_stats: E_lp_B_g_F (fit.py:461-472) over the observed controls. */
FCD_API int fcd_energy_terms(const double* S1, const double* S2, const double* S0, int32_t H,
                     const double* lqF, const double* qF, int64_t C,
                     const double* lqR, const double* qR, int32_t N, int32_t U,
                     const fcd_theta* theta_host, double elm, const void* solver_state,
                     double* out6, double* ws, void* stream);

/* Held-out scoring (csrc/fcd_patients.cu): with theta and q_F of a fitted model fixed, the free energy
 * (fcdiff/fit.py:142-155) is a sum over patient columns u; these entries keep the sums of `_eval_E_lp_R`,
 * `_eval_E_lM` and `_eval_E_lq_R` (fit.py:475-539) per patient instead of reducing them to one scalar.
 *   fcd_patient_terms: out4 [U][4] = {E_lM,u, E_lp_R,u, E_lq_R,u, sum_c sum_k qF[c,k] log M_k0(c,u)} -- the
 *     last is E_lM,u with every region typical.  The pair weights are those of the edge's own regions
 *     (n, m) = c_to_nm(c) (fit.py:489-511).  P / L: planes of the scored patients (fcd_resp_cache, all C edges);
 *     qF / fstate: q_F and its peak states; qR / lqR [N][U][2]; theta_host supplies pi, eta, epsilon.
 *     ws: fcd_patient_terms_ws_bytes(C, U) bytes of device scratch (no zero fill needed).  A patient's sums
 *     are bit-identical whichever other patients are scored in the same call: the row partition depends
 *     on C only and the partials are added in a fixed order.
 *   fcd_qR_change: out1[0] = max(out1[0], max_{n,u,s} |qR_new - qR_old|) over [N][U][2] (the caller zeroes out1
 *     first; the maximum of the region sweeps of fit.py:176-198 between two iterates); maxU [U] (may be NULL)
 *     receives each patient's maximum.  A NaN difference propagates. */
FCD_API int64_t fcd_patient_terms_ws_bytes(int64_t C, int32_t U);
FCD_API int fcd_patient_terms(const double* P, int64_t planeStride, const double* L, int64_t C, int32_t U, int64_t pitchU,
                      const double* qF, const uint8_t* fstate, const double* qR, const double* lqR, int32_t N,
                      const fcd_theta* theta_host, double* out4, double* ws, void* stream);
FCD_API int fcd_qR_change(const double* qR_old, const double* qR_new, int32_t N, int32_t U, double* maxU, double* out1,
                  void* stream);

/* Posteriors of the anomalous connections T and of the patients' connection states F~ (csrc/fcd_patients.cu;
 * no reference counterpart: the reference sums T and F~ out into M_kl, fcdiff/fit.py:409-444, and the sampler
 * draws them, fcdiff/model.py:141-188).  For edge c = (n, m) = c_to_nm(c) and patient u, with q_F[c,k] and the
 * pair weights w_l of the edge's own regions (fit.py:382-406):
 *   qT [C][U]       = sum_k q_F[c,k] sum_l w_l P(T = 1 | F = k, pair state l, b~[c,u])
 *   qFt [C][U][3]   = sum_k q_F[c,k] sum_l w_l P(F~ = j | F = k, pair state l, b~[c,u])   (may be NULL: not formed)
 *   expected [U]    = sum_c qT[c][u];   rate [C] = sum_u qT[c][u] / U
 * P: planes p_0, p_1, p_2 of the scored patients (fcd_resp_cache, all C edges, [3][C][pitchU] with planeStride);
 * qF / fstate: q_F and its peak states; qR [N][U][2] (16-byte aligned); theta_host supplies eta, epsilon.  qT is
 * always written (pass scratch when the map is not wanted).  ws: fcd_connection_ws_bytes(C, U) bytes of device
 * scratch (no zero fill needed).  A patient's maps and expected count are bit-identical whichever other patients
 * are in the call (the row partition depends on C only, the partials are added in a fixed order), and the three
 * reductions do not depend on whether qFt is written. */
FCD_API int64_t fcd_connection_ws_bytes(int64_t C, int32_t U);
FCD_API int fcd_connection_posteriors(const double* P, int64_t planeStride, int64_t C, int32_t U, int64_t pitchU,
                              const double* qF, const uint8_t* fstate, const double* qR, int32_t N,
                              const fcd_theta* theta_host, double* qT, double* qFt, double* expected, double* rate,
                              double* ws, void* stream);

/* Per-subject control log-likelihoods (csrc/fcd_patients.cu): one control's share of E_lp_B_g_F
 * (fcdiff/fit.py:461-472) for each new column, with the Gaussian log density of fit.py:111-114:
 *   out [S] = sum_c sum_k qF[c,k] (-((X[c][s] - mu_k) / sigma_k)^2 / 2 - log sigma_k - log sqrt(2 pi))
 * X [C][pitchS] edge-major columns (C = N(N-1)/2, pitchS >= S >= 1); qF [C][3]; theta_host supplies mu, sigma.
 * ws: fcd_control_terms_ws_bytes(C, S) bytes of device scratch (no zero fill needed).  A subject's value is
 * bit-identical whichever other subjects, S or pitchS are in the call: the row partition depends on C only and
 * the partials are added in a fixed order.  missing = 1 sums over the observed entries: a NaN X[c][s] adds
 * nothing (fit.py:461-472 with the entry marginalised), so that a subject's l_C and its patient free energy
 * cover the same entries.  missing = 0 takes every entry as observed; any other value is rejected. */
FCD_API int64_t fcd_control_terms_ws_bytes(int64_t C, int32_t S);
FCD_API int fcd_control_terms(const double* X, int64_t C, int32_t S, int64_t pitchS, const double* qF,
                              const fcd_theta* theta_host, double* out, double* ws, int32_t missing, void* stream);

/* Westfall-Young step-down max-T counts of a permutation test (csrc/fcd_permutation.cu; no reference
 * counterpart: the reference has no permutation driver, fcdiff/fit.py:56-82).  T [R1][pitch] (pitch >= K):
 * row 0 the observed statistics, rows 1..R1-1 those of relabelled data.  One family is the column range
 * [k0, k1), 0 <= k0 < k1 <= K; order [k1 - k0] (int64) lists its columns k, k0 <= k < k1, ascending by
 * (T[0][k], k): the permutation sigma, formed on the host and not checked here.  Then
 *   count_unc [k1 - k0] (by column, k - k0) = #{r : T[r][k] >= T[0][k]}
 *   count_sd  [k1 - k0] (by position j)     = #{r : max_{i <= j} T[r][sigma(i)] >= T[0][sigma(j)]}
 * so p[k] = count_unc / R1 and p_fwer[sigma(j)] = max_{i >= j} count_sd[i] / R1 (the suffix maximum is left
 * to the caller).  Both outputs are int64 and written whole; T must be finite (not checked here).  The counts
 * are exact integers: they do not depend on the launch shape or the order of the atomics.  1 <= R1 <= 2^20,
 * 1 <= K <= 2^24; larger sizes are rejected before any launch.  ws: fcd_maxt_ws_bytes(R1, K) bytes of device
 * scratch (no zero fill needed; 0 for sizes out of range). */
FCD_API int64_t fcd_maxt_ws_bytes(int64_t R1, int64_t K);
FCD_API int fcd_maxt_counts(const double* T, int64_t R1, int64_t K, int64_t pitch, const int64_t* order, int64_t k0,
                            int64_t k1, int64_t* count_unc, int64_t* count_sd, double* ws, void* stream);

/* K3c -- per-state sufficient statistics of the correlations for the control
 * and the patient group (north_star subsystem 3; the reference ships only
 * disabled pieces of a mu / sigma update, fcdiff/fit.py:232-237, 542-597,
 * 709-733; doc/methods.rst:715-944).  out[0..8] controls: n_j = H sum_c qF[c,j],
 * sum qF[c,j] S1[c], sum qF[c,j] S2[c]; out[9..17] patients: sum R_j, sum R_j x,
 * sum R_j x^2 with R_j(c,u) the posterior weight that patient edge (c,u) is in
 * state j.  Pooled, they are the EM (lower-bound) update of mu_j, sigma_j. */
FCD_API int fcd_state_moments(const double* S1, const double* S2, int32_t H,
                      const double* bt, const double* P, int64_t planeStride,
                      int64_t C, int32_t U, int64_t pitchU,
                      const double* qF, const double* qR, int32_t N, const int32_t* nm,
                      const fcd_theta* theta_host, double* out18, double* ws, void* stream);

/* ------------------------------------------------------- materialised API   */
/* The reference caches (C,H,3), (C,U,3) and (C,U,3,3) arrays and its tests
 * assign them directly (test_fcdiff/test_fit.py:440-446, 483-489).  These
 * entry points run the same steps from such arrays (API parity; the fused
 * path above never materialises them). */

/* `_update_lps` (fcdiff/fit.py:104-122): lpB [C][H][3], pBt [C][U][3],
 * lM [C][U][3][3] (k major, l minor), scipy.stats.norm op order.
 * missing = 1: the same caches of a fit with missing entries (fit.py:104-122 with NaN marginalised): a NaN
 * b[c,h] gives lpB[c][h][:] = 0, a NaN bt[c,u] gives pBt[c][u][:] = 1 and lM[c][u][:][:] = 0 (M_kl = eps_l +
 * (1 - eps_l) = 1, fit.py:427-430).  missing = 0 takes every entry as observed; any other value is rejected. */
FCD_API int fcd_materialize_lps(const double* b, const double* bt, int64_t C, int32_t H, int32_t U,
                        const fcd_theta* theta_host,
                        double* lpB, double* pBt, double* lM, int32_t missing, void* stream);

/* `_eval_M` (fcdiff/fit.py:409-430): M[i] from p[i][3], i < n. */
FCD_API int fcd_eval_M(const double* p, int64_t n, double eta, double epsilon, int32_t k, int32_t l,
               double* M, void* stream);

/* `_update_lq_F` from arrays (fcdiff/fit.py:157-174). */
FCD_API int fcd_lqF_from_arrays(const double* lpB, const double* lM, int64_t C, int32_t H, int32_t U,
                        const double* qR, int32_t N, const double* log_gamma_host,
                        double* lqF, void* stream);

/* W for `_update_lq_R` from a materialised lM: W_l = sum_k qF[c,k] lM[c,u,k,l], stored as
 * WT[u][c] = { W_0 - W_2, W_2 - W_1 } ([U][C][2], the layout fcd_estep_qR reads). */
FCD_API int fcd_region_weights_from_lM(const double* lM, int64_t C, int32_t U, const double* qF,
                               double* WT, void* stream);

/* `_eval_E_lM` (fcdiff/fit.py:489-511) from arrays. */
FCD_API int fcd_ElM_from_arrays(const double* qF, const double* qR, const double* lM,
                        int64_t C, int32_t N, int32_t U, double* out1, double* ws, void* stream);

/* `_eval_dE_dh` / `_eval_dE_de` (fcdiff/fit.py:600-664) from arrays:
 * out[0] = dE/d eta, out[1] = dE/d epsilon. norm [C][U][3], mix [C][U][3][3]. */
FCD_API int fcd_dE_from_arrays(const double* qR, const double* qF, const double* norm, const double* mix,
                       int64_t C, int32_t N, int32_t U, double eta, double epsilon,
                       double* out2, double* ws, void* stream);

/* `_eval_dlM_dh` / `_eval_dlM_de` (fcdiff/fit.py:618-641, 667-697), elementwise:
 * out[i] = (eps * norm[i][k] - 0.5 * eps * (norm[i][j] + norm[i][j'])) / mix[i]. */
FCD_API int fcd_dlM(const double* norm, const double* mix, int64_t n, double eps, int32_t k,
            double* out, void* stream);

/* `_eval_q_R_w` (fcdiff/fit.py:382-406): out[u][0..2] for the region pair (n, m). */
FCD_API int fcd_pair_weights(const double* qR, int32_t N, int32_t U, int32_t n, int32_t m,
                     double* out, void* stream);

/* sum_i a[i] * x[(i / a_div) % x_mod_or_n]: the broadcast dot products of
 * `_eval_E_lp_F`, `_eval_E_lp_B_g_F`, `_eval_E_lp_R`, `_eval_E_lq_F`,
 * `_eval_E_lq_R` (fcdiff/fit.py:447-486, 514-539).  See fit.py (host) for the
 * index maps used. out1[0] = sum_i a[ia(i)] * x[ix(i)] with
 *   ia(i) = (i / a_outer) * a_inner + i % a_inner   (a_outer >= a_inner)
 *   ix(i) = i % x_len. */
FCD_API int fcd_dot_broadcast(const double* a, int64_t a_outer, int64_t a_inner,
                      const double* x, int64_t x_len, int64_t n,
                      double* out1, double* ws, void* stream);

/* ------------------------------------------------------- sampler (K5)       */
/* Ancestral sampler of fcdiff/model.py:52-236 with counter-based Philox4x32-10
 * (key = seed, counter = (variable id, c, u)); util edge order everywhere.
 * Outputs (any may be NULL to skip): r [N][U] u8, t [C][U] u8, f [C][3] u8,
 * ft [C][U][3] u8, b [C][H] f64, bt [C][U] f64 (clipped to [-1,1]).
 * Each stage can also be driven from caller-provided parents (sample_T(r),
 * sample_F_tilde(f,t), sample_B(f,H), sample_B_tilde(f_tilde)). */
FCD_API int fcd_sample_R(uint64_t seed, uint64_t offset, int32_t N, int32_t U, double pi,
                 uint8_t* r, void* stream);
FCD_API int fcd_sample_T(uint64_t seed, uint64_t offset, const uint8_t* r, int32_t N, int32_t U,
                 double eta, int64_t c0, int64_t C, uint8_t* t, void* stream);
FCD_API int fcd_sample_F(uint64_t seed, uint64_t offset, int64_t c0, int64_t C,
                 const double* gamma3_host, uint8_t* f, void* stream);
FCD_API int fcd_sample_F_tilde(uint64_t seed, uint64_t offset, const uint8_t* f, const uint8_t* t,
                       int64_t c0, int64_t C, int32_t U, double epsilon, uint8_t* ft, void* stream);
FCD_API int fcd_sample_B(uint64_t seed, uint64_t offset, const uint8_t* f, int64_t c0, int64_t C, int32_t H,
                 const double* mu3_host, const double* sigma3_host, double* b, void* stream);
FCD_API int fcd_sample_B_tilde(uint64_t seed, uint64_t offset, const uint8_t* ft, int64_t c0, int64_t C, int32_t U,
                       const double* mu3_host, const double* sigma3_host, double* bt, void* stream);

/* ------------------------------------------------------- correlations (K1)  */
/* Region time series -> correlations (no reference counterpart; SURVEY 8 a11).
 * ts [S][N][T] float32.  Per subject: rows are centred and scaled to unit
 * norm, R = Z Z^T on tcgen05 tensor cores with error-compensated split-TF32
 * (3 MMAs per product), and the lower triangle is written in util edge order to
 * out[c][s0 + s] (float64, row pitch `pitch`), Fisher-z transformed
 * (atanh) when `fisher` != 0, else clipped to [-1, 1].
 * zws: device scratch of fcd_corr_workspace_bytes(S, N, T) bytes. */
FCD_API int64_t fcd_corr_workspace_bytes(int32_t S, int32_t N, int32_t T);
FCD_API int fcd_corr_fisherz(const float* ts, int32_t S, int32_t N, int32_t T,
                     double* out, int64_t pitch, int32_t s0, int32_t fisher,
                     void* zws, void* stream);
/* After fcd_corr_fisherz on the same ts / out / pitch / s0: a (subject, region) row with a non-finite
 * sample or of zero variance (the test the standardisation applies) has no usable time series; NaN (not
 * observed, fit.missing = "marginalize") is written to all N - 1 edges of that region in column s0 + s.
 * Every other entry is left as it is. */
FCD_API int fcd_corr_mark_missing(const float* ts, int32_t S, int32_t N, int32_t T,
                     double* out, int64_t pitch, int32_t s0, void* stream);

/* Correlations from cleaned time series: censored frames, per-subject scan lengths, confound regression.
 * ts [S][N][T] float32 (T = the longest subject; shorter subjects padded), keep [S][T] uint8 (a frame t
 * enters subject s's correlations iff keep[s][t] != 0; NULL: every frame), confounds [S][T][K] float64
 * frame-major (NULL iff K == 0; 0 <= K <= 64).  Per subject, over its kept frames only, every region row
 * is centred, cleared of the centred confounds by projection on their orthonormal basis (two passes of
 * modified Gram-Schmidt in fp64; a confound whose residual norm is <= 1e-10 of its raw norm is dropped,
 * rank[s] = the confounds kept, when rank != NULL), scaled to unit norm, and the Gram stage and output of
 * fcd_corr_fisherz follow: columns [s0, s0 + S) of the (C, pitch) matrix out, every other column
 * untouched.  r is then the partial correlation of the two regions given the confounds and a constant.
 * Samples and confounds of frames that are not kept are never read into arithmetic.  A region row with a
 * non-finite kept sample, or whose residual sum of squares is at most 2^-40 of its centred sum of squares
 * (zero variance when K == 0), is unusable: r = 0 on its edges, or NaN on its N - 1 edges when
 * mark_missing != 0.  With keep all ones and K == 0 the output has the bits of fcd_corr_fisherz (and,
 * with mark_missing, of fcd_corr_mark_missing after it).  Every subject needs at least K + 2 kept frames
 * (not checked here).  zws: device scratch of fcd_corr_clean_workspace_bytes(S, N, T, K) bytes. */
FCD_API int64_t fcd_corr_clean_workspace_bytes(int32_t S, int32_t N, int32_t T, int32_t K);
FCD_API int fcd_corr_fisherz_clean(const float* ts, int32_t S, int32_t N, int32_t T, const uint8_t* keep,
                     const double* confounds, int32_t K, double* out, int64_t pitch, int32_t s0,
                     int32_t fisher, int32_t mark_missing, int32_t* rank, void* zws, void* stream);

/* Partial correlations from cleaned time series: r_nm = -P_nm / sqrt(P_nn P_mm), P = Sigma^-1, Sigma the
 * Ledoit-Wolf shrunk correlation matrix of a subject's usable regions.  Inputs as fcd_corr_fisherz_clean
 * (ts, keep, confounds, K <= 64), and the same rows: over the kept frames each region row is centred, cleared
 * of the confounds, and scaled to unit variance with the 1/n_s normalisation (n_s the subject's kept frames),
 * all in fp64 (X, n_s x N_s).  R = X^T X / n_s, mu = tr(R) / N_s, and, when shrinkage < 0, Ledoit-Wolf as
 * sklearn.covariance.ledoit_wolf(X, assume_centered=True) computes it: d2 = |R - mu I|_F^2 / N_s,
 * b2 = min(d2, (sum_t |x_t|^4 / n_s - |R|_F^2) / (n_s N_s)), delta = b2 / d2 (0 unless b2 > 0); a
 * shrinkage in [0, 1] is delta itself.  Sigma = (1 - delta) R + delta mu I, inverted in fp64 (blocked
 * symmetric sweep, one CTA per subject); r goes through the clip / atanh of fcd_corr_fisherz into columns
 * [s0, s0 + S) of the (C, pitch) matrix out, every other column untouched.  With confounds r is the partial
 * correlation given all other regions, the confounds and a constant (at delta = 0); n_s is not reduced by
 * the K + 1 fitted columns.  An unusable region (the rule of fcd_corr_fisherz_clean) is left out of its
 * subject's problem: the subject's other edges and delta are those of its usable regions alone, and the
 * region's edges are 0, or NaN when mark_missing != 0.  delta = 1 gives r = 0 on every edge.  A pivot of
 * the inverse <= 2^-40 (Sigma singular to working precision: shrinkage 0 with n_s <= N + K, or collinear
 * regions) sets status[s] = 1 and writes NaN to all of column s0 + s; otherwise status[s] = 0.  rank[s]:
 * the confounds kept (when rank != NULL); shrinkage_out[s]: delta (when != NULL).  Subjects are processed
 * in batches inside the call; no result depends on the batch.  Every subject needs at least K + 2 kept
 * frames (not checked here).  zws: device scratch of fcd_corr_partial_workspace_bytes(S, N, T, K) bytes. */
FCD_API int64_t fcd_corr_partial_workspace_bytes(int32_t S, int32_t N, int32_t T, int32_t K);
FCD_API int fcd_corr_partial(const float* ts, int32_t S, int32_t N, int32_t T, const uint8_t* keep,
                     const double* confounds, int32_t K, double shrinkage, double* out, int64_t pitch,
                     int32_t s0, int32_t fisher, int32_t mark_missing, int32_t* rank, double* shrinkage_out,
                     int32_t* status, void* zws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FCDIFF_B200_H */
