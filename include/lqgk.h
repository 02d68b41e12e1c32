/* lqgk.h -- C ABI of liblqgk.so: B200 (sm_100a) kernels for the LQG inverse-optimal-control likelihood.
 *
 * Drop-in boundary for ONE hot path of RothkopfLab/lqg.  The reference has no FFI of its own (pure
 * Python/JAX); these entry points are what an XLA-FFI custom call (or ctypes / torch harness) binds in
 * place of the reference functions cited per entry.  All paths below are relative to the reference repo.
 *
 * Conventions
 *  - All buffers are caller-owned DEVICE memory.  No device allocation, no host synchronisation and no use of the
 *    default stream inside; kernels are enqueued on `stream` (a cudaStream_t passed as void*).
 *  - Return 0 (LQGK_OK) or a negative LQGK_E_* code; never throws.  Re-entrant: the only state is per host thread (the
 *    tuning knobs below and a pool of internal streams / events used to run independent kernels of one call side by side,
 *    always forked from and joined to `stream`).  lqgk_init() creates that pool up front; without it the first call of a
 *    thread creates it lazily, which is not possible while `stream` is being captured into a CUDA graph
 *    (-> LQGK_E_NOT_INITIALISED).  After lqgk_init() every entry point is capturable and replayable.
 *  - Matrices are row-major.  Every matrix has a leading parameter-sample axis and a time axis described by
 *    element strides: sample_stride 0 = shared by all samples, time_stride 0 = time-invariant
 *    (the reference stacks T copies: lqg/utils.py:6-35).
 *  - `_f32` / `_f64` select the I/O element type of matrices, gains, log-likelihoods and gradients.  The
 *    per-sample recursions always run in FP64 and the per-trial recursions in FP32 (DESIGN.md, precision).
 *  - Observations are FP32, time-major x_tm[T+1][N][d] (use lqgk_pack_obs_* once per dataset).
 *  - Dimension tuple (x, b, u, y, d) = (dynamics state, belief state, control, observation, observed-by-
 *    experimenter dims) must be one of the compiled instantiations (lqgk_dims_supported), else
 *    LQGK_E_UNSUPPORTED.
 */
#ifndef LQGK_H_
#define LQGK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LQGK_OK 0
#define LQGK_E_INVALID (-1)      /* null pointer / non-positive dimension / misaligned buffer          */
#define LQGK_E_UNSUPPORTED (-2)  /* dimension tuple not instantiated, or time-varying spec in the VJP  */
#define LQGK_E_WORKSPACE (-3)    /* workspace too small for even one 32-sample chunk                   */
#define LQGK_E_CUDA (-4)         /* a CUDA runtime call failed (see cudaGetLastError)                  */
#define LQGK_E_NOT_INITIALISED (-5) /* call under CUDA-graph capture before lqgk_init() on this thread */

typedef struct {
  int32_t S; /* parameter samples (systems) in this call                              */
  int32_t N; /* trials per system                                                     */
  int32_t T; /* time steps; observations have T+1 rows (lqg/system.py:233, SURVEY H7) */
  int32_t x, b, u, y, d;
  int64_t x_sample_stride; /* floats between the observation sets of consecutive samples in x_tm;
                              0 = all samples share one data set x_tm[T+1][N][d] (parameter sweeps);
                              (T+1)*N*d = every sample has its own data x_tm[S][T+1][N][d] (e.g. one sample per
                              experimental condition, lqg/infer/models.py:38-61) */
} LqgkDims;

typedef struct {
  const void* ptr;       /* NULL = absent (zeros / default)          */
  int64_t sample_stride; /* elements between samples, 0 = shared     */
  int64_t time_stride;   /* elements between time steps, 0 = const   */
} LqgkMat;

/* One LQG specification, mirrors lqg/spec.py:5-19 (LQGSpec).  For the dynamics side only A,B,F,V,W are read. */
typedef struct {
  LqgkMat A, B, F, V, W, Q, R;
  LqgkMat Qf;          /* absent -> Q at the last time step (lqg/utils.py:30)          */
  LqgkMat q, r, P, qf; /* affine terms, gains API only (zeros in every reference model) */
} LqgkSpec;

typedef struct {
  void* ptr;             /* NULL = gradient not wanted */
  int64_t sample_stride; /* elements between samples   */
} LqgkMatGrad;

/* Cotangents of a time-invariant spec (sum over time steps, SURVEY H6). */
typedef struct {
  LqgkMatGrad A, B, F, V, W, Q, R, Qf;
} LqgkSpecGrad;

/* ---- gains -------------------------------------------------------------------------------------------
 * lqgk_lqr_backward_*: replaces lqg/control/lqr.py:16-42  lqr.backward(spec, eps) -> Gains(L, l, H).
 *   Outputs L[S][T][u][b], l[S][T][u] (may be NULL), H[S][T][u][u] (may be NULL; the shifted Ht).
 * lqgk_kf_forward_*:   replaces lqg/belief/kf.py:6-21     kf.forward(spec, Sigma0) -> K.
 *   sigma0: [b][b] per sample (time_stride ignored); absent -> V[0] V[0]^T (lqg/system.py:158-161).
 *   Output K[S][T][b][y].
 * `d` and `N` in dims are ignored by the gains entry points and their adjoint (set d to any supported value, e.g. min(x, 2)). */
int lqgk_lqr_backward_f32(const LqgkDims* dims, const LqgkSpec* actor, double eps, float* L_out, float* l_out,
                          float* H_out, void* workspace, size_t workspace_bytes, void* stream);
int lqgk_lqr_backward_f64(const LqgkDims* dims, const LqgkSpec* actor, double eps, double* L_out, double* l_out,
                          double* H_out, void* workspace, size_t workspace_bytes, void* stream);
int lqgk_kf_forward_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, float* K_out,
                        void* workspace, size_t workspace_bytes, void* stream);
int lqgk_kf_forward_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double* K_out,
                        void* workspace, size_t workspace_bytes, void* stream);
/* lqgk_gains_vjp_*: reverse-mode adjoint of the two sweeps above (what jax.vjp of lqr.backward(spec, eps).L and of
 *   kf.forward(spec, Sigma0) computes in the reference).  L_bar[S][T][u][b] and K_bar[S][T][b][y] are the cotangents of L and
 *   K in the layouts of those outputs; either may be NULL (zero), not both.  eps and sigma0 as above.  The call recomputes
 *   both sweeps and keeps S_t / P_t in the workspace (no state from an earlier call), then runs the Riccati and Kalman
 *   adjoints; the eigen-shift of lqr.py:27-28 is held constant, as in lqgk_loglik_vjp_*.
 *   actor_grad receives the gradients of A, B, F, V, W, Q, R, Qf (any field may be NULL), sigma0_grad that of Sigma0 (may be
 *   NULL).  Defaulted inputs send their gradient to their source: Qf absent -> Q; sigma0 absent -> actor V.
 *   A, B, F, V, W, Q, R are required.  The affine terms q, r, qf are not read (L and K do not depend on them); a cross cost P
 *   and time-varying specs -> LQGK_E_UNSUPPORTED.  Workspace: lqgk_workspace_bytes(dims, LQGK_MODE_GAINS_VJP, max_chunk).
 *   Runs on `stream` alone (never on the internal streams), so it can be captured into a CUDA graph.                      */
int lqgk_gains_vjp_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double eps, const float* L_bar,
                       const float* K_bar, const LqgkSpecGrad* actor_grad, const LqgkMatGrad* sigma0_grad, void* workspace,
                       size_t workspace_bytes, void* stream);
int lqgk_gains_vjp_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkMat* sigma0, double eps, const double* L_bar,
                       const double* K_bar, const LqgkSpecGrad* actor_grad, const LqgkMatGrad* sigma0_grad, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---- likelihood ---------------------------------------------------------------------------------------
 * lqgk_loglik_fwd_*: replaces lqg/system.py:142-248  System.log_likelihood(x) (= conditional_moments +
 *   numpyro MultivariateNormal(...).to_event(1).log_prob).  Output ll[S][N].
 * lqgk_loglik_vjp_*: forward + reverse-mode adjoint in one call (what jax.value_and_grad of the above
 *   computes in the reference, lqg/infer/models.py:34,61,130).  ll_bar[S][N] are the cotangents of ll
 *   (NULL = all ones).  Time-invariant specs only.  Gradients of absent/defaulted inputs flow to their
 *   source (Qf absent -> Q; sigma0 absent -> actor V).                                                   */
int lqgk_loglik_fwd_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics,
                        const LqgkMat* sigma0, const float* x_tm, float* ll_out, void* workspace,
                        size_t workspace_bytes, void* stream);
int lqgk_loglik_fwd_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics,
                        const LqgkMat* sigma0, const float* x_tm, double* ll_out, void* workspace,
                        size_t workspace_bytes, void* stream);
int lqgk_loglik_vjp_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics,
                        const LqgkMat* sigma0, const float* x_tm, const float* ll_bar, float* ll_out,
                        const LqgkSpecGrad* actor_grad, const LqgkSpecGrad* dynamics_grad,
                        const LqgkMatGrad* sigma0_grad, void* workspace, size_t workspace_bytes, void* stream);
int lqgk_loglik_vjp_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics,
                        const LqgkMat* sigma0, const float* x_tm, const double* ll_bar, double* ll_out,
                        const LqgkSpecGrad* actor_grad, const LqgkSpecGrad* dynamics_grad,
                        const LqgkMatGrad* sigma0_grad, void* workspace, size_t workspace_bytes, void* stream);

/* ---- moments and simulation (the callers either side of the likelihood) -------------------------------------------------
 * lqgk_moments_*: replaces lqg/system.py:142-235 System.conditional_moments vmapped over trials, as used by
 *   belief_tracking_distribution (:250-257): predictive moments of the joint state (x, xhat)_{t+1} given x_{0..t}.
 *   Outputs mu[S][N][T][n] and Sigma[S][T][n][n] with n = x + b (either may be NULL).  Small systems (n <= 12) only.
 * lqgk_simulate_*: replaces lqg/system.py:62-140 System.simulate for S parameter samples x N trials, given the gains
 *   L[S][T][u][b], l[S][T][u] (NULL = 0) and K[S][T][b][y] (lqgk_lqr_backward_* / lqgk_kf_forward_*).  x0[x], xhat0[b]: initial
 *   state / belief (NULL = 0).  Noise: Philox4x32-10 counter stream keyed by (seed, trial) -- the reference's JAX threefry
 *   samples cannot be reproduced, the distribution is the same.  Outputs x[S][N][T+1][x] and optionally
 *   xhat[S][N][T+1][b], y[S][N][T][y], u[S][N][T][u].  Any dimension tuple with x, b, u, y <= 40.                        */
int lqgk_moments_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                     const float* x_tm, float* mu_out, float* Sigma_out, void* workspace, size_t workspace_bytes, void* stream);
int lqgk_moments_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkMat* sigma0,
                     const float* x_tm, double* mu_out, double* Sigma_out, void* workspace, size_t workspace_bytes, void* stream);
int lqgk_simulate_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const float* L, const float* l,
                      const float* K, const float* x0, const float* xhat0, uint64_t seed, float* x_out, float* xhat_out,
                      float* y_out, float* u_out, void* stream);
int lqgk_simulate_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const double* L, const double* l,
                      const double* K, const double* x0, const double* xhat0, uint64_t seed, double* x_out, double* xhat_out,
                      double* y_out, double* u_out, void* stream);

/* ---- signal-dependent noise (extension; NOT in the reference, see DESIGN.md and oracle/sdn_np.py) -------------
 * lqgk_sdn_gains_f64: Todorov (2005) alternating iterations for the control gains L and estimator gains K of
 *     x' = A x + B u + xi + sum_i eps_i C_i u,   y = H x + om + sum_i eta_i D_i x,
 *     xhat' = A xhat + B u + K (y - H xhat),     u = -L xhat,     cost = sum x'Qx + u'Ru + x_T' Qf x_T
 *   in ONE kernel (`sweeps` backward/forward sweeps starting from K = 0, then a final backward sweep).  With nc = nd = 0 a
 *   single sweep reproduces lqr.backward (lqg/control/lqr.py:16-42; L has the opposite sign: u = -L xhat) and the
 *   predictor-form Kalman gains.  All matrices FP64, time-invariant, row-major with a leading sample axis
 *   (sample_stride 0 = shared; time_stride ignored): A[b][b], B[b][u], H[y][b], C[nc][b][u], D[nd][y][b], Q[b][b],
 *   R[u][u], Qf[b][b] (absent -> Q), Om_xi[b][b], Om_omega[y][y] (noise covariances), Sigma1[b][b], xhat1[b].
 *   Outputs L[S][T][u][b], K[S][T][b][y], cost[S] (expected total cost; may be NULL).  (b, u, y) must be the belief / control
 *   / observation dims of a compiled small-system tuple.                                                                  */
typedef struct {
  int32_t S, T, b, u, y, nc, nd, sweeps;
} LqgkSdnDims;
typedef struct {
  LqgkMat A, B, H, C, D, Q, R, Qf, Om_xi, Om_omega, Sigma1, xhat1;
} LqgkSdnSpec;
int lqgk_sdn_gains_f64(const LqgkSdnDims* dims, const LqgkSdnSpec* spec, double* L_out, double* K_out, double* cost_out,
                       void* stream);
/* lqgk_sdn_gains_filter_f64: the same alternating iterations in the REFERENCE's conventions (filter form):
 *     u = L xhat,   xp = A xhat + B u,   xhat' = xp + K (y' - H xp),   y' = H x' + om + sum_i eta_i D_i x'   (y' observes x_{t+1}),
 *   i.e. lqg/system.py:110-124 with the multiplicative terms; Sigma1 / xhat1 are the prior covariance / mean of x_0.  With
 *   nc = nd = 0 ONE sweep reproduces lqr.backward (lqg/control/lqr.py:16-42; same sign) and kf.forward (lqg/belief/kf.py:6-21)
 *   exactly; the gains plug into lqgk_sdn_loglik_* / lqgk_simulate_*.  Derivation and validation: oracle/sdn_np.py
 *   (filter_backward_pass / filter_forward_pass: Monte Carlo cost, exact policy evaluation, coordinate-wise optimality).   */
int lqgk_sdn_gains_filter_f64(const LqgkSdnDims* dims, const LqgkSdnSpec* spec, double* L_out, double* K_out, double* cost_out,
                              void* stream);

/* lqgk_sdn_loglik_*: log-likelihood under signal-dependent noise -- the reference's experimenter-side filter
 *   (lqg/system.py:142-248, same filter-form conventions as lqg/system.py:110-124) extended by multiplicative noise
 *     x_{t+1} = A x_t + B u_t + V eps + sum_i eps'_i C_i u_t ,    y_t = F x_{t+1} + W eta + sum_j eta'_j D_j x_{t+1}
 *   with moment-matched Gaussian predictive distributions (oracle/sdn_np.py: sdn_log_likelihood).  EXTENSION: the reference
 *   has no such code, parity is pinned by Monte Carlo and by the exact reduction to lqgk_loglik_fwd_* when nc = nd = 0.
 *   The gains L[S][T][u][b], K[S][T][b][y] are inputs (lqgk_lqr_backward_* / lqgk_kf_forward_* of the actor's model, or any
 *   other solver).  noise->C: [nc][x][u], noise->D: [nd][y][x] per sample (sample_stride 0 = shared), nc, nd <= 4.  The
 *   covariance recursion is per (sample x trial) here -- one FP64 system per thread.  Time-invariant specs, joint dim <= 12.
 *   Output ll[S][N].                                                                                                      */
typedef struct {
  LqgkMat C, D;
  int32_t nc, nd;
} LqgkSdnNoise;
int lqgk_sdn_loglik_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise,
                        const float* L, const float* K, const float* x_tm, float* ll_out, void* stream);
int lqgk_sdn_loglik_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise,
                        const double* L, const double* K, const float* x_tm, double* ll_out, void* stream);
/* lqgk_sdn_simulate_*: lqgk_simulate_* for the generative model of lqgk_sdn_loglik_* (lqg/system.py:62-140 plus the multiplicative
 *   terms; oracle/sdn_np.py: sdn_simulate); noise == NULL or nc = nd = 0 draws exactly the trajectories of lqgk_simulate_*.      */
int lqgk_sdn_simulate_f32(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise,
                          const float* L, const float* l, const float* K, const float* x0, const float* xhat0, uint64_t seed,
                          float* x_out, float* xhat_out, float* y_out, float* u_out, void* stream);
int lqgk_sdn_simulate_f64(const LqgkDims* dims, const LqgkSpec* actor, const LqgkSpec* dynamics, const LqgkSdnNoise* noise,
                          const double* L, const double* l, const double* K, const double* x0, const double* xhat0, uint64_t seed,
                          double* x_out, double* xhat_out, double* y_out, double* u_out, void* stream);

/* ---- helpers ------------------------------------------------------------------------------------------ */
/* x[N][T+1][d] (f32 or f64, trial-major as in the reference) -> x_tm[T+1][N][d] float. */
int lqgk_pack_obs_f32(int32_t N, int32_t T1, int32_t d, const float* x, float* x_tm, void* stream);
int lqgk_pack_obs_f64(int32_t N, int32_t T1, int32_t d, const double* x, float* x_tm, void* stream);

#define LQGK_MODE_GAINS 0
#define LQGK_MODE_FWD 1
#define LQGK_MODE_VJP 2
#define LQGK_MODE_MOMENTS 3
#define LQGK_MODE_GAINS_VJP 4
/* Bytes of workspace that let `mode` process min(S, max_chunk) samples per internal chunk (max_chunk <= 0:
 * all S at once).  Any size >= lqgk_workspace_bytes(dims, mode, 32) is accepted; larger = fewer chunks.   */
size_t lqgk_workspace_bytes(const LqgkDims* dims, int mode, int32_t max_chunk);
int lqgk_dims_supported(const LqgkDims* dims);
const char* lqgk_strerror(int code);
const char* lqgk_version(void);
/* Text of the CUDA runtime's pending error (cudaPeekAtLastError) -- what went wrong behind an LQGK_E_CUDA return. */
const char* lqgk_last_cuda_error(void);
/* Creates the calling thread's internal streams / events for the current device (enough for `max_sample_slices` concurrent
 * sample slices, see lqgk_set_streams; 1 is the default configuration) and caches the device's SM count.  Optional unless
 * entry points are to be captured into CUDA graphs. */
int lqgk_init(int max_sample_slices);
/* Number of internal concurrent sample slices (streams) used by the likelihood entry points of the calling thread
 * (default 1 = everything on the caller's stream; 4 gives ~3 % at the benchmark size, see DESIGN.md).  Work is always forked from / joined to the caller's stream. */
int lqgk_set_streams(int n);
/* Kernel overlap inside one call: 0 keeps every chunk on one stream (no internal auxiliary streams); any other value
 * (1..7, default 6) lets the fused forward+adjoint call run the pipelined launch sequence of lqgk_set_pipeline over internal
 * auxiliary streams. */
int lqgk_set_kernel_overlap(int mask);
/* Pipelined launch sequence of the fused forward+adjoint call: chunks of at most `max_samples` parameter samples (default:
 * no limit; 0 = never) cut every sweep over time into `segments` segments (default 6) and run the sweeps of one direction as a
 * software pipeline over the internal streams (kf_fwd -> cov_fwd -> trial_fwd, then trial_rev -> cov_seq_rev -> contraction ->
 * kf_rev): at small sample counts every sweep is latency-bound and the chain of nine sweeps, not the arithmetic, sets the time of
 * one evaluation (a NUTS leapfrog).  Otherwise the same sequence runs as one segment on the chunk's stream, as do forward-only
 * calls and systems with joint dim > 12.  Results do not depend on the setting beyond FP64 summation order. */
int lqgk_set_pipeline(int max_samples, int segments);
/* Tuning knob: target number of (32-sample group x time-range) warps of the time-parallel contraction kernels. */
int lqgk_set_contrib_warps(int n);
/* Tuning knob: likelihood calls with at most n parameter samples run the covariance kernels one WARP per sample (shared-memory
 * matrices, lower per-step latency when the GPU is not full), larger calls one THREAD per sample (higher throughput).
 * Default 512 (measured crossover 512..1,024); 0 = always thread per sample.  Systems with joint dim > 12 always use the warp-per-sample kernels. */
int lqgk_set_warp_cov_max_samples(int n);
/* Per-kernel timing for bench.py: when enabled, every kernel launch of the calling thread's entry-point calls is
 * bracketed by CUDA events on the launching stream.  lqgk_profile_read() synchronises on those events, sums the
 * elapsed milliseconds (and launch counts) per kernel kind, resets the log and returns the number of kinds:
 * 0 pack, 1 lqr_fwd, 2 kf_fwd, 3 cov_fwd, 4 trial_fwd, 5 misc, 6 trial_rev, 7 cov_rev, 8 kf_rev, 9 lqr_rev, 10 unpack,
 * 11 cov_contrib, 12 reduce. */
int lqgk_profile_enable(int on);
int lqgk_profile_read(float* ms_by_kind, int32_t* launches_by_kind, int nkinds);
/* Start / end (ms, relative to the first recorded launch) and kind of every recorded launch; returns the count.
 * Call before lqgk_profile_read (which resets the log). */
int lqgk_profile_timeline(float* start_ms, float* end_ms, int32_t* kind, int max_entries);
/* Launches an FMA-saturating micro-kernel (fp64 != 0: DFMA, else FFMA) on `stream`; *flop_out = flops it executes.
 * Time it with CUDA events to obtain the measured CUDA-core peak used as the roofline denominator. `sink`: >= 8 bytes. */
int lqgk_peak_fma(int fp64, int iters, void* sink, void* stream, double* flop_out);
/* Number of kernel launches issued by the calling thread's last entry-point call (for bench accounting). */
int lqgk_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* LQGK_H_ */
