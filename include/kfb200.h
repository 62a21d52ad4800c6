/*
 * kfb200.h - C ABI of libkfb200.so: B200 (sm_100a) batched Kalman-filter
 * log-likelihood and reverse-mode gradient.
 *
 * This is the drop-in boundary for the ONE hot path of jessegrabowski/pymc_statespace:
 * what `BaseFilter.build_graph` (reference pymc_statespace/filters/kalman_filter.py:126-193)
 * computes with `pytensor.scan`, and what PyTensor autodiff of that scan computes for
 * `pm.Potential("log_likelihood")` (reference pymc_statespace/core/statespace.py:174).
 * The reference is pure Python (no FFI of its own); the binding a maintainer adds is the
 * ctypes stub shown in INTEGRATION.md.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer to float64 (or int32 where stated) unless the
 *    parameter name starts with `h_`; the caller owns every buffer; the library never
 *    allocates caller-visible memory and keeps no global state;
 *  - all calls are asynchronous on `stream` (a cudaStream_t passed as void*);
 *  - a "unit" is one independent recursion: unit u = draw * n_series + series;
 *    parameter matrices are indexed by draw (u / n_series), observations by series
 *    (u % n_series);
 *  - matrices are dense row-major with the reference's shapes: a0[m] P0[m,m] T[m,m] Z[p,m]
 *    R[m,r] H[p,p] Q[r,r] c[m] d[p], y[n,p] (NaN = missing observation);
 *  - `*_bs` is the stride in ELEMENTS between consecutive draws (series for y); 0 means the
 *    array is shared by all draws.  `*_ts` is the stride between consecutive time steps for
 *    a time-varying matrix (reference filters/utilities.py:1-20: 3-D, time-first); 0 = static;
 *  - errors: integer status (0 = OK), never C++ exceptions; numerical failures are reported
 *    per unit in `info[u]` (0 ok; t+1 > 0: innovation covariance F_t not positive definite at
 *    0-based step t; -(t+1) < 0: partially-missing y_t in a filter that only supports
 *    all-or-nothing rows - reference raises LinAlgError there, SURVEY.md A.2-Q2; KFB_INFO_DARE_FAILED:
 *    the steady-state covariance (DARE) of this draw did not converge / F_ss not positive definite)
 *    and the unit's loglik is NaN.
 */
#ifndef KFB200_H
#define KFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KFB_VERSION 100

typedef int32_t kfb_status;
enum {
  KFB_OK = 0,
  KFB_ERR_INVALID_ARG = 1,   /* null pointer / non-positive size / bad enum          */
  KFB_ERR_UNSUPPORTED = 2,   /* valid request this build has no kernel for           */
  KFB_ERR_WORKSPACE = 3,     /* workspace too small / missing                        */
  KFB_ERR_CUDA = 4           /* a CUDA runtime call failed (see kfb_last_cuda_error) */
};

/* FILTER_FACTORY keys, reference pymc_statespace/core/statespace.py:25-31 */
enum {
  KFB_STANDARD = 0,     /* StandardFilter         kalman_filter.py:255-284 */
  KFB_UNIVARIATE = 1,   /* UnivariateFilter       kalman_filter.py:444-505 */
  KFB_STEADY_STATE = 2, /* SteadyStateFilter      kalman_filter.py:354-441 */
  KFB_SINGLE = 3,       /* SingleTimeseriesFilter kalman_filter.py:321-351 */
  KFB_CHOLESKY = 4      /* CholeskyFilter         kalman_filter.py:287-318 */
};

/* info[] codes beyond "t + 1" / "-(t + 1)" (no series is this long) */
#define KFB_INFO_DARE_FAILED 0x40000001    /* steady_state: Riccati / Newton-Hewer iteration failed for this draw      */
#define KFB_INFO_BAD_STRUCTURE 0x40000003   /* a KFB_FLAG_Z_UNIT0 / _H_ZERO / _T_COMPANION promise does not hold for this unit */
#define KFB_INFO_NOT_STATIONARY 0x40000002 /* set by the host layer (KalmanLogp): stationary P0 requested but the      */
                                           /* Lyapunov doubling did not converge (spectral radius of T >= 1)            */
#define KFB_INFO_NOT_PSD 0x40000004        /* kfb_simulation_smoother: P0, Q or H is not positive semi-definite         */
                                           /* (kfb_forecast_paths: the start covariance, Q or H; kfb_impulse_response: Q) */

/* flags */
#define KFB_FLAG_CORRECTED 1u  /* strict_reference=False: fix SURVEY.md A.2 quirks Q1,Q4,Q5,Q6 */
#define KFB_FLAG_FORCE_COOP 2u /* testing: use the cooperative (shared-memory) kernels even   */
                               /* when a thread-per-unit instantiation exists                   */
#define KFB_FLAG_GENERIC_ADJOINT 4u /* testing: run the generic thread-per-unit kernels where the        */
                                    /* specialised k_endog = 1 forward / adjoint kernels would be used   */

/* Structure promises (k_endog = 1 only; verified per unit by the forward kernel, violations -> KFB_INFO_BAD_STRUCTURE):
 * the products with the known ones and zeros are not issued - same values, ~17 % fewer instructions per step.  Every
 * ARMA / local-level model of the reference has Z = [1, 0, ..] (models/SARIMAX.py:29-50, models/local_level.py:14-27) and
 * BayesianARMA has obs_cov = 0. */
#define KFB_FLAG_Z_UNIT0 8u   /* Z = [1, 0, .., 0] for every draw                                   */
#define KFB_FLAG_H_ZERO 16u   /* H = 0 for every draw (only honoured together with KFB_FLAG_Z_UNIT0) */
#define KFB_FLAG_NO_MISSING 64u  /* no observation is NaN.  Together with the three flags above the tape of the k_endog = 1
                                    kernels holds only what varies (a_t and the leading block of P_t: 24 instead of 40
                                    bytes per step at k_states 2); a missing observation is then reported per unit        */
#define KFB_FLAG_T_COMPANION 32u /* T = [t | e_0 .. e_{m-2}] for every draw: only the first column carries parameters
                                    (BayesianARMA / SARIMAX, reference models/SARIMAX.py:59-98).  Only honoured together
                                    with the two flags above; the columns >= 1 of the T gradient are then returned as 0 */

/* Time-parallel evaluation (k_endog = 1, k_states <= 4, standard / single / cholesky): one CTA per unit runs the filter
 * and its adjoint as blocked scans over time (Saerkkae & Garcia-Fernandez filtering elements forward, affine and
 * congruence scans backward), instead of one thread walking all n steps.  For few units and long series (one NUTS draw
 * per call); with many units the sequential kernels are faster.  Same outputs, gradients and info codes as without the
 * flag, to rounding (the sums run in another fixed order; two runs give identical bits).  Any other geometry with the
 * flag set returns KFB_ERR_UNSUPPORTED (k_endog > 1, k_states > 4, univariate, steady_state).  The structure promises
 * above are not used on this path (nothing is skipped or verified).  A unit whose parallel element is undefined at some
 * step (Z C Z^T + H = 0 there: an observation without noise given the previous state) is run by one thread of its CTA
 * with the sequential recursion; no info code marks it.  The forward pass always uses the tape part of the workspace. */
#define KFB_FLAG_TIME_PARALLEL 128u

/* Read by kfb_simulation_smoother only: a partly observed row y_t (some entries NaN, not all) is filtered on its
 * observed entries instead of failing the unit with -(t+1); predicted_covs must then come from kfb_masked_filter.
 * Without a partly observed row the result is the same, bit for bit, as without the flag. */
#define KFB_FLAG_PARTIAL_ROWS 256u

typedef struct kfb_desc {
  int32_t filter_kind;
  uint32_t flags;
  int64_t n_draws;  /* parameter draws                          */
  int64_t n_series; /* observation series (>=1); units = n_draws * n_series */
  int32_t n, m, p, r; /* time steps, k_states, k_endog, k_posdef */
  /* batch strides (elements); 0 = shared */
  int64_t y_bs, a0_bs, P0_bs, T_bs, Z_bs, R_bs, H_bs, Q_bs, c_bs, d_bs;
  /* time strides (elements); 0 = static.  steady_state and univariate take static matrices
     only (reference kalman_filter.py:421,482 fixed-signature steps)                        */
  int64_t T_ts, Z_ts, R_ts, H_ts, Q_ts, c_ts, d_ts;
} kfb_desc;

typedef struct kfb_inputs {
  const double *y, *a0, *P0, *T, *Z, *R, *H, *Q;
  const double *c, *d; /* may be NULL = zeros (initialize_intercepts, kalman_filter.py:37-51) */
} kfb_inputs;

/* Outputs of build_graph (kalman_filter.py:184-191), batched over units (leading dim U).
 * Any pointer may be NULL = not wanted.  loglik[U]; ll_obs[U,n]; filtered_states[U,n,m];
 * predicted_states[U,n+1,m] (a0 first); filtered_covs[U,n,m,m]; predicted_covs[U,n+1,m,m]
 * (P0 first); info[U] int32. */
typedef struct kfb_outputs {
  double *loglik, *ll_obs, *filtered_states, *predicted_states, *filtered_covs, *predicted_covs;
  int32_t *info;
} kfb_outputs;

/* Cotangents: the differentiated scalar per unit is
 *   g_loglik[u] * loglik[u] + sum_t g_ll_obs[u,t] * ll_obs[u,t];  NULL g_loglik = 1, NULL g_ll_obs = 0. */
typedef struct kfb_cotangents {
  const double *g_loglik, *g_ll_obs;
} kfb_cotangents;

/* Gradients, one block per UNIT (never reduced over shared inputs): a0[U,m] P0[U,m,m]
 * T[U,(n,)m,m] Z[U,(n,)p,m] R[U,(n,)m,r] H[U,(n,)p,p] Q[U,(n,)r,r] c[U,(n,)m] d[U,(n,)p] - the (n,)
 * dimension is present iff that input is time-varying.  NULL = not wanted. */
typedef struct kfb_grads {
  double *a0, *P0, *T, *Z, *R, *H, *Q, *c, *d;
} kfb_grads;

int32_t kfb_version(void);
const char *kfb_status_string(kfb_status s);
const char *kfb_last_cuda_error(void);

/* Bytes of device workspace kfb_forward / kfb_backward need.  `save_for_backward` != 0 adds
 * the forward-pass tape of predicted moments (a_t, P_t) the adjoint kernel reads back. */
kfb_status kfb_workspace_bytes(const kfb_desc *desc, int32_t save_for_backward, size_t *bytes);

/* Forward recursion: replaces the scan at kalman_filter.py:152-159 (and :388-395, :491-496). */
kfb_status kfb_forward(const kfb_desc *desc, const kfb_inputs *in, const kfb_outputs *out,
                       void *workspace, size_t workspace_bytes, int32_t save_for_backward,
                       void *stream);

/* Reverse-mode adjoint of kfb_forward wrt (a0,P0,T,Z,R,H,Q,c,d): replaces PyTensor's Scan.L_op
 * of the same graph (SURVEY.md section 8(a) row a10).  `workspace` must be the buffer a preceding
 * kfb_forward(..., save_for_backward=1) on the same desc/inputs filled. */
kfb_status kfb_backward(const kfb_desc *desc, const kfb_inputs *in, const kfb_cotangents *cot,
                        const kfb_grads *grads, void *workspace, size_t workspace_bytes,
                        void *stream);

/* RTS smoother (next row f2, not on the logp/grad path): reference KalmanSmoother.build_graph,
 * pymc_statespace/filters/kalman_smoother.py:56-104, static T, R, Q.  filtered_states[U,n,m], filtered_covs[U,n,m,m]
 * (outputs of kfb_forward) -> smoothed_states[U,n,m], smoothed_covs[U,n,m,m].  workspace: n_draws*m*m doubles
 * (m*m if R and Q are shared). */
kfb_status kfb_smoother(int64_t n_draws, int64_t n_series, int32_t n, int32_t m, int32_t r, const double *T,
                        int64_t T_bs, const double *R, int64_t R_bs, const double *Q, int64_t Q_bs,
                        const double *filtered_states, const double *filtered_covs, double *smoothed_states,
                        double *smoothed_covs, void *workspace, size_t workspace_bytes, void *stream);

/* kfb_smoother with flags (0: exactly kfb_smoother).  KFB_FLAG_TIME_PARALLEL: one CTA per unit and a blocked scan over
 * time of the smoothing elements (Saerkkae & Garcia-Fernandez 2021), then a walk of every chunk with the literal RTS
 * step; a unit whose scan disagrees with that walk (or meets a NaN) is re-run by the sequential recursion.  Faster for
 * few units over long series; results agree with the sequential smoother to rounding.  k_states 1..4, else
 * KFB_ERR_UNSUPPORTED; any other flag bit: KFB_ERR_INVALID_ARG.  Same workspace rule as kfb_smoother (no tape). */
kfb_status kfb_smoother_ex(int64_t n_draws, int64_t n_series, int32_t n, int32_t m, int32_t r, const double *T,
                           int64_t T_bs, const double *R, int64_t R_bs, const double *Q, int64_t Q_bs,
                           const double *filtered_states, const double *filtered_covs, double *smoothed_states,
                           double *smoothed_covs, void *workspace, size_t workspace_bytes, uint32_t flags, void *stream);

/* Stationary initial covariance: X = A X A^T + C with C = R Q R^T
 * (reference models/SARIMAX.py:100-107, models/VARMAX.py:143-150:
 *  solve_discrete_lyapunov(T, R Q R^T, method="bilinear")).  X[B,m,m]; info[B] (0 ok, 1 = no
 * convergence: spectral radius >= 1).  Backward: given Xbar[B,m,m] accumulates (+=) into
 * Abar[B,m,m], Rbar[B,m,r], Qbar[B,r,r] (any may be NULL). */
kfb_status kfb_lyapunov_forward(int64_t B, int32_t m, int32_t r, const double *A, int64_t A_bs,
                                const double *R, int64_t R_bs, const double *Q, int64_t Q_bs,
                                double *X, int32_t *info, void *stream);
kfb_status kfb_lyapunov_backward(int64_t B, int32_t m, int32_t r, const double *A, int64_t A_bs,
                                 const double *R, int64_t R_bs, const double *Q, int64_t Q_bs,
                                 const double *X, const double *Xbar, double *Abar, double *Rbar,
                                 double *Qbar, void *stream);

/* theta -> system matrices ("base + scatter(theta)": every reference model's update() is a
 * set_subtensor of theta slices into constant matrices, models/SARIMAX.py:59-98,
 * models/VARMAX.py:95-141, models/local_level.py:28-49).  `dst` is one packed block of
 * `block` doubles per draw, initialised from base[block]; dst[b, dst_idx[k]] = theta[b, src_idx[k]].
 * Backward: gtheta[b, src_idx[k]] += gdst[b, dst_idx[k]] (gtheta must be zeroed by the caller). */
kfb_status kfb_scatter_forward(int64_t B, int32_t n_theta, int32_t block, int32_t n_map,
                               const double *theta, const double *base, const int32_t *src_idx,
                               const int32_t *dst_idx, double *dst, void *stream);
kfb_status kfb_scatter_backward(int64_t B, int32_t n_theta, int32_t block, int32_t n_map,
                                const double *gdst, const int32_t *src_idx, const int32_t *dst_idx,
                                double *gtheta, void *stream);

/* The same for SEVERAL matrices in one launch each way (an evaluation scatters theta into 3-5 matrices: one launch
 * instead of one per matrix; the backward WRITES gtheta - no zeroing by the caller - summing over all segments). */
#define KFB_MAX_SCATTER_SEGMENTS 8
typedef struct kfb_scatter_seg {
  int32_t block;           /* doubles per draw of this matrix */
  int32_t n_map;           /* entries of src_idx / dst_idx */
  const double *base;      /* [block] constant part (forward only) */
  const int32_t *src_idx;  /* [n_map] theta index */
  const int32_t *dst_idx;  /* [n_map] element index */
  double *data;            /* forward: dst [B, block] (written); backward: gdst [B, block] (read) */
} kfb_scatter_seg;
kfb_status kfb_scatter_forward_multi(int64_t B, int32_t n_theta, int32_t n_seg, const kfb_scatter_seg *segs,
                                     const double *theta, void *stream);
kfb_status kfb_scatter_backward_multi(int64_t B, int32_t n_theta, int32_t n_seg, const kfb_scatter_seg *segs,
                                      double *gtheta, void *stream);

/* Batched simulation helpers (next row f4, not on the logp/grad path): reference pymc_statespace/utils/simulation.py.
 * The standard-normal draws are INPUTS (z_*), so the kernels are deterministic.
 * kfb_simulate = simulate_statespace (:29-62) for n_draws * sims_per_draw trajectories: z_state[S,n,r], z_obs[S,n,p]
 *   -> states[S,n,m], obs[S,n,p] (S = n_draws*sims_per_draw; x0[n_draws,m] may be NULL; info[S] = 1 if Q or H is
 *   not positive definite; H identically zero = no observation noise, as in the reference).
 * kfb_mvn_draws = conditional_simulation / numba_mvn_draws (:8-26): out[s,t,:] = mus[u,t,:] + chol(covs[u,t] +
 *   jitter[s] I) z[s,t,:], u = s / sims_per_unit; info[S] must be zero-initialised (receives t+1 of a failing block). */
kfb_status kfb_simulate(int64_t n_draws, int64_t sims_per_draw, int32_t n, int32_t m, int32_t p, int32_t r,
                        const double *T, int64_t T_bs, const double *Z, int64_t Z_bs, const double *R, int64_t R_bs,
                        const double *H, int64_t H_bs, const double *Q, int64_t Q_bs, const double *x0, int64_t x0_bs,
                        const double *z_state, const double *z_obs, double *states, double *obs, int32_t *info,
                        void *stream);
kfb_status kfb_mvn_draws(int64_t n_units, int64_t sims_per_unit, int32_t n, int32_t k, const double *mus,
                         const double *covs, const double *z, const double *jitter, double *out, int32_t *info,
                         void *stream);

/* Simulation smoother (Durbin & Koopman 2002, mean correction; not on the logp/grad path): joint draws of the state
 * paths x_0..x_{n-1} from p(x | y, theta), sims_per_unit of them per unit.  Model: x_0 ~ N(a0, P0), y_t = Z x_t + d +
 * eps_t (eps_t ~ N(0, H), t = 0..n-1), x_{t+1} = T x_t + c + R eta_t (eta_t ~ N(0, Q), t = 0..n-2) - the filters' model;
 * NOT kfb_simulate's shifted convention obs[t] = Z states[t-1].  Per simulation:
 *   1. x+_0 = a0 + S_P0 z_init, x+_{t+1} = T x+_t + c + R S_Q z_state_t, y+_t = Z x+_t + d + S_H z_obs_t
 *      (S_A S_A^T = A: lower Cholesky that accepts PSD input - a pivot at or below 1e-10 times the largest diagonal
 *      entry is zero and its column is zeroed, a pivot below -1e-10 times it is an error; H = 0: no observation noise);
 *   2. y* = y - y+; a*_0 = 0, v_t = y*_t - Z a*_t, a*_{t+1} = T a*_t + K_t v_t, K_t = T P_t Z^T F_t^-1;
 *   3. r_{n-1} = 0, r_{t-1} = Z^T F_t^-1 v_t + L_t^T r_t, L_t = T - K_t Z;
 *   4. xhat_0 = P0 r_{-1}, xhat_{t+1} = T xhat_t + R Q R^T r_t;   5. states[s, t] = x+_t + xhat_t.
 * A missing row (all of y_t NaN) has F_t^-1 = 0, K_t = 0.  With KFB_FLAG_PARTIAL_ROWS in desc->flags a partly observed
 * row (observed set o) has kfb_masked_filter's F_t^-1 and K_t (zero rows / columns for the missing entries) and
 * v_t = 0 on its missing entries; predicted_covs then come from kfb_masked_filter.
 * Inputs: desc gives sizes and batch strides; every time stride must be 0 (else KFB_ERR_UNSUPPORTED); filter_kind and
 * every other flag are ignored.  k_states, k_endog, k_posdef <= 32 (else KFB_ERR_UNSUPPORTED).  predicted_covs[U, n+1, m, m] is
 * the output of a preceding kfb_forward (standard filter, KFB_FLAG_CORRECTED) on the same desc and inputs
 * (its row 0 is not read: P_0 is the input P0).  Simulation
 * s = unit * sims_per_unit + k (S = U * sims_per_unit).  Normals, time-major: z_init[S, m], z_state[n-1, S, r] (may be
 * NULL if n = 1), z_obs[n, S, p].  c, d may be NULL.  Output states[S, n, m]; info[U] (written, no zeroing needed):
 * 0 ok, t+1 F_t not positive definite, -(t+1) y_t partly missing (never with KFB_FLAG_PARTIAL_ROWS), KFB_INFO_NOT_PSD;
 * a failing unit's paths are NaN.  Workspace (kfb_simulation_smoother_workspace_bytes), each term rounded up to 256 bytes, with U = n_draws * n_series
 * and S32 = S rounded up to a multiple of 32:  8 U n (m p + p p)  +  8 U (2 m m + m r + p p + r r)  +  8 n S32 p
 *   +  8 (n - 1) S32 m  +  4 U. */
kfb_status kfb_simulation_smoother_workspace_bytes(const kfb_desc *desc, int64_t sims_per_unit, size_t *bytes);
kfb_status kfb_simulation_smoother(const kfb_desc *desc, const kfb_inputs *in, const double *predicted_covs,
                                   int64_t sims_per_unit, const double *z_init, const double *z_state,
                                   const double *z_obs, double *states, int32_t *info, void *workspace,
                                   size_t workspace_bytes, void *stream);

/* The exact filter over data with partly observed rows (not on the logp/grad path): the predicted moments that
 * kfb_forward (standard filter, KFB_FLAG_CORRECTED) gives, for a sample in which some rows y_t have NaN in some entries
 * and not others (series released on different dates: the ragged edge of a multivariate sample, gaps inside it).
 * kfb_forward refuses such a row (-(t+1)); this filter conditions on its observed entries.  At step t with observed
 * set o, every product in the masked p x p form:
 *   F = Z_o P Z_o^T + H_oo,  K = T P Z^T F^-1 (zero columns for the missing entries),  v = y - Z a - d on o, 0 elsewhere,
 *   a <- T a + c + K v,  P <- T P L^T + R Q R^T (L = T - K Z), symmetrised.
 * An all-missing row has K = 0; a complete row is the ordinary update; a non-diagonal H enters through H_oo.  Outputs
 * predicted_states[U, n+1, m] and predicted_covs[U, n+1, m, m] (row 0: a0, P0) have kfb_forward's layout and meaning,
 * so kfb_simulation_smoother (with KFB_FLAG_PARTIAL_ROWS), kfb_forecast_paths and kfb_conditional_forecast read them
 * unchanged; either may be NULL, not both.  info[U] (written): 0, or t+1 if F_o is not positive definite at step t (that
 * unit's outputs are NaN); never -(t+1).  desc as in kfb_simulation_smoother (n >= 1; filter_kind and flags ignored;
 * every time stride 0, sizes <= 32, else KFB_ERR_UNSUPPORTED); y, a0, P0, T, Z, R, H, Q required, c, d may be NULL.
 * Workspace (kfb_masked_filter_workspace_bytes), rounded up to 256 bytes:  8 U (5 m m + 2 m p + 3 p p). */
kfb_status kfb_masked_filter_workspace_bytes(const kfb_desc *desc, size_t *bytes);
kfb_status kfb_masked_filter(const kfb_desc *desc, const kfb_inputs *in, double *predicted_states,
                             double *predicted_covs, int32_t *info, void *workspace, size_t workspace_bytes,
                             void *stream);

/* Forecast paths from the end of the sample (not on the logp/grad path): joint draws of x_n..x_{n+H-1} and
 * y_n..y_{n+H-1} given y_0..y_{n-1}, sims_per_unit of them per unit.  Same model as kfb_simulation_smoother.  The start
 * (a, P) of a unit is the state's distribution at the first forecast time: the predicted moments a_n, P_n of a
 * preceding kfb_forward (standard filter, KFB_FLAG_CORRECTED), copied into start_mean[U, m], start_cov[U, m, m].  (Run
 * that filter on y extended by H all-NaN rows and its predicted moments n..n+H-1 are the forecast's moments.)
 * Simulation s = unit * sims_per_unit + k with (a, P) = (start_mean[unit], start_cov[unit]):
 *   x_0 = a + S_P z_init[s];  for h = 0..H-1:  states[h, s] = x_h,  obs[h, s] = Z x_h + d + S_H z_obs[h, s],
 *                                              x_{h+1} = T x_h + c + R S_Q z_state[h, s]  (h < H-1)
 * with S_A the PSD lower factor of kfb_simulation_smoother.  Normals and outputs are time-major: z_init[S, m],
 * z_state[H-1, S, r] (may be NULL if H = 1), z_obs[H, S, p], states[H, S, m], obs[H, S, p]; either output may be NULL,
 * not both.  desc gives U = n_draws * n_series, m, p, r and the batch strides of T, Z, R, H, Q, c, d (c, d may be NULL);
 * desc->n, filter_kind, flags and in->y, a0, P0 are not read.  Every time stride must be 0 and k_states, k_endog,
 * k_posdef <= 32 (else KFB_ERR_UNSUPPORTED); horizon < 1, sims_per_unit < 1, a null required pointer or both outputs
 * NULL: KFB_ERR_INVALID_ARG.  info[U] (written, no zeroing needed): 0, or KFB_INFO_NOT_PSD if P, Q or H is not positive
 * semi-definite or the start has a NaN; a failing unit's paths are NaN.  Workspace
 * (kfb_forecast_paths_workspace_bytes), each term rounded up to 256 bytes:  8 U (m m + m r + p p + r r)  +  4 U. */
kfb_status kfb_forecast_paths_workspace_bytes(const kfb_desc *desc, int64_t sims_per_unit, size_t *bytes);
kfb_status kfb_forecast_paths(const kfb_desc *desc, const kfb_inputs *in, const double *start_mean,
                              const double *start_cov, int32_t horizon, int64_t sims_per_unit, const double *z_init,
                              const double *z_state, const double *z_obs, double *states, double *obs, int32_t *info,
                              void *workspace, size_t workspace_bytes, void *stream);

/* Conditional forecasts from the end of the sample (not on the logp/grad path): the law of x_n..x_{n+H-1} and
 * y_n..y_{n+H-1} given y_0..y_{n-1} AND the known future values cond[h, i] = y_{n+h, i} (NaN = free), and joint draws
 * of those paths (Banbura, Giannone & Lenza 2015: the simulation smoother over the window, with partly observed rows).
 * Same model and start as kfb_forecast_paths: (a, P) = (start_mean[u], start_cov[u]) are a_n, P_n of a preceding
 * kfb_forward (standard filter, KFB_FLAG_CORRECTED) over the n observations.  cond is [H, p] shared by every unit
 * (cond_bs = 0) or [U, H, p] (cond_bs = H p).  Per unit, with o / u the conditioned / free entries of step h and every
 * product in the masked p x p form:
 *   window filter  F = Z_o P Z_o^T + H_oo, K = T P Z^T F^-1, v = cond - Z a - d (0 on free entries), u_h = F^-1 v,
 *                  a <- T a + c + K v, P <- T P L^T + R Q R^T (L = T - K Z);
 *   smoother       r_{h-1} = Z^T (u_h - K^T r_h) + T^T r_h, N_{h-1} = Z^T F^-1 Z + L^T N_h L  (r = N = 0 after H-1);
 *   state_mean[u, h] = a_h + P_h r_{h-1}, state_cov[u, h] = P_h - P_h N_{h-1} P_h;
 *   G = H_uo H_oo^- (generalised inverse by the PSD factor's zero-pivot rule; 0 for a diagonal H), D = Z_u - G Z_o;
 *   obs_mean[u, h] = cond on conditioned entries, D x^ + d_u + G (cond_o - d_o) on free ones; obs_cov[u, h] =
 *   D V D^T + H_uu - G H_ou on the free block, 0 on every row and column of a conditioned entry.
 * Paths (sims_per_unit > 0; simulation s = unit * sims_per_unit + k): Durbin & Koopman's mean correction over the
 * window from x+_0 = a + S_P z_init[s] with the normals of kfb_forecast_paths (time-major z_init[S, m],
 * z_state[H-1, S, r] (may be NULL if H = 1), z_obs[H, S, p]); states[h, s] = x~_h, obs[h, s] = cond on conditioned
 * entries and Z_u x~ + d_u + eps+_u + G (cond_o - Z_o x~ - d_o - eps+_o) on free ones (eps+_h = S_H z_obs[h, s]).
 * With no condition these are kfb_forecast_paths' paths on the same normals.  sims_per_unit = 0: moments only (no
 * normal or path pointer is read).  Any moment output [U, H, m], [U, H, m, m], [U, H, p], [U, H, p, p] may be NULL; with
 * paths, states[H, S, m] or obs[H, S, p] may be NULL, not both.  desc as in kfb_forecast_paths, plus desc->n >= 0 (the
 * number of observations, used for info codes only).  info[U] (written): 0; n + h + 1 if F_o is not positive definite
 * at window step h (the numbering of a filter over n + H steps; e.g. a condition the model already determines without
 * noise); KFB_INFO_NOT_PSD if P, Q or H is not positive semi-definite or the start has a NaN.  Every output of a failing
 * unit is NaN.  Workspace (kfb_conditional_forecast_workspace_bytes), each term rounded up to 256 bytes, with
 * U = n_draws * n_series and S32 = U * sims_per_unit rounded up to a multiple of 32:
 *   8 U H (m p + 2 p p + p + m + m m)  +  8 U (2 m m + m r + p p + r r)  +  8 U (3 m m + 2 m p + 4 p p)  +  4 U
 *   +  8 H S32 p  +  8 (H - 1) S32 m. */
kfb_status kfb_conditional_forecast_workspace_bytes(const kfb_desc *desc, int32_t horizon, int64_t sims_per_unit,
                                                    size_t *bytes);
kfb_status kfb_conditional_forecast(const kfb_desc *desc, const kfb_inputs *in, const double *start_mean,
                                    const double *start_cov, int32_t horizon, const double *cond, int64_t cond_bs,
                                    int64_t sims_per_unit, const double *z_init, const double *z_state,
                                    const double *z_obs, double *state_mean, double *state_cov, double *obs_mean,
                                    double *obs_cov, double *states, double *obs, int32_t *info, void *workspace,
                                    size_t workspace_bytes, void *stream);

/* Impulse responses for every draw: column j of horizon h is T^h R S e_j (states[n_draws, H, m, r]) and Z T^h R S e_j
 * (obs[n_draws, H, p, r]), the response to shock j at time 0.  Either output may be NULL, not both.  desc gives
 * n_draws, m, p, r and the batch strides of T, Z, R, Q (every time stride 0, sizes <= 32, else KFB_ERR_UNSUPPORTED);
 * nothing else of desc or in is read.  A bad `shock` or horizon < 1: KFB_ERR_INVALID_ARG.  info[n_draws] (written):
 * 0, or KFB_INFO_NOT_PSD if Q is not positive semi-definite under KFB_SHOCK_STD / _CHOLESKY; that draw's responses
 * are NaN. */
#define KFB_SHOCK_UNIT 0     /* S = I                                        */
#define KFB_SHOCK_STD 1      /* S = diag(sqrt(diag Q)): one standard deviation */
#define KFB_SHOCK_CHOLESKY 2 /* S = PSD lower factor of Q: orthogonalised     */
kfb_status kfb_impulse_response(const kfb_desc *desc, const kfb_inputs *in, int32_t horizon, int32_t shock,
                                double *states, double *obs, int32_t *info, void *stream);

/* FP64 roofline denominator: `iters` dependent-chain DFMA rounds on every SM.  Returns through
 * h_flops the number of floating-point operations the launch executes (2 per FMA); the caller
 * times it with CUDA events.  sink[>= 1] receives a checksum so the work cannot be elided. */
kfb_status kfb_fp64_peak(int32_t iters, int32_t blocks, int32_t threads, double *sink,
                         double *h_flops, void *stream);

/* Same probe, but every FMA reads three DISTINCT registers (no operand reuse) - the rate dense small-matrix code can
 * actually sustain through the register file. */
kfb_status kfb_fp64_peak_distinct(int32_t iters, int32_t blocks, int32_t threads, double *sink, double *h_flops,
                                  void *stream);

/* How many kernels this library has launched in this process (bench.py "gpu_launches"). */
int64_t kfb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* KFB200_H */
