/*
 * libbnr -- C ABI of the B200-native Gibbs engine for Bayesian Network Regression.
 *
 * This is the drop-in boundary for the sampler hot path of BayesianNetworkRegression.jl:
 *   reference interface replaced                                   entry point(s) here
 *   -------------------------------------------------------------  ---------------------------------
 *   initialize_and_run! / run!        src/gibbs.jl:822-846,849-864  bnr_create, bnr_init_state, bnr_run
 *   initialize_variables!             src/gibbs.jl:191-224          bnr_init_state
 *   gibbs_sample! + update_* (x10)    src/gibbs.jl:663-677,267-636  bnr_run (whole sweeps), bnr_step (one conditional)
 *   sample_gig & friends              src/gig.jl:8-176              inside bnr_run / bnr_step(BNR_COND_D)
 *   rhat / return_psrf_VOI            src/convergence.jl:4-65,
 *                                     src/gibbs.jl:771-789          bnr_set_moment_window, bnr_rhat,
 *                                                                   bnr_moments_device, bnr_rhat_from_moments
 *   state Table columns (Results)     src/gibbs.jl:23-29,835-841    bnr_get_state, bnr_set_state, bnr_get_trace
 *   pmap over chains (one process     src/gibbs.jl:946-948          num_chains batched per handle (= per GPU);
 *   per chain)                                                      chain_offset keys the RNG by global chain id
 *
 * Host wrappers (Julia `ccall`, Python `ctypes`) keep everything else of Fit!/Summary: kwargs,
 * parameters.log, setup_X!, the PSRF control loop, DataFrames.  See INTEGRATION.md.
 *
 * Conventions
 *  - every function returns 0 on success, a negative BNR_E* code otherwise; bnr_last_error() gives
 *    a thread-local message.  No exceptions cross the ABI.
 *  - all host buffers are owned by the caller and never retained after the call returns;
 *    device memory, streams and CUDA graphs are owned by the handle.
 *  - matrices use the REFERENCE layout (Julia column-major): X is n x q with X[i + n*j];
 *    u is R x V with u[r + R*k]; M is R x R; pi is R x 3 with pi[r + R*c], columns = P(0),P(+1),P(-1);
 *    gamma/S have length q = V(V+1)/2 ordered as src/utils.jl:40-57 (column k, rows l = k..V, diagonal
 *    included).  Traces are returned iteration-fastest: out[it + rows*elem], so a Julia
 *    Array{Float64,3}(rows, d1, d2) can wrap the buffer directly.
 *  - all arithmetic is FP64.  Random numbers: Philox4x32-10, key = (seed, global chain id),
 *    counter = (sub-block, element, draw site, iteration): results do not depend on how chains are
 *    distributed over handles/GPUs or chain groups (bit for bit, with one exception: when a handle
 *    holds so few chains that the Gram SYRK splits its contraction -- num_chains x tiles < 148 and
 *    q >= 1024 -- the split count, hence the rounding of G, depends on the handle's chain count).
 *  - a handle is not thread-safe.
 */
#ifndef BNR_H
#define BNR_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNR_VERSION 200

/* error codes */
#define BNR_OK 0
#define BNR_EINVAL (-1)   /* bad argument */
#define BNR_ECUDA (-2)    /* CUDA runtime error (message in bnr_last_error) */
#define BNR_ENOMEM (-3)
#define BNR_ESTATE (-4)   /* call not valid in the current state (e.g. trace not recorded) */
#define BNR_ENODEV (-5)   /* no usable CUDA device: there is NO CPU fallback */

/* state variables (Results.state columns, src/gibbs.jl:835-841) */
enum {
  BNR_VAR_TAU2 = 0, BNR_VAR_U = 1, BNR_VAR_XI = 2, BNR_VAR_GAMMA = 3, BNR_VAR_S = 4, BNR_VAR_THETA = 5,
  BNR_VAR_DELTA = 6, BNR_VAR_M = 7, BNR_VAR_MU = 8, BNR_VAR_LAMBDA = 9, BNR_VAR_PI = 10, BNR_NUM_VARS = 11
};

/* conditionals, in gibbs_sample! order (src/gibbs.jl:666-675) */
enum {
  BNR_COND_TAU2 = 0, BNR_COND_U_XI = 1, BNR_COND_GAMMA = 2, BNR_COND_D = 3, BNR_COND_THETA = 4,
  BNR_COND_DELTA = 5, BNR_COND_M = 6, BNR_COND_MU = 7, BNR_COND_LAMBDA = 8, BNR_COND_PI = 9,
  BNR_NUM_CONDS = 10
};

/* auxiliary (intermediate) quantities exposed for level-1 parity tests; sizes in doubles per chain */
enum {
  BNR_AUX_TAU2_PARAMS = 0,   /* [2]        shape, scale of the InverseGamma                       */
  BNR_AUX_SIGMA_INV = 1,     /* [V*R*R]    per node Sigma^-1 (after jitter), R x R col-major       */
  BNR_AUX_SIGMA_CHOL = 2,    /* [V*R*R]    per node lower Cholesky factor of Sigma^-1              */
  BNR_AUX_MU_T = 3,          /* [V*R]      per node conditional mean of u_k                        */
  BNR_AUX_LOG_ODDS = 4,      /* [V]        log(w_bot / w_top); w = 1/(1+exp(.))                    */
  BNR_AUX_W = 5,             /* [q]        W = lower_triangle(u' Lambda u)                         */
  BNR_AUX_G = 6,             /* [n*n]      X D X' + I, col-major (symmetric, both triangles filled);
                                           QFORM: [q*q] the precision P = (X'X + D^-1)/tau2         */
  BNR_AUX_G_CHOL = 7,        /* [n*n]      its lower Cholesky factor (strict upper = 0); QFORM: [q*q] */
  BNR_AUX_RHS = 8,           /* [n]        a1 - a3                                                  */
  BNR_AUX_A4 = 9,            /* [n]        (X D X' + I)^-1 (a1 - a3); QFORM: [q] beta = gamma - W  */
  BNR_AUX_CHI = 10,          /* [q]        GIG chi_j = (gamma_j - W_j)^2 / tau2                     */
  BNR_AUX_THETA_PARAMS = 11, /* [2]        shape, scale                                             */
  BNR_AUX_DELTA_PARAMS = 12, /* [2]        a, b                                                     */
  BNR_AUX_M_PARAMS = 13,     /* [1+2*R*R]  df, Psi (col-major), chol(Psi) lower                     */
  BNR_AUX_MU_PARAMS = 14,    /* [2]        mean, sd                                                 */
  BNR_AUX_LAMBDA_LOGW = 15,  /* [R*3]      loglik_v - max_v loglik_v, [r + R*c], c over (0,+1,-1)    */
  BNR_AUX_LAMBDA_WEIGHTS = 16,/* [R*3]     unnormalised weights pi[r,c]*exp(logw)                   */
  BNR_AUX_PI_ALPHA = 17,     /* [R*3]      Dirichlet parameters                                     */
  BNR_AUX_GIG_USED = 18,     /* [q]        uniforms consumed per edge by the GIG sampler            */
  BNR_NUM_AUX = 19
};

/* per-chain status bits (bnr_status) -- the device-side analogue of the reference's exceptions
 * and stderr diagnostics (src/gibbs.jl:313-347, 385-402, 527-543) */
#define BNR_ST_JITTER 1        /* Sigma^-1 needed the 1e-5 / 4e-5 jitter ladder          */
#define BNR_ST_SIGMA_NOTPD 2   /* Sigma^-1 not PD even after the ladder (reference throws) */
#define BNR_ST_G_NOTPD 4       /* X D X' + I lost positive definiteness                  */
#define BNR_ST_GIG_CAP 8       /* GIG rejection loop hit the attempt cap                 */
#define BNR_ST_INJ_EXHAUSTED 16/* injected uniform stream too short (test mode)          */
#define BNR_ST_NAN 32          /* NaN mixture weight (reference falls back to Bernoulli(0.5)) */
#define BNR_ST_PSI_NOTPD 64    /* I + sum u u' not PD                                    */

typedef struct bnr_handle bnr_handle;

typedef struct bnr_params {
  int32_t n;                 /* samples                                                     */
  int32_t V;                 /* nodes; q = V(V+1)/2 columns of X                            */
  int32_t R;                 /* latent dimension, 1..BNR_MAX_R                              */
  int32_t num_chains;        /* chains advanced in lock-step by this handle (this GPU)      */
  int32_t chain_offset;      /* global id of local chain 0 (RNG key); 0 for single-GPU      */
  int32_t device;            /* CUDA device ordinal                                         */
  int32_t trace_full_chains; /* leading local chains whose FULL state is recorded per row   */
  int32_t trace_gamma_xi_all;/* !=0: record gamma and xi rows of every chain                */
  int64_t trace_rows;        /* capacity (rows) of the trace buffers; 0 = no traces         */
  uint64_t seed;
  double eta, zeta, iota, a_delta, b_delta, nu;   /* Fit! hyper-parameters (src/gibbs.jl:725) */
  int32_t gig_inject_len;    /* K: injected uniforms per edge in injection mode (default 64) */
  int32_t gamma_mode;        /* BNR_GAMMA_AUTO (cost model) | BNR_GAMMA_NFORM | BNR_GAMMA_QFORM              */
  int32_t chain_groups;      /* chain groups advanced by independent streams/graphs (0 = default 2, max 4);
                                a throughput knob only: results are identical for every value               */
  int32_t trace_gamma_xi_chains; /* when trace_gamma_xi_all == 0: leading local chains whose gamma / xi rows are
                                    recorded (chain 1 is all Results / Summary need when R-hat is streamed)    */
} bnr_params;

/* Formulation of the gamma draw (update_gamma!, src/gibbs.jl:420-438).  Both sample the same conditional
 * N(W + m, P^-1), P = (X'X + D^-1)/tau2:
 *  NFORM  the reference's literal Bhattacharya draw through the n x n system X D X' + I (n^2 q + n^3/3 flops);
 *         consumes z1 (q normals) and z2 (n normals).
 *  QFORM  factors the q x q precision P = L L' directly (q^3/3 flops): L w = X'(y - mu - X W)/tau2,
 *         L' beta = w + z, gamma = W + beta; consumes z (q normals, the z1 site).
 *  AUTO   picks the cheaper one: QFORM iff q^3/3 + 4 q^2 < n^2 q + n^3/3 (roughly n > 0.53 q). */
#define BNR_GAMMA_AUTO 0
#define BNR_GAMMA_NFORM 1
#define BNR_GAMMA_QFORM 2

#define BNR_MAX_R 16
/* Size limits (bnr_create returns BNR_EINVAL beyond them; the reference has none): R <= 16; the factored dimension --
 * n + 1 for the n x n form, q + 1 for the q x q form, rounded up to a multiple of 128 -- at most 32768 (n <= 32767 in
 * the n-form, V <= 255 in the q-form; above 8192 the back solve runs on a cluster of 8 CTAs per chain); V * R doubles +
 * a few R x R blocks must fit 200 KB of shared memory.  AUTO keeps the choice it made under the former 8192 limit
 * wherever that choice fits 8192, and otherwise picks the cheaper of the forms that fit 32768. */
#define BNR_MAX_FACTOR_DIM 32768

int bnr_version(void);
const char* bnr_last_error(void);
void bnr_default_params(bnr_params* p);

/* X: n x q column-major host array, y: n.  Copies both to the device (padded, L2-friendly). */
int bnr_create(const bnr_params* p, const double* X, const double* y, bnr_handle** out);
int bnr_destroy(bnr_handle* h);
/* bnr_destroy returns the handle's device buffers to a process-wide cache (cudaFree of gigabytes is slow and
 * synchronises the device); the next bnr_create reuses buffers of equal size.  bnr_set_cache_limit bounds the
 * cached bytes (default 4 GiB; 0 disables caching and trims), bnr_trim_cache releases everything cached. */
int bnr_set_cache_limit(int64_t bytes);
int bnr_trim_cache(void);

/* Row 1 of every chain from the priors (initialize_variables!), iteration counter := 0. */
int bnr_init_state(bnr_handle* h);

/* Advance every chain by n_iters Gibbs sweeps (asynchronous; bnr_sync waits). */
int bnr_run(bnr_handle* h, int64_t n_iters);
int bnr_sync(bnr_handle* h);
int bnr_iteration(bnr_handle* h, int64_t* completed_sweeps);
/* milliseconds of device time of the last bnr_run (CUDA events on the handle's stream) */
int bnr_last_run_ms(bnr_handle* h, float* ms);

/* Trace row bookkeeping: the next recorded sweep is written to row `row` (0-based). Row 0 is written by
 * bnr_init_state.  Mirrors run!'s `j` index incl. the purge_burn ring (src/gibbs.jl:851-861). */
int bnr_set_trace_row(bnr_handle* h, int64_t row);
int bnr_get_trace_row(bnr_handle* h, int64_t* row);
int bnr_copy_trace_rows(bnr_handle* h, int64_t dst_row, int64_t src_row, int64_t count); /* copy_table! */

/* Split-half streaming moments for R-hat: sweeps whose 1-based number s satisfies
 * first <= s < first+len contribute; halves are [first, first+len/2) and the last len/2 sweeps. */
int bnr_set_moment_window(bnr_handle* h, int64_t first_sweep, int64_t len);
/* Block moments, for R-hat windows that GROW (the doubling scheme, src/gibbs.jl:1051-1198): sweep s >= first_sweep
 * contributes to block (s - first_sweep) / block_len (nblocks blocks; 0 switches the feature off).
 * bnr_moments_from_blocks merges the blocks [first_block, first_block + nblocks) -- nblocks even, the first half of
 * them forming the first split chain -- into the split-half moments buffer, after which bnr_rhat /
 * bnr_export_moments work as usual.  No chain needs a trace for R-hat. */
int bnr_set_moment_blocks(bnr_handle* h, int64_t first_sweep, int64_t block_len, int32_t nblocks);
int bnr_moments_from_blocks(bnr_handle* h, int32_t first_block, int32_t nblocks);
/* device pointer to [chain][half(2)][param(V xi then q gamma)][mean, M2] and its length in doubles */
int bnr_moments_device(bnr_handle* h, double** dev_ptr, int64_t* count);
/* R-hat (src/convergence.jl:4-65) from gathered moments of total_chains chains; dev_moments is a DEVICE
 * pointer (e.g. the output of an NCCL all-gather of bnr_moments_device buffers), outputs are HOST. */
int bnr_rhat_from_moments(int device, const double* dev_moments, int32_t total_chains, int32_t V, int32_t q,
                          int64_t half_len, double* rhat_xi, double* rhat_gamma);
/* fill the moments buffer from rows [first_row, first_row+nrows) of the recorded gamma/xi traces instead
 * (exactly the rows return_psrf_VOI hands to rhat); needs trace_gamma_xi_all */
int bnr_moments_from_trace(bnr_handle* h, int64_t first_row, int64_t nrows);
/* draws per split chain behind the current moments buffer (len/2 of the window, or nrows/2) */
int bnr_moment_half_len(bnr_handle* h, int64_t* half_len);
/* convenience: R-hat over this handle's chains only */
int bnr_rhat(bnr_handle* h, double* rhat_xi, double* rhat_gamma);

/* current state of one local chain in reference layout */
int bnr_get_state(bnr_handle* h, int32_t chain, int32_t var, double* out);
int bnr_set_state(bnr_handle* h, int32_t chain, int32_t var, const double* in);
int bnr_var_size(bnr_handle* h, int32_t var, int64_t* n_elems);
/* rows [first,last) of a recorded variable, iteration-fastest: out[(it-first) + (last-first)*elem] */
int bnr_get_trace(bnr_handle* h, int32_t chain, int32_t var, int64_t first, int64_t last, double* out);
int bnr_status(bnr_handle* h, int32_t* status_per_chain);

/* copy the moments buffer into caller-owned DEVICE memory (e.g. the input of an NCCL all-gather) */
int bnr_export_moments(bnr_handle* h, double* dev_dst);
/* Summary on the device (Summary, src/gibbs.jl:1214-1250) over trace rows [first_row, first_row + nrows) of one
 * chain: per-edge mean and the order statistics sort(gamma_j)[rank_lo], sort(gamma_j)[rank_hi] (1-based ranks =
 * the reference's lw / hi indices, exact: radix select, no interpolation), per-node mean xi.  Outputs are HOST
 * arrays of q, q, q and V doubles (any may be NULL); rounding to 3 digits stays in the host wrapper. */
int bnr_summary(bnr_handle* h, int32_t chain, int64_t first_row, int64_t nrows, int64_t rank_lo, int64_t rank_hi,
                double* gamma_mean, double* gamma_lo, double* gamma_hi, double* xi_mean);

/* Effective sample size of xi (V) and gamma (q) over trace rows [first_row, first_row + nrows) of ALL chains
 * (BASELINE metric "gamma ESS/sec"; the reference has no ESS - estimator: multi-chain Geyer initial monotone
 * sequence on per-chain-centred autocovariances, no rank normalisation, lags 0..max_lag computed directly).
 * bnr_ess = accumulate + finish for this handle's chains.  Multi-GPU: every rank calls bnr_ess_accumulate, the
 * host all-gathers the two device buffers of bnr_ess_device (autocovariance sums [max_lag+1][V+q] and chain means
 * [chains][V+q]) and calls bnr_ess_from_stats on the gathered DEVICE buffers (nparts = ranks). Needs
 * trace_gamma_xi_all.  max_lag is clamped to an odd value <= nrows-1; bnr_ess_device reports the value used. */
int bnr_ess(bnr_handle* h, int64_t first_row, int64_t nrows, int32_t max_lag, double* ess_xi, double* ess_gamma);
int bnr_ess_accumulate(bnr_handle* h, int64_t first_row, int64_t nrows, int32_t max_lag);
int bnr_ess_device(bnr_handle* h, double** acov_sum, int64_t* n_acov, double** chain_mean, int64_t* n_mean,
                   int32_t* max_lag);
/* copy the two statistics buffers into caller-owned DEVICE memory (the inputs of the NCCL all-gathers) */
int bnr_export_ess(bnr_handle* h, double* dev_acov_dst, double* dev_means_dst);
int bnr_ess_from_stats(int device, const double* dev_acov_parts, int32_t nparts, const double* dev_chain_means,
                       int32_t total_chains, int32_t V, int32_t q, int64_t nrows, int32_t max_lag, double* ess_xi,
                       double* ess_gamma);

/* as bnr_ess_from_stats, plus the number of lags each Geyer sequence consumed (max_lag + 1 = the sequence had not
 * terminated inside the lag budget: that ESS is an upper bound); lags_* may be NULL */
int bnr_ess_from_stats_lags(int device, const double* dev_acov_parts, int32_t nparts, const double* dev_chain_means,
                            int32_t total_chains, int32_t V, int32_t q, int64_t nrows, int32_t max_lag,
                            double* ess_xi, double* ess_gamma, double* lags_xi, double* lags_gamma);
/* Streaming ESS statistics: the next `ndraws` sweeps accumulate their lagged products on the device while they run
 * (ring of the last max_lag + 8 centred draws + [max_lag + 1] products per chain and parameter), so NO chain needs a
 * trace (64 chains x 20 000 draws x 5150 parameters of traces would be 53 GB).  After those sweeps
 * bnr_ess_stream_finish fills the same two statistics buffers as bnr_ess_accumulate: bnr_ess_device / bnr_export_ess /
 * bnr_ess_from_stats then work unchanged (nrows = ndraws).  max_lag is clamped like in bnr_ess_accumulate. */
int bnr_ess_stream_begin(bnr_handle* h, int32_t max_lag, int64_t ndraws);
/* the same with an explicit window: the sweeps first_sweep .. first_sweep + ndraws - 1 (1-based sweep numbers, none of
 * them run yet) contribute */
int bnr_ess_stream_window(bnr_handle* h, int32_t max_lag, int64_t first_sweep, int64_t ndraws);
int bnr_ess_stream_finish(bnr_handle* h);

/* Predictions for new networks (posterior predictive of the response y).  X_new is m x q column-major, built like X
 * (setup_X!).  Every recorded row of every chain -- row 0 by bnr_init_state, then one per sweep at the current trace
 * row, moved by bnr_copy_trace_rows like the traces -- also writes m doubles to the chain's prediction table:
 *   BNR_PRED_MEAN        mu + X_new[j,:] gamma                       (credible interval of E[y | x_j])
 *   BNR_PRED_PREDICTIVE  mu + X_new[j,:] gamma + sqrt(tau2) z_j      (posterior predictive interval), z_j ~ N(0,1)
 *                        from its own Philox draw site (element j, the row's sweep number)
 * with the row's own state.  Predictions only read the state: the chains are bit-identical with and without them.
 * Rows never written hold NaN.  The table has its own capacity, so handles without traces can predict too. */
#define BNR_PRED_MEAN 0
#define BNR_PRED_PREDICTIVE 1
/* X_new: m x q column-major; rows: capacity of each chain's prediction table; m = 0 switches predictions off.
 * Only BNR_PRED_MEAN and BNR_PRED_PREDICTIVE are accepted here; BNR_PRED_LOGDENS is set by bnr_set_heldout. */
int bnr_set_predictors(bnr_handle* h, int32_t m, const double* X_new, int64_t rows, int32_t mode);
/* Held-out rows (K-fold cross-validation): the prediction table of m observations the chains do not train on, whose
 * responses y_held are known.  Every recorded row then holds, in place of the prediction,
 *   BNR_PRED_LOGDENS     -1/2 log(2 pi tau2) - (y_held[j] - mu - X_held[j,:] gamma)^2 / (2 tau2)
 * with the row's own state; no random numbers are drawn.  X_held: m x q column-major, y_held: m.  It replaces any
 * predictors the handle had (like a second bnr_set_predictors call); m = 0 switches it off.  The table is read with
 * bnr_get_prediction_trace and bnr_export_predictions. */
#define BNR_PRED_LOGDENS 2
int bnr_set_heldout(bnr_handle* h, int32_t m, const double* X_held, const double* y_held, int64_t rows);
/* rows [first, last) of one local chain, iteration-fastest: out[(r - first) + (last - first) * j] */
int bnr_get_prediction_trace(bnr_handle* h, int32_t chain, int64_t first, int64_t last, double* out);
/* rows [first_row, first_row + nrows) of every local chain into caller-owned DEVICE memory as [chain][row][m] */
int bnr_export_predictions(bnr_handle* h, int64_t first_row, int64_t nrows, double* dev_dst);
/* pooled mean and order statistics over `count` rows of m doubles at a DEVICE pointer; outputs are HOST arrays.  Ranks
 * are 1-based and exact (radix select, no interpolation); the result does not depend on how the rows were produced. */
int bnr_prediction_summary(int device, const double* dev_rows, int64_t count, int32_t m, int64_t rank_lo,
                           int64_t rank_hi, double* mean, double* lo, double* hi);

/* Pointwise log-likelihood (out-of-sample scoring: PSIS-LOO and WAIC).  Every recorded row of every chain -- row 0 by
 * bnr_init_state, then one per sweep at the current trace row, moved by bnr_copy_trace_rows like the traces -- also
 * writes n doubles to the chain's log-likelihood table:
 *   ll[i] = -1/2 log(2 pi tau2) - (y_i - mu - (X gamma)_i)^2 / (2 tau2)
 * with the row's own state.  It only reads the state: the chains are bit-identical with and without it.  Rows never
 * written hold NaN.  rows: capacity of each chain's table (C x rows x n x 8 bytes); 0 switches it off. */
int bnr_set_loglik(bnr_handle* h, int64_t rows);
/* rows [first, last) of one local chain, iteration-fastest: out[(r - first) + (last - first) * i] */
int bnr_get_loglik_trace(bnr_handle* h, int32_t chain, int64_t first, int64_t last, double* out);
/* rows [first_row, first_row + nrows) of every local chain into caller-owned DEVICE memory as [chain][row][n] */
int bnr_export_loglik(bnr_handle* h, int64_t first_row, int64_t nrows, double* dev_dst);
/* PSIS-LOO and WAIC of N pooled draws x n observations at a DEVICE pointer (row-major [N][n]), as the R package loo 2.x
 * computes them with r_eff = 1 (psis, gpdfit); outputs are HOST arrays of n.  The Pareto tail of ceil(min(0.2 N,
 * 3 sqrt N)) draws is sorted in one block's shared memory: beyond about 8e7 draws on a B200 the call returns
 * BNR_EINVAL.  Deterministic: the same table gives bit-identical results. */
int bnr_loo_summary(int device, const double* dev_rows, int64_t N, int32_t n, double* elpd_loo, double* p_loo,
                    double* pareto_k, double* elpd_waic, double* p_waic);
/* Pooled log-mean-exp of N rows of m doubles at a DEVICE pointer (row-major [N][m]): lpd[j] = log((1/N) sum_s
 * exp(rows[s][j])), a HOST array of m -- the held-out log predictive density of K-fold cross-validation.  The rows are
 * split over blocks whose partials are added in a fixed order: the same table gives bit-identical results.  No size
 * limit beyond the device memory of the input. */
int bnr_lpd_summary(int device, const double* dev_rows, int64_t N, int32_t m, double* lpd);

/* chain groups (independent streams / CUDA graphs) the handle runs */
int bnr_chain_groups(bnr_handle* h, int32_t* groups);
/* which gamma formulation the handle runs (BNR_GAMMA_NFORM / BNR_GAMMA_QFORM; AUTO is resolved at create) */
int bnr_gamma_mode(bnr_handle* h, int32_t* mode);
/* number of CUDA kernels launched by bnr_run on this handle so far (graph replays counted per kernel node) */
int bnr_launch_count(bnr_handle* h, int64_t* kernels);
/* one eager sweep with CUDA events between phases; ms[8] = tau2, (u,xi), gamma prep, SYRK, Cholesky, solves,
 * X'a4+gamma+GIG, X gamma + scalar conditionals + record */
int bnr_profile_sweep(bnr_handle* h, float* ms);

/* ---------------------------------------------------------------------------------------------------------------
 * bnr_fit: everything Fit!(X, y, R; ...) does between setup_X! and Results in one call -- chain generation with the
 * purge_burn ring (run!, src/gibbs.jl:849-864), the PSRF-driven "extend burn-in" loop (generate_samples!, 897-1020) or
 * the "doubling" loop (generate_samples_dbl!, 1051-1198; chosen when mingen > 0 && maxgen > 0 like Fit!, 744-750),
 * R-hat over all chains (return_psrf_VOI, 771-789), the Summary statistics of chain 1 (1214-1250) and optionally the
 * gamma / xi ESS.  A host wrapper only converts its arguments and wraps the returned buffers (INTEGRATION.md).
 *
 * Chains: base.num_chains chains PER DEVICE on n_devices GPUs of this process (devices base.device, base.device + 1,
 * ...); global chain ids (RNG keys) are base.chain_offset + (ext_rank * n_devices + d) * num_chains + local id.  The only
 * data that crosses NVLink are the split-half moments (32 (V + q) bytes per chain), the ESS statistics and, with
 * bnr_fit_predict, the retained predictions (8 m bytes per chain and draw) and, with bnr_fit_loo, the retained
 * log-likelihood rows (8 n bytes per chain and draw), exchanged with ncclAllGather inside the library (libnccl.so.2 is loaded at run time; without it, peer copies).  Several
 * PROCESSES can fit a share each (ext_world > 1): the library then calls `allgather` to exchange across processes.
 * --------------------------------------------------------------------------------------------------------------- */
#define BNR_STATE_NONE 0       /* no table of chain 1 is kept for bnr_fit_state */
#define BNR_STATE_GAMMA_XI 1   /* gamma and xi rows of chain 1 */
#define BNR_STATE_FULL 2       /* every state variable of chain 1 (what Results.state holds in the reference) */

/* all-gather across the processes that call bnr_fit together: every process contributes `count` doubles at dev_send
 * (device memory on `device`) and receives ext_world * count doubles, in rank order, at dev_recv.  Return 0 on success. */
typedef int (*bnr_allgather_fn)(void* ctx, int device, const double* dev_send, double* dev_recv, int64_t count);

typedef struct bnr_fit_params {
  bnr_params base;          /* n, V, R, num_chains (per device), chain_offset, device, seed, hyper-parameters, gamma_mode,
                               chain_groups; the trace_* fields are set by bnr_fit */
  int64_t nburn, nsamples;  /* traditional scheme */
  int64_t mingen, maxgen;   /* doubling scheme when both > 0 */
  double psrf_cutoff;
  int64_t purge_burn;       /* 0 = nothing */
  int32_t return_state;     /* BNR_STATE_* */
  int32_t n_devices;        /* GPUs of this process to shard the chains over (>= 1) */
  int32_t interval;         /* credible level of the device Summary (95) */
  int32_t ess_max_lag;      /* > 0: also the Geyer ESS of xi / gamma over the retained draws, lags 0..ess_max_lag */
  int32_t verbose;          /* != 0: the reference's "samples generated. Max PSRF ..." lines on stderr */
  int32_t ext_world, ext_rank;   /* multi-process use (0 / 1 = single process) */
  bnr_allgather_fn allgather;
  void* allgather_ctx;
} bnr_fit_params;

typedef struct bnr_fit_info {
  int64_t tot_generated;    /* rows generated per chain (the reference's tot_generated) */
  int64_t burn_in, sampled; /* Results.burn_in, Results.sampled: the retained draws are table rows burn_in .. burn_in + sampled - 1 (0-based) */
  int64_t rows;             /* rows of chain 1's table (bnr_fit_state) */
  int64_t n_psrf;           /* PSRF evaluations */
  int32_t streamed;         /* R-hat came from streamed (or block) moments: no chain but the first kept a trace */
  int32_t summary_ok, ess_ok;
  int32_t gamma_mode, status_or, total_chains, n_devices;
  int32_t exchange;         /* 0 none (one device), 1 NCCL, 2 peer copies */
} bnr_fit_info;

typedef struct bnr_fit_result bnr_fit_result;

void bnr_fit_default_params(bnr_fit_params* p);
const char* bnr_fit_last_error(void);
/* X: n x q column-major (the matrix setup_X! builds), y: n.  The result owns its handles until bnr_fit_free. */
int bnr_fit(const bnr_fit_params* p, const double* X, const double* y, bnr_fit_result** out);
int bnr_fit_get_info(const bnr_fit_result* r, bnr_fit_info* info);
int bnr_fit_rhat(const bnr_fit_result* r, double* rhat_xi, double* rhat_gamma);              /* [V], [q] */
int bnr_fit_summary(const bnr_fit_result* r, double* gamma_mean, double* gamma_lo, double* gamma_hi, double* xi_mean);
int bnr_fit_ess(const bnr_fit_result* r, double* ess_xi, double* ess_gamma);
/* rows 0 .. info.rows - 1 of one state variable of chain 1 in the reference layout (iteration fastest) */
int bnr_fit_state(bnr_fit_result* r, int32_t var, double* out);
/* the engine handle of one of the result's devices (valid until bnr_fit_free), e.g. for bnr_status / bnr_get_trace */
int bnr_fit_handle(bnr_fit_result* r, int32_t device_index, bnr_handle** h);
int bnr_fit_free(bnr_fit_result* r);
/* bnr_fit plus predictions for m new networks (X_new: m x q column-major, mode BNR_PRED_*); bnr_fit itself is unchanged
 * and issues exactly the same operations.  Every chain of every device and process keeps a prediction table of the
 * fit's row capacity; the retained rows of all chains are all-gathered in global-chain order (the same exchange as the
 * moments) and reduced on device 0.  The tables and the pooled buffer (total_chains x rows x m doubles) are allocated
 * before the first sweep: a fit that cannot hold them fails at once with BNR_ENOMEM. */
int bnr_fit_predict(const bnr_fit_params* p, const double* X, const double* y, int32_t m, const double* X_new,
                    int32_t mode, bnr_fit_result** out);
/* per new network: the mean and the order statistics of ranks round(N (100 - interval) / 200) and
 * round(N (1 - (100 - interval) / 200)) (Julia round) of the N = total_chains x sampled pooled draws; [m] each */
int bnr_fit_prediction(const bnr_fit_result* r, double* mean, double* lo, double* hi);
/* bnr_fit_predict (m = 0: no predictions) plus a pointwise log-likelihood table on every chain of every device and
 * process; the retained rows of all chains are all-gathered in global-chain order and reduced on device 0 by
 * bnr_loo_summary.  The tables (C x rows x n doubles per device), the export buffers and the pooled buffer
 * (total_chains x rows x n doubles) are allocated before the first sweep: a fit that cannot hold them fails at once
 * with BNR_ENOMEM.  All other outputs equal those of bnr_fit_predict with the same arguments. */
int bnr_fit_loo(const bnr_fit_params* p, const double* X, const double* y, int32_t m, const double* X_new,
                int32_t pred_mode, bnr_fit_result** out);
/* per observation [n]: elpd_loo, p_loo, Pareto k, elpd_waic, p_waic over the N = total_chains x sampled pooled draws;
 * BNR_ESTATE when the fit ran without bnr_fit_loo or kept fewer than 2 draws */
int bnr_fit_loo_pointwise(const bnr_fit_result* r, double* elpd_loo, double* p_loo, double* pareto_k,
                          double* elpd_waic, double* p_waic);
/* K-fold cross-validation (loo::kfold with r_eff = 1): observation i belongs to fold fold[i] in 1..K.  Fold f trains
 * on the rows with fold != f, in their original order, and holds out the rows with fold == f (bnr_set_heldout).  Every
 * fold is the fit bnr_fit makes of its training rows with chain_offset = base.chain_offset + f * num_chains (f 0-based)
 * on device base.device + f mod n_devices, bit for bit; all folds share one control loop, whose PSRF step sees the
 * maximum R-hat over every fold (NaN if any is NaN), and every fold's sweeps are launched before any is waited for.
 * Afterwards elpd_kfold[i] = log((1/S) sum_s N(y_i | mu_s + x_i gamma_s, tau2_s)) over the S = num_chains x sampled
 * retained draws of i's fold.  The held-out tables and export buffers are allocated before the first sweep: a run that
 * cannot hold them fails at once with BNR_ENOMEM.  Refused with BNR_EINVAL: K < 2, a label outside 1..K, an empty fold
 * or training set, ext_world > 1, ess_max_lag > 0.  On the result: bnr_fit_get_info gives total_chains = K x
 * num_chains and the devices used, bnr_fit_handle(r, f, ...) fold f's handle, bnr_fit_rhat the element-wise maximum
 * over the folds; bnr_fit_summary, bnr_fit_state, bnr_fit_prediction, bnr_fit_ess and bnr_fit_loo_pointwise return
 * BNR_ESTATE. */
int bnr_fit_kfold(const bnr_fit_params* p, const double* X, const double* y, int32_t K, const int32_t* fold,
                  bnr_fit_result** out);
/* elpd_kfold of every observation [n], in the original order */
int bnr_fit_kfold_pointwise(const bnr_fit_result* r, double* elpd_kfold);
/* the last R-hat of fold f (0-based) alone: [V], [q] */
int bnr_fit_kfold_rhat(const bnr_fit_result* r, int32_t f, double* rhat_xi, double* rhat_gamma);
/* The control flow of bnr_fit as a pure host function (no GPU): the engine operations a fit would issue when its k-th
 * PSRF evaluation returns psrf_max[k] as the maximum R-hat of both xi and gamma (NaN allowed; 0 beyond n_psrf).
 * ops: [cap_ops][4] = (op, a, b, c) with op  0 create(trace rows, all chains traced, full-state chains)  1 init
 *   2 run(a sweeps)  3 set trace row a  4 copy rows (dst a, src b, count c)  5 moment window(first sweep a, length b)
 *   6 moment blocks(first a, block length b, count c)  7 PSRF from trace rows [a, a + b)  8 PSRF from the streamed
 *   window  9 PSRF from blocks [a, a + b)  10 ESS window(first sweep a, length b).
 * Used by the CPU test-suite to check the loops against the restated reference (oracle/psrf_loops.py). */
int bnr_fit_plan(const bnr_fit_params* p, const double* psrf_max, int32_t n_psrf, int64_t* ops, int64_t cap_ops,
                 int64_t* n_ops, bnr_fit_info* info);
/* device-to-device copy helper for all-gather callbacks written in a host language without a CUDA binding */
int bnr_device_copy(int device, void* dev_dst, const void* dev_src, int64_t bytes);

/* ---- parity-test hooks (tests only) ---- */
/* Injected basic variates replacing Philox: host array [num_chains][per_chain], layout documented in
 * oracle/bnr_oracle.py:draw_layout (sweep) / init_layout (init).  NULL switches injection off. */
int bnr_set_injection(bnr_handle* h, const double* inj, int64_t per_chain);
int bnr_injection_size(bnr_handle* h, int32_t for_init, int64_t* per_chain);
/* Run ONE conditional of the sweep that would produce sweep number (completed+1), in place. */
int bnr_step(bnr_handle* h, int32_t cond);
/* bnr_step sequence bookkeeping: call after the 10th conditional to count the sweep as completed */
int bnr_finish_sweep(bnr_handle* h);
int bnr_enable_aux(bnr_handle* h, int32_t on);
int bnr_get_aux(bnr_handle* h, int32_t chain, int32_t aux_id, double* out, int64_t capacity);
/* the Cholesky-with-jitter ladder of update_u_xi! (src/gibbs.jl:322-347) applied by the device routine the sweep uses
 * to a caller-supplied R x R matrix (col-major): A_used = the matrix that finally factored (A, A + 1e-5 I or
 * A + 5e-5 I), L = its lower factor, status = BNR_ST_JITTER / BNR_ST_SIGMA_NOTPD bits */
int bnr_test_chol_jitter(bnr_handle* h, int32_t R, const double* A, double* A_used, double* L, int32_t* status);
/* raw basic variates of the production RNG for a draw site (lets the oracle replay Philox mode):
 * kind 0 = uniform, 1 = normal; fills out[count] with the first `count` values of stream
 * (iteration, site, element) of local chain `chain`. */
int bnr_rng_stream(bnr_handle* h, int32_t chain, int64_t iteration, int32_t site, int32_t element,
                   int32_t kind, int32_t count, double* out);
/* unit-scale Gamma(shape) variates from the same stream machinery (Marsaglia-Tsang) */
int bnr_rng_gamma(bnr_handle* h, int32_t chain, int64_t iteration, int32_t site, int32_t element,
                  double shape, int32_t count, double* out);

#ifdef __cplusplus
}
#endif
#endif /* BNR_H */
