// Host-callable launchers shared between the translation units of libbnr.
#pragma once
#include <cuda_runtime.h>
#include "bnr_engine.cuh"

// internal mirrors of include/bnr.h constants (kept in sync by a static_assert in bnr_api.cu)
#define BNR_ST_JITTER_ 1
#define BNR_ST_SIGMA_NOTPD_ 2
#define BNR_ST_G_NOTPD_ 4
#define BNR_ST_GIG_CAP_ 8
#define BNR_ST_INJ_EXHAUSTED_ 16
#define BNR_ST_NAN_ 32
#define BNR_ST_PSI_NOTPD_ 64
#define BNR_COND_THETA_ 4
#define BNR_COND_DELTA_ 5
#define BNR_COND_M_ 6
#define BNR_COND_MU_ 7
#define BNR_COND_LAMBDA_ 8
#define BNR_COND_PI_ 9

namespace bnr {

extern thread_local long long g_launches;   // kernels launched through the wrappers below (host-side count)

void launch_tau2(const Engine& e, cudaStream_t s);
void launch_uxi(const Engine& e, cudaStream_t s);
void launch_edge_prep(const Engine& e, int draw_v, cudaStream_t s);   // draw_v: 0 W only, 1 v = W + delta1, 2 v = z
void launch_rhs(const Engine& e, cudaStream_t s);                     // n-form a1 - a3; q-form (y - mu - X W)/tau2
void launch_gamma_gig(const Engine& e, int flags, cudaStream_t s);
void launch_finish(const Engine& e, int mask, cudaStream_t s);
void launch_init(const Engine& e, cudaStream_t s);
void launch_record(const Engine& e, int sweep_done, cudaStream_t s);
void launch_advance(const Engine& e, int inc_iter, cudaStream_t s);
void launch_test_chol_jitter(int R, const double* Ain, double* Aused, double* Lout, int* status, cudaStream_t s);
void launch_rng_dump(const Dims& d, int chain, long long iteration, int site, int element, int kind, double shape,
                     int count, double* out, cudaStream_t s);

// dense linear algebra (bnr_linalg.cu)
// out[c][m] = sum_k A(m,k) v[c][k];  trans=0: A = X (np x qp), out = e.xv-like [C][np], in [C][qp]
//                                     trans=1: A = X' (qp x np), out [C][qp], in [C][np]
void launch_x_times(const Engine& e, int trans, const double* in, double* out, double* splitk_ws, cudaStream_t s);
// the same product with any operand A (lda >= M, K = qp for trans 0); out == nullptr leaves the k-split partial products
// [splits][d.C][M] in splitk_ws without adding them (a single split included)
void launch_x_times(const Dims& d, int trans, const double* A, int lda, int M, int K, const double* in, double* out,
                    double* splitk_ws, cudaStream_t s);
size_t x_times_workspace_doubles(const Dims& d);
// predictions: partials of X_new gamma for every chain of the view into e.pred_ws (k_xmma<0>, pred_splits(d, mp) splits)
int pred_splits(const Dims& d, int mp);
void launch_pred_product(const Engine& e, cudaStream_t s);
// adds the partials in split order, mu_c and (predictive mode) sqrt(tau2_c) z_j, and stores the row at *e.trace_row
void launch_pred_record(const Engine& e, int sweep_done, cudaStream_t s);
// pointwise log-likelihood of the current state (needs e.xg == X gamma) into e.ll at *e.trace_row
void launch_loglik_record(const Engine& e, cudaStream_t s);
void launch_syrk_G(const Engine& e, cudaStream_t s);         // G_c = X diag(S_c) X' + I (lower tiles)
int syrk_splits(const Dims& d, int C);                        // k-splits launch_syrk_G uses for a batch of C chains
// launch_syrk_G computes the n-form Gram matrix on the INT8 tensor cores (Ozaki digit planes) for qp in
// [GRAM_I8_QP_MIN, GRAM_I8_QP_MAX], on the FP64 DMMA SYRK otherwise.  The rule depends on the shape only, never on the
// chain count: every chain grouping and graph / eager sweeps keep the same rounding.
constexpr int GRAM_I8_QP_MIN = 1024;
constexpr int GRAM_I8_QP_MAX = 18724;     // 7 qp 2^14 < 2^31: the int32 accumulators of the digit products are exact
bool gram_i8_selected(const Dims& d);
size_t gram_i8_plane_bytes(const Dims& d);                    // digit planes of one chain
// branch streams + events that let launch_cholesky run the off-diagonal panel updates next to the panel factorisation
// (works eagerly and under stream capture, where it becomes a fork/join of the graph)
struct ForkJoin {
  cudaStream_t side = nullptr;   // low priority: throughput work (the Gram SYRK)
  cudaStream_t side_hi = nullptr;// same priority as the main stream: the Cholesky's look-ahead branch (it feeds the
                                 // critical path two steps later and must not queue behind other groups' SYRK CTAs)
  cudaEvent_t fork = nullptr, join = nullptr;
  cudaEvent_t* pool = nullptr;   // 4 events per Cholesky panel (see launch_cholesky); owned by the handle
  int npool = 0;
};
// in-place lower Cholesky of every G_c (gdim x gdim); the forward solve L w = rhs rides along as a bordering row
void launch_cholesky(const Engine& e, double* rhs, const ForkJoin& fj, cudaStream_t s);
// rhs_c <- L_c^-T (rhs_c + addz_c); addz may be null
void launch_chol_solve(const Engine& e, double* rhs, const double* addz, cudaStream_t s);
void launch_xtx(const Dims& d, const double* XT, const double* ones, double* XtX, cudaStream_t s);   // X'X, once
void launch_build_P(const Engine& e, cudaStream_t s);        // q-form: P_c = (X'X + diag(1/S_c)) / tau2_c
int chol_max_dim();
int bwd_stream_max_dim();                                     // above it the back solve runs on a CTA cluster per chain
int bwd_cluster_capacity(int N);                              // resident back-solve clusters (0: none fits, < 0: error)
bool tmaps_check(const Engine& e);                            // all tensor maps of this handle's geometry encode
bool tmap_setup();                                            // resolves cuTensorMapEncodeTiled (false: driver without TMA maps)
void linalg_setup();                                          // one-time cudaFuncSetAttribute calls
void small_kernels_setup();

// posterior diagnostics on the device (bnr_diagnostics.cu)
void launch_summary_select(const double* rows, size_t rowlen, int off, int nelem, long long first, long long count,
                           long long rank_lo, long long rank_hi, double* mean_out, double* lo_out, double* hi_out,
                           cudaStream_t s);
// rows [first, first + N) of every chain of the (xi, gamma) trace table tr
void launch_chain_mean(const RowTable& tr, long long first, long long N, double* cmean, cudaStream_t s);
void launch_acov_sum(const RowTable& tr, long long first, long long N, int L, const double* cmean, double* acov,
                     cudaStream_t s);
// streaming ESS: per-sweep lagged-product accumulation (no all-chain trace) and its conversion into the statistics
// launch_acov_sum / launch_chain_mean produce (acov [L+1][P] summed over the local chains, chain means [C][P])
void launch_ess_stream(const Engine& e, cudaStream_t s);
void launch_ess_stream_finalize(const Engine& e, long long N, double* acov, double* cmean, cudaStream_t s);
// pooled predictions: mean and the exact order statistics (1-based ranks) of each of the m columns of rows[N][m];
// ws: pred_select_ws_bytes(N, m) bytes of device scratch
size_t pred_select_ws_bytes(long long N, int m);
void launch_pred_select(const double* rows, long long N, int m, long long rank_lo, long long rank_hi, double* mean,
                        double* lo, double* hi, void* ws, cudaStream_t s);
// pooled PSIS-LOO and WAIC of each of the n columns of rows[N][n] (loo 2.x psis / gpdfit, r_eff = 1); out: [5][n]
// (elpd_loo, p_loo, pareto_k, elpd_waic, p_waic).  ws: loo_ws_bytes(N, n) bytes; loo_tail_max() bounds the tail length
long long loo_tail_len(long long N);
long long loo_tail_max();
size_t loo_ws_bytes(long long N, int n);
void launch_loo(const double* rows, long long N, int n, double* out, void* ws, cudaStream_t s);
// pooled log-mean-exp of each of the m columns of rows[N][m]: lpd[j] = logsumexp_s rows[s][j] - log N (fixed order);
// ws: lpd_ws_bytes(N, m) bytes
size_t lpd_ws_bytes(long long N, int m);
void launch_lpd(const double* rows, long long N, int m, double* lpd, void* ws, cudaStream_t s);
void launch_ess_finish(const double* acov_parts, int nparts, const double* cmeans, int chains, int P, long long N,
                       int L, double* ess, double* lag_used, cudaStream_t s);
// split R-hat of [chains][2][nparams][2] moments (h draws per half); the split-half moments of mom from trace rows
// [first, first + nrows) of every chain of tr, or from blocks of blen sweeps (these two not counted in g_launches)
void launch_rhat(const double* mom, int chains, int nparams, long long h, double* out, cudaStream_t s);
void launch_moments_from_trace(const RowTable& tr, long long first, long long nrows, const SplitMoments& mom,
                               cudaStream_t s);
void launch_merge_blocks(const SplitMoments& mom, int chains, int first_block, int per_half, long long blen,
                         cudaStream_t s);

}  // namespace bnr
