// Device-side view of one handle: dimensions, data, per-chain state and workspaces (all FP64, SoA by chain).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "bnr_rng.cuh"

namespace bnr {

constexpr int MAX_R = 16;
constexpr int TILE_N = 128;   // n is padded to a multiple of this (SYRK / Cholesky tiles)
constexpr int TILE_K = 16;    // q is padded to a multiple of this (SYRK k-step)
constexpr int TAU2_MAX_BLOCKS = 32;   // blocks per chain of the tau2 reduction
constexpr int PART_BLOCK = 256;  // threads per block of the edge kernels (partials granularity)

struct Dims {
  int n, V, R, q, C;
  int C_total;        // chains of the whole handle (C is the count of the view: a chain group sees a part); schedule
                      // choices that change the rounding depend on C_total only, so chain groups never change results
  int np, qp;         // padded n (multiple of TILE_N) and q (multiple of TILE_K; of TILE_N in the q-form)
  int gmode;          // gamma draw: 1 = n x n Bhattacharya form (G = X D X' + I), 2 = q x q precision form
  int gdim;           // dimension of the matrix that is factored every sweep: np (n-form) or qp (q-form); always
                      // > n resp. q: the first padding row carries the right-hand side of the forward solve
  int nparts;         // edge-kernel blocks per chain = ceil(q / PART_BLOCK)
  int chain_offset;
  int chain_offset_local;   // index of this view's first chain inside the handle (0 for the handle itself)
  int gigK;           // injected uniforms per edge
  uint64_t seed;
  double eta, zeta, iota, a_delta, b_delta, nu;
};

// injected-variate layout of one chain (must equal oracle/bnr_oracle.py:draw_layout)
struct InjLayout {
  int64_t tau2, uxi, z1, z2, S, theta, Delta, M, mu, lambda, pi, total;
  __host__ __device__ static InjLayout make(int n, int V, int R, int K) {
    InjLayout l;
    const int64_t q = (int64_t)V * (V + 1) / 2;
    int64_t o = 0;
    l.tau2 = o; o += 1;
    l.uxi = o; o += (int64_t)V * (R + 1);
    l.z1 = o; o += q;
    l.z2 = o; o += n;
    l.S = o; o += q * K;
    l.theta = o; o += 1;
    l.Delta = o; o += 3;
    l.M = o; o += R + R * (R - 1) / 2;
    l.mu = o; o += 1;
    l.lambda = o; o += R;
    l.pi = o; o += 3 * R;
    l.total = o;
    return l;
  }
};

// init layout (oracle/bnr_oracle.py:init_layout)
struct InitLayout {
  int64_t S, pi, lambda, xi, M, u, gamma, total;
  __host__ __device__ static InitLayout make(int V, int R) {
    InitLayout l;
    const int64_t q = (int64_t)V * (V + 1) / 2;
    int64_t o = 0;
    l.S = o; o += q;
    l.pi = o; o += 3 * R;
    l.lambda = o; o += R;
    l.xi = o; o += V;
    l.M = o; o += R + R * (R - 1) / 2;
    l.u = o; o += (int64_t)V * R;
    l.gamma = o; o += q;
    l.total = o;
    return l;
  }
};

struct Aux {           // optional intermediate outputs for parity tests (nullptr when disabled)
  double* tau2_params;   // [C][2]
  double* sigma_inv;     // [C][V][R*R]
  double* sigma_chol;    // [C][V][R*R]
  double* mu_t;          // [C][V][R]
  double* log_odds;      // [C][V]
  double* chi;           // [C][qp]
  double* theta_params;  // [C][2]
  double* delta_params;  // [C][2]
  double* m_params;      // [C][1+2*R*R]
  double* mu_params;     // [C][2]
  double* lambda_logw;   // [C][R*3]
  double* lambda_w;      // [C][R*3]
  double* pi_alpha;      // [C][R*3]
  double* gig_used;      // [C][qp]
  double* G_copy;        // [C][gdim*gdim]  X D X' + I (n-form) or P (q-form) before factorisation
};

// One row of `width` doubles per chain and recorded sweep, chain-major: the layout of every table the record kernels
// write at *trace_row (traces, predictions, log-likelihood) and bnr_copy_trace_rows moves.  base == nullptr: off
struct RowTable {
  double* base; long long rows; int width; int chains;
  __host__ __device__ bool holds(int c, long long r) const { return base && c < chains && r < rows; }
  __host__ __device__ double* row(int c, long long r) const { return base + ((size_t)c * rows + r) * width; }
  // the chains [c0, c0 + Cg) of a chain group (only the leading `chains` chains have rows)
  RowTable view(int c0, int Cg) const {
    RowTable v = *this;
    v.chains = chains - c0 < 0 ? 0 : (chains - c0 > Cg ? Cg : chains - c0);
    v.base = base && v.chains > 0 ? row(c0, 0) : nullptr;
    return v;
  }
  size_t doubles() const { return (size_t)chains * rows * width; }
};

struct Engine {
  Dims d;
  // data (read-only, shared by all chains)
  const double* X;        // [qp][np] : column j of X padded to np rows (zeros beyond n and beyond q)
  const double* y;        // [np]
  const int2* edge_lk;    // [q] (l, k) of edge j, l >= k
  const double* XtX;      // [qp][qp] X'X, lower triangle, column-major (q-form only, computed once)
  // state, [C][...]
  double* tau2; double* u; double* u_alt; double* xi; double* gamma; double* S; double* theta;
  double* Delta; double* M; double* mu; double* lambda; double* pi;
  // workspaces
  double* W;        // [C][qp]  lower_triangle(u' Lambda u) with current u, lambda
  double* v;        // [C][qp]  W + delta1
  double* t;        // [C][qp]  X' a4
  double* xg;       // [C][np]  X gamma (cached between mu and the next tau2)
  double* xv;       // [C][np]  X (W + delta1)
  double* rhs;      // [C][np]  a1 - a3, then L^-1 rhs, then a4 (in place); q-form: (y - mu - X W)/tau2
  double* G;        // [C][gdim*gdim] col-major, lower triangle used
  double* syrk_ws;  // [C][syrk_ws_cap][gdim*gdim] partial Gram matrices of the k-split SYRK (nullptr: never split)
  int syrk_ws_cap;  // splits - 1, fixed per handle
  signed char* gram_planes;  // [C][7][np][qp] int8 digit planes of X diag(sqrt(S_c)) (INT8 Gram path, else nullptr)
  double* gram_rscale;       // [C][np] power-of-two row scales of the digit planes
  double* Linv;     // [C][gdim/128][128*128]  inverses of the 128 x 128 diagonal blocks of the factor (column-major)
  double* partials; // [C][nparts][2*MAX_R+1]  block partial sums: A_r, B_r (lambda), sum S
  double* tau2_part;      // [handle chains][2 * TAU2_MAX_BLOCKS] partial sums of the tau2 reduction (NOT offset per view)
  unsigned* tau2_ticket;  // [handle chains] arrival counters of its blocks
  int* status;      // [C]
  long long* iter;  // device scalar: completed sweeps
  long long* trace_row;   // device scalar: next trace row
  // moments [C][2][V+q][2] and window
  double* moments;
  long long* mom_window;  // device [5]: split-half window (first sweep, len), block moments (first sweep, block len, blocks)
  double* bmom;           // [C][bmom_nb][V+q][2] per-block (mean, M2): mergeable R-hat windows (doubling scheme)
  int bmom_nb;
  // streaming ESS statistics (bnr_ess_stream_begin; kernels in bnr_diagnostics.cu).  y_t = x_t - x_first per chain / parameter
  double* ess_ring;       // [C][ess_cap][V+q]  ring of the last ess_cap centred draws
  double* ess_head;       // [C][L][V+q]        the first L centred draws
  double* ess_acc;        // [C][L+1][V+q]      lagged products A_l = sum_t y_t y_(t-l)
  double* ess_sum;        // [C][2][V+q]        x_first, sum_t y_t
  const long long* ess_win;  // device [4]: first sweep, draws N, max lag L, ring capacity ess_cap
  int ess_L, ess_cap;
  // traces of the leading tr_full.chains / tr_gx.chains chains; both keep rows = the handle's trace capacity when off
  RowTable tr_full;       // full state rows (state_elem order)
  RowTable tr_gx;         // xi then gamma, width V+q
  // predictions for new networks (bnr_set_predictors; pred.base == nullptr: off).  Every recorded row r of chain c gets
  // pred.row(c, r)[j] = mu_c + X_new[j,:] gamma_c (+ sqrt(tau2_c) z_j in the predictive mode), width m
  RowTable pred;
  const double* Xp;       // [qp][pred_mp] X_new columns padded to pred_mp rows (a multiple of 128; zeros beyond m, q)
  int pred_mp, pred_mode, pred_splits;   // padded m, BNR_PRED_*, k-splits of the product X_new gamma
  double* pred_ws;        // split-K partials of X_new gamma, [pred_splits][C][pred_mp]; a chain group's view uses
                          // [pred_splits][Cg][pred_mp] at offset c0 * pred_splits * pred_mp
  // pointwise log-likelihood (bnr_set_loglik; ll.base == nullptr: off).  Every recorded row r of chain c gets
  // ll.row(c, r)[i] = log N(y_i | mu_c + (X gamma_c)_i, tau2_c) of the row's own state, width n
  RowTable ll;
  // injection
  const double* inj;  // [C][inj_stride] or nullptr
  long long inj_stride;
  Aux aux;
};

__device__ __forceinline__ RngKey chain_key(const Dims& d, int c) {
  return make_key(d.seed, (uint32_t)(d.chain_offset + c));
}

}  // namespace bnr
