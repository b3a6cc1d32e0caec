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

// Streamed (mean, M2) moments of the P = V + q parameters (xi then gamma) that R-hat reads: the split-half window
// [C][2][P][2] and the per-block moments [C][nblocks][P][2] that bnr_moments_from_blocks merges into any window made of
// whole blocks (the doubling scheme's growing window without all-chain traces).  blocks == nullptr: no block moments
struct SplitMoments {
  double* halves;
  long long* window;   // device [5]: split-half window (first sweep, len), blocks (first sweep, block len, count)
  double* blocks;
  int nblocks;         // block capacity of `blocks`
  int P;
  __host__ __device__ double* half(int c, int h, int p) const { return halves + (((size_t)c * 2 + h) * P + p) * 2; }
  __host__ __device__ double* block(int c, long long b, int p) const {
    return blocks + (((size_t)c * nblocks + b) * P + p) * 2;
  }
  // Welford step of draw x of sweep `sweep` into the half window and the block that hold the sweep (if any)
  __device__ void add(int c, int p, long long sweep, double x) const {
    const long long first = window[0], len = window[1];
    const long long h = len / 2, rel = sweep - first;
    if (len > 1 && rel >= 0 && rel < len) {
      int hf = -1;
      long long cnt = 0;
      if (rel < h) { hf = 0; cnt = rel + 1; }
      else if (rel >= len - h) { hf = 1; cnt = rel - (len - h) + 1; }
      if (hf >= 0) welford(half(c, hf, p), cnt, x);
    }
    const long long bfirst = window[2], blen = window[3], bcnt = window[4];
    if (blocks && bcnt > 0 && sweep >= bfirst) {
      const long long b = (sweep - bfirst) / blen;
      if (b < bcnt && b < nblocks) welford(block(c, b, p), (sweep - bfirst) % blen + 1, x);
    }
  }
  __device__ static void welford(double* m, long long cnt, double x) {
    double mean = (cnt == 1) ? 0.0 : m[0], m2 = (cnt == 1) ? 0.0 : m[1];
    const double dl = x - mean;
    mean += dl / (double)cnt;
    m2 += dl * (x - mean);
    m[0] = mean; m[1] = m2;
  }
  // the chains from c0 on of a chain group, which keeps its own device window record
  SplitMoments view(int c0, long long* group_window) const {
    SplitMoments v = *this;
    v.halves = half(c0, 0, 0);
    if (blocks) v.blocks = block(c0, 0, 0);
    v.window = group_window;
    return v;
  }
};

// Streamed ESS accumulators (bnr_ess_stream_begin; kernels in bnr_diagnostics.cu), per chain and parameter p < P with
// y_t = x_t - x_first: ring [C][cap][P] of the last cap centred draws, head [C][L][P] the first L, acc [C][L+1][P] the
// lagged products A_l = sum_t y_t y_(t-l), sum [C][2][P] x_first and sum_t y_t.  One allocation holds the four in this
// order.  ring == nullptr: off
struct EssStream {
  double *ring_, *head_, *acc_, *sum_;
  const long long* win;   // device [2]: first sweep, draws N
  int L, cap, P;
  __host__ __device__ bool on() const { return ring_ != nullptr; }
  __host__ __device__ double* ring(int c) const { return ring_ + (size_t)c * cap * P; }
  __host__ __device__ double* head(int c) const { return head_ + (size_t)c * L * P; }
  __host__ __device__ double* acc(int c) const { return acc_ + (size_t)c * (L + 1) * P; }
  __host__ __device__ double* sum(int c) const { return sum_ + (size_t)c * 2 * P; }
  size_t doubles(int C) const { return (size_t)C * P * ((size_t)cap + L + (L + 1) + 2); }
  void carve(double* base, int C) { ring_ = base; head_ = ring(C); acc_ = head(C); sum_ = acc(C); }
  EssStream view(int c0) const {
    EssStream v = *this;
    if (on()) { v.ring_ = ring(c0); v.head_ = head(c0); v.acc_ = acc(c0); v.sum_ = sum(c0); }
    return v;
  }
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
  double* tau2_part;      // [C][2 * TAU2_MAX_BLOCKS] partial sums of the tau2 reduction
  unsigned* tau2_ticket;  // [C] arrival counters of its blocks
  int* status;      // [C]
  long long* iter;  // device scalar: completed sweeps
  long long* trace_row;   // device scalar: next trace row
  SplitMoments mom;
  EssStream ess;
  // traces of the leading tr_full.chains / tr_gx.chains chains; both keep rows = the handle's trace capacity when off
  RowTable tr_full;       // full state rows (state_var order)
  RowTable tr_gx;         // xi then gamma, width V+q
  // predictions for new networks (bnr_set_predictors; pred.base == nullptr: off).  Every recorded row r of chain c gets
  // pred.row(c, r)[j] = mu_c + X_new[j,:] gamma_c (+ sqrt(tau2_c) z_j in the predictive mode), width m; for held-out
  // rows (bnr_set_heldout, BNR_PRED_LOGDENS) log N(y_held[j] | mu_c + X_new[j,:] gamma_c, tau2_c) instead
  RowTable pred;
  const double* Xp;       // [qp][pred_mp] X_new columns padded to pred_mp rows (a multiple of 128; zeros beyond m, q)
  const double* pred_y;   // [m] held-out responses (BNR_PRED_LOGDENS only, else nullptr)
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

// The state variables in BNR_VAR_* order, which is also their order in a full trace row: tau2, u[V*R], xi[V],
// gamma[q], S[q], theta, Delta, M[R*R], mu, lambda[R], pi[R*3].  Chain c holds `count` doubles of a variable at
// (e.*at) + c * stride.
constexpr int NUM_STATE_VARS = 11;
using EngineArray = double* Engine::*;
struct StateVar {
  EngineArray at;        // the member that holds the variable
  int count;             // elements per chain
  int stride;            // doubles between chains (qp for gamma and S)
  bool transposed;       // stored [r][3], the transpose of the reference's column-major (R, 3) order (pi): pi_stored
};
__host__ __device__ inline StateVar state_var(const Dims& d, int var) {
  const int R = d.R, V = d.V;
  switch (var) {
    case 0: return {&Engine::tau2, 1, 1, false};
    case 1: return {&Engine::u, V * R, V * R, false};
    case 2: return {&Engine::xi, V, V, false};
    case 3: return {&Engine::gamma, d.q, d.qp, false};
    case 4: return {&Engine::S, d.q, d.qp, false};
    case 5: return {&Engine::theta, 1, 1, false};
    case 6: return {&Engine::Delta, 1, 1, false};
    case 7: return {&Engine::M, R * R, R * R, false};
    case 8: return {&Engine::mu, 1, 1, false};
    case 9: return {&Engine::lambda, R, R, false};
    default: return {&Engine::pi, 3 * R, 3 * R, true};
  }
}
// offset of a variable in a full trace row; state_offset(d, NUM_STATE_VARS) is the row's width
__host__ __device__ inline int state_offset(const Dims& d, int var) {
  int o = 0;
  for (int v = 0; v < var; ++v) o += state_var(d, v).count;
  return o;
}
// where element el of the reference's (R, 3) order of pi is stored in the chain's [r][3]
__host__ __device__ inline int pi_stored(int el, int R) { return 3 * (el % R) + el / R; }

__device__ __forceinline__ RngKey chain_key(const Dims& d, int c) {
  return make_key(d.seed, (uint32_t)(d.chain_offset + c));
}

}  // namespace bnr
