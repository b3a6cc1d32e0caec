// C ABI of libbnr (see include/bnr.h): handle life-cycle, the sweep schedule (one CUDA graph per sweep),
// state / trace access in reference layout, streaming R-hat, and the parity-test hooks.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include "../../include/bnr.h"
#include "bnr_engine.cuh"
#include "bnr_kernels.h"

static_assert(BNR_ST_JITTER == BNR_ST_JITTER_ && BNR_ST_SIGMA_NOTPD == BNR_ST_SIGMA_NOTPD_ &&
              BNR_ST_G_NOTPD == BNR_ST_G_NOTPD_ && BNR_ST_GIG_CAP == BNR_ST_GIG_CAP_ &&
              BNR_ST_INJ_EXHAUSTED == BNR_ST_INJ_EXHAUSTED_ && BNR_ST_NAN == BNR_ST_NAN_ &&
              BNR_ST_PSI_NOTPD == BNR_ST_PSI_NOTPD_, "status bits out of sync");
static_assert(BNR_COND_THETA == BNR_COND_THETA_ && BNR_COND_DELTA == BNR_COND_DELTA_ && BNR_COND_M == BNR_COND_M_ &&
              BNR_COND_MU == BNR_COND_MU_ && BNR_COND_LAMBDA == BNR_COND_LAMBDA_ && BNR_COND_PI == BNR_COND_PI_,
              "conditional ids out of sync");
static_assert(BNR_MAX_R == bnr::MAX_R, "MAX_R out of sync");

using namespace bnr;

static thread_local std::string g_err;
// BNR_TIMING=1: wall-clock of the fixed-cost steps (create / graph build / destroy) on stderr
static const bool g_timing = getenv("BNR_TIMING") != nullptr;
static double wall_ms() {
  return 1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
namespace bnr { thread_local long long g_launches = 0; }
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
// NVTX range over a scope (SURVEY section 5): one per conditional of the sweep where the kernels are enqueued (eager
// sweeps, bnr_step, graph capture) and one per bnr_run; free when no tool is attached
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t _e = (call);                                                                             \
    if (_e != cudaSuccess)                                                                               \
      return fail(_e == cudaErrorMemoryAllocation ? BNR_ENOMEM : BNR_ECUDA,                              \
                  std::string(#call) + ": " + cudaGetErrorString(_e));                                   \
  } while (0)

// A chain group: a contiguous slice of the handle's chains advanced by its own stream and its own two-sweep CUDA
// graph.  Groups never synchronise with each other inside bnr_run, so while one group sits in its latency-bound
// phases (Cholesky panels, triangular solves, per-chain scalar kernels: <= one CTA per chain) the other group's
// DMMA SYRK keeps the remaining SMs busy.  Results do not depend on the grouping (RNG keyed by global chain id).
struct ChainGroup {
  Engine e;                      // view of the handle's arrays restricted to chains [c0, c0 + e.d.C)
  int c0 = 0;
  cudaStream_t stream = nullptr;
  // two-sweep graphs, one per parity of the u double buffer (index 1: e.u currently points at the second buffer), so an
  // eager sweep -- an odd sweep count -- does not throw the captured graphs away
  cudaGraph_t graph[2] = {nullptr, nullptr};
  cudaGraphExec_t gexec[2] = {nullptr, nullptr};
  cudaEvent_t done = nullptr;
  ForkJoin fj;                   // side stream of the Cholesky (off-diagonal panel updates)
  double* ws = nullptr;          // split-K workspace of this group
  long long* counters = nullptr; // device [2]: iter, trace_row of this group
  long long* mom_window = nullptr;
};
constexpr int MAX_GROUPS = 8;

// ---------------------------------------------------------------------------------------------------------
// Device-memory cache.  Releasing gigabytes with cudaFree costs 30 - 300 ms (occasionally seconds) and synchronises
// the device; a handle's buffers therefore go back to a process-wide cache keyed by (device, size) when the handle
// is destroyed and are handed to the next handle that asks for the same size (the common case: Fit called again on
// the same problem, or the PSRF loop of a wrapper re-creating engines).  bnr_set_cache_limit bounds what is kept
// (default 4 GiB per process), bnr_trim_cache releases it.
// ---------------------------------------------------------------------------------------------------------
namespace {
struct CacheBlock { void* p; size_t bytes; int device; };
std::mutex g_cache_mu;
std::vector<CacheBlock> g_cache;
size_t g_cache_bytes = 0;
size_t g_cache_limit = (size_t)4 << 30;

// best fit: the smallest cached block of the device that holds `bytes` without wasting more than a quarter of itself
// (+ 1 MiB); *got receives the block's true size
void* cache_take(int device, size_t bytes, size_t* got) {
  std::lock_guard<std::mutex> lk(g_cache_mu);
  size_t best = g_cache.size();
  for (size_t i = 0; i < g_cache.size(); ++i)
    if (g_cache[i].device == device && g_cache[i].bytes >= bytes && g_cache[i].bytes <= bytes + bytes / 4 + ((size_t)1 << 20) &&
        (best == g_cache.size() || g_cache[i].bytes < g_cache[best].bytes))
      best = i;
  if (best == g_cache.size()) return nullptr;
  void* p = g_cache[best].p;
  *got = g_cache[best].bytes;
  g_cache_bytes -= g_cache[best].bytes;
  g_cache[best] = g_cache.back();
  g_cache.pop_back();
  return p;
}
void cache_give(int device, void* p, size_t bytes) {
  {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    if (g_cache_bytes + bytes <= g_cache_limit) {
      g_cache.push_back({p, bytes, device});
      g_cache_bytes += bytes;
      return;
    }
  }
  cudaFree(p);
}
}  // namespace

struct bnr_handle {
  bnr_params p;
  Engine e;
  cudaStream_t stream = nullptr;
  ChainGroup groups[MAX_GROUPS];
  int n_groups = 0;
  bool graphs_ready[2] = {false, false};
  const double* u_first = nullptr;   // e.u at creation: the parity of the double buffer is (e.u != u_first)
  cudaEvent_t ev_fork = nullptr;
  ForkJoin fj;                   // side stream for eager sweeps on the whole chain set
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<std::pair<void*, size_t>> allocs;   // device buffers (pointer, bytes): returned to the cache on destroy
  double* ws = nullptr;          // split-K workspace
  double* d_inj = nullptr;       // injected variates
  long long inj_len = 0;
  bool aux_on = false;
  Aux aux_saved = {};
  long long win[5] = {0, 0, 0, 1, 0};   // host copy of the device window record (bnr_set_moment_window / _blocks)
  long long blk_len = 0;
  long long mom_half = 0;        // draws per split chain behind the current moments buffer
  long long launches = 0;        // kernels launched by bnr_run so far (graph replays included)
  long long graph_kernels = 0;   // kernels inside the captured two-sweep graphs (all groups)
  bool xg_valid = false;         // e.xg == X * gamma for the current state
  bool ran = false;
  double* d_rhat = nullptr;      // [V+q]
  double* d_tmp = nullptr;       // staging for get/set (max var size / trace chunk)
  size_t tmp_doubles = 0;
  // ESS statistics of the last bnr_ess_accumulate
  double* d_acov = nullptr;      // [max_lag + 1][V + q]  sum over local chains of the biased autocovariances
  double* d_cmean = nullptr;     // [C][V + q]
  int ess_lag = -1;
  long long ess_rows = 0;
  size_t acov_cap = 0;
  // streaming ESS (bnr_ess_stream_begin / _finish)
  long long* d_esswin = nullptr; // device [4]
  double* ess_stream_buf = nullptr;  // ring | head | lagged products | sums, reused across begin calls
  size_t ess_stream_cap = 0;     // its capacity in doubles
  long long ess_stream_N = 0;    // > 0 while a streaming window is armed
};

static int raw_alloc(bnr_handle* h, void** out, size_t bytes) {
  size_t got = bytes;
  void* p = cache_take(h->p.device, bytes, &got);
  if (!p) { CK(cudaMalloc(&p, bytes)); got = bytes; }
  h->allocs.push_back({p, got});
  *out = p;
  return 0;
}

// hand a buffer that a larger one supersedes back to the cache (instead of keeping it until bnr_destroy)
static void release_alloc(bnr_handle* h, void* p) {
  if (!p) return;
  for (size_t i = 0; i < h->allocs.size(); ++i)
    if (h->allocs[i].first == p) {
      cache_give(h->p.device, p, h->allocs[i].second);
      h->allocs[i] = h->allocs.back();
      h->allocs.pop_back();
      return;
    }
}

// short-lived device scratch of the handle-less entry points (bnr_rhat_from_moments, bnr_ess_from_stats): taken from
// and returned to the process-wide cache, so the steady state performs no cudaMalloc / cudaFree
struct Scratch {
  int device; void* p = nullptr; size_t bytes = 0;
  Scratch(int dev, size_t b) : device(dev), bytes((b + 255) / 256 * 256) {
    size_t got = bytes;
    p = cache_take(device, bytes, &got);
    if (p) bytes = got;
    else if (cudaMalloc(&p, bytes) != cudaSuccess) p = nullptr;
  }
  ~Scratch() { if (p) cache_give(device, p, bytes); }
};

template <typename T>
static int dalloc(bnr_handle* h, T** ptr, size_t count, bool zero = true) {
  void* p = nullptr;
  const size_t bytes = count * sizeof(T) + 16;
  int r = raw_alloc(h, &p, bytes);
  if (r) return r;
  if (zero) CK(cudaMemsetAsync(p, 0, bytes, h->stream));
  *ptr = (T*)p;
  return 0;
}
// the buffer of a row table whose shape is set; nan_fill: rows never written read as NaN.  A refusal names the table and
// its size and is cleared, so that it does not surface in a later call
static int alloc_table(bnr_handle* h, RowTable& t, bool nan_fill, const char* what) {
  if (int r = dalloc(h, &t.base, t.doubles(), false)) {
    cudaGetLastError();
    return fail(r, std::string(what) + " (" + std::to_string(8.0 * (double)t.doubles()) + " bytes): " + g_err);
  }
  if (nan_fill) CK(cudaMemsetAsync(t.base, 0xff, sizeof(double) * t.doubles(), h->stream));
  return BNR_OK;
}
#define DA(ptr, count)                          \
  do {                                          \
    int _r = dalloc(h, &(ptr), (count));        \
    if (_r) return _r;                          \
  } while (0)

extern "C" int bnr_version(void) { return BNR_VERSION; }
extern "C" const char* bnr_last_error(void) { return g_err.c_str(); }

extern "C" void bnr_default_params(bnr_params* p) {
  memset(p, 0, sizeof(*p));
  p->num_chains = 2;
  p->eta = 1.01; p->zeta = 1.0; p->iota = 1.0; p->a_delta = 1.0; p->b_delta = 1.0; p->nu = 10.0;
  p->trace_full_chains = 1; p->trace_gamma_xi_all = 1; p->gig_inject_len = 64;
}

static int var_size(const Dims& d, int var) {
  switch (var) {
    case BNR_VAR_TAU2: case BNR_VAR_THETA: case BNR_VAR_DELTA: case BNR_VAR_MU: return 1;
    case BNR_VAR_U: return d.R * d.V;
    case BNR_VAR_XI: return d.V;
    case BNR_VAR_GAMMA: case BNR_VAR_S: return d.q;
    case BNR_VAR_M: return d.R * d.R;
    case BNR_VAR_LAMBDA: return d.R;
    case BNR_VAR_PI: return 3 * d.R;
  }
  return -1;
}
// offset of a variable inside a full trace row (k_record / state_elem order)
static int row_offset(const Dims& d, int var) {
  const int R = d.R, V = d.V, q = d.q;
  const int o[BNR_NUM_VARS] = {0, 1, 1 + V * R, 1 + V * R + V, 1 + V * R + V + q, 1 + V * R + V + 2 * q,
                               2 + V * R + V + 2 * q, 3 + V * R + V + 2 * q, 3 + V * R + V + 2 * q + R * R,
                               4 + V * R + V + 2 * q + R * R, 4 + V * R + V + 2 * q + R * R + R};
  return o[var];
}

// the two branch streams of a stream (side at priority side_prio, side_hi at hi_prio), their fork / join events and the
// event pool of the Cholesky's look-ahead schedule: 4 per panel (launch_cholesky)
static int create_fork_join(ForkJoin& f, int panels, int side_prio, int hi_prio) {
  CK(cudaStreamCreateWithPriority(&f.side, cudaStreamNonBlocking, side_prio));
  CK(cudaStreamCreateWithPriority(&f.side_hi, cudaStreamNonBlocking, hi_prio));
  CK(cudaEventCreateWithFlags(&f.fork, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&f.join, cudaEventDisableTiming));
  f.npool = 4 * panels;
  f.pool = new cudaEvent_t[f.npool]();
  for (int i = 0; i < f.npool; ++i) CK(cudaEventCreateWithFlags(&f.pool[i], cudaEventDisableTiming));
  return BNR_OK;
}

// (also after a create_fork_join that failed part of the way)
static void destroy_fork_join(ForkJoin& f) {
  if (f.side) cudaStreamDestroy(f.side);
  if (f.side_hi) cudaStreamDestroy(f.side_hi);
  if (f.fork) cudaEventDestroy(f.fork);
  if (f.join) cudaEventDestroy(f.join);
  for (int i = 0; i < f.npool && f.pool; ++i)
    if (f.pool[i]) cudaEventDestroy(f.pool[i]);
  delete[] f.pool;
  f = ForkJoin();
}

static int create_impl(bnr_handle* h, const bnr_params* p, const double* X, const double* y);

extern "C" int bnr_create(const bnr_params* p, const double* X, const double* y, bnr_handle** out) {
  if (!p || !X || !y || !out) return fail(BNR_EINVAL, "null argument");
  if (p->n < 1 || p->V < 2 || p->R < 1 || p->R > BNR_MAX_R || p->num_chains < 1)
    return fail(BNR_EINVAL, "need n >= 1, V >= 2, 1 <= R <= 16, num_chains >= 1");
  if (!(p->nu > p->R - 1)) return fail(BNR_EINVAL, "nu must exceed R - 1 (InverseWishart degrees of freedom)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(BNR_ENODEV, "no CUDA device visible: libbnr has no CPU fallback");
  if (p->device < 0 || p->device >= ndev) return fail(BNR_EINVAL, "device ordinal out of range");
  CK(cudaSetDevice(p->device));
  int cc_major = 0;      // (cudaGetDeviceProperties takes anything from 1 to 120 ms; one attribute is all that is needed)
  CK(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, p->device));
  if (cc_major < 10) return fail(BNR_ENODEV, "libbnr is built for sm_100a (B200) only");

  bnr_handle* h = new bnr_handle();
  h->p = *p;
  const double t0 = wall_ms();
  const int rc = create_impl(h, p, X, y);
  if (g_timing) fprintf(stderr, "[bnr] bnr_create %.2f ms (%zu device buffers)\n", wall_ms() - t0, h->allocs.size());
  if (rc != BNR_OK) {
    const std::string msg = g_err;      // bnr_destroy must not clobber the reason
    bnr_destroy(h);
    g_err = msg;
    return rc;
  }
  *out = h;
  return BNR_OK;
}

// everything of bnr_create that can fail after the handle exists (the caller destroys the handle on failure)
static int create_impl(bnr_handle* h, const bnr_params* p, const double* X, const double* y) {
  if (h->p.gig_inject_len <= 0) h->p.gig_inject_len = 64;
  Dims& d = h->e.d;
  d.n = p->n; d.V = p->V; d.R = p->R; d.C = p->num_chains; d.C_total = p->num_chains;
  d.q = p->V * (p->V + 1) / 2;
  // n is padded to a multiple of 128 with AT LEAST one padding row: row n of the n x n system carries the right-hand
  // side of the forward solve through the factorisation (bnr_linalg.cu); same for q in the q-form
  d.np = (p->n + 1 + TILE_N - 1) / TILE_N * TILE_N;
  d.qp = (d.q + TILE_K - 1) / TILE_K * TILE_K;
  // gamma draw formulation (SURVEY 8d cost model): the q x q precision form costs q^3/3 + 4q^2 flops per
  // chain-iteration, the n x n Bhattacharya form (what the reference runs, src/gibbs.jl:429-436) n^2 q + n^3/3.
  // AUTO: the rule of the 8192 limit (q-form iff cheaper and qp128 <= 8192) wherever its choice has a factored dimension
  // <= 8192, so that no shape accepted then changes form; beyond, the cheaper of the forms that fit chol_max_dim().
  {
    const double qd = d.q, nd = d.n;
    const double cost_q = qd * qd * qd / 3.0 + 4.0 * qd * qd, cost_n = nd * nd * qd + nd * nd * nd / 3.0;
    const int qp128 = (d.q + 1 + TILE_N - 1) / TILE_N * TILE_N;
    const int small = bwd_stream_max_dim(), large = chol_max_dim();
    int mode = p->gamma_mode;
    if (mode != BNR_GAMMA_NFORM && mode != BNR_GAMMA_QFORM) {
      mode = (cost_q < cost_n && qp128 <= small) ? BNR_GAMMA_QFORM : BNR_GAMMA_NFORM;
      if ((mode == BNR_GAMMA_QFORM ? qp128 : d.np) > small) {
        const bool q_fits = qp128 <= large, n_fits = d.np <= large;
        mode = (q_fits && (cost_q < cost_n || !n_fits)) ? BNR_GAMMA_QFORM : BNR_GAMMA_NFORM;
      }
    }
    d.gmode = mode;
    if (mode == BNR_GAMMA_QFORM) d.qp = qp128;       // q-padded vectors double as right-hand sides of the q x q solve
    d.gdim = mode == BNR_GAMMA_QFORM ? d.qp : d.np;
  }
  d.nparts = (d.q + PART_BLOCK - 1) / PART_BLOCK;
  d.chain_offset = p->chain_offset;
  d.chain_offset_local = 0;
  d.gigK = h->p.gig_inject_len;
  d.seed = p->seed;
  d.eta = p->eta; d.zeta = p->zeta; d.iota = p->iota; d.a_delta = p->a_delta; d.b_delta = p->b_delta; d.nu = p->nu;
  // dynamic shared memory of the per-chain kernels grows with V*R
  const size_t need = sizeof(double) * ((size_t)d.V * d.R + 2 * d.R * d.R + 2 + 4 * (2 * d.V + 2 * d.R * d.R + 3 * d.R));
  if (need > 200 * 1024 || d.gdim > chol_max_dim()) {
    return fail(BNR_EINVAL, "problem too large for the per-chain shared-memory kernels (V*R > 200 KB of shared memory, or factored dimension > 32768: n <= 32767 in the n-form, V <= 255 in the q-form)");
  }
  CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CK(cudaEventCreate(&h->ev0));
  CK(cudaEventCreate(&h->ev1));
  linalg_setup();
  {
    // above 8192 the back solve is one cluster of 8 CTAs (~210 KB of shared memory each) per chain
    const int clusters = bwd_cluster_capacity(d.gdim);
    if (clusters < 0) return fail(BNR_ECUDA, "cudaOccupancyMaxActiveClusters failed for the cluster back solve");
    if (clusters == 0)
      return fail(BNR_ECUDA, "this device cannot co-schedule the back solve's cluster of 8 CTAs with ~210 KB of shared memory each (factored dimension > 8192)");
  }
  if (!tmap_setup()) return fail(BNR_ECUDA, "cuTensorMapEncodeTiled is not available from this driver (TMA tensor maps are required)");
  small_kernels_setup();

  Engine& e = h->e;
  const size_t C = d.C;
  const double t_create0 = wall_ms();
  double *dX, *dy;
  DA(dX, (size_t)d.qp * d.np);
  DA(dy, (size_t)d.np);
  // X: column-major n x q host -> padded columns of np rows
  CK(cudaMemcpy2DAsync(dX, (size_t)d.np * sizeof(double), X, (size_t)d.n * sizeof(double),
                       (size_t)d.n * sizeof(double), (size_t)d.q, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(dy, y, (size_t)d.n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  e.X = dX; e.y = dy;
  if (g_timing) { cudaStreamSynchronize(h->stream); fprintf(stderr, "[bnr]   X, y upload done at +%.2f ms\n", wall_ms() - t_create0); }
  std::vector<int2> lk(d.q);
  {
    int j = 0;
    for (int k = 0; k < d.V; ++k)
      for (int l = k; l < d.V; ++l) lk[j++] = make_int2(l, k);
  }
  int2* dlk;
  DA(dlk, (size_t)d.q);
  CK(cudaMemcpyAsync(dlk, lk.data(), sizeof(int2) * d.q, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  e.edge_lk = dlk;

  DA(e.tau2, C); DA(e.u, C * d.V * d.R); DA(e.u_alt, C * d.V * d.R); DA(e.xi, C * d.V);
  h->u_first = e.u;
  DA(e.gamma, C * d.qp); DA(e.S, C * d.qp); DA(e.theta, C); DA(e.Delta, C); DA(e.M, C * d.R * d.R);
  DA(e.mu, C); DA(e.lambda, C * d.R); DA(e.pi, C * 3 * d.R);
  DA(e.W, C * d.qp); DA(e.v, C * d.qp); DA(e.t, C * d.qp);
  DA(e.xg, C * d.np); DA(e.xv, C * d.np); DA(e.rhs, C * d.np);
  DA(e.G, C * d.gdim * d.gdim + 2048);
  DA(e.Linv, C * (size_t)(d.gdim / TILE_N) * TILE_N * TILE_N);
  // the blocks above the diagonal of every inverted panel are exact zeros that k_potf2_inv never writes
  CK(cudaMemsetAsync(e.Linv, 0, sizeof(double) * C * (size_t)(d.gdim / TILE_N) * TILE_N * TILE_N, h->stream));
  e.syrk_ws = nullptr; e.syrk_ws_cap = 0;
  e.gram_planes = nullptr; e.gram_rscale = nullptr;
  if (gram_i8_selected(d)) {
    DA(e.gram_planes, C * gram_i8_plane_bytes(d));
    DA(e.gram_rscale, C * d.np);
  } else if (d.gmode == BNR_GAMMA_NFORM) {
    // few chains x tiles: the SYRK splits its contraction (see launch_syrk_G).  The split count is fixed per handle
    // from its total chain count, so the chain grouping never changes the summation order.
    const int smax = syrk_splits(d, d.C);
    if (smax > 1) {
      e.syrk_ws_cap = smax - 1;
      DA(e.syrk_ws, C * (size_t)e.syrk_ws_cap * d.gdim * d.gdim);
    }
  }
  e.XtX = nullptr;
  if (d.gmode == BNR_GAMMA_QFORM) {
    // X'X once: row-major copy of X as the SYRK operand (k-major over the n samples), unit scales, no identity
    std::vector<double> xt((size_t)d.np * d.qp, 0.0), ones((size_t)d.np, 1.0);
    for (int j = 0; j < d.q; ++j)
      for (int i = 0; i < d.n; ++i) xt[(size_t)i * d.qp + j] = X[(size_t)i + (size_t)d.n * j];
    double *dXT = nullptr, *dOnes = nullptr, *dXtX = nullptr;
    DA(dXT, xt.size());              // (tracked by the handle: released below, or by bnr_destroy on a failure path)
    DA(dOnes, ones.size());
    DA(dXtX, (size_t)d.qp * d.qp);
    CK(cudaMemcpyAsync(dXT, xt.data(), xt.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(dOnes, ones.data(), ones.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    launch_xtx(d, dXT, dOnes, dXtX, h->stream);
    CK(cudaStreamSynchronize(h->stream));
    release_alloc(h, dXT);
    release_alloc(h, dOnes);
    e.XtX = dXtX;
  }
  DA(e.partials, C * d.nparts * (2 * MAX_R + 1));
  DA(e.tau2_part, C * 2 * TAU2_MAX_BLOCKS);
  DA(e.tau2_ticket, C);
  DA(e.status, C);
  DA(e.iter, 1); DA(e.trace_row, 1);
  DA(e.moments, C * 2 * (d.V + d.q) * 2);
  DA(e.mom_window, 5);
  e.bmom = nullptr; e.bmom_nb = 0;
  e.ess_ring = e.ess_head = e.ess_acc = e.ess_sum = nullptr; e.ess_win = nullptr; e.ess_L = e.ess_cap = 0;
  DA(h->d_esswin, 4);
  DA(h->ws, x_times_workspace_doubles(d));
  DA(h->d_rhat, (size_t)(d.V + d.q));
  const long long trace_rows = p->trace_rows > 0 ? p->trace_rows : 0;
  e.tr_full = {nullptr, trace_rows, 4 + d.V * d.R + d.V + 2 * d.q + d.R * d.R + d.R + 3 * d.R, 0};
  e.tr_gx = {nullptr, trace_rows, d.V + d.q, 0};
  if (trace_rows > 0) {
    e.tr_full.chains = p->trace_full_chains < 0 ? 0 : (p->trace_full_chains < d.C ? p->trace_full_chains : d.C);
    if (p->trace_gamma_xi_all) e.tr_gx.chains = d.C;
    else if (p->trace_gamma_xi_chains > 0) e.tr_gx.chains = p->trace_gamma_xi_chains < d.C ? p->trace_gamma_xi_chains : d.C;
  }
  // traces are not NaN-filled: a memset of a multi-GB trace would cost time at every create
  if (e.tr_full.chains > 0) if (int r = alloc_table(h, e.tr_full, false, "full-state trace")) return r;
  if (e.tr_gx.chains > 0) if (int r = alloc_table(h, e.tr_gx, false, "gamma/xi trace")) return r;
  {
    // chain groups (see ChainGroup): 2 by default once there are enough chains to split
    // default: 2 groups once the SYRK of half the chains fills the GPU for several waves; 4 when the chains are few
    // (then the per-group latency chain, not the tensor pipe, bounds the sweep and more of them must overlap)
    // measured on B200 (round 2, 100-sweep runs): 64 chains of config 3 with 2 / 3 / 4 / 6 / 8 groups -> 10.94 / 10.97 /
    // 11.02 / 11.17 / 11.29 ms per sweep; 32 chains: 2 / 3 / 4 -> 5.87 / 5.86 / 5.96 ms; 8 chains: 2 / 4 / 8 -> 2.02 /
    // 1.95 / 2.16 ms; config 4 (8 chains, split-K SYRK: every group's SYRK fills the GPU by itself): 2 / 4 -> 1.69 / 1.84
    // later in round 2 (look-ahead panel kernel): 8 chains of config 3 with 2 / 3 / 4 / 8 groups -> 1.86 / 1.79 / 1.85 /
    // 2.05 ms (three uneven groups of 2-3 chains: two concurrent SYRKs then leave ~40 SMs to the third group's panel
    // chain instead of 4), 16 chains: 2 / 3 / 4 / 8 -> 3.20 / 3.11 / 3.12 / 3.26; config 2 (q-form, no SYRK in the
    // sweep, pure latency chain): 1 / 2 / 4 / 8 -> 0.340 / 0.342 / 0.344 / 0.350
    // with the forked Cholesky updates at the panel chain's priority: 64 chains 2 / 3 / 4 / 5 / 6 groups -> 10.89 / 10.74 /
    // 10.80 / 10.89 / 10.95 ms; 32 chains 2 / 3 -> 5.76 / 5.52; config 5 (128 chains) 2 / 3 -> 1.80 / 1.77
    int ng_auto = d.C >= 6 ? 3 : (d.C >= 4 ? 4 : (d.C >= 2 ? 2 : 1));
    if (d.gmode == BNR_GAMMA_NFORM && d.C >= 4 && syrk_splits(d, d.C) > 1) ng_auto = 2;
    if (d.gmode == BNR_GAMMA_QFORM && d.C >= 2 && d.C < 24) ng_auto = 2;
    // INT8 Gram path: below 12 chains one group keeps the SMs busiest (measured on B200 at 1000 W, config 3, 100-sweep
    // runs: 8 chains 1 / 2 / 3 groups -> 1.36 / 1.44 / 1.41 ms; 12 chains -> 1.76 / 1.70 / 1.70 ms)
    if (gram_i8_selected(d) && d.C < 12) ng_auto = 1;
    int ng = p->chain_groups > 0 ? p->chain_groups : ng_auto;
    if (ng > MAX_GROUPS) ng = MAX_GROUPS;
    if (ng > d.C) ng = d.C;
    h->n_groups = ng;
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    const int panels = d.gdim / TILE_N;
    // eager sweeps on the whole chain set: both branches at the default priority
    if (int r = create_fork_join(h->fj, panels, 0, 0)) return r;
    // main stream: greatest priority (latency-bound kernels); side stream: least (SYRK, bulk panel updates)
    int plo = 0, phi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&plo, &phi));       // plo = least, phi = greatest (numerically lower)
    for (int g = 0; g < ng; ++g) {
      ChainGroup& G = h->groups[g];
      CK(cudaStreamCreateWithPriority(&G.stream, cudaStreamNonBlocking, phi));
      CK(cudaEventCreateWithFlags(&G.done, cudaEventDisableTiming));
      // look-ahead branch of the Cholesky: the priority of the main stream (one level lower was measured: config 3 at
      // 8 chains 1.77 -> 1.81 ms, nothing gained elsewhere)
      if (int r = create_fork_join(G.fj, panels, plo, phi)) return r;
      DA(G.ws, x_times_workspace_doubles(d));
      DA(G.counters, 2);
      DA(G.mom_window, 5);
    }
  }
  if (g_timing) { cudaStreamSynchronize(h->stream); fprintf(stderr, "[bnr]   buffers, streams, events at +%.2f ms\n", wall_ms() - t_create0); }
  h->tmp_doubles = (size_t)1 << 22;
  DA(h->d_tmp, h->tmp_doubles);
  e.inj = nullptr; e.inj_stride = 0;
  memset(&e.aux, 0, sizeof(e.aux));
  CK(cudaStreamSynchronize(h->stream));
  if (!tmaps_check(e)) return fail(BNR_ECUDA, "cuTensorMapEncodeTiled refused a tensor map of this problem's geometry");
  return BNR_OK;
}

static void drop_graph(bnr_handle* h);

extern "C" int bnr_trim_cache(void) {
  std::vector<CacheBlock> blocks;
  {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    blocks.swap(g_cache);
    g_cache_bytes = 0;
  }
  int cur = 0;
  cudaGetDevice(&cur);
  for (auto& b : blocks) { cudaSetDevice(b.device); cudaFree(b.p); }
  cudaSetDevice(cur);
  return BNR_OK;
}

extern "C" int bnr_set_cache_limit(int64_t bytes) {
  if (bytes < 0) return fail(BNR_EINVAL, "negative limit");
  { std::lock_guard<std::mutex> lk(g_cache_mu); g_cache_limit = (size_t)bytes; }
  if (bytes == 0) return bnr_trim_cache();
  return BNR_OK;
}

extern "C" int bnr_destroy(bnr_handle* h) {
  if (!h) return BNR_OK;
  const double t_destroy0 = wall_ms();
  cudaSetDevice(h->p.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  drop_graph(h);
  for (int g = 0; g < h->n_groups; ++g) {
    if (h->groups[g].stream) { cudaStreamSynchronize(h->groups[g].stream); cudaStreamDestroy(h->groups[g].stream); }
    if (h->groups[g].done) cudaEventDestroy(h->groups[g].done);
    destroy_fork_join(h->groups[g].fj);
  }
  destroy_fork_join(h->fj);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  for (auto& a : h->allocs) cache_give(h->p.device, a.first, a.second);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  if (g_timing) fprintf(stderr, "[bnr] bnr_destroy %.2f ms\n", wall_ms() - t_destroy0);
  return BNR_OK;
}

static void drop_graph(bnr_handle* h) {
  for (int g = 0; g < h->n_groups; ++g) {
    ChainGroup& G = h->groups[g];
    for (int par = 0; par < 2; ++par) {
      if (G.gexec[par]) { cudaGraphExecDestroy(G.gexec[par]); G.gexec[par] = nullptr; }
      if (G.graph[par]) { cudaGraphDestroy(G.graph[par]); G.graph[par] = nullptr; }
    }
  }
  h->graphs_ready[0] = h->graphs_ready[1] = false;
}

// X * gamma for the current state (cache used by tau2 and mu)
static void refresh_xg(bnr_handle* h) {
  launch_x_times(h->e, 0, h->e.gamma, h->e.xg, h->ws, h->stream);
  h->xg_valid = true;
}

// phase boundary k of a profiled sweep (bnr_profile_sweep: marks holds its 9 events); nothing in any other sweep
static void mark(cudaEvent_t* marks, int k, cudaStream_t s) {
  if (marks) cudaEventRecord(marks[k], s);
}

// the gamma conditional: W, v, X v, rhs, G, Cholesky, solves, X' a4, gamma (and optionally S + lambda statistics).
// syrk_forked: G = X D X' + I is already running on fj.side (enqueue_sweep forks it at the start of the sweep: it
// depends on nothing but last sweep's S); wait for it just before the factorisation.
static void run_gamma(Engine& e, double* ws, const ForkJoin& fj, cudaStream_t s, int gig_flags, bool syrk_forked = false,
                      cudaEvent_t* marks = nullptr) {
  if (e.d.gmode == BNR_GAMMA_QFORM) {
    // P = (X'X + D^-1)/tau2 = L L';  L w = X'(y - mu - X W)/tau2;  L' beta = w + z;  gamma = W + beta
    launch_edge_prep(e, 2, s);                        // W, v = z
    launch_x_times(e, 0, e.W, e.xv, ws, s);           // X W
    launch_rhs(e, s);                                 // (y - mu - X W)/tau2
    launch_x_times(e, 1, e.rhs, e.t, ws, s);          // t = X' rhs
    mark(marks, 3, s);
    launch_build_P(e, s);
    mark(marks, 4, s);
    launch_cholesky(e, e.t, fj, s);
    mark(marks, 5, s);
    launch_chol_solve(e, e.t, e.v, s);
    mark(marks, 6, s);
    launch_gamma_gig(e, (gig_flags & ~1) | ((gig_flags & 1) ? 4 : 0), s);
    return;
  }
  launch_edge_prep(e, 1, s);
  launch_x_times(e, 0, e.v, e.xv, ws, s);
  launch_rhs(e, s);
  mark(marks, 3, s);
  if (syrk_forked) cudaStreamWaitEvent(s, fj.join, 0);
  else launch_syrk_G(e, s);
  mark(marks, 4, s);
  launch_cholesky(e, e.rhs, fj, s);
  mark(marks, 5, s);
  launch_chol_solve(e, e.rhs, nullptr, s);
  mark(marks, 6, s);
  launch_x_times(e, 1, e.rhs, e.t, ws, s);
  launch_gamma_gig(e, gig_flags, s);
}

// the record block of the initial state (row 0) or of a finished sweep (sweep_done: also the streamed ESS lags): the
// trace rows, the prediction row, the log-likelihood row, then the row / iteration counters.  pred_forked: X_new gamma
// already runs on fj.side (join it), else it is launched here.  xg_stale: e.xg does not hold X gamma of the state, which
// the log-likelihood row reads.
static void enqueue_record(Engine& e, double* ws, const ForkJoin& fj, cudaStream_t s, bool sweep_done, bool pred_forked,
                           bool xg_stale) {
  launch_record(e, sweep_done, s);
  if (sweep_done && e.ess_ring) launch_ess_stream(e, s);
  if (e.pred.base) {
    if (pred_forked) cudaStreamWaitEvent(s, fj.join, 0);
    else launch_pred_product(e, s);
    launch_pred_record(e, sweep_done, s);
  }
  if (e.ll.base) {
    if (xg_stale) launch_x_times(e, 0, e.gamma, e.xg, ws, s);
    launch_loglik_record(e, s);
  }
  launch_advance(e, sweep_done, s);
}

// one full sweep in gibbs_sample! order (src/gibbs.jl:663-677).  The Gram SYRK (81 % of the sweep, pure throughput
// work) goes to the low-priority side stream right away; the latency-bound kernels stay on the high-priority main
// stream, so that they -- of this chain group and of the others -- get an SM as soon as any SYRK CTA retires instead
// of queueing behind the SYRK's remaining CTAs.
// marks (bnr_profile_sweep): events recorded at the 8 phase boundaries; the Gram SYRK and X_new gamma then run on s,
// so that each phase's events bracket its own kernels.
static void enqueue_sweep(Engine& e, double* ws, const ForkJoin& fj, cudaStream_t s, cudaEvent_t* marks = nullptr) {
  NvtxRange sweep("bnr sweep");
  mark(marks, 0, s);
  const bool fork_syrk = !marks && e.d.gmode == BNR_GAMMA_NFORM && !e.aux.G_copy;
  if (fork_syrk) {
    NvtxRange r("gamma: G = X D X' + I (forked)");
    cudaEventRecord(fj.fork, s);
    cudaStreamWaitEvent(fj.side, fj.fork, 0);
    launch_syrk_G(e, fj.side);
    cudaEventRecord(fj.join, fj.side);
  }
  { NvtxRange r("tau2"); launch_tau2(e, s); }
  mark(marks, 1, s);
  { NvtxRange r("u, xi"); launch_uxi(e, s); }
  std::swap(e.u, e.u_alt);          // u now holds the new draw (pointer swap is baked per captured sweep)
  mark(marks, 2, s);
  { NvtxRange r("gamma + D (GIG)"); run_gamma(e, ws, fj, s, 3, fork_syrk, marks); }
  mark(marks, 7, s);
  // predictions for new networks: X_new gamma depends on gamma only, so it runs on the side stream next to the scalar
  // conditionals and joins before k_pred_record, which needs the new mu (and tau2)
  const bool fork_pred = !marks && e.pred.base;
  if (fork_pred) {
    NvtxRange r("predictions: X_new gamma");
    cudaEventRecord(fj.fork, s);
    cudaStreamWaitEvent(fj.side, fj.fork, 0);
    launch_pred_product(e, fj.side);
    cudaEventRecord(fj.join, fj.side);
  }
  {
    NvtxRange r("theta, Delta, M, mu, Lambda, pi");
    launch_x_times(e, 0, e.gamma, e.xg, ws, s);
    launch_finish(e, (1 << BNR_COND_THETA) | (1 << BNR_COND_DELTA) | (1 << BNR_COND_M) | (1 << BNR_COND_MU) |
                         (1 << BNR_COND_LAMBDA) | (1 << BNR_COND_PI), s);
  }
  NvtxRange r("record");
  enqueue_record(e, ws, fj, s, true, fork_pred, false);
  mark(marks, 8, s);
}

// view of the handle's engine restricted to chains [c0, c0 + Cg): every per-chain array is chain-major, so the
// view is the same struct with offset pointers, a smaller C and a shifted global chain id
static Engine group_view(const bnr_handle* h, int c0, int Cg, long long* counters, long long* mom_window) {
  Engine v = h->e;
  const Dims& d = h->e.d;
  const size_t c = (size_t)c0;
  v.d.C = Cg;
  v.d.chain_offset = d.chain_offset + c0;
  v.d.chain_offset_local = c0;
  v.tau2 += c; v.theta += c; v.Delta += c; v.mu += c; v.status += c;
  v.u += c * d.V * d.R; v.u_alt += c * d.V * d.R; v.xi += c * d.V;
  v.gamma += c * d.qp; v.S += c * d.qp; v.W += c * d.qp; v.v += c * d.qp; v.t += c * d.qp;
  v.M += c * d.R * d.R; v.lambda += c * d.R; v.pi += c * 3 * d.R;
  v.xg += c * d.np; v.xv += c * d.np; v.rhs += c * d.np;
  v.G += c * d.gdim * d.gdim; if (v.syrk_ws) v.syrk_ws += c * (size_t)v.syrk_ws_cap * d.gdim * d.gdim; v.Linv += c * (size_t)(d.gdim / TILE_N) * TILE_N * TILE_N;
  if (v.gram_planes) { v.gram_planes += c * gram_i8_plane_bytes(d); v.gram_rscale += c * d.np; }
  v.partials += c * d.nparts * (2 * MAX_R + 1);
  v.moments += c * 2 * (d.V + d.q) * 2;
  if (v.bmom) v.bmom += c * (size_t)v.bmom_nb * (d.V + d.q) * 2;
  if (v.ess_ring) {
    const size_t P = (size_t)d.V + d.q;
    v.ess_ring += c * (size_t)v.ess_cap * P; v.ess_head += c * (size_t)v.ess_L * P;
    v.ess_acc += c * (size_t)(v.ess_L + 1) * P; v.ess_sum += c * 2 * P;
  }
  v.tr_full = v.tr_full.view(c0, Cg); v.tr_gx = v.tr_gx.view(c0, Cg);
  v.pred = v.pred.view(c0, Cg); v.ll = v.ll.view(c0, Cg);
  if (v.pred_ws) v.pred_ws += c * (size_t)v.pred_splits * v.pred_mp;
  v.iter = counters; v.trace_row = counters + 1; v.mom_window = mom_window;
  v.inj = nullptr; v.inj_stride = 0;
  memset(&v.aux, 0, sizeof(v.aux));
  return v;
}

// The u double buffer flips every sweep, so every group's graph holds TWO sweeps; odd counts run one sweep eagerly
// on the whole chain set.
static int build_graphs(bnr_handle* h) {
  const int par = (h->e.u != h->u_first) ? 1 : 0;
  if (h->graphs_ready[par]) return BNR_OK;
  const double t0 = wall_ms();
  const long long before = g_launches;
  const int C = h->e.d.C, ng = h->n_groups;
  for (int g = 0; g < ng; ++g) {
    ChainGroup& G = h->groups[g];
    const int c0 = (int)((long long)C * g / ng), c1 = (int)((long long)C * (g + 1) / ng);
    G.c0 = c0;
    G.e = group_view(h, c0, c1 - c0, G.counters, G.mom_window);
    Engine e = G.e;                  // the capture swaps u / u_alt twice on this copy
    CK(cudaStreamBeginCapture(G.stream, cudaStreamCaptureModeThreadLocal));
    enqueue_sweep(e, G.ws, G.fj, G.stream);
    enqueue_sweep(e, G.ws, G.fj, G.stream);
    CK(cudaStreamEndCapture(G.stream, &G.graph[par]));
    // node priorities = priorities of the streams the kernels were captured from (main: greatest, side: least)
    CK(cudaGraphInstantiate(&G.gexec[par], G.graph[par], cudaGraphInstantiateFlagUseNodePriority));
  }
  h->graph_kernels = g_launches - before;
  h->graphs_ready[par] = true;
  if (g_timing) fprintf(stderr, "[bnr] graph capture + instantiate (%d groups, %lld kernels) %.2f ms\n", ng, h->graph_kernels, wall_ms() - t0);
  return BNR_OK;
}

extern "C" int bnr_init_state(bnr_handle* h) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  CK(cudaMemsetAsync(e.iter, 0, sizeof(long long), h->stream));
  CK(cudaMemsetAsync(e.trace_row, 0, sizeof(long long), h->stream));
  CK(cudaMemsetAsync(e.status, 0, sizeof(int) * e.d.C, h->stream));
  launch_init(e, h->stream);
  enqueue_record(e, h->ws, h->fj, h->stream, false, false, true);     // X gamma_0: the cache is not valid after launch_init
  h->xg_valid = false;
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

extern "C" int bnr_run(bnr_handle* h, int64_t n_iters) {
  if (!h || n_iters < 0) return fail(BNR_EINVAL, "bad arguments");
  NvtxRange range("bnr_run");
  CK(cudaSetDevice(h->p.device));
  CK(cudaEventRecord(h->ev0, h->stream));
  if (!h->xg_valid) { const long long b0 = g_launches; refresh_xg(h); h->launches += g_launches - b0; }
  int64_t left = n_iters;
  if (h->e.inj == nullptr && !h->aux_on && left >= 2) {
    int r = build_graphs(h);
    if (r) return r;
    const int par = (h->e.u != h->u_first) ? 1 : 0;
    // fork: every group starts from the handle's counters and runs its sweeps without ever meeting the others
    CK(cudaEventRecord(h->ev_fork, h->stream));
    for (int g = 0; g < h->n_groups; ++g) {
      ChainGroup& G = h->groups[g];
      CK(cudaStreamWaitEvent(G.stream, h->ev_fork, 0));
      CK(cudaMemcpyAsync(G.counters, h->e.iter, sizeof(long long), cudaMemcpyDeviceToDevice, G.stream));
      CK(cudaMemcpyAsync(G.counters + 1, h->e.trace_row, sizeof(long long), cudaMemcpyDeviceToDevice, G.stream));
    }
    for (; left >= 2; left -= 2) {
      for (int g = 0; g < h->n_groups; ++g) CK(cudaGraphLaunch(h->groups[g].gexec[par], h->groups[g].stream));
      h->launches += h->graph_kernels;
    }
    // join
    for (int g = 0; g < h->n_groups; ++g) {
      CK(cudaEventRecord(h->groups[g].done, h->groups[g].stream));
      CK(cudaStreamWaitEvent(h->stream, h->groups[g].done, 0));
    }
    CK(cudaMemcpyAsync(h->e.iter, h->groups[0].counters, sizeof(long long), cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync(h->e.trace_row, h->groups[0].counters + 1, sizeof(long long), cudaMemcpyDeviceToDevice, h->stream));
  }
  for (; left > 0; --left) {
    // (an eager sweep flips the u buffers: the next graph run uses the graphs of the other parity)
    const long long before = g_launches;
    enqueue_sweep(h->e, h->ws, h->fj, h->stream);
    h->launches += g_launches - before;
  }
  CK(cudaEventRecord(h->ev1, h->stream));
  // an odd count left the double buffer on the other parity: capture that parity's graphs now, while the device is
  // still busy with what was just enqueued, instead of at the start of the next run
  if (h->e.inj == nullptr && !h->aux_on && (h->graphs_ready[0] || h->graphs_ready[1])) {
    int r = build_graphs(h);
    if (r) return r;
  }
  CK(cudaGetLastError());
  h->ran = true;
  return BNR_OK;
}

extern "C" int bnr_sync(bnr_handle* h) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  return BNR_OK;
}

extern "C" int bnr_last_run_ms(bnr_handle* h, float* ms) {
  if (!h || !ms || !h->ran) return fail(BNR_ESTATE, "no run recorded");
  CK(cudaSetDevice(h->p.device));
  CK(cudaEventSynchronize(h->ev1));
  CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return BNR_OK;
}

extern "C" int bnr_iteration(bnr_handle* h, int64_t* completed) {
  if (!h || !completed) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  long long v = 0;
  CK(cudaMemcpyAsync(&v, h->e.iter, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  *completed = v;
  return BNR_OK;
}

extern "C" int bnr_set_trace_row(bnr_handle* h, int64_t row) {
  if (!h || row < 0) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  long long v = row;
  CK(cudaMemcpyAsync(h->e.trace_row, &v, sizeof(v), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

extern "C" int bnr_get_trace_row(bnr_handle* h, int64_t* row) {
  if (!h || !row) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  long long v = 0;
  CK(cudaMemcpyAsync(&v, h->e.trace_row, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  *row = v;
  return BNR_OK;
}

extern "C" int bnr_copy_trace_rows(bnr_handle* h, int64_t dst, int64_t src, int64_t count) {
  if (!h || dst < 0 || src < 0 || count < 0) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  // every row table of the engine: the record kernels write all of them at *trace_row
  const struct { const RowTable& t; const char* range_msg; } all[] = {
      {e.tr_full, "rows out of range"}, {e.tr_gx, "rows out of range"},
      {e.pred, "rows beyond the prediction table"}, {e.ll, "rows beyond the log-likelihood table"}};
  bool any = false;
  int max_row = 0;
  for (const auto& a : all) {
    if (!a.t.base) continue;
    if (dst + count > a.t.rows || src + count > a.t.rows) return fail(BNR_EINVAL, a.range_msg);
    if (a.t.width > max_row) max_row = a.t.width;
    any = true;
  }
  if (!any) return BNR_OK;                  // this handle records no per-row tables: nothing to move
  if (count == 0 || dst == src) return BNR_OK;
  // rows are contiguous per chain; regions may overlap -> stage through one temporary (stream order keeps the chains apart)
  const bool overlap = !(dst + count <= src || src + count <= dst);
  Scratch sc(h->p.device, overlap ? (size_t)count * max_row * sizeof(double) : 256);
  if (overlap && !sc.p) return fail(BNR_ENOMEM, "device scratch allocation failed");
  for (const auto& a : all) {
    if (!a.t.base) continue;
    const size_t bytes = (size_t)count * a.t.width * sizeof(double);
    for (int c = 0; c < a.t.chains; ++c) {
      if (!overlap) {
        CK(cudaMemcpyAsync(a.t.row(c, dst), a.t.row(c, src), bytes, cudaMemcpyDeviceToDevice, h->stream));
      } else {
        CK(cudaMemcpyAsync(sc.p, a.t.row(c, src), bytes, cudaMemcpyDeviceToDevice, h->stream));
        CK(cudaMemcpyAsync(a.t.row(c, dst), sc.p, bytes, cudaMemcpyDeviceToDevice, h->stream));
      }
    }
  }
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

// device copy of the 5-entry window record (split-half window + block-moment configuration) for the handle and groups
static int push_windows(bnr_handle* h) {
  CK(cudaMemcpyAsync(h->e.mom_window, h->win, sizeof(h->win), cudaMemcpyHostToDevice, h->stream));
  for (int g = 0; g < h->n_groups; ++g)
    CK(cudaMemcpyAsync(h->groups[g].mom_window, h->win, sizeof(h->win), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

extern "C" int bnr_set_moment_window(bnr_handle* h, int64_t first, int64_t len) {
  if (!h || len < 0) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  h->win[0] = first; h->win[1] = len;
  int r = push_windows(h);
  if (r) return r;
  h->mom_half = len / 2;
  return BNR_OK;
}

extern "C" int bnr_set_moment_blocks(bnr_handle* h, int64_t first_sweep, int64_t block_len, int32_t nblocks) {
  if (!h || nblocks < 0 || (nblocks > 0 && block_len < 1)) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  const Dims& d = h->e.d;
  if (nblocks > h->e.bmom_nb) {
    CK(cudaStreamSynchronize(h->stream));
    drop_graph(h);                       // the group views carry the buffer pointer and its block capacity
    void* p = nullptr;
    release_alloc(h, h->e.bmom);
    h->e.bmom = nullptr; h->e.bmom_nb = 0;
    int r = raw_alloc(h, &p, sizeof(double) * (size_t)d.C * nblocks * (d.V + d.q) * 2);
    if (r) return r;
    h->e.bmom = (double*)p;
    h->e.bmom_nb = nblocks;
  }
  h->win[2] = first_sweep; h->win[3] = block_len > 0 ? block_len : 1; h->win[4] = nblocks;
  h->blk_len = block_len;
  return push_windows(h);
}

// merge blocks [first_block, first_block + nblocks) (nblocks even) into the split-half moments: Chan's pairwise update
// applied block after block in a fixed order.  grid = (ceil(P/128), C, 2)
__global__ void k_merge_blocks(const double* __restrict__ bmom, int nb_cap, int nparam, int first_block, int per_half,
                               long long blen, double* __restrict__ mom) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nparam) return;
  const int c = blockIdx.y, half = blockIdx.z;
  double n = 0.0, mean = 0.0, m2 = 0.0;
  for (int b = 0; b < per_half; ++b) {
    const double* m = bmom + (((size_t)c * nb_cap + first_block + half * per_half + b) * nparam + p) * 2;
    const double nb_ = (double)blen, delta = m[0] - mean, tot = n + nb_;
    mean += delta * nb_ / tot;
    m2 += m[1] + delta * delta * n * nb_ / tot;
    n = tot;
  }
  double* o = mom + (((size_t)c * 2 + half) * nparam + p) * 2;
  o[0] = mean; o[1] = m2;
}

extern "C" int bnr_moments_from_blocks(bnr_handle* h, int32_t first_block, int32_t nblocks) {
  if (!h || first_block < 0 || nblocks < 2 || (nblocks & 1)) return fail(BNR_EINVAL, "need an even number of blocks >= 2");
  CK(cudaSetDevice(h->p.device));
  if (!h->e.bmom || first_block + nblocks > (int)h->win[4]) return fail(BNR_ESTATE, "blocks not configured (bnr_set_moment_blocks)");
  const Dims& d = h->e.d;
  const int np_ = d.V + d.q;
  dim3 grid((np_ + 127) / 128, d.C, 2);
  k_merge_blocks<<<grid, 128, 0, h->stream>>>(h->e.bmom, h->e.bmom_nb, np_, first_block, nblocks / 2, h->blk_len, h->e.moments);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  h->mom_half = (long long)(nblocks / 2) * h->blk_len;
  return BNR_OK;
}

extern "C" int bnr_moments_device(bnr_handle* h, double** dev_ptr, int64_t* count) {
  if (!h || !dev_ptr || !count) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  *dev_ptr = h->e.moments;
  *count = (int64_t)h->e.d.C * 2 * (h->e.d.V + h->e.d.q) * 2;
  return BNR_OK;
}

extern "C" int bnr_rhat_from_moments(int device, const double* dev_moments, int32_t total_chains, int32_t V,
                                     int32_t q, int64_t half_len, double* rhat_xi, double* rhat_gamma) {
  if (!dev_moments || total_chains < 1 || half_len < 2) return fail(BNR_EINVAL, "bad arguments (need half_len >= 2)");
  CK(cudaSetDevice(device));
  Scratch sc(device, sizeof(double) * (V + q));
  if (!sc.p) return fail(BNR_ENOMEM, "device scratch allocation failed");
  double* d_out = (double*)sc.p;
  launch_rhat(dev_moments, total_chains, V + q, half_len, d_out, 0);
  std::vector<double> host(V + q);
  CK(cudaMemcpy(host.data(), d_out, sizeof(double) * (V + q), cudaMemcpyDeviceToHost));
  if (rhat_xi) memcpy(rhat_xi, host.data(), sizeof(double) * V);
  if (rhat_gamma) memcpy(rhat_gamma, host.data() + V, sizeof(double) * q);
  return BNR_OK;
}

// two-pass split-half moments of rows [first_row, first_row + nrows) of the gamma/xi traces (what
// return_psrf_VOI + rhat see, src/gibbs.jl:771-789).  grid = (ceil((V+q)/128), C, 2)
__global__ void k_moments_from_trace(RowTable tr, long long first, long long nrows, double* __restrict__ mom) {
  const int nparam = tr.width, p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nparam) return;
  const int c = blockIdx.y, half = blockIdx.z;
  const long long h = nrows / 2;
  const long long r0 = first + (half == 0 ? 0 : nrows - h);
  const double* __restrict__ base = tr.row(c, r0) + p;
  double s = 0.0;
  for (long long r = 0; r < h; ++r) s += base[(size_t)r * nparam];
  const double mean = s / (double)h;
  double m2 = 0.0;
  for (long long r = 0; r < h; ++r) { const double dl = base[(size_t)r * nparam] - mean; m2 += dl * dl; }
  double* m = mom + (((size_t)c * 2 + half) * nparam + p) * 2;
  m[0] = mean; m[1] = m2;
}

extern "C" int bnr_moments_from_trace(bnr_handle* h, int64_t first_row, int64_t nrows) {
  if (!h || first_row < 0 || nrows < 0) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  if (!e.tr_gx.base || e.tr_gx.chains < e.d.C)
    return fail(BNR_ESTATE, "gamma/xi traces of every chain are needed (trace_gamma_xi_all = 0): use the streaming "
                            "moments of bnr_set_moment_window instead");
  if (first_row + nrows > e.tr_gx.rows) return fail(BNR_EINVAL, "rows beyond trace capacity");
  if (nrows / 2 < 2) return fail(BNR_EINVAL, "need at least 4 rows");
  dim3 grid((e.tr_gx.width + 127) / 128, e.d.C, 2);
  k_moments_from_trace<<<grid, 128, 0, h->stream>>>(e.tr_gx, first_row, nrows, e.moments);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  h->mom_half = nrows / 2;
  return BNR_OK;
}

extern "C" int bnr_moment_half_len(bnr_handle* h, int64_t* half_len) {
  if (!h || !half_len) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  *half_len = h->mom_half;
  return BNR_OK;
}

extern "C" int bnr_rhat(bnr_handle* h, double* rhat_xi, double* rhat_gamma) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  CK(cudaSetDevice(h->p.device));
  if (h->mom_half < 2) return fail(BNR_ESTATE, "moment window too short for R-hat");
  const Dims& d = h->e.d;
  launch_rhat(h->e.moments, d.C, d.V + d.q, h->mom_half, h->d_rhat, h->stream);
  std::vector<double> host(d.V + d.q);
  CK(cudaMemcpyAsync(host.data(), h->d_rhat, sizeof(double) * (d.V + d.q), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (rhat_xi) memcpy(rhat_xi, host.data(), sizeof(double) * d.V);
  if (rhat_gamma) memcpy(rhat_gamma, host.data() + d.V, sizeof(double) * d.q);
  return BNR_OK;
}

extern "C" int bnr_var_size(bnr_handle* h, int32_t var, int64_t* n) {
  if (!h || !n || var < 0 || var >= BNR_NUM_VARS) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  *n = var_size(h->e.d, var);
  return BNR_OK;
}

static double* var_ptr(Engine& e, int c, int var) {
  const Dims& d = e.d;
  switch (var) {
    case BNR_VAR_TAU2: return e.tau2 + c;
    case BNR_VAR_U: return e.u + (size_t)c * d.V * d.R;
    case BNR_VAR_XI: return e.xi + (size_t)c * d.V;
    case BNR_VAR_GAMMA: return e.gamma + (size_t)c * d.qp;
    case BNR_VAR_S: return e.S + (size_t)c * d.qp;
    case BNR_VAR_THETA: return e.theta + c;
    case BNR_VAR_DELTA: return e.Delta + c;
    case BNR_VAR_M: return e.M + (size_t)c * d.R * d.R;
    case BNR_VAR_MU: return e.mu + c;
    case BNR_VAR_LAMBDA: return e.lambda + (size_t)c * d.R;
    case BNR_VAR_PI: return e.pi + (size_t)c * 3 * d.R;
  }
  return nullptr;
}

extern "C" int bnr_get_state(bnr_handle* h, int32_t chain, int32_t var, double* out) {
  if (!h || !out || chain < 0 || chain >= h->e.d.C || var < 0 || var >= BNR_NUM_VARS)
    return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  const int n = var_size(h->e.d, var), R = h->e.d.R;
  std::vector<double> tmp(n);
  CK(cudaMemcpyAsync(tmp.data(), var_ptr(h->e, chain, var), sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (var == BNR_VAR_PI) {
    for (int r = 0; r < R; ++r)
      for (int c = 0; c < 3; ++c) out[r + R * c] = tmp[3 * r + c];
  } else {
    memcpy(out, tmp.data(), sizeof(double) * n);
  }
  return BNR_OK;
}

extern "C" int bnr_set_state(bnr_handle* h, int32_t chain, int32_t var, const double* in) {
  if (!h || !in || chain < 0 || chain >= h->e.d.C || var < 0 || var >= BNR_NUM_VARS)
    return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  const int n = var_size(h->e.d, var), R = h->e.d.R;
  std::vector<double> tmp(in, in + n);
  if (var == BNR_VAR_PI)
    for (int r = 0; r < R; ++r)
      for (int c = 0; c < 3; ++c) tmp[3 * r + c] = in[r + R * c];
  CK(cudaMemcpyAsync(var_ptr(h->e, chain, var), tmp.data(), sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (var == BNR_VAR_GAMMA) h->xg_valid = false;
  return BNR_OK;
}

// gather rows [first,last) of one variable into iteration-fastest order
__global__ void k_gather_trace(const double* __restrict__ rows, size_t rowlen, int off, int nelem, long long first,
                               long long count, int pi_R, double* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= count * nelem) return;
  const long long it = idx % count;
  const int el = (int)(idx / count);
  int src = el;
  if (pi_R > 0) { const int r = el % pi_R, c = el / pi_R; src = 3 * r + c; }   // out is (R,3) column-major
  out[idx] = rows[(size_t)(first + it) * rowlen + off + src];
}

// the trace table that holds variable `var` of `chain` and the variable's offset in its rows (nullptr: not traced)
static const RowTable* traced(const Engine& e, int chain, int var, int* off) {
  if (e.tr_full.holds(chain, 0)) { *off = row_offset(e.d, var); return &e.tr_full; }
  if (e.tr_gx.holds(chain, 0) && (var == BNR_VAR_XI || var == BNR_VAR_GAMMA)) {
    *off = var == BNR_VAR_XI ? 0 : e.d.V;
    return &e.tr_gx;
  }
  return nullptr;
}

extern "C" int bnr_get_trace(bnr_handle* h, int32_t chain, int32_t var, int64_t first, int64_t last, double* out) {
  if (!h || !out || chain < 0 || chain >= h->e.d.C || var < 0 || var >= BNR_NUM_VARS || first < 0 || last < first)
    return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  if (last > e.tr_full.rows) return fail(BNR_EINVAL, "rows beyond trace capacity");
  const Dims& d = e.d;
  int off = 0;
  const RowTable* t = traced(e, chain, var, &off);
  if (!t) return fail(BNR_ESTATE, "this variable of this chain is not traced (see trace_full_chains / trace_gamma_xi_all)");
  const double* rows = t->row(chain, 0);
  const size_t rowlen = t->width;
  const int nelem = var_size(d, var);
  const long long count = last - first;
  if (count == 0) return BNR_OK;
  // chunk over elements so the staging buffer suffices
  const long long el_per_chunk = (long long)(h->tmp_doubles / (size_t)count);
  if (el_per_chunk < 1) return fail(BNR_EINVAL, "row range too long for the staging buffer; fetch fewer rows per call");
  for (int e0 = 0; e0 < nelem; e0 += (int)el_per_chunk) {
    const int ne = (int)((nelem - e0) < el_per_chunk ? (nelem - e0) : el_per_chunk);
    const long long tot = count * ne;
    if (var == BNR_VAR_PI) {
      if (ne != nelem) return fail(BNR_EINVAL, "row range too long for pi");
      k_gather_trace<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(rows, rowlen, off, ne, first, count, d.R, h->d_tmp);
    } else {
      k_gather_trace<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(rows, rowlen, off + e0, ne, first, count, 0, h->d_tmp);
    }
    CK(cudaMemcpyAsync(out + (size_t)e0 * count, h->d_tmp, sizeof(double) * tot, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  return BNR_OK;
}

extern "C" int bnr_status(bnr_handle* h, int32_t* status) {
  if (!h || !status) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  CK(cudaMemcpyAsync(status, h->e.status, sizeof(int) * h->e.d.C, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

// ---------------------------------------------------------------------------------------------------------
// parity-test hooks
// ---------------------------------------------------------------------------------------------------------
extern "C" int bnr_injection_size(bnr_handle* h, int32_t for_init, int64_t* per_chain) {
  if (!h || !per_chain) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  const Dims& d = h->e.d;
  *per_chain = for_init ? InitLayout::make(d.V, d.R).total : InjLayout::make(d.n, d.V, d.R, d.gigK).total;
  return BNR_OK;
}

extern "C" int bnr_set_injection(bnr_handle* h, const double* inj, int64_t per_chain) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  drop_graph(h);
  if (!inj) { h->e.inj = nullptr; h->e.inj_stride = 0; return BNR_OK; }
  const size_t total = (size_t)per_chain * h->e.d.C;
  if ((long long)total > h->inj_len) {
    void* p = nullptr;
    release_alloc(h, h->d_inj);
    h->d_inj = nullptr; h->inj_len = 0;
    int r = raw_alloc(h, &p, total * sizeof(double));
    if (r) return r;
    h->d_inj = (double*)p;
    h->inj_len = (long long)total;
  }
  CK(cudaMemcpy(h->d_inj, inj, total * sizeof(double), cudaMemcpyHostToDevice));
  h->e.inj = h->d_inj;
  h->e.inj_stride = per_chain;
  return BNR_OK;
}

extern "C" int bnr_enable_aux(bnr_handle* h, int32_t on) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  const Dims& d = e.d;
  const size_t C = d.C;
  CK(cudaStreamSynchronize(h->stream));
  drop_graph(h);
  if (!on) {
    if (h->aux_on) { h->aux_saved = e.aux; memset(&e.aux, 0, sizeof(e.aux)); }
    h->aux_on = false;
    return BNR_OK;
  }
  if (h->aux_on) return BNR_OK;
  if (h->aux_saved.tau2_params) {
    e.aux = h->aux_saved;
  } else {
    DA(e.aux.tau2_params, C * 2); DA(e.aux.sigma_inv, C * d.V * d.R * d.R); DA(e.aux.sigma_chol, C * d.V * d.R * d.R);
    DA(e.aux.mu_t, C * d.V * d.R); DA(e.aux.log_odds, C * d.V); DA(e.aux.chi, C * d.qp);
    DA(e.aux.theta_params, C * 2); DA(e.aux.delta_params, C * 2); DA(e.aux.m_params, C * (1 + 2 * d.R * d.R));
    DA(e.aux.mu_params, C * 2); DA(e.aux.lambda_logw, C * 3 * d.R); DA(e.aux.lambda_w, C * 3 * d.R);
    DA(e.aux.pi_alpha, C * 3 * d.R); DA(e.aux.gig_used, C * d.qp); DA(e.aux.G_copy, C * d.gdim * d.gdim);
    CK(cudaStreamSynchronize(h->stream));
  }
  h->aux_on = true;
  return BNR_OK;
}

extern "C" int bnr_get_aux(bnr_handle* h, int32_t chain, int32_t aux_id, double* out, int64_t capacity) {
  if (!h || !out || chain < 0 || chain >= h->e.d.C) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  if (!h->aux_on) return fail(BNR_ESTATE, "call bnr_enable_aux first");
  Engine& e = h->e;
  const Dims& d = e.d;
  const int R = d.R, V = d.V, RR = R * R;
  const double* src = nullptr;
  size_t n = 0;
  std::vector<double> tmp;
  switch (aux_id) {
    case BNR_AUX_TAU2_PARAMS: src = e.aux.tau2_params + 2 * chain; n = 2; break;
    case BNR_AUX_SIGMA_INV: src = e.aux.sigma_inv + (size_t)chain * V * RR; n = (size_t)V * RR; break;
    case BNR_AUX_SIGMA_CHOL: src = e.aux.sigma_chol + (size_t)chain * V * RR; n = (size_t)V * RR; break;
    case BNR_AUX_MU_T: src = e.aux.mu_t + (size_t)chain * V * R; n = (size_t)V * R; break;
    case BNR_AUX_LOG_ODDS: src = e.aux.log_odds + (size_t)chain * V; n = V; break;
    case BNR_AUX_W: src = e.W + (size_t)chain * d.qp; n = d.q; break;
    case BNR_AUX_RHS: case BNR_AUX_A4:
      if (d.gmode == BNR_GAMMA_QFORM) { src = e.t + (size_t)chain * d.qp; n = d.q; }   // beta = gamma - W
      else { src = e.rhs + (size_t)chain * d.np; n = d.n; }
      break;
    case BNR_AUX_CHI: src = e.aux.chi + (size_t)chain * d.qp; n = d.q; break;
    case BNR_AUX_THETA_PARAMS: src = e.aux.theta_params + 2 * chain; n = 2; break;
    case BNR_AUX_DELTA_PARAMS: src = e.aux.delta_params + 2 * chain; n = 2; break;
    case BNR_AUX_M_PARAMS: src = e.aux.m_params + (size_t)chain * (1 + 2 * RR); n = 1 + 2 * RR; break;
    case BNR_AUX_MU_PARAMS: src = e.aux.mu_params + 2 * chain; n = 2; break;
    case BNR_AUX_LAMBDA_LOGW: src = e.aux.lambda_logw + (size_t)chain * 3 * R; n = 3 * R; break;
    case BNR_AUX_LAMBDA_WEIGHTS: src = e.aux.lambda_w + (size_t)chain * 3 * R; n = 3 * R; break;
    case BNR_AUX_PI_ALPHA: src = e.aux.pi_alpha + (size_t)chain * 3 * R; n = 3 * R; break;
    case BNR_AUX_GIG_USED: src = e.aux.gig_used + (size_t)chain * d.qp; n = d.q; break;
    case BNR_AUX_G: case BNR_AUX_G_CHOL: {
      // m x m sub-block of the padded gdim x gdim matrix (m = n in the n-form, q in the q-form)
      const int m = d.gmode == BNR_GAMMA_QFORM ? d.q : d.n, N = d.gdim;
      const double* base = (aux_id == BNR_AUX_G ? e.aux.G_copy : e.G) + (size_t)chain * N * N;
      if (capacity < (int64_t)m * m) return fail(BNR_EINVAL, "capacity too small");
      tmp.resize((size_t)N * N);
      CK(cudaMemcpyAsync(tmp.data(), base, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      for (int j = 0; j < m; ++j)
        for (int i = 0; i < m; ++i) {
          double v = tmp[(size_t)j * N + i];
          if (aux_id == BNR_AUX_G_CHOL && i < j) v = 0.0;
          out[(size_t)j * m + i] = v;
        }
      return BNR_OK;
    }
    default: return fail(BNR_EINVAL, "unknown aux id");
  }
  if ((int64_t)n > capacity) return fail(BNR_EINVAL, "capacity too small");
  CK(cudaMemcpyAsync(out, src, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

// One conditional, in place, on the state as it stands (the reference's update_*!(state, i, ...) with rows
// i-1 / i merged: every variable holds its most recent value).
extern "C" int bnr_step(bnr_handle* h, int32_t cond) {
  if (!h || cond < 0 || cond >= BNR_NUM_CONDS) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  drop_graph(h);
  Engine& e = h->e;
  cudaStream_t s = h->stream;
  switch (cond) {
    case BNR_COND_TAU2:
      refresh_xg(h);
      launch_tau2(e, s);
      break;
    case BNR_COND_U_XI:
      launch_uxi(e, s);
      std::swap(e.u, e.u_alt);
      break;
    case BNR_COND_GAMMA:
      run_gamma(h->e, h->ws, h->fj, h->stream, 1);
      h->xg_valid = false;
      break;
    case BNR_COND_D:
      launch_edge_prep(e, 0, s);
      launch_gamma_gig(e, 2, s);
      break;
    case BNR_COND_THETA: case BNR_COND_LAMBDA:
      launch_edge_prep(e, 0, s);
      launch_gamma_gig(e, 0, s);       // refresh sum S and the lambda statistics from the current state
      launch_finish(e, 1 << cond, s);
      break;
    case BNR_COND_MU:
      refresh_xg(h);
      launch_finish(e, 1 << cond, s);
      break;
    default:
      launch_finish(e, 1 << cond, s);
      break;
  }
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

extern "C" int bnr_finish_sweep(bnr_handle* h) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  CK(cudaSetDevice(h->p.device));
  enqueue_record(h->e, h->ws, h->fj, h->stream, true, false, !h->xg_valid);
  if (h->e.ll.base) h->xg_valid = true;                       // (the log-likelihood row refreshed it)
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

// the jitter ladder of update_u_xi! (src/gibbs.jl:322-347) on a caller-supplied R x R matrix (col-major host arrays)
extern "C" int bnr_test_chol_jitter(bnr_handle* h, int32_t R, const double* A, double* A_used, double* L, int32_t* status) {
  if (!h || !A || !A_used || !L || !status || R < 1 || R > BNR_MAX_R) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  const size_t RR = (size_t)R * R;
  if (3 * RR + 1 > h->tmp_doubles) return fail(BNR_EINVAL, "staging buffer too small");
  double* d = h->d_tmp;
  CK(cudaMemcpyAsync(d, A, sizeof(double) * RR, cudaMemcpyHostToDevice, h->stream));
  launch_test_chol_jitter(R, d, d + RR, d + 2 * RR, reinterpret_cast<int*>(d + 3 * RR), h->stream);
  CK(cudaMemcpyAsync(A_used, d + RR, sizeof(double) * RR, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(L, d + 2 * RR, sizeof(double) * RR, cudaMemcpyDeviceToHost, h->stream));
  int st = 0;
  CK(cudaMemcpyAsync(&st, d + 3 * RR, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  *status = st;
  return BNR_OK;
}

static int rng_dump(bnr_handle* h, int chain, int64_t iteration, int site, int element, int kind, double shape,
                    int count, double* out) {
  if (!h || !out || count < 1 || chain < 0 || chain >= h->e.d.C) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  if ((size_t)count > h->tmp_doubles) return fail(BNR_EINVAL, "count too large");
  launch_rng_dump(h->e.d, chain, iteration, site, element, kind, shape, count, h->d_tmp, h->stream);
  CK(cudaMemcpyAsync(out, h->d_tmp, sizeof(double) * count, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

extern "C" int bnr_rng_stream(bnr_handle* h, int32_t chain, int64_t iteration, int32_t site, int32_t element,
                              int32_t kind, int32_t count, double* out) {
  if (kind != 0 && kind != 1) return fail(BNR_EINVAL, "kind must be 0 (uniform) or 1 (normal)");
  return rng_dump(h, chain, iteration, site, element, kind, 0.0, count, out);
}

extern "C" int bnr_rng_gamma(bnr_handle* h, int32_t chain, int64_t iteration, int32_t site, int32_t element,
                             double shape, int32_t count, double* out) {
  if (!(shape > 0.0)) return fail(BNR_EINVAL, "shape must be positive");
  return rng_dump(h, chain, iteration, site, element, 2, shape, count, out);
}

// ---------------------------------------------------------------------------------------------------------
// Summary on the device (src/gibbs.jl:1214-1250): mean and the two order statistics per edge, mean xi per node
// ---------------------------------------------------------------------------------------------------------
extern "C" int bnr_summary(bnr_handle* h, int32_t chain, int64_t first_row, int64_t nrows, int64_t rank_lo,
                           int64_t rank_hi, double* gamma_mean, double* gamma_lo, double* gamma_hi, double* xi_mean) {
  if (!h || chain < 0 || chain >= h->e.d.C || first_row < 0 || nrows < 1)
    return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  const Dims& d = e.d;
  if (first_row + nrows > e.tr_full.rows) return fail(BNR_EINVAL, "rows beyond trace capacity");
  if (rank_lo < 1 || rank_hi < 1 || rank_lo > nrows || rank_hi > nrows)
    return fail(BNR_EINVAL, "order-statistic ranks must lie in 1..nrows (the reference raises a BoundsError)");
  CK(cudaSetDevice(h->p.device));
  int off_g = 0, off_x = 0;
  const RowTable* t = traced(e, chain, BNR_VAR_GAMMA, &off_g);
  if (!t) return fail(BNR_ESTATE, "gamma/xi of this chain are not traced");
  traced(e, chain, BNR_VAR_XI, &off_x);     // (the same table)
  const double* rows = t->row(chain, 0);
  const size_t rowlen = t->width;
  if ((size_t)(3 * d.q + d.V) > h->tmp_doubles) return fail(BNR_EINVAL, "staging buffer too small");
  double* o = h->d_tmp;
  launch_summary_select(rows, rowlen, off_g, d.q, first_row, nrows, rank_lo, rank_hi, o, o + d.q, o + 2 * d.q, h->stream);
  launch_summary_select(rows, rowlen, off_x, d.V, first_row, nrows, 1, 1, o + 3 * d.q, nullptr, nullptr, h->stream);
  std::vector<double> host((size_t)3 * d.q + d.V);
  CK(cudaMemcpyAsync(host.data(), o, sizeof(double) * host.size(), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  if (gamma_mean) memcpy(gamma_mean, host.data(), sizeof(double) * d.q);
  if (gamma_lo) memcpy(gamma_lo, host.data() + d.q, sizeof(double) * d.q);
  if (gamma_hi) memcpy(gamma_hi, host.data() + 2 * d.q, sizeof(double) * d.q);
  if (xi_mean) memcpy(xi_mean, host.data() + 3 * d.q, sizeof(double) * d.V);
  return BNR_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Effective sample size of xi / gamma over rows [first_row, first_row + nrows) of every chain's trace
// ---------------------------------------------------------------------------------------------------------
extern "C" int bnr_ess_accumulate(bnr_handle* h, int64_t first_row, int64_t nrows, int32_t max_lag) {
  if (!h || first_row < 0 || nrows < 4 || max_lag < 1) return fail(BNR_EINVAL, "bad arguments (need nrows >= 4, max_lag >= 1)");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  const Dims& d = e.d;
  if (!e.tr_gx.base || e.tr_gx.chains < d.C)
    return fail(BNR_ESTATE, "gamma/xi traces of every chain are not recorded (trace_gamma_xi_all = 0)");
  if (first_row + nrows > e.tr_gx.rows) return fail(BNR_EINVAL, "rows beyond trace capacity");
  if (max_lag > nrows - 1) max_lag = (int32_t)(nrows - 1);
  if (!(max_lag & 1)) max_lag -= 1;                  // Geyer pairs (2t, 2t+1): keep the last lag odd
  if (max_lag < 1) max_lag = 1;
  CK(cudaSetDevice(h->p.device));
  const int P = d.V + d.q;
  const size_t need = (size_t)(max_lag + 1) * P;
  if (need > h->acov_cap) {
    void* pnew = nullptr;
    release_alloc(h, h->d_acov);
    h->d_acov = nullptr; h->acov_cap = 0;
    int r = raw_alloc(h, &pnew, need * sizeof(double));
    if (r) return r;
    h->d_acov = (double*)pnew;
    h->acov_cap = need;
  }
  if (!h->d_cmean) DA(h->d_cmean, (size_t)d.C * P);
  launch_chain_mean(e.tr_gx, first_row, nrows, h->d_cmean, h->stream);
  launch_acov_sum(e.tr_gx, first_row, nrows, max_lag, h->d_cmean, h->d_acov, h->stream);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  h->ess_lag = max_lag;
  h->ess_rows = nrows;
  return BNR_OK;
}

// Streaming variant: the next `ndraws` sweeps contribute their lagged products while they run (k_ess_stream), so no
// chain needs a trace.  bnr_ess_stream_finish turns the accumulators into the same two statistics buffers.
static int ess_stream_arm(bnr_handle* h, int32_t max_lag, int64_t first_sweep, int64_t ndraws) {
  if (!h || ndraws < 4 || max_lag < 1) return fail(BNR_EINVAL, "bad arguments (need ndraws >= 4, max_lag >= 1)");
  CK(cudaSetDevice(h->p.device));
  Engine& e = h->e;
  const Dims& d = e.d;
  if (max_lag > ndraws - 1) max_lag = (int32_t)(ndraws - 1);
  if (!(max_lag & 1)) max_lag -= 1;
  if (max_lag < 1) max_lag = 1;
  const int L = max_lag, cap = L + 8;
  const size_t P = (size_t)d.V + d.q, C = d.C;
  CK(cudaStreamSynchronize(h->stream));
  long long it = 0;
  CK(cudaMemcpyAsync(&it, e.iter, sizeof(it), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (first_sweep < 0) first_sweep = it + 1;
  if (first_sweep <= it) return fail(BNR_EINVAL, "the window must start after the sweeps already run");
  if (!e.ess_ring || e.ess_L != L) drop_graph(h);   // the sweep graphs gain the k_ess_stream node / its new geometry
  const size_t need = C * P * ((size_t)cap + L + (L + 1) + 2);
  if (need > h->ess_stream_cap) {
    void* pnew = nullptr;
    release_alloc(h, h->ess_stream_buf);
    h->ess_stream_buf = nullptr; h->ess_stream_cap = 0;
    int r = raw_alloc(h, &pnew, need * sizeof(double));
    if (r) return r;
    h->ess_stream_cap = need;
    h->ess_stream_buf = (double*)pnew;
    drop_graph(h);
  }
  e.ess_ring = h->ess_stream_buf;
  e.ess_head = e.ess_ring + C * P * cap;
  e.ess_acc = e.ess_head + C * P * L;
  e.ess_sum = e.ess_acc + C * P * (L + 1);
  e.ess_L = L; e.ess_cap = cap;
  e.ess_win = h->d_esswin;
  const long long win[4] = {first_sweep, ndraws, L, cap};
  CK(cudaMemcpyAsync(h->d_esswin, win, sizeof(win), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  const size_t acov_need = (size_t)(L + 1) * P;
  if (acov_need > h->acov_cap) {
    void* pnew = nullptr;
    release_alloc(h, h->d_acov);
    h->d_acov = nullptr; h->acov_cap = 0;
    int r = raw_alloc(h, &pnew, acov_need * sizeof(double));
    if (r) return r;
    h->d_acov = (double*)pnew;
    h->acov_cap = acov_need;
  }
  if (!h->d_cmean) DA(h->d_cmean, C * P);
  h->ess_stream_N = ndraws;
  h->ess_lag = -1;
  return BNR_OK;
}

// Streaming variant: the next `ndraws` sweeps contribute their lagged products while they run (k_ess_stream), so no
// chain needs a trace.  bnr_ess_stream_finish turns the accumulators into the same two statistics buffers.
extern "C" int bnr_ess_stream_begin(bnr_handle* h, int32_t max_lag, int64_t ndraws) {
  return ess_stream_arm(h, max_lag, -1, ndraws);
}

extern "C" int bnr_ess_stream_window(bnr_handle* h, int32_t max_lag, int64_t first_sweep, int64_t ndraws) {
  if (first_sweep < 1) return fail(BNR_EINVAL, "first_sweep is a 1-based sweep number");
  return ess_stream_arm(h, max_lag, first_sweep, ndraws);
}

extern "C" int bnr_ess_stream_finish(bnr_handle* h) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  if (h->ess_stream_N <= 0 || !h->e.ess_ring) return fail(BNR_ESTATE, "call bnr_ess_stream_begin first");
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  long long it = 0, win[4];
  CK(cudaMemcpy(&it, h->e.iter, sizeof(it), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(win, h->d_esswin, sizeof(win), cudaMemcpyDeviceToHost));
  if (it < win[0] + win[1] - 1)
    return fail(BNR_ESTATE, "the streaming window is not complete yet (run the remaining sweeps first)");
  launch_ess_stream_finalize(h->e, h->ess_stream_N, h->d_acov, h->d_cmean, h->stream);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  h->ess_lag = h->e.ess_L;
  h->ess_rows = h->ess_stream_N;
  h->ess_stream_N = 0;
  drop_graph(h);                         // later sweeps run without the accumulation kernel
  h->e.ess_ring = h->e.ess_head = h->e.ess_acc = h->e.ess_sum = nullptr;
  // (the buffer stays with the handle and is reused by the next bnr_ess_stream_begin)
  return BNR_OK;
}

extern "C" int bnr_ess_device(bnr_handle* h, double** acov_sum, int64_t* n_acov, double** chain_mean,
                              int64_t* n_mean, int32_t* max_lag) {
  if (!h || !acov_sum || !n_acov || !chain_mean || !n_mean || !max_lag) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  if (h->ess_lag < 0) return fail(BNR_ESTATE, "call bnr_ess_accumulate first");
  const int P = h->e.d.V + h->e.d.q;
  *acov_sum = h->d_acov; *n_acov = (int64_t)(h->ess_lag + 1) * P;
  *chain_mean = h->d_cmean; *n_mean = (int64_t)h->e.d.C * P;
  *max_lag = h->ess_lag;
  return BNR_OK;
}

extern "C" int bnr_export_ess(bnr_handle* h, double* dev_acov_dst, double* dev_means_dst) {
  if (!h || !dev_acov_dst || !dev_means_dst) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  if (h->ess_lag < 0) return fail(BNR_ESTATE, "call bnr_ess_accumulate first");
  const size_t P = (size_t)h->e.d.V + h->e.d.q;
  CK(cudaMemcpyAsync(dev_acov_dst, h->d_acov, sizeof(double) * (h->ess_lag + 1) * P, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(dev_means_dst, h->d_cmean, sizeof(double) * h->e.d.C * P, cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

extern "C" int bnr_ess_from_stats_lags(int device, const double* dev_acov_parts, int32_t nparts,
                                       const double* dev_chain_means, int32_t total_chains, int32_t V, int32_t q,
                                       int64_t nrows, int32_t max_lag, double* ess_xi, double* ess_gamma,
                                       double* lags_xi, double* lags_gamma) {
  if (!dev_acov_parts || !dev_chain_means || nparts < 1 || total_chains < 1 || nrows < 4 || max_lag < 1)
    return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(device));
  const int P = V + q;
  Scratch sc(device, sizeof(double) * 2 * P);
  if (!sc.p) return fail(BNR_ENOMEM, "device scratch allocation failed");
  double* d_out = (double*)sc.p;
  launch_ess_finish(dev_acov_parts, nparts, dev_chain_means, total_chains, P, nrows, max_lag, d_out, d_out + P, 0);
  std::vector<double> host((size_t)2 * P);
  CK(cudaMemcpy(host.data(), d_out, sizeof(double) * 2 * P, cudaMemcpyDeviceToHost));
  if (ess_xi) memcpy(ess_xi, host.data(), sizeof(double) * V);
  if (ess_gamma) memcpy(ess_gamma, host.data() + V, sizeof(double) * q);
  if (lags_xi) memcpy(lags_xi, host.data() + P, sizeof(double) * V);
  if (lags_gamma) memcpy(lags_gamma, host.data() + P + V, sizeof(double) * q);
  return BNR_OK;
}

extern "C" int bnr_ess_from_stats(int device, const double* dev_acov_parts, int32_t nparts,
                                  const double* dev_chain_means, int32_t total_chains, int32_t V, int32_t q,
                                  int64_t nrows, int32_t max_lag, double* ess_xi, double* ess_gamma) {
  return bnr_ess_from_stats_lags(device, dev_acov_parts, nparts, dev_chain_means, total_chains, V, q, nrows, max_lag,
                                 ess_xi, ess_gamma, nullptr, nullptr);
}

extern "C" int bnr_ess(bnr_handle* h, int64_t first_row, int64_t nrows, int32_t max_lag, double* ess_xi,
                       double* ess_gamma) {
  int r = bnr_ess_accumulate(h, first_row, nrows, max_lag);
  if (r) return r;
  const Dims& d = h->e.d;
  return bnr_ess_from_stats(h->p.device, h->d_acov, 1, h->d_cmean, d.C, d.V, d.q, nrows, h->ess_lag, ess_xi, ess_gamma);
}

extern "C" int bnr_gamma_mode(bnr_handle* h, int32_t* mode) {
  if (!h || !mode) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  *mode = h->e.d.gmode;
  return BNR_OK;
}

extern "C" int bnr_device_copy(int device, void* dev_dst, const void* dev_src, int64_t bytes) {
  if (!dev_dst || !dev_src || bytes < 0) return fail(BNR_EINVAL, "bad arguments");
  CK(cudaSetDevice(device));
  CK(cudaMemcpy(dev_dst, dev_src, (size_t)bytes, cudaMemcpyDeviceToDevice));
  return BNR_OK;
}

extern "C" int bnr_chain_groups(bnr_handle* h, int32_t* groups) {
  if (!h || !groups) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  *groups = h->n_groups;
  return BNR_OK;
}

extern "C" int bnr_launch_count(bnr_handle* h, int64_t* kernels) {
  if (!h || !kernels) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  *kernels = h->launches;
  return BNR_OK;
}

extern "C" int bnr_export_moments(bnr_handle* h, double* dev_dst) {
  if (!h || !dev_dst) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  const size_t n = (size_t)h->e.d.C * 2 * (h->e.d.V + h->e.d.q) * 2;
  CK(cudaMemcpyAsync(dev_dst, h->e.moments, n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

// One eager sweep (enqueue_sweep, on the handle's stream) with CUDA events between its phases.  ms[8]:
// 0 tau2, 1 (u,xi), 2 gamma prep (W, v, X v, rhs), 3 SYRK X D X' + I (q-form: P), 4 Cholesky, 5 triangular solves,
// 6 X' a4 + gamma + GIG, 7 X gamma + theta/Delta/M/mu/lambda/pi + record.
extern "C" int bnr_profile_sweep(bnr_handle* h, float* ms) {
  if (!h || !ms) return fail(BNR_EINVAL, "null argument");
  CK(cudaSetDevice(h->p.device));
  drop_graph(h);
  if (!h->xg_valid) refresh_xg(h);
  cudaEvent_t ev[9];
  for (int i = 0; i < 9; ++i) CK(cudaEventCreate(&ev[i]));
  enqueue_sweep(h->e, h->ws, h->fj, h->stream, ev);
  CK(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < 8; ++i) CK(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
  for (int i = 0; i < 9; ++i) cudaEventDestroy(ev[i]);
  CK(cudaGetLastError());
  return BNR_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Predictions for new networks: every recorded row of every chain also gets mu + X_new gamma (+ noise) per new network
// ---------------------------------------------------------------------------------------------------------
static void drop_predictors(bnr_handle* h) {
  Engine& e = h->e;
  release_alloc(h, const_cast<double*>(e.Xp));
  release_alloc(h, e.pred.base);
  release_alloc(h, e.pred_ws);
  e.Xp = nullptr; e.pred = {}; e.pred_ws = nullptr;
  e.pred_mp = e.pred_mode = e.pred_splits = 0;
}

// rows [first, last) of one chain of a row table into out[row + count * column] (iteration fastest, like the traces)
static int get_table_rows(bnr_handle* h, const RowTable& t, int chain, int64_t first, int64_t last, double* out) {
  CK(cudaSetDevice(h->p.device));
  const size_t count = (size_t)(last - first), w = (size_t)t.width;
  if (count == 0) return BNR_OK;
  std::vector<double> tmp(count * w);
  CK(cudaMemcpyAsync(tmp.data(), t.row(chain, first), sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  for (size_t r = 0; r < count; ++r)
    for (size_t j = 0; j < w; ++j) out[r + count * j] = tmp[r * w + j];
  return BNR_OK;
}

// rows [first_row, first_row + nrows) of every chain of a row table into dev_dst, [chain][nrows][width]
static int export_table_rows(bnr_handle* h, const RowTable& t, int64_t first_row, int64_t nrows, double* dev_dst) {
  CK(cudaSetDevice(h->p.device));
  if (nrows == 0) return BNR_OK;
  const size_t rowb = sizeof(double) * (size_t)t.width;
  CK(cudaMemcpy2DAsync(dev_dst, rowb * nrows, t.row(0, first_row), rowb * t.rows, rowb * nrows, (size_t)t.chains,
                       cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return BNR_OK;
}

extern "C" int bnr_set_predictors(bnr_handle* h, int32_t m, const double* X_new, int64_t rows, int32_t mode) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  if (m < 0) return fail(BNR_EINVAL, "m must be >= 0");
  if (mode != BNR_PRED_MEAN && mode != BNR_PRED_PREDICTIVE) return fail(BNR_EINVAL, "unknown prediction mode");
  if (m > 0 && !X_new) return fail(BNR_EINVAL, "null X_new");
  if (m > 0 && rows < 1) return fail(BNR_EINVAL, "the prediction table needs rows >= 1");
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  drop_graph(h);                       // the captured sweeps gain or lose the prediction nodes
  drop_predictors(h);
  if (m == 0) return BNR_OK;
  Engine& e = h->e;
  const Dims& d = e.d;
  const int mp = (m + TILE_N - 1) / TILE_N * TILE_N;
  const int ks = pred_splits(d, mp);
  RowTable pred = {nullptr, rows, m, d.C};
  if (int r = alloc_table(h, pred, true, "prediction table")) return r;
  double *xp = nullptr, *ws = nullptr;
  int r = dalloc(h, &xp, (size_t)d.qp * mp);
  if (!r) r = dalloc(h, &ws, (size_t)ks * d.C * mp, false);
  if (r) {
    cudaGetLastError();                // a refused cudaMalloc must not surface in a later call
    release_alloc(h, pred.base); release_alloc(h, xp); release_alloc(h, ws);
    return fail(r, "X_new and the split-K partials of the predictions (" +
                       std::to_string(8.0 * ((double)d.qp * mp + (double)ks * d.C * mp)) + " bytes): " + g_err);
  }
  // X_new: m x q column-major host -> columns padded to mp rows (zeros beyond m and beyond q, like X)
  CK(cudaMemcpy2DAsync(xp, (size_t)mp * sizeof(double), X_new, (size_t)m * sizeof(double), (size_t)m * sizeof(double),
                       (size_t)d.q, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  e.Xp = xp; e.pred = pred; e.pred_ws = ws;
  e.pred_mp = mp; e.pred_mode = mode; e.pred_splits = ks;
  return BNR_OK;
}

extern "C" int bnr_get_prediction_trace(bnr_handle* h, int32_t chain, int64_t first, int64_t last, double* out) {
  if (!h || !out || chain < 0 || chain >= h->e.d.C || first < 0 || last < first) return fail(BNR_EINVAL, "bad arguments");
  if (!h->e.pred.base) return fail(BNR_ESTATE, "no predictors set (bnr_set_predictors)");
  if (last > h->e.pred.rows) return fail(BNR_EINVAL, "rows beyond the prediction table");
  return get_table_rows(h, h->e.pred, chain, first, last, out);
}

extern "C" int bnr_export_predictions(bnr_handle* h, int64_t first_row, int64_t nrows, double* dev_dst) {
  if (!h || !dev_dst || first_row < 0 || nrows < 0) return fail(BNR_EINVAL, "bad arguments");
  if (!h->e.pred.base) return fail(BNR_ESTATE, "no predictors set (bnr_set_predictors)");
  if (first_row + nrows > h->e.pred.rows) return fail(BNR_EINVAL, "rows beyond the prediction table");
  return export_table_rows(h, h->e.pred, first_row, nrows, dev_dst);
}

extern "C" int bnr_prediction_summary(int device, const double* dev_rows, int64_t count, int32_t m, int64_t rank_lo,
                                      int64_t rank_hi, double* mean, double* lo, double* hi) {
  if (!dev_rows || count < 1 || m < 1) return fail(BNR_EINVAL, "bad arguments (need rows, count >= 1, m >= 1)");
  if (rank_lo < 1 || rank_hi < 1 || rank_lo > count || rank_hi > count)
    return fail(BNR_EINVAL, "order-statistic ranks must lie in 1..count");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(BNR_ENODEV, "no CUDA device visible: libbnr has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(BNR_EINVAL, "device ordinal out of range");
  CK(cudaSetDevice(device));
  const size_t outb = sizeof(double) * 3 * (size_t)m;
  Scratch sc(device, pred_select_ws_bytes(count, m) + outb);
  if (!sc.p) return fail(BNR_ENOMEM, "device scratch allocation failed");
  double* o = (double*)sc.p;
  launch_pred_select(dev_rows, count, m, rank_lo, rank_hi, o, o + m, o + 2 * m, o + 3 * m, 0);
  std::vector<double> host((size_t)3 * m);
  CK(cudaMemcpy(host.data(), o, outb, cudaMemcpyDeviceToHost));
  CK(cudaGetLastError());
  if (mean) memcpy(mean, host.data(), sizeof(double) * m);
  if (lo) memcpy(lo, host.data() + m, sizeof(double) * m);
  if (hi) memcpy(hi, host.data() + 2 * m, sizeof(double) * m);
  return BNR_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Pointwise log-likelihood: every recorded row of every chain also gets log p(y_i | state) for every observation i,
// the input of PSIS-LOO and WAIC (bnr_loo_summary)
// ---------------------------------------------------------------------------------------------------------
extern "C" int bnr_set_loglik(bnr_handle* h, int64_t rows) {
  if (!h) return fail(BNR_EINVAL, "null handle");
  if (rows < 0) return fail(BNR_EINVAL, "rows must be >= 0");
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  drop_graph(h);                       // the captured sweeps gain or lose the k_loglik_record node
  Engine& e = h->e;
  release_alloc(h, e.ll.base);
  e.ll = {};
  if (rows == 0) return BNR_OK;
  RowTable ll = {nullptr, rows, e.d.n, e.d.C};
  if (int r = alloc_table(h, ll, true, "log-likelihood table")) return r;
  CK(cudaStreamSynchronize(h->stream));
  e.ll = ll;
  return BNR_OK;
}

extern "C" int bnr_get_loglik_trace(bnr_handle* h, int32_t chain, int64_t first, int64_t last, double* out) {
  if (!h || !out || chain < 0 || chain >= h->e.d.C || first < 0 || last < first) return fail(BNR_EINVAL, "bad arguments");
  if (!h->e.ll.base) return fail(BNR_ESTATE, "no log-likelihood table (bnr_set_loglik)");
  if (last > h->e.ll.rows) return fail(BNR_EINVAL, "rows beyond the log-likelihood table");
  return get_table_rows(h, h->e.ll, chain, first, last, out);
}

extern "C" int bnr_export_loglik(bnr_handle* h, int64_t first_row, int64_t nrows, double* dev_dst) {
  if (!h || !dev_dst || first_row < 0 || nrows < 0) return fail(BNR_EINVAL, "bad arguments");
  if (!h->e.ll.base) return fail(BNR_ESTATE, "no log-likelihood table (bnr_set_loglik)");
  if (first_row + nrows > h->e.ll.rows) return fail(BNR_EINVAL, "rows beyond the log-likelihood table");
  return export_table_rows(h, h->e.ll, first_row, nrows, dev_dst);
}

extern "C" int bnr_loo_summary(int device, const double* dev_rows, int64_t N, int32_t n, double* elpd_loo,
                               double* p_loo, double* pareto_k, double* elpd_waic, double* p_waic) {
  if (!dev_rows || N < 2 || n < 1) return fail(BNR_EINVAL, "bad arguments (need rows, N >= 2 draws, n >= 1)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(BNR_ENODEV, "no CUDA device visible: libbnr has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(BNR_EINVAL, "device ordinal out of range");
  CK(cudaSetDevice(device));
  const long long M = loo_tail_len(N), Mmax = loo_tail_max();
  if (M > Mmax)
    return fail(BNR_EINVAL, "the Pareto tail of " + std::to_string(N) + " draws (" + std::to_string(M) +
                                " values) exceeds the " + std::to_string(Mmax) +
                                " values one block's shared memory holds (at most about " +
                                std::to_string((long long)((double)Mmax * Mmax / 9.0)) + " pooled draws)");
  const size_t outb = sizeof(double) * 5 * (size_t)n;
  Scratch sc(device, loo_ws_bytes(N, n) + outb);
  if (!sc.p) return fail(BNR_ENOMEM, "device scratch allocation failed");
  double* o = (double*)sc.p;
  launch_loo(dev_rows, N, n, o, o + 5 * (size_t)n, 0);
  std::vector<double> host((size_t)5 * n);
  CK(cudaMemcpy(host.data(), o, outb, cudaMemcpyDeviceToHost));
  CK(cudaGetLastError());
  double* dst[5] = {elpd_loo, p_loo, pareto_k, elpd_waic, p_waic};
  for (int k = 0; k < 5; ++k)
    if (dst[k]) memcpy(dst[k], host.data() + (size_t)k * n, sizeof(double) * n);
  return BNR_OK;
}
