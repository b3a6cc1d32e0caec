// bnr_fit: the whole chain generation behind Fit!(X, y, R; ...) in ONE C-ABI call -- what the reference does in
// generate_samples! / generate_samples_dbl! (src/gibbs.jl:897-1020, 1051-1198) around initialize_and_run! / run!
// (822-864) and return_psrf_VOI (771-789), plus the statistics Summary needs (1214-1250).
//
// The control flow is host code written against a small operations interface (Ops), implemented twice:
//   * DeviceOps  drives a flat list of libbnr handles through the public entry points of include/bnr.h.  The handles
//                are grouped into folds, a fold being the handles whose chains pool their statistics: bnr_fit shards
//                its chains over one fold of n_devices GPUs of this process (the split-half moments -- and the ESS
//                statistics -- are exchanged with ncclAllGather, then optionally across processes through a
//                caller-supplied all-gather); bnr_fit_kfold makes K folds of one handle each;
//   * PlanOps    records the operations and takes the PSRF maxima from the caller: bnr_fit_plan, a pure host function
//                that lets the control flow be tested without a GPU against the restated reference loops
//                (oracle/psrf_loops.py).
// Row / sweep conventions: table rows are 0-based here (the reference's row r is row r - 1), sweep s = 1, 2, ... is the
// s-th Gibbs sweep of a chain, row 0 holds the prior draw (sweep 0).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <chrono>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "../../include/bnr.h"

namespace {

thread_local std::string g_fit_err;
int ffail(int code, const std::string& msg) { g_fit_err = msg; return code; }

long long jround(double x) { return (long long)std::nearbyint(x); }   // Julia round(): ties to even

enum Op : long long {
  OP_CREATE = 0, OP_INIT = 1, OP_RUN = 2, OP_SET_ROW = 3, OP_COPY = 4, OP_WINDOW = 5, OP_BLOCKS = 6,
  OP_PSRF_TRACE = 7, OP_PSRF_STREAM = 8, OP_PSRF_BLOCKS = 9, OP_ESS_WINDOW = 10
};

struct Ops {
  virtual ~Ops() {}
  virtual int create(long long trace_rows, bool gx_all, int full_chains) = 0;
  virtual int init() = 0;
  virtual int run(long long n) = 0;
  virtual int set_row(long long r) = 0;
  virtual int copy(long long dst, long long src, long long cnt) = 0;
  virtual int iteration(long long* it) = 0;
  virtual int window(long long first, long long len) = 0;
  virtual int blocks(long long first, long long blk, int nb) = 0;
  virtual int ess_window(long long first, long long len) = 0;
  // mode 0: rows [a, a + b) of the traces; 1: the streamed window; 2: blocks [a, a + b).  Outputs max R-hat (NaN
  // propagates, like Julia's max(v...)).
  virtual int psrf(int mode, long long a, long long b, double* max_xi, double* max_gamma) = 0;
};

// run! (src/gibbs.jl:849-864) as device run segments: rows first_index .. (1-based) with the purge_burn ring
int run_rows(Ops& o, long long first_index, long long nburn, long long total, long long purge, long long capacity) {
  long long j = first_index, seg_start = j, seg_len = 0;
  for (long long i = first_index; i <= total; ++i) {
    if (j > capacity)
      // e.g. purge_burn = 1, or a purge_burn that does not divide nburn after the reference's normalisation: the ring
      // is not back at row purge_burn when burn-in ends and the retained rows run past the table
      return ffail(BNR_EINVAL, "row index beyond the state table (the reference raises a BoundsError for this "
                               "nburn / nsamples / purge_burn combination)");
    ++seg_len;
    if (purge > 0 && i < nburn && j == purge + 1) {
      if (int r = o.set_row(seg_start - 1)) return r;
      if (int r = o.run(seg_len)) return r;
      if (int r = o.copy(0, j - 1, 1)) return r;          // copy_table!(state, 1, j)
      j = 1;
      seg_start = 2; seg_len = 0;
    }
    ++j;
  }
  if (seg_len) {
    if (int r = o.set_row(seg_start - 1)) return r;
    if (int r = o.run(seg_len)) return r;
  }
  return 0;
}

long long normalise_purge(long long purge, long long nburn) {           // src/gibbs.jl:930-936
  if (purge > 0 && purge < nburn) {
    if (nburn % purge != 0) purge = purge - (nburn % purge);
    return purge;
  }
  return 0;
}

struct Outcome {
  long long tot_generated = 0, burn_in = 0, sampled = 0, rows = 0, n_psrf = 0;
  bool streamed = false;
};

// arm the streaming moments (and ESS statistics) for the last nsamp of the next `new_sweeps` sweeps
int stream_last(Ops& o, long long new_sweeps, long long nsamp, bool ess) {
  long long it = 0;
  if (int r = o.iteration(&it)) return r;
  const long long first = it + new_sweeps - nsamp + 1;
  if (int r = o.window(first, nsamp)) return r;
  if (ess) return o.ess_window(first, nsamp);
  return 0;
}

// generate_samples! (src/gibbs.jl:897-1020)
int fit_traditional(Ops& o, const bnr_fit_params& p, Outcome& out) {
  const long long nburn = p.nburn, nsamp = p.nsamples, total = nburn + nsamp, maxburn = nburn + nsamp;
  const long long purge = normalise_purge(p.purge_burn, nburn);
  const long long tot_save = purge > 0 ? nsamp + purge : total;
  // R-hat needs the retained draws of EVERY chain.  Whenever those are always the last nsamp generated sweeps, in
  // order, their split-half moments are streamed on the device and only chain 1 keeps a trace.  Without the purge
  // ring that holds iff nburn >= nsamp (the extension round moves total - nburn rows and regenerates nburn); with the
  // ring the rows nb+1 .. nb+nsamp are the last nsamp sweeps only when the ring never wraps inside them, i.e. when
  // the retained block is written in one piece after the last wrap: nsamp + purge <= nburn and nburn % purge == 0.
  const bool streamed = nburn >= nsamp && nsamp >= 1 &&
                        (purge == 0 || (nsamp + purge <= nburn && nburn % purge == 0 && nsamp % purge == 0));
  const bool ess = p.ess_max_lag > 0 && streamed;
  if (int r = o.create(tot_save, !streamed, p.return_state == BNR_STATE_FULL ? 1 : 0)) return r;
  if (int r = o.init()) return r;
  if (streamed)
    if (int r = stream_last(o, total - 1, nsamp, ess)) return r;
  if (int r = run_rows(o, 2, nburn, total, purge, tot_save)) return r;
  const long long nb = purge > 0 ? purge : nburn;
  long long tot_generated = nburn + nsamp;
  double mx = 0, mg = 0;
  if (int r = o.psrf(streamed ? 1 : 0, nb, nsamp, &mx, &mg)) return r;
  ++out.n_psrf;
  if (p.verbose) fprintf(stderr, "%lld samples generated. Max PSRF XI: %.2f. Max PSRF Gamma: %.2f\n", tot_generated, mx, mg);
  // (NaN > cutoff is false: a NaN R-hat ends this loop, as in the reference)
  while ((mx > p.psrf_cutoff || mg > p.psrf_cutoff) && tot_generated < maxburn + nsamp) {
    long long num2move;
    if (purge > 0) num2move = (nsamp + purge <= nburn) ? 1 : nsamp + purge - nburn;
    else num2move = total - nburn;
    if (int r = o.copy(0, tot_save - num2move, num2move)) return r;
    const long long a_total = num2move > 1 ? num2move + nburn : nburn;
    if (streamed)
      if (int r = stream_last(o, a_total - num2move, nsamp, ess)) return r;
    if (int r = run_rows(o, num2move + 1, nburn > nsamp ? nburn - nsamp + num2move : 0, a_total, purge, tot_save)) return r;
    tot_generated += a_total - num2move;
    if (int r = o.psrf(streamed ? 1 : 0, nb, nsamp, &mx, &mg)) return r;
    ++out.n_psrf;
    if (p.verbose)
      fprintf(stderr, "%lld samples generated. Max PSRF XI: %.3f. Max PSRF Gamma: %.3f\n", tot_generated, mx, mg);
  }
  out.tot_generated = tot_generated; out.burn_in = nb; out.sampled = nsamp; out.rows = tot_save; out.streamed = streamed;
  return 0;
}

// generate_samples_dbl! (src/gibbs.jl:1051-1198)
int fit_doubling(Ops& o, const bnr_fit_params& p, Outcome& out) {
  const long long mingen = p.mingen, maxgen = p.maxgen;
  const long long nburn = jround(mingen / 2.0);
  long long nsamp = mingen - nburn;
  const long long total = nburn + nsamp;
  const long long purge = normalise_purge(p.purge_burn, nburn);
  const long long tot_save = purge > 0 ? nsamp + purge : total;
  const long long halfburn = jround(mingen / 2.0);
  long long rounds = 0;
  if (maxgen > total) rounds = (maxgen - total + mingen - 1) / (mingen > 0 ? mingen : 1);
  long long capacity = nsamp + (rounds + 1) * halfburn + halfburn;
  if (capacity < tot_save) capacity = tot_save;
  // The retained window grows by mingen/2 draws per round.  When mingen is a multiple of 4 every window and every
  // split half is a whole number of blocks of mingen/4 sweeps: per-block moments are kept on the device and merged, and
  // only chain 1 keeps a trace.
  const bool blocked = mingen % 4 == 0 && mingen >= 8 && purge == 0;
  const long long blk = mingen / 4;
  if (int r = o.create(capacity, !blocked, p.return_state == BNR_STATE_FULL ? 1 : 0)) return r;
  if (blocked)
    if (int r = o.blocks(0, blk, (int)(4 * (rounds + 1)))) return r;
  if (int r = o.init()) return r;
  if (int r = run_rows(o, 2, nburn, total, purge, tot_save)) return r;
  const long long nb = purge > 0 ? purge : nburn;
  long long tot_generated = total, tot_samples = nsamp, tot_sze = tot_save, k = 0;
  double mx = 0, mg = 0;
  auto psrf = [&]() -> int {
    ++out.n_psrf;
    if (blocked) return o.psrf(2, 2 * (k + 1), 2 * (k + 1), &mx, &mg);
    return o.psrf(0, nb, nsamp, &mx, &mg);
  };
  if (int r = psrf()) return r;
  if (p.verbose) fprintf(stderr, "%lld samples generated. Max PSRF XI: %.3f. Max PSRF Gamma: %.3f\n", tot_generated, mx, mg);
  while ((mx > p.psrf_cutoff || mg > p.psrf_cutoff || std::isnan(mx) || std::isnan(mg)) && tot_generated < maxgen) {
    const long long num2move = tot_samples;
    tot_samples += halfburn;
    nsamp = tot_samples;
    const long long new_save = tot_samples + halfburn;
    if (int r = o.copy(0, tot_sze - num2move, num2move)) return r;
    if (int r = run_rows(o, num2move + 1, 0, new_save, purge, new_save)) return r;
    tot_sze = new_save;
    tot_generated += mingen;
    ++k;
    if (int r = psrf()) return r;
    if (p.verbose)
      fprintf(stderr, "%lld samples generated. Max PSRF XI: %.3f. Max PSRF Gamma: %.3f\n", tot_generated, mx, mg);
  }
  out.tot_generated = tot_generated; out.burn_in = nb; out.sampled = nsamp; out.rows = tot_sze; out.streamed = blocked;
  return 0;
}

int fit_loops(Ops& o, const bnr_fit_params& p, Outcome& out) {
  if (p.mingen > 0 && p.maxgen > 0) return fit_doubling(o, p, out);      // src/gibbs.jl:744-750
  return fit_traditional(o, p, out);
}

// ------------------------------------------------------------------------------------------------------------------
// PlanOps: the operation log of a fit whose PSRF maxima are given
// ------------------------------------------------------------------------------------------------------------------
struct PlanOps : Ops {
  const double* psrf_max; int n_psrf; int used = 0;
  std::vector<long long> log;
  long long sweeps = 0;
  void put(long long op, long long a = 0, long long b = 0, long long c = 0) { log.insert(log.end(), {op, a, b, c}); }
  int create(long long rows, bool gx_all, int full) override { put(OP_CREATE, rows, gx_all, full); return 0; }
  int init() override { put(OP_INIT); sweeps = 0; return 0; }
  int run(long long n) override { put(OP_RUN, n); sweeps += n; return 0; }
  int set_row(long long r) override { put(OP_SET_ROW, r); return 0; }
  int copy(long long d, long long s, long long c) override { put(OP_COPY, d, s, c); return 0; }
  int iteration(long long* it) override { *it = sweeps; return 0; }
  int window(long long f, long long l) override { put(OP_WINDOW, f, l); return 0; }
  int blocks(long long f, long long b, int nb) override { put(OP_BLOCKS, f, b, nb); return 0; }
  int ess_window(long long f, long long l) override { put(OP_ESS_WINDOW, f, l); return 0; }
  int psrf(int mode, long long a, long long b, double* mx, double* mg) override {
    put(mode == 0 ? OP_PSRF_TRACE : (mode == 1 ? OP_PSRF_STREAM : OP_PSRF_BLOCKS), a, b);
    const double v = used < n_psrf ? psrf_max[used] : 0.0;
    ++used;
    *mx = v; *mg = v;
    return 0;
  }
};

// ------------------------------------------------------------------------------------------------------------------
// NCCL, loaded at run time (libnccl.so.2: the copy a host process already has loaded -- e.g. torch's -- or the system one)
// ------------------------------------------------------------------------------------------------------------------
struct Nccl {
  void* lib = nullptr;
  int (*CommInitAll)(void**, int, const int*) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
  Nccl() {
    if (getenv("BNR_EXCHANGE") && !strcmp(getenv("BNR_EXCHANGE"), "peer")) return;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) return;
    CommInitAll = (int (*)(void**, int, const int*))dlsym(lib, "ncclCommInitAll");
    CommDestroy = (int (*)(void*))dlsym(lib, "ncclCommDestroy");
    AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(lib, "ncclAllGather");
    GroupStart = (int (*)())dlsym(lib, "ncclGroupStart");
    GroupEnd = (int (*)())dlsym(lib, "ncclGroupEnd");
    GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
    ok = CommInitAll && CommDestroy && AllGather && GroupStart && GroupEnd;
  }
};
Nccl& nccl() { static Nccl n; return n; }
constexpr int NCCL_DOUBLE = 8;     // ncclFloat64

#define CKF(call)                                                                                  \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) return ffail(BNR_ECUDA, std::string(#call) + ": " + cudaGetErrorString(_e)); \
  } while (0)
#define BN(call)                                                                                   \
  do {                                                                                             \
    int _r = (call);                                                                               \
    if (_r != BNR_OK) return ffail(_r, std::string(#call) + ": " + bnr_last_error());               \
  } while (0)

}  // namespace

// ------------------------------------------------------------------------------------------------------------------
// DeviceOps / the result object
// ------------------------------------------------------------------------------------------------------------------
struct bnr_fit_result {
  bnr_fit_params p;
  std::vector<bnr_handle*> h;          // the handles of every fold, fold by fold; h[0] holds chain 1
  std::vector<int> dev;                // the device of each handle
  std::vector<cudaStream_t> xs;        // exchange streams
  std::vector<void*> comms;            // NCCL communicators (empty: single device or peer-copy exchange)
  std::vector<double*> gbuf;           // per device: gathered buffer
  size_t gbuf_doubles = 0;
  double* xbuf = nullptr;              // device 0: buffer gathered across processes
  size_t xbuf_doubles = 0;
  int V = 0, q = 0, C = 0;
  Outcome out;
  // the handles whose chains pool their statistics: an ordinary fit is one fold over all its handles that holds
  // nothing out; bnr_fit_kfold makes one fold of one handle per held-out set
  struct Fold {
    int first = 0, handles = 1;        // its handles h[first .. first + handles)
    std::vector<int> held;             // the observations it holds out, in original order
    std::vector<double> rhat_xi, rhat_gamma;   // the R-hat of the last PSRF step over its chains
  };
  std::vector<Fold> folds;
  // rhat_*: the element-wise maximum over the folds (NaN wins)
  std::vector<double> rhat_xi, rhat_gamma, s_mean, s_lo, s_hi, s_xi, ess_xi, ess_gamma;
  bool summary_ok = false, ess_ok = false;
  // a per-row table pooled over the chains of each fold after the fit
  struct Pooled {
    const char* what;
    std::vector<int> width;            // per handle: doubles per row (empty: not requested)
    std::vector<double*> exp;          // per handle: the retained rows of its chains, [chain][row][width]
    bool ok = false;                   // its summary was computed
  };
  Pooled pred = {"predictions"};       // predictions for new networks (bnr_fit_predict), width m
  Pooled ll = {"log-likelihood"};      // pointwise log-likelihood for PSIS-LOO / WAIC (bnr_fit_loo), width n
  Pooled held = {"held-out log densities"};   // K-fold (bnr_fit_kfold): as wide as the fold holds out
  std::vector<double> elpd;            // K-fold: [n] elpd_kfold in original order
  bool kfold() const { return !held.width.empty(); }
  int pmode = 0;
  std::vector<double> p_mean, p_lo, p_hi;
  std::vector<double> l_pw[5];         // elpd_loo, p_loo, pareto_k, elpd_waic, p_waic per observation
  int gamma_mode = 0;
  int status_or = 0;
  int exchange = 0;                    // bnr_fit_info.exchange
  ~bnr_fit_result() {
    for (size_t d = 0; d < h.size(); ++d) {
      if (d < dev.size()) cudaSetDevice(dev[d]);
      if (d < gbuf.size() && gbuf[d]) cudaFree(gbuf[d]);
      for (Pooled* t : {&pred, &ll, &held})
        if (d < t->exp.size() && t->exp[d]) cudaFree(t->exp[d]);
      if (d < xs.size() && xs[d]) cudaStreamDestroy(xs[d]);
    }
    if (xbuf) { cudaSetDevice(dev[0]); cudaFree(xbuf); }
    if (!comms.empty() && nccl().ok)
      for (void* c : comms) if (c) nccl().CommDestroy(c);
    for (bnr_handle* hh : h) if (hh) bnr_destroy(hh);
  }
};

namespace {

// wall-clock accounting of a fit's phases (printed when BNR_FIT_TIMING is set): where the fixed cost of a short fit goes
struct PhaseClock {
  double t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
  struct Scope {
    PhaseClock& c; int i; double t0;
    Scope(PhaseClock& c_, int i_) : c(c_), i(i_), t0(now()) {}
    ~Scope() { c.t[i] += now() - t0; }
  };
};
enum { PH_CREATE = 0, PH_INIT, PH_RUN, PH_COPY, PH_PSRF, PH_SUMMARY, PH_ESS, PH_MISC };

// Julia's maximum(v): NaN if any element is NaN
double jmax(const std::vector<double>& v) {
  double m = -INFINITY;
  for (double x : v) { if (std::isnan(x)) return (double)NAN; if (x > m) m = x; }
  return m;
}

// one handle of a fit: the rows it trains on and, in K-fold cross-validation, the rows its fold holds out
struct Entry {
  int fold = 0, n = 0;
  const double* X = nullptr; const double* y = nullptr;   // training rows: the caller's X and y, or Xt and yt
  std::vector<double> Xt, yt, Xh, yh;                     // K-fold: the fold's rows, freed once its handle holds them
};

// a refused cudaMalloc of one of the buffers of a pooled table
int refuse(const char* buf, const char* what, size_t doubles) {
  cudaGetLastError();
  return ffail(BNR_ENOMEM, std::string("cannot allocate the ") + buf + " of the " + what + " (" +
                               std::to_string(doubles * sizeof(double)) + " bytes)");
}

struct DeviceOps : Ops {
  using Fold = bnr_fit_result::Fold;
  using Pooled = bnr_fit_result::Pooled;
  bnr_fit_result& R;
  std::vector<Entry> E;                // one per handle of R.h
  const double* X_new;
  PhaseClock clk;
  explicit DeviceOps(bnr_fit_result& r, const double* X_new_) : R(r), X_new(X_new_) {}
  int chains(const Fold& f) const { return R.C * f.handles * (R.p.ext_world > 1 ? R.p.ext_world : 1); }
  // the chains of some fold meet in gathers: it spans several handles (only an ordinary fit's one fold can), or the
  // fit spans several processes
  bool gathers() const { return R.h.size() > R.folds.size() || R.p.ext_world > 1; }

  int create(long long rows, bool gx_all, int full) override {
    PhaseClock::Scope sc(clk, PH_CREATE);
    const int H = (int)E.size(), nd = R.p.n_devices > 0 ? R.p.n_devices : 1;
    R.h.assign(H, nullptr); R.dev.assign(H, 0); R.xs.assign(H, nullptr); R.gbuf.assign(H, nullptr);
    for (Pooled* t : {&R.pred, &R.ll, &R.held}) t->exp.assign(t->width.size(), nullptr);
    R.V = R.p.base.V; R.q = R.V * (R.V + 1) / 2; R.C = R.p.base.num_chains;
    const int rank = R.p.ext_world > 1 ? R.p.ext_rank : 0;
    for (int i = 0; i < H; ++i) {
      Entry& e = E[i];
      bnr_params bp = R.p.base;
      bp.n = e.n;
      bp.device = R.p.base.device + i % nd;
      bp.chain_offset = R.p.base.chain_offset + (rank * H + i) * bp.num_chains;
      bp.trace_rows = rows;
      bp.trace_gamma_xi_all = gx_all ? 1 : 0;
      // a fold's chain 1 (first local chain of its first handle on rank 0 ... every rank keeps its own first chain) is
      // the one Results / Summary read; its other handles need traces only when R-hat is taken from trace rows
      const bool first = i == R.folds[e.fold].first;
      bp.trace_full_chains = first ? full : 0;
      bp.trace_gamma_xi_chains = first ? 1 : 0;
      if (!first && !gx_all) bp.trace_rows = 0;
      R.dev[i] = bp.device;
      BN(bnr_create(&bp, e.X, e.y, &R.h[i]));
      for (std::vector<double>* v : {&e.Xt, &e.yt}) std::vector<double>().swap(*v);
      // its tables before the next handle: creating every handle first made the create phase of a K-fold run with
      // all folds on one device 10 - 20 % slower (B200, 1000 W power limit)
      if (int r = create_tables(i, rows)) return r;
    }
    int32_t gm = 0;
    BN(bnr_gamma_mode(R.h[0], &gm));
    R.gamma_mode = gm;
    if (gathers()) {
      for (int i = 0; i < H; ++i) {
        CKF(cudaSetDevice(R.dev[i]));
        CKF(cudaStreamCreateWithFlags(&R.xs[i], cudaStreamNonBlocking));
      }
      if (H > 1 && nccl().ok) {
        R.comms.assign(H, nullptr);
        const int rc = nccl().CommInitAll(R.comms.data(), H, R.dev.data());
        if (rc != 0) {
          R.comms.clear();
          return ffail(BNR_ECUDA, std::string("ncclCommInitAll: ") + (nccl().GetErrorString ? nccl().GetErrorString(rc) : "error"));
        }
        R.exchange = 1;                                 // NCCL
      } else if (H > 1) {
        R.exchange = 2;                                 // peer copies
      }
    }
    return create_pooled(rows);
  }

  // handle i's prediction, log-likelihood and held-out tables of `rows` rows and their export buffers.  With the
  // pooled buffers of create_pooled they are all allocated before the first sweep: a fit that cannot hold them fails
  // here, not after the sampling
  int create_tables(int i, long long rows) {
    if (!R.pred.width.empty()) BN(bnr_set_predictors(R.h[i], R.pred.width[i], X_new, rows, R.pmode));
    if (!R.ll.width.empty()) BN(bnr_set_loglik(R.h[i], rows));
    if (R.kfold()) {
      Entry& e = E[i];
      BN(bnr_set_heldout(R.h[i], R.held.width[i], e.Xh.data(), e.yh.data(), rows));
      for (std::vector<double>* v : {&e.Xh, &e.yh}) std::vector<double>().swap(*v);
    }
    for (Pooled* t : {&R.pred, &R.ll, &R.held}) {
      if (t->width.empty()) continue;
      const size_t local = (size_t)R.C * rows * t->width[i];
      CKF(cudaSetDevice(R.dev[i]));
      if (cudaMalloc((void**)&t->exp[i], local * sizeof(double)) != cudaSuccess) {
        t->exp[i] = nullptr;
        return refuse("export buffer", t->what, local);
      }
    }
    return 0;
  }

  // the pooled buffers of the all-gather, sized for the widest table
  int create_pooled(long long rows) {
    const int H = (int)R.h.size(), world = R.p.ext_world > 1 ? R.p.ext_world : 1;
    int width = 0;
    const char* what = nullptr;
    for (Pooled* t : {&R.pred, &R.ll, &R.held}) {
      if (t->width.empty()) continue;
      width = std::max(width, *std::max_element(t->width.begin(), t->width.end()));
      what = t->what;
    }
    const size_t local = (size_t)R.C * rows * width;
    if (width > 0 && gathers()) {
      // gather_local / gather_ext reuse these buffers (they only grow)
      for (int i = 0; i < H; ++i) {
        CKF(cudaSetDevice(R.dev[i]));
        if (R.gbuf[i]) CKF(cudaFree(R.gbuf[i]));
        R.gbuf[i] = nullptr;
        if (cudaMalloc((void**)&R.gbuf[i], local * H * sizeof(double)) != cudaSuccess) {
          R.gbuf[i] = nullptr; R.gbuf_doubles = 0;
          return refuse("pooled buffer", what, local * H);
        }
      }
      R.gbuf_doubles = local * H;
      if (world > 1) {
        CKF(cudaSetDevice(R.dev[0]));
        if (cudaMalloc((void**)&R.xbuf, local * H * world * sizeof(double)) != cudaSuccess) {
          R.xbuf = nullptr;
          return refuse("pooled buffer", what, local * H * world);
        }
        R.xbuf_doubles = local * H * world;
      }
    }
    return 0;
  }

  // the retained rows of every chain of fold f in a pooled table, in global-chain order on the fold's first device
  // (*all), each handle's exported through export_rows
  int pool(const Outcome& o, const Fold& f, const Pooled& t, int (*export_rows)(bnr_handle*, int64_t, int64_t, double*),
           const double** all) {
    for (int i = f.first; i < f.first + f.handles; ++i) BN(export_rows(R.h[i], o.burn_in, o.sampled, t.exp[i]));
    *all = t.exp[f.first];
    if (f.handles > 1 || R.p.ext_world > 1) {
      const size_t cnt = (size_t)R.C * o.sampled * t.width[f.first];
      std::vector<const double*> src(t.exp.begin() + f.first, t.exp.begin() + f.first + f.handles);
      if (int r = gather_local(src, cnt)) return r;
      if (int r = gather_ext(cnt * f.handles, all)) return r;
    }
    return 0;
  }

  // Summary statistics of chain 1 on the device (src/gibbs.jl:1221-1236: lw / hi with Julia's round)
  int summary(const Outcome& o) {
    PhaseClock::Scope sc(clk, PH_SUMMARY);
    const long long nsamp = o.sampled;
    const double lower = (100 - (R.p.interval > 0 ? R.p.interval : 95)) / 200.0;
    const long long lw = jround(nsamp * lower), hi = jround(nsamp * (1.0 - lower));
    if (lw < 1 || hi > nsamp) return 0;
    R.s_mean.assign(R.q, 0); R.s_lo.assign(R.q, 0); R.s_hi.assign(R.q, 0); R.s_xi.assign(R.V, 0);
    if (bnr_summary(R.h[0], 0, o.burn_in, nsamp, lw, hi, R.s_mean.data(), R.s_lo.data(), R.s_hi.data(),
                    R.s_xi.data()) != BNR_OK)
      return ffail(BNR_ECUDA, std::string("bnr_summary: ") + bnr_last_error());
    R.summary_ok = true;
    return 0;
  }

  // pooled mean and order statistics of the predictions
  int predictions(const Outcome& o) {
    const Fold& f = R.folds[0];
    const long long N = (long long)chains(f) * o.sampled;
    const double lower = (100 - (R.p.interval > 0 ? R.p.interval : 95)) / 200.0;
    const long long lw = jround(N * lower), hi = jround(N * (1.0 - lower));
    if (o.sampled < 1 || lw < 1 || hi > N) return 0;
    const double* all = nullptr;
    if (int r = pool(o, f, R.pred, bnr_export_predictions, &all)) return r;
    const int m = R.pred.width[0];
    R.p_mean.assign(m, 0); R.p_lo.assign(m, 0); R.p_hi.assign(m, 0);
    BN(bnr_prediction_summary(R.dev[0], all, N, m, lw, hi, R.p_mean.data(), R.p_lo.data(), R.p_hi.data()));
    R.pred.ok = true;
    return 0;
  }

  // pooled PSIS-LOO and WAIC of the log-likelihood
  int loo(const Outcome& o) {
    const Fold& f = R.folds[0];
    const long long N = (long long)chains(f) * o.sampled;
    if (N < 2) return 0;
    const double* all = nullptr;
    if (int r = pool(o, f, R.ll, bnr_export_loglik, &all)) return r;
    const int n = R.ll.width[0];
    for (auto& v : R.l_pw) v.assign(n, 0);
    BN(bnr_loo_summary(R.dev[0], all, N, n, R.l_pw[0].data(), R.l_pw[1].data(), R.l_pw[2].data(), R.l_pw[3].data(),
                       R.l_pw[4].data()));
    R.ll.ok = true;
    return 0;
  }

  // elpd_kfold of every held-out observation: the log-mean-exp of its fold's retained rows of all chains
  int heldout(const Outcome& o) {
    R.elpd.assign(R.p.base.n, NAN);
    for (const Fold& f : R.folds) {
      const long long N = (long long)chains(f) * o.sampled;
      if (N < 1) return 0;
      const double* all = nullptr;
      if (int r = pool(o, f, R.held, bnr_export_predictions, &all)) return r;
      std::vector<double> lpd(f.held.size());
      BN(bnr_lpd_summary(R.dev[f.first], all, N, (int32_t)lpd.size(), lpd.data()));
      for (size_t j = 0; j < lpd.size(); ++j) R.elpd[f.held[j]] = lpd[j];
    }
    R.held.ok = true;
    return 0;
  }
  int init() override { PhaseClock::Scope sc(clk, PH_INIT); for (auto* h : R.h) BN(bnr_init_state(h)); return 0; }
  int run(long long n) override {
    PhaseClock::Scope sc(clk, PH_RUN);
    for (auto* h : R.h) BN(bnr_run(h, n));                 // asynchronous: all devices advance together
    for (auto* h : R.h) BN(bnr_sync(h));
    return 0;
  }
  int set_row(long long r) override { for (auto* h : R.h) BN(bnr_set_trace_row(h, r)); return 0; }
  int copy(long long d, long long s, long long c) override {
    PhaseClock::Scope sc(clk, PH_COPY);
    for (auto* h : R.h) BN(bnr_copy_trace_rows(h, d, s, c));
    return 0;
  }
  int iteration(long long* it) override { int64_t v = 0; BN(bnr_iteration(R.h[0], &v)); *it = v; return 0; }
  int window(long long f, long long l) override { for (auto* h : R.h) BN(bnr_set_moment_window(h, f, l)); return 0; }
  int blocks(long long f, long long b, int nb) override { for (auto* h : R.h) BN(bnr_set_moment_blocks(h, f, b, nb)); return 0; }
  int ess_window(long long f, long long l) override {
    for (auto* h : R.h) BN(bnr_ess_stream_window(h, R.p.ess_max_lag, f, l));
    return 0;
  }

  int ensure_gbuf(size_t doubles) {
    if (doubles <= R.gbuf_doubles) return 0;
    for (size_t d = 0; d < R.h.size(); ++d) {
      CKF(cudaSetDevice(R.dev[d]));
      if (R.gbuf[d]) CKF(cudaFree(R.gbuf[d]));
      R.gbuf[d] = nullptr;
      CKF(cudaMalloc((void**)&R.gbuf[d], doubles * sizeof(double)));
    }
    R.gbuf_doubles = doubles;
    return 0;
  }
  // every handle contributes src[d] (cnt doubles, device memory); afterwards gbuf[0] holds [handles][cnt] in handle
  // order (with NCCL every device holds it).  A fold that gathers spans every handle: see gathers()
  int gather_local(const std::vector<const double*>& src, size_t cnt) {
    const int nd = (int)R.h.size();
    if (int r = ensure_gbuf(cnt * nd)) return r;
    if (nd > 1 && !R.comms.empty()) {
      nccl().GroupStart();
      for (int d = 0; d < nd; ++d) {
        const int rc = nccl().AllGather(src[d], R.gbuf[d], cnt, NCCL_DOUBLE, R.comms[d], R.xs[d]);
        if (rc != 0) { nccl().GroupEnd(); return ffail(BNR_ECUDA, "ncclAllGather failed"); }
      }
      if (nccl().GroupEnd() != 0) return ffail(BNR_ECUDA, "ncclGroupEnd failed");
      for (int d = 0; d < nd; ++d) { CKF(cudaSetDevice(R.dev[d])); CKF(cudaStreamSynchronize(R.xs[d])); }
    } else {
      CKF(cudaSetDevice(R.dev[0]));
      for (int d = 0; d < nd; ++d)
        CKF(cudaMemcpyPeer(R.gbuf[0] + (size_t)d * cnt, R.dev[0], src[d], R.dev[d], cnt * sizeof(double)));
    }
    return 0;
  }
  // all-gather of gbuf[0][0 .. cnt) across the processes that call bnr_fit together; result pointer in *all
  int gather_ext(size_t cnt, const double** all) {
    *all = R.gbuf[0];
    if (R.p.ext_world <= 1) return 0;
    if (!R.p.allgather) return ffail(BNR_EINVAL, "ext_world > 1 needs an allgather callback");
    const size_t need = cnt * R.p.ext_world;
    CKF(cudaSetDevice(R.dev[0]));
    if (need > R.xbuf_doubles) {
      if (R.xbuf) CKF(cudaFree(R.xbuf));
      R.xbuf = nullptr;
      CKF(cudaMalloc((void**)&R.xbuf, need * sizeof(double)));
      R.xbuf_doubles = need;
    }
    const int rc = R.p.allgather(R.p.allgather_ctx, R.dev[0], R.gbuf[0], R.xbuf, (int64_t)cnt);
    if (rc != 0) return ffail(BNR_ECUDA, "the caller's all-gather callback failed");
    *all = R.xbuf;
    return 0;
  }

  int psrf(int mode, long long a, long long b, double* mx, double* mg) override {
    PhaseClock::Scope sc(clk, PH_PSRF);
    R.rhat_xi.assign(R.V, NAN); R.rhat_gamma.assign(R.q, NAN);
    for (Fold& f : R.folds) { f.rhat_xi.assign(R.V, NAN); f.rhat_gamma.assign(R.q, NAN); }
    if (mode != 2 && b / 2 < 2) { *mx = NAN; *mg = NAN; return 0; }
    for (auto* h : R.h) {
      if (mode == 0) BN(bnr_moments_from_trace(h, a, b));
      if (mode == 2) BN(bnr_moments_from_blocks(h, (int32_t)a, (int32_t)b));
    }
    int64_t half = 0;
    BN(bnr_moment_half_len(R.h[0], &half));
    if (half < 2) { *mx = NAN; *mg = NAN; return 0; }
    // element-wise maximum over the folds; NaN wins, so that jmax of it is jmax over all folds' values
    auto fold_max = [](std::vector<double>& acc, const std::vector<double>& v, bool first) {
      for (size_t i = 0; i < v.size(); ++i)
        if (first || std::isnan(v[i]) || (!std::isnan(acc[i]) && v[i] > acc[i])) acc[i] = v[i];
    };
    for (size_t k = 0; k < R.folds.size(); ++k) {
      Fold& f = R.folds[k];
      if (f.handles == 1 && R.p.ext_world <= 1) {
        BN(bnr_rhat(R.h[f.first], f.rhat_xi.data(), f.rhat_gamma.data()));
      } else {
        std::vector<const double*> src(f.handles);
        int64_t cnt = 0;
        for (int d = 0; d < f.handles; ++d) {
          double* ptr = nullptr;
          BN(bnr_moments_device(R.h[f.first + d], &ptr, &cnt));
          src[d] = ptr;
        }
        if (int r = gather_local(src, (size_t)cnt)) return r;
        const double* all = nullptr;
        if (int r = gather_ext((size_t)cnt * f.handles, &all)) return r;
        BN(bnr_rhat_from_moments(R.dev[f.first], all, chains(f), R.V, R.q, half, f.rhat_xi.data(),
                                 f.rhat_gamma.data()));
      }
      fold_max(R.rhat_xi, f.rhat_xi, k == 0);
      fold_max(R.rhat_gamma, f.rhat_gamma, k == 0);
    }
    *mx = jmax(R.rhat_xi); *mg = jmax(R.rhat_gamma);
    return 0;
  }

  // ESS of the retained draws from the streamed statistics (traditional scheme with streamed moments) or from the
  // traces of all chains
  int ess(const Outcome& o) {
    PhaseClock::Scope sc(clk, PH_ESS);
    const int L = R.p.ess_max_lag;
    if (L <= 0 || o.sampled < 4) return 0;
    if (o.streamed && !(R.p.mingen > 0 && R.p.maxgen > 0)) {
      for (auto* h : R.h) BN(bnr_ess_stream_finish(h));
    } else if (!o.streamed) {
      for (auto* h : R.h) BN(bnr_ess_accumulate(h, o.burn_in, o.sampled, L));
    } else {
      return 0;                                         // doubling scheme with block moments: no ESS statistics
    }
    std::vector<const double*> sa(R.h.size()), sm(R.h.size());
    int64_t na = 0, nm = 0;
    int32_t lag = 0;
    for (size_t d = 0; d < R.h.size(); ++d) {
      double *pa = nullptr, *pm = nullptr;
      BN(bnr_ess_device(R.h[d], &pa, &na, &pm, &nm, &lag));
      sa[d] = pa; sm[d] = pm;
    }
    R.ess_xi.assign(R.V, NAN); R.ess_gamma.assign(R.q, NAN);
    const int parts = (int)R.h.size() * (R.p.ext_world > 1 ? R.p.ext_world : 1);
    if (parts == 1) {
      BN(bnr_ess_from_stats(R.dev[0], sa[0], 1, sm[0], R.C, R.V, R.q, o.sampled, lag, R.ess_xi.data(), R.ess_gamma.data()));
    } else {
      // two exchanges: autocovariance sums, then chain means (kept in a private copy, the gather buffer is reused)
      if (int r = gather_local(sa, (size_t)na)) return r;
      const double* all_a = nullptr;
      if (int r = gather_ext((size_t)na * R.h.size(), &all_a)) return r;
      double* keep = nullptr;
      const size_t abytes = (size_t)na * parts * sizeof(double);
      CKF(cudaSetDevice(R.dev[0]));
      CKF(cudaMalloc((void**)&keep, abytes));
      CKF(cudaMemcpy(keep, all_a, abytes, cudaMemcpyDeviceToDevice));
      int rc = gather_local(sm, (size_t)nm);
      const double* all_m = nullptr;
      if (!rc) rc = gather_ext((size_t)nm * R.h.size(), &all_m);
      if (!rc && bnr_ess_from_stats(R.dev[0], keep, parts, all_m, chains(R.folds[0]), R.V, R.q, o.sampled, lag,
                                    R.ess_xi.data(), R.ess_gamma.data()) != BNR_OK)
        rc = ffail(BNR_ECUDA, std::string("bnr_ess_from_stats: ") + bnr_last_error());
      cudaSetDevice(R.dev[0]);
      cudaFree(keep);
      if (rc) return rc;
    }
    R.ess_ok = true;
    return 0;
  }
};

int check_params(const bnr_fit_params* p) {
  if (!p) return ffail(BNR_EINVAL, "null parameters");
  const bool dbl = p->mingen > 0 && p->maxgen > 0;
  if (!dbl && (p->nburn < 0 || p->nsamples < 1)) return ffail(BNR_EINVAL, "need nburn >= 0 and nsamples >= 1");
  if (p->n_devices < 0 || p->purge_burn < 0) return ffail(BNR_EINVAL, "negative n_devices / purge_burn");
  if (p->ext_world > 1 && (p->ext_rank < 0 || p->ext_rank >= p->ext_world)) return ffail(BNR_EINVAL, "bad ext_rank");
  return 0;
}

}  // namespace

extern "C" const char* bnr_fit_last_error(void) { return g_fit_err.c_str(); }

extern "C" void bnr_fit_default_params(bnr_fit_params* p) {
  memset(p, 0, sizeof(*p));
  bnr_default_params(&p->base);
  p->nburn = 30000; p->nsamples = 20000;            // Fit! defaults (src/gibbs.jl:725)
  p->psrf_cutoff = 1.01;
  p->return_state = BNR_STATE_FULL;
  p->n_devices = 1;
  p->interval = 95;
}

extern "C" int bnr_fit_plan(const bnr_fit_params* p, const double* psrf_max, int32_t n_psrf, int64_t* ops,
                            int64_t cap_ops, int64_t* n_ops, bnr_fit_info* info) {
  if (int r = check_params(p)) return r;
  if (!n_ops || (n_psrf > 0 && !psrf_max)) return ffail(BNR_EINVAL, "null argument");
  PlanOps o;
  o.psrf_max = psrf_max; o.n_psrf = n_psrf;
  Outcome out;
  if (int r = fit_loops(o, *p, out)) return r;
  const long long n = (long long)o.log.size() / 4;
  *n_ops = n;
  if (ops) {
    if (cap_ops < n) return ffail(BNR_EINVAL, "operation buffer too small");
    for (size_t i = 0; i < o.log.size(); ++i) ops[i] = o.log[i];
  }
  if (info) {
    memset(info, 0, sizeof(*info));
    info->tot_generated = out.tot_generated; info->burn_in = out.burn_in; info->sampled = out.sampled;
    info->rows = out.rows; info->n_psrf = out.n_psrf; info->streamed = out.streamed ? 1 : 0;
  }
  return BNR_OK;
}

// the folds of bnr_fit_kfold: labels checked, training and held-out rows of every fold in original order, one handle
// per fold
static int kfold_split(const bnr_fit_params* p, const double* X, const double* y, int32_t K, const int32_t* fold,
                       bnr_fit_result* R, std::vector<Entry>& E) {
  const int n = p->base.n, V = p->base.V;
  const size_t q = (size_t)V * (V + 1) / 2;
  std::vector<int> cnt(K, 0);
  for (int i = 0; i < n; ++i) {
    if (fold[i] < 1 || fold[i] > K)
      return ffail(BNR_EINVAL, "fold label " + std::to_string(fold[i]) + " of observation " + std::to_string(i + 1) +
                                   " lies outside 1.." + std::to_string(K));
    ++cnt[fold[i] - 1];
  }
  for (int f = 0; f < K; ++f) {
    if (cnt[f] == 0) return ffail(BNR_EINVAL, "fold " + std::to_string(f + 1) + " holds no observation");
    if (cnt[f] == n) return ffail(BNR_EINVAL, "fold " + std::to_string(f + 1) + " leaves an empty training set");
  }
  R->folds.assign(K, {});
  R->held.width = cnt;
  E.assign(K, {});
  for (int f = 0; f < K; ++f) {
    Entry& e = E[f];
    R->folds[f].first = e.fold = f;
    e.n = n - cnt[f];
    for (int i = 0; i < n; ++i) {
      const bool held = fold[i] == f + 1;
      (held ? e.yh : e.yt).push_back(y[i]);
      if (held) R->folds[f].held.push_back(i);
    }
    // column by column: X is column-major, so both sides are read and written in order
    e.Xt.resize((size_t)e.n * q); e.Xh.resize((size_t)cnt[f] * q);
    double *dt = e.Xt.data(), *dh = e.Xh.data();
    for (size_t j = 0; j < q; ++j) {
      const double* col = X + (size_t)n * j;
      for (int i = 0; i < n; ++i) *(fold[i] == f + 1 ? dh++ : dt++) = col[i];
    }
    e.X = e.Xt.data(); e.y = e.yt.data();
  }
  return 0;
}

// bnr_fit, bnr_fit_predict (m > 0: predictions for the m rows of X_new), bnr_fit_loo (loo: PSIS-LOO and WAIC) and
// bnr_fit_kfold (K > 0: the folds of `fold`, each scored on the observations it holds out)
static int fit_entry(const char* name, const bnr_fit_params* p, const double* X, const double* y, int32_t m,
                     const double* X_new, int32_t mode, bool loo, int32_t K, const int32_t* fold,
                     bnr_fit_result** res_out) {
  if (m < 0) return ffail(BNR_EINVAL, "m must be >= 0");
  if (m > 0 && !X_new) return ffail(BNR_EINVAL, "null X_new");
  if (mode != BNR_PRED_MEAN && mode != BNR_PRED_PREDICTIVE) return ffail(BNR_EINVAL, "unknown prediction mode");
  if (int r = check_params(p)) return r;
  if (!X || !y || !res_out) return ffail(BNR_EINVAL, "null argument");
  if (p->base.nu < p->base.R)
    // the reference builds this ArgumentError without throwing it (src/gibbs.jl:901-902); the InverseWishart draw is
    // undefined for nu <= R - 1, so the engine refuses
    return ffail(BNR_EINVAL, "nu must not be smaller than R");
  bnr_fit_result* R = new bnr_fit_result();
  R->p = *p;
  R->pmode = mode;
  DeviceOps o(*R, X_new);
  int rc = 0;
  if (K > 0) {
    rc = kfold_split(p, X, y, K, fold, R, o.E);
  } else {
    // one fold over n_devices handles that share the caller's rows and hold nothing out
    const int nd = p->n_devices > 0 ? p->n_devices : 1;
    R->folds.assign(1, {});
    R->folds[0].handles = nd;
    o.E.assign(nd, {0, p->base.n, X, y});
    if (m > 0) R->pred.width.assign(nd, m);
    if (loo) R->ll.width.assign(nd, p->base.n);
  }
  const double t_start = PhaseClock::now();
  if (!rc) rc = fit_loops(o, *p, R->out);
  if (!rc && K == 0) rc = o.summary(R->out);
  if (!rc && m > 0) rc = o.predictions(R->out);
  if (!rc && loo) rc = o.loo(R->out);
  if (!rc && K > 0) rc = o.heldout(R->out);
  if (!rc) rc = o.ess(R->out);
  if (!rc) {
    std::vector<int32_t> st(R->C);
    for (auto* h : R->h) {
      if (bnr_status(h, st.data()) != BNR_OK) { rc = ffail(BNR_ECUDA, bnr_last_error()); break; }
      for (int v : st) R->status_or |= v;
    }
  }
  if (getenv("BNR_FIT_TIMING"))
    fprintf(stderr, "%s %.1f ms: create %.1f  init %.1f  run %.1f  row copies %.1f  psrf %.1f  summary %.1f  ess %.1f\n",
            name, 1e3 * (PhaseClock::now() - t_start), 1e3 * o.clk.t[PH_CREATE], 1e3 * o.clk.t[PH_INIT],
            1e3 * o.clk.t[PH_RUN], 1e3 * o.clk.t[PH_COPY], 1e3 * o.clk.t[PH_PSRF], 1e3 * o.clk.t[PH_SUMMARY],
            1e3 * o.clk.t[PH_ESS]);
  if (rc) {
    const std::string msg = g_fit_err;
    delete R;
    g_fit_err = msg;
    return rc;
  }
  *res_out = R;
  return BNR_OK;
}

extern "C" int bnr_fit(const bnr_fit_params* p, const double* X, const double* y, bnr_fit_result** res_out) {
  return fit_entry("bnr_fit", p, X, y, 0, nullptr, BNR_PRED_MEAN, false, 0, nullptr, res_out);
}

extern "C" int bnr_fit_predict(const bnr_fit_params* p, const double* X, const double* y, int32_t m,
                               const double* X_new, int32_t mode, bnr_fit_result** res_out) {
  return fit_entry("bnr_fit_predict", p, X, y, m, X_new, mode, false, 0, nullptr, res_out);
}

extern "C" int bnr_fit_loo(const bnr_fit_params* p, const double* X, const double* y, int32_t m, const double* X_new,
                           int32_t pred_mode, bnr_fit_result** res_out) {
  return fit_entry("bnr_fit_loo", p, X, y, m, X_new, pred_mode, true, 0, nullptr, res_out);
}

extern "C" int bnr_fit_kfold(const bnr_fit_params* p, const double* X, const double* y, int32_t K, const int32_t* fold,
                             bnr_fit_result** res_out) {
  if (int r = check_params(p)) return r;             // before the K-fold rules read p
  if (!fold) return ffail(BNR_EINVAL, "null argument");
  if (K < 2) return ffail(BNR_EINVAL, "K-fold cross-validation needs K >= 2 folds");
  if (p->base.n < 2) return ffail(BNR_EINVAL, "K-fold cross-validation needs n >= 2 observations");
  if (p->base.V < 1) return ffail(BNR_EINVAL, "V must be >= 1");
  if (p->ext_world > 1) return ffail(BNR_EINVAL, "K-fold cross-validation runs in one process (ext_world must be <= 1)");
  if (p->ess_max_lag > 0) return ffail(BNR_EINVAL, "K-fold cross-validation computes no ESS (ess_max_lag must be 0)");
  return fit_entry("bnr_fit_kfold", p, X, y, 0, nullptr, BNR_PRED_MEAN, false, K, fold, res_out);
}

extern "C" int bnr_fit_kfold_pointwise(const bnr_fit_result* r, double* elpd_kfold) {
  if (!r || !elpd_kfold) return ffail(BNR_EINVAL, "null argument");
  if (!r->kfold()) return ffail(BNR_ESTATE, "not a K-fold result (bnr_fit_kfold)");
  if (!r->held.ok) return ffail(BNR_ESTATE, "no retained draws");
  memcpy(elpd_kfold, r->elpd.data(), sizeof(double) * r->elpd.size());
  return BNR_OK;
}

extern "C" int bnr_fit_kfold_rhat(const bnr_fit_result* r, int32_t f, double* rhat_xi, double* rhat_gamma) {
  if (!r) return ffail(BNR_EINVAL, "null result");
  if (!r->kfold()) return ffail(BNR_ESTATE, "not a K-fold result (bnr_fit_kfold)");
  if (f < 0 || f >= (int)r->folds.size()) return ffail(BNR_EINVAL, "fold index outside 0..K-1");
  if (rhat_xi) memcpy(rhat_xi, r->folds[f].rhat_xi.data(), sizeof(double) * r->V);
  if (rhat_gamma) memcpy(rhat_gamma, r->folds[f].rhat_gamma.data(), sizeof(double) * r->q);
  return BNR_OK;
}

static int not_kfold(const bnr_fit_result* r) {
  return r->kfold() ? ffail(BNR_ESTATE, "not available on a K-fold result (bnr_fit_kfold)") : 0;
}

extern "C" int bnr_fit_loo_pointwise(const bnr_fit_result* r, double* elpd_loo, double* p_loo, double* pareto_k,
                                     double* elpd_waic, double* p_waic) {
  if (!r) return ffail(BNR_EINVAL, "null result");
  if (int e = not_kfold(r)) return e;
  if (!r->ll.ok)
    return ffail(BNR_ESTATE, !r->ll.width.empty() ? "fewer than 2 retained draws for PSIS-LOO"
                                             : "the fit was run without the log-likelihood (bnr_fit_loo)");
  double* dst[5] = {elpd_loo, p_loo, pareto_k, elpd_waic, p_waic};
  for (int k = 0; k < 5; ++k)
    if (dst[k]) memcpy(dst[k], r->l_pw[k].data(), sizeof(double) * r->l_pw[k].size());
  return BNR_OK;
}

extern "C" int bnr_fit_prediction(const bnr_fit_result* r, double* mean, double* lo, double* hi) {
  if (!r) return ffail(BNR_EINVAL, "null result");
  if (int e = not_kfold(r)) return e;
  if (!r->pred.ok)
    return ffail(BNR_ESTATE, !r->pred.width.empty() ? "too few retained draws for the prediction interval"
                                               : "the fit was run without X_new (bnr_fit_predict)");
  if (mean) memcpy(mean, r->p_mean.data(), sizeof(double) * r->p_mean.size());
  if (lo) memcpy(lo, r->p_lo.data(), sizeof(double) * r->p_lo.size());
  if (hi) memcpy(hi, r->p_hi.data(), sizeof(double) * r->p_hi.size());
  return BNR_OK;
}

extern "C" int bnr_fit_get_info(const bnr_fit_result* r, bnr_fit_info* info) {
  if (!r || !info) return ffail(BNR_EINVAL, "null argument");
  memset(info, 0, sizeof(*info));
  info->tot_generated = r->out.tot_generated; info->burn_in = r->out.burn_in; info->sampled = r->out.sampled;
  info->rows = r->out.rows; info->n_psrf = r->out.n_psrf; info->streamed = r->out.streamed ? 1 : 0;
  info->summary_ok = r->summary_ok ? 1 : 0; info->ess_ok = r->ess_ok ? 1 : 0;
  info->gamma_mode = r->gamma_mode; info->status_or = r->status_or;
  info->total_chains = r->C * (int)r->h.size() * (r->p.ext_world > 1 ? r->p.ext_world : 1);
  std::vector<int> devs(r->dev);
  std::sort(devs.begin(), devs.end());
  info->n_devices = (int)(std::unique(devs.begin(), devs.end()) - devs.begin());
  info->exchange = r->exchange;
  return BNR_OK;
}

extern "C" int bnr_fit_rhat(const bnr_fit_result* r, double* rhat_xi, double* rhat_gamma) {
  if (!r) return ffail(BNR_EINVAL, "null result");
  if (rhat_xi) memcpy(rhat_xi, r->rhat_xi.data(), sizeof(double) * r->V);
  if (rhat_gamma) memcpy(rhat_gamma, r->rhat_gamma.data(), sizeof(double) * r->q);
  return BNR_OK;
}

extern "C" int bnr_fit_summary(const bnr_fit_result* r, double* gamma_mean, double* gamma_lo, double* gamma_hi,
                               double* xi_mean) {
  if (!r) return ffail(BNR_EINVAL, "null result");
  if (int e = not_kfold(r)) return e;
  if (!r->summary_ok)
    return ffail(BNR_ESTATE, "too few retained draws for the credible interval (the reference's Summary raises a BoundsError)");
  if (gamma_mean) memcpy(gamma_mean, r->s_mean.data(), sizeof(double) * r->q);
  if (gamma_lo) memcpy(gamma_lo, r->s_lo.data(), sizeof(double) * r->q);
  if (gamma_hi) memcpy(gamma_hi, r->s_hi.data(), sizeof(double) * r->q);
  if (xi_mean) memcpy(xi_mean, r->s_xi.data(), sizeof(double) * r->V);
  return BNR_OK;
}

extern "C" int bnr_fit_ess(const bnr_fit_result* r, double* ess_xi, double* ess_gamma) {
  if (!r) return ffail(BNR_EINVAL, "null result");
  if (int e = not_kfold(r)) return e;
  if (!r->ess_ok) return ffail(BNR_ESTATE, "no ESS statistics (ess_max_lag = 0, or the doubling scheme with block moments)");
  if (ess_xi) memcpy(ess_xi, r->ess_xi.data(), sizeof(double) * r->V);
  if (ess_gamma) memcpy(ess_gamma, r->ess_gamma.data(), sizeof(double) * r->q);
  return BNR_OK;
}

extern "C" int bnr_fit_state(bnr_fit_result* r, int32_t var, double* out) {
  if (!r || !out) return ffail(BNR_EINVAL, "null argument");
  if (int e = not_kfold(r)) return e;
  if (r->p.return_state == BNR_STATE_NONE) return ffail(BNR_ESTATE, "the fit was run with return_state = BNR_STATE_NONE");
  if (r->p.return_state == BNR_STATE_GAMMA_XI && var != BNR_VAR_GAMMA && var != BNR_VAR_XI)
    return ffail(BNR_ESTATE, "only gamma and xi were recorded (return_state = BNR_STATE_GAMMA_XI)");
  if (bnr_get_trace(r->h[0], 0, var, 0, r->out.rows, out) != BNR_OK) return ffail(BNR_ECUDA, bnr_last_error());
  return BNR_OK;
}

// device_index: the device's place among the result's devices, or the fold (0-based) of a K-fold result
extern "C" int bnr_fit_handle(bnr_fit_result* r, int32_t device_index, bnr_handle** h) {
  if (!r || !h || device_index < 0 || device_index >= (int)r->h.size()) return ffail(BNR_EINVAL, "bad arguments");
  *h = r->h[device_index];
  return BNR_OK;
}

extern "C" int bnr_fit_free(bnr_fit_result* r) {
  delete r;
  return BNR_OK;
}
