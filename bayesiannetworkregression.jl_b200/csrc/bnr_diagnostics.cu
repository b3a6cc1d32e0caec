// Posterior diagnostics computed on the device from the recorded traces (iteration-major rows):
//   * Summary (src/gibbs.jl:1214-1250): per-edge posterior mean and the two order statistics sort(gamma)[lw], [hi]
//     that bound the credible interval, per-node mean xi            -> k_summary_select (radix select, no sort)
//   * gamma / xi effective sample size (BASELINE metric "gamma ESS/sec"; not in the reference): multi-chain Geyer
//     initial-monotone-sequence estimator on direct-lag autocovariances -> k_chain_mean, k_acov_sum, k_ess_finish
// Everything is deterministic (fixed reduction orders, integer histograms).
#include "bnr_engine.cuh"
#include "bnr_kernels.h"

namespace bnr {

// ------------------------------------------------------------------------------------------------------------
// Summary: exact k-th order statistics by 8-bit MSB radix select on the order-preserving 64-bit key of a double.
// One block handles SUM_EPB adjacent parameters (64 contiguous bytes per trace row); thread t reads parameter
// t % SUM_EPB of rows t / SUM_EPB, t / SUM_EPB + 32, ...  Two ranks (lower / upper bound) are selected together.
// grid = ceil(nelem / SUM_EPB), block = 256.
// ------------------------------------------------------------------------------------------------------------
constexpr int SUM_EPB = 8;

__device__ __forceinline__ unsigned long long order_key(double x) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_to_double(unsigned long long k) {
  const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

__global__ void __launch_bounds__(256) k_summary_select(const double* __restrict__ rows, size_t rowlen, int off,
                                                        int nelem, long long first, long long count,
                                                        long long rank_lo, long long rank_hi,
                                                        double* __restrict__ mean_out, double* __restrict__ lo_out,
                                                        double* __restrict__ hi_out) {
  __shared__ int hist[2][SUM_EPB][256];
  __shared__ unsigned long long prefix[2][SUM_EPB];
  __shared__ long long remain[2][SUM_EPB];
  __shared__ double psum[32][SUM_EPB];
  const int tid = threadIdx.x, e = tid % SUM_EPB, lane = tid / SUM_EPB;   // 32 row lanes
  const int el = blockIdx.x * SUM_EPB + e;
  const bool live = el < nelem;
  const double* base = rows + (size_t)first * rowlen + off + (live ? el : 0);
  if (tid < 2 * SUM_EPB) {
    prefix[tid / SUM_EPB][tid % SUM_EPB] = 0ull;
    remain[tid / SUM_EPB][tid % SUM_EPB] = (tid / SUM_EPB == 0) ? rank_lo : rank_hi;   // 1-based ranks
  }
  double s = 0.0;
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
    for (int i = tid; i < 2 * SUM_EPB * 256; i += 256) (&hist[0][0][0])[i] = 0;
    __syncthreads();
    const unsigned long long p0 = prefix[0][e], p1 = prefix[1][e];
    if (live) {
      for (long long r = lane; r < count; r += 32) {
        const double x = base[(size_t)r * rowlen];
        if (pass == 0) s += x;
        const unsigned long long k = order_key(x);
        const unsigned long long hi = (pass == 0) ? 0ull : (k >> (shift + 8));
        const int dg = (int)((k >> shift) & 0xffull);
        if (hi == p0) atomicAdd(&hist[0][e][dg], 1);
        if (hi == p1) atomicAdd(&hist[1][e][dg], 1);
      }
    }
    __syncthreads();
    if (tid < 2 * SUM_EPB) {
      const int t = tid / SUM_EPB, ee = tid % SUM_EPB;
      long long rem = remain[t][ee];
      int b = 0;
      for (; b < 255; ++b) {
        const int cnt = hist[t][ee][b];
        if (rem <= cnt) break;
        rem -= cnt;
      }
      remain[t][ee] = rem;
      prefix[t][ee] = (prefix[t][ee] << 8) | (unsigned long long)b;
    }
    __syncthreads();
  }
  psum[lane][e] = s;
  __syncthreads();
  if (tid < SUM_EPB && blockIdx.x * SUM_EPB + tid < nelem) {
    double tot = 0.0;
    for (int l = 0; l < 32; ++l) tot += psum[l][tid];
    const int o = blockIdx.x * SUM_EPB + tid;
    mean_out[o] = tot / (double)count;
    if (lo_out) lo_out[o] = key_to_double(prefix[0][tid]);
    if (hi_out) hi_out[o] = key_to_double(prefix[1][tid]);
  }
}

void launch_summary_select(const double* rows, size_t rowlen, int off, int nelem, long long first, long long count,
                           long long rank_lo, long long rank_hi, double* mean_out, double* lo_out, double* hi_out,
                           cudaStream_t s) {
  ++g_launches;
  k_summary_select<<<(nelem + SUM_EPB - 1) / SUM_EPB, 256, 0, s>>>(rows, rowlen, off, nelem, first, count, rank_lo,
                                                                    rank_hi, mean_out, lo_out, hi_out);
}

// ------------------------------------------------------------------------------------------------------------
// Pooled predictions: mean and two exact order statistics of every column j of rows[N][m] (N = all retained draws of
// all chains: millions of rows, m ~ 100 columns).  k_summary_select's one-block-per-8-columns grid would leave most SMs
// idle here, so the rows are split over blocks too: per 8-bit digit pass (MSB first, the order key of k_summary_select)
//   k_pred_hist : grid (ceil(m / 8), RB), block 256 = 8 columns x 32 row lanes over rows [by * per, (by + 1) * per):
//                 a shared histogram of the digit among the keys that match the prefix picked so far, added into the
//                 global [2][m][256] integer histogram (order-free); pass 0 also writes the block's column sums
//   k_pred_pick : thread per (rank, column): walks the 256 bins, extends the prefix, clears the histogram
// and k_pred_mean adds the RB block sums of each column in block order.  RB depends on (N, m) only.
// ------------------------------------------------------------------------------------------------------------
constexpr int PS_EPB = 8;
constexpr long long PS_MIN_ROWS = 1024;    // rows per block at least

static int pred_select_row_blocks(long long N, int m) {
  const long long gx = (m + PS_EPB - 1) / PS_EPB;
  long long rb = (4 * 148 + gx - 1) / gx;
  const long long by_rows = (N + PS_MIN_ROWS - 1) / PS_MIN_ROWS;
  if (rb > by_rows) rb = by_rows;
  if (rb > 65535) rb = 65535;
  return rb < 1 ? 1 : (int)rb;
}

__global__ void __launch_bounds__(256) k_pred_hist(const double* __restrict__ rows, long long N, int m, long long per,
                                                   int pass, unsigned long long* __restrict__ hist,
                                                   const unsigned long long* __restrict__ prefix,
                                                   double* __restrict__ psum) {
  __shared__ unsigned int h[2][PS_EPB][256];
  __shared__ double ps[32][PS_EPB];
  const int tid = threadIdx.x, e = tid % PS_EPB, lane = tid / PS_EPB;
  const int el = blockIdx.x * PS_EPB + e;
  const bool live = el < m;
  const long long r0 = (long long)blockIdx.y * per, r1 = min(N, r0 + per);
  for (int i = tid; i < 2 * PS_EPB * 256; i += 256) (&h[0][0][0])[i] = 0u;
  __syncthreads();
  const int shift = 56 - 8 * pass;
  const unsigned long long p0 = (pass && live) ? prefix[el] : 0ull, p1 = (pass && live) ? prefix[m + el] : 0ull;
  double s = 0.0;
  if (live) {
    for (long long r = r0 + lane; r < r1; r += 32) {
      const double x = rows[(size_t)r * m + el];
      if (pass == 0) s += x;
      const unsigned long long k = order_key(x);
      const unsigned long long hi = pass == 0 ? 0ull : (k >> (shift + 8));
      const int dg = (int)((k >> shift) & 0xffull);
      if (hi == p0) atomicAdd(&h[0][e][dg], 1u);
      if (hi == p1) atomicAdd(&h[1][e][dg], 1u);
    }
  }
  __syncthreads();
  for (int i = tid; i < 2 * PS_EPB * 256; i += 256) {
    const int t = i / (PS_EPB * 256), ee = (i / 256) % PS_EPB, b = i % 256;
    const unsigned int v = (&h[0][0][0])[i];
    const int col = blockIdx.x * PS_EPB + ee;
    if (v && col < m) atomicAdd(&hist[((size_t)t * m + col) * 256 + b], (unsigned long long)v);
  }
  if (pass == 0) {
    ps[lane][e] = s;
    __syncthreads();
    if (tid < PS_EPB && blockIdx.x * PS_EPB + tid < m) {
      double tot = 0.0;
      for (int l = 0; l < 32; ++l) tot += ps[l][tid];
      psum[(size_t)blockIdx.y * m + blockIdx.x * PS_EPB + tid] = tot;
    }
  }
}

__global__ void k_pred_pick(int m, int pass, long long rank_lo, long long rank_hi, unsigned long long* __restrict__ hist,
                            unsigned long long* __restrict__ prefix, long long* __restrict__ remain) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;      // (rank t, column j) = (idx / m, idx % m)
  if (idx >= 2 * m) return;
  unsigned long long* hb = hist + (size_t)idx * 256;
  long long rem = pass == 0 ? (idx < m ? rank_lo : rank_hi) : remain[idx];
  int b = 0;
  for (; b < 255; ++b) {
    const long long cnt = (long long)hb[b];
    if (rem <= cnt) break;
    rem -= cnt;
  }
  remain[idx] = rem;
  prefix[idx] = ((pass == 0 ? 0ull : prefix[idx]) << 8) | (unsigned long long)b;
  for (int i = 0; i < 256; ++i) hb[i] = 0ull;
}

__global__ void k_pred_mean(int m, int rb, long long N, const double* __restrict__ psum,
                            const unsigned long long* __restrict__ prefix, double* __restrict__ mean,
                            double* __restrict__ lo, double* __restrict__ hi) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  double tot = 0.0;
  for (int b = 0; b < rb; ++b) tot += psum[(size_t)b * m + j];
  mean[j] = tot / (double)N;
  lo[j] = key_to_double(prefix[j]);
  hi[j] = key_to_double(prefix[m + j]);
}

// scratch: hist [2][m][256] | prefix [2][m] | remain [2][m] | psum [RB][m]
size_t pred_select_ws_bytes(long long N, int m) {
  return sizeof(unsigned long long) * ((size_t)2 * m * 256 + 4 * (size_t)m) +
         sizeof(double) * (size_t)pred_select_row_blocks(N, m) * m;
}

void launch_pred_select(const double* rows, long long N, int m, long long rank_lo, long long rank_hi, double* mean,
                        double* lo, double* hi, void* ws, cudaStream_t s) {
  const int rb = pred_select_row_blocks(N, m);
  const long long per = (N + rb - 1) / rb;
  unsigned long long* hist = (unsigned long long*)ws;
  unsigned long long* prefix = hist + (size_t)2 * m * 256;
  long long* remain = (long long*)(prefix + 2 * (size_t)m);
  double* psum = (double*)(remain + 2 * (size_t)m);
  cudaMemsetAsync(hist, 0, sizeof(unsigned long long) * (size_t)2 * m * 256, s);
  const dim3 grid((m + PS_EPB - 1) / PS_EPB, rb);
  for (int pass = 0; pass < 8; ++pass) {
    ++g_launches; k_pred_hist<<<grid, 256, 0, s>>>(rows, N, m, per, pass, hist, prefix, psum);
    ++g_launches; k_pred_pick<<<(2 * m + 127) / 128, 128, 0, s>>>(m, pass, rank_lo, rank_hi, hist, prefix, remain);
  }
  ++g_launches; k_pred_mean<<<(m + 127) / 128, 128, 0, s>>>(m, rb, N, psum, prefix, mean, lo, hi);
}

// ------------------------------------------------------------------------------------------------------------
// Pooled PSIS-LOO and WAIC of every column i of ll[N][n] (N pooled draws of the pointwise log-likelihood), as the R
// package loo 2.x computes them with r_eff = 1: log ratios -ll, shifted so that the largest is 0 (lw = min ll - ll); the
// tail is the M = ceil(min(0.2 N, 3 sqrt N)) largest lw, i.e. the M smallest ll; the generalised Pareto fit of
// Zhang & Stephens (gpdfit) replaces the tail by its quantiles; weights are truncated at 0.
//   launch_pred_select : ranks a = ll_(M), b = ll_(M+1) (the cutoff) and the column mean
//   k_loo_pass         : rows split over blocks like k_pred_hist (8 columns x 32 row lanes); per block and column the
//                        logsumexp partial of ll, sum (ll - mean)^2 and the non-tail weight sum sum_{ll > a} exp(b - ll);
//                        values below a are compacted into the column's tail through an integer cursor, values equal
//                        to a are counted
//   k_loo_tail         : block per column: the tail (cursor entries, then copies of a) sorted in shared memory, the
//                        GPD fit, smoothing, truncation and the block partials added in block order
// Every floating-point sum has a fixed order; the tail is sorted before use, so its compaction order does not matter.
// ------------------------------------------------------------------------------------------------------------
constexpr int LOO_TB = 512;     // threads of k_loo_tail

long long loo_tail_len(long long N) {
  const double S = (double)N;
  return (long long)ceil(fmin(0.2 * S, 3.0 * sqrt(S)));
}

// dynamic shared memory of k_loo_tail: tail [M] | reduction scratch [32] | broadcast [8] | theta [G] | l(theta) [G]
__host__ __device__ static int loo_grid(long long M) { return 30 + (int)floor(sqrt((double)M)); }
static size_t loo_tail_smem(long long M) { return sizeof(double) * ((size_t)M + 40 + 2 * (size_t)loo_grid(M)); }

long long loo_tail_max() {
  int dev = 0, optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  long long M = optin / 8 - 40 - 2 * loo_grid(optin / 8);
  while (M > 0 && loo_tail_smem(M) > (size_t)optin) --M;
  return M;
}

__global__ void __launch_bounds__(256) k_loo_pass(const double* __restrict__ rows, long long N, int n, long long per,
                                                  long long M, const double* __restrict__ mean,
                                                  const double* __restrict__ av, const double* __restrict__ bv,
                                                  double* __restrict__ part, unsigned long long* __restrict__ cnt,
                                                  double* __restrict__ tail) {
  __shared__ double red[4][32][PS_EPB];
  const int tid = threadIdx.x, e = tid % PS_EPB, lane = tid / PS_EPB;
  const int col = blockIdx.x * PS_EPB + e;
  const bool live = col < n;
  const long long r0 = (long long)blockIdx.y * per, r1 = min(N, r0 + per);
  double mx = -INFINITY, se = 0.0, sq = 0.0, w = 0.0;
  unsigned long long eq = 0;
  if (live) {
    const double mu = mean[col], a = av[col], b = bv[col];
    double* tl = tail + (size_t)col * M;
    for (long long r = r0 + lane; r < r1; r += 32) {
      const double x = rows[(size_t)r * n + col];
      if (x > mx) { se = se * exp(mx - x) + 1.0; mx = x; }
      else se += exp(x - mx);
      const double dv = x - mu;
      sq += dv * dv;
      if (x > a) w += exp(b - x);
      else if (x < a) tl[atomicAdd(&cnt[col], 1ull)] = x;
      else ++eq;
    }
    if (eq) atomicAdd(&cnt[n + col], eq);
  }
  red[0][lane][e] = mx; red[1][lane][e] = se; red[2][lane][e] = sq; red[3][lane][e] = w;
  __syncthreads();
  if (tid < PS_EPB && blockIdx.x * PS_EPB + tid < n) {
    double m = -INFINITY, s = 0.0, q = 0.0, ww = 0.0;
    for (int l = 0; l < 32; ++l) {
      const double m2 = red[0][l][tid], s2 = red[1][l][tid];
      if (s2 > 0.0) {
        if (m2 > m) { s = s * exp(m - m2) + s2; m = m2; }
        else s += s2 * exp(m2 - m);
      }
      q += red[2][l][tid];
      ww += red[3][l][tid];
    }
    double* p = part + ((size_t)blockIdx.y * n + blockIdx.x * PS_EPB + tid) * 4;
    p[0] = m; p[1] = s; p[2] = q; p[3] = ww;
  }
}

// the same value on every thread: warp trees, then the warps in order
__device__ double loo_block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
  return t;
}
__device__ double loo_block_max(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = -INFINITY;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t = fmax(t, red[i]);
  return t;
}

// out[k * n + col]: k = 0 elpd_loo, 1 p_loo, 2 pareto_k, 3 elpd_waic, 4 p_waic
__global__ void __launch_bounds__(LOO_TB) k_loo_tail(long long N, int n, long long M, int rb,
                                                     const double* __restrict__ part,
                                                     const unsigned long long* __restrict__ cnt,
                                                     const double* __restrict__ av, const double* __restrict__ bv,
                                                     const double* __restrict__ tail, double* __restrict__ out) {
  extern __shared__ double sm[];
  const int G = loo_grid(M);
  double* v = sm;              // the tail's ll values, sorted ascending
  double* red = v + M;
  double* bc = red + 32;
  double* th = bc + 8;
  double* lt = th + G;
  const int col = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  const long long below = (long long)cnt[col], eq = (long long)cnt[n + col];
  const double a = av[col], b = bv[col];
  for (long long i = tid; i < M; i += nt) v[i] = i < below ? tail[(size_t)col * M + i] : a;
  __syncthreads();
  // bitonic sort of M values without storing the padding to a power of two: every compare-exchange puts the larger
  // value at the higher index, so virtual +inf beyond M never moves and pairs reaching past M are skipped
  long long P = 1;
  while (P < M) P <<= 1;
  for (long long k = 2; k <= P; k <<= 1) {
    for (long long t = tid; t < P / 2; t += nt) {
      const long long h = k >> 1, blk = t / h, off = t % h;
      const long long i = blk * k + off, j = blk * k + k - 1 - off;
      if (j < M && v[i] > v[j]) { const double x = v[i]; v[i] = v[j]; v[j] = x; }
    }
    __syncthreads();
    for (long long d = k >> 2; d >= 1; d >>= 1) {
      for (long long t = tid; t < P / 2; t += nt) {
        const long long blk = t / d, off = t % d;
        const long long i = blk * 2 * d + off, j = i + d;
        if (j < M && v[i] > v[j]) { const double x = v[i]; v[i] = v[j]; v[j] = x; }
      }
      __syncthreads();
    }
  }
  // log weight of the tail value of ascending rank j (0-based): lw_j = min ll - ll_(M-1-j); cutoff = min ll - b
  const double mn = v[0], cut = mn - b, ec = exp(cut);
  const double Md = (double)M;
  double kh = INFINITY, sigma = 0.0;
  if (M >= 5 && v[0] != v[M - 1]) {
    const double xM = exp(mn - v[0]) - ec;
    const long long qi = (long long)floor(Md / 4.0 + 0.5) - 1;
    const double xs = exp(mn - v[M - 1 - qi]) - ec;
    for (int j = tid; j < G; j += nt) th[j] = 1.0 / xM + (1.0 - sqrt((double)G / (j + 0.5))) / (3.0 * xs);
    __syncthreads();
    for (int g = 0; g < G; ++g) {
      const double t = th[g];
      double s = 0.0;
      for (long long i = tid; i < M; i += nt) s += log1p(-t * (exp(mn - v[i]) - ec));
      s = loo_block_sum(s, red);
      if (tid == 0) {
        const double kk = s / Md;
        lt[g] = Md * (log(-t / kk) - kk - 1.0);
      }
    }
    __syncthreads();
    if (tid == 0) {
      double lm = -INFINITY;
      for (int g = 0; g < G; ++g) lm = fmax(lm, lt[g]);
      double z = 0.0;
      for (int g = 0; g < G; ++g) z += exp(lt[g] - lm);
      const double lse = lm + log(z);
      double thh = 0.0;
      for (int g = 0; g < G; ++g) thh += th[g] * exp(lt[g] - lse);
      bc[0] = thh;
    }
    __syncthreads();
    const double thh = bc[0];
    double s = 0.0;
    for (long long i = tid; i < M; i += nt) s += log1p(-thh * (exp(mn - v[i]) - ec));
    s = loo_block_sum(s, red);
    const double k0 = s / Md;
    sigma = -k0 / thh;
    kh = (Md * k0 + 5.0) / (Md + 10.0);
    if (isnan(kh)) kh = INFINITY;
  }
  const bool smooth = isfinite(kh);
  // smoothed, truncated log weight s_j of rank j and its raw lw_j
  auto smoothed = [&](long long j, double& lwr) {
    lwr = mn - v[M - 1 - j];
    double s = lwr;
    if (smooth) {
      const double p = ((double)j + 0.5) / Md;
      const double qq = kh == 0.0 ? -sigma * log1p(-p) : sigma * expm1(-kh * log1p(-p)) / kh;
      s = log(qq + ec);
    }
    return s > 0.0 ? 0.0 : s;
  };
  // lse(lw + ll) = mn + lse(t) with t_j = s_j - lw_j in the tail and t = 0 for the N - M others;
  // lse(lw) over the tail's s_j and the non-tail term cut + log W, W = sum_{ll > a} exp(b - ll) + (copies of a outside)
  double mt = 0.0, ms = -INFINITY;
  for (long long j = tid; j < M; j += nt) {
    double lwr;
    const double s = smoothed(j, lwr);
    mt = fmax(mt, s - lwr);
    ms = fmax(ms, s);
  }
  mt = loo_block_max(mt, red);
  ms = loo_block_max(ms, red);
  double st = 0.0, ss = 0.0;
  for (long long j = tid; j < M; j += nt) {
    double lwr;
    const double s = smoothed(j, lwr);
    st += exp(s - lwr - mt);
    ss += exp(s - ms);
  }
  st = loo_block_sum(st, red);
  ss = loo_block_sum(ss, red);
  if (tid == 0) {
    double m = -INFINITY, se = 0.0, sq = 0.0, w = 0.0;
    for (int y = 0; y < rb; ++y) {
      const double* p = part + ((size_t)y * n + col) * 4;
      if (p[1] > 0.0) {
        if (p[0] > m) { se = se * exp(m - p[0]) + p[1]; m = p[0]; }
        else se += p[1] * exp(p[0] - m);
      }
      sq += p[2];
      w += p[3];
    }
    w += (double)(below + eq - M);
    const double S = (double)N;
    const double lse_a = mn + mt + log((S - Md) * exp(-mt) + st);
    const double lnt = cut + log(w);
    const double mm = fmax(lnt, ms);
    const double lse_b = mm + log(exp(lnt - mm) + ss * exp(ms - mm));
    const double elpd = lse_a - lse_b;
    const double lpd = m + log(se) - log(S);
    const double pw = sq / (S - 1.0);
    out[col] = elpd;
    out[n + col] = lpd - elpd;
    out[2 * n + col] = kh;
    out[3 * n + col] = lpd - pw;
    out[4 * n + col] = pw;
  }
}

// scratch: select | mean, a, b [3][n] | partials [RB][n][4] | counters [2][n] | tails [n][M]
size_t loo_ws_bytes(long long N, int n) {
  const size_t sel = (pred_select_ws_bytes(N, n) + 255) / 256 * 256;
  return sel + sizeof(double) * ((size_t)3 * n + (size_t)pred_select_row_blocks(N, n) * n * 4) +
         sizeof(unsigned long long) * 2 * (size_t)n + sizeof(double) * (size_t)n * loo_tail_len(N);
}

void launch_loo(const double* rows, long long N, int n, double* out, void* ws, cudaStream_t s) {
  const long long M = loo_tail_len(N);
  const int rb = pred_select_row_blocks(N, n);
  const long long per = (N + rb - 1) / rb;
  char* p = (char*)ws;
  void* sel = p;
  p += (pred_select_ws_bytes(N, n) + 255) / 256 * 256;
  double* mean = (double*)p;
  double* av = mean + n;
  double* bv = av + n;
  double* part = bv + n;
  unsigned long long* cnt = (unsigned long long*)(part + (size_t)rb * n * 4);
  double* tail = (double*)(cnt + 2 * (size_t)n);
  launch_pred_select(rows, N, n, M, M + 1, mean, av, bv, sel, s);
  cudaMemsetAsync(cnt, 0, sizeof(unsigned long long) * 2 * (size_t)n, s);
  ++g_launches;
  k_loo_pass<<<dim3((n + PS_EPB - 1) / PS_EPB, rb), 256, 0, s>>>(rows, N, n, per, M, mean, av, bv, part, cnt, tail);
  const size_t smem = loo_tail_smem(M);
  cudaFuncSetAttribute(k_loo_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  ++g_launches;
  k_loo_tail<<<n, LOO_TB, smem, s>>>(N, n, M, rb, part, cnt, av, bv, tail, out);
}

// ------------------------------------------------------------------------------------------------------------
// ESS.  tr: the (xi, gamma) trace table, P = tr.width; window = rows [first, first + N).
//   k_chain_mean : cmean[c][p]                       grid = (ceil(P/128), C), block = 128
//   k_acov_sum   : acov[l][p] = sum_c 1/N sum_t (x_t - m_c)(x_{t+l} - m_c), l = 0 .. L (biased, per-chain centred)
//                  grid = (ceil(P/32), ceil((L+1)/64)), block = 256 = 32 parameters x 8 lag groups of 8 lags;
//                  row chunks of 128 are staged in shared memory, each thread slides an 8-lag register window.
//   k_ess_finish : Geyer initial monotone sequence over the pooled autocorrelations -> ess[p], thread per parameter
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_chain_mean(RowTable tr, long long first, long long N, double* __restrict__ cmean) {
  const int P = tr.width, p = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
  if (p >= P) return;
  const double* __restrict__ b = tr.row(c, first) + p;
  double s = 0.0;
  for (long long r = 0; r < N; ++r) s += b[(size_t)r * P];
  cmean[(size_t)c * P + p] = s / (double)N;
}

constexpr int AC_TCH = 128;    // rows per staged chunk
constexpr int AC_LB = 64;      // lags per block
constexpr size_t ACOV_SMEM = sizeof(double) * ((size_t)AC_TCH * 32 + (size_t)(AC_TCH + AC_LB) * 32);

__global__ void __launch_bounds__(256) k_acov_sum(RowTable tr, long long first, long long N, int L,
                                                  const double* __restrict__ cmean, double* __restrict__ acov) {
  const int P = tr.width, C = tr.chains;
  extern __shared__ double sm[];
  double* A = sm;                       // [AC_TCH][32]       x_t - m
  double* B = sm + AC_TCH * 32;         // [AC_TCH + 64][32]  x_{t + l0 + .} - m
  const int tid = threadIdx.x, pl = tid & 31, g = tid >> 5;
  const int p0 = blockIdx.x * 32, l0 = blockIdx.y * AC_LB;
  const int p = p0 + pl;
  double acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.0;
  for (int c = 0; c < C; ++c) {
    const double* base = tr.row(c, first);   // loaded through __ldg: a pointer taken from a struct is not __restrict__
    const double m = (p < P) ? cmean[(size_t)c * P + p] : 0.0;
    // every thread stages column pl of the tiles: its own parameter, so m is the right centre
    for (long long t0 = 0; t0 < N; t0 += AC_TCH) {
      __syncthreads();
      for (int r = g; r < AC_TCH; r += 8) {
        const long long t = t0 + r;
        A[r * 32 + pl] = (p < P && t < N) ? __ldg(base + (size_t)t * P + p) - m : 0.0;
      }
      for (int r = g; r < AC_TCH + AC_LB; r += 8) {
        const long long t = t0 + l0 + r;
        B[r * 32 + pl] = (p < P && t < N) ? __ldg(base + (size_t)t * P + p) - m : 0.0;
      }
      __syncthreads();
      // lags l0 + 8g + k, k = 0..7: acc[k] += A[t] * B[t + 8g + k]
      double w[8];
#pragma unroll
      for (int k = 0; k < 7; ++k) w[k + 1] = B[(8 * g + k) * 32 + pl];
#pragma unroll 8
      for (int t = 0; t < AC_TCH; ++t) {
#pragma unroll
        for (int k = 0; k < 7; ++k) w[k] = w[k + 1];
        w[7] = B[(t + 8 * g + 7) * 32 + pl];
        const double a = A[t * 32 + pl];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] += a * w[k];
      }
    }
  }
  if (p < P) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int l = l0 + 8 * g + k;
      if (l <= L) acov[(size_t)l * P + p] = acc[k] / (double)N;
    }
  }
}

// acov_parts: [nparts][L+1][P] (one part per rank), cmeans: [chains][P].  ess[p]; lag_used[p] = lags consumed
// (L + 1 when the Geyer sequence had not terminated inside the lag budget: the estimate is then an upper bound).
__global__ void k_ess_finish(const double* __restrict__ acov_parts, int nparts, const double* __restrict__ cmeans,
                             int chains, int P, long long N, int L, double* __restrict__ ess,
                             double* __restrict__ lag_used) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const size_t part = (size_t)(L + 1) * P;
  auto mean_acov = [&](int l) {
    double s = 0.0;
    for (int r = 0; r < nparts; ++r) s += acov_parts[r * part + (size_t)l * P + p];
    return s / (double)chains;
  };
  const double n = (double)N;
  const double W = mean_acov(0) * n / (n - 1.0);
  double B_over_n = 0.0;
  if (chains > 1) {
    double mm = 0.0;
    for (int c = 0; c < chains; ++c) mm += cmeans[(size_t)c * P + p];
    mm /= chains;
    for (int c = 0; c < chains; ++c) { const double dm = cmeans[(size_t)c * P + p] - mm; B_over_n += dm * dm; }
    B_over_n /= (chains - 1);
  }
  const double var_plus = W * (n - 1.0) / n + B_over_n;
  if (!(var_plus > 0.0)) { ess[p] = nan(""); if (lag_used) lag_used[p] = 0.0; return; }
  double tau = -1.0, prev = INFINITY;
  int t = 0;
  for (; t + 1 <= L && t + 1 < N; t += 2) {
    const double r0 = 1.0 - (W - mean_acov(t)) / var_plus;
    const double r1 = 1.0 - (W - mean_acov(t + 1)) / var_plus;
    double pair = r0 + r1;
    if (pair < 0.0) break;
    pair = pair < prev ? pair : prev;
    tau += 2.0 * pair;
    prev = pair;
  }
  const double nm = n * chains;
  const double floor_tau = 1.0 / log10(nm > 10.0 ? nm : 10.0);
  ess[p] = nm / (tau > floor_tau ? tau : floor_tau);
  if (lag_used) lag_used[p] = (double)t;
}

// ------------------------------------------------------------------------------------------------------------
// Streaming ESS statistics: the same (acov, chain means) as k_chain_mean + k_acov_sum, accumulated while the chains
// run, so that no chain needs a trace (64 chains x 20 000 draws x 5150 parameters would be 53 GB of traces).
// Per chain and parameter, with x_0 the first retained draw and y_t = x_t - x_0 (centring on a value of the chain
// itself keeps the raw lagged products well conditioned):
//     A_l = sum_{t >= l} y_t y_(t-l)  (l = 0..L),   S = sum_t y_t,   the first L draws (head) and the last L + ES_B (ring)
// and, at the end, with m = S / N, H_l = sum_{t < l} y_t, T_l = sum_{t >= N-l} y_t:
//     sum_{t >= l} (y_t - m)(y_(t-l) - m) = A_l - m (2 S - H_l - T_l) + (N - l) m^2 .
// k_ess_stream runs once per sweep (thread per (chain, parameter)): it appends the draw to the ring and, every ES_B
// draws (and at the last draw), adds the block's lagged products with a sliding ES_B-wide register window: one ring
// load and one read-modify-write of A_l per lag and per ES_B draws, i.e. 1/ES_B of the naive per-sweep traffic.
// grid = (ceil(P/128), C), block = 128.
// ------------------------------------------------------------------------------------------------------------
constexpr int ES_B = 8;

__global__ void __launch_bounds__(128) k_ess_stream(Engine e) {
  const Dims& d = e.d;
  const int P = d.V + d.q;
  const int p = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
  if (p >= P) return;
  const long long first = e.ess_win[0], N = e.ess_win[1];
  const int L = (int)e.ess_win[2], cap = (int)e.ess_win[3];
  const long long k = (*e.iter + 1) - first;        // index of this sweep's draw inside the window
  if (k < 0 || k >= N) return;
  const double x = (p < d.V) ? e.xi[c * d.V + p] : e.gamma[(size_t)c * d.qp + (p - d.V)];
  double* sum = e.ess_sum + (size_t)c * 2 * P;
  double* ring = e.ess_ring + (size_t)c * cap * P + p;
  double ref, S;
  if (k == 0) { ref = x; S = 0.0; sum[p] = ref; }
  else { ref = sum[p]; S = sum[P + p]; }
  const double y = x - ref;
  sum[P + p] = S + y;
  ring[(size_t)(k % cap) * P] = y;
  if (k < L) e.ess_head[((size_t)c * L + k) * P + p] = y;
  const int b = (int)(k % ES_B) + 1;
  if (b != ES_B && k != N - 1) return;
  // block of the b newest draws k0 .. k: A_l += sum_j y_(k0+j) y_(k0+j-l)
  const long long k0 = k - b + 1;
  double Y[ES_B], w[ES_B];
#pragma unroll
  for (int j = 0; j < ES_B; ++j) {
    Y[j] = (j < b) ? ring[(size_t)((k0 + j) % cap) * P] : 0.0;
    w[j] = Y[j];
  }
  double* A = e.ess_acc + (size_t)c * (L + 1) * P + p;
  const int lmax = (long long)L < k ? L : (int)k;
  const bool fresh = (k0 == 0);                     // first block of the window: A starts from zero
  for (int l = 0; l <= L; ++l) {
    if (l > 0) {
#pragma unroll
      for (int j = ES_B - 1; j > 0; --j) w[j] = w[j - 1];
      w[0] = (k0 - l >= 0) ? ring[(size_t)((k0 - l) % cap) * P] : 0.0;
    }
    if (l > lmax) { if (fresh) A[(size_t)l * P] = 0.0; continue; }
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < ES_B; ++j) s += Y[j] * ((k0 + j - l >= 0) ? w[j] : 0.0);
    A[(size_t)l * P] = (fresh ? 0.0 : A[(size_t)l * P]) + s;
  }
}

// acov[l][p] = sum_c (1/N) sum_{t >= l} (x_t - mean_c)(x_(t-l) - mean_c), cmean[c][p]; thread per parameter, chains in
// a fixed order (deterministic).  grid = ceil(P/128), block = 128.
__global__ void __launch_bounds__(128) k_ess_stream_finalize(Engine e, long long N, double* __restrict__ acov,
                                                             double* __restrict__ cmean) {
  const Dims& d = e.d;
  const int P = d.V + d.q, L = e.ess_L, cap = e.ess_cap;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const double n = (double)N;
  for (int c = 0; c < d.C; ++c) {
    const double ref = e.ess_sum[(size_t)c * 2 * P + p], S = e.ess_sum[(size_t)c * 2 * P + P + p];
    const double m = S / n;
    cmean[(size_t)c * P + p] = ref + m;
    const double* A = e.ess_acc + (size_t)c * (L + 1) * P + p;
    const double* head = e.ess_head + (size_t)c * L * P + p;
    const double* ring = e.ess_ring + (size_t)c * cap * P + p;
    double H = 0.0, T = 0.0;
    for (int l = 0; l <= L; ++l) {
      if (l >= 1) {
        H += head[(size_t)(l - 1) * P];
        T += ring[(size_t)((N - l) % cap) * P];
      }
      const double v = (A[(size_t)l * P] - m * (2.0 * S - H - T) + (n - l) * m * m) / n;
      acov[(size_t)l * P + p] = (c == 0 ? 0.0 : acov[(size_t)l * P + p]) + v;
    }
  }
}

void launch_ess_stream(const Engine& e, cudaStream_t s) {
  dim3 grid((e.d.V + e.d.q + 127) / 128, e.d.C);
  ++g_launches; k_ess_stream<<<grid, 128, 0, s>>>(e);
}

void launch_ess_stream_finalize(const Engine& e, long long N, double* acov, double* cmean, cudaStream_t s) {
  ++g_launches; k_ess_stream_finalize<<<(e.d.V + e.d.q + 127) / 128, 128, 0, s>>>(e, N, acov, cmean);
}

void launch_chain_mean(const RowTable& tr, long long first, long long N, double* cmean, cudaStream_t s) {
  dim3 grid((tr.width + 127) / 128, tr.chains);
  ++g_launches; k_chain_mean<<<grid, 128, 0, s>>>(tr, first, N, cmean);
}

void launch_acov_sum(const RowTable& tr, long long first, long long N, int L, const double* cmean, double* acov,
                     cudaStream_t s) {
  static bool attr = false;
  if (!attr) { cudaFuncSetAttribute(k_acov_sum, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ACOV_SMEM); attr = true; }
  dim3 grid((tr.width + 31) / 32, (L + 1 + AC_LB - 1) / AC_LB);
  ++g_launches; k_acov_sum<<<grid, 256, ACOV_SMEM, s>>>(tr, first, N, L, cmean, acov);
}

void launch_ess_finish(const double* acov_parts, int nparts, const double* cmeans, int chains, int P, long long N,
                       int L, double* ess, double* lag_used, cudaStream_t s) {
  ++g_launches; k_ess_finish<<<(P + 127) / 128, 128, 0, s>>>(acov_parts, nparts, cmeans, chains, P, N, L, ess, lag_used);
}

}  // namespace bnr
