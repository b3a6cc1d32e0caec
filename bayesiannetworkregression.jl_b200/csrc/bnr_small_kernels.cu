// Per-node, per-edge and scalar full-conditional kernels of the Gibbs sweep (everything except the dense
// linear algebra of the gamma draw, which lives in bnr_linalg.cu).  One launch advances ALL chains of the
// handle; chains are the outer grid dimension.  Reference semantics: src/gibbs.jl:267-636 (cited per kernel).
#include "bnr_engine.cuh"
#include "bnr_gig.cuh"
#include "bnr_kernels.h"

namespace bnr {

// ------------------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// deterministic block sum (fixed tree), result valid in every thread; blockDim.x multiple of 32, <= 1024
__device__ double block_sum(double v, double* sh /* >= 32 doubles */) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  double r = 0.0;
  for (int i = 0; i < nw; ++i) r += sh[i];
  return r;
}

// in-place lower Cholesky of a small col-major (ld = R) SPD matrix held in shared/local memory; single thread.
// Returns false when a pivot is not positive (matrix numerically not PD).
__device__ bool small_chol(double* A, int R) {
  for (int j = 0; j < R; ++j) {
    double d = A[j + R * j];
    for (int p = 0; p < j; ++p) d -= A[j + R * p] * A[j + R * p];
    if (!(d > 0.0)) return false;
    d = sqrt(d);
    A[j + R * j] = d;
    for (int i = j + 1; i < R; ++i) {
      double s = A[i + R * j];
      for (int p = 0; p < j; ++p) s -= A[i + R * p] * A[j + R * p];
      A[i + R * j] = s / d;
    }
  }
  return true;
}

// the same factorisation by one warp (lane i owns row i; identical summation order, so identical results): A is a
// col-major R x R SPD matrix in shared memory, R <= 32.  Every lane returns whether all pivots were positive.
__device__ bool warp_chol(double* A, int R, int lane) {
  bool ok = true;
  for (int j = 0; j < R; ++j) {
    double s = 0.0;
    if (lane >= j && lane < R) {
      s = A[lane + R * j];
      for (int p = 0; p < j; ++p) s -= A[lane + R * p] * A[j + R * p];
    }
    const double dj = __shfl_sync(0xffffffffu, s, j);
    if (!(dj > 0.0)) ok = false;
    const double rt = sqrt(dj);
    if (lane == j) A[j + R * j] = rt;
    else if (lane > j && lane < R) A[lane + R * j] = s / rt;
    __syncwarp();
  }
  return ok;
}

// Cholesky of a small SPD matrix with the reference's jitter ladder (src/gibbs.jl:322-347: on failure add 1e-5 I and
// retry, on a second failure a further 4e-5 I, then give up), by one warp.  In: A (col-major R x R, shared memory).
// Out: A = the Cholesky factor of the matrix that finally factored, A0 = that matrix; returns BNR_ST_JITTER_ /
// BNR_ST_SIGMA_NOTPD_ bits.
__device__ int warp_chol_ladder(double* A, double* A0, int R, int lane) {
  const int RR = R * R;
  int status = 0;
  for (int i = lane; i < RR; i += 32) A0[i] = A[i];
  __syncwarp();
  bool ok = warp_chol(A, R, lane);
  if (!ok) {
    status |= BNR_ST_JITTER_;
    if (lane < R) A0[lane + R * lane] += 1e-5;
    __syncwarp();
    for (int i = lane; i < RR; i += 32) A[i] = A0[i];
    __syncwarp();
    ok = warp_chol(A, R, lane);
    if (!ok) {
      if (lane < R) A0[lane + R * lane] += 4e-5;
      __syncwarp();
      for (int i = lane; i < RR; i += 32) A[i] = A0[i];
      __syncwarp();
      ok = warp_chol(A, R, lane);
      if (!ok) status |= BNR_ST_SIGMA_NOTPD_;
    }
  }
  return status;
}

// parity-test hook for the ladder alone (bnr_test_chol_jitter): one warp, matrix in / factor + used matrix + status out
__global__ void k_test_chol_jitter(int R, const double* __restrict__ Ain, double* __restrict__ Aused,
                                   double* __restrict__ Lout, int* __restrict__ status) {
  __shared__ double A[MAX_R * MAX_R], A0[MAX_R * MAX_R];
  const int lane = threadIdx.x;
  for (int i = lane; i < R * R; i += 32) A[i] = Ain[i];
  __syncwarp();
  const int st = warp_chol_ladder(A, A0, R, lane);
  __syncwarp();
  for (int i = lane; i < R * R; i += 32) {
    Aused[i] = A0[i];
    Lout[i] = (i % R >= i / R) ? A[i] : 0.0;
  }
  if (lane == 0) *status = st;
}

void launch_test_chol_jitter(int R, const double* Ain, double* Aused, double* Lout, int* status, cudaStream_t s) {
  k_test_chol_jitter<<<1, 32, 0, s>>>(R, Ain, Aused, Lout, status);
}

// ------------------------------------------------------------------------------------------------------------
// tau^2  (update_tau2!, src/gibbs.jl:267-277): InverseGamma(n/2 + q/2, 1/2 |y - mu - X gamma|^2 + 1/2 sum (gamma-W)^2/S)
// grid = (nb, C), block = 256: the two sums are split over nb = tau2_blocks(q) blocks per chain; the last block to
// finish (ticket counter) adds the partial sums in block order -- deterministic -- and draws.  X gamma comes from e.xg.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_tau2(Engine e) {
  extern __shared__ double sm[];
  __shared__ unsigned ticket;
  const Dims& d = e.d;
  const int c = blockIdx.y, tid = threadIdx.x, nb = gridDim.x, b = blockIdx.x;
  double* us = sm;                 // [V*R]
  double* lam = us + d.V * d.R;    // [R]
  double* red = lam + d.R;         // [32]
  for (int i = tid; i < d.V * d.R; i += blockDim.x) us[i] = e.u[(size_t)c * d.V * d.R + i];
  if (tid < d.R) lam[tid] = e.lambda[c * d.R + tid];
  __syncthreads();
  const double mu = e.mu[c];
  double s1 = 0.0;
  for (int i = b * blockDim.x + tid; i < d.n; i += nb * blockDim.x) {
    const double r = e.y[i] - mu - e.xg[(size_t)c * d.np + i];
    s1 += r * r;
  }
  double s2 = 0.0;
  for (int j = b * blockDim.x + tid; j < d.q; j += nb * blockDim.x) {
    const int2 lk = e.edge_lk[j];
    double w = 0.0;
    for (int r = 0; r < d.R; ++r) w += lam[r] * us[lk.y * d.R + r] * us[lk.x * d.R + r];
    const double g = e.gamma[(size_t)c * d.qp + j] - w;
    s2 += (g * g * 0.5) / e.S[(size_t)c * d.qp + j];
  }
  s1 = block_sum(s1, red);
  s2 = block_sum(s2, red);
  double* part = e.tau2_part + (size_t)c * 2 * TAU2_MAX_BLOCKS;
  if (tid == 0) {
    part[2 * b] = s1; part[2 * b + 1] = s2;
    __threadfence();
    ticket = atomicAdd(&e.tau2_ticket[c], 1u);
  }
  __syncthreads();
  if (ticket != (unsigned)(nb - 1)) return;
  if (tid == 0) {
    __threadfence();
    e.tau2_ticket[c] = 0u;      // ready for the next sweep
    const volatile double* vp = part;
    s1 = 0.0; s2 = 0.0;
    for (int k = 0; k < nb; ++k) { s1 += vp[2 * k]; s2 += vp[2 * k + 1]; }
    const long long it = *e.iter + 1;
    const double shape = 0.5 * d.n + 0.25 * (double)d.V * (d.V + 1);
    const double scale = 0.5 * s1 + s2;
    const InjLayout L = InjLayout::make(d.n, d.V, d.R, d.gigK);
    DrawStream st(chain_key(d, c), (uint32_t)it, SITE_TAU2, 0,
                  e.inj ? e.inj + (size_t)c * e.inj_stride + L.tau2 : nullptr, 1);
    const double g = st.gamma(shape);
    e.tau2[c] = scale / g;
    if (e.aux.tau2_params) { e.aux.tau2_params[2 * c] = shape; e.aux.tau2_params[2 * c + 1] = scale; }
  }
}

// ------------------------------------------------------------------------------------------------------------
// (u, xi)  (update_u_xi!, src/gibbs.jl:293-371; update_xi 385-402).  One warp per (chain, node); every node
// reads the PREVIOUS u of all other nodes (Jacobi), so u is double-buffered (e.u -> e.u_alt).
// The (V-1)-dimensional mixture odds of the reference are evaluated through the R x R identity
//   log(w_bot/w_top) = log(D/(1-D)) - 1/2 logdet M - 1/2 logdet Sigma^-1 + 1/2 b' Sigma b,   b = U' H^-1 gamma_k / tau2.
// grid = (ceil(V / 4), C), block = 128.
// ------------------------------------------------------------------------------------------------------------
constexpr int UXI_WARPS = 4;

__global__ void __launch_bounds__(32 * UXI_WARPS) k_uxi(Engine e) {
  extern __shared__ double sm[];
  const Dims& d = e.d;
  const int c = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int R = d.R, V = d.V, RR = R * R;
  double* ulam = sm;                       // [V*R]   u_prev[l][r] * lambda[r]
  double* Minv = ulam + V * R;             // [RR]
  double* Mch = Minv + RR;                 // [RR]    scratch for chol(M)
  double* misc = Mch + RR;                 // [2]     logdet M, ok flag
  double* wbase = misc + 2;
  const int per_warp = 2 * V + 2 * RR + 3 * R;
  double* hk = wbase + warp * per_warp;    // [V]  1/S_(k,l)
  double* gk = hk + V;                     // [V]  gamma_(k,l)/S_(k,l)
  double* A = gk + V;                      // [RR] Sigma^-1, then its Cholesky factor
  double* A0 = A + RR;                     // [RR] Sigma^-1 kept for aux / jitter
  double* bv = A0 + RR;                    // [R]
  double* mt = bv + R;                     // [R]
  double* zz = mt + R;                     // [R]

  const double* up = e.u + (size_t)c * V * R;
  for (int i = tid; i < V * R; i += blockDim.x) ulam[i] = up[i] * e.lambda[c * R + (i % R)];
  for (int i = tid; i < RR; i += blockDim.x) Mch[i] = e.M[(size_t)c * RR + i];
  __syncthreads();
  if (tid < 32) {
    // M^-1 and logdet M through the Cholesky factor of M, by warp 0: chol, then lane j inverts column j of L
    // (forward substitution, written over Minv as Linv), then Minv = Linv' Linv with the lanes over its entries
    const bool ok = warp_chol(Mch, R, lane);
    double* Li = A0;                        // warp 0's own scratch (its per-node use starts after the barrier)
    if (lane < R) {
      const int j = lane;
      for (int i = 0; i < j; ++i) Li[i + R * j] = 0.0;
      Li[j + R * j] = 1.0 / Mch[j + R * j];
      for (int i = j + 1; i < R; ++i) {
        double sv = 0.0;
        for (int p = j; p < i; ++p) sv -= Mch[i + R * p] * Li[p + R * j];
        Li[i + R * j] = sv / Mch[i + R * i];
      }
    }
    __syncwarp();
    for (int en = lane; en < RR; en += 32) {
      const int a = en % R, b = en / R;
      double sv = 0.0;
      for (int p = (a > b ? a : b); p < R; ++p) sv += Li[p + R * a] * Li[p + R * b];
      Minv[en] = sv;
    }
    if (lane == 0) {
      double ld = 0.0;
      for (int i = 0; i < R; ++i) ld += log(Mch[i + R * i]);
      misc[0] = 2.0 * ld;
      misc[1] = ok ? 1.0 : 0.0;
    }
  }
  __syncthreads();

  const int k = blockIdx.x * UXI_WARPS + warp;
  if (k >= V) return;
  const double tau2 = e.tau2[c];
  const double* Sg = e.S + (size_t)c * d.qp;
  const double* Gg = e.gamma + (size_t)c * d.qp;
  for (int l = lane; l < V; l += 32) {
    if (l == k) { hk[l] = 0.0; gk[l] = 0.0; continue; }
    const int hi = l > k ? l : k, lo = l > k ? k : l;
    const int j = lo * V - (lo * (lo - 1)) / 2 + (hi - lo);
    const double hinv = 1.0 / Sg[j];
    hk[l] = hinv;
    gk[l] = Gg[j] * hinv;
  }
  __syncwarp();
  const int ntri = R * (R + 1) / 2;
  for (int en = lane; en < ntri + R; en += 32) {
    if (en < ntri) {
      int a = 0, rem = en;            // (a, b) with b <= a, row-wise enumeration of the lower triangle
      while (rem > a) { rem -= a + 1; ++a; }
      const int b = rem;
      double s = 0.0;
      for (int l = 0; l < V; ++l) s += ulam[l * R + a] * ulam[l * R + b] * hk[l];
      s = s / tau2 + Minv[a + R * b];
      A[a + R * b] = s; A[b + R * a] = s;
    } else {
      const int a = en - ntri;
      double s = 0.0;
      for (int l = 0; l < V; ++l) s += ulam[l * R + a] * gk[l];
      bv[a] = s / tau2;
    }
  }
  __syncwarp();
  // Cholesky of Sigma^-1 with the reference's jitter ladder (src/gibbs.jl:322-347: +1e-5 I, then a further +4e-5 I),
  // by the whole warp; the O(R^2) solves and the sequential draws stay with lane 0
  int status = 0;
  if (misc[1] == 0.0) status |= BNR_ST_SIGMA_NOTPD_;
  status |= warp_chol_ladder(A, A0, R, lane);
  if (lane == 0) {
    // mu_t = Sigma b : solve L w = b, L' mu_t = w
    double ldA = 0.0;
    for (int i = 0; i < R; ++i) {
      double s = bv[i];
      for (int p = 0; p < i; ++p) s -= A[i + R * p] * mt[p];
      mt[i] = s / A[i + R * i];
      ldA += log(A[i + R * i]);
    }
    ldA *= 2.0;
    for (int i = R - 1; i >= 0; --i) {
      double s = mt[i];
      for (int p = i + 1; p < R; ++p) s -= A[p + R * i] * mt[p];
      mt[i] = s / A[i + R * i];
    }
    double quad = 0.0;
    for (int i = 0; i < R; ++i) quad += bv[i] * mt[i];
    const double Dl = e.Delta[c];
    const double lo = (log(Dl) - log1p(-Dl)) - 0.5 * misc[0] - 0.5 * ldA + 0.5 * quad;
    const double w = 1.0 / (1.0 + exp(lo));
    const long long it = *e.iter + 1;
    const InjLayout L = InjLayout::make(d.n, V, R, d.gigK);
    DrawStream st(chain_key(d, c), (uint32_t)it, SITE_UXI, (uint32_t)k,
                  e.inj ? e.inj + (size_t)c * e.inj_stride + L.uxi + (size_t)k * (R + 1) : nullptr, R + 1);
    const double ups = st.uniform();
    double xi;
    if (w <= 0.0) xi = 1.0;
    else if (w >= 1.0) xi = 0.0;
    else if (w != w) { xi = (ups <= 0.5) ? 1.0 : 0.0; status |= BNR_ST_NAN_; }
    else xi = (ups <= 1.0 - w) ? 1.0 : 0.0;
    for (int r = 0; r < R; ++r) zz[r] = st.normal();
    // inv(C.U) z : solve L' x = z
    for (int i = R - 1; i >= 0; --i) {
      double s = zz[i];
      for (int p = i + 1; p < R; ++p) s -= A[p + R * i] * zz[p];
      zz[i] = s / A[i + R * i];
    }
    double* un = e.u_alt + (size_t)c * V * R + (size_t)k * R;
    for (int r = 0; r < R; ++r) un[r] = xi * (mt[r] + zz[r]);
    e.xi[c * V + k] = xi;
    if (status) atomicOr(&e.status[c], status);
    if (e.aux.sigma_inv) {
      const size_t o = ((size_t)c * V + k);
      for (int a = 0; a < R; ++a)
        for (int b = 0; b < R; ++b) {
          e.aux.sigma_inv[o * RR + a + R * b] = A0[a + R * b];
          e.aux.sigma_chol[o * RR + a + R * b] = (a >= b) ? A[a + R * b] : 0.0;
        }
      for (int r = 0; r < R; ++r) e.aux.mu_t[o * R + r] = mt[r];
      e.aux.log_odds[o] = lo;
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// edge preparation for the gamma draw (update_gamma!, src/gibbs.jl:421-429): W = lower_triangle(u' Lambda u) with the
// NEW u and OLD lambda, delta1 = sqrt(tau2 S) z1, v = W + delta1.   grid = (nparts, C), block = PART_BLOCK.
// draw_v = 0 only refreshes W (step-mode helper).
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PART_BLOCK) k_edge_prep(Engine e, int draw_v) {
  extern __shared__ double sm[];
  const Dims& d = e.d;
  const int c = blockIdx.y, tid = threadIdx.x;
  double* us = sm;
  double* lam = us + d.V * d.R;
  for (int i = tid; i < d.V * d.R; i += blockDim.x) us[i] = e.u[(size_t)c * d.V * d.R + i];
  if (tid < d.R) lam[tid] = e.lambda[c * d.R + tid];
  __syncthreads();
  const int j = blockIdx.x * PART_BLOCK + tid;
  if (j >= d.q) return;
  const int2 lk = e.edge_lk[j];
  double w = 0.0;
  for (int r = 0; r < d.R; ++r) w += lam[r] * us[lk.y * d.R + r] * us[lk.x * d.R + r];
  const size_t o = (size_t)c * d.qp + j;
  e.W[o] = w;
  if (draw_v) {
    const long long it = *e.iter + 1;
    const InjLayout L = InjLayout::make(d.n, d.V, d.R, d.gigK);
    DrawStream st(chain_key(d, c), (uint32_t)it, SITE_GAMMA_Z1, (uint32_t)j,
                  e.inj ? e.inj + (size_t)c * e.inj_stride + L.z1 + j : nullptr, 1);
    const double z = st.normal();
    // n-form: v = W + delta1, delta1 = sqrt(tau2 S) z1;  q-form (draw_v == 2): the raw normal, used as L' beta = w + z
    e.v[o] = (draw_v == 2) ? z : w + sqrt(e.tau2[c] * e.S[o]) * z;
  }
}

// rhs = a1 - a3 = (y - mu - X(W + delta1))/tau - z2   (src/gibbs.jl:432-434).  grid = (ceil(np/256), C)
// q-form: rhs = (y - mu - X W)/tau2 (xv then holds X W); X' rhs is the linear term of the q x q system.
__global__ void __launch_bounds__(256) k_rhs(Engine e) {
  const Dims& d = e.d;
  const int c = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= d.np) return;
  double r = 0.0;
  if (i < d.n && d.gmode == 2) {
    r = (e.y[i] - e.mu[c] - e.xv[(size_t)c * d.np + i]) / e.tau2[c];
  } else if (i < d.n) {
    const long long it = *e.iter + 1;
    const InjLayout L = InjLayout::make(d.n, d.V, d.R, d.gigK);
    DrawStream st(chain_key(d, c), (uint32_t)it, SITE_GAMMA_Z2, (uint32_t)i,
                  e.inj ? e.inj + (size_t)c * e.inj_stride + L.z2 + i : nullptr, 1);
    const double tau = sqrt(e.tau2[c]);
    r = (e.y[i] - e.mu[c] - e.xv[(size_t)c * d.np + i]) / tau - st.normal();
  }
  e.rhs[(size_t)c * d.np + i] = r;
}

// ------------------------------------------------------------------------------------------------------------
// gamma finish + S (GIG) + lambda sufficient statistics, one thread per edge.
//   gamma_j = v_j + tau S_j t_j                      (src/gibbs.jl:435-436), t = X' a4
//   S_j ~ GIG(1/2, psi = theta_prev, chi = (gamma_j - W_j)^2 / tau2)   (update_D!, src/gibbs.jl:454-458, src/gig.jl)
//   partials: A_r = sum_j p_rj e_j/(tau2 S_j), B_r = sum_j p_rj^2/(tau2 S_j), sum S   (p_rj = u_rk u_rl, e = gamma - W)
// flags: 1 = finish gamma, 2 = draw S, 4 = finish gamma in the q-form (gamma = W + beta, beta in e.t).
// grid = (nparts, C), block = PART_BLOCK.
// ------------------------------------------------------------------------------------------------------------
// (3 blocks per SM: the rejection samplers are chains of dependent FP64 transcendental sequences, so the kernel is bound by
//  how many warps an SM can interleave -- 105 registers allowed 16 warps, 79 allow 24: config 4 1.404 -> 1.380 ms; 64
//  registers would spill)
__global__ void __launch_bounds__(PART_BLOCK, 3) k_gamma_gig(Engine e, int flags) {
  extern __shared__ double sm[];
  const Dims& d = e.d;
  const int c = blockIdx.y, tid = threadIdx.x, R = d.R;
  double* us = sm;                       // [V*R]
  double* red = us + d.V * d.R;          // [(2R+1) * 8]
  for (int i = tid; i < d.V * d.R; i += blockDim.x) us[i] = e.u[(size_t)c * d.V * d.R + i];
  __syncthreads();
  const int j = blockIdx.x * PART_BLOCK + tid;
  const double tau2 = e.tau2[c];
  double acc[2 * MAX_R + 1];
#pragma unroll
  for (int i = 0; i < 2 * MAX_R + 1; ++i) acc[i] = 0.0;
  if (j < d.q) {
    const size_t o = (size_t)c * d.qp + j;
    double g, s = e.S[o];
    if (flags & 4) {
      g = e.W[o] + e.t[o];
      e.gamma[o] = g;
    } else if (flags & 1) {
      g = e.v[o] + sqrt(tau2) * s * e.t[o];
      e.gamma[o] = g;
    } else {
      g = e.gamma[o];
    }
    const double ee = g - e.W[o];
    if (flags & 2) {
      const double chi = ee * ee / tau2;
      const long long it = *e.iter + 1;
      const InjLayout L = InjLayout::make(d.n, d.V, R, d.gigK);
      DrawStream st(chain_key(d, c), (uint32_t)it, SITE_S, (uint32_t)j,
                    e.inj ? e.inj + (size_t)c * e.inj_stride + L.S + (size_t)j * d.gigK : nullptr, d.gigK);
      bool capped = false;
      s = sample_gig(0.5, chi, e.theta[c], st, capped);
      e.S[o] = s;
      int status = 0;
      if (st.exhausted) status |= BNR_ST_INJ_EXHAUSTED_;
      else if (capped) status |= BNR_ST_GIG_CAP_;
      if (status) atomicOr(&e.status[c], status);
      if (e.aux.chi) { e.aux.chi[o] = chi; e.aux.gig_used[o] = e.inj ? (double)st.pos : 2.0 * st.sub; }
    }
    const int2 lk = e.edge_lk[j];
    const double inv = 1.0 / (tau2 * s);
    for (int r = 0; r < R; ++r) {
      const double p = us[lk.y * R + r] * us[lk.x * R + r];
      acc[r] = p * ee * inv;
      acc[R + r] = p * p * inv;
    }
    acc[2 * R] = s;
  }
  // deterministic block reduction of the 2R+1 partial sums
  const int lane = tid & 31, warp = tid >> 5, nv = 2 * R + 1;
  for (int i = 0; i < nv; ++i) {
    const double v = warp_sum(acc[i]);
    if (lane == 0) red[i * 8 + warp] = v;
  }
  __syncthreads();
  if (tid < nv) {
    double s = 0.0;
    for (int w = 0; w < PART_BLOCK / 32; ++w) s += red[tid * 8 + w];
    e.partials[((size_t)c * d.nparts + blockIdx.x) * (2 * MAX_R + 1) + tid] = s;
  }
}

// ------------------------------------------------------------------------------------------------------------
// scalar / small conditionals, one block per chain (mask selects which ones run; gibbs_sample! order):
//   theta (476-479), Delta (496-499 + sample_Beta 130-140), M (516-547), mu (565-570), lambda (586-613), pi (630-636)
// grid = C, block = 256.
// ------------------------------------------------------------------------------------------------------------
// The draws of the different conditionals are independent streams, so they run CONCURRENTLY on different warps
// (warp 1: theta, 2: Delta, 3: mu, 4..: the Bartlett variates of M, one stream per variate; 7: lambda / pi per r);
// warp 0 then does the R x R linear algebra of M.  A single sequential thread used to take ~40 us here.
__global__ void __launch_bounds__(256) k_finish(Engine e, int mask) {
  extern __shared__ double sm[];
  const Dims& d = e.d;
  const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, R = d.R, V = d.V, RR = R * R;
  double* us = sm;                 // [V*R]
  double* psi = us + V * R;        // [4 * RR]: Psi, chol(Psi), Bartlett factor, Y (M update)
  double* sums = psi + 4 * RR;     // [2*MAX_R+1]
  double* red = sums + 2 * MAX_R + 1;  // [32]
  const long long it = *e.iter + 1;
  const InjLayout L = InjLayout::make(d.n, V, R, d.gigK);
  const double* injc = e.inj ? e.inj + (size_t)c * e.inj_stride : nullptr;
  const RngKey key = chain_key(d, c);
  const bool do_theta = mask & (1 << BNR_COND_THETA_), do_delta = mask & (1 << BNR_COND_DELTA_);
  const bool do_M = mask & (1 << BNR_COND_M_), do_mu = mask & (1 << BNR_COND_MU_);
  const bool do_lam = mask & (1 << BNR_COND_LAMBDA_), do_pi = mask & (1 << BNR_COND_PI_);

  for (int i = tid; i < V * R; i += blockDim.x) us[i] = e.u[(size_t)c * V * R + i];
  if (tid < 2 * R + 1) {
    double s = 0.0;
    for (int p = 0; p < d.nparts; ++p) s += e.partials[((size_t)c * d.nparts + p) * (2 * MAX_R + 1) + tid];
    sums[tid] = s;
  }
  // block reductions first (every thread takes part): sum xi, #{xi != 0}, sum (y - X gamma)
  double sx = 0.0, nz = 0.0, sy = 0.0;
  if (do_delta || do_M) {
    for (int k = tid; k < V; k += blockDim.x) {
      const double x = e.xi[c * V + k];
      sx += x;
      nz += (fabs(x) > 0.1) ? 1.0 : 0.0;
    }
    sx = block_sum(sx, red);
    nz = block_sum(nz, red);
  }
  if (do_mu) {
    for (int i = tid; i < d.n; i += blockDim.x) sy += e.y[i] - e.xg[(size_t)c * d.np + i];
    sy = block_sum(sy, red);
  }
  __syncthreads();                 // us, sums complete
  double* Lp = psi + RR;           // chol(Psi), lower
  double* Ab = Lp + RR;            // Bartlett factor, lower
  double* Yw = Ab + RR;            // Y = A^-1 Lp'
  const double df = d.nu + nz;

  if (warp == 0 && do_M) {
    // Psi = I + sum_k u_k u_k'
    for (int en = lane; en < RR; en += 32) {
      const int a = en % R, b = en / R;
      double s = (a == b) ? 1.0 : 0.0;
      for (int k = 0; k < V; ++k) s += us[k * R + a] * us[k * R + b];
      psi[en] = s;
      Lp[en] = s;
    }
  } else if (warp == 1 && lane == 0 && do_theta) {
    const double shape = d.zeta + 0.5 * (double)V * (V + 1);
    const double scale = 2.0 / (2.0 * d.iota + sums[2 * R]);
    DrawStream st(key, (uint32_t)it, SITE_THETA, 0, injc ? injc + L.theta : nullptr, 1);
    e.theta[c] = st.gamma(shape) * scale;
    if (e.aux.theta_params) { e.aux.theta_params[2 * c] = shape; e.aux.theta_params[2 * c + 1] = scale; }
  } else if (warp == 2 && lane == 0 && do_delta) {
    const double a = d.a_delta + sx, b = d.b_delta + ((double)V - sx);
    DrawStream st(key, (uint32_t)it, SITE_DELTA, 0, injc ? injc + L.Delta : nullptr, 3);
    double dl;
    if (a > 0.0 && b > 0.0) {
      const double ga = st.gamma(a), gb = st.gamma(b);
      dl = ga / (ga + gb);
    } else if (a > 0.0) dl = 1.0;
    else if (b > 0.0) dl = 0.0;
    else {
      if (injc) { st.pos = 2; }
      dl = (st.uniform() < 0.5) ? 0.0 : 1.0;
    }
    e.Delta[c] = dl;
    if (e.aux.delta_params) { e.aux.delta_params[2 * c] = a; e.aux.delta_params[2 * c + 1] = b; }
  } else if (warp == 3 && lane == 0 && do_mu) {
    const double m = sy / d.n, sd = sqrt(e.tau2[c] / d.n);
    DrawStream st(key, (uint32_t)it, SITE_MU, 0, injc ? injc + L.mu : nullptr, 1);
    e.mu[c] = m + sd * st.normal();
    if (e.aux.mu_params) { e.aux.mu_params[2 * c] = m; e.aux.mu_params[2 * c + 1] = sd; }
  } else if (warp >= 4 && warp <= 6 && do_M) {
    // Bartlett variates, one Philox stream per variate (element = its index): R chi-squares (diagonal), then the
    // strictly-lower normals row by row -- the same order as the injected layout
    const int nvar = R + R * (R - 1) / 2;
    for (int v = (warp - 4) * 32 + lane; v < nvar; v += 96) {
      DrawStream st(key, (uint32_t)it, SITE_M, (uint32_t)v, injc ? injc + L.M + v : nullptr, 1);
      if (v < R) {
        const double ci = injc ? st.uniform() : 2.0 * st.gamma(0.5 * (df - v));
        Ab[v + R * v] = sqrt(ci);
      } else {
        int i = 1, rem = v - R;
        while (rem >= i) { rem -= i; ++i; }
        Ab[i + R * rem] = st.normal();
      }
    }
  } else if (warp == 7 && lane < R && (do_lam || do_pi)) {
    const int r = lane;
    const double vals[3] = {0.0, 1.0, -1.0};
    double lam_new = e.lambda[c * R + r];
    if (do_lam) {
      // loglik_v - loglik_(current) = (v - lam) A_r - 1/2 (v - lam)^2 B_r ; every r uses the OLD lambda elsewhere
      const double lam = lam_new, Ar = sums[r], Br = sums[R + r];
      double dl[3], mx = -1e300;
      for (int v = 0; v < 3; ++v) {
        const double dv = vals[v] - lam;
        dl[v] = dv * Ar - 0.5 * dv * dv * Br;
        mx = dl[v] > mx ? dl[v] : mx;
      }
      double w[3], tot = 0.0;
      for (int v = 0; v < 3; ++v) {
        w[v] = e.pi[((size_t)c * R + r) * 3 + v] * exp(dl[v] - mx);
        tot += w[v];
        if (e.aux.lambda_logw) {
          e.aux.lambda_logw[(size_t)c * 3 * R + r + R * v] = dl[v] - mx;
          e.aux.lambda_w[(size_t)c * 3 * R + r + R * v] = w[v];
        }
      }
      DrawStream st(key, (uint32_t)it, SITE_LAMBDA, (uint32_t)r, injc ? injc + L.lambda + r : nullptr, 1);
      const double t = st.uniform() * tot;
      int i = 0;
      double cw = w[0];
      while (cw < t && i < 2) { ++i; cw += w[i]; }
      lam_new = vals[i];
      if (tot != tot) atomicOr(&e.status[c], BNR_ST_NAN_);
    }
    if (do_pi) {
      double al[3] = {pow((double)(r + 1), d.eta), 1.0, 1.0};
      if (lam_new == 1.0) al[1] += 1.0;
      else if (lam_new == 0.0) al[0] += 1.0;
      else al[2] += 1.0;
      DrawStream st(key, (uint32_t)it, SITE_PI, (uint32_t)r, injc ? injc + L.pi + 3 * r : nullptr, 3);
      double g[3], tot = 0.0;
      for (int v = 0; v < 3; ++v) { g[v] = st.gamma(al[v]); tot += g[v]; }
      for (int v = 0; v < 3; ++v) {
        e.pi[((size_t)c * R + r) * 3 + v] = g[v] / tot;
        if (e.aux.pi_alpha) e.aux.pi_alpha[(size_t)c * 3 * R + r + R * v] = al[v];
      }
    }
    // (every r reads and writes only its own lambda_r / pi_r)
    if (do_lam) e.lambda[c * R + r] = lam_new;
  }
  if (!do_M) return;
  __syncthreads();                 // Psi / Lp (warp 0) and the Bartlett factor (warps 4-6) are in shared memory
  if (warp == 0) {
    // Cholesky of Psi, column by column: lane i owns row i (same summation order as small_chol)
    bool ok = true;
    for (int j = 0; j < R; ++j) {
      double sdot = 0.0;
      if (lane >= j && lane < R) {
        sdot = Lp[lane + R * j];
        for (int p = 0; p < j; ++p) sdot -= Lp[lane + R * p] * Lp[j + R * p];
      }
      const double dj = __shfl_sync(0xffffffffu, sdot, j);
      if (!(dj > 0.0)) ok = false;
      const double rt = sqrt(dj);
      if (lane == j) Lp[j + R * j] = rt;
      else if (lane > j && lane < R) Lp[lane + R * j] = sdot / rt;
      __syncwarp();
    }
    if (!ok && lane == 0) atomicOr(&e.status[c], BNR_ST_PSI_NOTPD_);
    // Y = A^-1 Lp'  (forward substitution; lane = column), then M = Y' Y (lanes over the R^2 entries)
    if (lane < R) {
      const int col = lane;
      for (int i = 0; i < R; ++i) {
        double sv = (col >= i) ? Lp[col + R * i] : 0.0;   // Lp'(i, col) = Lp(col, i)
        for (int p = 0; p < i; ++p) sv -= Ab[i + R * p] * Yw[p + R * col];
        Yw[i + R * col] = sv / Ab[i + R * i];
      }
    }
    __syncwarp();
    for (int en = lane; en < RR; en += 32) {
      const int a = en % R, b = en / R;
      double sv = 0.0;
      for (int p = 0; p < R; ++p) sv += Yw[p + R * a] * Yw[p + R * b];
      e.M[(size_t)c * RR + a + R * b] = sv;
    }
    if (e.aux.m_params) {
      double* o = e.aux.m_params + (size_t)c * (1 + 2 * RR);
      if (lane == 0) o[0] = df;
      for (int en = lane; en < RR; en += 32) {
        const int a = en % R, b = en / R;
        o[1 + a + R * b] = psi[a + R * b];
        o[1 + RR + a + R * b] = (a >= b) ? Lp[a + R * b] : 0.0;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// prior initialisation (initialize_variables!, src/gibbs.jl:191-224).  grid = C, block = 256.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_init(Engine e) {
  extern __shared__ double sm[];
  const Dims& d = e.d;
  const int c = blockIdx.x, tid = threadIdx.x, R = d.R, V = d.V, RR = R * R;
  double* us = sm;        // [V*R]
  double* lam = us + V * R;
  const InitLayout L = InitLayout::make(V, R);
  const double* injc = e.inj ? e.inj + (size_t)c * e.inj_stride : nullptr;
  const RngKey key = chain_key(d, c);
  const double theta = 0.5, tau2 = 1.0;
  const double eta = d.eta > 1.0 ? d.eta : 1.01;
  // S_j ~ Exponential(mean theta/2)
  for (int j = tid; j < d.q; j += blockDim.x) {
    DrawStream st(key, 0, SITE_INIT_S, (uint32_t)j, injc ? injc + L.S + j : nullptr, 1);
    const double ex = injc ? st.uniform() : -log(st.uniform());
    e.S[(size_t)c * d.qp + j] = ex * (theta / 2.0);
  }
  if (tid < R) {
    const int r = tid;
    DrawStream st(key, 0, SITE_INIT_PI, (uint32_t)r, injc ? injc + L.pi + 3 * r : nullptr, 3);
    const double al[3] = {pow((double)(r + 1), eta), 1.0, 1.0};
    double g[3], tot = 0.0;
    for (int v = 0; v < 3; ++v) { g[v] = st.gamma(al[v]); tot += g[v]; }
    double w[3];
    for (int v = 0; v < 3; ++v) { w[v] = g[v] / tot; e.pi[((size_t)c * R + r) * 3 + v] = w[v]; }
    DrawStream s2(key, 0, SITE_INIT_LAMBDA, (uint32_t)r, injc ? injc + L.lambda + r : nullptr, 1);
    const double t = s2.uniform() * (w[0] + w[1] + w[2]);
    int i = 0;
    double cw = w[0];
    while (cw < t && i < 2) { ++i; cw += w[i]; }
    const double vals[3] = {0.0, 1.0, -1.0};
    lam[r] = vals[i];
    e.lambda[c * R + r] = vals[i];
  }
  for (int k = tid; k < V; k += blockDim.x) {
    DrawStream st(key, 0, SITE_INIT_XI, (uint32_t)k, injc ? injc + L.xi + k : nullptr, 1);
    e.xi[c * V + k] = (st.uniform() <= 0.5) ? 1.0 : 0.0;
    DrawStream su(key, 0, SITE_INIT_U, (uint32_t)k, injc ? injc + L.u + (size_t)k * R : nullptr, R);
    for (int r = 0; r < R; ++r) {
      const double z = su.normal();
      us[k * R + r] = z;
      e.u[(size_t)c * V * R + k * R + r] = z;
    }
  }
  if (tid == 0) {
    e.theta[c] = theta; e.Delta[c] = 0.5; e.mu[c] = 1.0; e.tau2[c] = tau2;
    // M ~ InverseWishart(nu, I): Bartlett A, M = A^-T A^-1
    DrawStream st(key, 0, SITE_INIT_M, 0, injc ? injc + L.M : nullptr, R + R * (R - 1) / 2);
    double Ab[MAX_R * MAX_R], Y[MAX_R * MAX_R];
    for (int i = 0; i < R; ++i) {
      const double ci = injc ? st.uniform() : 2.0 * st.gamma(0.5 * (d.nu - i));
      Ab[i + R * i] = sqrt(ci);
    }
    for (int i = 0; i < R; ++i)
      for (int j = 0; j < i; ++j) Ab[i + R * j] = st.normal();
    for (int col = 0; col < R; ++col)
      for (int i = 0; i < R; ++i) {
        double s = (col == i) ? 1.0 : 0.0;
        for (int p = 0; p < i; ++p) s -= Ab[i + R * p] * Y[p + R * col];
        Y[i + R * col] = s / Ab[i + R * i];
      }
    for (int a = 0; a < R; ++a)
      for (int b = 0; b < R; ++b) {
        double s = 0.0;
        for (int p = 0; p < R; ++p) s += Y[p + R * a] * Y[p + R * b];
        e.M[(size_t)c * RR + a + R * b] = s;
      }
  }
  __syncthreads();
  for (int j = tid; j < d.q; j += blockDim.x) {
    const int2 lk = e.edge_lk[j];
    double w = 0.0;
    for (int r = 0; r < R; ++r) w += lam[r] * us[lk.y * R + r] * us[lk.x * R + r];
    DrawStream st(key, 0, SITE_INIT_GAMMA, (uint32_t)j, injc ? injc + L.gamma + j : nullptr, 1);
    const size_t o = (size_t)c * d.qp + j;
    e.gamma[o] = w + sqrt(tau2 * e.S[o]) * st.normal();
  }
}

// ------------------------------------------------------------------------------------------------------------
// trace rows + streaming split-half moments (replaces the T-row state Table and return_psrf_VOI's copies,
// src/gibbs.jl:835-841, 771-789).  grid = (ceil((V+q)/256), C), block = 256.
// Full trace rows hold the state variables in state_var order (bnr_engine.cuh)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_record(Engine e, int sweep_done /* 1: state belongs to sweep iter+1 */) {
  const Dims& d = e.d;
  const int c = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const long long sweep = *e.iter + (sweep_done ? 1 : 0);
  const long long row = *e.trace_row;
  const int np_ = d.V + d.q;
  if (p < np_) {
    const double x = (p < d.V) ? e.xi[c * d.V + p] : e.gamma[(size_t)c * d.qp + (p - d.V)];
    if (e.tr_gx.holds(c, row)) e.tr_gx.row(c, row)[p] = x;
    e.mom.add(c, p, sweep, x);
  }
  if (e.tr_full.holds(c, row)) {
    double* dst = e.tr_full.row(c, row);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e.tr_full.width; i += gridDim.x * blockDim.x) {
      int j = i;               // walk the state table to the variable that holds element i of the row
#pragma unroll
      for (int v = 0; v < NUM_STATE_VARS; ++v) {
        const StateVar s = state_var(d, v);
        if (j >= 0 && j < s.count) dst[i] = (e.*s.at)[(size_t)c * s.stride + j];
        j -= s.count;
      }
    }
  }
}

// one prediction row per chain: pred[c][row][j] = mu_c + sum_z partial_z[c][j] (z in split order) (+ sqrt(tau2_c) z_j,
// z_j from the SITE_PRED stream of element j at the row's sweep); held-out rows (mode 2) store
// -1/2 log(2 pi tau2_c) - (y_j - mu_c - sum_z partial_z[c][j])^2 / (2 tau2_c) and draw nothing.  grid = (ceil(m / 256), C)
__global__ void __launch_bounds__(256) k_pred_record(Engine e, int sweep_done /* 1: state belongs to sweep iter+1 */) {
  const int c = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  const long long row = *e.trace_row;
  if (j >= e.pred.width || !e.pred.holds(c, row)) return;
  const size_t stride = (size_t)e.d.C * e.pred_mp;
  const double* w = e.pred_ws + (size_t)c * e.pred_mp + j;
  double s = 0.0;
  for (int z = 0; z < e.pred_splits; ++z) s += w[z * stride];
  if (e.pred_mode == 2) {
    const double t2 = e.tau2[c];
    const double r = e.pred_y[j] - e.mu[c] - s;
    e.pred.row(c, row)[j] = -0.5 * log(6.283185307179586 * t2) - r * r / (2.0 * t2);
    return;
  }
  double v = e.mu[c] + s;
  if (e.pred_mode == 1) {
    const long long sweep = *e.iter + (sweep_done ? 1 : 0);
    DrawStream st(chain_key(e.d, c), (uint32_t)sweep, SITE_PRED, (uint32_t)j);
    v += sqrt(e.tau2[c]) * st.normal();
  }
  e.pred.row(c, row)[j] = v;
}

// one log-likelihood row per chain: ll[c][row][i] = -1/2 log(2 pi tau2_c) - (y_i - mu_c - (X gamma_c)_i)^2 / (2 tau2_c),
// X gamma from the cache e.xg (valid for the new gamma once launch_finish ran).  grid = (ceil(n / 256), C)
__global__ void __launch_bounds__(256) k_loglik_record(Engine e) {
  const int c = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  const long long row = *e.trace_row;
  if (i >= e.ll.width || !e.ll.holds(c, row)) return;
  const double t2 = e.tau2[c];
  const double r = e.y[i] - e.mu[c] - e.xg[(size_t)c * e.d.np + i];
  e.ll.row(c, row)[i] = -0.5 * log(6.283185307179586 * t2) - r * r / (2.0 * t2);
}

__global__ void k_advance(Engine e, int inc_iter) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (inc_iter) *e.iter += 1;
    *e.trace_row += 1;
  }
}

// raw streams for the parity tests (bnr_rng_stream / bnr_rng_gamma)
__global__ void k_rng_dump(Dims d, int chain, long long iteration, int site, int element, int kind, double shape,
                           int count, double* out) {
  if (threadIdx.x || blockIdx.x) return;
  DrawStream st(chain_key(d, chain), (uint32_t)iteration, (uint32_t)site, (uint32_t)element);
  for (int i = 0; i < count; ++i) out[i] = kind == 0 ? st.uniform() : (kind == 1 ? st.normal() : st.gamma(shape));
}

// ------------------------------------------------------------------------------------------------------------
// launch wrappers
// ------------------------------------------------------------------------------------------------------------
static size_t smem_u(const Dims& d) { return sizeof(double) * ((size_t)d.V * d.R + d.R + 64); }

// the per-chain kernels keep u (V x R doubles) in dynamic shared memory: allow more than the 48 KB default
// (bnr_create rejects problems beyond 200 KB)
void small_kernels_setup() {
  const int lim = 200 * 1024;
  cudaFuncSetAttribute(k_tau2, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_uxi, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_edge_prep, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_gamma_gig, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_init, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
}

int tau2_blocks(int q) {
  int nb = (q + 1023) / 1024;
  return nb < 1 ? 1 : (nb > TAU2_MAX_BLOCKS ? TAU2_MAX_BLOCKS : nb);
}
void launch_tau2(const Engine& e, cudaStream_t s) {
  dim3 grid(tau2_blocks(e.d.q), e.d.C);
  ++g_launches; k_tau2<<<grid, 256, smem_u(e.d), s>>>(e);
}
void launch_uxi(const Engine& e, cudaStream_t s) {
  const Dims& d = e.d;
  const size_t per_warp = 2 * d.V + 2 * d.R * d.R + 3 * d.R;
  const size_t sm = sizeof(double) * ((size_t)d.V * d.R + 2 * d.R * d.R + 2 + UXI_WARPS * per_warp);
  dim3 grid((d.V + UXI_WARPS - 1) / UXI_WARPS, d.C);
  ++g_launches; k_uxi<<<grid, 32 * UXI_WARPS, sm, s>>>(e);
}
void launch_edge_prep(const Engine& e, int draw_v, cudaStream_t s) {
  dim3 grid(e.d.nparts, e.d.C);
  ++g_launches; k_edge_prep<<<grid, PART_BLOCK, smem_u(e.d), s>>>(e, draw_v);
}
void launch_rhs(const Engine& e, cudaStream_t s) {
  dim3 grid((e.d.np + 255) / 256, e.d.C);
  ++g_launches; k_rhs<<<grid, 256, 0, s>>>(e);
}
void launch_gamma_gig(const Engine& e, int flags, cudaStream_t s) {
  dim3 grid(e.d.nparts, e.d.C);
  const size_t sm = sizeof(double) * ((size_t)e.d.V * e.d.R + (2 * MAX_R + 1) * 8);
  ++g_launches; k_gamma_gig<<<grid, PART_BLOCK, sm, s>>>(e, flags);
}
void launch_finish(const Engine& e, int mask, cudaStream_t s) {
  const size_t sm = sizeof(double) * ((size_t)e.d.V * e.d.R + 4 * e.d.R * e.d.R + 2 * MAX_R + 1 + 32);
  ++g_launches; k_finish<<<e.d.C, 256, sm, s>>>(e, mask);
}
void launch_init(const Engine& e, cudaStream_t s) {
  ++g_launches; k_init<<<e.d.C, 256, smem_u(e.d), s>>>(e);
}
void launch_record(const Engine& e, int sweep_done, cudaStream_t s) {
  dim3 grid((e.d.V + e.d.q + 255) / 256, e.d.C);
  ++g_launches; k_record<<<grid, 256, 0, s>>>(e, sweep_done);
}
void launch_pred_record(const Engine& e, int sweep_done, cudaStream_t s) {
  dim3 grid((e.pred.width + 255) / 256, e.d.C);
  ++g_launches; k_pred_record<<<grid, 256, 0, s>>>(e, sweep_done);
}
void launch_loglik_record(const Engine& e, cudaStream_t s) {
  dim3 grid((e.ll.width + 255) / 256, e.d.C);
  ++g_launches; k_loglik_record<<<grid, 256, 0, s>>>(e);
}
void launch_advance(const Engine& e, int inc_iter, cudaStream_t s) { k_advance<<<1, 32, 0, s>>>(e, inc_iter); }
void launch_rng_dump(const Dims& d, int chain, long long iteration, int site, int element, int kind, double shape,
                     int count, double* out, cudaStream_t s) {
  ++g_launches; k_rng_dump<<<1, 32, 0, s>>>(d, chain, iteration, site, element, kind, shape, count, out);
}

}  // namespace bnr
