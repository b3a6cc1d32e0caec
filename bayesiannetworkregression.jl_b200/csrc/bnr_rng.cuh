// Counter-based random numbers for the Gibbs engine: Philox4x32-10 (Salmon et al. 2011).
// key = (seed, global chain id), counter = (sub-block, element, draw site, iteration), so any draw
// of any chain can be regenerated independently of how chains are spread over GPUs.
// A DrawStream hands out U(0,1) / N(0,1) / Gamma(a,1) variates for ONE (iteration, site, element);
// in injection mode (parity tests) it reads them sequentially from a caller-provided array instead.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bnr {

// draw sites (Philox counter word 2)
enum Site : uint32_t {
  SITE_TAU2 = 1, SITE_UXI = 2, SITE_GAMMA_Z1 = 3, SITE_GAMMA_Z2 = 4, SITE_S = 5, SITE_THETA = 6,
  SITE_DELTA = 7, SITE_M = 8, SITE_MU = 9, SITE_LAMBDA = 10, SITE_PI = 11,
  SITE_PRED = 12,   // predictive noise of the predictions for new networks (k_pred_record); not an injected site
  SITE_INIT_S = 20, SITE_INIT_PI = 21, SITE_INIT_LAMBDA = 22, SITE_INIT_XI = 23, SITE_INIT_M = 24,
  SITE_INIT_U = 25, SITE_INIT_GAMMA = 26
};

__host__ __device__ inline void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3,
                                              uint32_t k0, uint32_t k1) {
  const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
  const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
  const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
  const uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
  const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
  c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c0, c1, c2, c3, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// 64 random bits -> double in the open interval (0,1) with 53-bit resolution
__host__ __device__ inline double u64_to_unit(uint32_t lo, uint32_t hi) {
  const uint64_t x = ((uint64_t)hi << 32) | lo;
  return ((double)(x >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}

struct RngKey {
  uint32_t k0, k1;
};

__host__ __device__ inline RngKey make_key(uint64_t seed, uint32_t global_chain) {
  RngKey k;
  k.k0 = (uint32_t)seed;
  k.k1 = (uint32_t)(seed >> 32) ^ (global_chain * 2654435761u);
  return k;
}

struct DrawStream {
  const double* inj;   // injected variates for this stream (nullptr = Philox)
  int pos;             // next injected value
  int inj_len;         // injected values available (exhaustion is flagged, not UB)
  RngKey key;
  uint32_t elem, site, iter;
  uint32_t sub;        // Philox blocks consumed so far
  double ubuf, nbuf;
  bool has_u, has_n, exhausted;

  __device__ DrawStream(RngKey k, uint32_t iteration, uint32_t site_, uint32_t element,
                        const double* injected = nullptr, int injected_len = 0)
      : inj(injected), pos(0), inj_len(injected_len), key(k), elem(element), site(site_), iter(iteration),
        sub(0), ubuf(0), nbuf(0), has_u(false), has_n(false), exhausted(false) {}

  __device__ double injected_next() {
    if (pos >= inj_len) { exhausted = true; return 0.5; }
    return inj[pos++];
  }

  __device__ void block(double& a, double& b) {
    uint32_t o[4];
    philox4x32_10(sub, elem, site, iter, key.k0, key.k1, o);
    ++sub;
    a = u64_to_unit(o[0], o[1]);
    b = u64_to_unit(o[2], o[3]);
  }

  __device__ double uniform() {
    if (inj) return injected_next();
    if (has_u) { has_u = false; return ubuf; }
    double a, b;
    block(a, b);
    ubuf = b; has_u = true;
    return a;
  }

  // normal() and gamma() are deliberately NOT inlined: every per-chain kernel draws a handful of variates from one or
  // two threads, i.e. this transcendental-heavy code runs once per launch and cold from the instruction cache (about
  // 10 cycles per instruction); one shared copy per module is fetched once instead of once per call site.
  __device__ __noinline__ double normal() {
    if (inj) return injected_next();
    if (has_n) { has_n = false; return nbuf; }
    double a, b;
    block(a, b);
    const double r = sqrt(-2.0 * log(a));
    double s, c;
    sincospi(2.0 * b, &s, &c);
    nbuf = r * s; has_n = true;
    return r * c;
  }

  // Gamma(shape, 1): Marsaglia & Tsang (2000); shape < 1 via the U^(1/shape) boost.
  __device__ __noinline__ double gamma(double shape) {
    if (inj) return injected_next();
    double boost = 1.0;
    if (shape < 1.0) {
      boost = pow(uniform(), 1.0 / shape);
      shape += 1.0;
    }
    const double d = shape - 1.0 / 3.0;
    const double c = 1.0 / sqrt(9.0 * d);
    for (int it = 0; it < 1000; ++it) {
      const double x = normal();
      double v = 1.0 + c * x;
      if (v <= 0.0) continue;
      v = v * v * v;
      const double u = uniform();
      if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) return boost * d * v;
    }
    return boost * d;  // unreachable in practice (acceptance > 95 % per attempt)
  }
};

}  // namespace bnr
