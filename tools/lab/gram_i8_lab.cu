// lab harness: time k_gram_slice and k_gram_i8 on their own, on synthetic data (not part of the product).
// Build variants (the macros exist only here, never in the library build):
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DLABNAME='"full"' tools/lab/gram_i8_lab.cu -lcuda
//   ... -DGI_LAB_LOADS_ONLY: the MMA thread waits for each stage and releases it without issuing (the TMA feed alone)
//   ... -DGI_LAB_MMA_ONLY:   the ring is filled once, then the k loop issues without waiting on TMA (the MMAs alone)
//   ... -DGS_LAB_NO_STORES:  both slicing kernels compute the digits but write no planes (rscale is written)
//   ... -DGS_LAB_NO_DIGITS:  both slicing kernels store placeholder words made from X, without the digit math
// Shapes: BASELINE config 3 (V = 100, n = 1000) with 64 chains and config 5 (V = 50, n = 500) with 128 chains.
// Times are the best of 7 event-timed launches after a warm-up launch.  'slice' is k_gram_slice as the library launches
// it (launch_gram_slice), 'ref' the previous kernel (32 rows x one chain per CTA, kept below as k_gram_slice_ref);
// 'write' is the plane bytes (7 np qp per chain) over the kernel time.
// `gram_i8_lab check` (full build only) compares the planes and row scales of both kernels byte for byte instead.
#include "../../bayesiannetworkregression.jl_b200/csrc/bnr_linalg.cu"
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>
namespace bnr { thread_local long long g_launches = 0; }
#ifndef LABNAME
#define LABNAME "full"
#endif

// the previous k_gram_slice, unchanged except for the lab macros: grid = (np / 32, C), block = 256
__global__ void __launch_bounds__(256) k_gram_slice_ref(const double* __restrict__ X, const double* __restrict__ S, int np,
                                                        int q, int qp, signed char* __restrict__ planes,
                                                        double* __restrict__ rscale) {
  using bnr::GI_S;
  __shared__ unsigned buf[GI_S][32][33];
  __shared__ double red[8][32];
  const int c = blockIdx.y, r0 = blockIdx.x * 32, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = r0 + lane;
  const double* Sc = S + (size_t)c * qp;
  double m = 0.0;
  for (int k0 = warp; k0 < q; k0 += 8 * 32) {
    const int kl = k0 + 8 * lane;
    const double sq = kl < q ? sqrt(Sc[kl]) : 0.0;
    const int nk = (q - k0 + 7) / 8 < 32 ? (q - k0 + 7) / 8 : 32;
    for (int j = 0; j < nk; ++j) m = fmax(m, fabs(X[row + (size_t)np * (k0 + 8 * j)] * __shfl_sync(0xffffffffu, sq, j)));
  }
  red[warp][lane] = m;
  __syncthreads();
  m = 0.0;
#pragma unroll
  for (int w = 0; w < 8; ++w) m = fmax(m, red[w][lane]);
  int p = 0;
  if (m > 0.0) {
    p = 54 - ilogb(m);
    if (ldexp(m, p) > 126.0 * 0x1p48) --p;
  }
  if (warp == 0) rscale[(size_t)c * np + row] = ldexp(1.0, -p);
  const int p1 = p > 1000 ? 1000 : p;
  const double sc1 = ldexp(1.0, p1), sc2 = ldexp(1.0, p - p1);
  signed char* out = planes + (size_t)c * GI_S * np * qp;
#if defined(GS_LAB_NO_STORES)
  unsigned sink = 0;
#endif
  for (int k0 = 0; k0 < qp; k0 += 128) {
    const int kl = k0 + warp * 16 + (lane & 15);
    const double sq = kl < q ? sqrt(Sc[kl]) : 0.0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int kw = warp * 4 + g;
      unsigned w[GI_S] = {0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int k = k0 + kw * 4 + b;
        const double sqk = __shfl_sync(0xffffffffu, sq, g * 4 + b);
        if (k < q) {
#if defined(GS_LAB_NO_DIGITS)
          const double xv = X[row + (size_t)np * k];
          w[b] |= (unsigned)__double2loint(xv) + (unsigned)__double2loint(sqk); w[4 + (b & 1)] |= __double2hiint(xv);
#else
          const long long M = __double2ll_rn(X[row + (size_t)np * k] * sqk * sc1 * sc2) + 0x808080808080ll;
          const unsigned lo = (unsigned)M ^ 0x80808080u, hi = (unsigned)(M >> 32) ^ 0x8080u;
#pragma unroll
          for (int i = 0; i < 4; ++i) w[GI_S - 1 - i] |= ((lo >> (8 * i)) & 255u) << (8 * b);
#pragma unroll
          for (int i = 0; i < 3; ++i) w[2 - i] |= ((hi >> (8 * i)) & 255u) << (8 * b);
#endif
        }
      }
#pragma unroll
      for (int s = 0; s < GI_S; ++s) buf[s][lane][kw] = w[s];
    }
    __syncthreads();
    for (int id = threadIdx.x; id < GI_S * 32 * 32; id += 256) {
      const int s = id >> 10, rr = (id >> 5) & 31, kw = id & 31;
      const int k = k0 + kw * 4;
#if defined(GS_LAB_NO_STORES)
      if (k < qp) sink ^= buf[s][rr][kw];
#else
      if (k < qp) *reinterpret_cast<unsigned*>(out + ((size_t)s * np + r0 + rr) * qp + k) = buf[s][rr][kw];
#endif
    }
    __syncthreads();
  }
#if defined(GS_LAB_NO_STORES)
  if (sink == 0x9e3779b9u) planes[0] = 1;
#endif
}

static int cdiv(int a, int b) { return (a + b - 1) / b; }

template <class F>
static float best_ms(F launch) {
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  launch();
  cudaDeviceSynchronize();
  float best = 1e30f;
  for (int r = 0; r < 7; ++r) {
    cudaEventRecord(e0); launch(); cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1); best = ms < best ? ms : best;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return best;
}

struct Problem {
  bnr::Engine e{};
  double *X = nullptr, *S = nullptr, *G = nullptr, *rs = nullptr;
  signed char* planes = nullptr;
  // X like bench.py's synthetic networks (48 % dense, X >= 0), S over 1e-12 .. 1e6.  edges: rows that are all zero,
  // dominated by one entry, or whose maximum is below 2^-946 (scale 2^p with p > 1000: sc1 sc2), and exact zeros in S
  Problem(int V, int n, int C, bool edges) {
    using namespace bnr;
    Dims& d = e.d;
    d.V = V; d.n = n; d.q = V * (V + 1) / 2; d.C = d.C_total = C; d.gmode = 1;
    d.np = cdiv(n + 1, 128) * 128; d.qp = cdiv(d.q, 16) * 16; d.gdim = d.np;
    std::mt19937_64 rng(V * 1000 + n);
    std::uniform_real_distribution<double> U(0.0, 1.0);
    std::vector<double> hx((size_t)d.np * d.qp, 0.0), hs((size_t)C * d.qp, 0.0);
    for (int k = 0; k < d.q; ++k)
      for (int i = 0; i < n; ++i) hx[(size_t)k * d.np + i] = U(rng) < 0.48 ? 0.13 + U(rng) : 0.0;
    for (int c = 0; c < C; ++c)
      for (int k = 0; k < d.q; ++k) hs[(size_t)c * d.qp + k] = exp(log(1e-12) + U(rng) * (log(1e6) - log(1e-12)));
    if (edges) {
      for (int k = 0; k < d.q; ++k) {
        hx[(size_t)k * d.np + 3] = 0.0;                                   // all-zero row
        hx[(size_t)k * d.np + 7] = (k % 3 == 0) ? 0x1p-990 * (1.0 + U(rng)) : 0.0;   // max below 2^-946
        hx[(size_t)k * d.np + n - 1] = (k % 5 == 0) ? 0x1p-1060 * (1.0 + U(rng)) : 0.0;  // subnormal entries
      }
      hx[(size_t)(d.q / 2) * d.np + 11] = 1e4;                           // dominated by one entry
      hx[(size_t)(d.q - 1) * d.np + 12] = 3e5;                           // ... in the last column
      for (int c = 0; c < C; ++c)
        for (int k = c % 11; k < d.q; k += 11) hs[(size_t)c * d.qp + k] = 0.0;   // exact zeros in S
    }
    cudaMalloc(&X, sizeof(double) * hx.size()); cudaMalloc(&S, sizeof(double) * hs.size());
    cudaMalloc(&G, sizeof(double) * (size_t)C * d.np * d.np); cudaMalloc(&rs, sizeof(double) * (size_t)C * d.np);
    cudaMalloc(&planes, (size_t)C * gram_i8_plane_bytes(d));
    cudaMemcpy(X, hx.data(), sizeof(double) * hx.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(S, hs.data(), sizeof(double) * hs.size(), cudaMemcpyHostToDevice);
    e.X = X; e.S = S; e.G = G; e.gram_planes = planes; e.gram_rscale = rs;
  }
  ~Problem() { cudaFree(X); cudaFree(S); cudaFree(G); cudaFree(rs); cudaFree(planes); }
  void slice_ref(signed char* p, double* r) const {
    const bnr::Dims& d = e.d;
    k_gram_slice_ref<<<dim3(d.np / 32, d.C), 256, 0, 0>>>(X, S, d.np, d.q, d.qp, p, r);
  }
};

static void run(const char* name, int V, int n, int C) {
  using namespace bnr;
  Problem pb(V, n, C, false);
  Engine& e = pb.e;
  const Dims& d = e.d;
  const float t_ref = best_ms([&] { pb.slice_ref(pb.planes, pb.rs); });
  const float t_slice = best_ms([&] { launch_gram_slice(e, 0); });
  const float t_i8 = best_ms([&] { launch_gram_i8_products(e, 0); });
  const float t_both = best_ms([&] { launch_syrk_G(e, 0); });
  const float t_fill = best_ms([&] { cudaMemsetAsync(pb.planes, 0, (size_t)C * gram_i8_plane_bytes(d), 0); });
  // operations and operand bytes of the 28 digit products over the stored 128 x 64 tiles
  const int T = d.np / GI_BM, nkb = cdiv(d.qp, GI_BK);
  const double tiles = (double)T * (T + 1) * C;
  const double ops = tiles * 28.0 * 2.0 * GI_BM * GI_BN * (double)nkb * GI_BK;
  const double feed = tiles * (double)nkb * GI_STAGE_BYTES;
  const double wr = (double)C * gram_i8_plane_bytes(d);
  printf("%-6s %-4s C=%-4d np=%-5d qp=%-5d slice %6.3f ms (write %5.2f TB/s of %.2f GB) ref %6.3f ms (%5.2f TB/s) | "
         "products %6.3f ms (%5.2f P int8 op/s, L2->SM %5.2f TB/s over %.1f GB) | both %6.3f ms | memset of the planes %6.3f ms "
         "(%5.2f TB/s)  err=%s\n",
         LABNAME, name, C, d.np, d.qp, t_slice, wr / (t_slice * 1e-3) / 1e12, wr / 1e9, t_ref, wr / (t_ref * 1e-3) / 1e12,
         t_i8, ops / (t_i8 * 1e-3) / 1e15, feed / (t_i8 * 1e-3) / 1e12, feed / 1e9, t_both, t_fill, wr / (t_fill * 1e-3) / 1e12,
         cudaGetErrorString(cudaGetLastError()));
}

__global__ void k_count_diff(const unsigned char* a, const unsigned char* b, size_t n, unsigned long long* cnt,
                             unsigned long long* first) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    if (a[i] != b[i]) { atomicAdd(cnt, 1ull); atomicMin(first, (unsigned long long)i); }
}

static unsigned long long count_diff(const void* a, const void* b, size_t n, unsigned long long* first) {
  unsigned long long *dc, h[2] = {0, ~0ull};
  cudaMalloc(&dc, 2 * sizeof(unsigned long long));
  cudaMemcpy(dc, h, sizeof(h), cudaMemcpyHostToDevice);
  k_count_diff<<<1184, 256>>>((const unsigned char*)a, (const unsigned char*)b, n, dc, dc + 1);
  cudaMemcpy(h, dc, sizeof(h), cudaMemcpyDeviceToHost);
  cudaFree(dc);
  *first = h[1];
  return h[0];
}

// planes and row scales of the launched kernel against the reference, byte for byte; both buffers start from different
// fill bytes, so a byte either kernel leaves unwritten shows as a difference
static bool check(const char* name, int V, int n, int C) {
  using namespace bnr;
  Problem pb(V, n, C, true);
  const Dims& d = pb.e.d;
  const size_t pbytes = (size_t)C * gram_i8_plane_bytes(d), rbytes = sizeof(double) * (size_t)C * d.np;
  signed char* ref_planes;
  double* ref_rs;
  cudaMalloc(&ref_planes, pbytes); cudaMalloc(&ref_rs, rbytes);
  cudaMemset(ref_planes, 0x5a, pbytes); cudaMemset(ref_rs, 0x5a, rbytes);
  cudaMemset(pb.planes, 0xa5, pbytes); cudaMemset(pb.rs, 0xa5, rbytes);
  pb.slice_ref(ref_planes, ref_rs);
  launch_gram_slice(pb.e, 0);
  cudaDeviceSynchronize();
  unsigned long long fp, fr;
  const unsigned long long dp = count_diff(pb.planes, ref_planes, pbytes, &fp), dr = count_diff(pb.rs, ref_rs, rbytes, &fr);
  const bool ok = dp == 0 && dr == 0 && cudaGetLastError() == cudaSuccess;
  printf("check  %-7s C=%-4d np=%-5d qp=%-5d planes %.3f GB: %llu bytes differ, rscale: %llu bytes differ  %s\n", name, C,
         d.np, d.qp, pbytes / 1e9, dp, dr, ok ? "identical" : "DIFFER");
  if (dp) printf("       first differing plane byte at %llu\n", fp);
  if (dr) printf("       first differing rscale byte at %llu\n", fr);
  cudaFree(ref_planes); cudaFree(ref_rs);
  return ok;
}

int main(int argc, char** argv) {
  bnr::linalg_setup();
  cudaDeviceProp p;
  cudaGetDeviceProperties(&p, 0);
  printf("# %s, %d SMs, k-block %d B, %d stages; slicing %d rows x %d chains per CTA\n", p.name, p.multiProcessorCount,
         bnr::GI_BK, bnr::GI_STAGES, bnr::GS_ROWS, bnr::GS_CB);
  if (argc > 1 && !strcmp(argv[1], "check")) {
#if defined(GS_LAB_NO_STORES) || defined(GS_LAB_NO_DIGITS) || defined(GI_LAB_LOADS_ONLY) || defined(GI_LAB_MMA_ONLY)
    printf("check needs the full build\n");
    return 2;
#else
    const int CB = bnr::GS_CB;
    bool ok = true;
    for (int C : {1, CB - 1, CB + 1, 64}) ok = check("c3", 100, 1000, C) && ok;
    for (int C : {1, CB - 1, CB + 1, 2 * CB + 1, 128}) ok = check("c5", 50, 500, C) && ok;
    for (int C : {1, CB - 1, CB + 1}) ok = check("qp1840", 60, 500, C) && ok;
    printf("check: %s\n", ok ? "all identical" : "FAILED");
    return ok ? 0 : 1;
#endif
  }
  run("c3", 100, 1000, 64);
  run("c5", 50, 500, 128);
  return 0;
}
