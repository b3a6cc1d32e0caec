// lab harness: time k_gram_slice and k_gram_i8 on their own, on synthetic data (not part of the product).
// Build variants (the macros exist only here, never in the library build):
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DLABNAME='"full"' tools/lab/gram_i8_lab.cu -lcuda
//   ... -DGI_LAB_LOADS_ONLY: the MMA thread waits for each stage and releases it without issuing (the TMA feed alone)
//   ... -DGI_LAB_MMA_ONLY:   the ring is filled once, then the k loop issues without waiting on TMA (the MMAs alone)
// Shapes: BASELINE config 3 (V = 100, n = 1000) with 64 chains and config 5 (V = 50, n = 500) with 128 chains.
// Times are the best of 7 event-timed launches after a warm-up launch.
#include "../../bayesiannetworkregression.jl_b200/csrc/bnr_linalg.cu"
#include <cstdio>
#include <random>
#include <vector>
namespace bnr { thread_local long long g_launches = 0; }
#ifndef LABNAME
#define LABNAME "full"
#endif

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

static void run(const char* name, int V, int n, int C) {
  using namespace bnr;
  Engine e{};
  Dims& d = e.d;
  d.V = V; d.n = n; d.q = V * (V + 1) / 2; d.C = d.C_total = C; d.gmode = 1;
  d.np = cdiv(n + 1, 128) * 128; d.qp = cdiv(d.q, 16) * 16; d.gdim = d.np;
  // X like bench.py's synthetic networks (48 % dense, X >= 0), S over 1e-12 .. 1e6
  std::mt19937_64 rng(V * 1000 + n);
  std::uniform_real_distribution<double> U(0.0, 1.0);
  std::vector<double> hx((size_t)d.np * d.qp, 0.0), hs((size_t)C * d.qp, 0.0);
  for (int k = 0; k < d.q; ++k)
    for (int i = 0; i < n; ++i) hx[(size_t)k * d.np + i] = U(rng) < 0.48 ? 0.13 + U(rng) : 0.0;
  for (int c = 0; c < C; ++c)
    for (int k = 0; k < d.q; ++k) hs[(size_t)c * d.qp + k] = exp(log(1e-12) + U(rng) * (log(1e6) - log(1e-12)));
  double *X, *S, *G, *rs;
  signed char* planes;
  cudaMalloc(&X, sizeof(double) * hx.size()); cudaMalloc(&S, sizeof(double) * hs.size());
  cudaMalloc(&G, sizeof(double) * (size_t)C * d.np * d.np); cudaMalloc(&rs, sizeof(double) * (size_t)C * d.np);
  cudaMalloc(&planes, (size_t)C * gram_i8_plane_bytes(d));
  cudaMemcpy(X, hx.data(), sizeof(double) * hx.size(), cudaMemcpyHostToDevice);
  cudaMemcpy(S, hs.data(), sizeof(double) * hs.size(), cudaMemcpyHostToDevice);
  e.X = X; e.S = S; e.G = G; e.gram_planes = planes; e.gram_rscale = rs;

  const float t_slice = best_ms([&] {
    k_gram_slice<<<dim3(d.np / 32, d.C), 256, 0, 0>>>(e.X, e.S, d.np, d.q, d.qp, e.gram_planes, e.gram_rscale);
  });
  const float t_i8 = best_ms([&] { launch_gram_i8_products(e, 0); });
  const float t_both = best_ms([&] { launch_syrk_G(e, 0); });
  // operations and operand bytes of the 28 digit products over the stored 128 x 64 tiles
  const int T = d.np / GI_BM, nkb = cdiv(d.qp, GI_BK);
  const double tiles = (double)T * (T + 1) * C;
  const double ops = tiles * 28.0 * 2.0 * GI_BM * GI_BN * (double)nkb * GI_BK;
  const double feed = tiles * (double)nkb * GI_STAGE_BYTES;
  printf("%-6s %-4s C=%-4d np=%-5d qp=%-5d slice %7.3f ms | products %7.3f ms (%5.2f P int8 op/s, L2->SM %5.2f TB/s over "
         "%.1f GB) | both %7.3f ms  err=%s\n",
         LABNAME, name, C, d.np, d.qp, t_slice, t_i8, ops / (t_i8 * 1e-3) / 1e15, feed / (t_i8 * 1e-3) / 1e12, feed / 1e9,
         t_both, cudaGetErrorString(cudaGetLastError()));
  cudaFree(X); cudaFree(S); cudaFree(G); cudaFree(rs); cudaFree(planes);
}

int main() {
  bnr::linalg_setup();
  cudaDeviceProp p;
  cudaGetDeviceProperties(&p, 0);
  printf("# %s, %d SMs, k-block %d B, %d stages\n", p.name, p.multiProcessorCount, bnr::GI_BK, bnr::GI_STAGES);
  run("c3", 100, 1000, 64);
  run("c5", 50, 500, 128);
  return 0;
}
