// lab harness: the pooled prediction select (launch_pred_select: rows split over blocks, global integer histograms)
// against k_summary_select (launch_summary_select: one block per 8 columns streams every row) on the same buffer of
// N rows x m doubles, as bnr_prediction_summary sees it after a fit (not part of the product).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 tools/lab/pred_select_lab.cu -o tools/lab/pred_select_lab
//   tools/lab/pred_select_lab [N] [m]        (default N = 64 x 20000, m = 100)
// Times are the best of 5 event-timed calls after a warm-up call; both must give the same order statistics bit for bit.
#include "../../bayesiannetworkregression.jl_b200/csrc/bnr_diagnostics.cu"
#include <cstdio>
#include <cstdlib>
#include <vector>
namespace bnr { thread_local long long g_launches = 0; }

__global__ void k_fill(double* x, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t o[4];
  bnr::philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 7u, 0u, 12345u, 678u, o);
  const double a = bnr::u64_to_unit(o[0], o[1]), b = bnr::u64_to_unit(o[2], o[3]);
  x[i] = 50.0 + 10.0 * sqrt(-2.0 * log(a)) * cospi(2.0 * b);
}

int main(int argc, char** argv) {
  const long long N = argc > 1 ? atoll(argv[1]) : 64LL * 20000;
  const int m = argc > 2 ? atoi(argv[2]) : 100;
  const long long lw = llrint(N * 0.025), hi = llrint(N * 0.975);
  double* rows = nullptr;
  const size_t n = (size_t)N * m;
  if (cudaMalloc(&rows, n * sizeof(double)) != cudaSuccess) { printf("alloc failed\n"); return 1; }
  k_fill<<<(unsigned)((n + 255) / 256), 256>>>(rows, n);
  double* out = nullptr;
  cudaMalloc(&out, 6 * (size_t)m * sizeof(double));
  void* ws = nullptr;
  cudaMalloc(&ws, bnr::pred_select_ws_bytes(N, m));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  auto best = [&](auto&& fn) {
    fn();
    float b = 1e30f;
    for (int r = 0; r < 5; ++r) {
      cudaEventRecord(e0);
      fn();
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      if (ms < b) b = ms;
    }
    return b;
  };
  const float t_sum = best([&] {
    bnr::launch_summary_select(rows, m, 0, m, 0, N, lw, hi, out, out + m, out + 2 * m, 0);
  });
  const float t_pred = best([&] {
    bnr::launch_pred_select(rows, N, m, lw, hi, out + 3 * m, out + 4 * m, out + 5 * m, ws, 0);
  });
  std::vector<double> h(6 * (size_t)m);
  cudaMemcpy(h.data(), out, h.size() * sizeof(double), cudaMemcpyDeviceToHost);
  int same = 1;
  double dmean = 0;
  for (int j = 0; j < m; ++j) {
    same &= h[m + j] == h[4 * m + j] && h[2 * m + j] == h[5 * m + j];
    dmean = fmax(dmean, fabs(h[j] - h[3 * m + j]) / fabs(h[j]));
  }
  const double gb = n * 8.0 / 1e9;
  printf("N = %lld rows x m = %d (%.2f GB), ranks %lld / %lld: k_summary_select %.3f ms, pooled select %.3f ms "
         "(%.1fx); order statistics identical: %s, largest relative mean difference %.1e; %s\n",
         N, m, gb, lw, hi, t_sum, t_pred, t_sum / t_pred, same ? "yes" : "NO", dmean,
         cudaGetErrorString(cudaGetLastError()));
  return same ? 0 : 1;
}
