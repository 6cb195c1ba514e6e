// Micro-probe for the EMD kernels on sm_100a: sustained MUFU.EX2 rate (ex2.approx.f32, what __expf issues) on a
// full grid, eight independent chains per thread so that latency does not bound it. Prints one JSON line:
// ex2 per second on the whole GPU, per SM and clock (SM clock from clock64 over the same window).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o ex2_probe ex2_probe.cu
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1);} } while (0)

constexpr int TPB = 512;
constexpr int CHAINS = 8;
constexpr int INNER = 256;

__global__ void __launch_bounds__(TPB) ex2_kernel(int iters, float* out, long long* cycles) {
  float v[CHAINS];
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) v[c] = -1e-3f * (threadIdx.x + c);
  const long long t0 = clock64();
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int j = 0; j < INNER; ++j) {
#pragma unroll
      for (int c = 0; c < CHAINS; ++c) asm volatile("ex2.approx.f32 %0, %0;" : "+f"(v[c]));
    }
  }
  const long long t1 = clock64();
  float s = 0;
#pragma unroll
  for (int c = 0; c < CHAINS; ++c) s += v[c];
  if (s == 12345.0f) out[0] = s;
  if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

int main(int argc, char** argv) {
  const int iters = argc > 1 ? atoi(argv[1]) : 200;
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = sms * 4;                 // 2048 threads per SM
  float* out; long long* cyc;
  CK(cudaMalloc(&out, sizeof(float)));
  CK(cudaMalloc(&cyc, sizeof(long long) * grid));
  ex2_kernel<<<grid, TPB>>>(2, out, cyc);   // warm-up
  CK(cudaDeviceSynchronize());
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
  CK(cudaEventRecord(a));
  ex2_kernel<<<grid, TPB>>>(iters, out, cyc);
  CK(cudaEventRecord(b));
  CK(cudaEventSynchronize(b));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, a, b));
  long long* h = (long long*)malloc(sizeof(long long) * grid);
  CK(cudaMemcpy(h, cyc, sizeof(long long) * grid, cudaMemcpyDeviceToHost));
  long long maxc = 0;
  for (int i = 0; i < grid; ++i) maxc = h[i] > maxc ? h[i] : maxc;
  const double ops = (double)grid * TPB * iters * INNER * CHAINS;
  const double per_sm = ops / sms;
  printf("{\"ex2_per_s\": %.6e, \"ex2_per_clk_per_sm\": %.3f, \"sm_clock_ghz\": %.3f, \"ms\": %.3f, \"sms\": %d}\n",
         ops / (ms * 1e-3), per_sm / (double)maxc, (double)maxc / (ms * 1e6), ms, sms);
  free(h);
  CK(cudaFree(out)); CK(cudaFree(cyc));
  return 0;
}
