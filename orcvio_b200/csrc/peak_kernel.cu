// FP64 peak micro-benchmarks (roofline denominators that MEASURED_PEAKS.json does not carry):
// dependent-chain-free DFMA throughput and mma.sync m8n8k4 f64 (DMMA) throughput.
#include <cuda_runtime.h>
#include "../../include/orcvio_b200.h"
#include "kernels.h"
#include "chol.cuh"

namespace {

__global__ void __launch_bounds__(256) k_dfma_peak(double* out, int iters, double seed) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
    a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

__global__ void __launch_bounds__(256) k_dmma_peak(double* out, int iters, double seed) {
  double a = seed + threadIdx.x * 1e-3, b = 1.0 + threadIdx.x * 1e-6;
  double c0 = 0, c1 = 0, d0 = 0, d1 = 0, e0 = 0, e1 = 0, f0 = 0, f1 = 0;
  for (int i = 0; i < iters; ++i) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(e0), "+d"(e1) : "d"(a), "d"(b));
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(f0), "+d"(f1) : "d"(a), "d"(b));
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((c0 + c1) + (d0 + d1)) + ((e0 + e1) + (f0 + f1));
}

// Dependent-chain latencies (cycles per operation) of the FP64 building blocks the factorisation
// kernels are made of: out[0] DFMA, [1] sqrt, [2] divide, [3] rsqrt, [4] shared-memory load,
// [5] __syncthreads with 512 threads, [6] warp shuffle (64-bit).
__global__ void __launch_bounds__(512) k_latency(double* out, double seed) {
  __shared__ double sm[64];
  const int tid = threadIdx.x;
  if (tid < 64) sm[tid] = (double)((tid + 1) & 63);
  __syncthreads();
  const int N = 256;
  double x = seed + 1.5;
  long long t0 = clock64();
  for (int i = 0; i < N; ++i) x = fma(x, 1.0000001, 1e-9);
  long long t1 = clock64();
  double r0 = (double)(t1 - t0) / N;
  double y = seed + 2.0;
  t0 = clock64();
  for (int i = 0; i < N; ++i) y = sqrt(y + 3.0);
  t1 = clock64();
  double r1 = (double)(t1 - t0) / N;
  double z = seed + 2.0;
  t0 = clock64();
  for (int i = 0; i < N; ++i) z = 1.0 / (z + 0.5);
  t1 = clock64();
  double r2 = (double)(t1 - t0) / N;
  double w = seed + 2.0;
  t0 = clock64();
  for (int i = 0; i < N; ++i) w = rsqrt(w + 3.0);
  t1 = clock64();
  double r3 = (double)(t1 - t0) / N;
  int idx = tid & 63;
  t0 = clock64();
  for (int i = 0; i < N; ++i) idx = (int)sm[idx];
  t1 = clock64();
  double r4 = (double)(t1 - t0) / N;
  t0 = clock64();
  for (int i = 0; i < N; ++i) __syncthreads();
  t1 = clock64();
  double r5 = (double)(t1 - t0) / N;
  double v = x;
  t0 = clock64();
  for (int i = 0; i < N; ++i) v = __shfl_xor_sync(0xffffffffu, v, 1) + 1.0;
  t1 = clock64();
  double r6 = (double)(t1 - t0) / N;
  if (tid == 0) {
    out[0] = r0; out[1] = r1; out[2] = r2; out[3] = r3; out[4] = r4; out[5] = r5; out[6] = r6;
    out[7] = x + y + z + w + idx + v;
  }
}


// Single-warp dependent latencies (cycles per operation; warp 0 of a 64-thread CTA runs alone, the second warp
// only idles): out[0] DFMA, [1] DMMA m8n8k4 dependent, [2] DMMA with 2 independent accumulators (per MMA),
// [3] with 4, [4] with 8, [5] 64-bit shuffle + add, [6] 16-byte shared load (pointer chase), [7] fence.acq_rel.cta
// after a shared store, [8] rcp.approx.ftz.f64, [9] DMMA dependent while the other warp of the scheduler... (unused)
__global__ void __launch_bounds__(64) k_latency1(double* out, double seed) {
  __shared__ __align__(16) double sm[128];
  const int tid = threadIdx.x;
  sm[tid] = (double)((2 * tid + 2) & 126);
  sm[tid + 64] = (double)((2 * tid + 2) & 126);
  __syncthreads();
  if (tid >= 32) return;
  const int N = 256;
  double r[10];
  long long t0, t1;
  double x = seed + 1.5;
  t0 = clock64();
#pragma unroll 8
  for (int i = 0; i < N; ++i) x = fma(x, 1.0000001, 1e-9);
  t1 = clock64();
  r[0] = (double)(t1 - t0) / N;
  double a = seed + tid * 1e-3, b = 1.0 + tid * 1e-6;
  double c[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) c[i] = 0.0;
  t0 = clock64();
#pragma unroll 8
  for (int i = 0; i < N; ++i)
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
  t1 = clock64();
  r[1] = (double)(t1 - t0) / N;
  t0 = clock64();
#pragma unroll 4
  for (int i = 0; i < N; ++i) {
#pragma unroll
    for (int u = 0; u < 2; ++u)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[2 * u]), "+d"(c[2 * u + 1]) : "d"(a), "d"(b));
  }
  t1 = clock64();
  r[2] = (double)(t1 - t0) / (2 * N);
  t0 = clock64();
#pragma unroll 2
  for (int i = 0; i < N; ++i) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[2 * u]), "+d"(c[2 * u + 1]) : "d"(a), "d"(b));
  }
  t1 = clock64();
  r[3] = (double)(t1 - t0) / (4 * N);
  t0 = clock64();
  for (int i = 0; i < N; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[2 * u]), "+d"(c[2 * u + 1]) : "d"(a), "d"(b));
  }
  t1 = clock64();
  r[4] = (double)(t1 - t0) / (8 * N);
  double v = x;
  t0 = clock64();
#pragma unroll 8
  for (int i = 0; i < N; ++i) v = __shfl_xor_sync(0xffffffffu, v, 1) + 1.0;
  t1 = clock64();
  r[5] = (double)(t1 - t0) / N;
  int idx = (2 * tid) & 126;
  t0 = clock64();
#pragma unroll 8
  for (int i = 0; i < N; ++i) idx = (int)(*reinterpret_cast<const double2*>(&sm[idx])).x;
  t1 = clock64();
  r[6] = (double)(t1 - t0) / N;
  t0 = clock64();
  for (int i = 0; i < N; ++i) {
    sm[tid] = v + i;
    asm volatile("fence.acq_rel.cta;" ::: "memory");
  }
  t1 = clock64();
  r[7] = (double)(t1 - t0) / N;
  double y = seed + 3.0;
  t0 = clock64();
#pragma unroll 8
  for (int i = 0; i < N; ++i) {
    double q;
    asm volatile("rcp.approx.ftz.f64 %0, %1;" : "=d"(q) : "d"(y));
    y = q + 2.0;
  }
  t1 = clock64();
  r[8] = (double)(t1 - t0) / N;
  r[9] = 0.0;
  double sink = x + v + y + idx + sm[tid];
#pragma unroll
  for (int i = 0; i < 16; ++i) sink += c[i];
  if (tid == 0) {
    for (int i = 0; i < 10; ++i) out[i] = r[i];
    out[10] = sink;
  }
}

}  // namespace

// Stand-alone run of the one-CTA Cholesky (chol.cuh) on a caller-supplied SPD matrix: the unit test
// and the per-phase clock profile of the routine both factorisation kernels are built on.
namespace ob {
template <bool PROF>
__global__ void __launch_bounds__(CHOL_THREADS) k_chol_probe(const double* Ain, const double* Xin, int m, int nx,
                                                             double* Lout, double* Xout, long long* prof) {
  extern __shared__ double sm[];
  __shared__ __align__(16) CholShared cs;
  double* A = sm;
  const int Tm = (m + 7) >> 3;
  chol_init(A, cs, m, nx);
  __syncthreads();
  for (int e = threadIdx.x; e < m * m; e += blockDim.x) {
    const int i = e / m, j = e - i * m;
    if (j <= i) A[chol_at(i, j, Tm)] = Ain[e];
  }
  for (int e = threadIdx.x; e < nx * m; e += blockDim.x) {
    const int q = e / m, k = e - q * m;
    A[chol_at(m + q, k, Tm)] = Xin[e];
  }
  cta_cholesky<PROF>(A, cs, nullptr, m, nx, prof);
  chol_for_rows(A, m, nx, 0, [&](int i, int k, double l) {
    if (i < m) Lout[(size_t)i * m + k] = l;
    else Xout[(size_t)(i - m) * m + k] = l;
  });
}
}  // namespace ob

extern "C" int orcvio_chol_probe(int m, int nx, const double* A, const double* X, double* L, double* Xs,
                                 long long* prof, int reps, float* us) {
  using namespace ob;
  if (m < 1 || m > ORCVIO_LEG + 6 * ORCVIO_MAX_OBS || nx < 0 || m + nx > CHOL_MAXR - 8 ||
      chol_smem_doubles(m, nx) * sizeof(double) > 225 * 1024) return ORCVIO_ERR_ARG;
  double *dA = nullptr, *dX = nullptr, *dL = nullptr, *dXs = nullptr;
  long long* dprof = nullptr;
  const size_t nA = (size_t)m * m, nX = (size_t)std::max(nx, 1) * m;
  if (cudaMalloc(&dA, nA * 8) != cudaSuccess) return ORCVIO_ERR_NO_DEVICE;
  cudaMalloc(&dX, nX * 8);
  cudaMalloc(&dL, nA * 8);
  cudaMalloc(&dXs, nX * 8);
  cudaMalloc(&dprof, 64 * 8 * sizeof(long long));
  cudaMemcpy(dA, A, nA * 8, cudaMemcpyHostToDevice);
  if (nx > 0) cudaMemcpy(dX, X, (size_t)nx * m * 8, cudaMemcpyHostToDevice);
  cudaMemset(dL, 0, nA * 8);
  cudaMemset(dprof, 0, 64 * 8 * sizeof(long long));
  const size_t smem = chol_smem_doubles(m, nx) * sizeof(double);
  auto kp = k_chol_probe<true>;
  auto kf = k_chol_probe<false>;
  cudaFuncSetAttribute(kp, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024);
  cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024);
  kp<<<1, CHOL_THREADS, smem>>>(dA, dX, m, nx, dL, dXs, dprof);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  kf<<<1, CHOL_THREADS, smem>>>(dA, dX, m, nx, dL, dXs, dprof);
  cudaEventRecord(e0);
  for (int r = 0; r < reps; ++r) kf<<<1, CHOL_THREADS, smem>>>(dA, dX, m, nx, dL, dXs, dprof);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  if (us) *us = 1e3f * ms / std::max(reps, 1);
  cudaMemcpy(L, dL, nA * 8, cudaMemcpyDeviceToHost);
  if (nx > 0) cudaMemcpy(Xs, dXs, (size_t)nx * m * 8, cudaMemcpyDeviceToHost);
  if (prof) cudaMemcpy(prof, dprof, 64 * 8 * sizeof(long long), cudaMemcpyDeviceToHost);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(dA); cudaFree(dX); cudaFree(dL); cudaFree(dXs); cudaFree(dprof);
  return cudaGetLastError() == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_latency_probe(double* cycles7) {
  double* out = nullptr;
  if (cudaMalloc(&out, 8 * sizeof(double)) != cudaSuccess) return ORCVIO_ERR_NO_DEVICE;
  k_latency<<<1, 512>>>(out, 0.25);
  k_latency<<<1, 512>>>(out, 0.25);
  double h[8];
  cudaMemcpy(h, out, sizeof(h), cudaMemcpyDeviceToHost);
  cudaFree(out);
  for (int i = 0; i < 7; ++i) cycles7[i] = h[i];
  return cudaGetLastError() == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_latency_probe1(double* cycles10) {
  double* out = nullptr;
  if (cudaMalloc(&out, 16 * sizeof(double)) != cudaSuccess) return ORCVIO_ERR_NO_DEVICE;
  k_latency1<<<1, 64>>>(out, 0.25);
  k_latency1<<<1, 64>>>(out, 0.25);
  double h[16];
  cudaMemcpy(h, out, sizeof(h), cudaMemcpyDeviceToHost);
  cudaFree(out);
  for (int i = 0; i < 10; ++i) cycles10[i] = h[i];
  return cudaGetLastError() == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}

extern "C" int orcvio_fp64_peak(double* dfma_tflops, double* dmma_tflops) {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return ORCVIO_ERR_NO_DEVICE;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int blocks = sms * 8, threads = 256, iters = 8192;
  double* out = nullptr;
  if (cudaMalloc(&out, (size_t)blocks * threads * sizeof(double)) != cudaSuccess) return ORCVIO_ERR_CUDA;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float ms = 0;
  for (int rep = 0; rep < 2; ++rep) {
    cudaEventRecord(e0);
    k_dfma_peak<<<blocks, threads>>>(out, iters, 1.0);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    cudaEventElapsedTime(&ms, e0, e1);
  }
  if (dfma_tflops) *dfma_tflops = 2.0 * 8 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
  for (int rep = 0; rep < 2; ++rep) {
    cudaEventRecord(e0);
    k_dmma_peak<<<blocks, threads>>>(out, iters, 1.0);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    cudaEventElapsedTime(&ms, e0, e1);
  }
  // one warp-level m8n8k4 = 8*8*4 MACs = 512 flop
  if (dmma_tflops) *dmma_tflops = 512.0 * 4 * iters * (double)blocks * (threads / 32) / (ms * 1e-3) / 1e12;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  return cudaGetLastError() == cudaSuccess ? ORCVIO_OK : ORCVIO_ERR_CUDA;
}
