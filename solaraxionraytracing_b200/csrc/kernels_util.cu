// kernels_util.cu — measurement helpers: FMA issue-rate micro-benchmarks.
//
// MEASURED_PEAKS.json records HBM and bf16 tensor peaks only; the ray-tracing kernels are bound by FP64 / FP32
// CUDA-core issue (no dense contraction on this path), so bench.py measures those two denominators itself, in
// the same run as the throughput number, with these kernels.
#include <cuda_runtime.h>

#include "kernels.h"
#include "sart_internal.h"

namespace sart {

// Folds the image replicas of a launch (fast_params.h: FastTables::nImgRep) into the handle's image and clears them.
__global__ void __launch_bounds__(256) k_fold_replicas(double* __restrict__ rep, double* __restrict__ rep2, int nRep,
                                                       size_t stride, size_t plane, double* __restrict__ image,
                                                       double* __restrict__ imageW2) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= plane) return;
  double a = 0.0, b = 0.0;
  for (int r = 0; r < nRep; ++r) {
    const double x = rep[size_t(r) * stride + i], y = rep2[size_t(r) * stride + i];
    if (x != 0.0 || y != 0.0) { a += x; b += y; rep[size_t(r) * stride + i] = 0.0; rep2[size_t(r) * stride + i] = 0.0; }
  }
  if (a != 0.0 || b != 0.0) { image[i] += a; imageW2[i] += b; }
}
cudaError_t launch_fold_replicas(double* rep, double* rep2, int nRep, size_t stride, size_t plane, double* image,
                                 double* imageW2, cudaStream_t s) {
  k_fold_replicas<<<unsigned((plane + 255) / 256), 256, 0, s>>>(rep, rep2, nRep, stride, plane, image, imageW2);
  return cudaGetLastError();
}

// Folds the spectra replicas of a launch (device_params.h: Spectra) into the handle's spectra and clears them. One block per
// element of the five arrays (eW, eW2, eN [nE1] | sW, sN [SART_MAX_SHELLS]); its threads split the replicas, so that the
// 1024 shell replicas cost 4 loads per thread instead of one thread's 1024 dependent ones.
__global__ void __launch_bounds__(256) k_fold_spectra(const __grid_constant__ Spectra rep, int nE1, const __grid_constant__ Spectra dst) {
  const int b = blockIdx.x;
  const bool energy = b < 3 * nE1;
  const int arr = energy ? b / nE1 : 3 + (b - 3 * nE1) / SART_MAX_SHELLS;
  const int k = energy ? b % nE1 : (b - 3 * nE1) % SART_MAX_SHELLS;
  const bool isCount = arr == 2 || arr == 4;
  unsigned long long* const src[5] = {reinterpret_cast<unsigned long long*>(rep.eW), reinterpret_cast<unsigned long long*>(rep.eW2),
                                      rep.eN, reinterpret_cast<unsigned long long*>(rep.sW), rep.sN};
  unsigned long long* const out[5] = {reinterpret_cast<unsigned long long*>(dst.eW), reinterpret_cast<unsigned long long*>(dst.eW2),
                                      dst.eN, reinterpret_cast<unsigned long long*>(dst.sW), dst.sN};
  const uint32_t nRep = (energy ? rep.eRepMask : rep.sRepMask) + 1u;
  const size_t stride = energy ? size_t(rep.eStride) : size_t(SART_MAX_SHELLS);
  double a = 0.0;
  unsigned long long n = 0ull;
  for (uint32_t r = threadIdx.x; r < nRep; r += blockDim.x) {
    unsigned long long* p = src[arr] + size_t(r) * stride + k;
    const unsigned long long v = *p;
    if (v) { *p = 0ull; if (isCount) n += v; else a += __longlong_as_double(v); }
  }
  for (int o = 16; o > 0; o >>= 1) { a += __shfl_down_sync(0xffffffffu, a, o); n += __shfl_down_sync(0xffffffffu, n, o); }
  __shared__ double sa[8];
  __shared__ unsigned long long sn[8];
  if ((threadIdx.x & 31) == 0) { sa[threadIdx.x >> 5] = a; sn[threadIdx.x >> 5] = n; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < int(blockDim.x >> 5); ++w) { a += sa[w]; n += sn[w]; }
    if (isCount) { if (n) out[arr][k] += n; }
    else if (a != 0.0) reinterpret_cast<double*>(out[arr])[k] += a;
  }
}
cudaError_t launch_fold_spectra(const Spectra& rep, int nE1, const Spectra& dst, cudaStream_t s) {
  k_fold_spectra<<<unsigned(3 * nE1 + 2 * SART_MAX_SHELLS), 256, 0, s>>>(rep, nE1, dst);
  return cudaGetLastError();
}

// Mass scan: adds the mass-major accumulators acc[bin][SART_MAX_MASSES] of a launch to the images [mass][bin] and clears them.
__global__ void __launch_bounds__(256) k_fold_mass_acc(double* __restrict__ acc, double* __restrict__ acc2, int nMasses,
                                                       size_t plane, double* __restrict__ image, double* __restrict__ imageW2) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;   // = bin * SART_MAX_MASSES + mass
  if (i >= plane * SART_MAX_MASSES) return;
  const int m = int(i % SART_MAX_MASSES);
  const size_t bin = i / SART_MAX_MASSES;
  const double a = acc[i], b = acc2[i];
  if (a != 0.0 || b != 0.0) {
    acc[i] = 0.0; acc2[i] = 0.0;
    if (m < nMasses) { image[size_t(m) * plane + bin] += a; imageW2[size_t(m) * plane + bin] += b; }
  }
}
cudaError_t launch_fold_mass_acc(double* acc, double* acc2, int nMasses, size_t plane, double* image, double* imageW2,
                                 cudaStream_t s) {
  const size_t n = plane * SART_MAX_MASSES;
  k_fold_mass_acc<<<unsigned((n + 255) / 256), 256, 0, s>>>(acc, acc2, nMasses, plane, image, imageW2);
  return cudaGetLastError();
}

template <typename T, int kChains>
__global__ void __launch_bounds__(256) k_fma_peak(T* out, T a, T b, int iters) {
  T acc[kChains];
#pragma unroll
  for (int c = 0; c < kChains; ++c) acc[c] = T(threadIdx.x + c);
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int c = 0; c < kChains; ++c) acc[c] = acc[c] * a + b;
  }
  T s = T(0);
#pragma unroll
  for (int c = 0; c < kChains; ++c) s += acc[c];
  if (s == T(-1.2345)) out[blockIdx.x * blockDim.x + threadIdx.x] = s;  // never true: keeps the loop alive
}

template <typename T>
static int measure(int device, double* tflops) {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(SART_ERR_CUDA, "cudaGetDeviceProperties failed");
  constexpr int kChains = 8;
  const int block = 256, grid = prop.multiProcessorCount * 8, iters = 20000;
  T* d = nullptr;
  if (cudaMalloc(&d, size_t(grid) * block * sizeof(T)) != cudaSuccess) return fail(SART_ERR_CUDA, "cudaMalloc failed");
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    k_fma_peak<T, kChains><<<grid, block>>>(d, T(1.0000001), T(1e-7), iters);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(d); return fail(SART_ERR_CUDA, "fma benchmark failed: %s", cudaGetErrorString(cudaGetLastError())); }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flop = 2.0 * double(kChains) * iters * double(grid) * block;
    const double tf = flop / (double(ms) * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  return SART_OK;
}

}  // namespace sart

extern "C" int sart_measure_fma_peak(int device, int fp64, double* tflops) {
  if (!tflops) return sart::fail(SART_ERR_ARG, "tflops is NULL");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) { cudaGetLastError(); return sart::fail(SART_ERR_CUDA, "no such CUDA device %d", device); }
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(device);
  const int rc = fp64 ? sart::measure<double>(device, tflops) : sart::measure<float>(device, tflops);
  cudaSetDevice(prev);
  return rc;
}
