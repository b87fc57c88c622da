// kernels_f32.cu — the single-precision fused Monte Carlo kernel (precision mode 2), sm_100a.
//
// Same decision sequence and weights as kernels_fast.cu (mode 1), with the geometry in FP32 instead of FP64. Mode 1's
// profile on B200 has the FP64 pipe and the XU pipe (MUFU seeds + FP64<->FP32 conversions around them) as its two
// busiest pipes and 76-80 registers per thread; FP32 runs on the 4x wider FMA pipe, needs no conversions and half
// the registers for the ray state. What makes FP32 sufficient here:
//   * the ray is (point, slopes) with |slope| < 0.1 and coordinates < 400 mm, so FP32 rounding is ~1e-5 mm in position
//     and ~1e-9 in direction (a few 1e-5 mm over the 1.5-7.5 m to the detector) — at or below the 1e-4 mm rounding
//     noise the reference itself carries from intersecting lines between points 1.5e14 mm apart (DESIGN.md §3);
//   * every difference of squares that decides a root or a hit is taken in factored form, (rho - R)(rho + R) with rho
//     from one rsqrt, instead of rho^2 - R^2, so no quadratic coefficient loses digits to cancellation;
//   * reciprocals / square roots are MUFU seeds plus one Newton step in FP32 (2-3 FFMA).
// Sampling (integer inverse-CDF search, Philox) and weights (FP32 factors, FP64 product and accumulation) are the very
// same code as mode 1 (fast_common.cuh), so a ray has the same emission shell, energy and exit-disc point in all modes.


#include "trace_f32.cuh"

namespace sart {
namespace fast {

// ---- fused kernel ---------------------------------------------------------------------------------------------
// A ray of stage A that is uncertain (rec.unc) goes to the re-trace queue whatever its code; stage B does the same at its
// own exits. A launch has at most kMaxRaysPerLaunch rays (fast_params.h), so the queue entry (ray index - first) fits 32 bits.
// kSpectra: the generic variant that also fills the spectra (sart_enable_spectra; fast_common.cuh: ImageSinkT). kBands: the
// generic variant that also fills the band images B (sart_enable_band_images), the spectra and the radial histogram checked at
// run time (k_trace_mc_f32_bands).
template <bool kWolter, bool kPlain, bool kAlias, bool kMargins, bool kSpectra, bool kBands>
__device__ __forceinline__ void f32_fused(const FastParams& P, const Geo32& G, const FastTables& T, double mAxion2, uint64_t first,
                                          uint64_t nRays, const PhiloxKeys& K, double* __restrict__ image,
                                          double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                                          const BandImages& B) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32<kAlias>(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill32<kAlias>(P, T, S);
  for (int i = threadIdx.x; i < kWarps32 * int(sizeof(WarpCounters) / 4); i += kBlock32) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  unsigned int* bandN = band_counts<kBands>();
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  auto sink = with_bands<kBands>(ImageSinkT<!kPlain, kSpectra>{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2,
                                                                 sumX, sumY, sumR}, B, bandN);
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  // 32-bit trip count + running 64-bit ray index: 5 loop instructions per ray instead of 12 (nRays <= kMaxRaysPerLaunch,
  // so the count fits)
  const uint64_t i0 = uint64_t(blockIdx.x) * kBlock32 + threadIdx.x;
  nIter = i0 < nRays ? unsigned((nRays - 1 - i0) / stride) + 1u : 0u;
  uint64_t ray = first + i0;
  uint32_t id = uint32_t(i0);
  const uint32_t stride32 = uint32_t(stride);
  for (unsigned k = nIter; k != 0u; --k, ray += stride, id += stride32) {
    Head32 hd;
    stage_a32_head<kPlain, false, kAlias>(P, T, S, K, ray, hd);
    Rec32 rec;
    rec.id = id;
    const int code = stage_a32<kWolter, false, kPlain, false, kAlias, kMargins>(P, G, T, S, hd, rec);
    finish32<kWolter, kPlain, false, kMargins>(P, G, T, S, code, rec, sink);
  }
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(0xffffffffu, nPassed, o);
    nTill += __shfl_down_sync(0xffffffffu, nTill, o);
    nIter += __shfl_down_sync(0xffffffffu, nIter, o);
    sumW += __shfl_down_sync(0xffffffffu, sumW, o);
    sumW2 += __shfl_down_sync(0xffffffffu, sumW2, o);
    sumX += __shfl_down_sync(0xffffffffu, sumX, o);
    sumY += __shfl_down_sync(0xffffffffu, sumY, o);
    sumR += __shfl_down_sync(0xffffffffu, sumR, o);
  }
  __syncwarp();
  if (lane == 0) flush_counters(counters, wc[warp], nIter, nPassed, nTill, sumW, sumW2, sumX, sumY, sumR);
  if (kBands) band_counts_flush(B, bandN);
}
template <bool kWolter, bool kPlain, bool kAlias, bool kMargins, bool kSpectra = false>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_f32(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G, const __grid_constant__ FastTables T,
               double mAxion2, uint64_t first, uint64_t nRays, const __grid_constant__ PhiloxKeys K, double* __restrict__ image,
               double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  f32_fused<kWolter, kPlain, kAlias, kMargins, kSpectra, false>(P, G, T, mAxion2, first, nRays, K, image, imageW2, counters,
                                                                BandImages{});
}
template <bool kWolter, bool kAlias, bool kMargins>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_f32_bands(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G, const __grid_constant__ FastTables T,
                     double mAxion2, uint64_t first, uint64_t nRays, const __grid_constant__ PhiloxKeys K,
                     double* __restrict__ image, double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                     const __grid_constant__ BandImages B) {
  f32_fused<kWolter, false, kAlias, kMargins, true, true>(P, G, T, mAxion2, first, nRays, K, image, imageW2, counters, B);
}
// The generic kind with the quantity histograms QH (sart_enable_quantity_hists; fast_common.cuh: QuantityHistSink), the band
// images B checked at run time. kQH = 1: the block's sums in shared memory, 2: in the block replicas QH.rw / QH.rw2. A copy
// of f32_fused rather than another instantiation of it: the kernels built from f32_fused keep the code they had before.
template <bool kWolter, bool kAlias, bool kMargins, int kQH>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_f32_qhists(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G, const __grid_constant__ FastTables T,
                      double mAxion2, uint64_t first, uint64_t nRays, const __grid_constant__ PhiloxKeys K,
                      double* __restrict__ image, double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                      const __grid_constant__ BandImages B, const __grid_constant__ QuantityHists QH) {
  constexpr bool kPlain = false;
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32<kAlias>(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill32<kAlias>(P, T, S);
  for (int i = threadIdx.x; i < kWarps32 * int(sizeof(WarpCounters) / 4); i += kBlock32) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  unsigned int* bandN = band_counts<true>();
  const QhistSmem qs = qhist_smem<kQH == 1>(tail + kWarps32 * sizeof(WarpCounters), QH);
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  QuantityHistSink<kQH == 1> sink{{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY, sumR}, P, B,
                                  bandN, band_replica(B), QH, qs, qhist_replica(QH)};
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  // 32-bit trip count + running 64-bit ray index: 5 loop instructions per ray instead of 12 (nRays <= kMaxRaysPerLaunch,
  // so the count fits)
  const uint64_t i0 = uint64_t(blockIdx.x) * kBlock32 + threadIdx.x;
  nIter = i0 < nRays ? unsigned((nRays - 1 - i0) / stride) + 1u : 0u;
  uint64_t ray = first + i0;
  uint32_t id = uint32_t(i0);
  const uint32_t stride32 = uint32_t(stride);
  for (unsigned k = nIter; k != 0u; --k, ray += stride, id += stride32) {
    Head32 hd;
    stage_a32_head<kPlain, false, kAlias>(P, T, S, K, ray, hd);
    Rec32 rec;
    rec.id = id;
    const int code = stage_a32<kWolter, false, kPlain, false, kAlias, kMargins>(P, G, T, S, hd, rec);
    finish32<kWolter, kPlain, false, kMargins>(P, G, T, S, code, rec, sink);
  }
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(0xffffffffu, nPassed, o);
    nTill += __shfl_down_sync(0xffffffffu, nTill, o);
    nIter += __shfl_down_sync(0xffffffffu, nIter, o);
    sumW += __shfl_down_sync(0xffffffffu, sumW, o);
    sumW2 += __shfl_down_sync(0xffffffffu, sumW2, o);
    sumX += __shfl_down_sync(0xffffffffu, sumX, o);
    sumY += __shfl_down_sync(0xffffffffu, sumY, o);
    sumR += __shfl_down_sync(0xffffffffu, sumR, o);
  }
  __syncwarp();
  if (lane == 0) flush_counters(counters, wc[warp], nIter, nPassed, nTill, sumW, sumW2, sumX, sumY, sumR);
  band_counts_flush(B, bandN);
  qhist_flush<kQH == 1>(QH, qs);
}

// ---- fused kernel with warp-level compaction between stage A and stage B (see kernels_fast.cu) ----------------
constexpr int kQueue32 = 64;
struct WarpQueue32 {
  float x0[kQueue32], y0[kQueue32], tx[kQueue32], ty[kQueue32], rho0[kQueue32], path2[kQueue32];
  int meta[kQueue32];   // hitLayer | (eIdx or emission shell) << 8 | clamped << 30 | uncertain << 31
  uint32_t we[kQueue32];   // energy word of the ray (solar source: the energy is resolved after the compaction)
  uint32_t id[kQueue32];   // ray index - first ray of the launch
};

template <bool kWolter, bool kPlain, bool kAlias, bool kMargins, bool kSpectra = false>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_f32_compact(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                       const __grid_constant__ FastTables T, double mAxion2, uint64_t first, uint64_t nRays,
                       const __grid_constant__ PhiloxKeys K, double* __restrict__ image, double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32<kAlias>(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  WarpQueue32* queues = reinterpret_cast<WarpQueue32*>(tail + kWarps32 * sizeof(WarpCounters));
  smem_fill32<kAlias>(P, T, S);
  for (int i = threadIdx.x; i < kWarps32 * int(sizeof(WarpCounters) / 4); i += kBlock32) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  __syncthreads();

  constexpr unsigned kFull = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  WarpQueue32& Q = queues[warp];
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  ImageSinkT<!kPlain, kSpectra> sink{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY, sumR};
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  uint64_t base = uint64_t(blockIdx.x) * kBlock32 + (threadIdx.x & ~31);
  const bool solar = kPlain || !P.testXray;
  int qn = 0;
  for (;;) {
    while (qn <= kQueue32 - 32 && base < nRays) {
      const uint64_t i = base + lane;
      base += stride;
      Rec32 rec;
      int code = SART_N_EXIT_CODES;
      if (i < nRays) {
        Head32 hd;
        stage_a32_head<kPlain, true, kAlias>(P, T, S, K, first + i, hd);
        rec.id = uint32_t(i);
        code = stage_a32<kWolter, false, kPlain, true, kAlias, kMargins>(P, G, T, S, hd, rec);
        ++nIter;
        if (code >= 0 && !(kMargins && rec.unc && sink.defer(rec.id))) sink.fail(code);
      }
      const unsigned m = __ballot_sync(kFull, code < 0);
      if (code < 0) {
        const int pos = qn + __popc(m & ((1u << lane) - 1u));
        Q.x0[pos] = rec.x0; Q.y0[pos] = rec.y0; Q.tx[pos] = rec.tx; Q.ty[pos] = rec.ty; Q.rho0[pos] = rec.rho0;
        Q.path2[pos] = rec.path2;
        Q.meta[pos] = rec.hitLayer | ((solar ? rec.rIdx : rec.eIdx) << 8) | (rec.clamped ? (1 << 30) : 0) | (rec.unc ? (1 << 31) : 0);
        Q.we[pos] = rec.we;
        Q.id[pos] = rec.id;
      }
      qn += __popc(m);
    }
    if (qn == 0) break;
    __syncwarp();
    const int take = qn < 32 ? qn : 32;
    if (lane < take) {
      const int pos = qn - take + lane;
      Rec32 rec;
      rec.x0 = Q.x0[pos]; rec.y0 = Q.y0[pos]; rec.tx = Q.tx[pos]; rec.ty = Q.ty[pos]; rec.rho0 = Q.rho0[pos];
      rec.path2 = Q.path2[pos];
      const int meta = Q.meta[pos];
      rec.hitLayer = meta & 0xff; rec.eIdx = (meta >> 8) & 0x3fffff; rec.clamped = (meta >> 30) & 1; rec.unc = meta < 0;
      rec.id = Q.id[pos];
      rec.bud = solar ? (0.0015f + float(rec.eIdx) * 0.0005f) : 1.0f;   // rs of the emission shell (rec.eIdx still holds it)
      if (solar) rec.eIdx = energy_index<kAlias>(P, T, rec.eIdx, Q.we[pos], rec.clamped);
      finish32<kWolter, kPlain, false, kMargins>(P, G, T, S, -1, rec, sink);
    }
    qn -= take;
    __syncwarp();
  }
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(kFull, nPassed, o);
    nTill += __shfl_down_sync(kFull, nTill, o);
    nIter += __shfl_down_sync(kFull, nIter, o);
    sumW += __shfl_down_sync(kFull, sumW, o);
    sumW2 += __shfl_down_sync(kFull, sumW2, o);
    sumX += __shfl_down_sync(kFull, sumX, o);
    sumY += __shfl_down_sync(kFull, sumY, o);
    sumR += __shfl_down_sync(kFull, sumR, o);
  }
  __syncwarp();
  if (lane == 0) flush_counters(counters, wc[warp], nIter, nPassed, nTill, sumW, sumW2, sumX, sumY, sumR);
}

// The same with the band images B, the generic kind (k_trace_mc_f32_bands). Its own copy of the kernel above: the plain variants
// of that kernel, compiled from a body shared with this one, came out with another register allocation than before the band
// images existed, and a run without them is to run the code it ran before.
template <bool kWolter, bool kAlias, bool kMargins>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_f32_compact_bands(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                             const __grid_constant__ FastTables T, double mAxion2, uint64_t first, uint64_t nRays,
                             const __grid_constant__ PhiloxKeys K, double* __restrict__ image, double* __restrict__ imageW2,
                             sart_counters_t* __restrict__ counters, const __grid_constant__ BandImages B) {
  constexpr bool kPlain = false;
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32<kAlias>(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  WarpQueue32* queues = reinterpret_cast<WarpQueue32*>(tail + kWarps32 * sizeof(WarpCounters));
  smem_fill32<kAlias>(P, T, S);
  for (int i = threadIdx.x; i < kWarps32 * int(sizeof(WarpCounters) / 4); i += kBlock32) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  unsigned int* bandN = band_counts<true>();
  __syncthreads();

  constexpr unsigned kFull = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  WarpQueue32& Q = queues[warp];
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  BandImageSink sink{{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY, sumR}, B, bandN,
                     band_replica(B)};
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  uint64_t base = uint64_t(blockIdx.x) * kBlock32 + (threadIdx.x & ~31);
  const bool solar = kPlain || !P.testXray;
  int qn = 0;
  for (;;) {
    while (qn <= kQueue32 - 32 && base < nRays) {
      const uint64_t i = base + lane;
      base += stride;
      Rec32 rec;
      int code = SART_N_EXIT_CODES;
      if (i < nRays) {
        Head32 hd;
        stage_a32_head<kPlain, true, kAlias>(P, T, S, K, first + i, hd);
        rec.id = uint32_t(i);
        code = stage_a32<kWolter, false, kPlain, true, kAlias, kMargins>(P, G, T, S, hd, rec);
        ++nIter;
        if (code >= 0 && !(kMargins && rec.unc && sink.defer(rec.id))) sink.fail(code);
      }
      const unsigned m = __ballot_sync(kFull, code < 0);
      if (code < 0) {
        const int pos = qn + __popc(m & ((1u << lane) - 1u));
        Q.x0[pos] = rec.x0; Q.y0[pos] = rec.y0; Q.tx[pos] = rec.tx; Q.ty[pos] = rec.ty; Q.rho0[pos] = rec.rho0;
        Q.path2[pos] = rec.path2;
        Q.meta[pos] = rec.hitLayer | ((solar ? rec.rIdx : rec.eIdx) << 8) | (rec.clamped ? (1 << 30) : 0) | (rec.unc ? (1 << 31) : 0);
        Q.we[pos] = rec.we;
        Q.id[pos] = rec.id;
      }
      qn += __popc(m);
    }
    if (qn == 0) break;
    __syncwarp();
    const int take = qn < 32 ? qn : 32;
    if (lane < take) {
      const int pos = qn - take + lane;
      Rec32 rec;
      rec.x0 = Q.x0[pos]; rec.y0 = Q.y0[pos]; rec.tx = Q.tx[pos]; rec.ty = Q.ty[pos]; rec.rho0 = Q.rho0[pos];
      rec.path2 = Q.path2[pos];
      const int meta = Q.meta[pos];
      rec.hitLayer = meta & 0xff; rec.eIdx = (meta >> 8) & 0x3fffff; rec.clamped = (meta >> 30) & 1; rec.unc = meta < 0;
      rec.id = Q.id[pos];
      rec.bud = solar ? (0.0015f + float(rec.eIdx) * 0.0005f) : 1.0f;   // rs of the emission shell (rec.eIdx still holds it)
      if (solar) rec.eIdx = energy_index<kAlias>(P, T, rec.eIdx, Q.we[pos], rec.clamped);
      finish32<kWolter, kPlain, false, kMargins>(P, G, T, S, -1, rec, sink);
    }
    qn -= take;
    __syncwarp();
  }
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(kFull, nPassed, o);
    nTill += __shfl_down_sync(kFull, nTill, o);
    nIter += __shfl_down_sync(kFull, nIter, o);
    sumW += __shfl_down_sync(kFull, sumW, o);
    sumW2 += __shfl_down_sync(kFull, sumW2, o);
    sumX += __shfl_down_sync(kFull, sumX, o);
    sumY += __shfl_down_sync(kFull, sumY, o);
    sumR += __shfl_down_sync(kFull, sumR, o);
  }
  __syncwarp();
  if (lane == 0) flush_counters(counters, wc[warp], nIter, nPassed, nTill, sumW, sumW2, sumX, sumY, sumR);
  band_counts_flush(B, bandN);
}
// The same with the quantity histograms QH as well (k_trace_mc_f32_qhists), the band images checked at run time; a copy for
// the same reason.
template <bool kWolter, bool kAlias, bool kMargins, int kQH>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_f32_compact_qhists(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                              const __grid_constant__ FastTables T, double mAxion2, uint64_t first, uint64_t nRays,
                              const __grid_constant__ PhiloxKeys K, double* __restrict__ image, double* __restrict__ imageW2,
                              sart_counters_t* __restrict__ counters, const __grid_constant__ BandImages B,
                              const __grid_constant__ QuantityHists QH) {
  constexpr bool kPlain = false;
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32<kAlias>(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  WarpQueue32* queues = reinterpret_cast<WarpQueue32*>(tail + kWarps32 * sizeof(WarpCounters));
  smem_fill32<kAlias>(P, T, S);
  for (int i = threadIdx.x; i < kWarps32 * int(sizeof(WarpCounters) / 4); i += kBlock32) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  unsigned int* bandN = band_counts<true>();
  const QhistSmem qs = qhist_smem<kQH == 1>(reinterpret_cast<unsigned char*>(queues + kWarps32), QH);
  __syncthreads();

  constexpr unsigned kFull = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  WarpQueue32& Q = queues[warp];
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  QuantityHistSink<kQH == 1> sink{{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY, sumR}, P, B,
                                  bandN, band_replica(B), QH, qs, qhist_replica(QH)};
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  uint64_t base = uint64_t(blockIdx.x) * kBlock32 + (threadIdx.x & ~31);
  const bool solar = kPlain || !P.testXray;
  int qn = 0;
  for (;;) {
    while (qn <= kQueue32 - 32 && base < nRays) {
      const uint64_t i = base + lane;
      base += stride;
      Rec32 rec;
      int code = SART_N_EXIT_CODES;
      if (i < nRays) {
        Head32 hd;
        stage_a32_head<kPlain, true, kAlias>(P, T, S, K, first + i, hd);
        rec.id = uint32_t(i);
        code = stage_a32<kWolter, false, kPlain, true, kAlias, kMargins>(P, G, T, S, hd, rec);
        ++nIter;
        if (code >= 0 && !(kMargins && rec.unc && sink.defer(rec.id))) sink.fail(code);
      }
      const unsigned m = __ballot_sync(kFull, code < 0);
      if (code < 0) {
        const int pos = qn + __popc(m & ((1u << lane) - 1u));
        Q.x0[pos] = rec.x0; Q.y0[pos] = rec.y0; Q.tx[pos] = rec.tx; Q.ty[pos] = rec.ty; Q.rho0[pos] = rec.rho0;
        Q.path2[pos] = rec.path2;
        Q.meta[pos] = rec.hitLayer | ((solar ? rec.rIdx : rec.eIdx) << 8) | (rec.clamped ? (1 << 30) : 0) | (rec.unc ? (1 << 31) : 0);
        Q.we[pos] = rec.we;
        Q.id[pos] = rec.id;
      }
      qn += __popc(m);
    }
    if (qn == 0) break;
    __syncwarp();
    const int take = qn < 32 ? qn : 32;
    if (lane < take) {
      const int pos = qn - take + lane;
      Rec32 rec;
      rec.x0 = Q.x0[pos]; rec.y0 = Q.y0[pos]; rec.tx = Q.tx[pos]; rec.ty = Q.ty[pos]; rec.rho0 = Q.rho0[pos];
      rec.path2 = Q.path2[pos];
      const int meta = Q.meta[pos];
      rec.hitLayer = meta & 0xff; rec.eIdx = (meta >> 8) & 0x3fffff; rec.clamped = (meta >> 30) & 1; rec.unc = meta < 0;
      rec.id = Q.id[pos];
      rec.bud = solar ? (0.0015f + float(rec.eIdx) * 0.0005f) : 1.0f;   // rs of the emission shell (rec.eIdx still holds it)
      if (solar) rec.eIdx = energy_index<kAlias>(P, T, rec.eIdx, Q.we[pos], rec.clamped);
      finish32<kWolter, kPlain, false, kMargins>(P, G, T, S, -1, rec, sink);
    }
    qn -= take;
    __syncwarp();
  }
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(kFull, nPassed, o);
    nTill += __shfl_down_sync(kFull, nTill, o);
    nIter += __shfl_down_sync(kFull, nIter, o);
    sumW += __shfl_down_sync(kFull, sumW, o);
    sumW2 += __shfl_down_sync(kFull, sumW2, o);
    sumX += __shfl_down_sync(kFull, sumX, o);
    sumY += __shfl_down_sync(kFull, sumY, o);
    sumR += __shfl_down_sync(kFull, sumR, o);
  }
  __syncwarp();
  if (lane == 0) flush_counters(counters, wc[warp], nIter, nPassed, nTill, sumW, sumW2, sumX, sumY, sumR);
  band_counts_flush(B, bandN);
  qhist_flush<kQH == 1>(QH, qs);
}
// ---- axion-mass scan with FP32 tracing (the per-mass weighting is fast_common.cuh's mass_scan_loop) --------------
template <bool kWolter, bool kMargins, int kPer, bool kSpectra, bool kRows = false>
__device__ __forceinline__ void f32_masses(const FastParams& P, const Geo32& G, const FastTables& T,
                                           const double* __restrict__ masses, int nMasses, uint64_t first, uint64_t nRays,
                                           const PhiloxKeys& K, double* __restrict__ image, double* __restrict__ imageW2,
                                           sart_counters_t* __restrict__ counters, const MassRows& R = MassRows{}) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill32(P, T, S);
  for (int i = threadIdx.x; i < kWarpsM * int(sizeof(WarpCounters) / 4); i += kBlockM) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  __syncthreads();
  mass_scan_loop<kPer, kSpectra, kRows>(P, T.rad, T.spec, R, masses, nMasses, first, nRays, image, imageW2, counters, wc,
                 [&](uint64_t ray, uint32_t id, RayResult& r) {
    RecordSink<false> sink{r, 0.0, T.rq, true};
    Head32 hd;
    stage_a32_head(P, T, S, K, ray, hd);
    Rec32 rec;
    rec.id = id;
    const int c0 = stage_a32<kWolter, false, false, false, false, kMargins>(P, G, T, S, hd, rec);
    finish32<kWolter, false, false, kMargins>(P, G, T, S, c0, rec, sink);
    return sink.unresolved;
  });
}
template <bool kWolter, bool kMargins, int kPer>
__global__ void __launch_bounds__(kBlockM, SART_F32_MINBLOCKS_M)
k_trace_mc_f32_masses(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                      const __grid_constant__ FastTables T, const double* __restrict__ masses, int nMasses, uint64_t first,
                      uint64_t nRays, const __grid_constant__ PhiloxKeys K, double* __restrict__ image, double* __restrict__ imageW2,
                      sart_counters_t* __restrict__ counters) {
  f32_masses<kWolter, kMargins, kPer, false>(P, G, T, masses, nMasses, first, nRays, K, image, imageW2, counters);
}
// The same with the per-mass spectra (sart_enable_mass_spectra; T.spec holds their accumulators, see mass_spec_add).
template <bool kWolter, bool kMargins, int kPer>
__global__ void __launch_bounds__(kBlockM, SART_F32_MINBLOCKS_M)
k_trace_mc_f32_masses_spectra(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                              const __grid_constant__ FastTables T, const double* __restrict__ masses, int nMasses,
                              uint64_t first, uint64_t nRays, const __grid_constant__ PhiloxKeys K, double* __restrict__ image,
                              double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  f32_masses<kWolter, kMargins, kPer, true>(P, G, T, masses, nMasses, first, nRays, K, image, imageW2, counters);
}
// The same with the per-mass radial histograms and band images R (sart_enable_mass_radial_hist / _band_images; their
// mass-minor accumulators, see mass_scan_loop), and with the per-mass spectra as well (kSpectra).
template <bool kWolter, bool kMargins, int kPer, bool kSpectra>
__global__ void __launch_bounds__(kBlockM, SART_F32_MINBLOCKS_M)
k_trace_mc_f32_masses_rows(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                           const __grid_constant__ FastTables T, const double* __restrict__ masses, int nMasses,
                           uint64_t first, uint64_t nRays, const __grid_constant__ PhiloxKeys K, double* __restrict__ image,
                           double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                           const __grid_constant__ MassRows R) {
  f32_masses<kWolter, kMargins, kPer, kSpectra, true>(P, G, T, masses, nMasses, first, nRays, K, image, imageW2, counters, R);
}

}  // namespace fast

#ifndef SART_NO_LAUNCHERS   // tools/micro/one_kernel.cu instantiates single kernels of this file for SASS inspection
// One launch of at most fast::kMaxRaysPerLaunch rays (api.cu cuts longer runs).
cudaError_t launch_mc_image_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                uint64_t first, uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                sart_counters_t* counters, int smCount, bool compact, cudaStream_t s, const BandImages& bands,
                                const QuantityHists& qh) {
  if (nRays == 0) return cudaSuccess;
  const LaunchVariant v = launch_variant(P, T);
  // the plain-run kernels compile the radial histogram, the spectra, the band images and the quantity histograms out
  const bool plain = v.plain && !T.rad.w && !T.spec.eW && !bands.w && !qh.w;
  const size_t smem = fast::smem_bytes32(P, fast::kWarps32, v.alias) + (compact ? fast::kWarps32 * sizeof(fast::WarpQueue32) : 0);
  // variant 0: inverse-CDF sampler, pure FP32; 1: inverse-CDF sampler with the margin tests (re-trace queue attached); 2: alias
  // sampler (no re-trace: its ray <-> index mapping is not the exact pipeline's)
  const int variant = v.alias ? 2 : (v.margins ? 1 : 0);
  auto run_smem = [&](size_t sm, auto kern, auto... extra) {
    cudaError_t e = fast::set_smem(kern, sm);
    if (e != cudaSuccess) return e;
    unsigned grid = 0;
    if ((e = grid_size(kern, fast::kBlock32, sm, nRays, smCount, 0, &grid)) != cudaSuccess) return e;
    kern<<<grid, fast::kBlock32, sm, s>>>(P, G, T, mAxion * mAxion, first, nRays, philox_round_keys(seed), image, imageW2, counters,
                                           extra...);
    return cudaGetLastError();
  };
  auto run = [&](auto kern, auto... bandArg) { return run_smem(smem, kern, bandArg...); };
  if (getenv("SART_DEBUG"))
    fprintf(stderr, "[sart] k_trace_mc_f32 compact=%d wolter=%d plain=%d alias=%d bands=%d qhists=%d (sampler=%d ra=%p ea=%p) "
            "smem=%zu\n", int(compact), int(v.wolter), int(plain), int(v.alias), bands.nBands, qh.nHists, T.sampler,
            (const void*)T.radiusAlias, (const void*)T.energyAlias, smem);
  if (qh.w) {   // the generic kind with the quantity histograms: everything else is checked at run time
    const bool smemSums = fast::qhist_sums_in_smem(smem, qh.entries);
    using KernQ = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, double, uint64_t, uint64_t, PhiloxKeys, double*,
                           double*, sart_counters_t*, BandImages, QuantityHists);
    // [compact][wolter][variant][sums in shared memory]
#define SART_VAR(K, W, A, M) {fast::K<W, A, M, 2>, fast::K<W, A, M, 1>}
#define SART_ROW(K, W) {SART_VAR(K, W, false, false), SART_VAR(K, W, false, true), SART_VAR(K, W, true, false)}
    static const KernQ table[2][2][3][2] = {{SART_ROW(k_trace_mc_f32_qhists, false), SART_ROW(k_trace_mc_f32_qhists, true)},
                                            {SART_ROW(k_trace_mc_f32_compact_qhists, false),
                                             SART_ROW(k_trace_mc_f32_compact_qhists, true)}};
#undef SART_ROW
#undef SART_VAR
    return run_smem(smem + fast::qhist_smem_bytes(qh.entries, smemSums),
                    table[compact ? 1 : 0][v.wolter ? 1 : 0][variant][smemSums ? 1 : 0], bands, qh);
  }
  if (bands.w) {   // the generic kind with the band images: the radial histogram and the spectra are checked at run time
    using KernB = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, double, uint64_t, uint64_t, PhiloxKeys, double*,
                           double*, sart_counters_t*, BandImages);
    // [compact][wolter][variant]
#define SART_ROW(K, W) {fast::K<W, false, false>, fast::K<W, false, true>, fast::K<W, true, false>}
    static const KernB table[2][2][3] = {{SART_ROW(k_trace_mc_f32_bands, false), SART_ROW(k_trace_mc_f32_bands, true)},
                                         {SART_ROW(k_trace_mc_f32_compact_bands, false), SART_ROW(k_trace_mc_f32_compact_bands, true)}};
#undef SART_ROW
    return run(table[compact ? 1 : 0][v.wolter ? 1 : 0][variant], bands);
  }
  using Kern = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, double, uint64_t, uint64_t, PhiloxKeys, double*, double*,
                        sart_counters_t*);
  // [compact][wolter][kind][variant]; kind 0: generic, 1: plain, 2: generic with the spectra
#define SART_ROW(K, W, PL, SP) {fast::K<W, PL, false, false, SP>, fast::K<W, PL, false, true, SP>, fast::K<W, PL, true, false, SP>}
#define SART_KINDS(K, W) {SART_ROW(K, W, false, false), SART_ROW(K, W, true, false), SART_ROW(K, W, false, true)}
  static const Kern table[2][2][3][3] = {{SART_KINDS(k_trace_mc_f32, false), SART_KINDS(k_trace_mc_f32, true)},
                                         {SART_KINDS(k_trace_mc_f32_compact, false), SART_KINDS(k_trace_mc_f32_compact, true)}};
#undef SART_KINDS
#undef SART_ROW
  const int kind = plain ? 1 : (T.spec.eW ? 2 : 0);
  return run(table[compact ? 1 : 0][v.wolter ? 1 : 0][kind][variant]);
}

cudaError_t launch_mc_image_f32_masses(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T,
                                       int nMasses, const double* dMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                                       double* acc, double* accW2, sart_counters_t* counters, int smCount, cudaStream_t s,
                                       const MassRows& rows) {
  if (nRays == 0) return cudaSuccess;
  const LaunchVariant v = launch_variant(P, T);
  const size_t smem = fast::smem_bytes32(P, fast::kWarpsM);
  auto run = [&](auto kern, auto... extra) {
    cudaError_t e = fast::set_smem(kern, smem);
    if (e != cudaSuccess) return e;
    unsigned grid = 0;
    if ((e = grid_size(kern, fast::kBlockM, smem, nRays, smCount, 0, &grid)) != cudaSuccess) return e;
    kern<<<grid, fast::kBlockM, smem, s>>>(P, G, T, dMasses, nMasses, first, nRays, philox_round_keys(seed), acc, accW2, counters,
                                           extra...);
    return cudaGetLastError();
  };
  using Kern = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, const double*, int, uint64_t, uint64_t, PhiloxKeys, double*,
                        double*, sart_counters_t*);
  constexpr int kAll = SART_MAX_MASSES / 32;
  const int per = nMasses <= 32 ? 0 : (nMasses <= 64 ? 1 : 2);
  // [spectra][wolter][margins][masses per lane]; spectra: T.spec holds the per-mass spectra accumulators
#define SART_ROW(K, W, M) {fast::K<W, M, 1>, fast::K<W, M, 2>, fast::K<W, M, kAll>}
#define SART_KERN(K) {{SART_ROW(K, false, false), SART_ROW(K, false, true)}, {SART_ROW(K, true, false), SART_ROW(K, true, true)}}
  if (rows.rad.w || rows.band.w) {
    using KernR = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, const double*, int, uint64_t, uint64_t, PhiloxKeys,
                           double*, double*, sart_counters_t*, MassRows);
    // [spectra][wolter][margins][masses per lane]
#define SART_ROW_S(W, M, S) {fast::k_trace_mc_f32_masses_rows<W, M, 1, S>, fast::k_trace_mc_f32_masses_rows<W, M, 2, S>, \
                             fast::k_trace_mc_f32_masses_rows<W, M, kAll, S>}
#define SART_KERN_S(S) {{SART_ROW_S(false, false, S), SART_ROW_S(false, true, S)}, {SART_ROW_S(true, false, S), SART_ROW_S(true, true, S)}}
    static const KernR table[2][2][2][3] = {SART_KERN_S(false), SART_KERN_S(true)};
#undef SART_KERN_S
#undef SART_ROW_S
    return run(table[T.spec.eW ? 1 : 0][v.wolter ? 1 : 0][v.margins ? 1 : 0][per], rows);
  }
  static const Kern table[2][2][2][3] = {SART_KERN(k_trace_mc_f32_masses), SART_KERN(k_trace_mc_f32_masses_spectra)};
#undef SART_KERN
#undef SART_ROW
  return run(table[T.spec.eW ? 1 : 0][v.wolter ? 1 : 0][v.margins ? 1 : 0][per]);
}

#endif  // SART_NO_LAUNCHERS

}  // namespace sart
