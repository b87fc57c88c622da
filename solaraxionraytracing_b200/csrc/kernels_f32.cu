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

#ifndef SART_F32_PAIR_DEFAULT
#define SART_F32_PAIR_DEFAULT 0
#endif

namespace sart {
namespace fast {

// ---- fused kernel ---------------------------------------------------------------------------------------------
// A ray of stage A that is uncertain (rec.unc) goes to the re-trace queue whatever its code; stage B does the same at its
// own exits. The launcher keeps nRays below 2^32, so the queue entry (ray index - first) fits 32 bits.
// kSpectra: the generic variant that also fills the spectra (sart_enable_spectra; fast_common.cuh: ImageSinkT).
template <bool kWolter, bool kPlain, bool kAlias, bool kMargins, bool kSpectra = false>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_f32(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G, const __grid_constant__ FastTables T,
               double mAxion2, uint64_t first, uint64_t nRays, const __grid_constant__ PhiloxKeys K, double* __restrict__ image,
               double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32<kAlias>(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill32<kAlias>(P, T, S);
  for (int i = threadIdx.x; i < kWarps32 * int(sizeof(WarpCounters) / 4); i += kBlock32) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  ImageSinkT<!kPlain, kSpectra> sink{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY, sumR};
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  // 32-bit trip count + running 64-bit ray index: 5 loop instructions per ray instead of 12 (the launcher keeps
  // nRays <= kMaxRaysPerLaunch, so the count fits)
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

// ---- axion-mass scan with FP32 tracing (the per-mass weighting is fast_common.cuh's mass_scan_loop) --------------
template <bool kWolter, bool kMargins, int kPer>
__global__ void __launch_bounds__(kBlockM, SART_F32_MINBLOCKS_M)
k_trace_mc_f32_masses(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                      const __grid_constant__ FastTables T, const double* __restrict__ masses, int nMasses, uint64_t first,
                      uint64_t nRays, const __grid_constant__ PhiloxKeys K, double* __restrict__ image, double* __restrict__ imageW2,
                      sart_counters_t* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill32(P, T, S);
  for (int i = threadIdx.x; i < kWarpsM * int(sizeof(WarpCounters) / 4); i += kBlockM) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  __syncthreads();
  mass_scan_loop<kPer>(P, T.rad, masses, nMasses, first, nRays, image, imageW2, counters, wc,
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

}  // namespace fast

#ifndef SART_NO_LAUNCHERS   // tools/micro/one_kernel.cu instantiates single kernels of this file for SASS inspection
cudaError_t launch_mc_image_f32x2(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion2,
                                  uint64_t first, uint64_t n, const PhiloxKeys& keys, double* image, double* imageW2,
                                  sart_counters_t* counters, int smCount, bool margins, cudaStream_t s);   // kernels_f32x2.cu

// Two rays per thread (kernels_f32x2.cu) for the plain run of a cone telescope without compaction. SART_F32_PAIR=0 / 1 in the
// environment overrides the default for A/B measurements and for the test that compares the two kernels ray set by ray set.
static bool pair_kernel_wanted() {
  const char* e = getenv("SART_F32_PAIR");
  return e ? (e[0] != '0') : (SART_F32_PAIR_DEFAULT != 0);
}

cudaError_t launch_mc_image_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                uint64_t first, uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                sart_counters_t* counters, int smCount, bool compact, cudaStream_t s) {
  if (nRays == 0) return cudaSuccess;
  const bool wolter = P.telKind == SART_TK_XMM || P.telKind == SART_TK_ABRIXAS;
  // alias sampler: solar source only (the X-ray test source draws no table values)
  const bool alias = T.sampler == SART_SAMPLER_ALIAS && !P.testXray && T.radiusAlias && T.energyAlias;
  const size_t smem = fast::smem_bytes32(P, fast::kWarps32, alias) + (compact ? fast::kWarps32 * sizeof(fast::WarpQueue32) : 0);
  const bool plain = !P.testXray && P.stage == SART_SK_VACUUM && !P.rotated && P.flags == 0 && P.reflKind != SART_RK_EFFECTIVE_AREA && !T.rad.w && !T.spec.eW;
  using Kern = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, double, uint64_t, uint64_t, PhiloxKeys, double*, double*,
                        sart_counters_t*);
  // [compact][wolter][kind][variant]; kind 0: generic, 1: plain, 2: generic with the spectra; variant 0: inverse-CDF sampler,
  // pure FP32; 1: inverse-CDF sampler with the margin tests (re-trace queue attached); 2: alias sampler (no re-trace: its
  // ray <-> index mapping is not the exact pipeline's)
#define SART_ROW(K, W, PL, SP) {fast::K<W, PL, false, false, SP>, fast::K<W, PL, false, true, SP>, fast::K<W, PL, true, false, SP>}
#define SART_KINDS(K, W) {SART_ROW(K, W, false, false), SART_ROW(K, W, true, false), SART_ROW(K, W, false, true)}
  static const Kern table[2][2][3][3] = {{SART_KINDS(k_trace_mc_f32, false), SART_KINDS(k_trace_mc_f32, true)},
                                         {SART_KINDS(k_trace_mc_f32_compact, false), SART_KINDS(k_trace_mc_f32_compact, true)}};
#undef SART_KINDS
#undef SART_ROW
  const bool margins = !alias && T.rq.cap != 0u;
  const int kind = plain ? 1 : (T.spec.eW ? 2 : 0);
  const Kern kern = table[compact ? 1 : 0][wolter ? 1 : 0][kind][alias ? 2 : (margins ? 1 : 0)];
  if (getenv("SART_DEBUG"))
    fprintf(stderr, "[sart] k_trace_mc_f32 compact=%d wolter=%d plain=%d alias=%d (sampler=%d ra=%p ea=%p) smem=%zu\n", int(compact),
            int(wolter), int(plain), int(alias), T.sampler, (const void*)T.radiusAlias, (const void*)T.energyAlias, smem);
  cudaError_t e = fast::set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  int perSM = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kern, fast::kBlock32, smem);
  if (e != cudaSuccess) return e;
  if (perSM < 1) perSM = 1;
  const uint64_t cap = uint64_t(smCount) * perSM;
  const PhiloxKeys keys = philox_round_keys(seed);
  const bool pairs = plain && !wolter && !compact && !alias && pair_kernel_wanted();
  for (uint64_t done = 0; done < nRays; done += fast::kMaxRaysPerLaunch) {   // one launch for anything below 6.9e10 rays
    const uint64_t n = nRays - done < fast::kMaxRaysPerLaunch ? nRays - done : fast::kMaxRaysPerLaunch;
    if (pairs) {
      e = launch_mc_image_f32x2(P, G, T, mAxion * mAxion, first + done, n, keys, image, imageW2, counters, smCount, margins, s);
      if (e != cudaSuccess) return e;
      continue;
    }
    const uint64_t want = (n + fast::kBlock32 - 1) / fast::kBlock32;
    const unsigned grid = unsigned(want < cap ? want : cap);
    kern<<<grid, fast::kBlock32, smem, s>>>(P, G, T, mAxion * mAxion, first + done, n, keys, image, imageW2, counters);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

cudaError_t launch_mc_image_f32_masses(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T,
                                       int nMasses, const double* dMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                                       double* acc, double* accW2, sart_counters_t* counters, int smCount, cudaStream_t s) {
  if (nRays == 0) return cudaSuccess;
  const bool wolter = P.telKind == SART_TK_XMM || P.telKind == SART_TK_ABRIXAS;
  const size_t smem = fast::smem_bytes32(P, fast::kWarpsM);
  const bool margins = T.rq.cap != 0u;
  using Kern = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, const double*, int, uint64_t, uint64_t, PhiloxKeys, double*,
                        double*, sart_counters_t*);
  constexpr int kAll = SART_MAX_MASSES / 32;
#define SART_ROW(W, M) {fast::k_trace_mc_f32_masses<W, M, 1>, fast::k_trace_mc_f32_masses<W, M, 2>, fast::k_trace_mc_f32_masses<W, M, kAll>}
  static const Kern table[2][2][3] = {{SART_ROW(false, false), SART_ROW(false, true)}, {SART_ROW(true, false), SART_ROW(true, true)}};
#undef SART_ROW
  const Kern kern = table[wolter ? 1 : 0][margins ? 1 : 0][nMasses <= 32 ? 0 : (nMasses <= 64 ? 1 : 2)];   // masses per lane
  cudaError_t e = fast::set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  int perSM = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kern, fast::kBlockM, smem);
  if (e != cudaSuccess) return e;
  if (perSM < 1) perSM = 1;
  const uint64_t want = (nRays + fast::kBlockM - 1) / fast::kBlockM;
  const uint64_t cap = uint64_t(smCount) * perSM;
  const unsigned grid = unsigned(want < cap ? want : cap);
  kern<<<grid, fast::kBlockM, smem, s>>>(P, G, T, dMasses, nMasses, first, nRays, philox_round_keys(seed), acc, accW2, counters);
  return cudaGetLastError();
}

#endif  // SART_NO_LAUNCHERS

}  // namespace sart
