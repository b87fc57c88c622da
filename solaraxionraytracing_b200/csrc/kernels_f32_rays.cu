// kernels_f32_rays.cu — the per-ray-record kernels of the single-precision pipeline (precision mode 2), sm_100a:
// traceAxionWrapper as a structure of arrays (sart_trace_mc_rays / sart_trace_words), the passed rays only, compacted
// (sart_trace_mc_passed), and tier (a): pre-sampled rays in HBM -> records in HBM (sart_trace_presampled). Device code of
// the pipeline: trace_f32.cuh.
#include "trace_f32.cuh"

namespace sart {
namespace fast {

// ---- per-ray records (traceAxionWrapper in FP32 mode) ----------------------------------------------------------
// `words` (optional, sart_trace_words): SoA [6][nRays] random words used instead of the Philox words of ray first + i.
// kLate: the energy is resolved by energy_index() after stage A, the way the compacting fused kernel does it (otherwise
// inside stage A, the way the plain fused kernel does it) — so the test hook reaches both forms of the search.
// An uncertain ray gets its FP32 record like any other and is queued; the exact pipeline overwrites the record afterwards.
template <bool kWolter, bool kPlain, bool kAlias, bool kLate = false>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_rays_f32(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                    const __grid_constant__ FastTables T, double mAxion2, uint64_t first, uint64_t nRays,
                    const __grid_constant__ PhiloxKeys K, const uint32_t* __restrict__ words, int32_t* __restrict__ oemit,
                    const __grid_constant__ sart_ray_out_t o) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32<kAlias>(P, smem, S, tail);
  smem_fill32<kAlias>(P, T, S);
  __syncthreads();
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  for (uint64_t i = uint64_t(blockIdx.x) * kBlock32 + threadIdx.x; i < nRays; i += stride) {
    RayResult r;
    RecordSink<true> sink{r, mAxion2, T.rq, false};
    Rec32 rec;
    rec.id = uint32_t(i);
    Head32 hd;
    if (words) {
#pragma unroll
      for (int k = 0; k < 6; ++k) hd.w[k] = words[size_t(k) * nRays + i];
    } else {
      ray_words(K, first + i, hd.w);
    }
    stage_a32_head_words<kPlain, kLate, kAlias>(P, T, S, hd);
    const int c0 = stage_a32<kWolter, false, kPlain, kLate, kAlias>(P, G, T, S, hd, rec);
    const bool solar = kPlain || !P.testXray;
    if (kLate && c0 < 0 && solar) rec.eIdx = energy_index<kAlias>(P, T, rec.rIdx, rec.we, rec.clamped);
    finish32<kWolter, kPlain>(P, G, T, S, c0, rec, sink);
    // energiesPre is set for every ray (rt:1818-1819), clipped or not: rays that end in stage A resolve their energy here
    double energy = double(P.srcEnergy);
    if (solar) {
      int eIdx = rec.eIdx;
      bool cl = false;
      if (c0 >= 0) eIdx = energy_index<kAlias>(P, T, hd.rIdx, hd.w[5], cl);
      energy = fmax(__ldg(T.energies + eIdx), 0.03);   // the f64 table value itself (rt:470-471)
    }
    store_record(P, o, i, r, mAxion2, energy);
    if (oemit) oemit[i] = hd.rIdx;
  }
}

// ---- per-ray records of the passed rays only, compacted (sart_trace_mc_passed) --------------------------------------
// Same tracing as k_trace_mc_rays_f32; a warp ballots its passed lanes, one lane reserves that many slots of the output
// with one atomic, and the lanes write their records side by side (coalesced). Uncertain rays are left to the exact
// pipeline's pass over the re-trace queue, which appends its own passed rays. Counters as in the fused kernel.
struct PassedSink {
  static constexpr bool kFold = true;
  static constexpr bool kRecord = true;    // the optional arrays of sart_passed_out_t include pathCB and deviationDet
  const FastTables& T;
  double m2;
  WarpCounters& wc;
  RayResult& out;
  bool& have;
  __device__ __forceinline__ bool defer(uint32_t id) {
    const int r = rq_push(T.rq, id);
    if (r == 2) atomicAdd(&wc.n_unresolved, 1u);
    return r == 1;
  }
  __device__ __forceinline__ void fail(int code) { atomicAdd(&wc.n_exit[code], 1u); }
  __device__ __forceinline__ void hit(const RayResult& h) { out = h; have = true; }
};

template <bool kWolter, bool kPlain>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_mc_passed_f32(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                      const __grid_constant__ FastTables T, double mAxion2, uint64_t first, uint64_t nRays,
                      const __grid_constant__ PhiloxKeys K, const __grid_constant__ sart_passed_out_t o,
                      unsigned int* __restrict__ count, unsigned int cap, uint32_t idBase,
                      sart_counters_t* __restrict__ counters) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill32(P, T, S);
  for (int i = threadIdx.x; i < kWarps32 * int(sizeof(WarpCounters) / 4); i += kBlock32) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  __syncthreads();
  constexpr unsigned kFull = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint64_t stride = uint64_t(gridDim.x) * kBlock32;
  for (uint64_t base = uint64_t(blockIdx.x) * kBlock32 + (threadIdx.x & ~31); base < nRays; base += stride) {   // warp-uniform
    const uint64_t i = base + lane;
    RayResult r;
    bool have = false;
    double wd = 0.0;
    bool passed = false;
    if (i < nRays) {
      ++nIter;
      PassedSink sink{T, mAxion2, wc[warp], r, have};
      Head32 hd;
      stage_a32_head<kPlain>(P, T, S, K, first + i, hd);
      Rec32 rec;
      rec.id = uint32_t(i);
      const int c0 = stage_a32<kWolter, false, kPlain>(P, G, T, S, hd, rec);
      finish32<kWolter, kPlain>(P, G, T, S, c0, rec, sink);
      if (have) {   // reached the weight stage: the tail of traceAxion (rt:2135-2221)
        const int code = finish_ray<true>(P, r, mAxion2, wd);
        if (code & SART_FLAG_PASSED_TILL_WINDOW) ++nTill;
        if (r.clamped) atomicAdd(&wc[warp].n_clamped, 1u);
        const int ec = code & SART_CODE_MASK;
        passed = ec == SART_EXIT_PASSED;
        if (passed) { ++nPassed; sumW += wd; sumW2 += wd * wd; sumX += r.x; sumY += r.y; sumR += r.r; }
        else atomicAdd(&wc[warp].n_exit[ec], 1u);
      }
    }
    const unsigned m = __ballot_sync(kFull, passed);
    if (m) {
      unsigned int slot0 = 0;
      if (lane == 0) slot0 = atomicAdd(count, unsigned(__popc(m)));
      slot0 = __shfl_sync(kFull, slot0, 0);
      const unsigned int slot = slot0 + __popc(m & ((1u << lane) - 1u));
      if (passed && slot < cap) {
        if (o.ray) o.ray[slot] = idBase + uint32_t(i);
        if (o.x) o.x[slot] = float(r.x);
        if (o.y) o.y[slot] = float(r.y);
        if (o.w) o.w[slot] = float(wd);
        if (o.shell) o.shell[slot] = uint8_t(r.shell);
        if (o.energy) o.energy[slot] = (kPlain || !P.testXray) ? float(fmax(__ldg(T.energies + r.eIdx), 0.03)) : P.srcEnergy;
        if (o.r) o.r[slot] = float(r.r);
        if (o.reflect) o.reflect[slot] = float(r.refl);
        if (o.transMagnet)
          o.transMagnet[slot] = float(double(r.pre) * conv_factor(P, r.convVac, r.gasGamma, r.gasE1, r.gasE2, r.gasInv2E, r.gasL, mAxion2));
        if (o.yaw) o.yaw[slot] = r.yaw;
        if (o.alpha1) o.alpha1[slot] = r.a1;
        if (o.alpha2) o.alpha2[slot] = r.a2;
        if (o.pathCB) o.pathCB[slot] = r.path;
        if (o.deviationDet) o.deviationDet[slot] = r.devDet;
        if (o.transProbArgon) o.transProbArgon[slot] = r.agas;
      }
    }
  }
  for (int ofs = 16; ofs > 0; ofs >>= 1) {
    nPassed += __shfl_down_sync(kFull, nPassed, ofs);
    nTill += __shfl_down_sync(kFull, nTill, ofs);
    nIter += __shfl_down_sync(kFull, nIter, ofs);
    sumW += __shfl_down_sync(kFull, sumW, ofs);
    sumW2 += __shfl_down_sync(kFull, sumW2, ofs);
    sumX += __shfl_down_sync(kFull, sumX, ofs);
    sumY += __shfl_down_sync(kFull, sumY, ofs);
    sumR += __shfl_down_sync(kFull, sumR, ofs);
  }
  __syncwarp();
  if (lane == 0) flush_counters(counters, wc[warp], nIter, nPassed, nTill, sumW, sumW2, sumX, sumY, sumR);
}

// ---- tier (a): pre-sampled rays, structure of arrays in HBM -> per-ray records in HBM -------------------------------
// 48 B in (origin x, y, z; exit-disc x, y; energy — f64, coalesced) and 32 B out (x, y, w f64; code, shell i32) per ray,
// plus whatever optional record arrays the caller asks for.
// The slopes are formed in FP64 from the caller's points (the origin is 1.5e14 mm away), everything after that is the
// FP32 pipeline. The energy is mapped to its index in the tabulated energies (the reference only ever traces tabulated
// energies, rt:470); an energy that is not a table value is traced at the nearest one and flagged INTERP_CLAMPED.
// kOptional: the caller wants optional record arrays (else only x, y, w, code, shell are formed and stored).
template <bool kWolter, bool kPlain, bool kMargins, bool kOptional>
__global__ void __launch_bounds__(kBlock32, SART_F32_MINBLOCKS)
k_trace_presampled_f32(const __grid_constant__ FastParams P, const __grid_constant__ Geo32 G,
                       const __grid_constant__ FastTables T, double mAxion2, size_t n, const double* __restrict__ origin,
                       const double* __restrict__ exitxy, const double* __restrict__ energy,
                       const __grid_constant__ sart_ray_out_t o) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem32 S;
  unsigned char* tail;
  smem_layout32(P, smem, S, tail);
  smem_fill32(P, T, S);
  __syncthreads();
  const size_t stride = size_t(gridDim.x) * kBlock32;
  for (size_t i = size_t(blockIdx.x) * kBlock32 + threadIdx.x; i < n; i += stride) {
    const double Ox = origin[i], Oy = origin[n + i], Oz = origin[2 * n + i];
    const double ex = exitxy[i], ey = exitxy[n + i], E = energy[i];
    Head32 hd;
    const double invD = rcp_nr(P.lengthB - Oz);
    hd.ex = float(ex); hd.ey = float(ey);
    hd.sx = float((ex - Ox) * invD); hd.sy = float((ey - Oy) * invD);
    // rounding noise of the reference's line O + lambda (E - O) (rt:481-492, 529-534) at pointExitCB: one ulp of the
    // origin's x / y, plus one ulp of its z seen through the slope
    hd.epsO = 4.4408921e-16f * (fabsf(float(Ox)) + fabsf(float(Oy)) + (fabsf(hd.sx) + fabsf(hd.sy)) * fabsf(float(Oz)));
    // energy -> index of the tabulated energy: uniform-grid guess, then the table decides
    const double Ec = fmax(E, 0.03);
    int k = int(rint((E - P.enE0) * P.enInvStep));
    k = k < 0 ? 0 : (k > P.nEnergies - 1 ? P.nEnergies - 1 : k);
    if (fmax(__ldg(T.energies + k), 0.03) != Ec) {
      k = lower_bound_window(T.energies, 0, P.nEnergies, Ec);   // first tabulated energy >= Ec
      if (k > P.nEnergies - 1) k = P.nEnergies - 1;
      if (k > 0 && fmax(__ldg(T.energies + k), 0.03) != Ec) {
        const double below = fmax(__ldg(T.energies + k - 1), 0.03);   // entries under 0.03 keV are traced at 0.03 (rt:471)
        if (below == Ec || fabs(below - Ec) < fabs(__ldg(T.energies + k) - Ec)) --k;
      }
    }
    hd.eIdx = k;
    hd.offGrid = fmax(__ldg(T.energies + k), 0.03) != Ec;
    RayResult r;
    RecordSink<true, kOptional> sink{r, mAxion2, T.rq, false};
    Rec32 rec;
    rec.id = uint32_t(i);
    const int c0 = stage_a32<kWolter, true, kPlain, false, false, kMargins>(P, G, T, S, hd, rec);
    finish32<kWolter, kPlain, true, kMargins>(P, G, T, S, c0, rec, sink);
    store_record<kOptional>(P, o, i, r, mAxion2, Ec);
  }
}

}  // namespace fast

cudaError_t launch_presampled_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                  size_t n, const double* origin, const double* exitxy, const double* energy,
                                  const sart_ray_out_t& o, int smCount, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const LaunchVariant v = launch_variant(P, T);   // pre-sampled rays have no source: the sampler plays no part
  const size_t smem = fast::smem_bytes32(P);
  using Kern = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, double, size_t, const double*, const double*, const double*,
                        sart_ray_out_t);
#define SART_ROW(W, PL) {{fast::k_trace_presampled_f32<W, PL, false, false>, fast::k_trace_presampled_f32<W, PL, false, true>}, \
                         {fast::k_trace_presampled_f32<W, PL, true, false>, fast::k_trace_presampled_f32<W, PL, true, true>}}
  static const Kern table[2][2][2][2] = {   // [wolter][plain][margins][optional arrays wanted]
      {SART_ROW(false, false), SART_ROW(false, true)}, {SART_ROW(true, false), SART_ROW(true, true)}};
#undef SART_ROW
  const bool optional = o.energy || o.reflect || o.transMagnet || o.yaw || o.alpha1 || o.alpha2 || o.pathCB || o.r ||
                        o.deviationDet || o.transProbArgon;
  const Kern kern = table[v.wolter ? 1 : 0][v.plain ? 1 : 0][v.margins ? 1 : 0][optional ? 1 : 0];
  cudaError_t e = fast::set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  unsigned grid = 0;
  if ((e = grid_size(kern, fast::kBlock32, smem, n, smCount, 0, &grid)) != cudaSuccess) return e;
  kern<<<grid, fast::kBlock32, smem, s>>>(P, G, T, mAxion * mAxion, n, origin, exitxy, energy, o);
  return cudaGetLastError();
}

cudaError_t launch_mc_passed_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                                 uint64_t first, uint64_t nRays, uint64_t seed, const sart_passed_out_t& o, unsigned int* count,
                                 unsigned int cap, uint32_t idBase, sart_counters_t* counters, int smCount, cudaStream_t s) {
  if (nRays == 0) return cudaSuccess;
  const LaunchVariant v = launch_variant(P, T);
  const size_t smem = fast::smem_bytes32(P);
  auto kern = v.wolter ? (v.plain ? fast::k_trace_mc_passed_f32<true, true> : fast::k_trace_mc_passed_f32<true, false>)
                       : (v.plain ? fast::k_trace_mc_passed_f32<false, true> : fast::k_trace_mc_passed_f32<false, false>);
  cudaError_t e = fast::set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  unsigned grid = 0;
  if ((e = grid_size(kern, fast::kBlock32, smem, nRays, smCount, 1, &grid)) != cudaSuccess) return e;
  kern<<<grid, fast::kBlock32, smem, s>>>(P, G, T, mAxion * mAxion, first, nRays, philox_round_keys(seed), o, count, cap, idBase, counters);
  return cudaGetLastError();
}

cudaError_t launch_mc_rays_f32(const fast::FastParams& P, const fast::Geo32& G, const fast::FastTables& T, double mAxion,
                               uint64_t first, uint64_t nRays, uint64_t seed, const sart_ray_out_t& o, int smCount,
                               cudaStream_t s, const uint32_t* words, bool lateEnergy, int32_t* emit) {
  if (nRays == 0) return cudaSuccess;
  const LaunchVariant v = launch_variant(P, T);
  const size_t smem = fast::smem_bytes32(P, fast::kWarps32, v.alias);
  using Kern = void (*)(fast::FastParams, fast::Geo32, fast::FastTables, double, uint64_t, uint64_t, PhiloxKeys, const uint32_t*,
                        int32_t*, sart_ray_out_t);
  static const Kern table[2][2][2] = {   // [wolter][plain][alias]
      {{fast::k_trace_mc_rays_f32<false, false, false>, fast::k_trace_mc_rays_f32<false, false, true>},
       {fast::k_trace_mc_rays_f32<false, true, false>, fast::k_trace_mc_rays_f32<false, true, true>}},
      {{fast::k_trace_mc_rays_f32<true, false, false>, fast::k_trace_mc_rays_f32<true, false, true>},
       {fast::k_trace_mc_rays_f32<true, true, false>, fast::k_trace_mc_rays_f32<true, true, true>}}};
  static const Kern late[2][2] = {   // [wolter][alias], generic (non-plain) variant: the hook of sart_trace_words
      {fast::k_trace_mc_rays_f32<false, false, false, true>, fast::k_trace_mc_rays_f32<false, false, true, true>},
      {fast::k_trace_mc_rays_f32<true, false, false, true>, fast::k_trace_mc_rays_f32<true, false, true, true>}};
  const Kern kern = lateEnergy ? late[v.wolter ? 1 : 0][v.alias ? 1 : 0] : table[v.wolter ? 1 : 0][v.plain ? 1 : 0][v.alias ? 1 : 0];
  cudaError_t e = fast::set_smem(kern, smem);
  if (e != cudaSuccess) return e;
  unsigned grid = 0;
  if ((e = grid_size(kern, fast::kBlock32, smem, nRays, smCount, 2, &grid)) != cudaSuccess) return e;
  kern<<<grid, fast::kBlock32, smem, s>>>(P, G, T, mAxion * mAxion, first, nRays, philox_round_keys(seed), words, emit, o);
  return cudaGetLastError();
}

}  // namespace sart
