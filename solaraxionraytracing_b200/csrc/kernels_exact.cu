// kernels_exact.cu — sm_100a kernels of the FP64 ("exact") pipeline and the CDF build.
// Compiled with -fmad=false: see trace_exact.cuh for why.
//
//   k_trace_presampled  tier-(a) kernel: SoA rays in (origin xyz, exit-disc xy, energy: 6 f64 = 48 B... see
//                       DESIGN.md for the byte count) -> SoA per-ray record out. One thread per ray.
//   k_trace_mc_rays     traceAxionWrapper drop-in (rt:2223-2244): Philox sampling + trace, per-ray records out.
//   k_trace_mc_image    fused run: Philox sampling + trace + prepareHeatmap (rt:818-842) + the counters of
//                       generateResultPlots (rt:2252-2257). Grid-stride over global ray indices.
//   k_build_cdf_rows / k_build_cdf_radius   initFullSetup's CDF build (rt:2679-2705).
#include <cuda_runtime.h>

#include "kernels.h"
#include "trace_exact.cuh"

namespace sart {

struct RayOutDev {  // sart_ray_out_t with device pointers
  double *x, *y, *w;
  int32_t *code, *shell;
  double *energy, *reflect, *transMagnet, *yaw, *alpha1, *alpha2, *pathCB, *r, *deviationDet, *transProbArgon;
};

__device__ __forceinline__ void store_ray(const RayOutDev& o, size_t i, const Geo& g, const Weights& w, const Final& f,
                                          bool weighted) {
  o.x[i] = f.x; o.y[i] = f.y; o.w[i] = f.w;
  o.code[i] = f.code;
  // shellNumber is assigned only at rt:2198, i.e. for rays that get past the window aperture
  const bool tail = weighted && !g.windowMiss;
  o.shell[i] = tail ? g.shell : -1;
  if (o.energy) o.energy[i] = g.energy;
  if (o.reflect) o.reflect[i] = weighted ? w.reflect : 0.0;
  if (o.transMagnet) o.transMagnet[i] = weighted ? f.transMagnet : 0.0;
  if (o.yaw) o.yaw[i] = g.ya;
  if (o.alpha1) o.alpha1[i] = g.alpha1;
  if (o.alpha2) o.alpha2[i] = g.alpha2;
  if (o.pathCB) o.pathCB[i] = g.pathCB;
  if (o.r) o.r[i] = f.r;
  if (o.deviationDet) o.deviationDet[i] = g.deviationDet;
  if (o.transProbArgon) o.transProbArgon[i] = tail ? w.absGas : 0.0;
}

__device__ __forceinline__ void trace_and_store(const Params& P, const Tables& T, double mAxion, V3 O, V3 E,
                                                double energy, int preClamped, const RayOutDev& out, size_t i, int eIdx = -1) {
  Geo g;
  trace_geometry<true>(P, T, O, E, energy, g);
  g.clamped |= preClamped;
  g.eIdx = eIdx;
  Weights w = {};
  Final f = {};
  if (g.code < 0) {
    ray_weights(P, T, g, w);
    ray_finish(P, g, w, mAxion, f);
    store_ray(out, i, g, w, f, true);
  } else {
    f.code = g.code | (g.clamped ? SART_FLAG_INTERP_CLAMPED : 0);
    store_ray(out, i, g, w, f, false);
  }
}

__global__ void __launch_bounds__(128)
k_trace_presampled(const __grid_constant__ Params P, const __grid_constant__ Tables T, double mAxion, size_t n,
                   const double* __restrict__ origin, const double* __restrict__ exitxy,
                   const double* __restrict__ energy, const __grid_constant__ RayOutDev out) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const V3 O = {origin[i], origin[n + i], origin[2 * n + i]};
  const V3 E = {exitxy[i], exitxy[n + i], P.lengthB};
  trace_and_store(P, T, mAxion, O, E, energy[i], 0, out, i);
}

// ---- re-trace kernels: the rays of a launch of the FP32 pipeline (kernels_f32.cu) whose decision margins were inside
// their error budgets, listed as offsets into the launch. Grid-stride over min(*count, cap) entries: the count is read on
// the device, so the host queues these launches without a synchronisation.
__global__ void __launch_bounds__(128)
k_retrace_presampled(const __grid_constant__ Params P, const __grid_constant__ Tables T, double mAxion, size_t n,
                     const double* __restrict__ origin, const double* __restrict__ exitxy,
                     const double* __restrict__ energy, const uint32_t* __restrict__ list,
                     const uint32_t* __restrict__ count, uint32_t cap, const __grid_constant__ RayOutDev out) {
  const uint32_t m = min(*count, cap);
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
    const size_t i = list[j];
    if (i >= n) continue;
    const V3 O = {origin[i], origin[n + i], origin[2 * n + i]};
    const V3 E = {exitxy[i], exitxy[n + i], P.lengthB};
    trace_and_store(P, T, mAxion, O, E, energy[i], 0, out, i);
  }
}

__device__ __forceinline__ void mc_ray_record(const Params& P, const Tables& T, double mAxion, uint64_t first, size_t n,
                                              uint64_t seed, const uint32_t* __restrict__ words, int32_t* __restrict__ emit,
                                              const RayOutDev& out, size_t i) {
  V3 O, E;
  double energy;
  int clamped = 0;
  uint32_t w[6];
  if (words) {   // sart_trace_words: caller-supplied random words, SoA [6][n]
    for (int k = 0; k < 6; ++k) w[k] = words[size_t(k) * n + i];
  } else {
    ray_words(seed, first + i, w);
  }
  if (emit) emit[i] = P.testXray ? 0 : min(lower_bound(T.fluxRadiusCDF, 0, P.nRadii, u01(w[2])), P.nRadii - 1);   // rIdx rt:437
  int eIdx = -1;
  if (!sample_ray_words(P, T, w, O, E, energy, clamped, &eIdx)) {
    out.x[i] = 0.0; out.y[i] = 0.0; out.w[i] = 0.0; out.code[i] = SART_EXIT_COLLIMATOR; out.shell[i] = -1;
    if (out.energy) out.energy[i] = energy;
    if (out.reflect) out.reflect[i] = 0.0;
    if (out.transMagnet) out.transMagnet[i] = 0.0;
    if (out.yaw) out.yaw[i] = 0.0;
    if (out.alpha1) out.alpha1[i] = 0.0;
    if (out.alpha2) out.alpha2[i] = 0.0;
    if (out.pathCB) out.pathCB[i] = 0.0;
    if (out.r) out.r[i] = 0.0;
    if (out.deviationDet) out.deviationDet[i] = 0.0;
    if (out.transProbArgon) out.transProbArgon[i] = 0.0;
    return;
  }
  trace_and_store(P, T, mAxion, O, E, energy, clamped, out, i, eIdx);
}

__global__ void __launch_bounds__(128)
k_trace_mc_rays(const __grid_constant__ Params P, const __grid_constant__ Tables T, double mAxion, uint64_t first,
                size_t n, uint64_t seed, const uint32_t* __restrict__ words, int32_t* __restrict__ emit,
                const __grid_constant__ RayOutDev out) {
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  mc_ray_record(P, T, mAxion, first, n, seed, words, emit, out, i);
}

__global__ void __launch_bounds__(128)
k_retrace_mc_rays(const __grid_constant__ Params P, const __grid_constant__ Tables T, double mAxion, uint64_t first,
                  size_t n, uint64_t seed, const uint32_t* __restrict__ words, const uint32_t* __restrict__ list,
                  const uint32_t* __restrict__ count, uint32_t cap, const __grid_constant__ RayOutDev out) {
  const uint32_t m = min(*count, cap);
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
    const size_t i = list[j];
    if (i < n) mc_ray_record(P, T, mAxion, first, n, seed, words, nullptr, out, i);
  }
}

// Re-trace pass of sart_trace_mc_passed: the queued rays traced exactly; those that pass are appended to the compacted
// records (single precision, like the FP32 kernel writes them), all of them are counted.
__global__ void __launch_bounds__(128)
k_retrace_mc_passed(const __grid_constant__ Params P, const __grid_constant__ Tables T, double mAxion, uint64_t first,
                    uint64_t seed, const uint32_t* __restrict__ list, const uint32_t* __restrict__ listCount, uint32_t listCap,
                    const __grid_constant__ sart_passed_out_t o, unsigned int* __restrict__ count, unsigned int cap,
                    uint32_t idBase, sart_counters_t* __restrict__ c) {
  auto addu = [](uint64_t* p, unsigned long long v) { atomicAdd(reinterpret_cast<unsigned long long*>(p), v); };
  const uint32_t m = min(*listCount, listCap);
  if (blockIdx.x == 0 && threadIdx.x == 0) addu(&c->n_retraced, m);
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
    const uint32_t i = list[j];
    V3 O, E;
    double energy;
    int clamped = 0;
    int eIdx = -1;
    if (!sample_ray(P, T, seed, first + i, O, E, energy, clamped, &eIdx)) { addu(&c->n_exit[SART_EXIT_COLLIMATOR], 1); continue; }
    Geo g;
    trace_geometry<true>(P, T, O, E, energy, g);
    g.clamped |= clamped;
    g.eIdx = eIdx;
    if (g.clamped) addu(&c->n_interp_clamped, 1);
    if (g.code >= 0) {
      addu(&c->n_exit[g.code], 1);
      if (g.code == SART_EXIT_NICKEL) addu(&c->n_hit_nickel, 1);
      continue;
    }
    Weights w;
    ray_weights(P, T, g, w);
    Final f;
    ray_finish(P, g, w, mAxion, f);
    if (f.code & SART_FLAG_PASSED_TILL_WINDOW) addu(&c->n_passed_till_window, 1);
    const int ec = f.code & SART_CODE_MASK;
    addu(&c->n_exit[ec], 1);
    if (ec != SART_EXIT_PASSED) continue;
    addu(&c->n_passed, 1);
    atomicAdd(&c->sum_w, f.w); atomicAdd(&c->sum_w2, f.w * f.w);
    atomicAdd(&c->sum_x, f.x); atomicAdd(&c->sum_y, f.y); atomicAdd(&c->sum_r, f.r);
    const unsigned int slot = atomicAdd(count, 1u);
    if (slot >= cap) continue;
    if (o.ray) o.ray[slot] = idBase + i;
    if (o.x) o.x[slot] = float(f.x);
    if (o.y) o.y[slot] = float(f.y);
    if (o.w) o.w[slot] = float(f.w);
    if (o.shell) o.shell[slot] = uint8_t(g.shell);
    if (o.energy) o.energy[slot] = float(g.energy);
    if (o.r) o.r[slot] = float(f.r);
    if (o.reflect) o.reflect[slot] = float(w.reflect);
    if (o.transMagnet) o.transMagnet[slot] = float(f.transMagnet);
    if (o.yaw) o.yaw[slot] = float(g.ya);
    if (o.alpha1) o.alpha1[slot] = float(g.alpha1);
    if (o.alpha2) o.alpha2[slot] = float(g.alpha2);
    if (o.pathCB) o.pathCB[slot] = float(g.pathCB);
    if (o.deviationDet) o.deviationDet[slot] = float(g.deviationDet);
    if (o.transProbArgon) o.transProbArgon[slot] = float(w.absGas);
  }
}

// ---- fused Monte Carlo run -------------------------------------------------------------------------------
// Block-level counters live in shared memory and are flushed once per block.
// 32-bit shared-memory counters (native ATOMS.ADD; the 64-bit and f64 shared-memory atomics this kernel used before are
// compare-and-swap loops that all 128 threads of a block fought over: a third of its instructions). A block sees fewer
// than 2^32 rays per launch (the launcher cuts a run into launches of at most 2^31 rays).
struct BlockCounters {
  unsigned int n_exit[16];   // geometric exits (mass independent); PASSED / ZERO_WEIGHT are per mass
  unsigned int n_clamped, pad[3];
};
// Sums of the first axion mass live in the registers of each thread and are reduced once at the end of the kernel.
struct ThreadSums {
  unsigned int n_rays = 0, n_passed = 0, n_zero = 0, n_till = 0;
  double sum_w = 0.0, sum_w2 = 0.0, sum_x = 0.0, sum_y = 0.0, sum_r = 0.0;
};
struct MassCounters {
  unsigned long long n_passed, n_zero, n_till_window, pad;
  double sum_w, sum_w2, sum_x, sum_y, sum_r;
};

// One ray of the fused run: sample, trace, weight for every axion mass, histogram (rt:1736-2221 + 818-842).
__device__ __forceinline__ void mc_image_ray(const Params& P, const Tables& T, int nMasses, const double* __restrict__ masses,
                                             uint64_t seed, uint64_t ray, double* __restrict__ image,
                                             double* __restrict__ imageW2, BlockCounters* bc, MassCounters* mc, ThreadSums& ts) {
  const double step = (P.chipCX * 2.0 - 0.0) / double(SART_IMAGE_BINS);  // (stop - start)/rows rt:828-830
  const double stepY = (P.chipCY * 2.0 - 0.0) / double(SART_IMAGE_BINS);
  V3 O, E;
  double energy;
  int clamped = 0;
  int eIdx = -1;
  if (!sample_ray(P, T, seed, ray, O, E, energy, clamped, &eIdx)) {
    atomicAdd(&bc->n_exit[SART_EXIT_COLLIMATOR], 1u);
    return;
  }
  Geo g;
  trace_geometry<false>(P, T, O, E, energy, g);
  g.clamped |= clamped;
  g.eIdx = eIdx;
  if (g.code >= 0) {
    atomicAdd(&bc->n_exit[g.code], 1u);
    if (g.clamped) atomicAdd(&bc->n_clamped, 1u);
    return;
  }
  Weights w;
  ray_weights(P, T, g, w);
  if (g.clamped) atomicAdd(&bc->n_clamped, 1u);
  if (g.windowMiss) atomicAdd(&bc->n_exit[SART_EXIT_WINDOW_APERTURE], 1u);
  for (int m = 0; m < nMasses; ++m) {
    Final f;
    ray_finish(P, g, w, masses[m], f);
    const int code = f.code & SART_CODE_MASK;
    if (m == 0) {   // the first (usually only) mass: per-thread registers
      if (f.code & SART_FLAG_PASSED_TILL_WINDOW) ++ts.n_till;
      if (code == SART_EXIT_ZERO_WEIGHT) ++ts.n_zero;
      if (code != SART_EXIT_PASSED) continue;
      ++ts.n_passed;
      ts.sum_w += f.w; ts.sum_w2 += f.w * f.w; ts.sum_x += f.x; ts.sum_y += f.y; ts.sum_r += f.r;
    } else {
      if (f.code & SART_FLAG_PASSED_TILL_WINDOW) atomicAdd(&mc[m].n_till_window, 1ull);
      if (code == SART_EXIT_ZERO_WEIGHT) atomicAdd(&mc[m].n_zero, 1ull);
      if (code != SART_EXIT_PASSED) continue;
      atomicAdd(&mc[m].n_passed, 1ull);
      atomicAdd(&mc[m].sum_w, f.w);
      atomicAdd(&mc[m].sum_w2, f.w * f.w);
      atomicAdd(&mc[m].sum_x, f.x);
      atomicAdd(&mc[m].sum_y, f.y);
      atomicAdd(&mc[m].sum_r, f.r);
    }
    // prepareHeatmap rt:839-842
    const double cx = floor((f.x - 0.0) / step), cy = floor((f.y - 0.0) / stepY);
    if (cx >= 0.0 && cx < double(SART_IMAGE_BINS) && cy >= 0.0 && cy < double(SART_IMAGE_BINS)) {
      const size_t bin = size_t(m) * SART_IMAGE_BINS * SART_IMAGE_BINS + size_t(int(cy)) * SART_IMAGE_BINS + size_t(int(cx));
      atomicAdd(image + bin, f.w);
      atomicAdd(imageW2 + bin, f.w * f.w);
    }
    if (T.rad.w && m == 0) {
      int b = int(f.r * T.rad.invStep);
      b = b < 0 ? 0 : (b > T.rad.nbins - 1 ? T.rad.nbins - 1 : b);
      atomicAdd(T.rad.w + b, f.w);
      atomicAdd(T.rad.n + b, 1ull);
    }
    // spectra (sart_enable_spectra, single mass): the X-ray source's rays carry no table index and go to bin nEnergies
    if (T.spec.eW && m == 0) spec_add(T.spec, g.eIdx >= 0 ? g.eIdx : P.nEnergies, g.shell, f.w);
  }
}

#ifndef SART_EXACT_MINBLOCKS
#define SART_EXACT_MINBLOCKS 6   // 85 registers instead of 108: 24 instead of 16 warps per SM for this latency-bound kernel (+5 %; 8 is slower)
#endif
// `list` != nullptr: trace the rays first + list[j], j < min(*listCount, listCap), instead of first + [0, nRays).
__global__ void __launch_bounds__(128, SART_EXACT_MINBLOCKS)
k_trace_mc_image(const __grid_constant__ Params P, const __grid_constant__ Tables T, int nMasses,
                 const double* __restrict__ masses, uint64_t first, uint64_t nRays, uint64_t seed,
                 const uint32_t* __restrict__ list, const uint32_t* __restrict__ listCount, uint32_t listCap,
                 double* __restrict__ image, double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  extern __shared__ unsigned char smem_raw[];
  BlockCounters* bc = reinterpret_cast<BlockCounters*>(smem_raw);
  MassCounters* mc = reinterpret_cast<MassCounters*>(smem_raw + sizeof(BlockCounters));
  unsigned long long* nRaysBlock = &mc[0].pad;   // rays of this block (zeroed with the mass counters)
  for (int k = threadIdx.x; k < int(sizeof(BlockCounters) / 4); k += blockDim.x)
    reinterpret_cast<unsigned int*>(bc)[k] = 0u;
  for (int k = threadIdx.x; k < int(nMasses * sizeof(MassCounters) / 8); k += blockDim.x)
    reinterpret_cast<unsigned long long*>(mc)[k] = 0ull;
  __syncthreads();

  const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
  ThreadSums ts;
  // One loop for both modes, so that the per-ray code (8500 SASS instructions, most of them inlined f64 libm) exists once:
  // this kernel waits for instruction fetches more than for anything else (profiles/README.md).
  // List mode: the re-trace of the uncertain rays of an FP32 launch, which has counted them in n_rays already.
  const bool listMode = list != nullptr;
  const uint64_t total = listMode ? uint64_t(min(*listCount, listCap)) : nRays;
  for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
    const uint64_t ray = first + (listMode ? uint64_t(list[i]) : i);
    if (!listMode) ++ts.n_rays;
    mc_image_ray(P, T, nMasses, masses, seed, ray, image, imageW2, bc, mc, ts);
  }
  if (listMode && blockIdx.x == 0 && threadIdx.x == 0)
    for (int m = 0; m < nMasses; ++m) atomicAdd(reinterpret_cast<unsigned long long*>(&counters[m].n_retraced), (unsigned long long)total);
  // the thread sums of the first mass: warp shuffle, then one shared-memory atomic per warp and quantity
  for (int o = 16; o > 0; o >>= 1) {
    ts.n_rays += __shfl_down_sync(0xffffffffu, ts.n_rays, o);
    ts.n_passed += __shfl_down_sync(0xffffffffu, ts.n_passed, o);
    ts.n_zero += __shfl_down_sync(0xffffffffu, ts.n_zero, o);
    ts.n_till += __shfl_down_sync(0xffffffffu, ts.n_till, o);
    ts.sum_w += __shfl_down_sync(0xffffffffu, ts.sum_w, o);
    ts.sum_w2 += __shfl_down_sync(0xffffffffu, ts.sum_w2, o);
    ts.sum_x += __shfl_down_sync(0xffffffffu, ts.sum_x, o);
    ts.sum_y += __shfl_down_sync(0xffffffffu, ts.sum_y, o);
    ts.sum_r += __shfl_down_sync(0xffffffffu, ts.sum_r, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(nRaysBlock, (unsigned long long)ts.n_rays);
    atomicAdd(&mc[0].n_passed, (unsigned long long)ts.n_passed);
    atomicAdd(&mc[0].n_zero, (unsigned long long)ts.n_zero);
    atomicAdd(&mc[0].n_till_window, (unsigned long long)ts.n_till);
    atomicAdd(&mc[0].sum_w, ts.sum_w); atomicAdd(&mc[0].sum_w2, ts.sum_w2);
    atomicAdd(&mc[0].sum_x, ts.sum_x); atomicAdd(&mc[0].sum_y, ts.sum_y); atomicAdd(&mc[0].sum_r, ts.sum_r);
  }
  __syncthreads();
  // flush
  for (int m = threadIdx.x; m < nMasses; m += blockDim.x) {
    sart_counters_t* c = counters + m;
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_rays), *nRaysBlock);
    for (int e = 1; e < SART_N_EXIT_CODES; ++e)
      if (e != SART_EXIT_ZERO_WEIGHT && bc->n_exit[e])
        atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_exit[e]), (unsigned long long)bc->n_exit[e]);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_exit[SART_EXIT_PASSED]), mc[m].n_passed);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_exit[SART_EXIT_ZERO_WEIGHT]), mc[m].n_zero);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_passed), mc[m].n_passed);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_passed_till_window), mc[m].n_till_window);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_hit_nickel), (unsigned long long)bc->n_exit[SART_EXIT_NICKEL]);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_interp_clamped), (unsigned long long)bc->n_clamped);
    atomicAdd(&c->sum_w, mc[m].sum_w);
    atomicAdd(&c->sum_w2, mc[m].sum_w2);
    atomicAdd(&c->sum_x, mc[m].sum_x);
    atomicAdd(&c->sum_y, mc[m].sum_y);
    atomicAdd(&c->sum_r, mc[m].sum_r);
  }
}

// ---- CDF build rt:2679-2705 -------------------------------------------------------------------------------
// One thread walks one radius row sequentially (the reference's summation order => identical bits).
__global__ void k_build_cdf_rows(int nR, int nE, const double* __restrict__ radii, const double* __restrict__ energies,
                                 const double* __restrict__ emRates, double* __restrict__ rowTotals,
                                 double* __restrict__ cdfs) {
  const int iRad = blockIdx.x * blockDim.x + threadIdx.x;
  if (iRad >= nR) return;
  const double radius = radii[iRad];
  const double* em = emRates + size_t(iRad) * nE;
  double* row = cdfs + size_t(iRad) * nE;
  double diffSum = 0.0;
  for (int iE = 0; iE < nE; ++iE) {
    const double e = energies[iE];
    const double diffFlux = em[iE] * (e * e) * radius * radius;
    diffSum += diffFlux;
    row[iE] = diffSum;
  }
  rowTotals[iRad] = diffSum;
  const double integral = row[nE - 1];
  for (int iE = 0; iE < nE; ++iE) row[iE] = row[iE] / integral;
}
__global__ void k_build_cdf_radius(int nR, const double* __restrict__ rowTotals, double* __restrict__ radiusCDF) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  double acc = 0.0;
  for (int i = 0; i < nR; ++i) { acc += rowTotals[i]; radiusCDF[i] = acc; }
  const double integral = radiusCDF[nR - 1];
  for (int i = 0; i < nR; ++i) radiusCDF[i] = radiusCDF[i] / integral;
}

// ---- prepareHeatmap rt:818-842 for host-provided points -------------------------------------------------------
__global__ void k_heatmap(int rows, int cols, double start_x, double step_x, double start_y, double step_y, size_t n,
                          const double* __restrict__ X, const double* __restrict__ Y, const double* __restrict__ W,
                          double norm, double* __restrict__ result, unsigned long long* __restrict__ nBad) {
  const size_t stride = size_t(gridDim.x) * blockDim.x;
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const double cx = floor((X[i] - start_x) / step_x), cy = floor((Y[i] - start_y) / step_y);
    if (cx >= 0.0 && cx < double(cols) && cy >= 0.0 && cy < double(rows))
      atomicAdd(result + size_t(cy) * cols + size_t(cx), 1 * W[i] / norm);
    else
      atomicAdd(nBad, 1ull);
  }
}

cudaError_t launch_heatmap(int rows, int cols, double start_x, double step_x, double start_y, double step_y, size_t n,
                           const double* X, const double* Y, const double* W, double norm, double* result,
                           unsigned long long* nBad, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const int block = 256;
  size_t want = (n + block - 1) / block;
  const unsigned grid = unsigned(want < 148 * 8 ? want : 148 * 8);
  k_heatmap<<<grid, block, 0, s>>>(rows, cols, start_x, step_x, start_y, step_y, n, X, Y, W, norm, result, nBad);
  return cudaGetLastError();
}

// ---- launchers --------------------------------------------------------------------------------------------
static RayOutDev to_dev(const sart_ray_out_t& o) {
  return RayOutDev{o.x, o.y, o.w, o.code, o.shell, o.energy, o.reflect, o.transMagnet, o.yaw,
                   o.alpha1, o.alpha2, o.pathCB, o.r, o.deviationDet, o.transProbArgon};
}

cudaError_t launch_presampled_exact(const Params& P, const Tables& T, double mAxion, size_t n, const double* origin,
                                    const double* exitxy, const double* energy, const sart_ray_out_t& out,
                                    cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const int block = 128;
  const unsigned grid = unsigned((n + block - 1) / block);
  k_trace_presampled<<<grid, block, 0, s>>>(P, T, mAxion, n, origin, exitxy, energy, to_dev(out));
  return cudaGetLastError();
}

cudaError_t launch_mc_rays_exact(const Params& P, const Tables& T, double mAxion, uint64_t first, size_t n,
                                 uint64_t seed, const sart_ray_out_t& out, cudaStream_t s, const uint32_t* words, int32_t* emit) {
  if (n == 0) return cudaSuccess;
  const int block = 128;
  const unsigned grid = unsigned((n + block - 1) / block);
  k_trace_mc_rays<<<grid, block, 0, s>>>(P, T, mAxion, first, n, seed, words, emit, to_dev(out));
  return cudaGetLastError();
}

cudaError_t launch_mc_image_exact(const Params& P, const Tables& T, int nMasses, const double* masses, uint64_t first,
                                  uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                  sart_counters_t* counters, int smCount, cudaStream_t s) {
  if (nRays == 0) return cudaSuccess;
  const int block = 128;
  const size_t smem = sizeof(BlockCounters) + size_t(nMasses) * sizeof(MassCounters);
  int perSM = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_trace_mc_image, block, smem);
  if (e != cudaSuccess) return e;
  if (perSM < 1) perSM = 1;
  uint64_t want = (nRays + block - 1) / block;
  uint64_t cap = uint64_t(smCount) * perSM;  // one resident wave; the grid-stride loop covers the rest
  const unsigned grid = unsigned(want < cap ? want : cap);
  k_trace_mc_image<<<grid, block, smem, s>>>(P, T, nMasses, masses, first, nRays, seed, nullptr, nullptr, 0u, image, imageW2,
                                             counters);
  return cudaGetLastError();
}

// ---- re-trace launchers (fixed grids: the list length lives on the device) -------------------------------------
cudaError_t launch_retrace_mc_image(const Params& P, const Tables& T, int nMasses, const double* masses, uint64_t first,
                                    uint64_t seed, const fast::RetraceQueue& q, double* image, double* imageW2,
                                    sart_counters_t* counters, int smCount, cudaStream_t s) {
  const int block = 128;
  const size_t smem = sizeof(BlockCounters) + size_t(nMasses) * sizeof(MassCounters);
  int perSM = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_trace_mc_image, block, smem);
  if (e != cudaSuccess) return e;
  if (perSM < 1) perSM = 1;
  // one resident wave (the list length lives on the device): latency-bound FP64 code wants every warp slot it can get
  k_trace_mc_image<<<unsigned(smCount * perSM), block, smem, s>>>(P, T, nMasses, masses, first, 0, seed, q.list, q.count, q.cap, image,
                                                                 imageW2, counters);
  return cudaGetLastError();
}
cudaError_t launch_retrace_mc_rays(const Params& P, const Tables& T, double mAxion, uint64_t first, size_t n, uint64_t seed,
                                   const uint32_t* words, const fast::RetraceQueue& q, const sart_ray_out_t& out, int smCount,
                                   cudaStream_t s) {
  k_retrace_mc_rays<<<unsigned(smCount) * 4u, 128, 0, s>>>(P, T, mAxion, first, n, seed, words, q.list, q.count, q.cap, to_dev(out));
  return cudaGetLastError();
}
cudaError_t launch_retrace_mc_passed(const Params& P, const Tables& T, double mAxion, uint64_t first, uint64_t seed,
                                     const fast::RetraceQueue& q, const sart_passed_out_t& o, unsigned int* count, unsigned int cap,
                                     uint32_t idBase, sart_counters_t* counters, int smCount, cudaStream_t s) {
  k_retrace_mc_passed<<<unsigned(smCount) * 4u, 128, 0, s>>>(P, T, mAxion, first, seed, q.list, q.count, q.cap, o, count, cap, idBase,
                                                           counters);
  return cudaGetLastError();
}
cudaError_t launch_retrace_presampled(const Params& P, const Tables& T, double mAxion, size_t n, const double* origin,
                                      const double* exitxy, const double* energy, const fast::RetraceQueue& q,
                                      const sart_ray_out_t& out, int smCount, cudaStream_t s) {
  k_retrace_presampled<<<unsigned(smCount) * 4u, 128, 0, s>>>(P, T, mAxion, n, origin, exitxy, energy, q.list, q.count, q.cap,
                                                            to_dev(out));
  return cudaGetLastError();
}

cudaError_t launch_build_cdfs(int nR, int nE, const double* radii, const double* energies, const double* emRates,
                              double* rowTotals, double* cdfs, double* radiusCDF, cudaStream_t s) {
  k_build_cdf_rows<<<(nR + 63) / 64, 64, 0, s>>>(nR, nE, radii, energies, emRates, rowTotals, cdfs);
  k_build_cdf_radius<<<1, 32, 0, s>>>(nR, rowTotals, radiusCDF);
  return cudaGetLastError();
}

}  // namespace sart
