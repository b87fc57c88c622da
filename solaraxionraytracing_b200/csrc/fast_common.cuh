// fast_common.cuh — pieces shared by the throughput pipelines (kernels_fast.cu: FP64 algebra, kernels_f32.cu: FP32
// geometry): MUFU-seeded arithmetic, the integer inverse-CDF search, the reflectivity lookup, the conversion probability,
// the per-ray outcome record and the sinks that turn an outcome into counters / image contributions.
#pragma once
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdlib>

#include "fast_params.h"
#include "kernels.h"
#include "philox.cuh"

namespace sart {
namespace fast {

#ifndef SART_FAST_BLOCK
#define SART_FAST_BLOCK 256
#endif
#ifndef SART_FAST_MINBLOCKS
#define SART_FAST_MINBLOCKS 3
#endif
constexpr int kBlock = SART_FAST_BLOCK;
constexpr int kWarps = kBlock / 32;

// ---- FP64 divide / sqrt from FP32 seeds ---------------------------------------------------------------------
// MUFU.RCP / MUFU.RSQ seeds (2^-23 relative); the *_rn intrinsics and rsqrtf() expand to range checks + slow paths.
__device__ __forceinline__ float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rsqrt_approx(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ double rcp_nr(double x) {
  double r = double(rcp_approx(float(x)));
  const double e = fma(-x, r, 1.0);
  return fma(r, e, r);
}
__device__ __forceinline__ double rsqrt_nr(double x) {
  double y = double(rsqrt_approx(float(x)));
  const double h = 0.5 * x * y;
  return fma(y, fma(-h, y, 0.5), y);  // y * (1.5 - 0.5 x y^2)
}

// sin/cos(2 pi u), u in [0, 1): MUFU.SIN/COS on the argument shifted into [-pi, pi) where their absolute error is
// 2^-21.4; these only set the sampled emission direction / exit-disc point (a 5e-7 relative shift of a random point).
__device__ __forceinline__ void sincos_2pi(float u, float& s, float& c) {
  const float t = 6.283185307179586f * (u - 0.5f);
  s = -__sinf(t);
  c = -__cosf(t);
}
// asin / atan for small arguments (grazing angles <= 0.1 rad, slopes <= 0.1): odd series, relative error < 1e-7.
__device__ __forceinline__ float asin_small(float x) {
  // series of asin, relative error < 1e-7 for |x| <= 0.1 (grazing angles <= 5.7 deg); beyond that it is still monotone
  // and the reflectivity lookup clamps at angleMax (1.5 deg), so the exact value does not matter
  const float x2 = x * x;
  return x * fmaf(x2, fmaf(x2, 0.075f, 0.16666667f), 1.0f);
}
__device__ __forceinline__ float atan_small(float x) {
  if (fabsf(x) > 0.1f) return atanf(x);
  const float x2 = x * x;
  return x * fmaf(x2, fmaf(x2, 0.2f, -0.33333334f), 1.0f);
}

struct D3 { double x, y, z; };

// rkEffectiveArea (rt:1553-1562): the two angle polynomials of the LLNL effective-area parametrisation, pitch and yaw in
// degrees; the ray's "reflectivity" is their product times the telescope transmission at its energy (FastTables::telTrans).
__device__ __forceinline__ float eff_area_angles(float p, float y) {
  const float tp = fmaf(p, fmaf(p, fmaf(p, fmaf(p, 0.0008f, 1e-04f), -0.4489f), -0.3116f), 96.787f) * 0.01f;
  const float ty = fmaf(y, fmaf(y, fmaf(y, fmaf(y, fmaf(y, fmaf(y, 6.0e-7f, -1.0e-5f), -0.0001f), 0.0034f), -0.0292f), -0.1534f), 99.959f) * 0.01f;
  return tp * ty;
}

// XMM's central blocker with a hole pattern (rt:1674-1688; lineIntersectsObject rt:494-527): does the point (x, y) of the
// telescope entrance plane lie inside one of the nHoles holes of half size R? Hole l = -half .. half sits at
// (2 (l + sign l) R, 0) for odd l and at (0, 2 l R) for even l. `edge` returns the distance [mm] of the point to the
// nearest edge line (or circle) of any hole — conservative for the margin test: also edges that do not bound the shape
// there count. Distances along the diagonal axes of the star / diamond are scaled by 1 / sqrt 2, the factor by which a
// displacement of the point can grow in those coordinates.
template <class F>
__device__ __forceinline__ bool in_hole(int holeType, int nHoles, F R, F x, F y, F& edge) {
  const int half = nHoles / 2;   // nHoles - ceil(nHoles / 2)
  const F k = F(0.7071067811865476);
  bool any = false;
  edge = F(1e30);
  auto near = [&](F a, F bound, F scale) { const F d = fabs(fabs(a) - bound) * scale; edge = d < edge ? d : edge; };
  for (int l = -half; l <= half; ++l) {
    F cx = F(0), cy = F(0);
    if (l != 0) {
      if ((abs(l) & 1) == 0) cy = F(2 * l) * R;
      else cx = F(2 * (l + (l > 0 ? 1 : -1))) * R;
    }
    const F ix = x - cx, iy = y - cy;
    const F tx = (ix - iy) * k, ty = (ix + iy) * k;
    const F ax = fabs(ix), ay = fabs(iy), atx = fabs(tx), aty = fabs(ty);
    const F R16 = R * F(16);
    bool in = false;
    switch (holeType) {
      case SART_HT_CIRCLE: {
        const F r = sqrt(ix * ix + iy * iy);
        in = r < R;
        near(r, R, F(1));
        break;
      }
      case SART_HT_STAR:
        in = (atx < R && aty < R16) || (aty < R && atx < R16);
        near(tx, R, k); near(ty, R, k); near(tx, R16, k); near(ty, R16, k);
        // fall through: the star is the cross plus the same cross turned by 45 degrees
      case SART_HT_CROSS:
        in = in || (ax < R && ay < R16) || (ay < R && ax < R16);
        near(ix, R, F(1)); near(iy, R, F(1)); near(ix, R16, F(1)); near(iy, R16, F(1));
        break;
      case SART_HT_SQUARE:
        in = ax < R && ay < R;
        near(ix, R, F(1)); near(iy, R, F(1));
        break;
      case SART_HT_DIAMOND:
        in = atx < R && aty < R;
        near(tx, R, k); near(ty, R, k);
        break;
      default: break;
    }
    any = any || in;
  }
  return any;
}

__device__ __forceinline__ void rad_add(const RadialHist& h, double r, double w) {
  int b = int(r * h.invStep);
  b = b < 0 ? 0 : (b > h.nbins - 1 ? h.nbins - 1 : b);
  atomicAdd(h.w + b, w);
  atomicAdd(h.n + b, 1ull);
}

// Spectra of the throughput kernels (device_params.h: Spectra, spec_add). The energy bins spread the lanes of a warp over
// hundreds of addresses; the shell bins are a handful (4 for LLNL), so the lanes of a warp that hit the same shell first
// sum their weights through the warp and one of them adds (measured on CAST+LLNL, 1e9 rays: one add per lane made the
// spectra cost 73 % of the kernel, the same-address adds of a warp being serialised in L2).
__device__ __forceinline__ void spec_add_warp(const Spectra& s, int eBin, int shell, double w) {
  const uint32_t e = (blockIdx.x & s.eRepMask) * s.eStride + uint32_t(eBin);
  atomicAdd(s.eW + e, w);
  atomicAdd(s.eW2 + e, w * w);
  atomicAdd(s.eN + e, 1ull);
  const unsigned peers = __match_any_sync(__activemask(), shell);
  double sum = 0.0;
  for (unsigned m = peers; m; m &= m - 1u) sum += __shfl_sync(peers, w, __ffs(m) - 1);
  if ((threadIdx.x & 31u) == unsigned(__ffs(peers) - 1)) {
    const uint32_t k = ((blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) & s.sRepMask) * uint32_t(SART_MAX_SHELLS) + uint32_t(shell);
    atomicAdd(s.sW + k, sum);
    atomicAdd(s.sN + k, (unsigned long long)__popc(peers));
  }
}

// ---- shared memory layout -----------------------------------------------------------------------------------
struct WarpCounters { unsigned int n_exit[16]; unsigned int n_clamped; unsigned int n_unresolved; unsigned int pad[2]; };

// ---- re-trace queue (fast_params.h: RetraceQueue) ------------------------------------------------------------------
// 1: queued (the exact pipeline will trace the ray and account for it), 2: the queue is full (the ray keeps its FP32
// outcome and is counted as unresolved), 0: re-tracing is off.
__device__ __forceinline__ int rq_push(const RetraceQueue& q, uint32_t id) {
  if (q.cap == 0u) return 0;
  const uint32_t slot = atomicAdd(q.count, 1u);
  if (slot < q.cap) { q.list[slot] = id; return 1; }
  return 2;
}
constexpr int kCodeDeferred = 0x40;   // RayResult::code of a ray that went to the re-trace queue (mass scan)

// lowerBound restricted to the guide window [lo, hi]
__device__ __forceinline__ int lower_bound_window(const double* __restrict__ a, int lo, int hi, double key) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Number of the 4 ascending thresholds that are <= w. The thresholds are non-decreasing (build_thresholds), so the
// middle one decides which of t.x / t.z is still open: 3 compares + 1 select instead of 4 compares + 4 selects.
__device__ __forceinline__ int count_le(const uint4& t, uint32_t w) {
  const bool upper = w >= t.y;
  const uint32_t m = upper ? t.z : t.x;
  return (upper ? 2 : 0) + int(w >= m) + int(w >= t.w);
}
// lowerBound over u32 thresholds beyond the 8 prefetched ones (windows wider than 8 entries: flat CDF tails), on
// [from, hi]: the caller passes hi = the next bucket's guide entry, which bounds the answer from above (api.cu
// build_guide), so the search runs over the bucket's window instead of over the rest of the row (CAST+LLNL tables:
// 4.4 instead of 9.8 dependent loads for the 0.5 % of the rays that get here).
static __device__ __noinline__ int thr_search_tail(const uint32_t* __restrict__ thr, int from, int hi, uint32_t w) {
  int lo = from;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (w >= thr[mid]) lo = mid + 1; else hi = mid;   // generic load: the radius thresholds live in shared memory
  }
  return lo;
}
// Upper end of the search window of bucket k of a guide with nBuckets entries: g[k + 1], or n for the last bucket.
__device__ __forceinline__ int guide_upper(const uint16_t* __restrict__ guide, uint32_t k, uint32_t nBuckets, int n) {
  if (k + 1 < nBuckets) { const int g = int(guide[k + 1]); return g < n ? g : n; }
  return n;
}

// Reflectivity at grazing angle alphaDeg from the row pre-interpolated at the ray's energy: linear in the angle.
// (Variants measured on B200 and rejected: rows of overlapping 16-byte quads — one load per lookup, but the table grows by
// a third and CAST+LLNL, whose tables already fill most of one L2 partition, loses 25 %; one aligned 16-byte load plus a
// conditional second one — slower, 35.2 -> 37.6 ms: 16 bytes per lane through L1TEX cost more than the requests saved.)
__device__ __forceinline__ float refl_lookup(const FastParams& P, const float* __restrict__ row, float alphaDeg, bool& clamped,
                                             uint32_t rowOff = 0u) {   // rowOff: 32-bit element offset of the row in `row`
  const float x = fminf(fmaxf(alphaDeg, P.angleMin), P.angleMax);   // NaN -> angleMin
  clamped |= (x != alphaDeg);
  const float fx = (x - P.angleMin) * P.invReflDx;
  int i = int(fx);
  if (i > P.nAngles - 2) i = P.nAngles - 2;
  const float* cell = row + (rowOff + uint32_t(i));   // one 32-bit add + one wide multiply-add per lookup
  const float z0 = __ldg(cell), z1 = __ldg(cell + 1);
  return fmaf(fx - float(i), z1 - z0, z0);
}

// What trace_one knows about a ray. `code` is the exit code of a geometric early return, or -1 when the ray reached
// the weight stage; then weight(m_a) = wPre * conv(m_a) * wPost (finish_ray), so a mass scan re-uses one traced ray.
struct RayResult {
  int code;
  int bin;        // image bin or -1
  int shell;
  bool windowMiss, clamped;
  double wPre;    // reflectivity * cos(yaw) * He absorption        (everything before the window, without P(a->gamma))
  double wPost;   // window or strongback * detector gas * exposure (0 when the window aperture is missed)
  double x, y, r;
  // conversion probability pieces: vacuum convVac = (g B L / 2)^2; gas: Gamma, L, exp(-Gamma L), exp(-Gamma L/2), 1/(2E)
  float convVac, gasGamma, gasE1, gasE2, gasInv2E;   // gasE1 holds 1 - exp(-Gamma L / 2), gasE2 exp(-Gamma L / 2) (conv_factor)
  double gasL;
  // the rest of the Axion record (rt:192-221) for the per-ray entry points; dead code in the fused kernels
  int eIdx;                 // index of the tabulated energy (the X-ray source energy sits at nEnergies)
  double refl;              // reflect rt:2126
  float pre;                // cos(yaw) * He absorption: transmissionMagnet = pre * conversion probability rt:2120
  float yaw, a1, a2;        // yawAngles rt:2123, grazing angles [deg]
  float path;               // pathCB rt:1843
  float devDet;             // deviationDet rt:2085
  float agas;               // transProbArgon rt:2193
};

// Conversion probability for axion mass^2 m2 (computeMagnetTransmission rt:1582-1625 without the cos(ya) factor).
// gasA = 1 - exp(-Gamma L / 2) (from expm1f), gasE2 = exp(-Gamma L / 2). The reference's bracket
//   1 + exp(-Gamma L) - 2 exp(-Gamma L / 2) cos(q L)  =  (1 - exp(-Gamma L / 2))^2 + 4 exp(-Gamma L / 2) sin^2(q L / 2)
// is evaluated in the second form: at the resonance m_a = m_gamma (q -> 0) with a thin gas (Gamma L ~ 1e-4) the first one
// is (Gamma L)^2 / 4 ~ 1e-9 left over from terms of order 1 — nothing in FP32: half the rays of a scan point at the
// resonance came out with weight zero (tests/test_gpu_retrace.py: test_mass_scan_counters_equal_exact_on_1e8_rays).
__device__ __forceinline__ double conv_factor(const FastParams& P, float convVac, float gasGamma, float gasA, float gasE2,
                                              float gasInv2E, double gasL, double m2) {
  if (P.flags & SART_CF_IGNORE_CONV_PROB) return 1.0;
  if (P.stage == SART_SK_VACUUM) return double(convVac);
  const double q = fabs(P.gasMgamma2 - m2) * double(gasInv2E);   // momentumTransfer am:63-68
  double ph = q * gasL;   // phase reduced in FP64 before the FP32 sine
  ph = fma(-6.283185307179586, rint(ph * 0.15915494309189535), ph);   // [-pi, pi]
  // sin of the half phase, |x| <= pi / 2, with RELATIVE accuracy also for a tiny phase (the MUFU sine has an absolute one):
  // the odd series to x^11 (remainder x^13 / 13! <= 6e-8 at pi / 2), 7 instructions, no range reduction needed
  const float x = float(0.5 * ph), x2 = x * x;
  const float sh = x * fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, -2.5052108e-8f, 2.7557319e-6f), -1.9841270e-4f),
                                                   8.3333333e-3f), -0.16666667f), 1.0f);
  const double g = double(gasGamma);
  const double den = fma(q, q, 0.25 * g * g);
  const double term2 = den > 1e-30 ? rcp_nr(den) : 1.0 / den;   // rcp_nr seeds in FP32: a resonance in a near-vacuum leaves its range
  const double a = double(gasA), s2 = double(sh) * double(sh);   // FP64 products: (Gamma L)^2 may leave the FP32 range
  return P.gasTerm1 * term2 * fma(a, a, 4.0 * double(gasE2) * s2);
}
// Tail of traceAxion for one axion mass: exit code | flags and the final weight.
template <bool kFolded>
__device__ __forceinline__ int finish_ray(const FastParams& P, const RayResult& r, double m2, double& w) {
  const double w0 = kFolded ? r.wPre
                            : r.wPre * conv_factor(P, r.convVac, r.gasGamma, r.gasE1, r.gasE2, r.gasInv2E, r.gasL, m2);
  int flags = (w0 != 0.0) ? SART_FLAG_PASSED_TILL_WINDOW : 0;
  if (r.clamped) flags |= SART_FLAG_INTERP_CLAMPED;
  w = 0.0;
  if (r.windowMiss) return SART_EXIT_WINDOW_APERTURE | flags;
  w = w0 * r.wPost;
  return ((w != 0.0) ? SART_EXIT_PASSED : SART_EXIT_ZERO_WEIGHT) | flags;
}

// transmissionMagnet of a ray that reached the weight stage (rt:2120) for axion mass^2 m2: the record's value
// (store_record) and the quantity histograms' (QuantityHistSink).
__device__ __forceinline__ double trans_magnet(const FastParams& P, const RayResult& r, double m2) {
  return double(r.pre) * conv_factor(P, r.convVac, r.gasGamma, r.gasE1, r.gasE2, r.gasInv2E, r.gasL, m2);
}

// The Axion record (rt:192-221) of one ray of the throughput pipelines, written to the structure of arrays `o` (device
// pointers). Fields of the weight stage (reflect, transmissionMagnet, yawAngles, the grazing angles, pathCB, deviationDet)
// are defined for the rays that reach it — exit codes PASSED, ZERO_WEIGHT, WINDOW_APERTURE, which is every ray
// generateResultPlots (rt:2246-2289) reads them from — and 0 for rays clipped before; x, y, r, shellNumber and
// transProbArgon for the rays past the window aperture, like the exact pipeline (kernels_exact.cu: store_ray).
// kOptional = false: the caller asked for none of the optional arrays (the launcher checks the pointers), so neither their
// null tests nor the values behind them are compiled in.
template <bool kOptional = true>
__device__ __forceinline__ void store_record(const FastParams& P, const sart_ray_out_t& o, size_t i, const RayResult& r,
                                             double m2, double energyKeV) {
  int code = r.code;
  double wd = 0.0;
  const bool weighted = r.code < 0;
  if (weighted) code = finish_ray<true>(P, r, m2, wd);
  else if (r.clamped) code |= SART_FLAG_INTERP_CLAMPED;
  const int ec = code & SART_CODE_MASK;
  const bool tail = ec == SART_EXIT_PASSED || ec == SART_EXIT_ZERO_WEIGHT;
  o.x[i] = tail ? r.x : 0.0; o.y[i] = tail ? r.y : 0.0; o.w[i] = wd; o.code[i] = code; o.shell[i] = tail ? r.shell : -1;
  if (!kOptional) return;
  if (o.energy) o.energy[i] = energyKeV;
  if (o.reflect) o.reflect[i] = weighted ? r.refl : 0.0;
  if (o.transMagnet) o.transMagnet[i] = weighted ? trans_magnet(P, r, m2) : 0.0;
  if (o.yaw) o.yaw[i] = weighted ? double(r.yaw) : 0.0;
  if (o.alpha1) o.alpha1[i] = weighted ? double(r.a1) : 0.0;
  if (o.alpha2) o.alpha2[i] = weighted ? double(r.a2) : 0.0;
  if (o.pathCB) o.pathCB[i] = weighted ? double(r.path) : 0.0;
  if (o.r) o.r[i] = tail ? r.r : 0.0;
  if (o.deviationDet) o.deviationDet[i] = weighted ? double(r.devDet) : 0.0;
  if (o.transProbArgon) o.transProbArgon[i] = tail ? double(r.agas) : 0.0;
}

// Sink that keeps the outcome as a RayResult (per-ray records, mass scan).
template <bool kFoldT, bool kRecordT = true>
struct RecordSink {
  static constexpr bool kFold = kFoldT;
  static constexpr bool kRecord = kRecordT;   // false: the record fields nobody reads (pathCB, deviationDet) are not computed
  RayResult& out;
  double m2;
  const RetraceQueue& rq;
  bool dropDeferred;   // mass scan: a queued ray is dropped here (code = kCodeDeferred); the per-ray entry points write the
                       // FP32 record anyway and the exact pipeline overwrites it
  bool unresolved = false;
  __device__ __forceinline__ bool defer(uint32_t id) {
    const int r = rq_push(rq, id);
    unresolved |= (r == 2);
    if (r == 1 && dropDeferred) { fail(kCodeDeferred); return true; }
    return false;
  }
  __device__ __forceinline__ void fail(int code) {
    out.code = code; out.clamped = false; out.windowMiss = false; out.bin = -1; out.shell = -1;
    out.x = out.y = out.r = 0.0; out.wPre = out.wPost = 0.0;
    out.refl = 0.0; out.pre = out.yaw = out.a1 = out.a2 = out.devDet = out.agas = 0.f;
  }
  __device__ __forceinline__ void hit(const RayResult& h) { out = h; out.code = -1; }
};

// Sink of the fused kernels: the tail of traceAxion (rt:2135-2221) + prepareHeatmap (rt:839-842) for one axion mass,
// applied where the ray's outcome becomes known. Sums live in the caller's registers, exit counts in the warp's
// shared-memory counters.
// kRadial = false compiles the optional radial histogram out (the plain-run kernel variants; the launcher takes the generic
// variant when sart_enable_radial_hist is on). kSpectra = false compiles the spectra out: the FP32 launcher has generic
// variants with and without them, so that a run without spectra runs the code it ran before they existed (measured on
// BabyIAXO+XMM: the spectra code compiled in but off made the compacting kernel 4 % slower).
template <bool kRadial, bool kSpectra = kRadial>
struct ImageSinkT {
  static constexpr bool kFold = true;
  static constexpr bool kRecord = false;
  const FastTables& T;
  double m2;
  double* __restrict__ image;
  double* __restrict__ imageW2;
  uint32_t rep;   // element offset of this block's image replica (32-bit: one wide multiply-add per address)
  WarpCounters& wc;
  unsigned int &nPassed, &nTill;
  double &sumW, &sumW2, &sumX, &sumY, &sumR;
  __device__ __forceinline__ bool defer(uint32_t id) {
    const int r = rq_push(T.rq, id);
    if (r == 2) atomicAdd(&wc.n_unresolved, 1u);
    return r == 1;
  }
  __device__ __forceinline__ void fail(int code) { atomicAdd(&wc.n_exit[code], 1u); }
  __device__ __forceinline__ void hit(const RayResult& h) {
    const double w0 = h.wPre;   // conversion probability already folded in
    if (w0 != 0.0) ++nTill;                                   // passedTillWindow rt:2135-2136
    if (h.clamped) atomicAdd(&wc.n_clamped, 1u);
    if (h.windowMiss) { atomicAdd(&wc.n_exit[SART_EXIT_WINDOW_APERTURE], 1u); return; }
    const double wd = w0 * h.wPost;
    if (wd != 0.0) {                                          // passed rt:2220
      ++nPassed;
      sumW += wd; sumW2 += wd * wd; sumX += h.x; sumY += h.y; sumR += h.r;
#ifndef SART_NO_IMAGE_ATOMICS   // (experiment switch: measures what the histogram atomics cost)
      if (h.bin >= 0) {
        const uint32_t at = rep + uint32_t(h.bin);
        atomicAdd(image + at, wd);
        atomicAdd(imageW2 + at, wd * wd);
      }
#endif
      if (kRadial && T.rad.w) rad_add(T.rad, h.r, wd);
      if (kSpectra && T.spec.eW) spec_add_warp(T.spec, h.eIdx, h.shell, wd);
    } else {
      atomicAdd(&wc.n_exit[SART_EXIT_ZERO_WEIGHT], 1u);
    }
  }
};
using ImageSink = ImageSinkT<true>;

// Sink of the band-image kernel variants (sart_enable_band_images): the generic sink, with the radial histogram and the
// spectra checked at run time, plus the band images B (device_params.h: BandImages; here their replicas, bandRep this block's
// replica) and the block's per-band counts bandN in shared memory, which the kernel flushes once at its end. A derived sink,
// so that ImageSinkT, and every kernel variant built on it, stays what it was before the band images existed.
// A passed ray of weight wd into the band images of a throughput kernel: its band's count in shared memory, Σw and Σw² into
// replica bandRep of its band's plane.
__device__ __forceinline__ void band_hit(const BandImages& B, unsigned int* bandN, uint32_t bandRep, const RayResult& h,
                                         double wd) {
  const unsigned k = __ldg(B.band + h.eIdx);
  if (k == kNoBand) return;
  atomicAdd(bandN + k, 1u);
  if (h.bin < 0) return;
  const uint32_t at = bandRep + k * uint32_t(SART_IMAGE_BINS * SART_IMAGE_BINS) + uint32_t(h.bin);
  atomicAdd(B.w + at, wd);
  atomicAdd(B.w2 + at, wd * wd);
}
struct BandImageSink : ImageSinkT<true, true> {
  const BandImages& B;
  unsigned int* bandN;
  uint32_t bandRep;
  __device__ __forceinline__ void hit(const RayResult& h) {
    ImageSinkT<true, true>::hit(h);
    const double wd = h.wPre * h.wPost;   // the weight ImageSinkT::hit tested
    if (h.windowMiss || wd == 0.0) return;
    band_hit(B, bandN, bandRep, h, wd);
  }
};

// The block's per-band counts of the band-image kernel variants (BandImageSink::bandN): shared memory, zeroed by the threads
// 0 .. SART_MAX_BANDS - 1 before the kernel's first __syncthreads, added to the handle's counts once at the end of the
// kernel (one global atomic per band and block instead of one per ray). nullptr without band images.
template <bool kBands>
__device__ __forceinline__ unsigned int* band_counts() {
  if constexpr (kBands) {
    __shared__ unsigned int n[SART_MAX_BANDS];
    if (threadIdx.x < SART_MAX_BANDS) n[threadIdx.x] = 0u;
    return n;
  } else {
    return nullptr;
  }
}
__device__ __forceinline__ uint32_t band_replica(const BandImages& B) { return (blockIdx.x & B.repMask) * B.repStride; }
// The sink of a fused kernel body shared by a variant without band images (kBands = false: `sink` itself) and one with them.
template <bool kBands, class Sink>
__device__ __forceinline__ auto with_bands(const Sink& sink, const BandImages& B, unsigned int* bandN) {
  if constexpr (kBands) return BandImageSink{sink, B, bandN, band_replica(B)};
  else return sink;
}
__device__ __forceinline__ void band_counts_flush(const BandImages& B, const unsigned int* n) {
  __syncthreads();
  if (threadIdx.x < unsigned(B.nBands) && n[threadIdx.x]) atomicAdd(B.n + threadIdx.x, (unsigned long long)n[threadIdx.x]);
}

// ---- quantity histograms of the throughput kernels (sart_enable_quantity_hists; device_params.h: QuantityHists) ------
// The record quantity q (SART_Q_*) of a ray that passed, as store_record writes it.
__device__ __forceinline__ double record_quantity(const FastParams& P, const RayResult& h, double m2, int q) {
  switch (q) {
    case SART_Q_REFLECT: return h.refl;
    case SART_Q_TRANS_MAGNET: return trans_magnet(P, h, m2);
    case SART_Q_YAW: return double(h.yaw);
    case SART_Q_ALPHA1: return double(h.a1);
    case SART_Q_ALPHA2: return double(h.a2);
    case SART_Q_PATH_CB: return double(h.path);
    case SART_Q_DEVIATION_DET: return double(h.devDet);
    default: return double(h.agas);
  }
}

// The block-private part of the histograms in dynamic shared memory, behind everything else the kernel keeps there: the
// counts as u32 (a block traces fewer than 2^32 rays), and with kSmemSums also Σw and Σw² as f64, so that a passed ray costs
// shared-memory atomics only and the block adds its entries into the handle's arrays once, at its end (the f64 adds are
// CAS loops in shared memory: ATOMS.CAST.SPIN.64). Without kSmemSums the sums go to the block replicas in global memory
// (QuantityHists::rw, rw2) instead.
struct QhistSmem {
  double* w;
  double* w2;
  unsigned int* n;
};
// Bytes the launcher adds to the block's dynamic shared memory (16 for the alignment of the part).
__host__ __device__ inline size_t qhist_smem_bytes(int entries, bool sums) {
  return 16 + ((size_t(entries) * (sums ? 20 : 4) + 15) & ~size_t(15));
}
// The launchers' choice between the two: the replicas, unless SART_QHIST_SMEM is set and the block, `smem` bytes without the
// histograms, still fits the per-block limit with the sums. Measured on B200 (tools/bench_quantity_hists.py, 1e9 rays,
// 2 and 8 histograms at 256 bins, CAST+LLNL and BabyIAXO+XMM): the two within 2 % of each other, the replicas ahead in
// three of the four cases.
inline bool qhist_sums_in_smem(size_t smem, int entries) {
  if (!std::getenv("SART_QHIST_SMEM")) return false;
  int dev = 0, optin = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
    return false;
  return smem + qhist_smem_bytes(entries, true) <= size_t(optin);
}
// Lays the part over `base` (the end of the kernel's own shared memory) and zeroes it; before the kernel's first
// __syncthreads.
template <bool kSmemSums>
__device__ __forceinline__ QhistSmem qhist_smem(unsigned char* base, const QuantityHists& Q) {
  QhistSmem s;
  const int e = Q.entries;
  unsigned char* p = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(base) + 15) & ~uintptr_t(15));
  if (kSmemSums) {
    s.w = reinterpret_cast<double*>(p); s.w2 = s.w + e; s.n = reinterpret_cast<unsigned int*>(s.w2 + e);
  } else {
    s.w = s.w2 = nullptr; s.n = reinterpret_cast<unsigned int*>(p);
  }
  for (int i = threadIdx.x; i < e; i += blockDim.x) {
    s.n[i] = 0u;
    if (kSmemSums) { s.w[i] = 0.0; s.w2[i] = 0.0; }
  }
  return s;
}
// The block's entries into the handle's arrays: the counts, and with kSmemSums the sums; once, at the end of the kernel.
template <bool kSmemSums>
__device__ __forceinline__ void qhist_flush(const QuantityHists& Q, const QhistSmem& s) {
  __syncthreads();
  for (int e = threadIdx.x; e < Q.entries; e += blockDim.x) {
    const unsigned int c = s.n[e];
    if (!c) continue;
    atomicAdd(Q.n + e, (unsigned long long)c);
    if (kSmemSums) { atomicAdd(Q.w + e, s.w[e]); atomicAdd(Q.w2 + e, s.w2[e]); }
  }
}

// Sink of the quantity-histogram kernel variants: the generic sink with the radial histogram and the spectra checked at run
// time, the band images checked at run time (B.w), and the histograms Q. kRecord: pathCB and deviationDet are computed,
// as for a per-ray record. A derived sink like BandImageSink, so that every kernel variant without the histograms stays
// what it was.
template <bool kSmemSums>
struct QuantityHistSink : ImageSinkT<true, true> {
  static constexpr bool kRecord = true;
  const FastParams& P;
  const BandImages& B;
  unsigned int* bandN;
  uint32_t bandRep;
  const QuantityHists& Q;
  QhistSmem s;
  uint32_t qRep;   // element offset of this block's replica of the sums (without kSmemSums)
  __device__ __forceinline__ void hit(const RayResult& h) {
    ImageSinkT<true, true>::hit(h);
    const double wd = h.wPre * h.wPost;   // the weight ImageSinkT::hit tested
    if (h.windowMiss || wd == 0.0) return;
    if (B.w) band_hit(B, bandN, bandRep, h, wd);
    // The lanes of a warp that hit the same entry first sum through the warp and one of them adds (as spec_add_warp): a
    // distribution piles most rays into a few entries, and same-address f64 adds are serialised (in shared memory a CAS
    // loop per add).
    for (int j = 0; j < Q.nHists; ++j) {
      const uint32_t e = uint32_t(Q.off[j] + qhist_entry(Q, j, record_quantity(P, h, m2, Q.quantity[j])));
      const unsigned active = __activemask();
      const unsigned peers = __match_any_sync(active, e);
      double sw = 0.0, sw2 = 0.0;
      if (peers == 0xffffffffu) {   // the whole warp in one entry (a distribution's peak): 5 butterfly steps, not 32 shuffles
        sw = wd; sw2 = wd * wd;
        for (int o = 16; o > 0; o >>= 1) {
          sw += __shfl_xor_sync(peers, sw, o);
          sw2 += __shfl_xor_sync(peers, sw2, o);
        }
      } else {
        for (unsigned m = peers; m; m &= m - 1u) {
          const double x = __shfl_sync(peers, wd, __ffs(m) - 1);
          sw += x;
          sw2 += x * x;
        }
      }
      if ((threadIdx.x & 31u) != unsigned(__ffs(peers) - 1)) continue;
      atomicAdd(s.n + e, unsigned(__popc(peers)));
      if (kSmemSums) {
        atomicAdd(s.w + e, sw);
        atomicAdd(s.w2 + e, sw2);
      } else {
        atomicAdd(Q.rw + (qRep + e), sw);
        atomicAdd(Q.rw2 + (qRep + e), sw2);
      }
    }
  }
};
__device__ __forceinline__ uint32_t qhist_replica(const QuantityHists& Q) { return (blockIdx.x & Q.repMask) * Q.repStride; }
// The sink of a fused kernel body shared by the variants without quantity histograms (kQH = 0: with_bands) and those with
// them (kQH = 1: sums in shared memory, 2: sums in the block replicas).
template <bool kBands, int kQH, class Sink>
__device__ __forceinline__ auto with_extras(const Sink& sink, const FastParams& P, const BandImages& B, unsigned int* bandN,
                                            const QuantityHists& Q, const QhistSmem& qs) {
  if constexpr (kQH != 0)
    return QuantityHistSink<kQH == 1>{sink, P, B, bandN, band_replica(B), Q, qs, qhist_replica(Q)};
  else
    return with_bands<kBands>(sink, B, bandN);
}

// ---- axion-mass scan: the part shared by the FP64-algebra and the FP32 tracing --------------------------------
// Per-mass spectra of the mass-scan kernels (sart_enable_mass_spectra), in FastTables::spec: accumulators laid out like
// the image's, [bin][SART_MAX_MASSES] (eW, eW2: bin = energy index, nEnergies for the X-ray source) and
// [shell][SART_MAX_MASSES] (sW), so that the 32 mass lanes of a warp add to consecutive addresses. The counts eN / sN are
// 32-bit arrays of the same shapes: a launch has at most kMaxRaysPerLaunch = 2^31 rays, so no bin overflows before
// k_fold_mass_spectra widens it into the handle's 64-bit counts, and a warp's 32 lanes touch 128 bytes instead of 256.
__device__ __forceinline__ void mass_spec_add(const Spectra& a, int m, int eBin, int shell, double w) {
  const uint32_t e = uint32_t(eBin) * SART_MAX_MASSES + uint32_t(m), k = uint32_t(shell) * SART_MAX_MASSES + uint32_t(m);
  atomicAdd(a.eW + e, w);
  atomicAdd(a.eW2 + e, w * w);
  atomicAdd(reinterpret_cast<unsigned int*>(a.eN) + e, 1u);
  atomicAdd(a.sW + k, w);
  atomicAdd(reinterpret_cast<unsigned int*>(a.sN) + k, 1u);
}

// Rays are traced once (lanes = rays) by `trace(global ray index, RayResult&)`; each ray that reaches the weight stage
// is then broadcast through the warp and weighted for all M masses at once with lanes = masses (mass lane + 32 k), so
// the per-mass sums live in registers of the lane that owns the mass and need no reduction. `image` / `imageW2` are the
// mass-major accumulators [bin][SART_MAX_MASSES] (see k_fold_mass_acc).
// kPer = masses per lane (1, 2 or SART_MAX_MASSES / 32): the launcher picks the smallest that holds nMasses, because the
// per-mass sums are 15 registers per mass and lane (with 4 masses per lane the FP32 kernel spilled: 80 registers, 112 bytes).
// kSpectra: the passed ray-masses also go to the per-mass spectra `spec` (mass_spec_add); false compiles them out.
// kRows: the passed ray-masses also go to the per-mass radial histograms and band images R that are on (device_params.h:
// MassRows; here mass-minor accumulators like the image's: Σw [bin][SART_MAX_MASSES] and a 32-bit count of the same shape
// for the radial histograms, Σw and Σw² [band][256 * 256][SART_MAX_MASSES] and a 32-bit count [band][SART_MAX_MASSES] for
// the band images, which k_fold_mass_acc / k_fold_mass_hist add into the handle's rows after every launch of at most
// kMaxRaysPerLaunch rays). The tracing lane resolves its ray's radial bin and band, so that two integers go through the
// broadcast. The band counts are
// a few hundred addresses that every passed ray-mass of the grid would add to, so a block counts them in shared memory and
// adds them into the accumulators once, at its end (measured on B200, config 4, 4 bands: with the counts in global memory
// the band images cost 5.98x the plain scan).
template <int kPer, bool kSpectra, bool kRows = false, class Trace>
__device__ __forceinline__ void mass_scan_loop(const FastParams& P, const RadialHist& rad, const Spectra& spec, const MassRows& R,
                                               const double* __restrict__ masses, int nMasses, uint64_t first, uint64_t nRays,
                                               double* __restrict__ image, double* __restrict__ imageW2,
                                               sart_counters_t* __restrict__ counters, WarpCounters* wc, Trace trace) {
  static_assert(kPer >= 1 && kPer <= SART_MAX_MASSES / 32, "masses per lane");
  constexpr unsigned kFull = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double m2[kPer], sumW[kPer], sumW2[kPer], sumX[kPer], sumY[kPer], sumR[kPer];
  unsigned int nPassed[kPer], nZero[kPer], nTill[kPer];
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int m = lane + 32 * k;
    const double mm = m < nMasses ? masses[m] : 0.0;
    m2[k] = mm * mm;
    sumW[k] = sumW2[k] = sumX[k] = sumY[k] = sumR[k] = 0.0;
    nPassed[k] = nZero[k] = nTill[k] = 0u;
  }
  unsigned int nIter = 0;
  unsigned int* bandN = nullptr;   // kRows: the block's band counts [band][SART_MAX_MASSES]
  if constexpr (kRows) {
    __shared__ unsigned int n[SART_MAX_BANDS * SART_MAX_MASSES];
    for (int i = threadIdx.x; i < SART_MAX_BANDS * SART_MAX_MASSES; i += blockDim.x) n[i] = 0u;
    __syncthreads();
    bandN = n;
  }
  const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
  for (uint64_t b = uint64_t(blockIdx.x) * blockDim.x + (threadIdx.x & ~31); b < nRays; b += stride) {   // warp-uniform
    const uint64_t i = b + lane;
    const bool valid = i < nRays;
    RayResult r;
    r.code = SART_N_EXIT_CODES;
    if (valid) {
      if (trace(first + i, uint32_t(i), r)) atomicAdd(&wc[warp].n_unresolved, 1u);
      ++nIter;
      if (r.code == kCodeDeferred) { r.clamped = false; }   // queued for the exact pipeline, which accounts for it
      else if (r.code >= 0) atomicAdd(&wc[warp].n_exit[r.code], 1u);
      else if (r.windowMiss) atomicAdd(&wc[warp].n_exit[SART_EXIT_WINDOW_APERTURE], 1u);
      if (r.clamped) atomicAdd(&wc[warp].n_clamped, 1u);
    }
    int radBin = 0, band = kNoBand;   // kRows: this lane's ray's radial bin and band
    if (kRows && valid && r.code < 0) {
      if (R.rad.w) {
        radBin = int(r.r * R.rad.invStep);
        radBin = radBin < 0 ? 0 : (radBin > R.rad.nbins - 1 ? R.rad.nbins - 1 : radBin);
      }
      if (R.band.w) band = __ldg(R.band.band + r.eIdx);
    }
    unsigned alive = __ballot_sync(kFull, valid && r.code < 0);
    while (alive) {
      const int src = __ffs(alive) - 1;
      alive &= alive - 1;
      const double wPre = __shfl_sync(kFull, r.wPre, src), wPost = __shfl_sync(kFull, r.wPost, src);
      const double gasL = __shfl_sync(kFull, r.gasL, src);
      const float convVac = __shfl_sync(kFull, r.convVac, src), gG = __shfl_sync(kFull, r.gasGamma, src);
      const float gE1 = __shfl_sync(kFull, r.gasE1, src), gE2 = __shfl_sync(kFull, r.gasE2, src);
      const float gI = __shfl_sync(kFull, r.gasInv2E, src);
      const double x = __shfl_sync(kFull, r.x, src), y = __shfl_sync(kFull, r.y, src), rr = __shfl_sync(kFull, r.r, src);
      const int bin = __shfl_sync(kFull, r.bin, src);
      const bool miss = __shfl_sync(kFull, int(r.windowMiss), src) != 0;
      const int eBin = kSpectra ? __shfl_sync(kFull, r.eIdx, src) : 0, shell = kSpectra ? __shfl_sync(kFull, r.shell, src) : 0;
      const int rBin = kRows ? __shfl_sync(kFull, radBin, src) : 0, bBand = kRows ? __shfl_sync(kFull, band, src) : int(kNoBand);
#pragma unroll
      for (int k = 0; k < kPer; ++k) {
        const int m = lane + 32 * k;
        if (m >= nMasses) continue;
        const double w0 = wPre * conv_factor(P, convVac, gG, gE1, gE2, gI, gasL, m2[k]);
        if (w0 != 0.0) ++nTill[k];
        if (miss) continue;
        const double w = w0 * wPost;
        if (w != 0.0) {
          ++nPassed[k];
          sumW[k] += w; sumW2[k] += w * w; sumX[k] += x; sumY[k] += y; sumR[k] += rr;
          if (bin >= 0) {
            // mass-major accumulators [bin][SART_MAX_MASSES]: the 32 lanes (= 32 masses) of this warp add to 256
            // consecutive bytes instead of to 32 image planes 512 KiB apart; k_fold_mass_acc transposes afterwards
            atomicAdd(image + size_t(bin) * SART_MAX_MASSES + m, w);
            atomicAdd(imageW2 + size_t(bin) * SART_MAX_MASSES + m, w * w);
          }
          if (m == 0 && rad.w) rad_add(rad, rr, w);   // the radial histogram follows the first mass, as in the exact kernel
          if (kSpectra) mass_spec_add(spec, m, eBin, shell, w);
          if (kRows && R.rad.w) {
            const uint32_t at = uint32_t(rBin) * SART_MAX_MASSES + uint32_t(m);
            atomicAdd(R.rad.w + at, w);
            atomicAdd(reinterpret_cast<unsigned int*>(R.rad.n) + at, 1u);
          }
          if (kRows && bBand != int(kNoBand)) {
            atomicAdd(bandN + (uint32_t(bBand) * SART_MAX_MASSES + uint32_t(m)), 1u);
            if (bin >= 0) {
              const uint32_t at = (uint32_t(bBand) * uint32_t(SART_IMAGE_BINS * SART_IMAGE_BINS) + uint32_t(bin)) * SART_MAX_MASSES +
                                  uint32_t(m);
              atomicAdd(R.band.w + at, w);
              atomicAdd(R.band.w2 + at, w * w);
            }
          }
        } else {
          ++nZero[k];
        }
      }
    }
  }
  // ---- flush: the lane that owns a mass adds its sums; geometric exits are the same for every mass
  for (int o = 16; o > 0; o >>= 1) nIter += __shfl_down_sync(kFull, nIter, o);
  nIter = __shfl_sync(kFull, nIter, 0);
  __syncwarp();
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int m = lane + 32 * k;
    if (m >= nMasses) continue;
    sart_counters_t* c = counters + m;
    auto addu = [](uint64_t* p, unsigned long long v) { if (v) atomicAdd(reinterpret_cast<unsigned long long*>(p), v); };
    addu(&c->n_rays, nIter);
    addu(&c->n_exit[SART_EXIT_PASSED], nPassed[k]);
    addu(&c->n_exit[SART_EXIT_ZERO_WEIGHT], nZero[k]);
    addu(&c->n_passed, nPassed[k]);
    addu(&c->n_passed_till_window, nTill[k]);
    for (int e = 1; e < SART_N_EXIT_CODES; ++e)
      if (e != SART_EXIT_ZERO_WEIGHT) addu(&c->n_exit[e], wc[warp].n_exit[e]);
    addu(&c->n_hit_nickel, wc[warp].n_exit[SART_EXIT_NICKEL]);
    addu(&c->n_interp_clamped, wc[warp].n_clamped);
    addu(&c->n_unresolved, wc[warp].n_unresolved);
    atomicAdd(&c->sum_w, sumW[k]); atomicAdd(&c->sum_w2, sumW2[k]);
    atomicAdd(&c->sum_x, sumX[k]); atomicAdd(&c->sum_y, sumY[k]); atomicAdd(&c->sum_r, sumR[k]);
  }
  if constexpr (kRows) {
    __syncthreads();
    for (int i = threadIdx.x; i < R.band.nBands * SART_MAX_MASSES; i += blockDim.x)
      if (bandN[i]) atomicAdd(reinterpret_cast<unsigned int*>(R.band.n) + i, bandN[i]);
  }
}

}  // namespace fast
}  // namespace sart
