// device_params.h — the POD blocks the kernels read: run-wide scalars (passed as a __grid_constant__ kernel
// parameter) and one constant record per mirror shell (a small array in HBM, L1/L2 resident).
//
// Everything here is derived ONCE on the host from sart_setup_t (derive.cpp). The reference recomputes these
// per ray inside traceAxion (tan/cos/sin of the shell angle, r2..r5, distanceMirrors, distDet, lengthTelescope,
// rotation sines/cosines: src/raytracer.nim:1879-1884, 1951-1957, 1971-1973, 2070-2072, 639-644, 669-672,
// 702-715); hoisting them does not change a single bit because each value is produced by the same expression.
#pragma once
#include <cstdint>

#include "../../include/sart.h"

namespace sart {

// Per-shell constants, f64. Names follow the reference's variables.
struct ShellF64 {
  double R1;        // allR1[j]
  double R1pT;      // allR1[j] + allThickness[j]   (glass front rt:1942-1943; nickel test of the shell above rt:1722)
  double r1sq;      // R1*R1
  double r4;        // rt:1954-1956
  double r4sq;
  double distanceMirrors;  // cos(beta)*(xSep + lMirror)  rt:1973
  double distDet;   // rt:2070-2072
  double ddWin;     // distDet / cos(pipesTurned)              rt:811
  double ddEnd;     // (distDet + depthDet) / cos(pipesTurned) rt:2081, 811
  // cone, mirror 1 (angle = beta, distMirr = 0): tan, tan^2, r1*tan, (2 r1)*tan, distMirr + lMirror*cos(angle)
  double tan1, k1, r1tan1, two_r1_tan1, zmax1;
  // cone, mirror 2 (angle = 3 beta, radius r4, distMirr = distanceMirrors)
  double tan2, k2, r4tan2, two_r4_tan2, zmax2;
  // paraboloid (mirror 1 of XMM/Abrixas, angle = beta)  rt:669-676, 743-746
  double p_r3, p_e, p_r3sq, p_el, p_r3tan, p_r3_2tan;
  // hyperboloid (mirror 2 of XMM/Abrixas, angle = 3 beta)  rt:702-715, 749-758
  double h_r3, h_e, h_g, h_r3sq, h_el, h_gll, h_2g, h_nden, h_r3tan, h_r3_2tan;
};

struct Params {
  // enums / counts
  int32_t telKind, nShells, reflKind, nCoatings, stage, experiment, nStripHalf, testXray;
  uint32_t flags;
  int32_t layers[SART_MAX_COATINGS];
  int32_t holeType, numberOfHoles, parallelSource;
  int32_t shellsMonotonic;   // R1 strictly increasing and no glass reaching the next shell: the shell scan may stop early
  // sun + sampling
  double sunX, sunY, sunZ, radiusSun;
  // magnet / pipes (z of the clip planes, radii)
  double radiusCB, lengthB, zExitCB, zPipe1, zPipe2, rPipe1;
  double B, g_agamma, tesla_to_eV2, m_to_inv_eV;
  double pGas, tGas, roomTemp, radiusCB_m;  // pGas = pGasRoom/roomTemp*tGas rt:1601
  // telescope frame
  double cosTX, sinTX, cosTY, sinTY, halfLenTel, oeX, oeY;
  double lMirror, fL;  // fL = distanceDetectorXRT
  double holeInOptics;
  // detector plane
  double cosPipe, sinPipe, dShift, lateralShift, transversalShift;
  double radiusWindow, chipCX, chipCY, cosTheta, sinTheta, stripDist, stripWidth;
  double exposureFactor;
  // X-ray test source rt:1765-1806
  double srcX, srcY, srcZ, srcRadius, srcEnergy, colZ;
  // reflectivity grid
  int32_t nAngles, nReflEnergies;
  double angleMin, angleMax, reflEMin, reflEMax, reflDx, reflDy;
  // solar model
  int32_t nRadii, nEnergies;
};

// Optional weighted radial histogram of the passed rays (pointdataR rt:2202) for the containment radii of
// generateResultPlots (rt:2459-2527): bin = floor(r * invStep), the last bin collects everything beyond. w == nullptr: off.
struct RadialHist {
  double* w;                 // [nbins] sum of weights
  unsigned long long* n;     // [nbins] number of rays
  double invStep;
  int32_t nbins, pad;
};

// Optional spectra of the passed rays (sart_enable_spectra): Σw, Σw² and the ray count per energy bin (the index of the
// ray's tabulated energy, rt:470; bin nEnergies = the X-ray source), Σw and the ray count per mirror shell (shellNumber
// rt:2198). eW == nullptr: off. Replica r of the energy arrays starts r * eStride elements in, replica r of the shell
// arrays r * SART_MAX_SHELLS; a block adds into energy replica (block & eRepMask) and a warp into shell replica
// (global warp & sRepMask). Masks 0 = the arrays themselves (the exact kernels; the throughput kernels get replicas that a
// fold kernel adds up after the launch). 64 bytes: the kernel parameters behind a table block keep their 16-byte alignment.
struct Spectra {
  double* eW;
  double* eW2;
  unsigned long long* eN;
  double* sW;
  unsigned long long* sN;
  uint32_t eStride, eRepMask, sRepMask, pad[3];
};
static_assert(sizeof(Spectra) == 64, "Spectra: 64 bytes");

#if defined(__CUDACC__)
__device__ __forceinline__ void spec_add(const Spectra& s, int eBin, int shell, double w) {
  const uint32_t e = (blockIdx.x & s.eRepMask) * s.eStride + uint32_t(eBin);
  atomicAdd(s.eW + e, w);
  atomicAdd(s.eW2 + e, w * w);
  atomicAdd(s.eN + e, 1ull);
  const uint32_t k = ((blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) & s.sRepMask) * uint32_t(SART_MAX_SHELLS) + uint32_t(shell);
  atomicAdd(s.sW + k, w);
  atomicAdd(s.sN + k, 1ull);
}
#endif

// Table pointers (device memory).
struct Tables {
  const double* energies;
  const double* fluxRadiusCDF;
  const double* diffFluxCDFs;
  const double* reflectivity;
  const double *sbX, *sbY, *wdX, *wdY, *gaX, *gaY, *ttX, *ttY;
  int32_t sbN, wdN, gaN, ttN;
  const ShellF64* shells;
  RadialHist rad;
  // Optional guide tables of the two CDFs (null: search the whole table): guide[k] = lowerBound(cdf, k / nBuckets), so the
  // lower bound of a uniform of bucket k lies in [guide[k], guide[k + 1]] and the binary search of rt:437 / rt:464 runs over
  // that window instead of over the whole CDF — the same index, a fraction of the dependent loads.
  const uint16_t* radiusGuide;   // [kRadGuide]
  const uint16_t* energyGuide;   // [nRadii][kEnGuide]
  // Optional (null: interpolate per ray): window / strongback / detector-gas factors of rt:2165-2190 at each tabulated
  // energy, evaluated on the host by the very expression the device uses (eval_linear1d: same IEEE operations, no
  // contraction on either side => the same bits). A Monte Carlo ray's energy is a table value (rt:470), so its three
  // 10-step binary searches with dependent loads become one 32-byte record.
  const struct EnergyFactors* energyFactors;   // [nEnergies]
  Spectra spec;   // optional (last member: the offsets of the fields above stay those of the kernels built without it)
};
struct EnergyFactors {
  double window, strongback, gas;
  int32_t clamped;   // bit 0 / 1 / 2: the energy lies outside the window / strongback / gas grid
  int32_t pad;
};

// Guide-table buckets per CDF row; the bucket of the uniform (w + 0.5) 2^-32 is w >> (32 - bits). Sized so that the
// flat tails of the CDFs (hundreds of entries sharing 1e-3 of the probability) still resolve within the 8 thresholds
// the kernel prefetches for all but ~1e-3 of the rays: radius guide 16 KiB of shared memory, energy guide 4 KiB per row (larger guides cost more in L1/L2 capacity than they save: measured).
#ifndef SART_RAD_GUIDE_BITS
#define SART_RAD_GUIDE_BITS 13
#endif
#ifndef SART_EN_GUIDE_BITS
#define SART_EN_GUIDE_BITS 11
#endif
constexpr int kRadGuideBits = SART_RAD_GUIDE_BITS, kRadGuide = 1 << kRadGuideBits;
constexpr int kEnGuideBits = SART_EN_GUIDE_BITS, kEnGuide = 1 << kEnGuideBits;
// Sampling cells of the single-precision pipeline (fast_params.h: SampleCell): the word's top bits pick a cell that holds
// the answer for every word of the cell up to its first threshold; only a ray at or past the first threshold of a cell
// with two or more thresholds searches (thr_search_tail). A cell covers 2^-bits of the probability, so the share of such
// rays is below the share of such cells: 0.7 % (radius) and 0.9 % (energy) at 13 bits on the bench tables — per warp that
// is one slow path in five launches of the search, which is what the size buys (measured on CAST+LLNL, 1e9 rays:
// 12/11 bits 27.4 ms, 13/12 bits 26.4 ms, 13/13 bits 26.0 ms; the guide + 8 prefetched thresholds before: 28.2 ms).
// Radius cells live in shared memory (64 KiB), energy cells in global memory (64 KiB per emission shell, 129 MB for
// 1968 shells; a ray reads one 8-byte cell of it).
#ifndef SART_RAD_CELL_BITS
#define SART_RAD_CELL_BITS 13
#endif
#ifndef SART_EN_CELL_BITS
#define SART_EN_CELL_BITS 13
#endif
constexpr int kRadCellBits = SART_RAD_CELL_BITS, kRadCells = 1 << kRadCellBits;
constexpr int kEnCellBits = SART_EN_CELL_BITS, kEnCells = 1 << kEnCellBits;
// Entries per row of a u32 threshold table: the row rounded up to 4 entries plus 8 saturated pad entries, so that two
// 16-byte loads from any 4-aligned start inside the row stay inside the row's storage.
#if defined(__CUDACC__)
__host__ __device__
#endif
inline int thr_pitch(int n) { return ((n + 3) & ~3) + 8; }

}  // namespace sart
