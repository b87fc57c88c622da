// fast_params.h — POD blocks of the "fast" pipeline (kernels_fast.cu), filled on the host by derive_fast.cpp.
#pragma once
#include <cstdint>

#include <vector_types.h>

#include "device_params.h"

namespace sart {
namespace fast {

// Shell record in shared memory (built from ShellF64 on the host, see derive_fast_shells).
struct ShellFast {
  double R1, R1pT, r1sq;
  double tan1, zmax1, cosb, sinb;
  double r4, tan2, dm, zmax2, cos3b, sin3b;
  double ddWin, distDet;
  // Wolter-I
  double p_e, p_c0, p_r3sq, p_r3tan;                       // paraboloid: rho^2 = r3^2 + e (l - z); c0 = r3^2 + e l
  double h_e, h_g, h_r3sq, h_r3tan, h_inv_nden;            // hyperboloid: rho^2 = r3^2 + e (l-z) + g (l-z)^2
  int32_t coat;   // reflectivity table of this shell: layers.lowerBound(hitLayer) (rt:1573) in bits 0..7; bit 8: the
                  // lower bound ran past the last coating (the reference would raise; the exact pipeline clamps and flags)
  int32_t pad_;
};
constexpr int kCoatMask = 0xff, kCoatClamped = 0x100;
static_assert(sizeof(ShellFast) % 16 == 8, "odd number of doubles keeps shared-memory rows off the same banks");

struct FastParams {
  // geometry (FP64)
  double radiusCB2, lengthB, dzExitCB, dzPipe1, dzPipe2, rPipe12;  // dz* = plane z - lengthB
  double cosTX, sinTX, cosTY, sinTY, halfLenTel, oeX, oeY, zExitCBtel;  // zExitCBtel = zExitCB - zPipe2
  double lMirror, cosPipe, sinPipe, dShift, lateralShift, transversalShift;
  double radiusWindow2, chipCX, chipCY, cosTheta, sinTheta, stripDist, stripWidth, invStripPitch, invBinX, invBinY;
  double sunDist, radiusSun, radiusCB;
  double shellRhoMin, shellInvStep;   // uniform radial grid -> first candidate shell (shellGuide)
  double depthOverCos;                // depthDet / cos(pipesTurned): distance of the second detector plane (deviationDet rt:2081-2085)
  // weights (FP32)
  float convK;         // (g*1e-9 * B*T2eV2 * 1e-3*m2eV / 2)^2: conversionProb = convK * pathCB^2 (rt:363-365)
  float exposure;
  float angleMin, angleMax, invReflDx;
  // gas stage (FP64 constants of axionMassforMagnet.nim)
  double gasGamma0, gasMgamma2, gasTerm1, gasRhoPipe100, gasRhoMagnet100;
  // X-ray source
  double srcX, srcY, srcZ, srcRadius, colDz, srcRadius2;
  float srcEnergy;
  double enE0, enInvStep;   // uniform-grid guess of an energy's index in the tabulated energies (pre-sampled rays)
  int32_t telKind, nShells, reflKind, nCoatings, stage, nStripHalf, testXray, parallelSource;
  int32_t layers[SART_MAX_COATINGS];
  uint32_t flags;
  int32_t nRadii, nEnergies, nAngles, nReflEnergies, shellsMonotonic, srcEIdx;
  int32_t nShellGuide, rotated;
  int32_t pipesFree, padP_;   // solar Monte Carlo rays cannot reach the pipe walls (kernels_f32.cu, stage A)
  // XMM's central blocker with holes (rt:1674-1688): hole shape, number of holes and half size [mm]
  int32_t holeType, numberOfHoles;
  double holeInOptics;
};

// ---- single-precision pipeline (kernels_f32.cu): the same blocks rounded to FP32, plus a few derived values that
// keep its arithmetic free of cancellation (radii instead of squared radii: C = (rho - R)(rho + R))
struct ShellF32 {
  float R1, R1pT, tan1, zmax1, cosb, sinb;
  float r4, tan2, dm, zmax2, cos3b, sin3b;
  float ddWin;
  float p_e, p_R0, p_r3sq, p_r3tan;                        // p_R0 = sqrt(r3^2 + e l): paraboloid radius at z = 0
  float h_e, h_g, h_r3sq, h_r3tan, h_inv_nden;
  int32_t coat;
  // the z intervals of the two mirrors as centre and half length ("hit" is |z - mid| < half, its margin ||z - mid| - half|),
  // and two per-shell factors of the error budgets (kernels_f32.cu)
  float zmid1, zhalf1, zmid2, zhalf2;
  float twoR;     // 2 R of mirror 1 at z = 0 (R1, or p_R0 for a paraboloid): budget of C = twoR * budget of rho
  float tan2p;    // tan(3 beta) + 0.01: how fast the gap between the ray and mirror 2 changes along z
};
static_assert(sizeof(ShellF32) == 116, "29 words: an odd stride keeps shared-memory rows off the same banks");

// ---- error budgets of the FP32 decisions (derive_fast.cpp: derive_tolerances; DESIGN.md section 3b). Every hit/miss
// decision of the FP32 pipeline has a margin (rho^2 - R^2, the discriminant, z - z_end, ...). A margin inside the budget
// of what FP32 rounding, the fast sampling arithmetic and the reference's own f64 rounding noise can move makes the ray
// "uncertain": it is handed to the exact FP64 pipeline (trace_exact.cuh) through the re-trace queue, so that the
// classification of every ray is the exact pipeline's. All budgets carry the handle's retrace scale (sart_set_retrace;
// 0 = pure FP32).
// Field order of Tol32 and Geo32: the order in which the plain fused kernel uses them, in 16-byte groups — constants come
// from the kernel's parameter bank one LDC / LDCU per use, and neighbours that are used together load as one.
struct alignas(16) Tol32 {
  // lateral position budget before the mirrors [mm], Monte Carlo rays: latA + latS rs + latT (|sx| + |sy|)   (rs = emission
  // radius / solar radius), and the same at the detector plane (det*); lat / det neighbours load as one 64-bit constant
  // and go through one packed multiply-add (trace_f32.cuh: ray_budget2)
  float latS, detS, latT, detT;
  float latA, detA;
  float twoRcb;                      // 2 R of the squared-radius compares (bore; pipes and window below)
  float circCB;                      // circ2 R^2 for the bore: |rho^2 - R^2| < 2 R lat + circ2 R^2
  float entK;                        // budget of the bore entrance test (z = 0, intersected separately by the reference) / budget of the other planes
  float rho;                         // + rounding of a radial distance at the telescope entrance
  float discRel;                     // a negative discriminant above -discRel hb^2 may be a rounding artefact
  float zrel;                        // relative rounding of a root
  float nick;                        // rounding part of the nickel test's budget: sinA lMirror + zrel (largest shell gap)
  float angLo;                       // angleMax - ang: grazing angles from here on touch the end of the reflectivity grid
  float twoRwin, circWin;            // detector window aperture
  int32_t chipInside;                // the chip edge can cut inside the window aperture (else the aperture decides alone)
  float twoRpipe, circPipe;          // pipes
  float circ2;
  float latTpre, detTpre;            // pre-sampled rays: latA + latTpre (|sx| + |sy|) + latRef epsO, epsO = the rounding
                                     //   noise of the reference's line through the caller's origin (kernels_f32.cu)
  float latRef, detRef;
  float spider;                      // rounding of the Chebyshev spider polynomial (in units of cos(n phi))
  float cond;                        // the reference's quadratic formula loses hb^2 / |A C| digits (rt:646-658): dz |q| += cond hb^2 / |A|
  float ang;                         // grazing angle against the end of the reflectivity grid [deg]
  float sinA;                        // absolute rounding of sin(alpha)
};

struct alignas(16) Geo32 {
  float radiusSun, lengthBplusSun, radiusCB, radiusCB2;
  float lengthB, dzExitCB, lengthB2, dzPipe2;
  float oeX, oeY, shellRhoMin, shellInvStep;
  float lMirror, zExitCBtel, cosPipe, sinPipe;
  float dShift, depthOverCos, lateralShift, transversalShift;   // depthOverCos = ddEnd - ddWin = depthDet / cos(pipesTurned): the second detector plane of deviationDet (rt:2081-2085)
  float chipCX, chipCY, radiusWindow2, cosTheta;   // (chipCX, chipCY), (invBinX, invBinY), (oeX, oeY), (lateralShift,
  float sinTheta, stripDist, stripWidth, invStripPitch;   //  transversalShift): 8-byte aligned pairs for the packed x / y arithmetic
  float invBinX, invBinY, dzPipe1, rPipe12;
  float cosTX, sinTX, cosTY, sinTY, halfLenTel;
  float srcX, srcY, srcRadius, srcRadius2, invSrcDz, colDz;
  float holeR;   // holeInOptics
  Tol32 tol;
};

// Re-trace queue of a launch: offsets (ray index - first ray of the launch) of the uncertain rays. count[0] counts the
// pushes (it may run past cap: the pushes beyond cap are refused and the ray keeps its FP32 outcome, counted in
// sart_counters_t::n_unresolved).
struct RetraceQueue {
  uint32_t* list;
  uint32_t* count;
  uint32_t cap, pad;
};
// Rays per launch of the FP32 kernels: queue entries (ray index - first ray of the launch) and the fused kernel's per-thread
// trip count are 32-bit. api.cu cuts longer runs into launches of at most this many rays.
constexpr uint64_t kMaxRaysPerLaunch = uint64_t(1) << 31;

// Radial lookup of the shell search (rt:1932-1957) for the FP32 kernels: the radial buckets of the shell guide are fine
// enough to hold at most one boundary (a shell's front radius R1 or the outer edge R1 + thickness of its glass) each,
// so one 8-byte record decides the outcome: sel holds the outcome below / at / above the boundary B, one byte each
// (bits 0-7, 8-15, 16-23): a shell number < 64, or 64 + exit code.
struct ShellCell {
  float B;
  uint32_t sel;
};
constexpr int kShellCellFail = 64;

struct EnergyLUT {  // one record per tabulated energy index (16 B, one LDG.128)
  // strongback transmission = Tstrongback * 2^sbExp: 200 um of silicon transmit 1e-60 at 0.9 keV, far below the FP32
  // range, and a weight must keep its value there, not only its non-zeroness. The exponent is the low 16 bits of sbExp
  // (signed; 0 wherever FP32 holds the value); bits 16.. say which interpolations of the exact pipeline clamp at this
  // energy (kLutClamp*: SART_FLAG_INTERP_CLAMPED of the rays that evaluate them). sbExp == 0 for an ordinary energy.
  int32_t sbExp;
  float Twindow, Tstrongback, Agas;
};
constexpr int kLutClampWindow = 1, kLutClampStrongback = 2, kLutClampGas = 4, kLutClampRefl = 8;
struct GasLUT {     // buffer-gas stage only
  float massAtt;   // exp(logMassAttenuation(E)) am:70-73
  float inv2E;     // 1 / (2 E[eV])
};

// One cell of a sampling table (mode 2): the words w with w >> (32 - bits) == k. base = number of thresholds below the
// cell (the answer for words below the cell's first threshold thr0; 0xffffffff when the cell holds none), n = number of
// thresholds inside it. Answer = base + (w >= thr0) when n < 2; otherwise the thresholds base + 1 .. base + n - 1 are
// searched (thr_search_tail). The last cell is given n >= 2 when it holds a saturated threshold, so that the all-ones word
// always reaches the slow path and its f64 fallback. Indices are 16-bit (sart_create checks nRadii, nEnergies < 65536).
struct alignas(8) SampleCell { uint32_t thr0; uint32_t baseN; };   // baseN = base | min(n, 0xffff) << 16

struct FastTables {
  // Inverse-CDF sampling (rt:437, 464) in integers: with u = (w + 0.5) 2^-32, cdf[i] < u  <=>  w >= thr[i], where
  // thr[i] is the smallest such 32-bit word (saturated at 0xffffffff; that word falls back to the f64 tables).
  const double* radiusCDF;       // [nRadii] f64, fallback only
  const uint32_t* radiusThr;     // [thr_pitch(nRadii)]
  const uint16_t* radiusGuide;   // [kRadGuide] g[k] = lowerBound(cdf, k/kRadGuide): the search for a word of bucket k starts there
  const double* energyCDF;       // [nRadii][nEnergies] f64, fallback only
  const uint32_t* energyThr;     // [nRadii][thr_pitch(nEnergies)]
  const uint16_t* energyGuide;   // [nRadii][kEnGuide]
  const SampleCell* radiusCells; // [kRadCells]          (mode 2; modes 0 / 1 use the guides above)
  const SampleCell* energyCells; // [nRadii][kEnCells]
  const double* energies;        // [nEnergies] keV (pre-sampled rays: energy -> index)
  const EnergyLUT* elut;         // [nEnergies + 1]
  const GasLUT* glut;            // [nEnergies + 1]
  // reflectivity pre-interpolated along the energy axis at every tabulated energy: [coat][nEnergies + 1][nAngles];
  // the per-ray lookup is then linear in the grazing angle only (same value as the bilinear form of rt:1567-1578)
  const float* reflE;
  // rkEffectiveArea (rt:1553-1562): the telescope transmission at every tabulated energy, [nEnergies + 1]; the ray's
  // "reflectivity" is this value times two polynomials in its pitch and yaw angles
  const float* telTrans;
  const ShellFast* shells;    // [nShells]
  const ShellF32* shells32;   // [nShells] the same records in single precision (kernels_f32.cu)
  const uint8_t* shellGuide;  // [nShellGuide]: smallest j with R1[j] > lower edge of the radial bucket
  const ShellCell* shellTab;  // [nShellGuide] (kernels_f32.cu)
  // Alias tables (sart_set_sampler(SART_SAMPLER_ALIAS), kernels_f32.cu): the same discrete distributions as the
  // thresholds above — P(i) = (thr[i] - thr[i-1]) 2^-32 — as Walker/Vose tables, one 32-bit entry per index:
  // bits 31..11 = the bucket's own share in units of 2^-21, bits 10..0 = the alias index. A word w selects bucket
  // k = (w n) >> 32 and keeps it when the low 32 bits of w n are below the share, else takes the alias: one lookup, no
  // search. Needs n <= 2048; null when unavailable.
  const uint32_t* radiusAlias;   // [nRadii]
  const uint32_t* energyAlias;   // [nRadii][nEnergies]
  int32_t sampler, pad2_;        // SART_SAMPLER_* for this launch
  RadialHist rad;             // optional (w == nullptr: off)
  // Image replicas: block b adds into replica b % nImgRep of the image / w^2 image it is handed (replica r starts
  // imgRepStride doubles after replica 0); 0 or 1 = the image itself. The focal spot concentrates ~1e9 atomic adds per
  // launch on a few hundred bins; spreading them over replicas removes the same-address serialisation in L2.
  int32_t nImgRep, pad_;
  uint64_t imgRepStride;
  RetraceQueue rq;            // cap == 0: re-tracing off
  // optional spectra of the passed rays (device_params.h: Spectra; the generic kernel variants only). Last member, so that
  // the plain-run kernels, which compile them out, read every other field at the offset they always had.
  Spectra spec;
};

}  // namespace fast
}  // namespace sart
