/* sart.h — C-ABI boundary of the B200-native solar-axion ray tracer.
 *
 * This header is the drop-in seam for ONE path of jovoy/SolarAxionRayTracing:
 * the per-ray pipeline `traceAxion` (src/raytracer.nim:1736-2221) as driven by
 * `traceAxionWrapper` (src/raytracer.nim:2223-2244) from
 * `calculateFluxFractions` (src/raytracer.nim:2755-2776), plus the weighted
 * detector histogram `prepareHeatmap` (src/raytracer.nim:818-842) that
 * consumes its output and the CDF build in `initFullSetup`
 * (src/raytracer.nim:2679-2705) that feeds it.
 *
 * The reference has no FFI for this path; each entry point below names the
 * Nim proc (file:line) whose role it takes. INTEGRATION.md shows the Nim
 * `{.importc, dynlib.}` stubs a maintainer would add.
 *
 * Conventions: plain C, no exceptions cross the boundary, every function
 * returns 0 on success and a negative sart_status on failure; the message is
 * available from sart_last_error() (thread-local). A handle owns one CUDA
 * device and one stream and is not thread-safe. All host pointers are owned by
 * the caller; tables and setup are copied at sart_create(). There is NO CPU
 * fallback: without a CUDA device sart_create() fails with SART_ERR_CUDA.
 */
#ifndef SART_H
#define SART_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SART_ABI_VERSION 2
#define SART_MAX_SHELLS 64   /* XMM has 58 shells (raytracer.nim:1289-1313) */
#define SART_MAX_COATINGS 8  /* LLNL has 4 coating recipes (raytracer.nim:1167) */
#define SART_IMAGE_BINS 256  /* prepareHeatmap(256, 256, ...) raytracer.nim:2629 */
#define SART_MAX_MASSES 64   /* axion masses traced per launch in a mass scan */

typedef enum {
  SART_OK = 0,
  SART_ERR_ARG = -1,     /* bad argument */
  SART_ERR_CUDA = -2,    /* CUDA runtime error / no device */
  SART_ERR_CONFIG = -3,  /* unsupported setup combination (reference: doAssert false) */
  SART_ERR_NOMEM = -4
} sart_status;

/* ---- enums mirroring the reference's (raytracer.nim:16-46, 59-64, 164-167, 223-230) ---- */
typedef enum { SART_ES_CAST = 0, SART_ES_BABYIAXO = 1 } sart_experiment_kind;
typedef enum { SART_TK_LLNL = 0, SART_TK_XMM = 1, SART_TK_CUSTOM_BABYIAXO = 2,
               SART_TK_ABRIXAS = 3, SART_TK_OTHER = 4 } sart_telescope_kind;
typedef enum { SART_SK_VACUUM = 0, SART_SK_GAS = 1 } sart_stage_kind;
typedef enum { SART_DK_INGRID2017 = 0, SART_DK_INGRID2018 = 1, SART_DK_INGRIDIAXO = 2 } sart_detector_kind;
typedef enum { SART_WY_2017 = 0, SART_WY_2018 = 1, SART_WY_IAXO = 2 } sart_window_year;
typedef enum { SART_HT_NONE = 0, SART_HT_CROSS = 1, SART_HT_STAR = 2, SART_HT_CIRCLE = 3,
               SART_HT_SQUARE = 4, SART_HT_DIAMOND = 5 } sart_hole_type;
typedef enum { SART_RK_EFFECTIVE_AREA = 0, SART_RK_SINGLE_COATING = 1,
               SART_RK_MULTI_COATING = 2 } sart_reflectivity_kind;

/* ConfigFlags (raytracer.nim:223-230) as a bit set: bit = ordinal of the Nim enum. */
enum {
  SART_CF_IGNORE_DET_WINDOW = 1u << 0,
  SART_CF_IGNORE_GAS_ABS = 1u << 1,
  SART_CF_IGNORE_REFLECTION = 1u << 2,
  SART_CF_IGNORE_CONV_PROB = 1u << 3,
  SART_CF_XRAY_TEST = 1u << 4,
  SART_CF_READ_MAGNET_CONFIG = 1u << 5,
  SART_CF_READ_DET_INSTALL_CONFIG = 1u << 6
};

/* Where a ray left traceAxion (one value per early `return` of raytracer.nim:1736-2221). */
typedef enum {
  SART_EXIT_PASSED = 0,         /* reached the end, weight != 0        rt:2220 */
  SART_EXIT_MISSED_BORE = 1,    /* no entrance disc, no single wall hit rt:1825 */
  SART_EXIT_CLIP_EXIT_CB = 2,   /* rt:1846-1848 */
  SART_EXIT_CLIP_PIPE_VT3 = 3,  /* rt:1856-1858 */
  SART_EXIT_CLIP_PIPE_XRT = 4,  /* rt:1866-1868 */
  SART_EXIT_OPAQUE = 5,         /* spider / blocker                      rt:1910-1914 */
  SART_EXIT_OUTSIDE_SHELLS = 6, /* rt:1934 */
  SART_EXIT_GLASS_FRONT = 7,    /* rt:1942-1944 */
  SART_EXIT_NICKEL = 8,         /* rt:2040-2046 */
  SART_EXIT_NO_MIRROR_HIT = 9,  /* almostEqual test                      rt:2051-2057 */
  SART_EXIT_WINDOW_APERTURE = 10, /* rt:2139-2147 */
  SART_EXIT_ZERO_WEIGHT = 11,   /* reached the end with weight == 0      rt:2220 */
  SART_EXIT_COLLIMATOR = 12,    /* X-ray test source only                rt:1800-1801 */
  SART_N_EXIT_CODES = 13
} sart_exit_code;
/* `code` words carry the exit code in bits 0..7 and these flags above it. */
#define SART_CODE_MASK 0xff
#define SART_FLAG_PASSED_TILL_WINDOW 0x100 /* Axion.passedTillWindow rt:2135-2136 */
#define SART_FLAG_INTERP_CLAMPED 0x200     /* an interpolation argument left its grid; the reference would raise */

/* ---- setup: the read-only parameters of FullRaytraceSetup (raytracer.nim:232-242) as one POD ---- */
typedef struct {
  double lengthColdbore, B, lengthB, radiusCB, pGasRoom, tGas; /* Magnet rt:83-89 (mm, T, mm, mm, bar, K) */
} sart_magnet_t;

typedef struct {
  double cb2vt3_length, cb2vt3_radius;   /* Pipes.coldBoreToVT3 rt:125-140 */
  double vt3xrt_length, vt3xrt_radius;   /* Pipes.vt3ToXRT */
  double distanceCBAxisXRTAxis;
  double pipesTurned;                    /* degree */
} sart_pipes_t;

typedef struct {
  int32_t kind;                 /* sart_telescope_kind */
  int32_t nShells;
  int32_t numberOfHoles;
  int32_t holeType;             /* sart_hole_type */
  int32_t reflKind;             /* sart_reflectivity_kind */
  int32_t nCoatings;
  int32_t layers[SART_MAX_COATINGS]; /* Reflectivity.layers rt:78 */
  double optics_entrance[3], optics_exit[3];
  double telescope_turned_x, telescope_turned_y; /* degree */
  double lMirror, holeInOptics;
  double allThickness[SART_MAX_SHELLS];
  double allR1[SART_MAX_SHELLS];
  double allXsep[SART_MAX_SHELLS];
  double allAngles[SART_MAX_SHELLS];  /* degree */
} sart_telescope_t;               /* Telescope rt:91-105 */

typedef struct {
  int32_t active, parallel;
  double energy, distance, radius, offAxisUp, offAxisLeft, activity, lengthCol;
} sart_test_source_t;             /* TestXraySource rt:108-122 */

typedef struct {
  double distanceDetectorXRT, distanceWindowFocalPlane, lateralShift, transversalShift;
} sart_detector_install_t;        /* DetectorInstallation rt:146-153 */

typedef struct {
  int32_t windowYear;             /* sart_window_year */
  int32_t numberOfStrips;
  double stripDistWindow, stripWidthWindow, detectorWindowAperture;
  double theta;                   /* rad */
  double radiusWindow, openApertureRatio, windowThickness, alThickness, depthDet;
} sart_detector_t;                /* DetectorSetup rt:170-184 (interpolators live in sart_tables_t) */

typedef struct {
  double radiusSun, distanceSunEarth; /* rt:249-250 */
  double roomTemp, mAxion, g_agamma;  /* rt:254-256 (K, eV, GeV^-1) */
  double chipXMax, chipYMax;          /* rt:260-266 */
  double tesla_to_eV2;                /* unchained toNaturalUnit(T)      */
  double m_to_inv_eV;                 /* unchained toNaturalUnit(m)      */
  double exposureFactor;              /* rt:2207-2212 (1.0 with cfXrayTest) */
} sart_consts_t;

typedef struct {
  uint32_t abi_version;           /* SART_ABI_VERSION */
  uint32_t flags;                 /* SART_CF_* bit set */
  int32_t experiment;             /* sart_experiment_kind */
  int32_t stage;                  /* sart_stage_kind */
  int32_t detectorKind;           /* sart_detector_kind */
  int32_t reserved0;
  sart_magnet_t magnet;
  sart_pipes_t pipes;
  sart_telescope_t telescope;
  sart_test_source_t testSource;
  sart_detector_install_t detectorInstall;
  sart_detector_t detector;
  sart_consts_t consts;
} sart_setup_t;                   /* ExperimentSetup rt:155-162 + DetectorSetup + globals */

/* 1-D linear interpolator on a sorted irregular grid (numericalnim newLinear1D; rt:1522-1527). */
typedef struct { int32_t n; int32_t reserved; const double* x; const double* y; } sart_interp1d_t;

/* ---- tables: everything the reference loads from resources/ for the path ---- */
typedef struct {
  /* solar model, after the CDF build of rt:2679-2705 */
  int32_t nRadii, nEnergies;
  const double* energies;        /* [nEnergies] keV, ascending                       rt:2657-2662 */
  const double* fluxRadiusCDF;   /* [nRadii]                                         rt:2705 */
  const double* diffFluxCDFs;    /* [nRadii][nEnergies] row-major                    rt:2704 */
  /* reflectivity (angle-major: refl[c][iAngle][iEnergy])                            rt:1174-1208 */
  int32_t nCoatings, nAngles, nReflEnergies, reserved;
  double angleMin, angleMax;     /* degree */
  double reflEnergyMin, reflEnergyMax; /* keV */
  const double* reflectivity;    /* [nCoatings][nAngles][nReflEnergies] */
  /* detector chain (keV grids)                                                      rt:1499-1527 */
  sart_interp1d_t strongbackTransmission, windowTransmission, gasAbsorption;
  sart_interp1d_t telescopeTransmission; /* only rkEffectiveArea (rt:1245-1249); n = 0 otherwise */
} sart_tables_t;

/* ---- per-ray outputs (structure of arrays; the Axion record rt:192-221 transposed) ---- */
typedef struct {
  /* required */
  double* x;        /* pointdataX  (chip frame, mm)  rt:2214 */
  double* y;        /* pointdataY                    rt:2215 */
  double* w;        /* weights                       rt:2216 */
  int32_t* code;    /* sart_exit_code | SART_FLAG_*  */
  int32_t* shell;   /* shellNumber                   rt:2198 (-1 if never assigned) */
  /* optional: NULL to skip */
  double* energy;        /* energiesPre / energiesAx   rt:1819, 2197 */
  double* reflect;       /* rt:2126 */
  double* transMagnet;   /* transmissionMagnet rt:2120 */
  double* yaw;           /* yawAngles rt:2123 */
  double* alpha1;        /* grazing angle on mirror 1, degree */
  double* alpha2;
  double* pathCB;        /* rt:1843 */
  double* r;             /* pointdataR rt:2202 */
  double* deviationDet;  /* rt:2085 */
  double* transProbArgon;/* rt:2193 */
} sart_ray_out_t;

/* Whole-run counters: the stdout counters of generateResultPlots (rt:2253-2257, 2276-2278, 886). */
typedef struct {
  uint64_t n_rays;
  uint64_t n_exit[16];           /* histogram over sart_exit_code */
  uint64_t n_passed;             /* Axion.passed */
  uint64_t n_passed_till_window; /* Axion.passedTillWindow */
  uint64_t n_hit_nickel;         /* Axion.hitNickel */
  uint64_t n_interp_clamped;     /* rays where an interpolation argument was clamped */
  uint64_t n_retraced;           /* precision mode 2: rays whose FP32 decision margins were inside the error budget and
                                    that were therefore traced by the exact FP64 pipeline instead (sart_set_retrace) */
  uint64_t n_unresolved;         /* such rays that did not fit the re-trace queue and kept their FP32 outcome (0 in
                                    practice: the queue holds 6 % of a launch) */
  double sum_w;                  /* Σ weights | passed  (performAngularScan rt:2800; "total flux" rt:885) */
  double sum_w2;
  double sum_x, sum_y, sum_r;    /* unweighted sums over passed rays (means of rt:2276-2278) */
} sart_counters_t;

typedef struct sart_handle sart_handle_t;

/* ---- library ---- */
const char* sart_last_error(void);
int sart_abi_version(void);
size_t sart_sizeof_setup(void);
size_t sart_sizeof_tables(void);
size_t sart_sizeof_counters(void);
int sart_device_count(void);

/* ---- host-side setup constructors (C++; replace newExperimentSetup rt:1411-1423, newDetectorSetup
 * rt:1464-1528 minus file I/O, calcWindowVals rt:1431-1462 and the globals rt:248-272). Same defaults as
 * the reference for every (experiment, detector, stage, telescope) it implements; SART_ERR_CONFIG where the
 * reference does `doAssert false` (tkOther, tkCustomBabyIAXO). */
int sart_init_setup(int experiment, int detectorKind, int stage, int telescope, uint32_t flags,
                    sart_setup_t* out);
int sart_calc_window_vals(double radiusWindow, int numberOfStrips, double openApertureRatio,
                          double* width, double* dist);

/* ---- handle ---- */
/* Copies setup + tables to `device` (HBM), derives the per-shell constant blocks. */
int sart_create(const sart_setup_t* setup, const sart_tables_t* tables, int device, sart_handle_t** out);
void sart_destroy(sart_handle_t* h);
/* Replace the setup of a live handle (tables stay resident): performAngularScan mutates
 * telescope_turned_y between runs (rt:2794-2798). */
int sart_update_setup(sart_handle_t* h, const sart_setup_t* setup);
/* Axion masses for the buffer-gas scan; default is the single value setup.consts.mAxion (rt:255). */
int sart_set_axion_masses(sart_handle_t* h, int n, const double* masses_eV);
/* 0 = "exact": FP64, the reference's operation order (bit-faithful hit/miss classification);
 * 1 = "fast": FP64 algebra on (point, slopes) + FP32 weights (closer to exact arithmetic than the reference itself);
 * 2 = "f32": the same formulation with FP32 geometry (positions to ~1e-4 mm, the reference's own rounding level).
 * Every reflectivity kind (rt:1533-1580, rkEffectiveArea included) and XMM hole type (rt:1674-1688) runs in all three modes;
 * modes 1 and 2 return SART_ERR_CONFIG for shells that overlap / are not in ascending order and for more than 64 holes. */
int sart_set_precision(sart_handle_t* h, int mode);
/* Precision modes 1 and 2 only: 1 = compact the rays that survive bore, pipes, vetoes and glass fronts into full warps before the
 * mirror stage (pays off when most rays are clipped, e.g. BabyIAXO + XMM); 0 = one ray per lane throughout. Results are
 * identical ray by ray. Default: chosen at sart_create from the setup (on for XMM/Abrixas, off for LLNL). */
int sart_set_compaction(sart_handle_t* h, int mode);
int sart_has_precision(int mode); /* 1 if this build has the pipeline for `mode` */
/* Precision mode 2 only. Every hit/miss decision of the FP32 pipeline (rho < R at the bore exit and the pipes rt:481-492,
 * the spider and the shell boundaries rt:1635-1704, 1932-1944, the mirror roots rt:646-658, the nickel test rt:1706-1734,
 * the window aperture and the strongback strips rt:2139-2185) has a margin; a ray with a margin inside the error budget of
 * that decision — FP32 rounding, the fast sampling arithmetic, and the reference's own f64 rounding noise — is "uncertain".
 * mode 1 (default): uncertain rays are traced by the exact FP64 pipeline instead, right after the FP32 kernel on the same
 * stream, so every ray has the exit code of precision mode 0 (counted in sart_counters_t::n_retraced; ~1e-4 .. 3e-3 of the
 * rays). mode 0: pure FP32 (about 1e-5 of the rays then differ in their exit code). `scale` multiplies every budget
 * (1 = the derived budgets; tests use it to show the safety factor they carry). Not applied with SART_SAMPLER_ALIAS. */
int sart_set_retrace(sart_handle_t* h, int mode, double scale);
void* sart_stream(sart_handle_t* h); /* cudaStream_t the handle launches on */

/* ---- CDF build on the device (replaces rt:2679-2705). emRates is [nRadii][nEnergies] row-major,
 * radii are fractions of the solar radius. Outputs are host arrays. Sequential per-row sums in the
 * reference's order, so the result is bit-identical to a scalar loop. */
int sart_build_cdfs(int device, int nRadii, int nEnergies, const double* radii, const double* energies,
                    const double* emRates, double* fluxRadiusCDF, double* diffFluxCDFs);

/* ---- emission-rate table of the solar model (src/readOpacityFile.nim `calculateOpacities` :598-860, the
 * opacity-free processes): emRates[nRadii][nEnergies] row-major, ready for sart_build_cdfs. temp_K, rho_gcm3 [nRadii]
 * and massFractions [nRadii][29] are the AGSS09 columns Temp, Rho and H1..Ni in file order (readSolarModel.nim:3-7);
 * radius i is 0.0015 + 0.0005 i solar radii (:793). `processes` is a SART_EM_* bit set; couplings as in the reference
 * (g_ae = 1e-13, gagamma = 1e-12, ganuclei = 1e-15 at :641-645). FB/BB (term1 :369-371) and the transverse plasmon
 * (:439-452) need the un-shipped OPCD opacities and are not produced. */
enum {
  SART_EM_PRIMAKOFF = 1u << 0,    /* primakoff      readOpacityFile.nim:384-413 */
  SART_EM_COMPTON = 1u << 1,      /* comptonEmrate  :360-362 */
  SART_EM_EE_BREMS = 1u << 2,     /* bremsEmrate    :364-367 (fNew :312-326) */
  SART_EM_FREE_FREE = 1u << 3,    /* freefreeEmrate :378-381 */
  SART_EM_IRON57 = 1u << 4,       /* iron           :454-466 */
  SART_EM_LONG_PLASMON = 1u << 5  /* longPlasmon    :421-437 in the limit of zero opacity */
};
int sart_emission_rates(int device, int nRadii, const double* temp_K, const double* rho_gcm3,
                        const double* massFractions, int nEnergies, const double* energies_keV, uint32_t processes,
                        double g_ae, double gagamma, double ganuclei, double* emRates);

/* ---- tier (a): trace pre-sampled rays. Replaces the body of traceAxion after the sampling block
 * (rt:1811-2221). origin_xyz = SoA [3][n] (rayOrigin), exit_xy = SoA [2][n] (pointExitCBMagneticField x,y;
 * z = lengthB), energy_keV [n]. Host buffers; copies are inside the call. Precision 0 and 1 run the exact FP64 pipeline
 * (every output array), precision 2 the FP32 pipeline (x, y, w, code, shell, energy, r; other optional arrays zeroed;
 * the energy must be one of the tabulated energies as in the reference, rt:470 — otherwise the nearest one is traced
 * and the ray is flagged SART_FLAG_INTERP_CLAMPED). */
int sart_trace_presampled(sart_handle_t* h, size_t n, const double* origin_xyz, const double* exit_xy,
                          const double* energy_keV, const sart_ray_out_t* out);
/* Same with DEVICE pointers (inputs resident in HBM, outputs left in HBM); asynchronous on sart_stream(). */
int sart_trace_presampled_dev(sart_handle_t* h, size_t n, const double* d_origin_xyz, const double* d_exit_xy,
                              const double* d_energy_keV, const sart_ray_out_t* d_out);

/* ---- the literal traceAxionWrapper drop-in (rt:2223-2244): Monte Carlo sampling (rt:1754-1764) from the
 * counter-based generator Philox4x32-10 (key = seed, counter = global ray index) + trace; per-ray records
 * out. Host buffers. Ray i of the call is global ray first_ray + i, so any split of a run over calls,
 * streams or GPUs traces the same rays. */
int sart_trace_mc_rays(sart_handle_t* h, uint64_t first_ray, size_t n, uint64_t seed, const sart_ray_out_t* out);

/* ---- the same drop-in for consumers that only read the rays that PASS (generateResultPlots rt:2246-2289 filters
 * `axions.filterIt(it.passed)` before it touches any field): the records of the passed rays only, compacted on the device
 * and in single precision where the pipeline computes in single precision, so that the clipped rays (14 % CAST+LLNL, 77 %
 * BabyIAXO+XMM) are not shipped over PCIe at all. Order is arbitrary; `ray` tells which ray a record belongs to (ray index
 * - first_ray). Every array is optional (NULL to skip) and must hold `capacity` records; *n_passed returns how many rays
 * passed (SART_ERR_ARG if more than capacity: the first `capacity` records are valid). counters (optional, host): the
 * whole-run counters of these rays, as sart_read_image would return them. Precision mode 2, inverse-CDF sampler, single
 * axion mass; uncertain rays are re-traced in FP64 like everywhere else (sart_set_retrace). */
typedef struct {
  uint32_t* ray;         /* ray index - first_ray */
  float* x;              /* pointdataX (chip frame, mm) rt:2214 */
  float* y;              /* pointdataY rt:2215 */
  float* w;              /* weights rt:2216 */
  uint8_t* shell;        /* shellNumber rt:2198 */
  float* energy;         /* energiesAx [keV] rt:2197 */
  float* r;              /* pointdataR rt:2202 */
  float* reflect;        /* rt:2126 */
  float* transMagnet;    /* transmissionMagnet rt:2120 */
  float* yaw;            /* yawAngles rt:2123 */
  float* alpha1;         /* grazing angles [deg] */
  float* alpha2;
  float* pathCB;         /* rt:1843 */
  float* deviationDet;   /* rt:2085 */
  float* transProbArgon; /* rt:2193 */
} sart_passed_out_t;
int sart_trace_mc_passed(sart_handle_t* h, uint64_t first_ray, uint64_t n, uint64_t seed, size_t capacity,
                         const sart_passed_out_t* out, uint64_t* n_passed, sart_counters_t* counters);

/* ---- test hook: sart_trace_mc_rays with the six random words of every ray supplied by the caller (SoA [6][n]: phi_sun,
 * theta_sun, radius, disc r, disc phi, energy; uniform = (word + 0.5) 2^-32) instead of drawn from Philox, so that tests
 * can drive the integer inverse-CDF search (rt:437, 464) through its corners — word 0, word 0xffffffff, the words on
 * either side of every CDF entry, flat CDF tails. Precision modes 0 and 2, solar source. late_energy != 0 (mode 2)
 * resolves the energy after the clip stages, the way the compacting fused kernel does; 0 inside them, like the plain one.
 * out->energy is filled for every ray, clipped or not (energiesPre, rt:1818-1819). */
int sart_trace_words(sart_handle_t* h, size_t n, const uint32_t* words, int late_energy, const sart_ray_out_t* out,
                     int32_t* emission_shell /* optional [n]: the radius index rt:437 of every ray */);

/* ---- fused run: sample + trace + prepareHeatmap (rt:818-842, 256x256 over the 14x14 mm chip, norm = 1).
 * Accumulates (+=) into the handle's device-resident image/counters; asynchronous. With M axion masses set
 * (sart_set_axion_masses) the image is [M][256][256]. In precision modes 1 and 2 the kernel adds into internal replicas
 * (single mass) or mass-major accumulators (mass scan) that a small second kernel folds into the image on the same
 * stream right after the trace kernel: when the call returns, everything it did is queued on sart_stream(). */
int sart_trace_mc(sart_handle_t* h, uint64_t first_ray, uint64_t n_rays, uint64_t seed);
int sart_reset_image(sart_handle_t* h);
/* Optional weighted radial histogram of the passed rays, for the 68 % / 95.5 % containment radii of
 * generateResultPlots (rt:2459-2527, which sorts pointdataR of every passed ray): bin = floor(pointdataR * nbins / r_max),
 * the last bin also collects r >= r_max. Filled by sart_trace_mc for a single axion mass, cleared by sart_reset_image.
 * nbins = 0 switches it off (default). sum_w / counts are host arrays [nbins] (either may be NULL). */
int sart_enable_radial_hist(sart_handle_t* h, int nbins, double r_max);
int sart_read_radial_hist(sart_handle_t* h, double* sum_w, uint64_t* counts);
/* Optional weighted spectra of the rays that PASS (weight != 0, rt:2220) in sart_trace_mc, single axion mass — the
 * reductions generateResultPlots (rt:2246-2635) makes over energiesAx, shellNumber and weights, without per-ray records:
 * energy bin i < nEnergies = tabulated energy i (a Monte Carlo ray's energy is a table value, rt:470), bin nEnergies = the
 * X-ray test source's energy; shell bin j = shellNumber (rt:2198). Accumulated (+=) like the image and cleared by
 * sart_reset_image; filled in every precision mode, by the FP32 kernel and by the FP64 re-trace of its uncertain rays
 * alike, so precision 2 has the counts of precision 0. With spectra on, precision modes 1 and 2 run the generic kernel
 * variant (as with the radial histogram) and sart_trace_mc with more than one axion mass fails with SART_ERR_CONFIG.
 * sart_angular_scan, sart_trace_mc_rays, sart_trace_mc_passed, sart_trace_presampled(_dev) and sart_trace_words leave
 * them untouched. on != 0 synchronises, then (re)allocates and zeroes them; on = 0 switches them off (default). */
int sart_enable_spectra(sart_handle_t* h, int on);
/* Synchronises and copies out; host arrays, any may be NULL: energy_* [nEnergies + 1], shell_* [SART_MAX_SHELLS].
 * SART_ERR_ARG when the spectra are off. */
int sart_read_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                      double* shell_sum_w, uint64_t* shell_counts);
/* Device pointers for collectives (ncclAllReduce / torch.distributed on the caller's side). */
double* sart_image_dev(sart_handle_t* h);       /* [M][256][256] Σw  */
double* sart_image_w2_dev(sart_handle_t* h);    /* [M][256][256] Σw² */
void* sart_counters_dev(sart_handle_t* h);      /* sart_counters_t[M] on the device */
size_t sart_image_len(sart_handle_t* h);        /* M*256*256 */
/* ---- multi-GPU: the one collective of the path. Rays shard over GPUs by global ray index with no exchange while tracing;
 * afterwards the images and counters — all additive — are summed over the GPUs by ONE ncclAllReduce(sum, f64) over
 * {image, sum-of-squares image, counters} (the reference has no counterpart: its only parallel construct is the Weave loop
 * of rt:2234-2244 inside one process). The sum lands in a separate "merged" buffer of every handle: the handle's own
 * accumulators are untouched, so steps can go on accumulating and the call can be repeated. NCCL is loaded with dlopen at
 * first use (SART_ERR_CONFIG if libnccl.so.2 is absent).
 *   one process per GPU (MPI / torchrun): rank 0 calls sart_comm_unique_id, ships the 128 bytes to the other ranks by
 *     whatever transport the host has, every rank calls sart_comm_init_rank, then sart_allreduce(&h, 1);
 *   one process, n GPUs: sart_comm_init_all(handles, n) (handles on distinct devices), then sart_allreduce(handles, n).
 * Asynchronous on the handles' streams; sart_read_merged synchronises and copies the merged result out. */
#define SART_COMM_ID_BYTES 128
int sart_comm_unique_id(char id[SART_COMM_ID_BYTES]);
int sart_comm_init_rank(sart_handle_t* h, int n_ranks, int rank, const char id[SART_COMM_ID_BYTES]);
int sart_comm_init_all(sart_handle_t* const* handles, int n);
void sart_comm_destroy(sart_handle_t* h);   /* also done by sart_destroy */
int sart_allreduce(sart_handle_t* const* handles, int n);
int sart_read_merged(sart_handle_t* h, double* image, double* image_w2, sart_counters_t* counters);

/* Synchronise and copy out. image/image_w2 may be NULL. counters is [M]. */
int sart_read_image(sart_handle_t* h, double* image, double* image_w2, sart_counters_t* counters);
int sart_synchronize(sart_handle_t* h);

/* ---- performAngularScan (rt:2778-2815): n_angles runs of n_rays_per_angle rays each, run i with
 * telescope_turned_y = angles_deg[i] (rt:2794-2798) and everything else as in the handle's setup. All runs are
 * queued on the handle's stream without host synchronisation (only the by-value parameter block changes between scan
 * points); scan point i traces the global rays first_ray + [i*n, (i+1)*n), so a scan split over GPUs by blocks of scan
 * points (first_ray = first point * n) traces the same rays as an unsplit one. fluxes[i] = sum of the weights of the passed rays
 * (rt:2800, un-normalised; the reference then divides by the maximum, rt:2801-2802). counters [n_angles] and images
 * [n_angles][256][256] are optional host arrays (NULL to skip). Leaves the handle's own setup and image untouched. */
int sart_angular_scan(sart_handle_t* h, int n_angles, const double* angles_deg, uint64_t first_ray,
                      uint64_t n_rays_per_angle, uint64_t seed, double* fluxes, sart_counters_t* counters, double* images);

/* ---- prepareHeatmap (rt:818-842), general form, for per-ray records held by the host (e.g. the output of
 * sart_trace_mc_rays filtered by `passed`): result[floor((y-start_y)/dy)][floor((x-start_x)/dx)] += w/norm on the
 * GPU. result is a host array [numberOfRows*numberOfColumns], overwritten. Points outside the grid are counted in
 * *n_out_of_range (may be NULL) instead of raising IndexDefect like the reference. */
int sart_prepare_heatmap(sart_handle_t* h, int numberOfRows, int numberOfColumns, double start_x, double stop_x,
                         double start_y, double stop_y, size_t n, const double* data_X, const double* data_Y,
                         const double* weight1, double norm, double* result, uint64_t* n_out_of_range);

/* ---- measurement helper: dense FMA issue rate of the CUDA cores (fp64 != 0: DFMA, else FFMA) in TFLOP/s, best of a
 * few launches. bench.py uses it as the roofline denominator of the compute-bound trace kernels. */
int sart_measure_fma_peak(int device, int fp64, double* tflops);

/* ---- Philox helper exported for tests: the 6 uniforms of global ray `ray` in the order the reference
 * draws them (rt:433-436, 418-419, 464): phi_sun, theta_sun, u_radius, u_disk_r, u_disk_phi, u_energy. */
void sart_ray_uniforms(uint64_t seed, uint64_t ray, double u[6]);

/* ---- the integer form of the inverse-CDF sampling (host helper, exported for tests): thr[i] = the smallest 32-bit
 * word w whose uniform u = (w + 0.5) 2^-32 satisfies cdf[i] < u, saturated at 0xffffffff. lowerBound(cdf, u) (rt:437,
 * 464) is then the number of thresholds <= w, for every w < 0xffffffff. */
void sart_cdf_thresholds(const double* cdf, int n, uint32_t* thr);

/* ---- sampler of the emission shell and the energy (rt:437, 464). SART_SAMPLER_INVERSE_CDF (default) is the reference's
 * lowerBound(cdf, u) as exact integer work: the ray a (seed, index) pair denotes is the same in every precision mode and in
 * the CPU oracle. SART_SAMPLER_ALIAS draws from the very same discrete distributions — P(i) = the number of 32-bit words
 * the inverse-CDF search maps to i, over 2^32 — through Walker/Vose alias tables: one table lookup instead of a search
 * (+13 % rays/s on CAST+LLNL). The distributions agree to ~1e-9 per index, the (seed, index) -> ray mapping does not:
 * runs agree with the other modes and the oracle statistically (tier b), not ray by ray. Honoured by sart_trace_mc (single
 * mass), sart_angular_scan and sart_trace_mc_rays in precision mode 2; those calls fail with SART_ERR_CONFIG in any other
 * configuration while it is selected. The X-ray test source draws no table values and is unaffected. */
enum { SART_SAMPLER_INVERSE_CDF = 0, SART_SAMPLER_ALIAS = 1 };
int sart_set_sampler(sart_handle_t* h, int sampler);
/* Host helper, exported for tests: the alias entries of the distribution the n thresholds `thr` (sart_cdf_thresholds)
 * define. entries[k]: bits 31..11 = the share of bucket k that stays with index k, in units of 2^-21 of the bucket;
 * bits 10..0 = the index that receives the rest. A 32-bit word w selects k = (w n) >> 32 and takes index k when the low 32
 * bits of w n are below (entries[k] & 0xfffff800), else the alias. n <= 2048 (entries are zeroed otherwise). */
void sart_alias_table(const uint32_t* thr, int n, uint32_t* entries);

/* ---- the radial lookup table of the shell search (host helper, exported for tests). The FP32 kernels replace the
 * scan of rt:1932-1957 (hit shell = first j with R1[j] > rho; glass front of the shell below rt:1942-1944; outside the
 * last shell rt:1934) by one record of a uniform radial table. For n radial distances rho [mm] this returns the outcome
 * through the table (via_table) and through the scan (via_scan): the shell number (< 64), or 64 + the SART_EXIT_* code.
 * SART_ERR_CONFIG when the shells are too closely spaced for the table (the throughput modes then refuse the setup). */
int sart_shell_lookup(const sart_setup_t* setup, int n, const float* rho, int32_t* via_table, int32_t* via_scan);

/* ---- the error budgets of the FP32 decisions (host helper, exported for tests and for the curious): for a Monte Carlo ray
 * of this setup with slopes |sx| + |sy| = slope_sum and emission radius rs (in solar radii), the lateral position budget
 * before the mirrors and at the detector plane [mm], as the kernels of precision mode 2 form them (sart_set_retrace;
 * DESIGN.md section 3b), and whether the pipe tests are skipped for this setup (no solar ray can reach the pipe wall).
 * nRadii: rows of the solar table (the outermost emission shell bounds the slopes). */
int sart_error_budgets(const sart_setup_t* setup, int nRadii, double scale, double slope_sum, double rs, double* lat_mm,
                       double* det_mm, int* pipes_free);

/* ---- which pipelines take this setup (host helper; no device needed). Returns 1 when precision modes 1 and 2 can run it,
 * 0 when only the exact pipeline can — `why` (optional, at most why_len bytes incl. the terminator) then says what is in
 * the way — and a negative SART_ERR_* for an invalid setup. Since round 2 the throughput modes cover every reflectivity
 * kind (rt:1533-1580) and XMM hole type (rt:1674-1688) of the reference; they refuse shells that overlap or are not in
 * ascending order of radius and hole patterns of more than 64 holes. (Mode 2 in addition needs its radial shell table:
 * sart_shell_lookup tells.) */
int sart_throughput_supported(const sart_setup_t* setup, char* why, int why_len);

#ifdef __cplusplus
}
#endif
#endif /* SART_H */
