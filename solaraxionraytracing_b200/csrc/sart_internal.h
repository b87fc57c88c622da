// sart_internal.h — private to libsart.so: the handle and its optional accumulators, error reporting, launcher prototypes.
#pragma once
#include <cstdarg>
#include <cstddef>
#include <cstdint>

#include <initializer_list>
#include <vector>

#include "../../include/sart.h"
#include "device_params.h"
#include "fast_params.h"

typedef struct CUstream_st* cudaStream_t;

namespace sart {

// Records the message for sart_last_error() and returns `code`.
int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));

// Host derivation of the kernel parameter blocks (derive.cpp).
void derive_params(const sart_setup_t& s, const sart_tables_t* tb, Params* p);
void derive_shells(const sart_setup_t& s, ShellF64* shells /* [SART_MAX_SHELLS] */);

namespace fast {
bool supported(const sart_setup_t& s, const char** why);
void derive_shells(const sart_setup_t& s, const ShellF64* exactShells, ShellFast* out);
void derive_params(const sart_setup_t& s, const Params& P, FastParams* f);
void derive_f32(const FastParams& f, const ShellFast* shells, int nShells, Geo32* g, ShellF32* out, float tolScale = 1.0f);
void derive_tolerances(const FastParams& f, const ShellFast* shells, int nShells, float scale, Tol32* t);
bool build_shell_table(const Geo32& g, const ShellF32* shells, int nShells, int nBuckets, std::vector<ShellCell>* out);
bool build_alias_table(const uint32_t* thr, int n, uint32_t* out /* [n] */);
int classify_radius(const ShellF32* shells, int nShells, float rho);
int shell_table_lookup(const Geo32& g, const std::vector<ShellCell>& tab, float rho);
void build_shell_guide(const sart_setup_t& s, FastParams* f, std::vector<uint8_t>* guide);
void build_energy_lut(int nE, const double* energies, const sart_interp1d_t& sb, const sart_interp1d_t& wd,
                      const sart_interp1d_t& ga, double srcEnergy, double reflEMin, double reflEMax,
                      std::vector<EnergyLUT>* out,
                      std::vector<GasLUT>* gout);
void refl_at_energy(const Params& P, const float* z, double E, float* out);
void build_tel_trans(int nE, const double* energies, const sart_interp1d_t& tt, double srcEnergy, std::vector<float>* out);
void build_sample_cells(const uint32_t* thr, int n, int bits, SampleCell* out /* [1 << bits] */);
}  // namespace fast

}  // namespace sart

namespace sart {
// sart_allreduce (comm.cu): the counters travel as f64 words behind the two images
constexpr int kCounterWords = int(sizeof(sart_counters_t) / 8);
inline size_t merged_words(int nMasses) {
  return size_t(nMasses) * (2 * size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS + size_t(kCounterWords));
}

// sart_allreduce_outputs (comm.cu): int64 words of the descriptor the ranks exchange, in sart_handle::d_desc
constexpr int kDescCapacity = 128;

// Bump allocator over one device buffer: every piece starts on a 256-byte boundary. Over a null base it only measures, so a
// layout is written once and run twice: over nullptr to size the buffer, then over the allocation to hand out its pointers.
struct Carve {
  unsigned char* base;
  size_t off = 0;
  explicit Carve(void* b = nullptr) : base(static_cast<unsigned char*>(b)) {}
  template <class T> void take(T*& p, size_t count) {
    p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off = (off + count * sizeof(T) + 255) & ~size_t(255);
  }
};

// The optional accumulators of the passed rays, each switched on and off by its own entry point: the radial histogram
// (sart_enable_radial_hist), the spectra (sart_enable_spectra), the per-mass spectra (sart_enable_mass_spectra), the
// band images (sart_enable_band_images), the quantity histograms (sart_enable_quantity_hists), the per-mass radial
// histograms (sart_enable_mass_radial_hist) and the per-mass band images (sart_enable_mass_band_images).
enum AccumKind { kRadialHist, kSpectra, kMassSpectra, kBandImages, kQuantityHists, kMassRadialHist, kMassBandImages, kAccums };
constexpr AccumKind kAllAccums[kAccums] = {kRadialHist, kSpectra, kMassSpectra, kBandImages, kQuantityHists, kMassRadialHist,
                                           kMassBandImages};
// The per-mass accumulators: one row per axion mass, filled by the mass-scan kernels.
constexpr bool per_mass(AccumKind k) { return k == kMassSpectra || k == kMassRadialHist || k == kMassBandImages; }

// One block of an accumulator: the handle's own (sart_handle::accum) or its merged copy (sart_handle::merged_accum), both
// one allocation laid out by the same code (api.cu: alloc_accum). blob == nullptr: off (and bins == 0).
struct Accum {
  void* blob = nullptr;
  size_t bytes = 0;
  int bins = 0;         // (per-mass) radial histogram: its bins per row; (per-mass) spectra: energy bins per row, nEnergies + 1;
                        // (per-mass) band images: bands per row; quantity histograms: their entries, Σ(nbins + 2)
  double rmax = 0.0;    // (per-mass) radial histogram: its range
  double edges[SART_MAX_BANDS + 1] = {};   // (per-mass) band images: the bins + 1 band edges [keV]
  int n_qhists = 0;                        // quantity histograms: their specs, in the caller's order
  sart_quantity_hist_t qspecs[SART_N_QUANTITIES] = {};
  RadialHist rad{};     // (per-mass) radial histogram: w, n [bins], per mass one such row
  Spectra spec{};       // (per-mass) spectra: eW, eW2, eN, sW, sN; the per-mass spectra have one row per mass (eRow, sRow)
  BandImages band{};    // (per-mass) band images: w, w2 [bins][256][256], n [bins], per mass one such row; the handle's
                        // block also its energy -> band table
  QuantityHists qh{};   // quantity histograms: w, w2, n [bins]; the handle's block also the specs and the replicas rw, rw2
  int valid = 0;        // merged copy: it holds the sums of the last sart_allreduce_outputs for the masses set
  // The handle's own block only: the buffers the throughput kernels add into instead (api.cu: carve_throughput), which the
  // fold after every launch adds into the arrays above and clears. The spectra's replicas, the per-mass spectra's
  // mass-minor accumulators, the band images' replicas (tput_band, which also holds the energy -> band table), the
  // per-mass radial histograms' and band images' mass-minor accumulators (tput_rad, tput_band); the radial histogram has
  // none, the quantity histograms keep theirs in qh.
  void* tput_blob = nullptr;
  Spectra tput{};
  BandImages tput_band{};
  RadialHist tput_rad{};
};

// Rows of accumulator k for nMasses axion masses: one per mass for the per-mass accumulators (allocated for SART_MAX_MASSES,
// read and merged for the masses set), one for the others.
inline size_t accum_rows(AccumKind k, int nMasses) { return per_mass(k) ? size_t(nMasses) : 1; }

// The arrays of an accumulator: f(a.array, b.array, count) for every device array of a pair of blocks of kind k (a block
// and itself, or a handle's block and its merged copy) in layout order, `count` elements for `rows` rows of a.bins bins.
// The only place that lists them; an element is an f64 sum (double) or a u64 count (unsigned long long).
template <class A, class B, class F>
inline void accum_arrays(AccumKind k, A& a, B& b, size_t rows, F&& f) {
  const size_t e = rows * size_t(a.bins), s = rows * SART_MAX_SHELLS;
  if (k == kRadialHist || k == kMassRadialHist) {
    f(a.rad.w, b.rad.w, e); f(a.rad.n, b.rad.n, e);
    return;
  }
  if (k == kBandImages || k == kMassBandImages) {
    const size_t p = e * SART_IMAGE_BINS * SART_IMAGE_BINS;
    f(a.band.w, b.band.w, p); f(a.band.w2, b.band.w2, p); f(a.band.n, b.band.n, e);
    return;
  }
  if (k == kQuantityHists) {
    f(a.qh.w, b.qh.w, e); f(a.qh.w2, b.qh.w2, e); f(a.qh.n, b.qh.n, e);
    return;
  }
  f(a.spec.eW, b.spec.eW, e); f(a.spec.eW2, b.spec.eW2, e); f(a.spec.eN, b.spec.eN, e);
  f(a.spec.sW, b.spec.sW, s); f(a.spec.sN, b.spec.sN, s);
}

// api.cu: a block of accumulator k with `bins` bins (rmax: the radial histogram's range), allocated and carved but not
// cleared. On failure `a` stays empty and the error is recorded.
int alloc_accum(AccumKind k, int bins, double rmax, Accum* a);
// api.cu: the reader behind sart_read_radial_hist / _spectra / _mass_spectra / ... and their sart_read_merged_* twins. Copies the
// rows in use of accumulator k, the handle's own block or its merged copy, into the caller's arrays `host`, one per array
// in the order of accum_arrays (NULL: skipped), and synchronises. `off`: the error while there is nothing to read.
int read_accum(sart_handle* h, AccumKind k, bool merged, std::initializer_list<void*> host, const char* off);
}  // namespace sart

struct sart_handle {
  int device = -1;
  cudaStream_t stream = nullptr;
  sart_setup_t setup;
  sart::Params params;
  sart::Tables tables;          // device pointers
  void* table_blob = nullptr;   // one allocation backing every table
  size_t table_bytes = 0;
  int precision = 0;            // 0 exact f64, 1 fast (f64 algebra + f32 weights), 2 f32 geometry
  int compact = 0;              // fast mode: warp-level compaction between the clip stages and the mirrors
  int compact_user = 0;         // set by sart_set_compaction: sart_update_setup keeps it instead of re-running the pilot
  int have_solar = 0, n_refl_coatings = 0, have_tel_transmission = 0;   // which caller tables sart_create uploaded
  double pilot_survival = 1.0;  // fraction of launched rays that reach the mirrors (pilot run at create)
  // "fast" pipeline: parameter block, LUTs and f32 reflectivity in a second allocation
  int fast_ok = 0;
  const char* fast_why = "";
  int sampler = 0;      // SART_SAMPLER_*
  int alias_ok = 0;     // alias tables built (nRadii, nEnergies <= 2048)
  int f32_ok = 0;   // precision mode 2 also needs the radial shell table (derive_fast.cpp: build_shell_table)
  sart::fast::FastParams fparams;
  sart::fast::FastTables ftables;
  sart::fast::Geo32 geo32;      // single-precision geometry block of precision mode 2
  void* fast_blob = nullptr;
  std::vector<float> h_refl32;  // host copy of the reflectivity (f32) for rebuilding the X-ray-source row
  std::vector<double> h_energies, h_tab[4][2];  // host copies (energies; strongback/window/gas/telescope transmission x,y) for LUT rebuilds
  int sm_count = 148;
  int n_masses = 1;
  int masses_default = 1;       // masses[0] still mirrors setup.consts.mAxion
  int image_masses = 0;         // mass planes the image buffers were allocated for
  double masses[SART_MAX_MASSES] = {0};
  double* d_masses = nullptr;   // [SART_MAX_MASSES]
  long long* d_desc = nullptr;  // [kDescCapacity] the descriptor of sart_allreduce_outputs (comm.cu: describe_outputs)
  // one allocation of merged_words(n_masses) doubles: image [n_masses][256][256] | w^2 image | counter words (the send
  // buffer of sart_allreduce); d_image_w2 points into it
  double* d_image = nullptr;
  double* d_image_w2 = nullptr;
  // NCCL communicator of this handle (comm.cu) and the result of the last sart_allreduce, laid out like the block above
  void* comm = nullptr;
  int comm_ranks = 0, comm_rank = 0;
  double* d_merged = nullptr;
  int merged_masses = 0, merged_valid = 0;
  sart_counters_t* d_counters = nullptr;  // [n_masses]
  // image replicas of the throughput kernels (cleared by the fold that follows every launch)
  double* d_rep = nullptr;      // [2][n_rep][256*256]
  double* d_mass_acc = nullptr; // [2][256*256][SART_MAX_MASSES] mass-major accumulators of the mass-scan kernel
  int n_rep = 0;
  size_t rep_stride = 0;        // doubles between two replicas
  // re-trace queue of precision mode 2 (fast_params.h: RetraceQueue): [0] = push count, entries from word 64 on
  uint32_t* d_queue = nullptr;
  size_t queue_cap = 0;
  int retrace = 1;              // sart_set_retrace: uncertain FP32 rays are re-traced in FP64
  float retrace_scale = 1.0f;   // multiplies every error budget (Tol32)
  // the optional accumulators (indexed by sart::AccumKind): the handle's arrays, which the exact kernels and the re-trace
  // add into directly (the radial histogram also reaches the kernels through tables.rad / ftables.rad, the others only
  // through sart_trace_mc), and their merged copies, the sums over all ranks of the last sart_allreduce_outputs
  sart::Accum accum[sart::kAccums], merged_accum[sart::kAccums];
  // staging for the host-pointer entry points
  void* d_stage = nullptr;
  size_t stage_bytes = 0;
  cudaStream_t stream_in = nullptr, stream_out = nullptr;   // copy streams of the chunked host-buffer paths
  void* ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // cudaEvent_t: inputs landed / kernel done / outputs landed, x2 buffers
  void* h_stage = nullptr;      // pinned: the record counts of the two buffers of sart_trace_mc_passed
};
