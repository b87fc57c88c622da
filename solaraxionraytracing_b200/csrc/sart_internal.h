// sart_internal.h — private to libsart.so: the handle, error reporting, launcher prototypes.
#pragma once
#include <cstdarg>
#include <cstddef>
#include <cstdint>

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
  size_t fast_shell_off = 0, fast_shell32_off = 0, fast_lut_off = 0, fast_glut_off = 0, fast_tt_off = 0, fast_sguide_off = 0, fast_stab_off = 0, fast_refl_off = 0;
  std::vector<float> h_refl32;  // host copy of the reflectivity (f32) for rebuilding the X-ray-source row
  std::vector<double> h_energies, h_tab[4][2];  // host copies (energies; strongback/window/gas/telescope transmission x,y) for LUT rebuilds
  int sm_count = 148;
  size_t shell_offset = 0;      // byte offset of the ShellF64 array inside table_blob
  int n_masses = 1;
  int masses_default = 1;       // masses[0] still mirrors setup.consts.mAxion
  int image_masses = 0;         // mass planes the image buffers were allocated for
  double masses[SART_MAX_MASSES] = {0};
  double* d_masses = nullptr;   // [SART_MAX_MASSES]
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
  // optional radial histogram of the passed rays (sart_enable_radial_hist)
  double* d_rad_w = nullptr;
  unsigned long long* d_rad_n = nullptr;
  int rad_bins = 0;
  double rad_rmax = 0.0;
  // optional spectra of the passed rays (sart_enable_spectra), one allocation each: the handle's arrays (the exact kernels
  // and the re-trace add into them directly) and the replicas of the throughput kernels (device_params.h: Spectra), which
  // the fold after every launch adds up and clears. Only sart_trace_mc hands them to a kernel.
  void* d_spec = nullptr;
  void* d_spec_rep = nullptr;
  sart::Spectra spec{}, spec_rep{};   // spec.eW == nullptr: off
  int spec_e1 = 0;                    // energy bins: nEnergies + 1 (the last one is the X-ray source's)
  // staging for the host-pointer entry points
  void* d_stage = nullptr;
  size_t stage_bytes = 0;
  cudaStream_t stream_in = nullptr, stream_out = nullptr;   // copy streams of the chunked host-buffer paths
  void* ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // cudaEvent_t: inputs landed / kernel done / outputs landed, x2 buffers
  void* h_stage = nullptr;      // pinned
  size_t h_stage_bytes = 0;
};
