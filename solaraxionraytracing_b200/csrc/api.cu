// api.cu — the C-ABI of libsart.so (include/sart.h): handle lifetime, table upload, launches, read-back.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "kernels.h"
#include "philox.cuh"
#include "sart_internal.h"

namespace sart {

static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}

static int cuda_fail(cudaError_t e, const char* what) {
  return fail(SART_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

#define SART_CUDA(call)                                  \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

static size_t align256(size_t n) { return (n + 255) & ~size_t(255); }

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static int validate(const sart_setup_t* s, const sart_tables_t* t) {
  if (!s) return fail(SART_ERR_ARG, "setup is NULL");
  if (s->abi_version != SART_ABI_VERSION) return fail(SART_ERR_ARG, "setup.abi_version %u != %u", s->abi_version, SART_ABI_VERSION);
  const sart_telescope_t& tel = s->telescope;
  if (tel.kind != SART_TK_LLNL && tel.kind != SART_TK_XMM && tel.kind != SART_TK_ABRIXAS)
    return fail(SART_ERR_CONFIG, "The telescope kind %d does not have any opaque structures implemented yet.", tel.kind);
  if (tel.nShells < 1 || tel.nShells > SART_MAX_SHELLS) return fail(SART_ERR_ARG, "telescope.nShells %d out of range", tel.nShells);
  if (tel.nCoatings < 0 || tel.nCoatings > SART_MAX_COATINGS) return fail(SART_ERR_ARG, "telescope.nCoatings out of range");
  if (!t) return SART_OK;
  if (!s->testSource.active) {
    if (t->nRadii < 1 || t->nEnergies < 1 || !t->energies || !t->fluxRadiusCDF || !t->diffFluxCDFs)
      return fail(SART_ERR_ARG, "solar model tables missing");
    if (t->nRadii > 65535 || t->nEnergies > 65535) return fail(SART_ERR_ARG, "solar model tables too large for the guide tables");
  }
  if (!(s->flags & SART_CF_IGNORE_REFLECTION)) {
    if (tel.reflKind == SART_RK_EFFECTIVE_AREA) {
      if (t->telescopeTransmission.n < 2) return fail(SART_ERR_ARG, "telescopeTransmission table missing");
    } else {
      if (!t->reflectivity || t->nAngles < 2 || t->nReflEnergies < 2) return fail(SART_ERR_ARG, "reflectivity table missing");
      const int need = tel.reflKind == SART_RK_MULTI_COATING ? tel.nCoatings : 1;
      if (t->nCoatings < need) return fail(SART_ERR_ARG, "reflectivity table has %d coatings, telescope needs %d", t->nCoatings, need);
    }
  }
  if (t->strongbackTransmission.n < 2 || t->windowTransmission.n < 2 || t->gasAbsorption.n < 2)
    return fail(SART_ERR_ARG, "detector transmission tables missing");
  return SART_OK;
}

// Guide table of a CDF row: g[k] = lowerBound(cdf, k/K). For a uniform u in bucket k (k/K <= u < (k+1)/K) the answer of
// lowerBound(cdf, u) is >= g[k], and usually g[k] or g[k] + 1: the device counts thresholds from there.
static void build_guide(const double* cdf, int n, int nBuckets, uint16_t* out) {
  int pos = 0;
  for (int k = 0; k < nBuckets; ++k) {
    const double key = double(k) / double(nBuckets);
    while (pos < n && cdf[pos] < key) ++pos;
    out[k] = uint16_t(pos);
  }
}

// Smallest 32-bit word w with c < (w + 0.5) 2^-32, i.e. "cdf entry < uniform of word w" <=> w >= threshold. Exact:
// c 2^32 is a power-of-two scaling and its fractional part is compared with 0.5. Saturates at 0xffffffff (c within
// 1.5 2^-32 of 1, or NaN rows of shells that emit nothing); the kernel sends that one word to the f64 table.
static uint32_t cdf_threshold(double c) {
  if (c != c) return 0xffffffffu;
  if (!(c > 0.0)) return 0u;
  const double x = c * 4294967296.0, k = std::floor(x);
  const double t = k + ((x - k) >= 0.5 ? 1.0 : 0.0);
  return t >= 4294967295.0 ? 0xffffffffu : uint32_t(t);
}
static void build_thresholds(const double* cdf, int n, uint32_t* out /* [thr_pitch(n)] */) {
  const int pitch = thr_pitch(n);
  // non-decreasing by construction for a cumulative sum of non-negative rates; enforced, because the device counts
  // "thresholds <= w" assuming it (count_le)
  uint32_t prev = 0u;
  for (int i = 0; i < n; ++i) { prev = std::max(prev, cdf_threshold(cdf[i])); out[i] = prev; }
  for (int i = n; i < pitch; ++i) out[i] = 0xffffffffu;
}

struct Blob {  // bump allocator over one device allocation
  unsigned char* base = nullptr;
  size_t off = 0;
  std::vector<std::pair<size_t, std::vector<unsigned char>>> pending;
  template <class T> size_t add(const T* src, size_t count) {
    const size_t bytes = count * sizeof(T);
    const size_t at = off;
    std::vector<unsigned char> v(bytes);
    if (bytes) std::memcpy(v.data(), src, bytes);
    pending.emplace_back(at, std::move(v));
    off = align256(off + bytes);
    return at;
  }
};

// numericalnim newLinear1D.eval as the device evaluates it (trace_exact.cuh: eval_linear1d), operation for operation: this
// translation unit's host code is compiled without contraction, the device code with -fmad=false, so both produce the same
// bits.
static double eval_linear1d_host(const sart_interp1d_t& t, double x, int* clamped) {
  const int n = t.n;
  if (n < 2 || !t.x || !t.y) { *clamped = 1; return (n == 1 && t.y) ? t.y[0] : 0.0; }
  const double x0 = t.x[0], xn = t.x[n - 1];
  if (!(x >= x0)) { *clamped = 1; x = x0; }
  if (!(x <= xn)) { *clamped = 1; x = xn; }
  int lo = 0, hi = n - 1;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (t.x[mid] <= x) lo = mid; else hi = mid;
  }
  const double xl = t.x[lo], yl = t.y[lo];
  const double slope = (t.y[lo + 1] - yl) / (t.x[lo + 1] - xl);
  return yl + (x - xl) * slope;
}

static int upload_tables(sart_handle* h, const sart_tables_t* t) {
  Blob b;
  size_t oEn = 0, oRC = 0, oDC = 0, oRefl = 0;
  const bool solar = t->nRadii > 0 && t->energies;
  if (solar) {
    oEn = b.add(t->energies, t->nEnergies);
    oRC = b.add(t->fluxRadiusCDF, t->nRadii);
    oDC = b.add(t->diffFluxCDFs, size_t(t->nRadii) * t->nEnergies);
  }
  const bool refl = t->reflectivity && t->nCoatings > 0;
  if (refl) oRefl = b.add(t->reflectivity, size_t(t->nCoatings) * t->nAngles * t->nReflEnergies);
  const sart_interp1d_t* I[4] = {&t->strongbackTransmission, &t->windowTransmission, &t->gasAbsorption, &t->telescopeTransmission};
  size_t oX[4] = {0, 0, 0, 0}, oY[4] = {0, 0, 0, 0};
  for (int k = 0; k < 4; ++k)
    if (I[k]->n > 0 && I[k]->x && I[k]->y) { oX[k] = b.add(I[k]->x, I[k]->n); oY[k] = b.add(I[k]->y, I[k]->n); }
  std::vector<sart::ShellF64> shells(SART_MAX_SHELLS);
  derive_shells(h->setup, shells.data());
  const size_t oSh = b.add(shells.data(), shells.size());
  // window / strongback / detector-gas factors at each tabulated energy (device_params.h: EnergyFactors)
  std::vector<EnergyFactors> ef;
  size_t oEf = 0;
  if (solar) {
    ef.resize(size_t(t->nEnergies));
    for (int i = 0; i < t->nEnergies; ++i) {
      const double E = t->energies[i] > 0.03 ? t->energies[i] : 0.03;   // rt:470-471
      int cw = 0, cs = 0, cg = 0;
      ef[size_t(i)].window = eval_linear1d_host(t->windowTransmission, E, &cw);
      ef[size_t(i)].strongback = eval_linear1d_host(t->strongbackTransmission, E, &cs);
      ef[size_t(i)].gas = eval_linear1d_host(t->gasAbsorption, E, &cg);
      ef[size_t(i)].clamped = cw | (cs << 1) | (cg << 2);
      ef[size_t(i)].pad = 0;
    }
    oEf = b.add(ef.data(), ef.size());
  }

  if (h->table_blob) { cudaFree(h->table_blob); h->table_blob = nullptr; }
  SART_CUDA(cudaMalloc(&h->table_blob, b.off ? b.off : 256));
  h->table_bytes = b.off;
  unsigned char* base = static_cast<unsigned char*>(h->table_blob);
  for (auto& pr : b.pending)
    if (!pr.second.empty()) SART_CUDA(cudaMemcpyAsync(base + pr.first, pr.second.data(), pr.second.size(), cudaMemcpyHostToDevice, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));

  Tables& T = h->tables;
  std::memset(&T, 0, sizeof T);
  if (solar) {
    T.energies = reinterpret_cast<const double*>(base + oEn);
    T.fluxRadiusCDF = reinterpret_cast<const double*>(base + oRC);
    T.diffFluxCDFs = reinterpret_cast<const double*>(base + oDC);
  }
  if (refl) T.reflectivity = reinterpret_cast<const double*>(base + oRefl);
  const double** PX[4] = {&T.sbX, &T.wdX, &T.gaX, &T.ttX};
  const double** PY[4] = {&T.sbY, &T.wdY, &T.gaY, &T.ttY};
  int32_t* PN[4] = {&T.sbN, &T.wdN, &T.gaN, &T.ttN};
  for (int k = 0; k < 4; ++k)
    if (I[k]->n > 0 && I[k]->x && I[k]->y) {
      *PX[k] = reinterpret_cast<const double*>(base + oX[k]);
      *PY[k] = reinterpret_cast<const double*>(base + oY[k]);
      *PN[k] = I[k]->n;
    }
  T.shells = reinterpret_cast<const ShellF64*>(base + oSh);
  if (solar) T.energyFactors = reinterpret_cast<const EnergyFactors*>(base + oEf);
  h->shell_offset = oSh;
  h->have_solar = solar ? 1 : 0;
  h->n_refl_coatings = refl ? t->nCoatings : 0;
  h->have_tel_transmission = (I[3]->n >= 2 && I[3]->x && I[3]->y) ? 1 : 0;
  return SART_OK;
}

// sart_update_setup may only move to setups the tables uploaded at sart_create cover (validate() checked them against
// the setup of that moment only).
static int validate_update(const sart_handle* h, const sart_setup_t* s) {
  int rc = validate(s, nullptr);
  if (rc) return rc;
  if (!s->testSource.active && !h->have_solar)
    return fail(SART_ERR_ARG, "sart_update_setup: the solar source needs the solar model tables, and this handle was created without them");
  if (!(s->flags & SART_CF_IGNORE_REFLECTION)) {
    if (s->telescope.reflKind == SART_RK_EFFECTIVE_AREA) {
      if (!h->have_tel_transmission)
        return fail(SART_ERR_ARG, "sart_update_setup: rkEffectiveArea needs the telescopeTransmission table, and this handle was created without it");
    } else {
      const int need = s->telescope.reflKind == SART_RK_MULTI_COATING ? s->telescope.nCoatings : 1;
      if (h->n_refl_coatings < need)
        return fail(SART_ERR_ARG, "sart_update_setup: the setup needs %d reflectivity coatings, the handle holds %d", need, h->n_refl_coatings);
    }
  }
  return SART_OK;
}

// Builds / refreshes the device data of the fast pipeline. `t` may be NULL on a setup update (tables unchanged).
static int upload_fast(sart_handle* h, const sart_tables_t* t) {
  const char* why = "";
  h->fast_ok = fast::supported(h->setup, &why) ? 1 : 0;
  h->fast_why = why;
  h->f32_ok = 0;
  const Params& P = h->params;
  if (t) {   // host copies for later LUT rebuilds, kept whether or not this setup can use the throughput pipelines
    h->h_energies.assign(t->energies ? t->energies : nullptr, t->energies ? t->energies + t->nEnergies : nullptr);
    const sart_interp1d_t* I[4] = {&t->strongbackTransmission, &t->windowTransmission, &t->gasAbsorption, &t->telescopeTransmission};
    for (int k = 0; k < 4; ++k) {
      if (I[k]->n < 1 || !I[k]->x || !I[k]->y) { h->h_tab[k][0].clear(); h->h_tab[k][1].clear(); continue; }
      h->h_tab[k][0].assign(I[k]->x, I[k]->x + I[k]->n);
      h->h_tab[k][1].assign(I[k]->y, I[k]->y + I[k]->n);
    }
    const size_t nRefl = t->reflectivity ? size_t(t->nCoatings) * t->nAngles * t->nReflEnergies : 0;
    h->h_refl32.resize(nRefl);
    // a reflectivity that is non-zero in f64 stays non-zero in the f32 copy: `passed` means weight != 0 (rt:2220), and
    // multilayer tables reach 1e-50 at large angles
    for (size_t i = 0; i < nRefl; ++i) {
      const double v = t->reflectivity[i];
      h->h_refl32[i] = (v != 0.0 && std::fabs(v) < 1.2e-38) ? float(std::copysign(1.2e-38, v)) : float(v);
    }
  }
  if (!h->fast_ok) return SART_OK;
  if (!t && !h->fast_blob) {
    // the derived sampling tables (thresholds, guides, reflectivity rows) are built from the caller's tables at
    // sart_create only; a handle created with a setup the throughput pipelines do not support never got them
    h->fast_ok = 0;
    h->fast_why = "the handle was created with a setup the throughput pipelines do not support; create a new handle for this setup";
    return SART_OK;
  }
  sart_interp1d_t I[4];
  for (int k = 0; k < 4; ++k) I[k] = sart_interp1d_t{int32_t(h->h_tab[k][0].size()), 0, h->h_tab[k][0].data(), h->h_tab[k][1].data()};
  fast::derive_params(h->setup, P, &h->fparams);
  if (h->h_energies.size() > 1) {
    h->fparams.enE0 = h->h_energies.front();
    h->fparams.enInvStep = double(h->h_energies.size() - 1) / (h->h_energies.back() - h->h_energies.front());
  }
  std::vector<ShellF64> sh64(SART_MAX_SHELLS);
  derive_shells(h->setup, sh64.data());
  std::vector<fast::ShellFast> shf(SART_MAX_SHELLS);
  fast::derive_shells(h->setup, sh64.data(), shf.data());
  std::vector<uint8_t> sguide;
  fast::build_shell_guide(h->setup, &h->fparams, &sguide);
  if (sguide.size() > 4096) return fail(SART_ERR_CONFIG, "shell guide too large (%zu)", sguide.size());
  std::vector<fast::ShellF32> sh32(SART_MAX_SHELLS);
  fast::derive_f32(h->fparams, shf.data(), h->setup.telescope.nShells, &h->geo32, sh32.data(), h->retrace_scale);
  std::vector<fast::ShellCell> stab;
  h->f32_ok = fast::build_shell_table(h->geo32, sh32.data(), h->setup.telescope.nShells, int(sguide.size()), &stab) ? 1 : 0;
  if (!h->f32_ok) stab.assign(sguide.size(), fast::ShellCell{0.f, 0u});   // mode 1 (its own shell scan) stays available
  const int nE = int(h->h_energies.size());
  std::vector<fast::EnergyLUT> lut;
  std::vector<fast::GasLUT> glut;
  // the "reflectivity grid" whose ends set the clamped flag of an energy: the reflectivity table's energy axis, or the
  // abscissae of the telescope transmission for rkEffectiveArea (trace_exact.cuh: ray_weights)
  const bool effArea = P.reflKind == SART_RK_EFFECTIVE_AREA;
  const double rEMin = effArea ? (I[3].n >= 2 ? I[3].x[0] : INFINITY) : P.reflEMin;
  const double rEMax = effArea ? (I[3].n >= 2 ? I[3].x[I[3].n - 1] : -INFINITY) : P.reflEMax;
  fast::build_energy_lut(nE, h->h_energies.data(), I[0], I[1], I[2], h->setup.testSource.energy, rEMin, rEMax, &lut, &glut);
  std::vector<float> telTrans;
  fast::build_tel_trans(nE, h->h_energies.data(), I[3], h->setup.testSource.energy, &telTrans);
  const int nCoat = P.nAngles > 0 && !h->h_refl32.empty() ? int(h->h_refl32.size() / (size_t(P.nAngles) * P.nReflEnergies)) : 0;
  const size_t reflRow = size_t(P.nAngles), reflPlane = reflRow * (size_t(nE) + 1);
  // the throughput kernels address table rows with 32-bit element offsets
  if (size_t(std::max(nCoat, 1)) * reflPlane >= (size_t(1) << 31) ||
      size_t(std::max(P.nRadii, 1)) * thr_pitch(std::max(P.nEnergies, 1)) >= (size_t(1) << 31) ||
      size_t(std::max(P.nRadii, 1)) * kEnGuide >= (size_t(1) << 31) ||
      size_t(std::max(P.nRadii, 1)) * kEnCells >= (size_t(1) << 31))
    return fail(SART_ERR_CONFIG, "tables too large for the throughput pipelines (a table exceeds 2^31 elements)");
  unsigned char* base = static_cast<unsigned char*>(h->fast_blob);
  if (t) {
    // layout: shells | shell guide (4 KiB) | lut | gas lut | radius guide | energy guide | reflE
    size_t off = 0;
    h->fast_shell_off = off; off += align256(shf.size() * sizeof(fast::ShellFast));
    h->fast_shell32_off = off; off += align256(size_t(SART_MAX_SHELLS) * sizeof(fast::ShellF32));
    h->fast_sguide_off = off; off += 4096;
    h->fast_stab_off = off; off += 4096 * sizeof(fast::ShellCell);
    h->fast_lut_off = off; off += align256(lut.size() * sizeof(fast::EnergyLUT));
    h->fast_glut_off = off; off += align256(glut.size() * sizeof(fast::GasLUT));
    h->fast_tt_off = off; off += align256(telTrans.size() * sizeof(float));
    const size_t rgOff = off; off += align256(size_t(kRadGuide) * 2);
    const size_t egOff = off; off += align256(size_t(std::max(P.nRadii, 1)) * kEnGuide * 2);
    const size_t rtOff = off; off += align256(size_t(thr_pitch(std::max(P.nRadii, 1))) * 4);
    const size_t etOff = off; off += align256(size_t(std::max(P.nRadii, 1)) * thr_pitch(std::max(P.nEnergies, 1)) * 4);
    const size_t rcOff = off; off += align256(size_t(kRadCells) * sizeof(fast::SampleCell));
    const size_t ecOff = off; off += align256(size_t(std::max(P.nRadii, 1)) * kEnCells * sizeof(fast::SampleCell));
    h->fast_refl_off = off; off += align256(size_t(std::max(nCoat, 1)) * reflPlane * sizeof(float));
    // alias tables of the same distributions (sart_set_sampler), when the packed 11-bit alias index can hold them
    const bool aliasFits = P.nRadii > 0 && t->fluxRadiusCDF && P.nRadii <= 2048 && P.nEnergies <= 2048;
    const size_t raOff = off; off += aliasFits ? align256(size_t(P.nRadii) * 4) : 0;
    const size_t eaOff = off; off += aliasFits ? align256(size_t(P.nRadii) * P.nEnergies * 4) : 0;
    h->alias_ok = 0;
    if (h->fast_blob) { cudaFree(h->fast_blob); h->fast_blob = nullptr; }
    SART_CUDA(cudaMalloc(&h->fast_blob, off + 256));
    base = static_cast<unsigned char*>(h->fast_blob);
    if (P.nRadii > 0 && t->fluxRadiusCDF) {
      const int ep = thr_pitch(P.nEnergies);
      std::vector<uint16_t> rg(kRadGuide), eg(size_t(P.nRadii) * kEnGuide);
      std::vector<uint32_t> rth(size_t(thr_pitch(P.nRadii))), eth(size_t(P.nRadii) * ep);
      build_guide(t->fluxRadiusCDF, P.nRadii, kRadGuide, rg.data());
      build_thresholds(t->fluxRadiusCDF, P.nRadii, rth.data());
      for (int r = 0; r < P.nRadii; ++r) {
        build_guide(t->diffFluxCDFs + size_t(r) * P.nEnergies, P.nEnergies, kEnGuide, eg.data() + size_t(r) * kEnGuide);
        build_thresholds(t->diffFluxCDFs + size_t(r) * P.nEnergies, P.nEnergies, eth.data() + size_t(r) * ep);
      }
      SART_CUDA(cudaMemcpy(base + rgOff, rg.data(), rg.size() * 2, cudaMemcpyHostToDevice));
      SART_CUDA(cudaMemcpy(base + egOff, eg.data(), eg.size() * 2, cudaMemcpyHostToDevice));
      SART_CUDA(cudaMemcpy(base + rtOff, rth.data(), rth.size() * 4, cudaMemcpyHostToDevice));
      SART_CUDA(cudaMemcpy(base + etOff, eth.data(), eth.size() * 4, cudaMemcpyHostToDevice));
      {
        std::vector<fast::SampleCell> rc(kRadCells), ec(size_t(P.nRadii) * kEnCells);
        fast::build_sample_cells(rth.data(), P.nRadii, kRadCellBits, rc.data());
        for (int r = 0; r < P.nRadii; ++r)
          fast::build_sample_cells(eth.data() + size_t(r) * ep, P.nEnergies, kEnCellBits, ec.data() + size_t(r) * kEnCells);
        SART_CUDA(cudaMemcpy(base + rcOff, rc.data(), rc.size() * sizeof(fast::SampleCell), cudaMemcpyHostToDevice));
        SART_CUDA(cudaMemcpy(base + ecOff, ec.data(), ec.size() * sizeof(fast::SampleCell), cudaMemcpyHostToDevice));
      }
      if (aliasFits) {
        std::vector<uint32_t> ra(size_t(P.nRadii)), ea(size_t(P.nRadii) * P.nEnergies);
        bool ok = fast::build_alias_table(rth.data(), P.nRadii, ra.data());
        for (int r = 0; ok && r < P.nRadii; ++r)
          ok = fast::build_alias_table(eth.data() + size_t(r) * ep, P.nEnergies, ea.data() + size_t(r) * P.nEnergies);
        if (ok) {
          SART_CUDA(cudaMemcpy(base + raOff, ra.data(), ra.size() * 4, cudaMemcpyHostToDevice));
          SART_CUDA(cudaMemcpy(base + eaOff, ea.data(), ea.size() * 4, cudaMemcpyHostToDevice));
          h->alias_ok = 1;
        }
      }
    }
    // reflectivity interpolated along energy at each tabulated energy
    if (nCoat > 0) {
      std::vector<float> re(size_t(nCoat) * reflPlane), line(size_t(P.nAngles));
      for (int c = 0; c < nCoat; ++c) {
        const float* z = h->h_refl32.data() + size_t(c) * P.nAngles * P.nReflEnergies;
        for (int i = 0; i <= nE; ++i) {
          fast::refl_at_energy(P, z, i < nE ? std::max(0.03, h->h_energies[i]) : h->setup.testSource.energy, line.data());
          std::copy(line.begin(), line.end(), re.begin() + size_t(c) * reflPlane + size_t(i) * reflRow);
        }
      }
      SART_CUDA(cudaMemcpy(base + h->fast_refl_off, re.data(), re.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    fast::FastTables& F = h->ftables;
    F.energies = h->tables.energies;
    F.radiusCDF = h->tables.fluxRadiusCDF;
    F.energyCDF = h->tables.diffFluxCDFs;
    F.radiusGuide = reinterpret_cast<const uint16_t*>(base + rgOff);
    F.energyGuide = reinterpret_cast<const uint16_t*>(base + egOff);
    F.radiusThr = reinterpret_cast<const uint32_t*>(base + rtOff);
    F.energyThr = reinterpret_cast<const uint32_t*>(base + etOff);
    F.radiusCells = reinterpret_cast<const fast::SampleCell*>(base + rcOff);
    F.energyCells = reinterpret_cast<const fast::SampleCell*>(base + ecOff);
    F.elut = reinterpret_cast<const fast::EnergyLUT*>(base + h->fast_lut_off);
    F.glut = reinterpret_cast<const fast::GasLUT*>(base + h->fast_glut_off);
    F.reflE = reinterpret_cast<const float*>(base + h->fast_refl_off);
    F.telTrans = reinterpret_cast<const float*>(base + h->fast_tt_off);
    F.shells = reinterpret_cast<const fast::ShellFast*>(base + h->fast_shell_off);
    F.shells32 = reinterpret_cast<const fast::ShellF32*>(base + h->fast_shell32_off);
    F.shellGuide = reinterpret_cast<const uint8_t*>(base + h->fast_sguide_off);
    F.shellTab = reinterpret_cast<const fast::ShellCell*>(base + h->fast_stab_off);
    F.radiusAlias = h->alias_ok ? reinterpret_cast<const uint32_t*>(base + raOff) : nullptr;
    F.energyAlias = h->alias_ok ? reinterpret_cast<const uint32_t*>(base + eaOff) : nullptr;
    F.sampler = h->alias_ok ? h->sampler : SART_SAMPLER_INVERSE_CDF;
    // the exact pipeline narrows its two CDF searches with the same guide tables (device_params.h: Tables)
    const bool solarGuides = P.nRadii > 0 && t->fluxRadiusCDF;
    h->tables.radiusGuide = solarGuides ? F.radiusGuide : nullptr;
    h->tables.energyGuide = solarGuides ? F.energyGuide : nullptr;
  } else if (nCoat > 0) {
    // setup update: only the X-ray-source row (index nE) of each coating can have changed
    std::vector<float> row(reflRow), line(size_t(P.nAngles));
    for (int c = 0; c < nCoat; ++c) {
      fast::refl_at_energy(P, h->h_refl32.data() + size_t(c) * P.nAngles * P.nReflEnergies, h->setup.testSource.energy, line.data());
      std::copy(line.begin(), line.end(), row.begin());
      SART_CUDA(cudaMemcpy(base + h->fast_refl_off + (size_t(c) * reflPlane + size_t(nE) * reflRow) * sizeof(float),
                           row.data(), reflRow * sizeof(float), cudaMemcpyHostToDevice));
    }
  }
  SART_CUDA(cudaMemcpy(base + h->fast_shell_off, shf.data(), shf.size() * sizeof(fast::ShellFast), cudaMemcpyHostToDevice));
  SART_CUDA(cudaMemcpy(base + h->fast_shell32_off, sh32.data(), sh32.size() * sizeof(fast::ShellF32), cudaMemcpyHostToDevice));
  SART_CUDA(cudaMemcpy(base + h->fast_lut_off, lut.data(), lut.size() * sizeof(fast::EnergyLUT), cudaMemcpyHostToDevice));
  SART_CUDA(cudaMemcpy(base + h->fast_glut_off, glut.data(), glut.size() * sizeof(fast::GasLUT), cudaMemcpyHostToDevice));
  SART_CUDA(cudaMemcpy(base + h->fast_tt_off, telTrans.data(), telTrans.size() * sizeof(float), cudaMemcpyHostToDevice));
  SART_CUDA(cudaMemcpy(base + h->fast_sguide_off, sguide.data(), sguide.size(), cudaMemcpyHostToDevice));
  SART_CUDA(cudaMemcpy(base + h->fast_stab_off, stab.data(), stab.size() * sizeof(fast::ShellCell), cudaMemcpyHostToDevice));
  return SART_OK;
}

static int ensure_image(sart_handle* h, int nMasses) {
  const size_t len = size_t(nMasses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
  if (h->d_image && h->image_masses == nMasses) return SART_OK;
  cudaFree(h->d_image); cudaFree(h->d_counters);   // d_image_w2 points into d_image's block
  h->d_image = nullptr; h->d_image_w2 = nullptr; h->d_counters = nullptr; h->image_masses = 0; h->merged_valid = 0;
  SART_CUDA(cudaMalloc(&h->d_image, merged_words(nMasses) * sizeof(double)));
  h->d_image_w2 = h->d_image + len;
  SART_CUDA(cudaMalloc(&h->d_counters, size_t(nMasses) * sizeof(sart_counters_t)));
  h->image_masses = nMasses;
  SART_CUDA(cudaMemsetAsync(h->d_image, 0, merged_words(nMasses) * sizeof(double), h->stream));
  SART_CUDA(cudaMemsetAsync(h->d_counters, 0, size_t(nMasses) * sizeof(sart_counters_t), h->stream));
  return SART_OK;
}

static int ensure_stage(sart_handle* h, size_t bytes);

// Re-trace queue for a launch of n rays of the FP32 pipeline: room for 6 % of them (measured: 0.01 - 0.3 % are
// uncertain), cleared on the stream. Returns a queue with cap = 0 when re-tracing is off.
constexpr uint64_t kRetraceChunk = uint64_t(1) << 31;   // rays per launch: queue entries are 32-bit offsets
static int begin_queue(sart_handle* h, uint64_t n, fast::RetraceQueue* q) {
  *q = fast::RetraceQueue{nullptr, nullptr, 0u, 0u};
  if (!h->retrace || n == 0) return SART_OK;
  const size_t want = size_t(std::min<uint64_t>(n, std::max<uint64_t>(n / 16 + 65536, 1u << 20)));
  if (h->queue_cap < want) {
    SART_CUDA(cudaStreamSynchronize(h->stream));
    cudaFree(h->d_queue);
    h->d_queue = nullptr; h->queue_cap = 0;
    SART_CUDA(cudaMalloc(&h->d_queue, (want + 64) * sizeof(uint32_t)));
    h->queue_cap = want;
  }
  SART_CUDA(cudaMemsetAsync(h->d_queue, 0, 64 * sizeof(uint32_t), h->stream));
  q->list = h->d_queue + 64; q->count = h->d_queue; q->cap = uint32_t(std::min<size_t>(h->queue_cap, 0xffffffffu));
  return SART_OK;
}

// Replica buffers for the single-mass throughput kernels. SART_IMG_REPLICAS overrides the count (1 = off).
static int ensure_replicas(sart_handle* h) {
  if (h->n_rep > 0) return SART_OK;
  int n = 8;   // measured on B200, CAST+LLNL, 1e9 rays: 1 replica 43.8 ms, 4 / 16 / 64 replicas 36.1 ms
  if (const char* e = std::getenv("SART_IMG_REPLICAS")) n = std::max(1, std::min(256, std::atoi(e)));
  h->n_rep = n;
  h->rep_stride = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS;
  if (const char* e = std::getenv("SART_IMG_REP_SKEW")) h->rep_stride += size_t(std::max(0, std::atoi(e)));   // experiment: replicas not 512 KiB apart
  if (n > 1) {
    const size_t bytes = size_t(2) * n * h->rep_stride * sizeof(double);
    SART_CUDA(cudaMalloc(&h->d_rep, bytes));
    SART_CUDA(cudaMemsetAsync(h->d_rep, 0, bytes, h->stream));
  }
  return SART_OK;
}

// Chooses the fast kernel variant for this setup from a pilot run: warp compaction pays off only when a large
// fraction of the launched rays is removed before the mirrors (measured: BabyIAXO+XMM 0.33 survive, +35 %; CAST+LLNL
// 0.93 survive, -13 %).
static int autotune(sart_handle* h) {
  h->compact = 0;
  if (!h->fast_ok || h->setup.testSource.active) return SART_OK;
  const size_t plane = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS;
  const size_t bytes = 2 * plane * sizeof(double) + sizeof(sart_counters_t);
  int rc = ensure_stage(h, bytes);
  if (rc) return rc;
  unsigned char* base = static_cast<unsigned char*>(h->d_stage);
  SART_CUDA(cudaMemsetAsync(base, 0, bytes, h->stream));
  const uint64_t n = 1u << 17;
  sart_counters_t* dc = reinterpret_cast<sart_counters_t*>(base + 2 * plane * sizeof(double));
  fast::FastTables pilotTables = h->ftables;
  pilotTables.rad = RadialHist{};   // the pilot rays must not reach the user's radial histogram
  SART_CUDA(launch_mc_image_fast(h->fparams, pilotTables, h->setup.consts.mAxion, 0, n, 0x5eedull,
                                 reinterpret_cast<double*>(base), reinterpret_cast<double*>(base) + plane, dc,
                                 h->sm_count, false, h->stream));
  sart_counters_t c;
  SART_CUDA(cudaMemcpyAsync(&c, dc, sizeof c, cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  uint64_t early = 0;
  for (int e = SART_EXIT_MISSED_BORE; e <= SART_EXIT_GLASS_FRONT; ++e) early += c.n_exit[e];
  h->pilot_survival = c.n_rays ? 1.0 - double(early) / double(c.n_rays) : 1.0;
  h->compact = h->pilot_survival < 0.6 ? 1 : 0;
  return SART_OK;
}

static int ensure_stage(sart_handle* h, size_t bytes) {
  if (h->stage_bytes >= bytes) return SART_OK;
  if (h->d_stage) cudaFree(h->d_stage);
  h->d_stage = nullptr; h->stage_bytes = 0;
  SART_CUDA(cudaMalloc(&h->d_stage, bytes));
  h->stage_bytes = bytes;
  return SART_OK;
}

// One allocation of spectra (device_params.h: Spectra), 8-byte words: eW | eW2 | eN, each eRep x eStride | sW | sN, each
// sRep x SART_MAX_SHELLS.
static size_t spectra_bytes(int eStride, int eRep, int sRep) {
  return 3 * align256(size_t(eRep) * eStride * 8) + 2 * align256(size_t(sRep) * SART_MAX_SHELLS * 8);
}
static Spectra carve_spectra(void* base, int eStride, int eRep, int sRep) {
  unsigned char* p = static_cast<unsigned char*>(base);
  const size_t e = align256(size_t(eRep) * eStride * 8), s = align256(size_t(sRep) * SART_MAX_SHELLS * 8);
  Spectra r{};
  r.eW = reinterpret_cast<double*>(p);
  r.eW2 = reinterpret_cast<double*>(p + e);
  r.eN = reinterpret_cast<unsigned long long*>(p + 2 * e);
  r.sW = reinterpret_cast<double*>(p + 3 * e);
  r.sN = reinterpret_cast<unsigned long long*>(p + 3 * e + s);
  r.eStride = uint32_t(eStride); r.eRepMask = uint32_t(eRep - 1); r.sRepMask = uint32_t(sRep - 1);
  return r;
}

// Parameter block of `s` for a live handle: setup-derived fields recomputed, table-derived fields kept.
static void rederive_params(const sart_handle* h, const sart_setup_t& s, Params* p) {
  const Params old = h->params;
  derive_params(s, nullptr, p);
  p->nAngles = old.nAngles; p->nReflEnergies = old.nReflEnergies;
  p->angleMin = old.angleMin; p->angleMax = old.angleMax;
  p->reflEMin = old.reflEMin; p->reflEMax = old.reflEMax;
  p->reflDx = old.reflDx; p->reflDy = old.reflDy;
  p->nRadii = old.nRadii; p->nEnergies = old.nEnergies;
}

}  // namespace sart

using namespace sart;

extern "C" {

const char* sart_last_error(void) { return g_err; }
int sart_abi_version(void) { return SART_ABI_VERSION; }
size_t sart_sizeof_setup(void) { return sizeof(sart_setup_t); }
size_t sart_sizeof_tables(void) { return sizeof(sart_tables_t); }
size_t sart_sizeof_counters(void) { return sizeof(sart_counters_t); }
int sart_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

void sart_cdf_thresholds(const double* cdf, int n, uint32_t* thr) {
  if (!cdf || !thr || n < 0) return;
  for (int i = 0; i < n; ++i) thr[i] = cdf_threshold(cdf[i]);
}

int sart_shell_lookup(const sart_setup_t* setup, int n, const float* rho, int32_t* via_table, int32_t* via_scan) {
  if (!setup || n < 0 || (n > 0 && (!rho || !via_table || !via_scan))) return fail(SART_ERR_ARG, "sart_shell_lookup: bad argument");
  const int nS = setup->telescope.nShells;
  if (nS < 1 || nS > SART_MAX_SHELLS) return fail(SART_ERR_ARG, "sart_shell_lookup: nShells = %d", nS);
  std::vector<ShellF64> sh64(SART_MAX_SHELLS);
  derive_shells(*setup, sh64.data());
  std::vector<fast::ShellFast> shf(SART_MAX_SHELLS);
  fast::derive_shells(*setup, sh64.data(), shf.data());
  fast::FastParams F;
  std::memset(&F, 0, sizeof F);
  std::vector<uint8_t> sguide;
  fast::build_shell_guide(*setup, &F, &sguide);
  fast::Geo32 G;
  std::vector<fast::ShellF32> sh32(SART_MAX_SHELLS);
  fast::derive_f32(F, shf.data(), nS, &G, sh32.data());
  std::vector<fast::ShellCell> tab;
  if (sguide.size() > 4096 || !fast::build_shell_table(G, sh32.data(), nS, int(sguide.size()), &tab))
    return fail(SART_ERR_CONFIG, "shell radii too closely spaced for the radial lookup table");
  for (int i = 0; i < n; ++i) {
    via_table[i] = fast::shell_table_lookup(G, tab, rho[i]);
    via_scan[i] = fast::classify_radius(sh32.data(), nS, rho[i]);
  }
  return SART_OK;
}

int sart_error_budgets(const sart_setup_t* setup, int nRadii, double scale, double slope_sum, double rs, double* lat_mm,
                       double* det_mm, int* pipes_free) {
  int rc = validate(setup, nullptr);
  if (rc) return rc;
  if (!(scale >= 0.0) || nRadii < 1) return fail(SART_ERR_ARG, "sart_error_budgets: bad argument");
  Params P;
  derive_params(*setup, nullptr, &P);
  P.nRadii = nRadii;
  fast::FastParams F;
  fast::derive_params(*setup, P, &F);
  std::vector<ShellF64> sh64(SART_MAX_SHELLS);
  derive_shells(*setup, sh64.data());
  std::vector<fast::ShellFast> shf(SART_MAX_SHELLS);
  fast::derive_shells(*setup, sh64.data(), shf.data());
  fast::Tol32 t;
  fast::derive_tolerances(F, shf.data(), setup->telescope.nShells, float(scale), &t);
  if (lat_mm) *lat_mm = double(t.latA) + double(t.latS) * rs + double(t.latT) * slope_sum;
  if (det_mm) *det_mm = double(t.detA) + double(t.detS) * rs + double(t.detT) * slope_sum;
  if (pipes_free) *pipes_free = F.pipesFree;
  return SART_OK;
}

int sart_throughput_supported(const sart_setup_t* setup, char* why, int why_len) {
  int rc = validate(setup, nullptr);
  if (rc) return rc;
  const char* w = "";
  const bool ok = fast::supported(*setup, &w);
  if (why && why_len > 0) { std::strncpy(why, ok ? "" : w, size_t(why_len)); why[why_len - 1] = 0; }
  return ok ? 1 : 0;
}

void sart_ray_uniforms(uint64_t seed, uint64_t ray, double u[6]) {
  uint32_t w[6];
  ray_words(seed, ray, w);
  for (int i = 0; i < 6; ++i) u[i] = u01(w[i]);
}

int sart_create(const sart_setup_t* setup, const sart_tables_t* tables, int device, sart_handle_t** out) {
  if (!out) return fail(SART_ERR_ARG, "sart_create: out is NULL");
  *out = nullptr;
  if (!tables) return fail(SART_ERR_ARG, "sart_create: tables is NULL");
  int rc = validate(setup, tables);
  if (rc) return rc;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(SART_ERR_CUDA, "no CUDA device available (%s); libsart has no CPU fallback",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(SART_ERR_ARG, "device %d out of range (0..%d)", device, ndev - 1);
  SART_CUDA(cudaSetDevice(device));
  sart_handle* h = new (std::nothrow) sart_handle();
  if (!h) return fail(SART_ERR_NOMEM, "out of host memory");
  h->device = device;
  h->setup = *setup;
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) { delete h; return cuda_fail(e, "cudaGetDeviceProperties"); }
  h->sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) { delete h; return cuda_fail(e, "cudaStreamCreate"); }
  derive_params(h->setup, tables, &h->params);
  if ((rc = upload_tables(h, tables))) { sart_destroy(h); return rc; }
  if ((rc = upload_fast(h, tables))) { sart_destroy(h); return rc; }
  if ((e = cudaMalloc(&h->d_masses, SART_MAX_MASSES * sizeof(double))) != cudaSuccess) { sart_destroy(h); return cuda_fail(e, "cudaMalloc"); }
  h->n_masses = 1;
  h->masses[0] = setup->consts.mAxion;
  if ((e = cudaMemcpyAsync(h->d_masses, h->masses, sizeof(double), cudaMemcpyHostToDevice, h->stream)) != cudaSuccess) { sart_destroy(h); return cuda_fail(e, "cudaMemcpyAsync"); }
  if ((rc = ensure_image(h, 1))) { sart_destroy(h); return rc; }
  if ((rc = autotune(h))) { sart_destroy(h); return rc; }
  if ((e = cudaStreamSynchronize(h->stream)) != cudaSuccess) { sart_destroy(h); return cuda_fail(e, "cudaStreamSynchronize"); }
  *out = h;
  return SART_OK;
}

void sart_destroy(sart_handle_t* h) {
  if (!h) return;
  if (h->device >= 0) cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  sart_comm_destroy(h);
  cudaFree(h->table_blob); cudaFree(h->fast_blob); cudaFree(h->d_masses); cudaFree(h->d_image); cudaFree(h->d_merged);
  cudaFree(h->d_counters); cudaFree(h->d_stage); cudaFree(h->d_rad_w); cudaFree(h->d_rad_n); cudaFree(h->d_rep); cudaFree(h->d_mass_acc);
  cudaFree(h->d_queue); cudaFree(h->d_spec); cudaFree(h->d_spec_rep);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->stream_in) cudaStreamDestroy(h->stream_in);
  if (h->stream_out) cudaStreamDestroy(h->stream_out);
  for (void* e : h->ev) if (e) cudaEventDestroy(static_cast<cudaEvent_t>(e));
  delete h;
}

// The setup-dependent part of a handle: sart_update_setup applies a new setup to it and puts the old one back (host state
// and the device-side records derived from it) if any step fails, so a failed update leaves the handle as it was.
static int apply_setup(sart_handle* h, const sart_setup_t& s, bool retune) {
  h->setup = s;
  rederive_params(h, h->setup, &h->params);
  std::vector<ShellF64> shells(SART_MAX_SHELLS);
  derive_shells(h->setup, shells.data());
  SART_CUDA(cudaStreamSynchronize(h->stream));
  SART_CUDA(cudaMemcpyAsync(static_cast<unsigned char*>(h->table_blob) + h->shell_offset, shells.data(),
                            shells.size() * sizeof(ShellF64), cudaMemcpyHostToDevice, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  int rc = upload_fast(h, nullptr);
  if (rc) return rc;
  if (h->precision >= 1 && !h->fast_ok) h->precision = 0;
  if (h->precision == 2 && !h->f32_ok) h->precision = 1;
  if (retune && !h->compact_user) rc = autotune(h);
  return rc;
}

int sart_update_setup(sart_handle_t* h, const sart_setup_t* setup) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  int rc = validate_update(h, setup);
  if (rc) return rc;
  DeviceGuard dg(h->device);
  const sart_setup_t old = h->setup;
  const int oldPrecision = h->precision, oldCompact = h->compact;
  const double oldSurvival = h->pilot_survival;
  // the pilot run that chooses the kernel variant measures how many rays the bore, pipes and entrance structures remove:
  // repeat it only when that geometry changes (not for every step of an angle or detector-position scan)
  const bool retune = std::memcmp(&old.magnet, &setup->magnet, sizeof old.magnet) != 0 ||
                      std::memcmp(&old.pipes, &setup->pipes, sizeof old.pipes) != 0 ||
                      old.telescope.kind != setup->telescope.kind || old.telescope.nShells != setup->telescope.nShells ||
                      old.testSource.active != setup->testSource.active || old.experiment != setup->experiment;
  rc = apply_setup(h, *setup, retune);
  if (rc) {
    char msg[sizeof g_err];
    std::snprintf(msg, sizeof msg, "%s", g_err);
    h->precision = oldPrecision;
    apply_setup(h, old, false);   // best effort: the old setup was valid for this handle
    h->precision = oldPrecision; h->compact = oldCompact; h->pilot_survival = oldSurvival;
    return fail(rc, "sart_update_setup failed, previous setup kept: %s", msg);
  }
  if (h->n_masses == 1 && h->masses_default) {
    h->masses[0] = setup->consts.mAxion;
    SART_CUDA(cudaMemcpyAsync(h->d_masses, h->masses, sizeof(double), cudaMemcpyHostToDevice, h->stream));
    SART_CUDA(cudaStreamSynchronize(h->stream));
  }
  return SART_OK;
}

int sart_set_axion_masses(sart_handle_t* h, int n, const double* masses_eV) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (n < 1 || n > SART_MAX_MASSES || !masses_eV) return fail(SART_ERR_ARG, "sart_set_axion_masses: need 1..%d masses", SART_MAX_MASSES);
  DeviceGuard dg(h->device);
  SART_CUDA(cudaStreamSynchronize(h->stream));
  int rc = ensure_image(h, n);
  if (rc) {   // the old buffers are gone: fall back to a state every entry point can work with
    h->n_masses = 1;
    if (ensure_image(h, 1) != SART_OK) h->n_masses = 0;
    return rc;
  }
  std::memcpy(h->masses, masses_eV, n * sizeof(double));
  h->n_masses = n;
  h->masses_default = 0;
  SART_CUDA(cudaMemcpyAsync(h->d_masses, h->masses, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

int sart_set_precision(sart_handle_t* h, int mode) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (mode < 0 || mode > 2) return fail(SART_ERR_ARG, "unknown precision mode %d", mode);
  if (mode >= 1 && !h->fast_ok) return fail(SART_ERR_CONFIG, "fast pipeline unavailable for this setup: %s", h->fast_why);
  if (mode == 2 && !h->f32_ok)
    return fail(SART_ERR_CONFIG, "FP32 pipeline unavailable for this setup: shell radii too closely spaced for its radial lookup table");
  h->precision = mode;
  return SART_OK;
}

int sart_has_precision(int mode) { return mode >= 0 && mode <= 2; }

int sart_set_sampler(sart_handle_t* h, int sampler) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (sampler != SART_SAMPLER_INVERSE_CDF && sampler != SART_SAMPLER_ALIAS) return fail(SART_ERR_ARG, "unknown sampler %d", sampler);
  if (sampler == SART_SAMPLER_ALIAS && !h->alias_ok)
    return fail(SART_ERR_CONFIG, "alias tables unavailable (need a solar table with at most 2048 radii and 2048 energies, and a "
                                 "setup the throughput pipelines support)");
  h->sampler = sampler;
  h->ftables.sampler = sampler;
  return SART_OK;
}

void sart_alias_table(const uint32_t* thr, int n, uint32_t* entries) {
  if (!thr || !entries || n < 1) return;
  if (!fast::build_alias_table(thr, n, entries)) std::memset(entries, 0, size_t(n) * 4);
}

int sart_set_retrace(sart_handle_t* h, int mode, double scale) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (mode < 0 || mode > 1 || !(scale >= 0.0) || scale > 1e6) return fail(SART_ERR_ARG, "sart_set_retrace: mode 0/1, scale in [0, 1e6]");
  DeviceGuard dg(h->device);
  h->retrace = mode;
  if (float(scale) != h->retrace_scale) {
    h->retrace_scale = float(scale);
    if (h->fast_ok) {   // the budgets live in the FP32 geometry block
      SART_CUDA(cudaStreamSynchronize(h->stream));
      int rc = upload_fast(h, nullptr);
      if (rc) return rc;
    }
  }
  return SART_OK;
}

int sart_set_compaction(sart_handle_t* h, int mode) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (mode < 0 || mode > 1) return fail(SART_ERR_ARG, "compaction mode must be 0 or 1");
  h->compact = mode;
  h->compact_user = 1;   // an explicit choice survives sart_update_setup
  return SART_OK;
}

void* sart_stream(sart_handle_t* h) { return h ? h->stream : nullptr; }

int sart_build_cdfs(int device, int nR, int nE, const double* radii, const double* energies, const double* emRates,
                    double* fluxRadiusCDF, double* diffFluxCDFs) {
  if (nR < 1 || nE < 1 || !radii || !energies || !emRates || !fluxRadiusCDF || !diffFluxCDFs)
    return fail(SART_ERR_ARG, "sart_build_cdfs: bad argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(SART_ERR_CUDA, "no CUDA device available; libsart has no CPU fallback"); }
  if (device < 0 || device >= ndev) return fail(SART_ERR_ARG, "device %d out of range", device);
  DeviceGuard dg(device);
  const size_t cells = size_t(nR) * nE;
  double *dR = nullptr, *dE = nullptr, *dEm = nullptr, *dTot = nullptr, *dC = nullptr, *dRC = nullptr;
  int rc = SART_OK;
  cudaError_t e;
#define TRY(call) if (rc == SART_OK && (e = (call)) != cudaSuccess) rc = cuda_fail(e, #call)
  TRY(cudaMalloc(&dR, nR * sizeof(double)));
  TRY(cudaMalloc(&dE, nE * sizeof(double)));
  TRY(cudaMalloc(&dEm, cells * sizeof(double)));
  TRY(cudaMalloc(&dTot, nR * sizeof(double)));
  TRY(cudaMalloc(&dC, cells * sizeof(double)));
  TRY(cudaMalloc(&dRC, nR * sizeof(double)));
  TRY(cudaMemcpy(dR, radii, nR * sizeof(double), cudaMemcpyHostToDevice));
  TRY(cudaMemcpy(dE, energies, nE * sizeof(double), cudaMemcpyHostToDevice));
  TRY(cudaMemcpy(dEm, emRates, cells * sizeof(double), cudaMemcpyHostToDevice));
  TRY(launch_build_cdfs(nR, nE, dR, dE, dEm, dTot, dC, dRC, nullptr));
  TRY(cudaDeviceSynchronize());
  TRY(cudaMemcpy(diffFluxCDFs, dC, cells * sizeof(double), cudaMemcpyDeviceToHost));
  TRY(cudaMemcpy(fluxRadiusCDF, dRC, nR * sizeof(double), cudaMemcpyDeviceToHost));
#undef TRY
  cudaFree(dR); cudaFree(dE); cudaFree(dEm); cudaFree(dTot); cudaFree(dC); cudaFree(dRC);
  return rc;
}

int sart_emission_rates(int device, int nR, const double* temp, const double* rho, const double* frac, int nE,
                        const double* energies, uint32_t processes, double g_ae, double gagamma, double ganuclei,
                        double* emRates) {
  if (nR < 1 || nE < 1 || !temp || !rho || !frac || !energies || !emRates) return fail(SART_ERR_ARG, "sart_emission_rates: bad argument");
  if (processes == 0 || (processes >> 6)) return fail(SART_ERR_ARG, "sart_emission_rates: unknown process bits 0x%x", processes);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(SART_ERR_CUDA, "no CUDA device available; libsart has no CPU fallback"); }
  if (device < 0 || device >= ndev) return fail(SART_ERR_ARG, "device %d out of range", device);
  DeviceGuard dg(device);
  const size_t cells = size_t(nR) * nE;
  double *dT = nullptr, *dRho = nullptr, *dF = nullptr, *dE = nullptr, *dEm = nullptr;
  void* dSt = nullptr;
  int rc = SART_OK;
  cudaError_t e;
#define TRY(call) if (rc == SART_OK && (e = (call)) != cudaSuccess) rc = cuda_fail(e, #call)
  TRY(cudaMalloc(&dT, nR * sizeof(double)));
  TRY(cudaMalloc(&dRho, nR * sizeof(double)));
  TRY(cudaMalloc(&dF, size_t(nR) * 29 * sizeof(double)));
  TRY(cudaMalloc(&dE, nE * sizeof(double)));
  TRY(cudaMalloc(&dEm, cells * sizeof(double)));
  TRY(cudaMalloc(&dSt, size_t(nR) * 80));
  TRY(cudaMemcpy(dT, temp, nR * sizeof(double), cudaMemcpyHostToDevice));
  TRY(cudaMemcpy(dRho, rho, nR * sizeof(double), cudaMemcpyHostToDevice));
  TRY(cudaMemcpy(dF, frac, size_t(nR) * 29 * sizeof(double), cudaMemcpyHostToDevice));
  TRY(cudaMemcpy(dE, energies, nE * sizeof(double), cudaMemcpyHostToDevice));
  TRY(launch_emission_rates(nR, nE, dT, dRho, dF, dE, processes, g_ae, gagamma, ganuclei, dSt, dEm, nullptr));
  TRY(cudaDeviceSynchronize());
  TRY(cudaMemcpy(emRates, dEm, cells * sizeof(double), cudaMemcpyDeviceToHost));
#undef TRY
  cudaFree(dT); cudaFree(dRho); cudaFree(dF); cudaFree(dE); cudaFree(dEm); cudaFree(dSt);
  return rc;
}

static int check_out(const sart_ray_out_t* out) {
  if (!out || !out->x || !out->y || !out->w || !out->code || !out->shell)
    return fail(SART_ERR_ARG, "sart_ray_out_t: x, y, w, code and shell are required");
  return SART_OK;
}

// One batch of pre-sampled rays, device pointers. Precision 2: the FP32 kernel writes every record and queues the rays
// whose decision margins are inside their error budgets; the exact kernel then overwrites those records.
static int launch_presampled(sart_handle* h, size_t m, const double* dO, const double* dX, const double* dE,
                             const sart_ray_out_t& dev) {
  if (h->precision == 2 && h->ftables.energies) {
    if (m > kRetraceChunk) return fail(SART_ERR_ARG, "sart_trace_presampled: at most 2^31 rays per call in precision mode 2");
    fast::FastTables ft = h->ftables;
    int rc = begin_queue(h, m, &ft.rq);
    if (rc) return rc;
    SART_CUDA(launch_presampled_f32(h->fparams, h->geo32, ft, h->masses[0], m, dO, dX, dE, dev, h->sm_count, h->stream));
    if (ft.rq.cap)
      SART_CUDA(launch_retrace_presampled(h->params, h->tables, h->masses[0], m, dO, dX, dE, ft.rq, dev, h->sm_count, h->stream));
  } else {
    SART_CUDA(launch_presampled_exact(h->params, h->tables, h->masses[0], m, dO, dX, dE, dev, h->stream));
  }
  return SART_OK;
}

int sart_trace_presampled_dev(sart_handle_t* h, size_t n, const double* d_origin, const double* d_exit,
                              const double* d_energy, const sart_ray_out_t* d_out) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  int rc = check_out(d_out);
  if (rc) return rc;
  if (n && (!d_origin || !d_exit || !d_energy)) return fail(SART_ERR_ARG, "sart_trace_presampled: NULL input");
  DeviceGuard dg(h->device);
  return launch_presampled(h, n, d_origin, d_exit, d_energy, *d_out);
}

// Lays a device-side sart_ray_out_t over the staging buffer; returns bytes used.
static size_t carve_out(unsigned char* base, size_t n, const sart_ray_out_t& host, sart_ray_out_t* dev) {
  size_t off = 0;
  auto takeD = [&](double* hostp) -> double* {
    if (!hostp) return nullptr;
    double* p = reinterpret_cast<double*>(base + off);
    off = align256(off + n * sizeof(double));
    return p;
  };
  auto takeI = [&](int32_t* hostp) -> int32_t* {
    if (!hostp) return nullptr;
    int32_t* p = reinterpret_cast<int32_t*>(base + off);
    off = align256(off + n * sizeof(int32_t));
    return p;
  };
  dev->x = takeD(host.x); dev->y = takeD(host.y); dev->w = takeD(host.w);
  dev->code = takeI(host.code); dev->shell = takeI(host.shell);
  dev->energy = takeD(host.energy); dev->reflect = takeD(host.reflect); dev->transMagnet = takeD(host.transMagnet);
  dev->yaw = takeD(host.yaw); dev->alpha1 = takeD(host.alpha1); dev->alpha2 = takeD(host.alpha2);
  dev->pathCB = takeD(host.pathCB); dev->r = takeD(host.r); dev->deviationDet = takeD(host.deviationDet);
  dev->transProbArgon = takeD(host.transProbArgon);
  return off;
}

static int copy_out(sart_handle* h, size_t n, const sart_ray_out_t& host, const sart_ray_out_t& dev) {
#define CPD(f) if (host.f) SART_CUDA(cudaMemcpyAsync(host.f, dev.f, n * sizeof(*host.f), cudaMemcpyDeviceToHost, h->stream))
  CPD(x); CPD(y); CPD(w); CPD(code); CPD(shell); CPD(energy); CPD(reflect); CPD(transMagnet); CPD(yaw); CPD(alpha1);
  CPD(alpha2); CPD(pathCB); CPD(r); CPD(deviationDet); CPD(transProbArgon);
#undef CPD
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

// Offsets a host-side sart_ray_out_t by `a` rays.
static sart_ray_out_t offset_out(const sart_ray_out_t& o, size_t a) {
  sart_ray_out_t r = o;
#define OFF(f) if (r.f) r.f += a
  OFF(x); OFF(y); OFF(w); OFF(code); OFF(shell); OFF(energy); OFF(reflect); OFF(transMagnet); OFF(yaw); OFF(alpha1);
  OFF(alpha2); OFF(pathCB); OFF(r); OFF(deviationDet); OFF(transProbArgon);
#undef OFF
  return r;
}


int sart_trace_presampled(sart_handle_t* h, size_t n, const double* origin, const double* exitxy, const double* energy,
                          const sart_ray_out_t* out) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  int rc = check_out(out);
  if (rc) return rc;
  if (n == 0) return SART_OK;
  if (!origin || !exitxy || !energy) return fail(SART_ERR_ARG, "sart_trace_presampled: NULL input");
  DeviceGuard dg(h->device);
  // Chunks of up to 1 Mi rays through two device-side buffers: the host->device copies of chunk k+1, the kernel of
  // chunk k and the device->host copies of chunk k-1 run on three streams at once (PCIe is full duplex; with pinned
  // host arrays the call is bound by the larger of the two directions, 48 B/ray in, instead of by their sum).
  const size_t chunk = size_t(1) << 20, m0 = n < chunk ? n : chunk;
  const size_t inBytes = align256(3 * m0 * sizeof(double)) + align256(2 * m0 * sizeof(double)) + align256(m0 * sizeof(double));
  sart_ray_out_t probe;
  const size_t outBytes = carve_out(nullptr, m0, *out, &probe);
  const size_t bufBytes = inBytes + outBytes;
  const int nbuf = n > chunk ? 2 : 1;
  if ((rc = ensure_stage(h, nbuf * bufBytes))) return rc;
  if (nbuf == 2 && !h->stream_in) {
    SART_CUDA(cudaStreamCreateWithFlags(&h->stream_in, cudaStreamNonBlocking));
    SART_CUDA(cudaStreamCreateWithFlags(&h->stream_out, cudaStreamNonBlocking));
    for (int i = 0; i < 6; ++i) SART_CUDA(cudaEventCreateWithFlags(reinterpret_cast<cudaEvent_t*>(&h->ev[i]), cudaEventDisableTiming));
  }
  cudaStream_t sIn = nbuf == 2 ? h->stream_in : h->stream, sOut = nbuf == 2 ? h->stream_out : h->stream;
  auto ev = [&](int kind, int b) { return static_cast<cudaEvent_t>(h->ev[kind * 2 + b]); };   // 0 in, 1 kernel, 2 out
  size_t k = 0;
  for (size_t a = 0; a < n; a += chunk, ++k) {
    const size_t m = n - a < chunk ? n - a : chunk;
    const int b = int(k & 1);
    unsigned char* base = static_cast<unsigned char*>(h->d_stage) + size_t(b) * bufBytes;
    double* dO = reinterpret_cast<double*>(base);
    double* dX = reinterpret_cast<double*>(base + align256(3 * m0 * sizeof(double)));
    double* dE = reinterpret_cast<double*>(base + align256(3 * m0 * sizeof(double)) + align256(2 * m0 * sizeof(double)));
    sart_ray_out_t dev;
    carve_out(base + inBytes, m, *out, &dev);
    if (nbuf == 2 && k >= 2) SART_CUDA(cudaStreamWaitEvent(sIn, ev(1, b), 0));      // kernel of chunk k-2 has read this buffer
    for (int c = 0; c < 3; ++c) SART_CUDA(cudaMemcpyAsync(dO + c * m, origin + c * n + a, m * sizeof(double), cudaMemcpyHostToDevice, sIn));
    for (int c = 0; c < 2; ++c) SART_CUDA(cudaMemcpyAsync(dX + c * m, exitxy + c * n + a, m * sizeof(double), cudaMemcpyHostToDevice, sIn));
    SART_CUDA(cudaMemcpyAsync(dE, energy + a, m * sizeof(double), cudaMemcpyHostToDevice, sIn));
    if (nbuf == 2) {
      SART_CUDA(cudaEventRecord(ev(0, b), sIn));
      SART_CUDA(cudaStreamWaitEvent(h->stream, ev(0, b), 0));
      if (k >= 2) SART_CUDA(cudaStreamWaitEvent(h->stream, ev(2, b), 0));           // outputs of chunk k-2 have left this buffer
    }
    if ((rc = launch_presampled(h, m, dO, dX, dE, dev))) return rc;
    if (nbuf == 2) {
      SART_CUDA(cudaEventRecord(ev(1, b), h->stream));
      SART_CUDA(cudaStreamWaitEvent(sOut, ev(1, b), 0));
    }
    const sart_ray_out_t host = offset_out(*out, a);
#define CPD(f) if (host.f) SART_CUDA(cudaMemcpyAsync(host.f, dev.f, m * sizeof(*host.f), cudaMemcpyDeviceToHost, sOut))
    CPD(x); CPD(y); CPD(w); CPD(code); CPD(shell); CPD(energy); CPD(reflect); CPD(transMagnet); CPD(yaw); CPD(alpha1);
    CPD(alpha2); CPD(pathCB); CPD(r); CPD(deviationDet); CPD(transProbArgon);
#undef CPD
    if (nbuf == 2) SART_CUDA(cudaEventRecord(ev(2, b), sOut));
  }
  if (nbuf == 2) { SART_CUDA(cudaStreamSynchronize(sIn)); SART_CUDA(cudaStreamSynchronize(sOut)); }
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

int sart_trace_mc_rays(sart_handle_t* h, uint64_t first_ray, size_t n, uint64_t seed, const sart_ray_out_t* out) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  int rc = check_out(out);
  if (rc) return rc;
  if (n == 0) return SART_OK;
  DeviceGuard dg(h->device);
  if (h->sampler == SART_SAMPLER_ALIAS && h->precision != 2)
    return fail(SART_ERR_CONFIG, "the alias sampler needs precision mode 2");
  sart_ray_out_t probe;
  const size_t outBytes = carve_out(nullptr, n, *out, &probe);
  if ((rc = ensure_stage(h, outBytes))) return rc;
  sart_ray_out_t dev;
  carve_out(static_cast<unsigned char*>(h->d_stage), n, *out, &dev);
  if (h->precision == 2) {
    if (n > kRetraceChunk) return fail(SART_ERR_ARG, "sart_trace_mc_rays: at most 2^31 rays per call");
    fast::FastTables ft = h->ftables;
    const bool alias = h->sampler == SART_SAMPLER_ALIAS;   // another ray <-> index mapping than the exact pipeline's: no re-trace
    if (!alias && (rc = begin_queue(h, n, &ft.rq))) return rc;
    SART_CUDA(launch_mc_rays_f32(h->fparams, h->geo32, ft, h->masses[0], first_ray, n, seed, dev, h->sm_count, h->stream));
    if (ft.rq.cap)
      SART_CUDA(launch_retrace_mc_rays(h->params, h->tables, h->masses[0], first_ray, n, seed, nullptr, ft.rq, dev, h->sm_count, h->stream));
  } else if (h->precision == 1) {
    SART_CUDA(launch_mc_rays_fast(h->fparams, h->ftables, h->masses[0], first_ray, n, seed, dev, h->sm_count, h->stream));
  } else {
    SART_CUDA(launch_mc_rays_exact(h->params, h->tables, h->masses[0], first_ray, n, seed, dev, h->stream));
  }
  return copy_out(h, n, *out, dev);
}

int sart_trace_mc_passed(sart_handle_t* h, uint64_t first_ray, uint64_t n, uint64_t seed, size_t capacity,
                         const sart_passed_out_t* out, uint64_t* n_passed, sart_counters_t* counters) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (!out || !n_passed) return fail(SART_ERR_ARG, "sart_trace_mc_passed: out and n_passed are required");
  *n_passed = 0;
  if (h->precision != 2) return fail(SART_ERR_CONFIG, "sart_trace_mc_passed: precision mode 2");
  if (h->sampler != SART_SAMPLER_INVERSE_CDF || h->n_masses != 1)
    return fail(SART_ERR_CONFIG, "sart_trace_mc_passed: inverse-CDF sampler and a single axion mass");
  if (n > (uint64_t(1) << 32)) return fail(SART_ERR_ARG, "sart_trace_mc_passed: at most 2^32 rays per call (32-bit ray offsets)");
  DeviceGuard dg(h->device);
  // the fields of sart_passed_out_t in declaration order: host pointer and element size
  void* const hostp[15] = {out->ray, out->x, out->y, out->w, out->shell, out->energy, out->r, out->reflect, out->transMagnet,
                           out->yaw, out->alpha1, out->alpha2, out->pathCB, out->deviationDet, out->transProbArgon};
  const size_t esize[15] = {4, 4, 4, 4, 1, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4};
  // chunks of 2^24 rays through two device buffers: the kernels of chunk k + 1 run while the records of chunk k (whose
  // number the host learns from a 4-byte read) cross PCIe on a second stream
  const uint64_t chunk = std::min<uint64_t>(std::max<uint64_t>(n, 1), uint64_t(1) << 24);
  size_t off[15], bufBytes = 256;   // [0, 256): the record count of the chunk
  for (int f = 0; f < 15; ++f) { off[f] = bufBytes; if (hostp[f]) bufBytes += align256(size_t(chunk) * esize[f]); }
  const size_t cntOff = 2 * bufBytes;
  int rc = ensure_stage(h, cntOff + align256(sizeof(sart_counters_t)));
  if (rc) return rc;
  if (!h->stream_in) {
    SART_CUDA(cudaStreamCreateWithFlags(&h->stream_in, cudaStreamNonBlocking));
    SART_CUDA(cudaStreamCreateWithFlags(&h->stream_out, cudaStreamNonBlocking));
    for (int i = 0; i < 6; ++i) SART_CUDA(cudaEventCreateWithFlags(reinterpret_cast<cudaEvent_t*>(&h->ev[i]), cudaEventDisableTiming));
  }
  if (!h->h_stage) { SART_CUDA(cudaHostAlloc(&h->h_stage, 256, cudaHostAllocDefault)); h->h_stage_bytes = 256; }
  unsigned int* hcount = static_cast<unsigned int*>(h->h_stage);
  unsigned char* base = static_cast<unsigned char*>(h->d_stage);
  sart_counters_t* dCnt = reinterpret_cast<sart_counters_t*>(base + cntOff);
  SART_CUDA(cudaMemsetAsync(dCnt, 0, sizeof(sart_counters_t), h->stream));
  auto evDone = [&](int b) { return static_cast<cudaEvent_t>(h->ev[b]); };
  auto evCopied = [&](int b) { return static_cast<cudaEvent_t>(h->ev[2 + b]); };
  auto devOut = [&](int b) {
    sart_passed_out_t d;
    unsigned char* p = base + size_t(b) * bufBytes;
    void** dp[15] = {(void**)&d.ray, (void**)&d.x, (void**)&d.y, (void**)&d.w, (void**)&d.shell, (void**)&d.energy, (void**)&d.r,
                     (void**)&d.reflect, (void**)&d.transMagnet, (void**)&d.yaw, (void**)&d.alpha1, (void**)&d.alpha2,
                     (void**)&d.pathCB, (void**)&d.deviationDet, (void**)&d.transProbArgon};
    for (int f = 0; f < 15; ++f) *dp[f] = hostp[f] ? static_cast<void*>(p + off[f]) : nullptr;
    return d;
  };
  uint64_t total = 0;
  bool overflow = false;
  auto finish = [&](uint64_t k) -> int {   // chunk k: wait for its kernels, learn its record count, send the records home
    const int b = int(k & 1);
    SART_CUDA(cudaEventSynchronize(evDone(b)));
    const uint64_t c = std::min<uint64_t>(hcount[b], chunk);
    const uint64_t room = total < capacity ? capacity - total : 0;
    const uint64_t take = std::min(c, room);
    if (take < c) overflow = true;
    unsigned char* p = base + size_t(b) * bufBytes;
    for (int f = 0; f < 15 && take; ++f)
      if (hostp[f])
        SART_CUDA(cudaMemcpyAsync(static_cast<unsigned char*>(hostp[f]) + total * esize[f], p + off[f], take * esize[f],
                                  cudaMemcpyDeviceToHost, h->stream_out));
    SART_CUDA(cudaEventRecord(evCopied(b), h->stream_out));
    total += c;
    return SART_OK;
  };
  uint64_t k = 0;
  for (uint64_t done = 0; done < n; done += chunk, ++k) {
    const uint64_t m = std::min<uint64_t>(n - done, chunk);
    const int b = int(k & 1);
    unsigned int* dCount = reinterpret_cast<unsigned int*>(base + size_t(b) * bufBytes);
    if (k >= 2) SART_CUDA(cudaStreamWaitEvent(h->stream, evCopied(b), 0));   // the records of chunk k - 2 have left this buffer
    SART_CUDA(cudaMemsetAsync(dCount, 0, 256, h->stream));
    fast::FastTables ft = h->ftables;
    if ((rc = begin_queue(h, m, &ft.rq))) return rc;
    const sart_passed_out_t d = devOut(b);
    SART_CUDA(launch_mc_passed_f32(h->fparams, h->geo32, ft, h->masses[0], first_ray + done, m, seed, d, dCount, unsigned(chunk),
                                   uint32_t(done), dCnt, h->sm_count, h->stream));
    if (ft.rq.cap)
      SART_CUDA(launch_retrace_mc_passed(h->params, h->tables, h->masses[0], first_ray + done, seed, ft.rq, d, dCount, unsigned(chunk),
                                         uint32_t(done), dCnt, h->sm_count, h->stream));
    SART_CUDA(cudaMemcpyAsync(hcount + b, dCount, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->stream));
    SART_CUDA(cudaEventRecord(evDone(b), h->stream));
    if (k >= 1 && (rc = finish(k - 1))) return rc;
  }
  if (k >= 1 && (rc = finish(k - 1))) return rc;
  if (counters) SART_CUDA(cudaMemcpyAsync(counters, dCnt, sizeof(sart_counters_t), cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream_out));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  *n_passed = total;
  if (overflow) return fail(SART_ERR_ARG, "sart_trace_mc_passed: %llu rays passed, the output arrays hold %zu", (unsigned long long)total, capacity);
  return SART_OK;
}

int sart_trace_words(sart_handle_t* h, size_t n, const uint32_t* words, int late_energy, const sart_ray_out_t* out,
                     int32_t* emission_shell) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  int rc = check_out(out);
  if (rc) return rc;
  if (n == 0) return SART_OK;
  if (!words) return fail(SART_ERR_ARG, "sart_trace_words: words is NULL");
  if (h->precision == 1) return fail(SART_ERR_CONFIG, "sart_trace_words: precision mode 0 or 2 (mode 1 runs the same integer search code as mode 2)");
  if (h->setup.testSource.active) return fail(SART_ERR_CONFIG, "sart_trace_words: solar source only");
  if (late_energy && h->precision != 2) return fail(SART_ERR_CONFIG, "sart_trace_words: late_energy is a variant of precision mode 2");
  DeviceGuard dg(h->device);
  sart_ray_out_t probe;
  const size_t outBytes = carve_out(nullptr, n, *out, &probe);
  const size_t wBytes = align256(6 * n * sizeof(uint32_t)), eBytes = align256(n * sizeof(int32_t));
  if ((rc = ensure_stage(h, outBytes + wBytes + eBytes))) return rc;
  unsigned char* base = static_cast<unsigned char*>(h->d_stage);
  sart_ray_out_t dev;
  carve_out(base, n, *out, &dev);
  uint32_t* dW = reinterpret_cast<uint32_t*>(base + outBytes);
  int32_t* dEmit = emission_shell ? reinterpret_cast<int32_t*>(base + outBytes + wBytes) : nullptr;
  SART_CUDA(cudaMemcpyAsync(dW, words, 6 * n * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  if (h->precision == 2) {
    if (n > kRetraceChunk) return fail(SART_ERR_ARG, "sart_trace_words: at most 2^31 rays per call");
    fast::FastTables ft = h->ftables;
    if (h->sampler != SART_SAMPLER_ALIAS && (rc = begin_queue(h, n, &ft.rq))) return rc;
    SART_CUDA(launch_mc_rays_f32(h->fparams, h->geo32, ft, h->masses[0], 0, n, 0, dev, h->sm_count, h->stream, dW,
                                 late_energy != 0, dEmit));
    if (ft.rq.cap)
      SART_CUDA(launch_retrace_mc_rays(h->params, h->tables, h->masses[0], 0, n, 0, dW, ft.rq, dev, h->sm_count, h->stream));
  } else {
    SART_CUDA(launch_mc_rays_exact(h->params, h->tables, h->masses[0], 0, n, 0, dev, h->stream, dW, dEmit));
  }
  if (dEmit) SART_CUDA(cudaMemcpyAsync(emission_shell, dEmit, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  return copy_out(h, n, *out, dev);
}

int sart_trace_mc(sart_handle_t* h, uint64_t first_ray, uint64_t n_rays, uint64_t seed) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (!h->d_image) return fail(SART_ERR_NOMEM, "the image buffers of this handle could not be allocated");
  DeviceGuard dg(h->device);
  if (h->sampler == SART_SAMPLER_ALIAS && (h->precision != 2 || h->n_masses > 1))
    return fail(SART_ERR_CONFIG, "the alias sampler needs precision mode 2 and a single axion mass");
  if (h->spec.eW && h->n_masses > 1) return fail(SART_ERR_CONFIG, "sart_trace_mc: the spectra need a single axion mass");
  // Precision 2: launches of at most 2^31 rays, each followed on the same stream by the exact pipeline's pass over the
  // rays the FP32 kernel queued as uncertain (it adds them to the same image and counters). Not with the alias sampler,
  // whose ray <-> index mapping is not the exact pipeline's.
  const bool retrace = h->precision == 2 && h->retrace && h->sampler != SART_SAMPLER_ALIAS;
  if (h->precision >= 1 && h->n_masses > 1) {
    const size_t plane = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS, accLen = plane * SART_MAX_MASSES;
    if (!h->d_mass_acc) {
      SART_CUDA(cudaMalloc(&h->d_mass_acc, 2 * accLen * sizeof(double)));
      SART_CUDA(cudaMemsetAsync(h->d_mass_acc, 0, 2 * accLen * sizeof(double), h->stream));
    }
    if (h->precision == 2) {
      for (uint64_t done = 0; done < n_rays; done += kRetraceChunk) {
        const uint64_t n = std::min<uint64_t>(n_rays - done, kRetraceChunk);
        fast::FastTables ft = h->ftables;
        int rc = retrace ? begin_queue(h, n, &ft.rq) : SART_OK;
        if (rc) return rc;
        SART_CUDA(launch_mc_image_f32_masses(h->fparams, h->geo32, ft, h->n_masses, h->d_masses, first_ray + done, n, seed,
                                             h->d_mass_acc, h->d_mass_acc + accLen, h->d_counters, h->sm_count, h->stream));
        if (ft.rq.cap)
          SART_CUDA(launch_retrace_mc_image(h->params, h->tables, h->n_masses, h->d_masses, first_ray + done, seed, ft.rq,
                                            h->d_image, h->d_image_w2, h->d_counters, h->sm_count, h->stream));
      }
    } else {
      SART_CUDA(launch_mc_image_fast_masses(h->fparams, h->ftables, h->n_masses, h->d_masses, first_ray, n_rays, seed,
                                            h->d_mass_acc, h->d_mass_acc + accLen, h->d_counters, h->sm_count, h->stream));
    }
    SART_CUDA(launch_fold_mass_acc(h->d_mass_acc, h->d_mass_acc + accLen, h->n_masses, plane, h->d_image, h->d_image_w2,
                                   h->stream));
    return SART_OK;
  }
  if (h->precision >= 1) {
    int rc = ensure_replicas(h);
    if (rc) return rc;
    const size_t plane = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS;
    fast::FastTables ft = h->ftables;
    ft.spec = h->spec_rep;   // the spectra replicas, or off
    double *img = h->d_image, *img2 = h->d_image_w2;
    if (h->n_rep > 1) {
      ft.nImgRep = h->n_rep; ft.imgRepStride = h->rep_stride;
      img = h->d_rep; img2 = h->d_rep + size_t(h->n_rep) * h->rep_stride;
    }
    if (h->precision == 2) {
      for (uint64_t done = 0; done < n_rays; done += kRetraceChunk) {
        const uint64_t n = std::min<uint64_t>(n_rays - done, kRetraceChunk);
        if (retrace && (rc = begin_queue(h, n, &ft.rq))) return rc;
        SART_CUDA(launch_mc_image_f32(h->fparams, h->geo32, ft, h->masses[0], first_ray + done, n, seed, img, img2,
                                      h->d_counters, h->sm_count, h->compact != 0, h->stream));
        if (ft.rq.cap) {
          Tables et = h->tables;
          if (!ft.rad.w) et.rad = RadialHist{};
          et.spec = h->spec;   // the re-traced rays belong in the spectra as much as in the image
          SART_CUDA(launch_retrace_mc_image(h->params, et, 1, h->d_masses, first_ray + done, seed, ft.rq, h->d_image,
                                            h->d_image_w2, h->d_counters, h->sm_count, h->stream));
        }
      }
    } else {
      SART_CUDA(launch_mc_image_fast(h->fparams, ft, h->masses[0], first_ray, n_rays, seed, img, img2, h->d_counters,
                                     h->sm_count, h->compact != 0, h->stream));
    }
    if (h->n_rep > 1)
      SART_CUDA(launch_fold_replicas(img, img2, h->n_rep, h->rep_stride, plane, h->d_image, h->d_image_w2, h->stream));
    if (h->spec.eW) SART_CUDA(launch_fold_spectra(h->spec_rep, h->spec_e1, h->spec, h->stream));
    return SART_OK;
  }
  Tables et = h->tables;
  et.spec = h->spec;
  SART_CUDA(launch_mc_image_exact(h->params, et, h->n_masses, h->d_masses, first_ray, n_rays, seed, h->d_image,
                                  h->d_image_w2, h->d_counters, h->sm_count, h->stream));
  return SART_OK;
}

int sart_reset_image(sart_handle_t* h) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  DeviceGuard dg(h->device);
  const size_t len = size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
  SART_CUDA(cudaMemsetAsync(h->d_image, 0, 2 * len * sizeof(double), h->stream));   // image | w^2 image: one block
  SART_CUDA(cudaMemsetAsync(h->d_counters, 0, size_t(h->n_masses) * sizeof(sart_counters_t), h->stream));
  if (h->rad_bins > 0) {
    SART_CUDA(cudaMemsetAsync(h->d_rad_w, 0, size_t(h->rad_bins) * sizeof(double), h->stream));
    SART_CUDA(cudaMemsetAsync(h->d_rad_n, 0, size_t(h->rad_bins) * sizeof(unsigned long long), h->stream));
  }
  if (h->spec.eW) SART_CUDA(cudaMemsetAsync(h->d_spec, 0, spectra_bytes(h->spec_e1, 1, 1), h->stream));
  return SART_OK;
}

int sart_enable_spectra(sart_handle_t* h, int on) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  DeviceGuard dg(h->device);
  SART_CUDA(cudaStreamSynchronize(h->stream));
  cudaFree(h->d_spec); cudaFree(h->d_spec_rep);
  h->d_spec = nullptr; h->d_spec_rep = nullptr; h->spec = Spectra{}; h->spec_rep = Spectra{}; h->spec_e1 = 0;
  if (!on) return SART_OK;
  const int nE1 = h->params.nEnergies + 1;
  // Replicas of the throughput kernels (powers of two; SART_SPEC_E_REPLICAS / SART_SPEC_S_REPLICAS override them for
  // measurements). The energy bins spread the passed rays over hundreds of addresses, like the focal spot the image
  // replicas serve: one replica per block residue. The shell bins are a handful of addresses (4 for LLNL): one per warp.
  auto pow2 = [](const char* env, int dflt) {
    int n = dflt;
    if (const char* e = std::getenv(env)) n = std::max(1, std::min(1 << 16, std::atoi(e)));
    int p = 1;
    while (p * 2 <= n) p *= 2;
    return p;
  };
  const int eRep = pow2("SART_SPEC_E_REPLICAS", 32), sRep = pow2("SART_SPEC_S_REPLICAS", 1024);
  const uint32_t eStride = uint32_t((nE1 + 31) & ~31);
  SART_CUDA(cudaMalloc(&h->d_spec, spectra_bytes(nE1, 1, 1)));
  SART_CUDA(cudaMalloc(&h->d_spec_rep, spectra_bytes(int(eStride), eRep, sRep)));
  SART_CUDA(cudaMemsetAsync(h->d_spec, 0, spectra_bytes(nE1, 1, 1), h->stream));
  SART_CUDA(cudaMemsetAsync(h->d_spec_rep, 0, spectra_bytes(int(eStride), eRep, sRep), h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  h->spec = carve_spectra(h->d_spec, nE1, 1, 1);
  h->spec_rep = carve_spectra(h->d_spec_rep, int(eStride), eRep, sRep);
  h->spec_e1 = nE1;
  return SART_OK;
}

int sart_read_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                      double* shell_sum_w, uint64_t* shell_counts) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (!h->spec.eW) return fail(SART_ERR_ARG, "sart_read_spectra: no spectra enabled (sart_enable_spectra)");
  DeviceGuard dg(h->device);
  const size_t e = size_t(h->spec_e1) * 8, s = size_t(SART_MAX_SHELLS) * 8;
  if (energy_sum_w) SART_CUDA(cudaMemcpyAsync(energy_sum_w, h->spec.eW, e, cudaMemcpyDeviceToHost, h->stream));
  if (energy_sum_w2) SART_CUDA(cudaMemcpyAsync(energy_sum_w2, h->spec.eW2, e, cudaMemcpyDeviceToHost, h->stream));
  if (energy_counts) SART_CUDA(cudaMemcpyAsync(energy_counts, h->spec.eN, e, cudaMemcpyDeviceToHost, h->stream));
  if (shell_sum_w) SART_CUDA(cudaMemcpyAsync(shell_sum_w, h->spec.sW, s, cudaMemcpyDeviceToHost, h->stream));
  if (shell_counts) SART_CUDA(cudaMemcpyAsync(shell_counts, h->spec.sN, s, cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

int sart_enable_radial_hist(sart_handle_t* h, int nbins, double r_max) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (nbins < 0 || nbins > (1 << 24) || (nbins > 0 && !(r_max > 0.0))) return fail(SART_ERR_ARG, "sart_enable_radial_hist: bad argument");
  DeviceGuard dg(h->device);
  SART_CUDA(cudaStreamSynchronize(h->stream));
  cudaFree(h->d_rad_w); cudaFree(h->d_rad_n);
  h->d_rad_w = nullptr; h->d_rad_n = nullptr; h->rad_bins = 0; h->rad_rmax = 0.0;
  RadialHist r{};
  if (nbins > 0) {
    SART_CUDA(cudaMalloc(&h->d_rad_w, size_t(nbins) * sizeof(double)));
    SART_CUDA(cudaMalloc(&h->d_rad_n, size_t(nbins) * sizeof(unsigned long long)));
    SART_CUDA(cudaMemsetAsync(h->d_rad_w, 0, size_t(nbins) * sizeof(double), h->stream));
    SART_CUDA(cudaMemsetAsync(h->d_rad_n, 0, size_t(nbins) * sizeof(unsigned long long), h->stream));
    h->rad_bins = nbins; h->rad_rmax = r_max;
    r.w = h->d_rad_w; r.n = h->d_rad_n; r.invStep = double(nbins) / r_max; r.nbins = nbins;
  }
  h->tables.rad = r;
  h->ftables.rad = r;
  return SART_OK;
}

int sart_read_radial_hist(sart_handle_t* h, double* sum_w, uint64_t* counts) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (h->rad_bins < 1) return fail(SART_ERR_ARG, "sart_read_radial_hist: no radial histogram enabled");
  DeviceGuard dg(h->device);
  if (sum_w) SART_CUDA(cudaMemcpyAsync(sum_w, h->d_rad_w, size_t(h->rad_bins) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (counts) SART_CUDA(cudaMemcpyAsync(counts, h->d_rad_n, size_t(h->rad_bins) * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

double* sart_image_dev(sart_handle_t* h) { return h ? h->d_image : nullptr; }
double* sart_image_w2_dev(sart_handle_t* h) { return h ? h->d_image_w2 : nullptr; }
void* sart_counters_dev(sart_handle_t* h) { return h ? h->d_counters : nullptr; }
size_t sart_image_len(sart_handle_t* h) { return h ? size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS : 0; }

int sart_read_image(sart_handle_t* h, double* image, double* image_w2, sart_counters_t* counters) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  DeviceGuard dg(h->device);
  const size_t len = size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
  if (image) SART_CUDA(cudaMemcpyAsync(image, h->d_image, len * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (image_w2) SART_CUDA(cudaMemcpyAsync(image_w2, h->d_image_w2, len * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (counters) SART_CUDA(cudaMemcpyAsync(counters, h->d_counters, size_t(h->n_masses) * sizeof(sart_counters_t), cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

int sart_prepare_heatmap(sart_handle_t* h, int rows, int cols, double start_x, double stop_x, double start_y,
                         double stop_y, size_t n, const double* X, const double* Y, const double* W, double norm,
                         double* result, uint64_t* n_out_of_range) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (rows < 1 || cols < 1 || !result || (n && (!X || !Y || !W))) return fail(SART_ERR_ARG, "sart_prepare_heatmap: bad argument");
  DeviceGuard dg(h->device);
  const size_t cells = size_t(rows) * cols;
  const size_t bytes = align256(cells * sizeof(double)) + 256 + 3 * align256(n * sizeof(double));
  int rc = ensure_stage(h, bytes);
  if (rc) return rc;
  unsigned char* base = static_cast<unsigned char*>(h->d_stage);
  double* dRes = reinterpret_cast<double*>(base);
  unsigned long long* dBad = reinterpret_cast<unsigned long long*>(base + align256(cells * sizeof(double)));
  double* dX = reinterpret_cast<double*>(base + align256(cells * sizeof(double)) + 256);
  double* dY = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(dX) + align256(n * sizeof(double)));
  double* dW = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(dY) + align256(n * sizeof(double)));
  SART_CUDA(cudaMemsetAsync(dRes, 0, align256(cells * sizeof(double)) + 256, h->stream));
  if (n) {
    SART_CUDA(cudaMemcpyAsync(dX, X, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    SART_CUDA(cudaMemcpyAsync(dY, Y, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    SART_CUDA(cudaMemcpyAsync(dW, W, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  }
  // stepsize_X = (stop_x - start_x)/numberOfRows, stepsize_Y = (stop_y - start_y)/numberOfColumns (rt:828-830)
  const double step_x = (stop_x - start_x) / double(rows), step_y = (stop_y - start_y) / double(cols);
  SART_CUDA(launch_heatmap(rows, cols, start_x, step_x, start_y, step_y, n, dX, dY, dW, norm, dRes, dBad, h->stream));
  unsigned long long bad = 0;
  SART_CUDA(cudaMemcpyAsync(result, dRes, cells * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaMemcpyAsync(&bad, dBad, sizeof bad, cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  if (n_out_of_range) *n_out_of_range = bad;
  return SART_OK;
}

int sart_angular_scan(sart_handle_t* h, int n_angles, const double* angles_deg, uint64_t first_ray,
                      uint64_t n_rays_per_angle, uint64_t seed, double* fluxes, sart_counters_t* counters, double* images) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (n_angles < 1 || !angles_deg || !fluxes) return fail(SART_ERR_ARG, "sart_angular_scan: bad argument");
  if (h->n_masses != 1) return fail(SART_ERR_ARG, "sart_angular_scan: set a single axion mass");
  if (h->sampler == SART_SAMPLER_ALIAS && h->precision != 2)
    return fail(SART_ERR_CONFIG, "the alias sampler needs precision mode 2");
  DeviceGuard dg(h->device);
  const size_t plane = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS;
  const size_t imgBytes = align256(size_t(n_angles) * plane * sizeof(double));
  const size_t bytes = 2 * imgBytes + align256(size_t(n_angles) * sizeof(sart_counters_t));
  int rc = ensure_stage(h, bytes);
  if (rc) return rc;
  unsigned char* base = static_cast<unsigned char*>(h->d_stage);
  double* dImg = reinterpret_cast<double*>(base);
  double* dImg2 = reinterpret_cast<double*>(base + imgBytes);
  sart_counters_t* dCnt = reinterpret_cast<sart_counters_t*>(base + 2 * imgBytes);
  SART_CUDA(cudaMemsetAsync(base, 0, bytes, h->stream));
  // One launch per scan point, queued back to back on the handle's stream: only the by-value parameter block differs
  // (the rotation of the telescope frame), the tables and shell records in HBM are shared, nothing synchronises.
  fast::FastTables ft = h->ftables;
  Tables et = h->tables;
  ft.rad = RadialHist{}; et.rad = RadialHist{};
  for (int i = 0; i < n_angles; ++i) {
    sart_setup_t s = h->setup;
    s.telescope.telescope_turned_y = angles_deg[i];   // rt:2796
    Params P;
    rederive_params(h, s, &P);
    const uint64_t first = first_ray + uint64_t(i) * n_rays_per_angle;   // every scan point traces its own rays, like the reference
    if (h->precision >= 1) {
      fast::FastParams F;
      fast::derive_params(s, P, &F);
      F.shellRhoMin = h->fparams.shellRhoMin; F.shellInvStep = h->fparams.shellInvStep; F.nShellGuide = h->fparams.nShellGuide;
      if (h->precision == 2) {
        fast::Geo32 G;
        std::vector<fast::ShellF32> unused(SART_MAX_SHELLS);
        fast::derive_f32(F, nullptr, 0, &G, unused.data());
        // error budgets: the handle's (they depend on the shells, which do not turn), doubled where the rotation of the
        // telescope frame adds rounding steps
        G.tol = h->geo32.tol;
        if (F.rotated && !h->fparams.rotated) { G.tol.latA *= 2.0f; G.tol.detA *= 2.0f; }
        for (uint64_t done = 0; done < n_rays_per_angle; done += kRetraceChunk) {
          const uint64_t n = std::min<uint64_t>(n_rays_per_angle - done, kRetraceChunk);
          fast::FastTables fq = ft;
          if (h->retrace && h->sampler != SART_SAMPLER_ALIAS && (rc = begin_queue(h, n, &fq.rq))) return rc;
          SART_CUDA(launch_mc_image_f32(F, G, fq, h->masses[0], first + done, n, seed, dImg + size_t(i) * plane,
                                        dImg2 + size_t(i) * plane, dCnt + i, h->sm_count, h->compact != 0, h->stream));
          if (fq.rq.cap)
            SART_CUDA(launch_retrace_mc_image(P, et, 1, h->d_masses, first + done, seed, fq.rq, dImg + size_t(i) * plane,
                                              dImg2 + size_t(i) * plane, dCnt + i, h->sm_count, h->stream));
        }
        continue;
      }
      SART_CUDA(launch_mc_image_fast(F, ft, h->masses[0], first, n_rays_per_angle, seed, dImg + size_t(i) * plane,
                                     dImg2 + size_t(i) * plane, dCnt + i, h->sm_count, h->compact != 0, h->stream));
    } else {
      SART_CUDA(launch_mc_image_exact(P, et, 1, h->d_masses, first, n_rays_per_angle, seed, dImg + size_t(i) * plane,
                                      dImg2 + size_t(i) * plane, dCnt + i, h->sm_count, h->stream));
    }
  }
  std::vector<sart_counters_t> cnt;
  cnt.resize(size_t(n_angles));
  SART_CUDA(cudaMemcpyAsync(cnt.data(), dCnt, cnt.size() * sizeof(sart_counters_t), cudaMemcpyDeviceToHost, h->stream));
  if (images) SART_CUDA(cudaMemcpyAsync(images, dImg, size_t(n_angles) * plane * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < n_angles; ++i) fluxes[i] = cnt[size_t(i)].sum_w;   // axions.filterIt(it.passed).mapIt(it.weights).sum() rt:2800
  if (counters) std::memcpy(counters, cnt.data(), cnt.size() * sizeof(sart_counters_t));
  return SART_OK;
}

int sart_synchronize(sart_handle_t* h) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  DeviceGuard dg(h->device);
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

}  // extern "C"
