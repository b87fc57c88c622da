// api.cu — the C-ABI of libsart.so (include/sart.h): handle lifetime, table upload, launches, read-back.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <type_traits>
#include <vector>

#include "host_cuda.h"
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

// Synchronous host -> device copy of n elements into a table the kernels only read.
template <class T> static cudaError_t put(const T* dst, const T* src, size_t n) {
  return cudaMemcpy(const_cast<T*>(dst), src, n * sizeof(T), cudaMemcpyHostToDevice);
}

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
  const bool solar = t->nRadii > 0 && t->energies;
  const bool refl = t->reflectivity && t->nCoatings > 0;
  const sart_interp1d_t* I[4] = {&t->strongbackTransmission, &t->windowTransmission, &t->gasAbsorption, &t->telescopeTransmission};
  std::vector<sart::ShellF64> shells(SART_MAX_SHELLS);
  derive_shells(h->setup, shells.data());
  // window / strongback / detector-gas factors at each tabulated energy (device_params.h: EnergyFactors)
  std::vector<EnergyFactors> ef;
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
  }

  Tables& T = h->tables;
  std::memset(&T, 0, sizeof T);
  const double** PX[4] = {&T.sbX, &T.wdX, &T.gaX, &T.ttX};
  const double** PY[4] = {&T.sbY, &T.wdY, &T.gaY, &T.ttY};
  int32_t* PN[4] = {&T.sbN, &T.wdN, &T.gaN, &T.ttN};
  struct Copy { const void* dst; const void* src; size_t bytes; };
  std::vector<Copy> copies;
  auto layout = [&](Carve c) {   // every table: its place in table_blob and the host array it is filled from
    copies.clear();
    auto add = [&](auto*& dst, const auto* src, size_t n) { c.take(dst, n); copies.push_back({dst, src, n * sizeof *src}); };
    if (solar) {
      add(T.energies, t->energies, t->nEnergies);
      add(T.fluxRadiusCDF, t->fluxRadiusCDF, t->nRadii);
      add(T.diffFluxCDFs, t->diffFluxCDFs, size_t(t->nRadii) * t->nEnergies);
    }
    if (refl) add(T.reflectivity, t->reflectivity, size_t(t->nCoatings) * t->nAngles * t->nReflEnergies);
    for (int k = 0; k < 4; ++k)
      if (I[k]->n > 0 && I[k]->x && I[k]->y) { add(*PX[k], I[k]->x, I[k]->n); add(*PY[k], I[k]->y, I[k]->n); *PN[k] = I[k]->n; }
    add(T.shells, shells.data(), shells.size());
    if (solar) add(T.energyFactors, ef.data(), ef.size());
    return c.off;
  };
  const size_t bytes = layout(Carve());
  if (h->table_blob) { cudaFree(h->table_blob); h->table_blob = nullptr; }
  SART_CUDA(cudaMalloc(&h->table_blob, bytes));
  h->table_bytes = bytes;
  layout(Carve(h->table_blob));
  for (const Copy& c : copies)
    if (c.bytes) SART_CUDA(cudaMemcpyAsync(const_cast<void*>(c.dst), c.src, c.bytes, cudaMemcpyHostToDevice, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
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
  fast::FastTables& F = h->ftables;
  if (t) {
    // the exact pipeline narrows its two CDF searches with the same guide tables (device_params.h: Tables)
    const bool solarGuides = P.nRadii > 0 && t->fluxRadiusCDF;
    // alias tables of the same distributions (sart_set_sampler), when the packed 11-bit alias index can hold them
    const bool aliasFits = solarGuides && P.nRadii <= 2048 && P.nEnergies <= 2048;
    const size_t nR = size_t(std::max(P.nRadii, 1));
    auto layout = [&](Carve c) {
      c.take(F.shells, shf.size()); c.take(F.shells32, sh32.size());
      c.take(F.shellGuide, 4096); c.take(F.shellTab, 4096);
      c.take(F.elut, lut.size()); c.take(F.glut, glut.size()); c.take(F.telTrans, telTrans.size());
      c.take(F.radiusGuide, kRadGuide); c.take(F.energyGuide, nR * kEnGuide);
      c.take(F.radiusThr, thr_pitch(int(nR))); c.take(F.energyThr, nR * thr_pitch(std::max(P.nEnergies, 1)));
      c.take(F.radiusCells, kRadCells); c.take(F.energyCells, nR * kEnCells);
      c.take(F.reflE, size_t(std::max(nCoat, 1)) * reflPlane);
      c.take(F.radiusAlias, aliasFits ? nR : 0); c.take(F.energyAlias, aliasFits ? nR * P.nEnergies : 0);
      return c.off;
    };
    const size_t bytes = layout(Carve());
    h->alias_ok = 0;
    if (h->fast_blob) { cudaFree(h->fast_blob); h->fast_blob = nullptr; }
    SART_CUDA(cudaMalloc(&h->fast_blob, bytes));
    layout(Carve(h->fast_blob));
    if (solarGuides) {
      const int ep = thr_pitch(P.nEnergies);
      std::vector<uint16_t> rg(kRadGuide), eg(size_t(P.nRadii) * kEnGuide);
      std::vector<uint32_t> rth(size_t(thr_pitch(P.nRadii))), eth(size_t(P.nRadii) * ep);
      build_guide(t->fluxRadiusCDF, P.nRadii, kRadGuide, rg.data());
      build_thresholds(t->fluxRadiusCDF, P.nRadii, rth.data());
      for (int r = 0; r < P.nRadii; ++r) {
        build_guide(t->diffFluxCDFs + size_t(r) * P.nEnergies, P.nEnergies, kEnGuide, eg.data() + size_t(r) * kEnGuide);
        build_thresholds(t->diffFluxCDFs + size_t(r) * P.nEnergies, P.nEnergies, eth.data() + size_t(r) * ep);
      }
      SART_CUDA(put(F.radiusGuide, rg.data(), rg.size()));
      SART_CUDA(put(F.energyGuide, eg.data(), eg.size()));
      SART_CUDA(put(F.radiusThr, rth.data(), rth.size()));
      SART_CUDA(put(F.energyThr, eth.data(), eth.size()));
      {
        std::vector<fast::SampleCell> rc(kRadCells), ec(size_t(P.nRadii) * kEnCells);
        fast::build_sample_cells(rth.data(), P.nRadii, kRadCellBits, rc.data());
        for (int r = 0; r < P.nRadii; ++r)
          fast::build_sample_cells(eth.data() + size_t(r) * ep, P.nEnergies, kEnCellBits, ec.data() + size_t(r) * kEnCells);
        SART_CUDA(put(F.radiusCells, rc.data(), rc.size()));
        SART_CUDA(put(F.energyCells, ec.data(), ec.size()));
      }
      if (aliasFits) {
        std::vector<uint32_t> ra(size_t(P.nRadii)), ea(size_t(P.nRadii) * P.nEnergies);
        bool ok = fast::build_alias_table(rth.data(), P.nRadii, ra.data());
        for (int r = 0; ok && r < P.nRadii; ++r)
          ok = fast::build_alias_table(eth.data() + size_t(r) * ep, P.nEnergies, ea.data() + size_t(r) * P.nEnergies);
        if (ok) {
          SART_CUDA(put(F.radiusAlias, ra.data(), ra.size()));
          SART_CUDA(put(F.energyAlias, ea.data(), ea.size()));
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
      SART_CUDA(put(F.reflE, re.data(), re.size()));
    }
    F.energies = h->tables.energies;
    F.radiusCDF = h->tables.fluxRadiusCDF;
    F.energyCDF = h->tables.diffFluxCDFs;
    if (!h->alias_ok) { F.radiusAlias = nullptr; F.energyAlias = nullptr; }
    F.sampler = h->alias_ok ? h->sampler : SART_SAMPLER_INVERSE_CDF;
    h->tables.radiusGuide = solarGuides ? F.radiusGuide : nullptr;
    h->tables.energyGuide = solarGuides ? F.energyGuide : nullptr;
  } else if (nCoat > 0) {
    // setup update: only the X-ray-source row (index nE) of each coating can have changed
    std::vector<float> row(reflRow), line(size_t(P.nAngles));
    for (int c = 0; c < nCoat; ++c) {
      fast::refl_at_energy(P, h->h_refl32.data() + size_t(c) * P.nAngles * P.nReflEnergies, h->setup.testSource.energy, line.data());
      std::copy(line.begin(), line.end(), row.begin());
      SART_CUDA(put(F.reflE + size_t(c) * reflPlane + size_t(nE) * reflRow, row.data(), reflRow));
    }
  }
  SART_CUDA(put(F.shells, shf.data(), shf.size()));
  SART_CUDA(put(F.shells32, sh32.data(), sh32.size()));
  SART_CUDA(put(F.elut, lut.data(), lut.size()));
  SART_CUDA(put(F.glut, glut.data(), glut.size()));
  SART_CUDA(put(F.telTrans, telTrans.data(), telTrans.size()));
  SART_CUDA(put(F.shellGuide, sguide.data(), sguide.size()));
  SART_CUDA(put(F.shellTab, stab.data(), stab.size()));
  return SART_OK;
}

// Lays block `a` of accumulator k (bins and rmax set) over `base` (nullptr: only measures): the arrays of accum_arrays for
// SART_MAX_MASSES masses, each on a 256-byte boundary. Returns their bytes.
static size_t carve_accum(AccumKind k, void* base, Accum* a) {
  Carve c(base);
  accum_arrays(k, *a, *a, accum_rows(k, SART_MAX_MASSES), [&](auto*& p, auto*&, size_t n) { c.take(p, n); });
  if (k == kRadialHist || k == kMassRadialHist) { a->rad.invStep = double(a->bins) / a->rmax; a->rad.nbins = a->bins; }
  if (k == kMassSpectra) { a->spec.eRow = uint32_t(a->bins); a->spec.sRow = uint32_t(SART_MAX_SHELLS); }
  if (k == kBandImages || k == kMassBandImages) a->band.nBands = a->bins;
  return c.off;
}

// A failed allocation of accumulator k: the CUDA error, except that the per-mass radial histograms and band images, which
// take SART_MAX_MASSES rows (about 3 x 64 MiB per band), report an out-of-memory device as SART_ERR_NOMEM.
static int accum_alloc_fail(AccumKind k, cudaError_t e, size_t bytes) {
  if (e == cudaErrorMemoryAllocation && (k == kMassRadialHist || k == kMassBandImages))
    return fail(SART_ERR_NOMEM, "cudaMalloc (accumulator): no room for %zu bytes on the device", bytes);
  return cuda_fail(e, "cudaMalloc (accumulator)");
}

int alloc_accum(AccumKind k, int bins, double rmax, Accum* a) {
  *a = Accum{};
  a->bins = bins; a->rmax = rmax;
  const size_t bytes = carve_accum(k, nullptr, a);
  const cudaError_t e = cudaMalloc(&a->blob, bytes);
  if (e != cudaSuccess) { *a = Accum{}; return accum_alloc_fail(k, e, bytes); }
  a->bytes = bytes;
  carve_accum(k, a->blob, a);
  return SART_OK;
}

// The buffers the throughput kernels of accumulator k add into (Accum::tput, tput_band), laid over `base` (nullptr: only
// measures); returns their bytes. The spectra's replicas (device_params.h: Spectra): eW | eW2 | eN, each eRep x eStride |
// sW | sN, each sRep x SART_MAX_SHELLS. The per-mass spectra's mass-minor accumulators (fast_common.cuh: mass_spec_add):
// eW | eW2 | 32-bit eN, each [nE1][SART_MAX_MASSES] | sW | 32-bit sN, each [SART_MAX_SHELLS][SART_MAX_MASSES]. The band
// images' replicas (device_params.h: BandImages): w | w2, each bRep x [bins][256][256], and the band of each of the nE1
// energy bins, which the exact kernels read through the handle's block (a->band) as well; their counts are the handle's. The
// quantity histograms' replicas of Σw and Σw² (device_params.h: QuantityHists::rw, rw2), each qRep x bins, in a->qh itself.
// The per-mass radial histograms' mass-minor accumulators (fast_common.cuh: mass_scan_loop): w | 32-bit n, each
// [bins][SART_MAX_MASSES]. The per-mass band images' mass-minor accumulators: w | w2, each [bins][256][256][SART_MAX_MASSES] |
// 32-bit n [bins][SART_MAX_MASSES], and the band table as for the band images.
static size_t carve_throughput(AccumKind k, int nE1, int eRep, int sRep, int bRep, int qRep, void* base, Accum* a) {
  Carve c(base);
  Spectra* r = &a->tput;
  *r = Spectra{};
  if (k == kSpectra) {
    const uint32_t eStride = uint32_t((nE1 + 31) & ~31);
    const size_t e = size_t(eRep) * eStride, s = size_t(sRep) * SART_MAX_SHELLS;
    c.take(r->eW, e); c.take(r->eW2, e); c.take(r->eN, e); c.take(r->sW, s); c.take(r->sN, s);
    r->eStride = eStride; r->eRepMask = uint32_t(eRep - 1); r->sRepMask = uint32_t(sRep - 1);
  } else if (k == kMassSpectra) {
    const size_t e = size_t(nE1) * SART_MAX_MASSES, s = size_t(SART_MAX_SHELLS) * SART_MAX_MASSES;
    unsigned int *eN, *sN;
    c.take(r->eW, e); c.take(r->eW2, e); c.take(eN, e); c.take(r->sW, s); c.take(sN, s);
    r->eN = reinterpret_cast<unsigned long long*>(eN); r->sN = reinterpret_cast<unsigned long long*>(sN);
  } else if (k == kBandImages) {
    BandImages& b = a->tput_band;
    b = a->band;
    const size_t len = size_t(a->bins) * SART_IMAGE_BINS * SART_IMAGE_BINS;
    c.take(b.w, size_t(bRep) * len); c.take(b.w2, size_t(bRep) * len); c.take(b.band, size_t(nE1));
    b.repStride = uint32_t(len); b.repMask = uint32_t(bRep - 1);
    a->band.band = b.band;
  } else if (k == kMassRadialHist) {
    RadialHist& m = a->tput_rad;
    m = a->rad;
    unsigned int* n;
    c.take(m.w, size_t(a->bins) * SART_MAX_MASSES); c.take(n, size_t(a->bins) * SART_MAX_MASSES);
    m.n = reinterpret_cast<unsigned long long*>(n);
  } else if (k == kMassBandImages) {
    BandImages& b = a->tput_band;
    b = a->band;
    const size_t len = size_t(a->bins) * SART_IMAGE_BINS * SART_IMAGE_BINS * SART_MAX_MASSES;
    unsigned int* n;
    c.take(b.w, len); c.take(b.w2, len); c.take(n, size_t(a->bins) * SART_MAX_MASSES); c.take(b.band, size_t(nE1));
    b.n = reinterpret_cast<unsigned long long*>(n);
    a->band.band = b.band;
  } else if (k == kQuantityHists) {
    QuantityHists& q = a->qh;
    c.take(q.rw, size_t(qRep) * size_t(a->bins)); c.take(q.rw2, size_t(qRep) * size_t(a->bins));
    q.repStride = uint32_t(a->bins); q.repMask = uint32_t(qRep - 1);
  }
  return c.off;
}

// The (per-mass) band images' table of the energy bins from bin `from` on (sart_enable_band_images,
// sart_enable_mass_band_images; device_params.h: BandImages): the band of the energy a per-ray record reports,
// max(0.03 keV, energies[i]) for tabulated energy i (rt:470-471) and the X-ray source's energy for bin nEnergies.
static int put_band_table(sart_handle* h, AccumKind k, int from) {
  const Accum& a = h->accum[k];
  const int nE = h->params.nEnergies;
  auto band_of = [&](double E) {
    for (int b = 0; b < a.bins; ++b)
      if (a.edges[b] <= E && E < a.edges[b + 1]) return uint8_t(b);
    return kNoBand;
  };
  std::vector<uint8_t> t(size_t(nE) + 1);
  for (int i = from; i <= nE; ++i)
    t[size_t(i)] = band_of(i == nE ? h->setup.testSource.energy
                                   : (size_t(i) < h->h_energies.size() ? std::max(0.03, h->h_energies[size_t(i)]) : NAN));
  SART_CUDA(cudaMemcpyAsync(const_cast<uint8_t*>(a.band.band) + from, t.data() + from, size_t(nE + 1 - from),
                            cudaMemcpyHostToDevice, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

// Switches accumulator k off: frees the handle's block, its throughput buffers and its merged copy. The other accumulators
// and their merged copies stay as they are.
static void free_accum(sart_handle* h, AccumKind k) {
  cudaFree(h->accum[k].blob); cudaFree(h->accum[k].tput_blob); cudaFree(h->merged_accum[k].blob);
  h->accum[k] = Accum{};
  h->merged_accum[k] = Accum{};
  if (k == kRadialHist) h->tables.rad = h->ftables.rad = RadialHist{};
}

// The specs of the quantity histograms into their device view (device_params.h: QuantityHists), bins = their entries.
static void put_qhist_specs(Accum& a, int n, const sart_quantity_hist_t* specs) {
  QuantityHists& q = a.qh;
  a.n_qhists = n;
  q.nHists = n; q.entries = a.bins;
  int off = 0;
  for (int j = 0; j < n; ++j) {
    a.qspecs[j] = specs[j];
    q.quantity[j] = specs[j].quantity; q.nbins[j] = specs[j].nbins; q.off[j] = off;
    q.lo[j] = specs[j].lo; q.hi[j] = specs[j].hi; q.inv[j] = double(specs[j].nbins) / (specs[j].hi - specs[j].lo);
    off += specs[j].nbins + 2;
  }
}

// Accumulator k on with `bins` bins: the handle's block and its throughput buffers, allocated, cleared and carved; the band
// images also get their `edges` and energy -> band table, the quantity histograms their `n_q` specs `qspecs`.
static int new_accum(sart_handle* h, AccumKind k, int bins, double rmax, const double* edges, int n_q,
                     const sart_quantity_hist_t* qspecs) {
  Accum& a = h->accum[k];
  int rc = alloc_accum(k, bins, rmax, &a);
  if (rc) return rc;
  if (edges) std::copy(edges, edges + bins + 1, a.edges);
  if (qspecs) put_qhist_specs(a, n_q, qspecs);
  // Replicas of the spectra (powers of two; SART_SPEC_E_REPLICAS / SART_SPEC_S_REPLICAS override them for measurements).
  // The energy bins spread the passed rays over hundreds of addresses, like the focal spot the image replicas serve: one
  // replica per block residue. The shell bins are a handful of addresses (4 for LLNL): one per warp. The band images have a
  // focal spot per band plane, like the image: 8 replicas (SART_BAND_REPLICAS overrides it; measured on B200, CAST+LLNL, 4
  // bands, 1e9 rays: 1 replica 39.5 ms, 8 replicas 31.4 ms, 16 replicas at 16 bands no faster than 8). The quantity
  // histograms' sums go to 8 replicas only in the kernels whose block leaves no room for them in shared memory.
  auto pow2 = [](const char* env, int dflt) {
    int n = dflt;
    if (const char* e = std::getenv(env)) n = std::max(1, std::min(1 << 16, std::atoi(e)));
    int p = 1;
    while (p * 2 <= n) p *= 2;
    return p;
  };
  const int eRep = pow2("SART_SPEC_E_REPLICAS", 32), sRep = pow2("SART_SPEC_S_REPLICAS", 1024);
  const int bRep = std::min(pow2("SART_BAND_REPLICAS", 8), 64);
  const int qRep = std::min(pow2("SART_QHIST_REPLICAS", 8), 64);
  const int nE1 = h->params.nEnergies + 1;
  const size_t tputBytes = carve_throughput(k, nE1, eRep, sRep, bRep, qRep, nullptr, &a);
  if (tputBytes) {
    const cudaError_t e = cudaMalloc(&a.tput_blob, tputBytes);
    if (e != cudaSuccess) { a.tput_blob = nullptr; return accum_alloc_fail(k, e, tputBytes); }
  }
  SART_CUDA(cudaMemsetAsync(a.blob, 0, a.bytes, h->stream));
  if (tputBytes) SART_CUDA(cudaMemsetAsync(a.tput_blob, 0, tputBytes, h->stream));
  SART_CUDA(cudaStreamSynchronize(h->stream));
  carve_throughput(k, nE1, eRep, sRep, bRep, qRep, a.tput_blob, &a);
  if (k == kRadialHist) h->tables.rad = h->ftables.rad = a.rad;
  return k == kBandImages || k == kMassBandImages ? put_band_table(h, k, 0) : SART_OK;
}

// What every sart_enable_* does after its own checks: synchronises, switches accumulator k off, and with bins > 0 on again,
// cleared. A failure leaves it off.
static int set_accum(sart_handle* h, AccumKind k, int bins, double rmax = 0.0, const double* edges = nullptr, int n_q = 0,
                     const sart_quantity_hist_t* qspecs = nullptr) {
  DeviceGuard dg(h->device);
  SART_CUDA(cudaStreamSynchronize(h->stream));
  free_accum(h, k);
  const int rc = bins > 0 ? new_accum(h, k, bins, rmax, edges, n_q, qspecs) : SART_OK;
  if (rc) {
    free_accum(h, k);
    cudaGetLastError();   // a failed cudaMalloc must not surface at the next launch
  }
  return rc;
}

// Clears the handle's block of accumulator k on its stream (nothing while it is off).
static int clear_accum(sart_handle* h, AccumKind k) {
  if (h->accum[k].blob) SART_CUDA(cudaMemsetAsync(h->accum[k].blob, 0, h->accum[k].bytes, h->stream));
  return SART_OK;
}

int read_accum(sart_handle* h, AccumKind k, bool merged, std::initializer_list<void*> host, const char* off) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  const Accum& a = merged ? h->merged_accum[k] : h->accum[k];
  if (merged ? !a.valid : !a.blob) return fail(SART_ERR_ARG, "%s", off);
  DeviceGuard dg(h->device);
  void* const* hp = host.begin();
  cudaError_t e = cudaSuccess;
  accum_arrays(k, a, a, accum_rows(k, h->n_masses), [&](auto* d, auto*, size_t n) {
    void* p = *hp++;
    if (p && e == cudaSuccess) e = cudaMemcpyAsync(p, d, n * sizeof *d, cudaMemcpyDeviceToHost, h->stream);
  });
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  return e == cudaSuccess ? SART_OK : cuda_fail(e, "cudaMemcpyAsync (accumulator, device to host)");
}

static int ensure_image(sart_handle* h, int nMasses) {
  const size_t len = size_t(nMasses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
  if (h->d_image && h->image_masses == nMasses) return SART_OK;
  for (AccumKind k : kAllAccums) {   // a new mass list: the per-mass rows of the old one are meaningless
    if (!per_mass(k)) continue;
    if (const int rc = clear_accum(h, k)) return rc;
    h->merged_accum[k].valid = 0;
  }
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

// A run of the FP32 pipeline: launches of at most fast::kMaxRaysPerLaunch rays, each followed on the same stream by the
// exact pipeline's pass over the rays it queued as uncertain. f32(done, m, q) launches rays [done, done + m) of the run with
// queue q attached (cap 0: none), retrace(done, m, q) traces the rays in q. `queue`: whether the run may be re-traced at all
// (begin_queue attaches no queue either while re-tracing is switched off).
template <class F32, class Retrace>
static int f32_then_retrace(sart_handle* h, uint64_t n, bool queue, F32&& f32, Retrace&& retrace) {
  for (uint64_t done = 0; done < n; done += fast::kMaxRaysPerLaunch) {
    const uint64_t m = std::min<uint64_t>(n - done, fast::kMaxRaysPerLaunch);
    fast::RetraceQueue q{};
    if (queue) {
      const int rc = begin_queue(h, m, &q);
      if (rc) return rc;
    }
    SART_CUDA(f32(done, m, q));
    if (q.cap) SART_CUDA(retrace(done, m, q));
  }
  return SART_OK;
}

// Replica buffers for the single-mass throughput kernels. SART_IMG_REPLICAS overrides the count (1 = off).
static int ensure_replicas(sart_handle* h) {
  if (h->n_rep > 0) return SART_OK;
  int n = 8;   // measured on B200, CAST+LLNL, 1e9 rays: 1 replica 43.8 ms, 4 / 16 / 64 replicas 36.1 ms
  if (const char* e = std::getenv("SART_IMG_REPLICAS")) n = std::max(1, std::min(256, std::atoi(e)));
  h->n_rep = n;
  h->rep_stride = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS;
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
  double *img, *img2;
  sart_counters_t* dc;
  auto layout = [&](Carve c) { c.take(img, plane); c.take(img2, plane); c.take(dc, 1); return c.off; };
  const size_t bytes = layout(Carve());
  int rc = ensure_stage(h, bytes);
  if (rc) return rc;
  layout(Carve(h->d_stage));
  SART_CUDA(cudaMemsetAsync(h->d_stage, 0, bytes, h->stream));
  const uint64_t n = 1u << 17;
  fast::FastTables pilotTables = h->ftables;
  pilotTables.rad = RadialHist{};   // the pilot rays must not reach the user's radial histogram
  SART_CUDA(launch_mc_image_fast(h->fparams, pilotTables, h->setup.consts.mAxion, 0, n, 0x5eedull, img, img2, dc,
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

// The copy streams and events of the two chunked host-buffer paths (sart_trace_presampled, sart_trace_mc_passed), created
// on first use.
static int ensure_copy_streams(sart_handle* h) {
  if (h->stream_in) return SART_OK;
  SART_CUDA(cudaStreamCreateWithFlags(&h->stream_in, cudaStreamNonBlocking));
  SART_CUDA(cudaStreamCreateWithFlags(&h->stream_out, cudaStreamNonBlocking));
  for (int i = 0; i < 6; ++i) SART_CUDA(cudaEventCreateWithFlags(reinterpret_cast<cudaEvent_t*>(&h->ev[i]), cudaEventDisableTiming));
  return SART_OK;
}

// Copies records [0, n) of the device arrays `dev` into records [first, first + n) of the caller's arrays `host` on stream
// s, for every array the caller asked for. Out: sart_ray_out_t or sart_passed_out_t.
template <class Out>
static int copy_records(const Out& host, size_t first, const Out& dev, size_t n, cudaStream_t s) {
  cudaError_t e = cudaSuccess;
  auto copy = [&](auto* hp, auto* dp) {
    if (hp && e == cudaSuccess) e = cudaMemcpyAsync(hp + first, dp, n * sizeof *hp, cudaMemcpyDeviceToHost, s);
  };
  if constexpr (std::is_same_v<Out, sart_ray_out_t>) ray_out_fields(host, dev, copy);
  else passed_out_fields(host, dev, copy);
  return e == cudaSuccess ? SART_OK : cuda_fail(e, "cudaMemcpyAsync (records, device to host)");
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
  if ((e = cudaMalloc(&h->d_desc, kDescCapacity * sizeof(long long))) != cudaSuccess) { sart_destroy(h); return cuda_fail(e, "cudaMalloc"); }
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
  cudaFree(h->d_counters); cudaFree(h->d_stage); cudaFree(h->d_rep); cudaFree(h->d_mass_acc); cudaFree(h->d_queue);
  cudaFree(h->d_desc);
  for (AccumKind k : kAllAccums) free_accum(h, k);
  cudaFreeHost(h->h_stage);
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
  SART_CUDA(cudaMemcpyAsync(const_cast<ShellF64*>(h->tables.shells), shells.data(), shells.size() * sizeof(ShellF64),
                            cudaMemcpyHostToDevice, h->stream));
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
  // the band of the X-ray source's energy bin, like its reflectivity row (upload_fast)
  for (AccumKind k : {kBandImages, kMassBandImages})
    if (h->accum[k].blob && old.testSource.energy != setup->testSource.energy && (rc = put_band_table(h, k, h->params.nEnergies)))
      return rc;
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
    if (m > fast::kMaxRaysPerLaunch) return fail(SART_ERR_ARG, "sart_trace_presampled: at most 2^31 rays per call in precision mode 2");
    fast::FastTables ft = h->ftables;
    return f32_then_retrace(h, m, true,   // one launch
        [&](uint64_t, uint64_t, const fast::RetraceQueue& q) {
          ft.rq = q;
          return launch_presampled_f32(h->fparams, h->geo32, ft, h->masses[0], m, dO, dX, dE, dev, h->sm_count, h->stream);
        },
        [&](uint64_t, uint64_t, const fast::RetraceQueue& q) {
          return launch_retrace_presampled(h->params, h->tables, h->masses[0], m, dO, dX, dE, q, dev, h->sm_count, h->stream);
        });
  }
  SART_CUDA(launch_presampled_exact(h->params, h->tables, h->masses[0], m, dO, dX, dE, dev, h->stream));
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

// Lays a device-side sart_ray_out_t of n rays over `c`: an array for every array the caller asked for.
static void carve_out(Carve& c, size_t n, const sart_ray_out_t& host, sart_ray_out_t* dev) {
  ray_out_fields(host, *dev, [&](auto* hp, auto*& dp) { if (hp) c.take(dp, n); else dp = nullptr; });
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
  const int nbuf = n > chunk ? 2 : 1;
  double *dO[2], *dX[2], *dE[2];
  sart_ray_out_t dev[2];
  auto layout = [&](Carve c) {   // a buffer: origin [3][m0] | exit [2][m0] | energy [m0] | records of m0 rays
    for (int b = 0; b < nbuf; ++b) {
      c.take(dO[b], 3 * m0); c.take(dX[b], 2 * m0); c.take(dE[b], m0);
      carve_out(c, m0, *out, &dev[b]);
    }
    return c.off;
  };
  if ((rc = ensure_stage(h, layout(Carve())))) return rc;
  layout(Carve(h->d_stage));
  if (nbuf == 2 && (rc = ensure_copy_streams(h))) return rc;
  cudaStream_t sIn = nbuf == 2 ? h->stream_in : h->stream, sOut = nbuf == 2 ? h->stream_out : h->stream;
  auto ev = [&](int kind, int b) { return static_cast<cudaEvent_t>(h->ev[kind * 2 + b]); };   // 0 in, 1 kernel, 2 out
  size_t k = 0;
  for (size_t a = 0; a < n; a += chunk, ++k) {
    const size_t m = n - a < chunk ? n - a : chunk;
    const int b = int(k & 1);
    if (nbuf == 2 && k >= 2) SART_CUDA(cudaStreamWaitEvent(sIn, ev(1, b), 0));      // kernel of chunk k-2 has read this buffer
    for (int c = 0; c < 3; ++c) SART_CUDA(cudaMemcpyAsync(dO[b] + c * m, origin + c * n + a, m * sizeof(double), cudaMemcpyHostToDevice, sIn));
    for (int c = 0; c < 2; ++c) SART_CUDA(cudaMemcpyAsync(dX[b] + c * m, exitxy + c * n + a, m * sizeof(double), cudaMemcpyHostToDevice, sIn));
    SART_CUDA(cudaMemcpyAsync(dE[b], energy + a, m * sizeof(double), cudaMemcpyHostToDevice, sIn));
    if (nbuf == 2) {
      SART_CUDA(cudaEventRecord(ev(0, b), sIn));
      SART_CUDA(cudaStreamWaitEvent(h->stream, ev(0, b), 0));
      if (k >= 2) SART_CUDA(cudaStreamWaitEvent(h->stream, ev(2, b), 0));           // outputs of chunk k-2 have left this buffer
    }
    if ((rc = launch_presampled(h, m, dO[b], dX[b], dE[b], dev[b]))) return rc;
    if (nbuf == 2) {
      SART_CUDA(cudaEventRecord(ev(1, b), h->stream));
      SART_CUDA(cudaStreamWaitEvent(sOut, ev(1, b), 0));
    }
    if ((rc = copy_records(*out, a, dev[b], m, sOut))) return rc;
    if (nbuf == 2) SART_CUDA(cudaEventRecord(ev(2, b), sOut));
  }
  if (nbuf == 2) { SART_CUDA(cudaStreamSynchronize(sIn)); SART_CUDA(cudaStreamSynchronize(sOut)); }
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

// Per-ray records of n Monte Carlo rays into the caller's arrays `out`: global rays first .. first + n - 1 of `seed`, or, with
// `words`, the caller's random words (host, SoA [6][n]). `late` and `emit` (host, may be NULL) are sart_trace_words'
// late_energy and emission shells.
static int trace_records(sart_handle* h, uint64_t first, size_t n, uint64_t seed, const uint32_t* words, bool late,
                         int32_t* emit, const sart_ray_out_t& out) {
  sart_ray_out_t dev;
  uint32_t* dW = nullptr;
  int32_t* dEmit = nullptr;
  auto layout = [&](Carve c) {
    carve_out(c, n, out, &dev);
    if (words) c.take(dW, 6 * n);
    if (emit) c.take(dEmit, n);
    return c.off;
  };
  int rc = ensure_stage(h, layout(Carve()));
  if (rc) return rc;
  layout(Carve(h->d_stage));
  if (words) SART_CUDA(cudaMemcpyAsync(dW, words, 6 * n * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  if (h->precision == 2) {
    fast::FastTables ft = h->ftables;
    // the alias sampler has another ray <-> index mapping than the exact pipeline's: no re-trace
    rc = f32_then_retrace(h, n, h->sampler != SART_SAMPLER_ALIAS,   // one launch
        [&](uint64_t, uint64_t, const fast::RetraceQueue& q) {
          ft.rq = q;
          return launch_mc_rays_f32(h->fparams, h->geo32, ft, h->masses[0], first, n, seed, dev, h->sm_count, h->stream, dW,
                                    late, dEmit);
        },
        [&](uint64_t, uint64_t, const fast::RetraceQueue& q) {
          return launch_retrace_mc_rays(h->params, h->tables, h->masses[0], first, n, seed, dW, q, dev, h->sm_count, h->stream);
        });
    if (rc) return rc;
  } else if (h->precision == 1) {
    SART_CUDA(launch_mc_rays_fast(h->fparams, h->ftables, h->masses[0], first, n, seed, dev, h->sm_count, h->stream));
  } else {
    SART_CUDA(launch_mc_rays_exact(h->params, h->tables, h->masses[0], first, n, seed, dev, h->stream, dW, dEmit));
  }
  if (dEmit) SART_CUDA(cudaMemcpyAsync(emit, dEmit, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  if ((rc = copy_records(out, 0, dev, n, h->stream))) return rc;
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
  if (h->precision == 2 && n > fast::kMaxRaysPerLaunch) return fail(SART_ERR_ARG, "sart_trace_mc_rays: at most 2^31 rays per call");
  return trace_records(h, first_ray, n, seed, nullptr, false, nullptr, *out);
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
  // chunks of 2^24 rays through two device buffers: the kernels of chunk k + 1 run while the records of chunk k (whose
  // number the host learns from a 4-byte read) cross PCIe on a second stream
  const uint64_t chunk = std::min<uint64_t>(std::max<uint64_t>(n, 1), uint64_t(1) << 24);
  unsigned int* dCount[2];
  sart_passed_out_t dev[2];
  sart_counters_t* dCnt;
  auto layout = [&](Carve c) {   // two buffers (the record count of the chunk | its records), then the run's counters
    for (int b = 0; b < 2; ++b) {
      c.take(dCount[b], 1);
      passed_out_fields(*out, dev[b], [&](auto* hp, auto*& dp) { if (hp) c.take(dp, chunk); else dp = nullptr; });
    }
    c.take(dCnt, 1);
    return c.off;
  };
  int rc = ensure_stage(h, layout(Carve()));
  if (rc) return rc;
  layout(Carve(h->d_stage));
  if ((rc = ensure_copy_streams(h))) return rc;
  if (!h->h_stage) SART_CUDA(cudaHostAlloc(&h->h_stage, 2 * sizeof(unsigned int), cudaHostAllocDefault));
  unsigned int* hcount = static_cast<unsigned int*>(h->h_stage);
  SART_CUDA(cudaMemsetAsync(dCnt, 0, sizeof(sart_counters_t), h->stream));
  auto evDone = [&](int b) { return static_cast<cudaEvent_t>(h->ev[b]); };
  auto evCopied = [&](int b) { return static_cast<cudaEvent_t>(h->ev[2 + b]); };
  uint64_t total = 0;
  bool overflow = false;
  auto finish = [&](uint64_t k) -> int {   // chunk k: wait for its kernels, learn its record count, send the records home
    const int b = int(k & 1);
    SART_CUDA(cudaEventSynchronize(evDone(b)));
    const uint64_t c = std::min<uint64_t>(hcount[b], chunk);
    const uint64_t room = total < capacity ? capacity - total : 0;
    const uint64_t take = std::min(c, room);
    if (take < c) overflow = true;
    if (take) {
      const int rc = copy_records(*out, total, dev[b], take, h->stream_out);
      if (rc) return rc;
    }
    SART_CUDA(cudaEventRecord(evCopied(b), h->stream_out));
    total += c;
    return SART_OK;
  };
  uint64_t k = 0;
  for (uint64_t done = 0; done < n; done += chunk, ++k) {
    const uint64_t m = std::min<uint64_t>(n - done, chunk);
    const int b = int(k & 1);
    if (k >= 2) SART_CUDA(cudaStreamWaitEvent(h->stream, evCopied(b), 0));   // the records of chunk k - 2 have left this buffer
    SART_CUDA(cudaMemsetAsync(dCount[b], 0, sizeof(unsigned int), h->stream));
    fast::FastTables ft = h->ftables;
    rc = f32_then_retrace(h, m, true,   // one launch
        [&](uint64_t, uint64_t, const fast::RetraceQueue& q) {
          ft.rq = q;
          return launch_mc_passed_f32(h->fparams, h->geo32, ft, h->masses[0], first_ray + done, m, seed, dev[b], dCount[b],
                                      unsigned(chunk), uint32_t(done), dCnt, h->sm_count, h->stream);
        },
        [&](uint64_t, uint64_t, const fast::RetraceQueue& q) {
          return launch_retrace_mc_passed(h->params, h->tables, h->masses[0], first_ray + done, seed, q, dev[b], dCount[b],
                                          unsigned(chunk), uint32_t(done), dCnt, h->sm_count, h->stream);
        });
    if (rc) return rc;
    SART_CUDA(cudaMemcpyAsync(hcount + b, dCount[b], sizeof(unsigned int), cudaMemcpyDeviceToHost, h->stream));
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
  if (h->precision == 2 && n > fast::kMaxRaysPerLaunch) return fail(SART_ERR_ARG, "sart_trace_words: at most 2^31 rays per call");
  DeviceGuard dg(h->device);
  return trace_records(h, 0, n, 0, words, late_energy != 0, emission_shell, *out);
}

// A fused image run of one axion mass in the handle's precision mode, with the parameter blocks and table views the caller
// prepared (the handle's, or those of a scan point). The throughput kernels add into img / img2, which ft may spread over
// replicas, and into the band images `band`; the exact kernels (mode 0, and the re-trace of mode 2) add into exImg / exImg2
// and `exBand`. All add into `counters` and into the quantity histograms `qh` (the exact kernels into its arrays, the
// throughput kernels from shared memory or through its replicas). Band images off: band.w == exBand.w == nullptr; quantity
// histograms off: qh.w == nullptr.
static int trace_image(sart_handle* h, const Params& P, const fast::FastParams& F, const fast::Geo32& G, fast::FastTables ft,
                       const Tables& et, uint64_t first, uint64_t n, uint64_t seed, double* img, double* img2, double* exImg,
                       double* exImg2, sart_counters_t* counters, const BandImages& band = {}, const BandImages& exBand = {},
                       const QuantityHists& qh = {}) {
  if (h->precision == 0) {
    SART_CUDA(launch_mc_image_exact(P, et, 1, h->d_masses, first, n, seed, exImg, exImg2, counters, h->sm_count, h->stream,
                                    exBand, qh));
    return SART_OK;
  }
  if (h->precision == 1) {
    SART_CUDA(launch_mc_image_fast(F, ft, h->masses[0], first, n, seed, img, img2, counters, h->sm_count, h->compact != 0,
                                   h->stream, band, qh));
    return SART_OK;
  }
  // the alias sampler has another ray <-> index mapping than the exact pipeline's: no re-trace
  return f32_then_retrace(h, n, h->sampler != SART_SAMPLER_ALIAS,
      [&](uint64_t done, uint64_t m, const fast::RetraceQueue& q) {
        ft.rq = q;
        return launch_mc_image_f32(F, G, ft, h->masses[0], first + done, m, seed, img, img2, counters, h->sm_count,
                                   h->compact != 0, h->stream, band, qh);
      },
      [&](uint64_t done, uint64_t, const fast::RetraceQueue& q) {
        return launch_retrace_mc_image(P, et, 1, h->d_masses, first + done, seed, q, exImg, exImg2, counters, h->sm_count,
                                       h->stream, exBand, qh);
      });
}

// The folds that follow a run of the throughput kernels with the accumulators `acc` (the handle's, or the rows of a scan
// point): the replicas of the spectra, the band images and the quantity histograms, which belong to the handle, are added
// into acc's arrays and cleared.
static int fold_accums(sart_handle* h, const Accum* acc) {
  const Accum &spec = acc[kSpectra], &bands = acc[kBandImages], &qhists = acc[kQuantityHists];
  if (spec.blob) SART_CUDA(launch_fold_spectra(spec.tput, spec.bins, spec.spec, h->stream));
  if (bands.blob) {
    const BandImages& r = bands.tput_band;
    SART_CUDA(launch_fold_replicas(r.w, r.w2, int(r.repMask) + 1, r.repStride, r.repStride, bands.band.w, bands.band.w2, h->stream));
  }
  if (qhists.blob) {   // the replicas hold sums only where the kernel kept them out of shared memory; zeros cost no adds
    const QuantityHists& q = qhists.qh;
    SART_CUDA(launch_fold_replicas(q.rw, q.rw2, int(q.repMask) + 1, q.repStride, size_t(q.entries), q.w, q.w2, h->stream));
  }
  return SART_OK;
}

int sart_trace_mc(sart_handle_t* h, uint64_t first_ray, uint64_t n_rays, uint64_t seed) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (!h->d_image) return fail(SART_ERR_NOMEM, "the image buffers of this handle could not be allocated");
  DeviceGuard dg(h->device);
  if (h->sampler == SART_SAMPLER_ALIAS && (h->precision != 2 || h->n_masses > 1))
    return fail(SART_ERR_CONFIG, "the alias sampler needs precision mode 2 and a single axion mass");
  const Accum &spec = h->accum[kSpectra], &mspec = h->accum[kMassSpectra];
  const Accum &mrad = h->accum[kMassRadialHist], &mbands = h->accum[kMassBandImages];
  const bool massRows = mrad.blob || mbands.blob;
  const bool perMass = mspec.blob || massRows;   // the per-mass accumulators run the mass-scan kernels for every M
  if (spec.blob && h->n_masses > 1) return fail(SART_ERR_CONFIG, "sart_trace_mc: the spectra need a single axion mass");
  if (spec.blob && massRows)   // the mass-scan kernels fill the per-mass spectra, not these
    return fail(SART_ERR_CONFIG, "sart_trace_mc: the spectra need a single axion mass and the per-mass radial histograms "
                                 "and band images off (use sart_enable_mass_spectra)");
  if (mspec.blob && h->sampler == SART_SAMPLER_ALIAS)
    return fail(SART_ERR_CONFIG, "sart_trace_mc: the per-mass spectra run the mass-scan kernels, which need the inverse-CDF sampler");
  if (massRows && h->sampler == SART_SAMPLER_ALIAS)
    return fail(SART_ERR_CONFIG, "sart_trace_mc: the per-mass radial histograms and band images run the mass-scan kernels, "
                                 "which need the inverse-CDF sampler");
  const Accum& bands = h->accum[kBandImages];
  if (bands.blob && (h->n_masses > 1 || perMass))
    return fail(SART_ERR_CONFIG, "sart_trace_mc: the band images need a single axion mass and the per-mass spectra, radial "
                                 "histograms and band images off");
  const Accum& qhists = h->accum[kQuantityHists];
  if (qhists.blob && (h->n_masses > 1 || perMass))
    return fail(SART_ERR_CONFIG, "sart_trace_mc: the quantity histograms need a single axion mass and the per-mass spectra, "
                                 "radial histograms and band images off");
  const size_t plane = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS;
  int rc = SART_OK;
  // A mass scan, or any run with a per-mass accumulator on (one contract for every mass list, M = 1 included): the exact
  // kernels add the per-mass spectra, radial histograms and band images into the handle's rows directly, the throughput
  // kernels into mass-minor accumulators that k_fold_mass_spectra, k_fold_mass_hist and k_fold_mass_acc add up after every
  // launch.
  if (h->n_masses > 1 || perMass) {
    Tables et = h->tables;
    et.spec = mspec.spec;   // or off
    const MassRows rows{mrad.rad, mbands.band}, acc{mrad.tput_rad, mbands.tput_band};   // or off
    if (h->precision == 0) {
      SART_CUDA(launch_mc_image_exact(h->params, et, h->n_masses, h->d_masses, first_ray, n_rays, seed, h->d_image,
                                      h->d_image_w2, h->d_counters, h->sm_count, h->stream, {}, {}, rows));
      return SART_OK;
    }
    const size_t accLen = plane * SART_MAX_MASSES;
    if (!h->d_mass_acc) {
      SART_CUDA(cudaMalloc(&h->d_mass_acc, 2 * accLen * sizeof(double)));
      SART_CUDA(cudaMemsetAsync(h->d_mass_acc, 0, 2 * accLen * sizeof(double), h->stream));
    }
    fast::FastTables ft = h->ftables;
    ft.spec = mspec.tput;   // or off
    // the 32-bit counts of the per-mass accumulators are folded after every launch of at most kMaxRaysPerLaunch rays
    auto fold_spectra = [&]() {
      cudaError_t e = cudaSuccess;
      if (mspec.blob) e = launch_fold_mass_spectra(mspec.tput, h->n_masses, mspec.bins, mspec.spec, h->stream);
      if (e == cudaSuccess && mrad.blob)
        e = launch_fold_mass_hist(acc.rad.w, reinterpret_cast<unsigned int*>(acc.rad.n), h->n_masses, mrad.bins, mrad.rad.w,
                                  mrad.rad.n, h->stream);
      if (e == cudaSuccess && mbands.blob)
        e = launch_fold_mass_hist(nullptr, reinterpret_cast<unsigned int*>(acc.band.n), h->n_masses, mbands.bins, nullptr,
                                  mbands.band.n, h->stream);
      if (e == cudaSuccess && mbands.blob)
        e = launch_fold_mass_acc(acc.band.w, acc.band.w2, h->n_masses, size_t(mbands.bins) * plane, mbands.band.w, mbands.band.w2,
                                 h->stream);
      return e;
    };
    if (h->precision == 2) {
      rc = f32_then_retrace(h, n_rays, true,   // the alias sampler was refused above
          [&](uint64_t done, uint64_t m, const fast::RetraceQueue& q) {
            ft.rq = q;
            const cudaError_t e = launch_mc_image_f32_masses(h->fparams, h->geo32, ft, h->n_masses, h->d_masses, first_ray + done,
                                                             m, seed, h->d_mass_acc, h->d_mass_acc + accLen, h->d_counters,
                                                             h->sm_count, h->stream, acc);
            return e != cudaSuccess ? e : fold_spectra();
          },
          [&](uint64_t done, uint64_t, const fast::RetraceQueue& q) {
            return launch_retrace_mc_image(h->params, et, h->n_masses, h->d_masses, first_ray + done, seed, q, h->d_image,
                                           h->d_image_w2, h->d_counters, h->sm_count, h->stream, {}, {}, rows);
          });
      if (rc) return rc;
    } else if (!perMass) {
      SART_CUDA(launch_mc_image_fast_masses(h->fparams, ft, h->n_masses, h->d_masses, first_ray, n_rays, seed,
                                            h->d_mass_acc, h->d_mass_acc + accLen, h->d_counters, h->sm_count, h->stream));
    } else {
      for (uint64_t done = 0; done < n_rays; done += fast::kMaxRaysPerLaunch) {
        const uint64_t m = std::min<uint64_t>(n_rays - done, fast::kMaxRaysPerLaunch);
        SART_CUDA(launch_mc_image_fast_masses(h->fparams, ft, h->n_masses, h->d_masses, first_ray + done, m, seed,
                                              h->d_mass_acc, h->d_mass_acc + accLen, h->d_counters, h->sm_count, h->stream, acc));
        SART_CUDA(fold_spectra());
      }
    }
    SART_CUDA(launch_fold_mass_acc(h->d_mass_acc, h->d_mass_acc + accLen, h->n_masses, plane, h->d_image, h->d_image_w2,
                                   h->stream));
    return SART_OK;
  }
  Tables et = h->tables;
  et.spec = spec.spec;   // mode 0 and the re-trace of mode 2 add into the spectra directly
  fast::FastTables ft = h->ftables;
  double *img = h->d_image, *img2 = h->d_image_w2;
  if (h->precision >= 1) {
    if ((rc = ensure_replicas(h))) return rc;
    ft.spec = spec.tput;   // the spectra replicas, or off
    if (h->n_rep > 1) {
      ft.nImgRep = h->n_rep; ft.imgRepStride = h->rep_stride;
      img = h->d_rep; img2 = h->d_rep + size_t(h->n_rep) * h->rep_stride;
    }
  }
  // band images: the throughput kernels add into their replicas, the exact kernels into the handle's arrays
  rc = trace_image(h, h->params, h->fparams, h->geo32, ft, et, first_ray, n_rays, seed, img, img2, h->d_image, h->d_image_w2,
                   h->d_counters, bands.tput_band, bands.band, qhists.qh);
  if (rc || h->precision == 0) return rc;
  if (h->n_rep > 1)
    SART_CUDA(launch_fold_replicas(img, img2, h->n_rep, h->rep_stride, plane, h->d_image, h->d_image_w2, h->stream));
  return fold_accums(h, h->accum);
}

int sart_reset_image(sart_handle_t* h) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  DeviceGuard dg(h->device);
  const size_t len = size_t(h->n_masses) * SART_IMAGE_BINS * SART_IMAGE_BINS;
  SART_CUDA(cudaMemsetAsync(h->d_image, 0, 2 * len * sizeof(double), h->stream));   // image | w^2 image: one block
  SART_CUDA(cudaMemsetAsync(h->d_counters, 0, size_t(h->n_masses) * sizeof(sart_counters_t), h->stream));
  for (AccumKind k : kAllAccums)
    if (int rc = clear_accum(h, k)) return rc;
  return SART_OK;
}

// The argument checks of sart_enable_band_images and sart_enable_mass_band_images.
static int check_band_edges(int n_bands, const double* edges_keV, const char* who) {
  if (n_bands < 0 || n_bands > SART_MAX_BANDS || (n_bands > 0 && !edges_keV))
    return fail(SART_ERR_ARG, "%s: need 1..%d bands and their edges, or 0 (off)", who, SART_MAX_BANDS);
  for (int b = 0; n_bands > 0 && b <= n_bands; ++b)
    if (!std::isfinite(edges_keV[b]) || edges_keV[b] < 0.0 || (b > 0 && !(edges_keV[b] > edges_keV[b - 1])))
      return fail(SART_ERR_ARG, "%s: the band edges must be finite, >= 0 and strictly ascending", who);
  return SART_OK;
}

int sart_enable_mass_radial_hist(sart_handle_t* h, int nbins, double r_max) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (nbins < 0 || nbins > (1 << 24) || (nbins > 0 && !(r_max > 0.0)))
    return fail(SART_ERR_ARG, "sart_enable_mass_radial_hist: bad argument");
  if (nbins > 0 && h->accum[kRadialHist].blob)
    return fail(SART_ERR_CONFIG, "sart_enable_mass_radial_hist: the single-mass radial histogram is on (sart_enable_radial_hist); "
                                 "switch it off first");
  return set_accum(h, kMassRadialHist, nbins, r_max);
}

int sart_read_mass_radial_hist(sart_handle_t* h, double* sum_w, uint64_t* counts) {
  return read_accum(h, kMassRadialHist, false, {sum_w, counts},
                    "sart_read_mass_radial_hist: no per-mass radial histograms enabled (sart_enable_mass_radial_hist)");
}

int sart_enable_mass_band_images(sart_handle_t* h, int n_bands, const double* edges_keV) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (int rc = check_band_edges(n_bands, edges_keV, "sart_enable_mass_band_images")) return rc;
  if (n_bands > 0 && h->accum[kBandImages].blob)
    return fail(SART_ERR_CONFIG, "sart_enable_mass_band_images: the single-mass band images are on (sart_enable_band_images); "
                                 "switch them off first");
  return set_accum(h, kMassBandImages, n_bands, 0.0, edges_keV);
}

int sart_read_mass_band_images(sart_handle_t* h, double* image, double* image_w2, uint64_t* counts) {
  return read_accum(h, kMassBandImages, false, {image, image_w2, counts},
                    "sart_read_mass_band_images: no per-mass band images enabled (sart_enable_mass_band_images)");
}

int sart_enable_mass_spectra(sart_handle_t* h, int on) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (on && h->accum[kSpectra].blob)
    return fail(SART_ERR_CONFIG, "sart_enable_mass_spectra: the single-mass spectra are on (sart_enable_spectra); switch them off first");
  return set_accum(h, kMassSpectra, on ? h->params.nEnergies + 1 : 0);
}

int sart_read_mass_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                           double* shell_sum_w, uint64_t* shell_counts) {
  return read_accum(h, kMassSpectra, false, {energy_sum_w, energy_sum_w2, energy_counts, shell_sum_w, shell_counts},
                    "sart_read_mass_spectra: no per-mass spectra enabled (sart_enable_mass_spectra)");
}

int sart_enable_spectra(sart_handle_t* h, int on) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (on && h->accum[kMassSpectra].blob)
    return fail(SART_ERR_CONFIG, "sart_enable_spectra: the per-mass spectra are on (sart_enable_mass_spectra); switch them off first");
  return set_accum(h, kSpectra, on ? h->params.nEnergies + 1 : 0);   // the last energy bin is the X-ray source's
}

int sart_read_spectra(sart_handle_t* h, double* energy_sum_w, double* energy_sum_w2, uint64_t* energy_counts,
                      double* shell_sum_w, uint64_t* shell_counts) {
  return read_accum(h, kSpectra, false, {energy_sum_w, energy_sum_w2, energy_counts, shell_sum_w, shell_counts},
                    "sart_read_spectra: no spectra enabled (sart_enable_spectra)");
}

int sart_enable_band_images(sart_handle_t* h, int n_bands, const double* edges_keV) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (int rc = check_band_edges(n_bands, edges_keV, "sart_enable_band_images")) return rc;
  if (n_bands > 0 && h->accum[kMassBandImages].blob)
    return fail(SART_ERR_CONFIG, "sart_enable_band_images: the per-mass band images are on (sart_enable_mass_band_images); "
                                 "switch them off first");
  return set_accum(h, kBandImages, n_bands, 0.0, edges_keV);
}

int sart_read_band_images(sart_handle_t* h, double* image, double* image_w2, uint64_t* counts) {
  return read_accum(h, kBandImages, false, {image, image_w2, counts},
                    "sart_read_band_images: no band images enabled (sart_enable_band_images)");
}

int sart_enable_quantity_hists(sart_handle_t* h, int n, const sart_quantity_hist_t* hists) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (n < 0 || n > SART_N_QUANTITIES || (n > 0 && !hists))
    return fail(SART_ERR_ARG, "sart_enable_quantity_hists: need 1..%d histograms and their specs, or 0 (off)", SART_N_QUANTITIES);
  int entries = 0;
  unsigned seen = 0;
  for (int j = 0; j < n; ++j) {
    const sart_quantity_hist_t& q = hists[j];
    if (q.quantity < 0 || q.quantity >= SART_N_QUANTITIES || (seen & (1u << q.quantity)))
      return fail(SART_ERR_ARG, "sart_enable_quantity_hists: histogram %d: unknown or repeated quantity %d", j, int(q.quantity));
    if (q.nbins < 1 || q.nbins > SART_MAX_QHIST_BINS)
      return fail(SART_ERR_ARG, "sart_enable_quantity_hists: histogram %d: need 1..%d bins", j, SART_MAX_QHIST_BINS);
    if (!std::isfinite(q.lo) || !std::isfinite(q.hi) || !(q.lo < q.hi))
      return fail(SART_ERR_ARG, "sart_enable_quantity_hists: histogram %d: lo and hi must be finite with lo < hi", j);
    seen |= 1u << q.quantity;
    entries += q.nbins + 2;
  }
  return set_accum(h, kQuantityHists, entries, 0.0, nullptr, n, hists);
}

int sart_read_quantity_hists(sart_handle_t* h, double* sum_w, double* sum_w2, uint64_t* counts) {
  return read_accum(h, kQuantityHists, false, {sum_w, sum_w2, counts},
                    "sart_read_quantity_hists: no quantity histograms enabled (sart_enable_quantity_hists)");
}

int sart_enable_radial_hist(sart_handle_t* h, int nbins, double r_max) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (nbins < 0 || nbins > (1 << 24) || (nbins > 0 && !(r_max > 0.0))) return fail(SART_ERR_ARG, "sart_enable_radial_hist: bad argument");
  if (nbins > 0 && h->accum[kMassRadialHist].blob)
    return fail(SART_ERR_CONFIG, "sart_enable_radial_hist: the per-mass radial histograms are on (sart_enable_mass_radial_hist); "
                                 "switch them off first");
  return set_accum(h, kRadialHist, nbins, r_max);
}

int sart_read_radial_hist(sart_handle_t* h, double* sum_w, uint64_t* counts) {
  return read_accum(h, kRadialHist, false, {sum_w, counts}, "sart_read_radial_hist: no radial histogram enabled");
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
  double *dRes, *dX, *dY, *dW;
  unsigned long long* dBad;
  auto layout = [&](Carve c) { c.take(dRes, cells); c.take(dBad, 1); c.take(dX, n); c.take(dY, n); c.take(dW, n); return c.off; };
  int rc = ensure_stage(h, layout(Carve()));
  if (rc) return rc;
  layout(Carve(h->d_stage));
  SART_CUDA(cudaMemsetAsync(dRes, 0, cells * sizeof(double), h->stream));
  SART_CUDA(cudaMemsetAsync(dBad, 0, sizeof *dBad, h->stream));
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

// The caller's arrays of accumulator k in a sart_scan_out_t, in the order of accum_arrays, into p; returns their number (0:
// an accumulator without rows in a scan).
static int scan_out_arrays(const sart_scan_out_t& o, AccumKind k, void** p) {
  switch (k) {
    case kRadialHist: p[0] = o.radial_sum_w; p[1] = o.radial_counts; return 2;
    case kSpectra:
      p[0] = o.energy_sum_w; p[1] = o.energy_sum_w2; p[2] = o.energy_counts; p[3] = o.shell_sum_w; p[4] = o.shell_counts;
      return 5;
    case kBandImages: p[0] = o.band_image; p[1] = o.band_image_w2; p[2] = o.band_counts; return 3;
    case kQuantityHists: p[0] = o.qhist_sum_w; p[1] = o.qhist_sum_w2; p[2] = o.qhist_counts; return 3;
    default: return 0;
  }
}

// sart_angular_scan, and with `out` sart_angular_scan_outputs: then every single-mass accumulator the handle has on also
// gets one row per scan point, in the stage buffer next to the images, copied into the caller's arrays `out` at the end.
// Without `out` the scan runs the kernels a run without accumulators runs.
static int angular_scan(sart_handle* h, int n_angles, const double* angles_deg, uint64_t first_ray, uint64_t n_rays_per_angle,
                        uint64_t seed, double* fluxes, sart_counters_t* counters, double* images, const sart_scan_out_t* out) {
  DeviceGuard dg(h->device);
  const size_t plane = size_t(SART_IMAGE_BINS) * SART_IMAGE_BINS;
  double *dImg, *dImg2;
  sart_counters_t* dCnt;
  Accum rows[kAccums];   // bins > 0: the [n_angles] rows of accumulator k, shaped like the handle's
  auto layout = [&](Carve c) {
    c.take(dImg, size_t(n_angles) * plane); c.take(dImg2, size_t(n_angles) * plane); c.take(dCnt, size_t(n_angles));
    void* unused[5];
    for (AccumKind k : kAllAccums) {
      if (!out || !h->accum[k].blob || !scan_out_arrays(*out, k, unused)) continue;
      rows[k] = Accum{};
      rows[k].bins = h->accum[k].bins;
      accum_arrays(k, rows[k], rows[k], size_t(n_angles), [&](auto*& p, auto*&, size_t n) { c.take(p, n); });
    }
    return c.off;
  };
  const size_t bytes = layout(Carve());
  int rc = ensure_stage(h, bytes);
  if (rc && out) {
    cudaGetLastError();   // the failed cudaMalloc must not surface at the next launch
    return fail(SART_ERR_NOMEM, "sart_angular_scan_outputs: no room for the %zu bytes of the scan points' images and rows", bytes);
  }
  if (rc) return rc;
  layout(Carve(h->d_stage));
  SART_CUDA(cudaMemsetAsync(h->d_stage, 0, bytes, h->stream));
  // One launch per scan point, queued back to back on the handle's stream: only the by-value parameter block differs
  // (the rotation of the telescope frame), the tables and shell records in HBM are shared, nothing synchronises.
  for (int i = 0; i < n_angles; ++i) {
    // The accumulators of scan point i: the handle's, with every array the kernels add into directly moved to row i. The
    // replicas of the throughput kernels stay the handle's: each fold below clears them for the next point.
    Accum v[kAccums];
    for (AccumKind k : kAllAccums) {
      if (!rows[k].bins) continue;
      v[k] = h->accum[k];
      accum_arrays(k, v[k], rows[k], 1, [&](auto*& p, auto* r, size_t n) { p = r + size_t(i) * n; });
    }
    v[kBandImages].tput_band.n = v[kBandImages].band.n;   // the band counts are never replicated
    fast::FastTables ft = h->ftables;
    Tables et = h->tables;
    ft.rad = et.rad = v[kRadialHist].rad;
    ft.spec = v[kSpectra].tput;
    et.spec = v[kSpectra].spec;
    sart_setup_t s = h->setup;
    s.telescope.telescope_turned_y = angles_deg[i];   // rt:2796
    Params P;
    rederive_params(h, s, &P);
    fast::FastParams F{};
    fast::Geo32 G{};
    if (h->precision >= 1) {
      fast::derive_params(s, P, &F);
      F.shellRhoMin = h->fparams.shellRhoMin; F.shellInvStep = h->fparams.shellInvStep; F.nShellGuide = h->fparams.nShellGuide;
    }
    if (h->precision == 2) {
      std::vector<fast::ShellF32> unused(SART_MAX_SHELLS);
      fast::derive_f32(F, nullptr, 0, &G, unused.data());
      // error budgets: the handle's (they depend on the shells, which do not turn), doubled where the rotation of the
      // telescope frame adds rounding steps
      G.tol = h->geo32.tol;
      if (F.rotated && !h->fparams.rotated) { G.tol.latA *= 2.0f; G.tol.detA *= 2.0f; }
    }
    const uint64_t first = first_ray + uint64_t(i) * n_rays_per_angle;   // every scan point traces its own rays, like the reference
    double *img = dImg + size_t(i) * plane, *img2 = dImg2 + size_t(i) * plane;
    if ((rc = trace_image(h, P, F, G, ft, et, first, n_rays_per_angle, seed, img, img2, img, img2, dCnt + i,
                          v[kBandImages].tput_band, v[kBandImages].band, v[kQuantityHists].qh)))
      return rc;
    if (h->precision >= 1 && (rc = fold_accums(h, v))) return rc;
  }
  std::vector<sart_counters_t> cnt;
  cnt.resize(size_t(n_angles));
  SART_CUDA(cudaMemcpyAsync(cnt.data(), dCnt, cnt.size() * sizeof(sart_counters_t), cudaMemcpyDeviceToHost, h->stream));
  if (images) SART_CUDA(cudaMemcpyAsync(images, dImg, size_t(n_angles) * plane * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  for (AccumKind k : kAllAccums) {
    if (!rows[k].bins) continue;
    void* host[5] = {};
    scan_out_arrays(*out, k, host);
    void* const* hp = host;
    cudaError_t e = cudaSuccess;
    accum_arrays(k, rows[k], rows[k], size_t(n_angles), [&](auto* d, auto*, size_t n) {
      void* p = *hp++;
      if (p && e == cudaSuccess) e = cudaMemcpyAsync(p, d, n * sizeof *d, cudaMemcpyDeviceToHost, h->stream);
    });
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync (scan rows, device to host)");
  }
  SART_CUDA(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < n_angles; ++i) fluxes[i] = cnt[size_t(i)].sum_w;   // axions.filterIt(it.passed).mapIt(it.weights).sum() rt:2800
  if (counters) std::memcpy(counters, cnt.data(), cnt.size() * sizeof(sart_counters_t));
  return SART_OK;
}

// The checks both scan entry points make.
static int check_scan(sart_handle* h, int n_angles, const double* angles_deg, double* fluxes, const char* who) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  if (n_angles < 1 || !angles_deg || !fluxes) return fail(SART_ERR_ARG, "%s: bad argument", who);
  if (h->n_masses != 1) return fail(SART_ERR_ARG, "%s: set a single axion mass", who);
  if (h->sampler == SART_SAMPLER_ALIAS && h->precision != 2)
    return fail(SART_ERR_CONFIG, "the alias sampler needs precision mode 2");
  return SART_OK;
}

int sart_angular_scan(sart_handle_t* h, int n_angles, const double* angles_deg, uint64_t first_ray,
                      uint64_t n_rays_per_angle, uint64_t seed, double* fluxes, sart_counters_t* counters, double* images) {
  const int rc = check_scan(h, n_angles, angles_deg, fluxes, "sart_angular_scan");
  return rc ? rc : angular_scan(h, n_angles, angles_deg, first_ray, n_rays_per_angle, seed, fluxes, counters, images, nullptr);
}

int sart_angular_scan_outputs(sart_handle_t* h, int n_angles, const double* angles_deg, uint64_t first_ray,
                              uint64_t n_rays_per_angle, uint64_t seed, double* fluxes, sart_counters_t* counters,
                              double* images, const sart_scan_out_t* out) {
  int rc = check_scan(h, n_angles, angles_deg, fluxes, "sart_angular_scan_outputs");
  if (rc) return rc;
  if (h->accum[kMassSpectra].blob)
    return fail(SART_ERR_CONFIG, "sart_angular_scan_outputs: the per-mass spectra are on; a scan fills single-mass rows only");
  if (h->accum[kMassRadialHist].blob || h->accum[kMassBandImages].blob)
    return fail(SART_ERR_CONFIG, "sart_angular_scan_outputs: the per-mass radial histograms or band images are on; a scan fills "
                                 "single-mass rows only");
  const sart_scan_out_t none{};
  if (!out) out = &none;
  static const char* const names[kAccums] = {"radial histogram", "spectra", "per-mass spectra", "band images",
                                             "quantity histograms", "per-mass radial histograms", "per-mass band images"};
  bool any = false;
  for (AccumKind k : kAllAccums) {
    void* p[5];
    const int np = scan_out_arrays(*out, k, p);
    any |= np > 0 && h->accum[k].blob != nullptr;
    for (int j = 0; j < np && !h->accum[k].blob; ++j)
      if (p[j]) return fail(SART_ERR_ARG, "sart_angular_scan_outputs: an output array for the %s, which the handle has off", names[k]);
  }
  if (!any)
    return fail(SART_ERR_ARG, "sart_angular_scan_outputs: no radial histogram, spectra, band images or quantity histograms "
                              "are on (sart_angular_scan scans without them)");
  return angular_scan(h, n_angles, angles_deg, first_ray, n_rays_per_angle, seed, fluxes, counters, images, out);
}

int sart_synchronize(sart_handle_t* h) {
  if (!h) return fail(SART_ERR_ARG, "handle is NULL");
  DeviceGuard dg(h->device);
  SART_CUDA(cudaStreamSynchronize(h->stream));
  return SART_OK;
}

}  // extern "C"
