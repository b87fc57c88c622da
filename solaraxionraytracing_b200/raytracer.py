"""Host-side mirror of the reference's driver for the per-ray path, on top of the C-ABI (include/sart.h).

Names follow src/raytracer.nim: `initFullSetup` (rt:2637-2753) builds a `FullRaytraceSetup` (rt:232-242),
`traceAxionWrapper` (rt:2223-2244) fills per-ray `Axion` records (here a structure of arrays),
`calculateFluxFractions` (rt:2755-2776) runs the whole Monte Carlo and returns the 256x256 detector image that
`prepareHeatmap` (rt:818-842) would build, plus the counters `generateResultPlots` prints (rt:2252-2257).
Everything numeric happens in libsart.so on the GPU; this module only moves numpy arrays across the boundary.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import abi, tables as _tables
from ._lib import SartError, check, lib  # noqa: F401  (re-exported)
from .output import BandImages, QuantityHist, ScanOutputs, Spectra, check_quantity_hist_specs, quantity_hist_edges


def _dp(a: np.ndarray):
    return a.ctypes.data_as(abi.c_double_p)


def _ptr(a: np.ndarray):
    """A float64 or uint64 array as the ctypes pointer the C-ABI takes."""
    return a.ctypes.data_as(abi.c_double_p if a.dtype == np.float64 else C.POINTER(C.c_uint64))


def fast_available() -> bool:
    """True if this build of libsart has the mixed-precision ("fast") pipeline."""
    return bool(lib.sart_has_precision(1))


def flags_from_cli(ignoreDetWindow=False, ignoreGasAbs=False, ignoreConvProb=False, ignoreReflection=False,
                   xrayTest=False, magnet=False, detectorInstall=False) -> int:
    """The flag set `main` builds from its CLI switches (rt:2842-2849)."""
    f = 0
    if ignoreDetWindow: f |= abi.CF_IGNORE_DET_WINDOW
    if ignoreGasAbs: f |= abi.CF_IGNORE_GAS_ABS
    if ignoreConvProb: f |= abi.CF_IGNORE_CONV_PROB
    if ignoreReflection: f |= abi.CF_IGNORE_REFLECTION
    if xrayTest: f |= abi.CF_XRAY_TEST
    if magnet: f |= abi.CF_READ_MAGNET_CONFIG
    if detectorInstall: f |= abi.CF_READ_DET_INSTALL_CONFIG
    return f


def newExperimentSetup(experiment, detector, stage, telescope, flags: int = 0) -> abi.Setup:
    """newExperimentSetup (rt:1411-1423) + newDetectorSetup (rt:1464-1496): C++ constructors in libsart.
    Accepts the reference's enum strings ("CAST", "InGrid2018", "vacuum", "LLNL") or the integer kinds."""
    def kind(v, table):
        if isinstance(v, str):
            if v not in table:
                raise ValueError(f"invalid enum value {v!r}; expected one of {sorted(table)}")  # parseEnum raises
            return table[v]
        return int(v)
    s = abi.Setup()
    check(lib.sart_init_setup(kind(experiment, abi.EXPERIMENT_KINDS), kind(detector, abi.DETECTOR_KINDS),
                              kind(stage, abi.STAGE_KINDS), kind(telescope, abi.TELESCOPE_KINDS), flags, C.byref(s)))
    return s


def calcWindowVals(radiusWindow: float, numberOfStrips: int, openApertureRatio: float):
    """calcWindowVals (rt:1431-1462) -> (width, dist) in mm."""
    w, d = C.c_double(), C.c_double()
    check(lib.sart_calc_window_vals(radiusWindow, numberOfStrips, openApertureRatio, C.byref(w), C.byref(d)))
    return w.value, d.value


def buildCdfs(emission: _tables.EmissionTable, device: int = 0):
    """The CDF build of initFullSetup (rt:2679-2705) on the GPU -> (fluxRadiusCDF [nR], diffFluxCDFs [nR, nE])."""
    radii = np.ascontiguousarray(emission.radii, dtype=np.float64)
    en = np.ascontiguousarray(emission.energies, dtype=np.float64)
    em = np.ascontiguousarray(emission.emRates, dtype=np.float64)
    nR, nE = em.shape
    rc = np.empty(nR)
    dc = np.empty((nR, nE))
    check(lib.sart_build_cdfs(device, nR, nE, _dp(radii), _dp(en), _dp(em), _dp(rc), _dp(dc)))
    return rc, dc


def calculateEmissionRates(solarModel: _tables.SolarModel | None = None, processes=("primakoff",), nElems: int = 1500,
                           g_ae: float = 1e-13, gagamma: float = 1e-12, ganuclei: float = 1e-15,
                           device: int = 0) -> _tables.EmissionTable:
    """The opacity-free part of calculateOpacities (src/readOpacityFile.nim:598-860) on the GPU: emission rates on
    energies = linspace(1e-3, 15, nElems) keV (:608-609) for every radius of the solar model. `processes` names
    SART_EM_* terms ("primakoff", "compton", "ee_brems", "free_free", "iron57", "long_plasmon")."""
    sm = solarModel or _tables.solar_model_packaged()
    bits = 0
    for p in processes:
        if p not in abi.EM_PROCESSES:
            raise ValueError(f"unknown emission process {p!r}; expected one of {sorted(abi.EM_PROCESSES)}")
        bits |= abi.EM_PROCESSES[p]
    energies = np.linspace(1e-3, 15.0, nElems)
    T = np.ascontiguousarray(sm.temp_K, dtype=np.float64)
    rho = np.ascontiguousarray(sm.rho_gcm3, dtype=np.float64)
    fr = np.ascontiguousarray(sm.mass_fractions, dtype=np.float64)
    em = np.empty((T.size, nElems))
    check(lib.sart_emission_rates(device, T.size, _dp(T), _dp(rho), _dp(fr), nElems, _dp(energies), bits, g_ae, gagamma,
                                  ganuclei, _dp(em)))
    radii = 0.0015 + 0.0005 * np.arange(T.size)   # readOpacityFile.nim:793
    return _tables.EmissionTable(radii=radii, energies=energies, emRates=em)


@dataclass
class FullRaytraceSetup:
    """FullRaytraceSetup (rt:232-242)."""
    expSetup: abi.Setup
    tables: _tables.TableSet
    outpath: str = "out"

    @property
    def flags(self) -> int:
        return self.expSetup.flags


class AxionBatch:
    """Per-ray results, the `Axion` record (rt:192-221) as a structure of numpy arrays."""

    def __init__(self, n: int, optional: bool = True, pinned=None):
        self.n = n
        def alloc(dtype=np.float64):
            return np.zeros(n, dtype=dtype)
        self.x = alloc(); self.y = alloc(); self.w = alloc()
        self.code = alloc(np.int32); self.shell = alloc(np.int32)
        for name in abi.RAY_OUT_OPTIONAL:   # optional: True / False, or the names of the optional arrays wanted
            want = (name in optional) if isinstance(optional, (tuple, list, set)) else bool(optional)
            setattr(self, name, alloc() if want else None)

    def c_struct(self) -> abi.RayOut:
        o = abi.RayOut()
        o.x, o.y, o.w = _dp(self.x), _dp(self.y), _dp(self.w)
        o.code = self.code.ctypes.data_as(abi.c_int32_p)
        o.shell = self.shell.ctypes.data_as(abi.c_int32_p)
        for name in abi.RAY_OUT_OPTIONAL:
            a = getattr(self, name)
            if a is not None:
                setattr(o, name, _dp(a))
        return o

    @property
    def exit_code(self) -> np.ndarray:
        return self.code & abi.CODE_MASK

    @property
    def passed(self) -> np.ndarray:          # Axion.passed
        return self.exit_code == abi.EXIT_PASSED

    @property
    def passedTillWindow(self) -> np.ndarray:  # Axion.passedTillWindow
        return (self.code & abi.FLAG_PASSED_TILL_WINDOW) != 0

    @property
    def hitNickel(self) -> np.ndarray:       # Axion.hitNickel
        return self.exit_code == abi.EXIT_NICKEL


@dataclass
class RunResult:
    image: np.ndarray        # [M, 256, 256] (M = number of axion masses), image[m, y, x] like heatmaptable2 rt:2629
    image_w2: np.ndarray     # sum of squared weights per bin (Monte Carlo variance)
    counters: list           # one dict per mass


class RayTracer:
    """One GPU's ray-tracing context: owns a sart_handle_t (tables resident in HBM, one stream)."""

    def __init__(self, fullSetup: FullRaytraceSetup, device: int = 0):
        self.fullSetup = fullSetup
        self._h = abi.H()
        self._tstruct = fullSetup.tables.c_struct()
        check(lib.sart_create(C.byref(fullSetup.expSetup), C.byref(self._tstruct), device, C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h:
            lib.sart_destroy(self._h)
            self._h = abi.H()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- configuration
    def update_setup(self, setup: abi.Setup):
        check(lib.sart_update_setup(self._h, C.byref(setup)))
        self.fullSetup.expSetup = setup

    def set_axion_masses(self, masses):
        m = np.ascontiguousarray(masses, dtype=np.float64)
        check(lib.sart_set_axion_masses(self._h, m.size, _dp(m)))

    def set_precision(self, mode: int):
        check(lib.sart_set_precision(self._h, mode))

    def set_sampler(self, sampler: int):
        """abi.SAMPLER_INVERSE_CDF (default: the reference's lowerBound, same rays as the oracle) or abi.SAMPLER_ALIAS
        (same distributions through alias tables: statistical parity only, precision mode 2)."""
        check(lib.sart_set_sampler(self._h, sampler))

    def set_retrace(self, mode: int = 1, scale: float = 1.0):
        """Precision mode 2: re-trace the rays whose FP32 decision margins are inside their error budgets with the exact
        FP64 pipeline (default on); `scale` multiplies the budgets."""
        check(lib.sart_set_retrace(self._h, mode, scale))

    def set_compaction(self, mode: int):
        check(lib.sart_set_compaction(self._h, mode))

    @property
    def n_masses(self) -> int:
        return lib.sart_image_len(self._h) // (abi.IMAGE_BINS * abi.IMAGE_BINS)

    @property
    def stream(self) -> int:
        return lib.sart_stream(self._h) or 0

    # -- tier (a): pre-sampled rays
    def trace_presampled(self, origin_xyz, exit_xy, energy, optional: bool = True) -> AxionBatch:
        origin_xyz = np.ascontiguousarray(origin_xyz, dtype=np.float64)
        exit_xy = np.ascontiguousarray(exit_xy, dtype=np.float64)
        energy = np.ascontiguousarray(energy, dtype=np.float64)
        n = energy.size
        if origin_xyz.shape != (3, n) or exit_xy.shape != (2, n):
            raise ValueError("origin_xyz must be [3, n] and exit_xy [2, n] (structure of arrays)")
        out = AxionBatch(n, optional)
        o = out.c_struct()
        check(lib.sart_trace_presampled(self._h, n, _dp(origin_xyz), _dp(exit_xy), _dp(energy), C.byref(o)))
        return out

    def trace_presampled_dev(self, n: int, d_origin: int, d_exit: int, d_energy: int, d_out: abi.RayOut):
        """Device-pointer variant (asynchronous on `stream`)."""
        check(lib.sart_trace_presampled_dev(self._h, n, d_origin, d_exit, d_energy, C.byref(d_out)))

    # -- traceAxionWrapper: Monte Carlo rays, per-ray records
    def traceAxionWrapper(self, bufLen: int, seed: int = 299792458, first_ray: int = 0,
                          optional: bool = True) -> AxionBatch:
        out = AxionBatch(bufLen, optional)
        o = out.c_struct()
        check(lib.sart_trace_mc_rays(self._h, first_ray, bufLen, seed, C.byref(o)))
        return out

    def trace_passed(self, n: int, seed: int = 299792458, first_ray: int = 0, fields=("ray", "x", "y", "w", "shell"),
                     capacity: int | None = None, buffers: dict | None = None):
        """sart_trace_mc_passed: the records of the rays that pass only, compacted on the GPU, single precision. Returns
        (dict of numpy arrays cut to the number of passed rays, counters dict). `buffers` supplies pre-allocated
        (e.g. pinned) arrays by field name."""
        cap = int(capacity if capacity is not None else n)
        dtypes = {name: np.dtype(t) for name, t in abi.PASSED_OUT_FIELDS}
        arrays = {}
        po = abi.PassedOut()
        for name in fields:
            a = buffers[name] if buffers and name in buffers else np.empty(cap, dtype=dtypes[name])
            assert a.dtype == dtypes[name] and a.size >= cap and a.flags.c_contiguous
            arrays[name] = a
            setattr(po, name, a.ctypes.data_as(C.POINTER(dict(abi.PASSED_OUT_FIELDS)[name])))
        npass = C.c_uint64(0)
        cnt = abi.Counters()
        check(lib.sart_trace_mc_passed(self._h, first_ray, n, seed, cap, C.byref(po), C.byref(npass), C.byref(cnt)))
        return {k: v[:npass.value] for k, v in arrays.items()}, cnt.as_dict()

    def trace_words(self, words, late_energy: bool = False, optional: bool = True) -> AxionBatch:
        """Test hook (sart_trace_words): traceAxionWrapper with caller-supplied random words [6, n] instead of Philox."""
        w = np.ascontiguousarray(words, dtype=np.uint32)
        if w.ndim != 2 or w.shape[0] != 6:
            raise ValueError("words must be [6, n]")
        out = AxionBatch(w.shape[1], optional)
        o = out.c_struct()
        out.emission_shell = np.empty(w.shape[1], dtype=np.int32)
        check(lib.sart_trace_words(self._h, w.shape[1], w.ctypes.data_as(C.POINTER(C.c_uint32)), int(late_energy),
                                   C.byref(o), out.emission_shell.ctypes.data_as(abi.c_int32_p)))
        return out

    # -- fused run
    def trace_mc(self, n_rays: int, seed: int = 299792458, first_ray: int = 0):
        """Asynchronous: accumulates into the device image."""
        check(lib.sart_trace_mc(self._h, first_ray, n_rays, seed))

    def reset_image(self):
        check(lib.sart_reset_image(self._h))

    def _default_r_max(self, r_max: float | None) -> float:
        if r_max is None:
            c = self.fullSetup.expSetup.consts
            r_max = 0.5 * float(np.hypot(c.chipXMax, c.chipYMax)) * 1.0001
        return r_max

    def enable_radial_hist(self, nbins: int = 16384, r_max: float | None = None):
        """Radial histogram of the passed rays (for the containment radii); r_max defaults to the chip diagonal / 2."""
        r_max = self._default_r_max(r_max)
        check(lib.sart_enable_radial_hist(self._h, nbins, r_max))
        self._rad = (nbins, r_max)

    # Each accumulator's host arrays for `rows` rows (one read, the masses of a mass scan, or the scan points of
    # angular_scan_outputs), in the order the C-ABI takes them, and the function that cuts them into one result per row.
    def _radial_rows(self, rows: int, shape=None):
        nbins, r_max = shape or self._rad
        w = np.empty((rows, nbins))
        n = np.empty((rows, nbins), dtype=np.uint64)
        edges = np.linspace(0.0, r_max, nbins + 1)
        return (w, n), lambda: [(edges.copy(), w[k], n[k]) for k in range(rows)]

    def _read_radial(self, read):
        arrays, split = self._radial_rows(1)
        check(read(self._h, *map(_ptr, arrays)))
        return split()[0]

    def read_radial_hist(self):
        """(bin edges [nbins + 1], sum of weights [nbins], ray counts [nbins])."""
        return self._read_radial(lib.sart_read_radial_hist)

    def enable_mass_radial_hist(self, nbins: int = 16384, r_max: float | None = None):
        """Radial histogram of the rays that pass in trace_mc for every axion mass of set_axion_masses
        (sart_enable_mass_radial_hist), binned like enable_radial_hist, from the one traced ray per mass scan; nbins = 0
        switches them off. Switching them on clears them; trace_mc then runs the mass-scan kernels for any number of masses.
        Not together with enable_radial_hist or the alias sampler."""
        r_max = self._default_r_max(r_max)
        check(lib.sart_enable_mass_radial_hist(self._h, nbins, r_max))
        self._mass_rad = (nbins, r_max)

    def _read_mass_radial(self, read):
        arrays, split = self._radial_rows(self.n_masses, getattr(self, "_mass_rad", (0, 1.0)))
        check(read(self._h, *map(_ptr, arrays)))
        return split()

    def read_mass_radial_hist(self) -> list[tuple]:
        """One (bin edges, sum of weights, ray counts) per axion mass, in the order of set_axion_masses, accumulated since
        enable_mass_radial_hist / reset_image (raises SartError while they are off); each ready for
        output.containment_radii_from_hist."""
        return self._read_mass_radial(lib.sart_read_mass_radial_hist)

    def read_merged_mass_radial_hist(self) -> list[tuple]:
        """read_mass_radial_hist of the last allreduce_outputs (raises SartError without one)."""
        return self._read_mass_radial(lib.sart_read_merged_mass_radial_hist)

    def enable_spectra(self, on: bool = True):
        """Energy spectrum and per-shell flux of the rays that pass in trace_mc (single axion mass; sart_enable_spectra).
        Switching them on clears them; precision modes 1 and 2 then run their generic kernel variant."""
        check(lib.sart_enable_spectra(self._h, int(bool(on))))
        self._spectra_on = bool(on)

    def _spectra_rows(self, rows: int):
        """Each Spectra with the energies of the bins: the tabulated energies, then the X-ray source's (NaN without a
        source); shells cut to the telescope's."""
        en = np.asarray(self.fullSetup.tables.energies if self.fullSetup.tables.energies is not None else [], dtype=np.float64)
        nE1 = en.size + 1
        w, w2 = np.empty((rows, nE1)), np.empty((rows, nE1))
        n = np.empty((rows, nE1), dtype=np.uint64)
        sw = np.empty((rows, abi.MAX_SHELLS))
        sn = np.empty((rows, abi.MAX_SHELLS), dtype=np.uint64)
        s = self.fullSetup.expSetup
        src = s.testSource.energy if s.testSource.active else np.nan
        ns = s.telescope.nShells
        energies = np.append(en, src)
        return (w, w2, n, sw, sn), lambda: [Spectra(energies.copy(), w[k], w2[k], n[k], sw[k, :ns].copy(), sn[k, :ns].copy())
                                            for k in range(rows)]

    def _read_spectra_rows(self, read, rows: int) -> list[Spectra]:
        """`rows` spectra copied out by `read` (sart_read_spectra / sart_read_mass_spectra)."""
        arrays, split = self._spectra_rows(rows)
        check(read(self._h, *map(_ptr, arrays)))
        return split()

    def read_spectra(self) -> Spectra:
        """The spectra accumulated since enable_spectra / reset_image (raises SartError while they are off)."""
        return self._read_spectra_rows(lib.sart_read_spectra, 1)[0]

    def enable_mass_spectra(self, on: bool = True):
        """Energy spectrum and per-shell flux of the rays that pass in trace_mc, for every axion mass of set_axion_masses
        (sart_enable_mass_spectra), from the one traced ray per mass scan. Switching them on clears them; trace_mc then runs
        the mass-scan kernels for any number of masses. Not together with enable_spectra or the alias sampler."""
        check(lib.sart_enable_mass_spectra(self._h, int(bool(on))))

    def read_mass_spectra(self) -> list[Spectra]:
        """One Spectra per axion mass, in the order of set_axion_masses, accumulated since enable_mass_spectra /
        reset_image (raises SartError while they are off)."""
        return self._read_spectra_rows(lib.sart_read_mass_spectra, self.n_masses)

    def enable_band_images(self, edges_keV=None):
        """Detector images of the rays that pass in trace_mc per energy band [edges[b], edges[b + 1]) keV (single axion mass;
        sart_enable_band_images); None switches them off. Switching them on clears them."""
        if edges_keV is None:
            check(lib.sart_enable_band_images(self._h, 0, None))
            self._band_edges = None
            return
        e = np.ascontiguousarray(edges_keV, dtype=np.float64)
        check(lib.sart_enable_band_images(self._h, e.size - 1 if e.size > 1 else -1, _dp(e)))   # one edge: no band, refused
        self._band_edges = e.copy()

    def _band_rows(self, rows: int, edges=False):
        edges = getattr(self, "_band_edges", None) if edges is False else edges
        nb = 0 if edges is None else edges.size - 1
        img = np.empty((rows, nb, abi.IMAGE_BINS, abi.IMAGE_BINS))
        img2 = np.empty_like(img)
        n = np.empty((rows, nb), dtype=np.uint64)
        return (img, img2, n), lambda: [BandImages(edges.copy(), img[k], img2[k], n[k]) for k in range(rows)]

    def _read_bands(self, read) -> BandImages:
        arrays, split = self._band_rows(1)
        check(read(self._h, *map(_ptr, arrays)))
        return split()[0]

    def read_band_images(self) -> BandImages:
        """The band images accumulated since enable_band_images / reset_image (raises SartError while they are off)."""
        return self._read_bands(lib.sart_read_band_images)

    def read_merged_band_images(self) -> BandImages:
        """read_band_images of the last allreduce_outputs (raises SartError without one)."""
        return self._read_bands(lib.sart_read_merged_band_images)

    def enable_mass_band_images(self, edges_keV=None):
        """Band images (as enable_band_images) of the rays that pass in trace_mc for every axion mass of set_axion_masses
        (sart_enable_mass_band_images), from the one traced ray per mass scan; None switches them off. Switching them on
        clears them; trace_mc then runs the mass-scan kernels for any number of masses. Not together with
        enable_band_images or the alias sampler. Device memory: about 3 x 64 MiB per band."""
        if edges_keV is None:
            check(lib.sart_enable_mass_band_images(self._h, 0, None))
            self._mass_band_edges = None
            return
        e = np.ascontiguousarray(edges_keV, dtype=np.float64)
        check(lib.sart_enable_mass_band_images(self._h, e.size - 1 if e.size > 1 else -1, _dp(e)))   # one edge: refused
        self._mass_band_edges = e.copy()

    def _read_mass_bands(self, read) -> list[BandImages]:
        arrays, split = self._band_rows(self.n_masses, getattr(self, "_mass_band_edges", None))
        check(read(self._h, *map(_ptr, arrays)))
        return split()

    def read_mass_band_images(self) -> list[BandImages]:
        """One BandImages per axion mass, in the order of set_axion_masses, accumulated since enable_mass_band_images /
        reset_image (raises SartError while they are off)."""
        return self._read_mass_bands(lib.sart_read_mass_band_images)

    def read_merged_mass_band_images(self) -> list[BandImages]:
        """read_mass_band_images of the last allreduce_outputs (raises SartError without one)."""
        return self._read_mass_bands(lib.sart_read_merged_mass_band_images)

    def enable_quantity_hists(self, specs=None):
        """Weighted histograms of per-ray record quantities of the rays that pass in trace_mc (single axion mass;
        sart_enable_quantity_hists): specs [(name, nbins, lo, hi), ...], names from abi.QUANTITIES (the fields of
        sart_ray_out_t); None or [] switches them off. Switching them on clears them."""
        specs = check_quantity_hist_specs(specs or [])
        arr = (abi.QuantityHistSpec * max(len(specs), 1))()
        for k, (name, nbins, lo, hi) in enumerate(specs):
            arr[k] = abi.QuantityHistSpec(abi.QUANTITIES.index(name), nbins, lo, hi)
        check(lib.sart_enable_quantity_hists(self._h, len(specs), arr if specs else None))
        self._qhist_specs = specs or None

    def _qhist_rows(self, rows: int):
        specs = getattr(self, "_qhist_specs", None) or []
        n = sum(nb + 2 for _, nb, _, _ in specs)
        w, w2 = np.empty((rows, n)), np.empty((rows, n))
        c = np.empty((rows, n), dtype=np.uint64)

        def split():
            out = []
            for k in range(rows):
                row, off = [], 0
                for name, nb, lo, hi in specs:
                    sl = slice(off, off + nb + 2)
                    row.append(QuantityHist(name, quantity_hist_edges(nb, lo, hi), w[k, sl].copy(), w2[k, sl].copy(),
                                            c[k, sl].copy()))
                    off += nb + 2
                out.append(row)
            return out
        return (w, w2, c), split

    def _read_qhists(self, read) -> list[QuantityHist]:
        arrays, split = self._qhist_rows(1)
        check(read(self._h, *map(_ptr, arrays)))
        return split()[0]

    def read_quantity_hists(self) -> list[QuantityHist]:
        """The quantity histograms accumulated since enable_quantity_hists / reset_image, one output.QuantityHist per spec
        (raises SartError while they are off)."""
        return self._read_qhists(lib.sart_read_quantity_hists)

    def read_merged_quantity_hists(self) -> list[QuantityHist]:
        """read_quantity_hists of the last allreduce_outputs (raises SartError without one)."""
        return self._read_qhists(lib.sart_read_merged_quantity_hists)

    def synchronize(self):
        check(lib.sart_synchronize(self._h))

    def image_dev(self) -> tuple[int, int, int]:
        """(device pointer of the image, of the w^2 image, number of doubles each) for collectives."""
        return lib.sart_image_dev(self._h), lib.sart_image_w2_dev(self._h), lib.sart_image_len(self._h)

    def counters_dev(self) -> int:
        return lib.sart_counters_dev(self._h)

    def angular_scan(self, angles_deg, n_rays_per_angle: int, seed: int = 299792458, want_images: bool = False,
                     first_ray: int = 0):
        """sart_angular_scan: (fluxes [n], counters [n dicts], images [n, 256, 256] or None)."""
        a = np.ascontiguousarray(angles_deg, dtype=np.float64)
        fl = np.empty(a.size)
        cnt = (abi.Counters * a.size)()
        img = np.empty((a.size, abi.IMAGE_BINS, abi.IMAGE_BINS)) if want_images else None
        check(lib.sart_angular_scan(self._h, a.size, _dp(a), first_ray, n_rays_per_angle, seed, _dp(fl), cnt,
                                    _dp(img) if want_images else None))
        return fl, [c.as_dict() for c in cnt], img

    def angular_scan_outputs(self, angles_deg, n_rays_per_angle: int, seed: int = 299792458, want_images: bool = False,
                             first_ray: int = 0) -> ScanOutputs:
        """sart_angular_scan_outputs: angular_scan, plus for every scan point a row of each accumulator this tracer has on
        (enable_radial_hist, enable_spectra, enable_band_images, enable_quantity_hists): what a fused run of that point's
        rays would add to a freshly reset tracer. The tracer's own accumulators, image and counters stay as they are.
        Raises SartError when none of the four is on."""
        a = np.ascontiguousarray(angles_deg, dtype=np.float64)
        n = a.size
        fl = np.empty(n)
        cnt = (abi.Counters * n)()
        img = np.empty((n, abi.IMAGE_BINS, abi.IMAGE_BINS)) if want_images else None
        on = {"radial": getattr(self, "_rad", (0, 0.0))[0] > 0, "spectra": getattr(self, "_spectra_on", False),
              "bands": getattr(self, "_band_edges", None) is not None, "qhists": bool(getattr(self, "_qhist_specs", None))}
        rows = {"radial": self._radial_rows, "spectra": self._spectra_rows, "bands": self._band_rows,
                "qhists": self._qhist_rows}
        out = abi.ScanOut()
        split = {}
        for kind, fields in abi.SCAN_OUT_FIELDS.items():
            if on[kind]:
                arrays, split[kind] = rows[kind](n)
                for (name, _), arr in zip(fields, arrays):
                    setattr(out, name, _ptr(arr))
        check(lib.sart_angular_scan_outputs(self._h, n, _dp(a), first_ray, n_rays_per_angle, seed, _dp(fl), cnt,
                                            _dp(img) if want_images else None, C.byref(out)))
        got = {kind: f() for kind, f in split.items()}
        return ScanOutputs(a.copy(), fl, [c.as_dict() for c in cnt], img, got.get("radial"), got.get("spectra"),
                           got.get("bands"), got.get("qhists"))

    # -- multi-GPU (sart_allreduce): one NCCL all-reduce of image | w^2 image | counters into a separate merged buffer
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(abi.COMM_ID_BYTES)
        check(lib.sart_comm_unique_id(buf))
        return buf.raw

    def comm_init_rank(self, n_ranks: int, rank: int, unique_id: bytes):
        if len(unique_id) != abi.COMM_ID_BYTES:
            raise ValueError("unique_id must be the 128 bytes of comm_unique_id()")
        check(lib.sart_comm_init_rank(self._h, n_ranks, rank, C.create_string_buffer(unique_id, abi.COMM_ID_BYTES)))

    def allreduce(self):
        """Asynchronous on `stream`; the tracer's own image keeps accumulating, the sum over ranks is read_merged()."""
        hs = (abi.H * 1)(self._h)
        check(lib.sart_allreduce(hs, 1))

    def allreduce_outputs(self):
        """sart_allreduce_outputs for this rank (every rank calls it): sums the radial histogram, the (per-mass) spectra, the
        band images and the quantity histograms that are on over all ranks into merged copies, read with the read_merged_*
        methods. Synchronises."""
        hs = (abi.H * 1)(self._h)
        check(lib.sart_allreduce_outputs(hs, 1))

    def read_merged_radial_hist(self):
        """read_radial_hist of the last allreduce_outputs (raises SartError without one)."""
        return self._read_radial(lib.sart_read_merged_radial_hist)

    def read_merged_spectra(self) -> Spectra:
        """read_spectra of the last allreduce_outputs (raises SartError without one)."""
        return self._read_spectra_rows(lib.sart_read_merged_spectra, 1)[0]

    def read_merged_mass_spectra(self) -> list[Spectra]:
        """read_mass_spectra of the last allreduce_outputs (raises SartError without one)."""
        return self._read_spectra_rows(lib.sart_read_merged_mass_spectra, self.n_masses)

    def read_merged(self, want_w2: bool = True) -> RunResult:
        m = self.n_masses
        img = np.empty((m, abi.IMAGE_BINS, abi.IMAGE_BINS))
        img2 = np.empty_like(img) if want_w2 else None
        cnt = (abi.Counters * m)()
        check(lib.sart_read_merged(self._h, _dp(img), _dp(img2) if want_w2 else None, cnt))
        return RunResult(img, img2, [c.as_dict() for c in cnt])

    def read_image(self, want_w2: bool = True) -> RunResult:
        m = self.n_masses
        img = np.empty((m, abi.IMAGE_BINS, abi.IMAGE_BINS))
        img2 = np.empty_like(img) if want_w2 else None
        cnt = (abi.Counters * m)()
        check(lib.sart_read_image(self._h, _dp(img), _dp(img2) if want_w2 else None, cnt))
        return RunResult(img, img2, [c.as_dict() for c in cnt])


PRECISION_NAMES = ("exact", "fast", "f32")


def set_fastest_precision(tracer: RayTracer, want: int, warn=None) -> int:
    """Sets precision mode `want`, else the fastest slower one this setup supports (f32 -> fast -> exact); returns the
    mode set. `warn` receives a message for every mode the setup refuses."""
    for mode in range(want, 0, -1):
        try:
            tracer.set_precision(mode)
            return mode
        except SartError as e:
            if warn:
                warn(f"precision {PRECISION_NAMES[mode]} is not available for this setup ({e}); falling back")
    tracer.set_precision(0)
    return 0


def initFullSetup(setup, detectorSetup, stage, telescope, flags: int = 0, tables: _tables.TableSet | None = None,
                  emission: _tables.EmissionTable | None = None, reflectivity=None, device: int = 0,
                  outpath: str = "out") -> FullRaytraceSetup:
    """initFullSetup (rt:2637-2753). `tables` wins if given; otherwise the CDFs are built on the GPU from
    `emission` (default: the synthetic full-size table) and the packaged detector-chain tables are used."""
    exp = newExperimentSetup(setup, detectorSetup, stage, telescope, flags)
    if tables is None:
        if emission is None:
            emission = _tables.synthetic_emission()
        rc, dc = buildCdfs(emission, device)
        if reflectivity is None:
            reflectivity = _tables.synthetic_reflectivity(max(1, exp.telescope.nCoatings))
        tables = _tables.TableSet(energies=emission.energies, fluxRadiusCDF=rc, diffFluxCDFs=dc,
                                  reflectivity=reflectivity, **_tables.detector_tables_packaged())
    return FullRaytraceSetup(expSetup=exp, tables=tables, outpath=outpath)


def calculateFluxFractions(raytraceSetup: FullRaytraceSetup, nRays: int = 1_000_000, seed: int = 299792458,
                           device: int = 0, tracer: RayTracer | None = None) -> RunResult:
    """calculateFluxFractions (rt:2755-2776): trace `nRays` axions (NumberOfPointsSun = 1_000_000 in the
    reference, rt:251) and return the detector image + counters."""
    own = tracer is None
    t = tracer or RayTracer(raytraceSetup, device)
    try:
        t.reset_image()
        t.trace_mc(nRays, seed)
        return t.read_image()
    finally:
        if own:
            t.close()


def prepareHeatmap(tracer: RayTracer, numberOfRows, numberOfColumns, start_x, stop_x, start_y, stop_y, data_X, data_Y,
                   weight1, norm):
    """prepareHeatmap (rt:818-842) for per-ray records held by the host; histogrammed on the GPU
    (sart_prepare_heatmap). Returns (heatmap [rows, cols], number of points outside the grid)."""
    X = np.ascontiguousarray(data_X, dtype=np.float64)
    Y = np.ascontiguousarray(data_Y, dtype=np.float64)
    W = np.ascontiguousarray(weight1, dtype=np.float64)
    out = np.empty((numberOfRows, numberOfColumns))
    bad = C.c_uint64(0)
    check(lib.sart_prepare_heatmap(tracer._h, numberOfRows, numberOfColumns, start_x, stop_x, start_y, stop_y, X.size,
                                   _dp(X), _dp(Y), _dp(W), norm, _dp(out), C.byref(bad)))
    return out, bad.value


def performAngularScan(fullSetup: FullRaytraceSetup, angularScanMin: float, angularScanMax: float,
                       numAngularScanPoints: int = 50, nRays: int = 1_000_000, seed: int = 299792458, device: int = 0,
                       tracer: RayTracer | None = None, rank: int = 0, world: int = 1, group=None):
    """performAngularScan (rt:2778-2815): relative flux versus telescope_turned_y. Returns (angles [deg],
    relative flux = flux / max flux, absolute fluxes). With world > 1 the scan points are dealt to the
    ranks in contiguous blocks (no exchange while tracing) and the per-point fluxes are summed over `group` at the end."""
    from .multi_gpu import shard
    angles = np.linspace(angularScanMin, angularScanMax, numAngularScanPoints)
    lo, cnt = shard(numAngularScanPoints, rank, world)   # a contiguous block of scan points per rank
    fluxes = np.zeros(numAngularScanPoints)
    if cnt:
        own = tracer is None
        t = tracer or RayTracer(fullSetup, device)
        try:
            # scan point i always traces the global rays [i*nRays, (i+1)*nRays), whichever rank owns it
            fluxes[lo:lo + cnt], _, _ = t.angular_scan(angles[lo:lo + cnt], nRays, seed, first_ray=lo * nRays)
        finally:
            if own:
                t.close()
    if world > 1:
        import torch
        import torch.distributed as dist
        tf = torch.from_numpy(fluxes)
        dist.all_reduce(tf, op=dist.ReduceOp.SUM, group=group)
        fluxes = tf.numpy()
    return angles, fluxes / fluxes.max(), fluxes
