"""Command line of the ray tracer: the switches of the reference's `main` (src/raytracer.nim:2817-2865, cligen
`dispatch main`) driving the GPU path.

  python -m solaraxionraytracing_b200 [--ignoreDetWindow] [--ignoreGasAbs] [--ignoreConvProb] [--ignoreReflection]
      [--xrayTest] [--detectorInstall] [--magnet] [--angularScanMin A --angularScanMax B --numAngularScanPoints N]
      [--noPlots] [--config FILE | --configPath DIR] [--nRays N] [--precision f32|fast|exact] [--writeSpectra]
      [--energyBands E0,E1,...] [--histogram NAME:NBINS:LO:HI ...] [--massScanRadii] [--massScanBands E0,E1,...]
      [--device D | --devices 0,1,... | --devices all]

Inputs the reference reads from `resources/` and that are not shipped with it (solar_model_dataframe.csv, the two
reflectivity HDF5 files) are taken from [Resources] when present, else generated: Primakoff emission rates from AGSS09
on the GPU and the packaged Henke gold reflectivity (XMM) / the synthetic multilayer tables (LLNL).
"""
from __future__ import annotations

import argparse
import sys
from pathlib import Path

import numpy as np


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(prog="raytracer", description=__doc__.split("\n\n")[0])
    for flag in ("ignoreDetWindow", "ignoreGasAbs", "ignoreConvProb", "ignoreReflection", "xrayTest", "detectorInstall",
                 "magnet", "noPlots"):
        ap.add_argument(f"--{flag}", action="store_true")
    ap.add_argument("--angularScanMin", type=float, default=0.0)
    ap.add_argument("--angularScanMax", type=float, default=0.0)
    ap.add_argument("--numAngularScanPoints", type=int, default=50)
    ap.add_argument("--config", default="", help="path to a config.toml")
    ap.add_argument("--configPath", default="", help="directory holding config.toml")
    ap.add_argument("--nRays", type=float, default=None, help="NumberOfPointsSun (rt:251); default [Run].nRays or 1e6")
    ap.add_argument("--seed", type=int, default=None, help="default [Run].seed or 299792458 (rt:276)")
    ap.add_argument("--precision", choices=["f32", "fast", "exact"], default=None)
    ap.add_argument("--sampler", choices=["inverse_cdf", "alias"], default=None,
                    help="alias: emission shell / energy from alias tables of the same distributions (f32, single mass)")
    ap.add_argument("--writeSpectra", action="store_true",
                    help="also write the energy spectrum and the per-shell flux of the detected rays as CSV files next to "
                         "the image (a single-mass run then takes the generic kernel variant; a mass scan writes one pair "
                         "of files per mass, suffixed _ma{m}eV, an angular scan one pair per scan point, suffixed "
                         "_angle{a}deg)")
    ap.add_argument("--energyBands", default=None,
                    help="also write one detector image per energy band: comma-separated band edges in keV, e.g. 0.5,2,4,8 "
                         "(2 to 17 values, ascending) writes axion_image_{year}_E0.5-2keV.csv and so on next to the image "
                         "(an angular scan: one set per scan point, suffixed _angle{a}deg); a single axion mass only (a mass "
                         "scan: --massScanBands)")
    ap.add_argument("--histogram", action="append", default=None, metavar="NAME:NBINS:LO:HI",
                    help="also write a weighted histogram of a per-ray record quantity of the passed rays, e.g. "
                         "transMagnet:256:0:1e-20, to axion_hist_{NAME}_{year}.csv next to the image (NBINS regular bins over "
                         "[LO, HI) plus an underflow and an overflow row); repeatable, each quantity once; NAME is one of "
                         "reflect, transMagnet, yaw, alpha1, alpha2, pathCB, deviationDet, transProbArgon; an angular scan "
                         "writes one file per scan point, suffixed _angle{a}deg; a single axion mass only. With an angular "
                         "scan, each of these three switches also writes the containment radii of every scan point to "
                         "angular_scan_telescope_y_radii.csv")
    ap.add_argument("--massScanRadii", action="store_true",
                    help="a mass scan (several axion masses) also writes the 68 %% / 95.5 %% containment radii of every mass "
                         "to mass_scan_radii.csv, from one traced ray per mass scan (a single axion mass: the radii are in "
                         "the image CSV; see also --energyBands)")
    ap.add_argument("--massScanBands", default=None, metavar="E0,E1,...",
                    help="a mass scan also writes one detector image per energy band and mass, "
                         "axion_image_{year}_E{lo}-{hi}keV_ma{m}eV.csv, with that mass's containment radii in the radius "
                         "columns, and mass_scan_radii.csv as --massScanRadii; band edges as --energyBands (a single axion "
                         "mass: --energyBands)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--devices", default=None,
                    help="trace on several GPUs: a comma-separated list of CUDA ordinals or `all`. A fused run shards the "
                         "rays over them and merges image, counters, radial histogram and spectra with NCCL; an angular "
                         "scan deals each a contiguous block of scan points. The output files are those of one GPU")
    ap.add_argument("--outputPath", default="", help="overrides [Resources].outputPath")
    ap.add_argument("--allowSynthetic", action="store_true",
                    help="continue with stand-in tables (and a warning) when a [Resources] input file is missing; the "
                         "reference stops in that case")
    return ap


def parse_devices(text: str, n_visible: int) -> list[int]:
    """The value of --devices: `all` (every visible device) or distinct, comma-separated ordinals below `n_visible`."""
    if text.strip() == "all":
        if n_visible < 1:
            raise ValueError("no CUDA device is visible")
        return list(range(n_visible))
    try:
        devices = [int(x) for x in text.split(",")]
    except ValueError:
        raise ValueError(f"expected `all` or comma-separated device ordinals, got {text!r}") from None
    for k, d in enumerate(devices):
        if d in devices[:k]:
            raise ValueError(f"device {d} is listed twice")
        if not 0 <= d < n_visible:
            raise ValueError(f"device {d} does not exist ({n_visible} visible)")
    return devices


def visible_devices() -> int:
    from ._lib import lib
    return lib.sart_device_count()


def parse_args(argv=None) -> argparse.Namespace:
    ap = build_parser()
    a = ap.parse_args(argv)
    if a.devices is not None:
        if a.device != 0:
            ap.error("--devices and --device exclude each other")
        try:
            a.devices = parse_devices(a.devices, visible_devices())
        except ValueError as e:
            ap.error(f"--devices: {e}")
    if a.energyBands is not None:
        from .output import parse_energy_bands
        try:
            a.energyBands = parse_energy_bands(a.energyBands)
        except ValueError as e:
            ap.error(f"--energyBands: {e}")
    if a.massScanBands is not None:
        from .output import parse_energy_bands
        try:
            a.massScanBands = parse_energy_bands(a.massScanBands)
        except ValueError as e:
            ap.error(f"--massScanBands: {e}")
    if a.histogram is not None:
        from .output import check_quantity_hist_specs, parse_quantity_hist
        try:
            a.histogram = check_quantity_hist_specs([parse_quantity_hist(t) for t in a.histogram])
        except ValueError as e:
            ap.error(f"--histogram: {e}")
    return a


def _substitute(what: str, missing, used: str, allow: bool):
    """The reference fails hard when a [Resources] file is missing (rt:2647, 1174, 1498). A stand-in changes the physics
    of the result, so it is used only with --allowSynthetic, and never silently."""
    msg = f"{what}: {missing} not found"
    if not allow:
        raise SystemExit(f"raytracer: {msg}. The reference stops here; pass --allowSynthetic to continue with {used}.")
    print(f"WARNING: {msg}; using {used}. The image and flux below do NOT come from the reference's input data.",
          file=sys.stderr)


def load_tables(rt, tables, res, setup, device: int, allow_synthetic: bool = False):
    """initFullSetup's inputs (rt:2645-2705, 1160-1249, 1498-1527): files under [Resources] when they exist."""
    from . import abi
    base = Path(res.resourcePath)
    csv = base / res.solarModelFile
    if res.solarModelFile and csv.is_file():
        em = tables.read_solar_model_dataframe(csv)
    else:
        raw = base / res.rawSolarModel
        have_raw = bool(res.rawSolarModel) and raw.is_file()
        _substitute("solar model", csv, "Primakoff-only emission rates computed on the GPU from "
                    + (str(raw) if have_raw else "the packaged AGSS09 model"), allow_synthetic)
        sm = tables.read_solar_model(raw) if have_raw else None
        em = rt.calculateEmissionRates(sm, ("primakoff",), device=device)
    rc, dc = rt.buildCdfs(em, device)
    llnl = setup.telescope.kind == abi.TK_LLNL
    extra = {}
    refl = None
    if setup.telescope.reflKind == abi.RK_EFFECTIVE_AREA:
        # rkEffectiveArea (rt:1245-1249): the telescope transmission comes from llnlEfficiency, no reflectivity table
        eff = base / (res.llnlEfficiency or "llnl_xray_telescope_cast_effective_area.csv")
        if not eff.is_file():
            raise SystemExit(f"raytracer: rkEffectiveArea needs the effective-area table {eff}")
        header = eff.read_text().splitlines()[0].split(",")
        if "Energy[keV]" not in header or "Transmission" not in header:
            # the shipped csv has Energy[keV], EffectiveArea[cm^2] only; the reference reads df["Transmission"] (rt:1247-1248)
            # and fails on it as well (the conversion from the effective area is `when false`, rt:1238-1244)
            raise SystemExit(f"raytracer: {eff} has no 'Transmission' column (columns: {header}); the reference needs it too")
        data = np.loadtxt(eff, delimiter=",", skiprows=1)
        extra["telescopeTransmission"] = (data[:, header.index("Energy[keV]")], data[:, header.index("Transmission")])
    else:
        h5 = base / (res.llnlReflFile if llnl else res.goldReflFile)
        if h5.is_file():
            refl, extra["angleLim"], extra["reflEnergyLim"] = tables.reflectivity_from_h5(h5, setup.telescope.nCoatings if llnl else None)
        elif llnl:
            _substitute("LLNL multilayer reflectivity", h5, "SYNTHETIC multilayer tables (made-up coatings)", allow_synthetic)
            refl = tables.synthetic_reflectivity(max(1, setup.telescope.nCoatings))
        else:
            _substitute("gold reflectivity", h5, "the packaged Henke gold data (resources/reflectivity.zip, coarser grid)", allow_synthetic)
            refl = tables.gold_reflectivity_packaged()
    try:
        det = tables.detector_tables_from_resources(base, setup.detector.windowThickness, setup.detector.alThickness)
    except OSError as e:
        _substitute("detector transmission tables", e.filename or base, "the packaged copies of the reference's own .tsv files", True)
        det = tables.detector_tables_packaged()
    return tables.TableSet(energies=em.energies, fluxRadiusCDF=rc, diffFluxCDFs=dc, reflectivity=refl, **extra, **det)


def write_fused_outputs(result, radial_hist, spectra, masses, setup, outpath, bands=None, qhists=None, mass_radial=None,
                        mass_bands=None):
    """The files of a fused run: the image CSV and containment radii (at most one mass), or the per-mass images of a mass
    scan; with `spectra` also the spectra CSVs (one Spectra, or one per mass); with `bands` (output.BandImages, at most one
    mass) one image CSV per energy band; with `qhists` (output.QuantityHist list, at most one mass) one CSV per histogram;
    with `mass_radial` (a mass scan: one radial histogram per mass) mass_scan_radii.csv, and with `mass_bands` (one
    output.BandImages per mass) one image CSV per band and mass (output.write_mass_scan_outputs)."""
    from . import output
    if len(masses) <= 1:
        radii = output.containment_radii_from_hist(*radial_hist)
        path = output.generateResultPlots(result, setup.detector.windowYear, outpath, radii=radii,
                                          chipXMax=setup.consts.chipXMax, chipYMax=setup.consts.chipYMax)
        print("wrote", path)
        if bands is not None:
            for p in output.write_band_image_csvs(bands, setup.detector.windowYear, outpath, radii,
                                                  setup.consts.chipXMax, setup.consts.chipYMax):
                print("wrote", p)
        if qhists is not None:
            for p in output.write_quantity_hist_csvs(qhists, setup.detector.windowYear, outpath):
                print("wrote", p)
        if spectra is not None:
            for p in output.write_spectra_csvs(spectra, setup.detector.windowYear, outpath):
                print("wrote", p)
    else:   # mass scan: one image per mass, total flux per mass on stdout
        Path(outpath).mkdir(parents=True, exist_ok=True)
        for m, c in zip(masses, result.counters):
            print(f"m_a = {m:.6g} eV: passed {c['n_passed']}, total flux {c['sum_w']:.6e}")
        np.save(Path(outpath) / "axion_images_mass_scan.npy", result.image)
        if spectra is not None:
            for p in output.write_mass_spectra_csvs(spectra, masses, setup.detector.windowYear, outpath):
                print("wrote", p)
        if mass_radial is not None:
            for p in output.write_mass_scan_outputs(masses, mass_radial, mass_bands, setup.detector.windowYear, outpath,
                                                    setup.consts.chipXMax, setup.consts.chipYMax):
                print("wrote", p)


def write_angular_scan(angles, rel, outpath):
    print("Angle [deg], relative flux")
    for ang, r in zip(angles, rel):
        print(f"{ang:.4f}, {r:.6f}")
    Path(outpath).mkdir(parents=True, exist_ok=True)
    np.savetxt(Path(outpath) / "angular_scan_telescope_y.csv", np.column_stack([angles, rel]), delimiter=",",
               header="Angle [deg],relative flux", comments="")


def write_angular_scan_outputs(scan, setup, outpath):
    """The files of an angular scan with accumulators (output.ScanOutputs): those of write_angular_scan, the containment
    radii of every scan point and its spectra, band images and quantity histograms (output.write_scan_outputs)."""
    from . import output
    write_angular_scan(scan.angles, scan.fluxes / scan.fluxes.max(), outpath)
    for p in output.write_scan_outputs(scan, setup.detector.windowYear, outpath, setup.consts.chipXMax, setup.consts.chipYMax):
        print("wrote", p)


def main(argv=None) -> int:
    a = parse_args(argv)
    from . import abi, config as cfgmod, multi_gpu, raytracer as rt, tables
    cfg_file = a.config or (str(Path(a.configPath) / "config.toml") if a.configPath else None)
    flags = rt.flags_from_cli(a.ignoreDetWindow, a.ignoreGasAbs, a.ignoreConvProb, a.ignoreReflection, a.xrayTest,
                              a.magnet, a.detectorInstall)
    print("Flags:", {n for n, on in vars(a).items() if on is True and n != "noPlots"})
    setup, res = cfgmod.setup_from_config(cfg_file, flags)
    run = cfgmod.parseRun(cfgmod.load_config(cfg_file))
    if a.energyBands is not None and len(run.mAxion) > 1:
        build_parser().error("--energyBands: the band images need a single axion mass, and the configuration sets a mass scan "
                             "(use --massScanBands)")
    mass_outputs = a.massScanRadii or a.massScanBands is not None
    if mass_outputs and (len(run.mAxion) <= 1 or a.angularScanMin != a.angularScanMax):
        which = "--massScanBands" if a.massScanBands is not None else "--massScanRadii"
        build_parser().error(f"{which}: needs a mass scan (several axion masses in [Run] mAxion) without an angular scan; a "
                             "single axion mass writes its radii with the image and its band images with --energyBands")
    if a.histogram is not None and len(run.mAxion) > 1:
        build_parser().error("--histogram: the quantity histograms need a single axion mass, and the configuration sets a mass scan")
    a.nRays = run.nRays if a.nRays is None else a.nRays
    a.seed = run.seed if a.seed is None else a.seed
    a.precision = a.precision or run.precision
    outpath = a.outputPath or res.outputPath
    devices = a.devices or [a.device]
    tb = load_tables(rt, tables, res, setup, devices[0], a.allowSynthetic)
    fs = rt.FullRaytraceSetup(setup, tb, outpath)
    n = int(a.nRays)
    want = {"exact": 0, "fast": 1, "f32": 2}[a.precision]
    sampler = abi.SAMPLER_ALIAS if (a.sampler or run.sampler) == "alias" else None
    warn = lambda msg: print(msg, file=sys.stderr)   # noqa: E731
    single = len(run.mAxion) <= 1
    fused = a.angularScanMin == a.angularScanMax
    # an angular scan of one axion mass writes the files of these switches once per scan point, with its containment radii
    scan_outputs = single and (a.writeSpectra or a.energyBands is not None or a.histogram is not None)
    if a.devices is not None:
        if fused:
            print("start")
            try:
                r = multi_gpu.trace_on_devices(fs, devices, n, a.seed, precision=want, sampler=sampler,
                                               masses=run.mAxion or None, radial_hist=single, spectra=a.writeSpectra,
                                               bands=a.energyBands, quantity_hists=a.histogram,
                                               mass_radial_hist=mass_outputs, mass_bands=a.massScanBands, warn=warn)
            except rt.SartError as e:
                if "NCCL" in str(e):
                    raise SystemExit(f"raytracer: {e}") from None
                raise
            write_fused_outputs(r.result, r.radial_hist, r.spectra, run.mAxion, setup, outpath, r.band_images, r.quantity_hists,
                                r.mass_radial_hists, r.mass_band_images)
        elif scan_outputs:
            scan = multi_gpu.angular_scan_outputs_on_devices(fs, devices, a.angularScanMin, a.angularScanMax,
                                                             a.numAngularScanPoints, n, a.seed, precision=want,
                                                             sampler=sampler, masses=run.mAxion or None, radial_hist=True,
                                                             spectra=a.writeSpectra, bands=a.energyBands,
                                                             quantity_hists=a.histogram, warn=warn)
            write_angular_scan_outputs(scan, setup, outpath)
        else:
            angles, rel, _ = multi_gpu.angular_scan_on_devices(fs, devices, a.angularScanMin, a.angularScanMax,
                                                               a.numAngularScanPoints, n, a.seed, precision=want,
                                                               sampler=sampler, masses=run.mAxion or None, warn=warn)
            write_angular_scan(angles, rel, outpath)
        return 0
    with rt.RayTracer(fs, a.device) as tr:
        rt.set_fastest_precision(tr, want, warn)
        if sampler is not None:
            tr.set_sampler(sampler)
        if run.mAxion:
            tr.set_axion_masses(run.mAxion)
        if fused:
            print("start")
            if single:
                tr.enable_radial_hist()
            if a.writeSpectra:   # a mass scan: one pair of spectra files per mass
                tr.enable_spectra() if single else tr.enable_mass_spectra()
            if a.energyBands is not None:
                tr.enable_band_images(a.energyBands)
            if a.histogram is not None:
                tr.enable_quantity_hists(a.histogram)
            if mass_outputs:
                tr.enable_mass_radial_hist()
            if a.massScanBands is not None:
                tr.enable_mass_band_images(a.massScanBands)
            tr.reset_image()
            tr.trace_mc(n, a.seed)
            result = tr.read_image()
            spectra = None
            if a.writeSpectra:
                spectra = tr.read_spectra() if single else tr.read_mass_spectra()
            bands = tr.read_band_images() if a.energyBands is not None else None
            qhists = tr.read_quantity_hists() if a.histogram is not None else None
            write_fused_outputs(result, tr.read_radial_hist() if single else None, spectra, run.mAxion, setup, outpath, bands,
                                qhists, tr.read_mass_radial_hist() if mass_outputs else None,
                                tr.read_mass_band_images() if a.massScanBands is not None else None)
        elif scan_outputs:
            tr.enable_radial_hist()
            if a.writeSpectra:
                tr.enable_spectra()
            if a.energyBands is not None:
                tr.enable_band_images(a.energyBands)
            if a.histogram is not None:
                tr.enable_quantity_hists(a.histogram)
            angles = np.linspace(a.angularScanMin, a.angularScanMax, a.numAngularScanPoints)
            write_angular_scan_outputs(tr.angular_scan_outputs(angles, n, a.seed), setup, outpath)
        else:
            angles, rel, _ = rt.performAngularScan(fs, a.angularScanMin, a.angularScanMax, a.numAngularScanPoints, n,
                                                   a.seed, tracer=tr)
            write_angular_scan(angles, rel, outpath)
    return 0


if __name__ == "__main__":
    sys.exit(main())
