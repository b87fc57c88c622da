"""Command line of the ray tracer: the switches of the reference's `main` (src/raytracer.nim:2817-2865, cligen
`dispatch main`) driving the GPU path.

  python -m solaraxionraytracing_b200 [--ignoreDetWindow] [--ignoreGasAbs] [--ignoreConvProb] [--ignoreReflection]
      [--xrayTest] [--detectorInstall] [--magnet] [--angularScanMin A --angularScanMax B --numAngularScanPoints N]
      [--noPlots] [--config FILE | --configPath DIR] [--nRays N] [--precision f32|fast|exact] [--writeSpectra]
      [--device D]

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
                         "the image (single-mass runs; the run then takes the generic kernel variant)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--outputPath", default="", help="overrides [Resources].outputPath")
    ap.add_argument("--allowSynthetic", action="store_true",
                    help="continue with stand-in tables (and a warning) when a [Resources] input file is missing; the "
                         "reference stops in that case")
    return ap


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


def main(argv=None) -> int:
    a = build_parser().parse_args(argv)
    from . import abi, config as cfgmod, output, raytracer as rt, tables
    cfg_file = a.config or (str(Path(a.configPath) / "config.toml") if a.configPath else None)
    flags = rt.flags_from_cli(a.ignoreDetWindow, a.ignoreGasAbs, a.ignoreConvProb, a.ignoreReflection, a.xrayTest,
                              a.magnet, a.detectorInstall)
    print("Flags:", {n for n, on in vars(a).items() if on is True and n != "noPlots"})
    setup, res = cfgmod.setup_from_config(cfg_file, flags)
    run = cfgmod.parseRun(cfgmod.load_config(cfg_file))
    a.nRays = run.nRays if a.nRays is None else a.nRays
    a.seed = run.seed if a.seed is None else a.seed
    a.precision = a.precision or run.precision
    outpath = a.outputPath or res.outputPath
    tb = load_tables(rt, tables, res, setup, a.device, a.allowSynthetic)
    fs = rt.FullRaytraceSetup(setup, tb, outpath)
    n = int(a.nRays)
    with rt.RayTracer(fs, a.device) as tr:
        want = {"exact": 0, "fast": 1, "f32": 2}[a.precision]
        for mode in range(want, -1, -1):     # f32 -> fast -> exact: the fastest pipeline that supports this setup
            try:
                tr.set_precision(mode)
                break
            except rt.SartError as e:
                print(f"precision {['exact', 'fast', 'f32'][mode]} is not available for this setup ({e}); falling back",
                      file=sys.stderr)
        if (a.sampler or run.sampler) == "alias":
            tr.set_sampler(abi.SAMPLER_ALIAS)
        if run.mAxion:
            tr.set_axion_masses(run.mAxion)
        if a.angularScanMin == a.angularScanMax:
            print("start")
            spectra = a.writeSpectra and len(run.mAxion) <= 1
            if a.writeSpectra and not spectra:
                print("--writeSpectra: spectra are written for single-mass runs only", file=sys.stderr)
            if len(run.mAxion) <= 1:
                tr.enable_radial_hist()
            if spectra:
                tr.enable_spectra()
            tr.reset_image()
            tr.trace_mc(n, a.seed)
            result = tr.read_image()
            if len(run.mAxion) <= 1:
                radii = output.containment_radii_from_hist(*tr.read_radial_hist())
                path = output.generateResultPlots(result, setup.detector.windowYear, outpath, radii=radii,
                                                  chipXMax=setup.consts.chipXMax, chipYMax=setup.consts.chipYMax)
                print("wrote", path)
                if spectra:
                    for p in output.write_spectra_csvs(tr.read_spectra(), setup.detector.windowYear, outpath):
                        print("wrote", p)
            else:   # mass scan: one image per mass, total flux per mass on stdout
                Path(outpath).mkdir(parents=True, exist_ok=True)
                for m, c in zip(run.mAxion, result.counters):
                    print(f"m_a = {m:.6g} eV: passed {c['n_passed']}, total flux {c['sum_w']:.6e}")
                np.save(Path(outpath) / "axion_images_mass_scan.npy", result.image)
        else:
            angles, rel, _ = rt.performAngularScan(fs, a.angularScanMin, a.angularScanMax, a.numAngularScanPoints, n,
                                                   a.seed, tracer=tr)
            print("Angle [deg], relative flux")
            for ang, r in zip(angles, rel):
                print(f"{ang:.4f}, {r:.6f}")
            Path(outpath).mkdir(parents=True, exist_ok=True)
            np.savetxt(Path(outpath) / "angular_scan_telescope_y.csv", np.column_stack([angles, rel]), delimiter=",",
                       header="Angle [deg],relative flux", comments="")
    return 0


if __name__ == "__main__":
    sys.exit(main())
