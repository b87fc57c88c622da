"""Outputs of a run: the stdout counters and containment radii of `generateResultPlots` (src/raytracer.nim:2246-2635)
and the detector-image CSV of `plotHeatmap` (rt:856-921). Plots (ggplotnim PDFs/PNGs) are presentation and out of scope.

The reference sorts `pointdataR` of every passed ray (rt:2459-2527). `containment_radii` restates that on per-ray
records (traceAxionWrapper output); `containment_radii_from_hist` gives the same four radii from the weighted radial
histogram the fused GPU run fills (sart_enable_radial_hist), to within one histogram bin — no per-ray data leaves the
GPU for a 1e9-ray run.
"""
from __future__ import annotations

from dataclasses import dataclass
from pathlib import Path

import numpy as np

from . import abi

WINDOW_YEAR_NAMES = abi.WINDOW_YEAR_NAMES   # `$windowYear` (rt:43-46): "2017", "2018", "BabyIAXO"


def _nim_round(x: float) -> int:
    """std/math round: half away from zero."""
    return int(np.floor(abs(x) + 0.5) * (1 if x >= 0 else -1))


@dataclass
class ContainmentRadii:
    rSigma1: float    # 68 % of the passed rays (count) inside
    rSigma2: float    # 95.5 %
    rSigma1W: float   # 68 % of the summed weight inside (the value handed to plotHeatmap, rt:2635)
    rSigma2W: float   # 95.5 %


def containment_radii(pointdataR, weights) -> ContainmentRadii:
    """rt:2459-2527 on the passed rays' radii and weights, including its quirks: the weighted scan starts at index
    round(0.63 n) + 1, so a weighted radius stays 0 when its threshold is crossed before that index."""
    R = np.asarray(pointdataR, dtype=np.float64)
    W = np.asarray(weights, dtype=np.float64)
    n = R.size
    if n == 0:
        return ContainmentRadii(0.0, 0.0, 0.0, 0.0)
    order = np.argsort(R, kind="stable")
    Rs, Ws = R[order], W[order]
    s1, s2 = _nim_round(n * 0.68), _nim_round(n * 0.955)
    r1 = float(Rs[s1 - 1]) if s1 >= 1 else 0.0
    r2 = float(Rs[s2 - 1]) if s2 >= 1 else 0.0
    cum = np.cumsum(Ws)
    total = float(cum[-1])
    k0 = _nim_round(n * 0.63)
    idx = np.arange(n)
    in1 = (idx > k0) & (cum < total * 0.68)
    in2 = (idx > k0) & (cum < total * 0.955) & (cum >= total * 0.68)
    r1w = float(Rs[np.nonzero(in1)[0][-1]]) if in1.any() else 0.0
    r2w = float(Rs[np.nonzero(in2)[0][-1]]) if in2.any() else 0.0
    return ContainmentRadii(r1, r2, r1w, r2w)


def containment_radii_from_hist(edges, sum_w, counts) -> ContainmentRadii:
    """The same four radii from a radial histogram (bin edges [nb + 1], sum of weights and ray counts per bin); inside
    the bin where a threshold is crossed the radius is interpolated linearly."""
    edges = np.asarray(edges, dtype=np.float64)
    w = np.asarray(sum_w, dtype=np.float64)
    c = np.asarray(counts, dtype=np.float64)
    n = c.sum()
    if n == 0:
        return ContainmentRadii(0.0, 0.0, 0.0, 0.0)

    def quantile(cum, target):
        j = int(np.searchsorted(cum, target, side="left"))
        j = min(j, cum.size - 1)
        below = cum[j - 1] if j > 0 else 0.0
        step = cum[j] - below
        f = (target - below) / step if step > 0 else 0.0
        return float(edges[j] + f * (edges[j + 1] - edges[j]))

    cc, cw = np.cumsum(c), np.cumsum(w)
    r1, r2 = quantile(cc, _nim_round(n * 0.68)), quantile(cc, _nim_round(n * 0.955))
    total = float(cw[-1])
    r63 = quantile(cc, _nim_round(n * 0.63) + 1)
    r1w, r2w = quantile(cw, total * 0.68), quantile(cw, total * 0.955)
    # the reference only looks beyond the 63 % count index (rt:2502-2510)
    r1w = r1w if r1w > r63 else 0.0
    r2w = r2w if r2w > r63 else 0.0
    return ContainmentRadii(r1, r2, r1w, r2w)


CSV_COLUMNS = ["x", "y", "photon flux", "yr0", "yr02", "x-position [mm]", "y-position [mm]", "xr", "xrneg", "yr", "xr2",
               "xrneg2", "yr2"]


def axion_image_table(image: np.ndarray, rSigma1: float, rSigma2: float, chipXMax: float = 14.0,
                      chipYMax: float = 14.0) -> dict[str, np.ndarray]:
    """The data frame of plotHeatmap (rt:863-896) as columns: row k = y * width + x, `photon flux` = image[y, x],
    yr0 / yr02 = linspace(-rSigma, rSigma, width^2), the circle columns offset by the chip centre (rt:873)."""
    img = np.asarray(image, dtype=np.float64)
    assert img.ndim == 2 and img.shape[0] == img.shape[1]
    width = img.shape[0]
    n = width * width
    ys, xs = np.divmod(np.arange(n), width)
    offset = chipXMax / 2.0           # ChipCenterX rt:265
    yr0, yr02 = np.linspace(-rSigma1, rSigma1, n), np.linspace(-rSigma2, rSigma2, n)
    with np.errstate(invalid="ignore"):
        c1, c2 = np.sqrt(rSigma1 * rSigma1 - yr0 * yr0), np.sqrt(rSigma2 * rSigma2 - yr02 * yr02)
    return {"x": xs, "y": ys, "photon flux": img.reshape(-1), "yr0": yr0, "yr02": yr02,
            "x-position [mm]": xs * chipXMax / width, "y-position [mm]": ys * chipYMax / width,
            "xr": c1 + offset, "xrneg": -c1 + offset, "yr": yr0 + offset,
            "xr2": c2 + offset, "xrneg2": -c2 + offset, "yr2": yr02 + offset}


def write_axion_image_csv(path: str | Path, image: np.ndarray, rSigma1: float, rSigma2: float, chipXMax: float = 14.0,
                          chipYMax: float = 14.0, precision: int = 17) -> Path:
    """`df.writeCsv(outpath / "axion_image_{year}{suffix}.csv")` (rt:896): one header line with the 13 column names,
    65 536 rows. Numbers are written with `precision` significant digits (datamancer's writeCsv default is 4; the
    default here round-trips f64 — pass precision=4 for byte-compatible files)."""
    tab = axion_image_table(image, rSigma1, rSigma2, chipXMax, chipYMax)
    path = Path(path)
    path.parent.mkdir(parents=True, exist_ok=True)
    cols = [tab[c] for c in CSV_COLUMNS]
    fmt = f"%.{precision}g"
    with open(path, "w") as f:
        f.write(",".join(CSV_COLUMNS) + "\n")
        for k in range(cols[0].size):
            f.write(f"{int(cols[0][k])},{int(cols[1][k])}," + ",".join(fmt % c[k] for c in cols[2:]) + "\n")
    return path


def read_axion_image_csv(path: str | Path) -> tuple[np.ndarray, dict[str, np.ndarray]]:
    """Reads a CSV written by the reference or by write_axion_image_csv back into (image [w, w], columns)."""
    with open(path) as f:
        header = f.readline().rstrip("\n").split(",")
    data = np.genfromtxt(path, delimiter=",", skip_header=1)
    cols = {name: data[:, i] for i, name in enumerate(header)}
    width = int(round(np.sqrt(data.shape[0])))
    img = np.zeros((width, width))
    img[cols["y"].astype(int), cols["x"].astype(int)] = cols["photon flux"]
    return img, cols


def result_summary(counters: dict, radii: ContainmentRadii | None = None, image: np.ndarray | None = None) -> str:
    """The lines generateResultPlots and plotHeatmap echo (rt:2253-2257, 2276-2278, 2512-2513, 886)."""
    n = max(1, counters["n_passed"])
    lines = [f"Passed axions {counters['n_passed']}",
             f"Passed axions until the Window {counters['n_passed_till_window']}",
             f"Number of X-rays hitting nickel: {counters['n_hit_nickel']}",
             f"{counters['sum_x'] / n}", f"{counters['sum_y'] / n}", f"{counters['sum_r'] / n}",
             "Extracted all data!"]
    if radii is not None:
        lines += [f"{radii.rSigma1W}vs {radii.rSigma1}", f"{radii.rSigma2W}vs {radii.rSigma2}"]
    lines.append("all plots done, now to heatmap!")
    if image is not None:
        lines.append(f"The total flux arriving in the detector is: {float(np.sum(image))}")
    return "\n".join(lines)


@dataclass
class Spectra:
    """Weighted spectra of the passed rays of a run: per energy bin (bin i < nE = tabulated energy i, bin nE = the X-ray
    source's energy) and per mirror shell (shellNumber rt:2198) the sum of weights, of squared weights and the ray count."""
    energies_keV: np.ndarray   # [nE + 1]: the tabulated energies, then the source energy (NaN without an X-ray source)
    sum_w: np.ndarray          # [nE + 1]
    sum_w2: np.ndarray         # [nE + 1]
    counts: np.ndarray         # [nE + 1] uint64
    shell_sum_w: np.ndarray    # [nShells]
    shell_counts: np.ndarray   # [nShells] uint64


def spectra_from_records(energy_keV, shell, weights, energies, source_energy: float | None = None,
                         n_shells: int = abi.MAX_SHELLS) -> Spectra:
    """The spectra of per-ray records (traceAxionWrapper output), the host-side counterpart of the fused run's
    (RayTracer.read_spectra). Rays with weight != 0 are the passed ones (rt:2220). Bins are energy INDICES: a record
    reports fmax(energies[i], 0.03) keV (rt:470-471), so the index is recovered from the value; table energies below
    0.03 keV all report 0.03 and are credited to the first of them. With `source_energy` (an X-ray source run, which draws no
    table energies) every ray goes to bin nE."""
    E = np.asarray(energy_keV, dtype=np.float64)
    S = np.asarray(shell, dtype=np.int64)
    W = np.asarray(weights, dtype=np.float64)
    en = np.asarray(energies, dtype=np.float64)
    nE = en.size
    sel = W != 0.0
    E, S, W = E[sel], S[sel], W[sel]
    if source_energy is not None:
        idx = np.full(E.size, nE, dtype=np.int64)
    else:
        reported = np.maximum(en, 0.03)
        idx = np.searchsorted(reported, E, side="left")
        ok = (idx < nE) & (reported[np.minimum(idx, nE - 1)] == E)
        if not ok.all():
            raise ValueError(f"{int((~ok).sum())} record energies are not tabulated energies")
    if S.size and (S.min() < 0 or S.max() >= n_shells):
        raise ValueError("shell numbers of passed rays outside [0, n_shells)")
    src = np.nan if source_energy is None else float(source_energy)
    return Spectra(energies_keV=np.append(en, src),
                   sum_w=np.bincount(idx, weights=W, minlength=nE + 1),
                   sum_w2=np.bincount(idx, weights=W * W, minlength=nE + 1),
                   counts=np.bincount(idx, minlength=nE + 1).astype(np.uint64),
                   shell_sum_w=np.bincount(S, weights=W, minlength=n_shells),
                   shell_counts=np.bincount(S, minlength=n_shells).astype(np.uint64))


SPECTRUM_COLUMNS = ["Energy [keV]", "flux", "flux error", "rays"]
SHELL_FLUX_COLUMNS = ["shell", "flux", "rays"]


def _write_columns(path: str | Path, header: list[str], cols: list[np.ndarray], ints: set[int], precision: int) -> Path:
    path = Path(path)
    path.parent.mkdir(parents=True, exist_ok=True)
    fmt = f"%.{precision}g"
    with open(path, "w") as f:
        f.write(",".join(header) + "\n")
        for k in range(cols[0].size):
            f.write(",".join(str(int(c[k])) if j in ints else fmt % c[k] for j, c in enumerate(cols)) + "\n")
    return path


def write_energy_spectrum_csv(path: str | Path, spectra: Spectra, precision: int = 17) -> Path:
    """The energy spectrum of the detected flux: one row per energy bin with a known energy (the source bin is left out
    without an X-ray source), columns `Energy [keV]`, `flux` (Σw), `flux error` (√Σw²) and `rays`."""
    keep = np.isfinite(spectra.energies_keV)
    return _write_columns(path, SPECTRUM_COLUMNS, [spectra.energies_keV[keep], spectra.sum_w[keep],
                                                   np.sqrt(spectra.sum_w2[keep]), spectra.counts[keep]], {3}, precision)


def write_shell_flux_csv(path: str | Path, spectra: Spectra, precision: int = 17) -> Path:
    """The detected flux per mirror shell: columns `shell`, `flux` (Σw) and `rays`."""
    n = spectra.shell_sum_w.size
    return _write_columns(path, SHELL_FLUX_COLUMNS, [np.arange(n), spectra.shell_sum_w, spectra.shell_counts], {0, 2},
                          precision)


def read_columns_csv(path: str | Path) -> dict[str, np.ndarray]:
    """Reads a CSV written by write_energy_spectrum_csv / write_shell_flux_csv back into its columns."""
    with open(path) as f:
        header = f.readline().rstrip("\n").split(",")
    data = np.loadtxt(path, delimiter=",", skiprows=1, ndmin=2)
    return {name: data[:, i] for i, name in enumerate(header)}


def write_spectra_csvs(spectra: Spectra, windowYear: int, outpath: str | Path, suffix: str = "",
                       precision: int = 17) -> tuple[Path, Path]:
    """`axion_energy_spectrum_{year}{suffix}.csv` and `axion_shell_flux_{year}{suffix}.csv` next to the image CSV."""
    year = WINDOW_YEAR_NAMES.get(windowYear, str(windowYear))
    return (write_energy_spectrum_csv(Path(outpath) / f"axion_energy_spectrum_{year}{suffix}.csv", spectra, precision),
            write_shell_flux_csv(Path(outpath) / f"axion_shell_flux_{year}{suffix}.csv", spectra, precision))


def mass_suffix(mAxion: float) -> str:
    """File-name suffix of one axion mass of a mass scan: `_ma{m:.6g}eV`."""
    return f"_ma{mAxion:.6g}eV"


def write_mass_spectra_csvs(spectra: list[Spectra], masses, windowYear: int, outpath: str | Path,
                            precision: int = 17) -> list[Path]:
    """The spectra of a mass scan (RayTracer.read_mass_spectra), one pair of write_spectra_csvs files per mass:
    `axion_energy_spectrum_{year}_ma{m:.6g}eV.csv` and `axion_shell_flux_{year}_ma{m:.6g}eV.csv`."""
    masses = [float(m) for m in masses]
    if len(spectra) != len(masses):
        raise ValueError(f"{len(spectra)} spectra for {len(masses)} masses")
    if len({mass_suffix(m) for m in masses}) != len(masses):
        raise ValueError("two masses of the scan share a file name (they agree to 6 significant digits)")
    paths: list[Path] = []
    for s, m in zip(spectra, masses):
        paths.extend(write_spectra_csvs(s, windowYear, outpath, suffix=mass_suffix(m), precision=precision))
    return paths


@dataclass
class BandImages:
    """Detector images of the passed rays of a run per energy band (RayTracer.enable_band_images): band b holds the rays
    whose energy lies in [edges[b], edges[b + 1]) keV."""
    edges: np.ndarray       # [B + 1] keV, strictly ascending
    image: np.ndarray       # [B, 256, 256] Σw, image[b, y, x] like the run's image
    image_w2: np.ndarray    # [B, 256, 256] Σw²
    counts: np.ndarray      # [B] uint64: the passed rays of each band, in the image or not


def parse_energy_bands(text: str) -> list[float]:
    """The value of --energyBands: 2 .. abi.MAX_BANDS + 1 comma-separated edges in keV, finite, >= 0 and strictly
    ascending ("0.5,2,4,8": three bands)."""
    try:
        edges = [float(x) for x in text.split(",")]
    except ValueError:
        raise ValueError(f"expected comma-separated energies in keV, got {text!r}") from None
    if not 2 <= len(edges) <= abi.MAX_BANDS + 1:
        raise ValueError(f"need 2 to {abi.MAX_BANDS + 1} edges (1 to {abi.MAX_BANDS} bands), got {len(edges)}")
    if not all(np.isfinite(e) and e >= 0.0 for e in edges) or any(b <= a for a, b in zip(edges, edges[1:])):
        raise ValueError(f"the edges must be finite, >= 0 and strictly ascending, got {text!r}")
    return edges


def band_suffix(lo: float, hi: float) -> str:
    """File-name suffix of the energy band [lo, hi) keV: `_E{lo:g}-{hi:g}keV`."""
    return f"_E{lo:g}-{hi:g}keV"


def write_band_image_csvs(bands: BandImages, windowYear: int, outpath: str | Path, radii: ContainmentRadii | None = None,
                          chipXMax: float = 14.0, chipYMax: float = 14.0, precision: int = 17, suffix: str = "") -> list[Path]:
    """One write_axion_image_csv file per energy band, `axion_image_{year}_E{lo:g}-{hi:g}keV{suffix}.csv`, next to the run's
    image. The radius columns carry `radii`, the containment radii of the whole run: per-band radii are not computed."""
    edges = [float(e) for e in bands.edges]
    if len(edges) != bands.image.shape[0] + 1:
        raise ValueError(f"{len(edges)} edges for {bands.image.shape[0]} band images")
    names = [band_suffix(lo, hi) for lo, hi in zip(edges, edges[1:])]
    if len(set(names)) != len(names):
        raise ValueError("two bands share a file name (their edges agree to 6 significant digits)")
    radii = radii or ContainmentRadii(0.0, 0.0, 0.0, 0.0)
    year = WINDOW_YEAR_NAMES.get(windowYear, str(windowYear))
    return [write_axion_image_csv(Path(outpath) / f"axion_image_{year}{sfx}{suffix}.csv", img, radii.rSigma1W, radii.rSigma2W,
                                  chipXMax, chipYMax, precision) for sfx, img in zip(names, bands.image)]


@dataclass
class QuantityHist:
    """Weighted histogram of one per-ray record quantity of the passed rays of a run (RayTracer.enable_quantity_hists).
    Entry 0 is the underflow (v < lo), entries 1 .. nbins the regular bins [edges[k-1], edges[k]), entry nbins + 1 the
    overflow (v >= hi or NaN)."""
    name: str               # a field of sart_ray_out_t: abi.QUANTITIES
    edges: np.ndarray       # [nbins + 1] lo + (hi - lo) k / nbins
    sum_w: np.ndarray       # [nbins + 2] Σw
    sum_w2: np.ndarray      # [nbins + 2] Σw²
    counts: np.ndarray      # [nbins + 2] uint64


def check_quantity_hist_specs(specs) -> list[tuple[str, int, float, float]]:
    """The specs of RayTracer.enable_quantity_hists, [(name, nbins, lo, hi), ...], checked like sart_enable_quantity_hists
    checks them: at most one histogram per quantity, names from abi.QUANTITIES, 1 .. abi.MAX_QHIST_BINS bins, lo and hi
    finite with lo < hi. Raises ValueError."""
    out = []
    for spec in specs:
        try:
            name, nbins, lo, hi = spec
        except (TypeError, ValueError):
            raise ValueError(f"a histogram spec is (name, nbins, lo, hi), got {spec!r}") from None
        if name not in abi.QUANTITIES:
            raise ValueError(f"unknown quantity {name!r}; one of {', '.join(abi.QUANTITIES)}")
        if any(name == o[0] for o in out):
            raise ValueError(f"quantity {name!r} is histogrammed twice")
        if isinstance(nbins, bool) or int(nbins) != nbins or not 1 <= int(nbins) <= abi.MAX_QHIST_BINS:
            raise ValueError(f"{name}: need 1 to {abi.MAX_QHIST_BINS} bins, got {nbins!r}")
        lo, hi = float(lo), float(hi)
        if not (np.isfinite(lo) and np.isfinite(hi) and lo < hi):
            raise ValueError(f"{name}: lo and hi must be finite with lo < hi, got {lo!r}, {hi!r}")
        out.append((name, int(nbins), lo, hi))
    return out


def parse_quantity_hist(text: str) -> tuple[str, int, float, float]:
    """One value of --histogram: `NAME:NBINS:LO:HI`, e.g. `transMagnet:256:0:1e-20`."""
    parts = text.split(":")
    if len(parts) != 4:
        raise ValueError(f"expected NAME:NBINS:LO:HI, got {text!r}")
    name, nbins, lo, hi = parts
    try:
        n, a, b = int(nbins), float(lo), float(hi)
    except ValueError:
        raise ValueError(f"expected NAME:NBINS:LO:HI with an integer NBINS and numbers LO, HI, got {text!r}") from None
    return check_quantity_hist_specs([(name, n, a, b)])[0]


def quantity_hist_entries(values, nbins: int, lo: float, hi: float) -> np.ndarray:
    """The entry of each value in a histogram of `nbins` bins over [lo, hi), the binning of sart_enable_quantity_hists bit
    for bit: 0 if v < lo, nbins + 1 if not v < hi (NaN included), else 1 + fmin(floor((v - lo) * inv), nbins - 1) with
    inv = nbins / (hi - lo), every operation rounded on its own."""
    v = np.asarray(values, dtype=np.float64)
    lo, hi = np.float64(lo), np.float64(hi)
    inv = np.float64(nbins) / (hi - lo)
    with np.errstate(invalid="ignore", over="ignore"):
        reg = 1.0 + np.fmin(np.floor((v - lo) * inv), np.float64(nbins - 1))
        e = np.where(v < lo, 0.0, np.where(~(v < hi), np.float64(nbins + 1), reg))
    return e.astype(np.int64)


def quantity_hists_from_records(records, specs) -> list[QuantityHist]:
    """The quantity histograms of per-ray records (an AxionBatch of RayTracer.trace_mc_rays, or anything with the arrays `w`
    and those the specs name), the host-side counterpart of RayTracer.read_quantity_hists: the rays with w != 0 (rt:2220)
    are counted, each with the value of its record."""
    W = np.asarray(records.w, dtype=np.float64)
    sel = W != 0.0
    W = W[sel]
    out = []
    for name, nbins, lo, hi in check_quantity_hist_specs(specs):
        v = getattr(records, name)
        if v is None:
            raise ValueError(f"the records have no {name!r} array")
        e = quantity_hist_entries(np.asarray(v, dtype=np.float64)[sel], nbins, lo, hi)
        out.append(QuantityHist(name, quantity_hist_edges(nbins, lo, hi),
                                np.bincount(e, weights=W, minlength=nbins + 2),
                                np.bincount(e, weights=W * W, minlength=nbins + 2),
                                np.bincount(e, minlength=nbins + 2).astype(np.uint64)))
    return out


def quantity_hist_edges(nbins: int, lo: float, hi: float) -> np.ndarray:
    """The nbins + 1 edges of the regular bins, lo + (hi - lo) k / nbins (the last one exactly hi)."""
    e = lo + (hi - lo) * (np.arange(nbins + 1, dtype=np.float64) / nbins)
    e[-1] = hi
    return e


QUANTITY_HIST_COLUMNS = ["lower edge", "upper edge", "flux", "flux error", "rays"]


def write_quantity_hist_csvs(hists: list[QuantityHist], windowYear: int, outpath: str | Path,
                             precision: int = 17, suffix: str = "") -> list[Path]:
    """One `axion_hist_{name}_{year}{suffix}.csv` per histogram next to the image CSV: columns `lower edge`, `upper edge`, `flux`
    (Σw), `flux error` (√Σw²) and `rays`, one row per entry; the underflow row has the lower edge -inf, the overflow row
    (NaN values included) the upper edge inf."""
    year = WINDOW_YEAR_NAMES.get(windowYear, str(windowYear))
    paths = []
    for h in hists:
        lower = np.concatenate(([-np.inf], h.edges))
        upper = np.concatenate((h.edges, [np.inf]))
        paths.append(_write_columns(Path(outpath) / f"axion_hist_{h.name}_{year}{suffix}.csv", QUANTITY_HIST_COLUMNS,
                                    [lower, upper, h.sum_w, np.sqrt(h.sum_w2), h.counts], {4}, precision))
    return paths


@dataclass
class ScanOutputs:
    """An angular scan with its accumulators (RayTracer.angular_scan_outputs): per scan point the flux, the counters, the
    image, and a row of every accumulator that was on (None for those that were off)."""
    angles: np.ndarray                                  # [n] telescope_turned_y [deg]
    fluxes: np.ndarray                                  # [n] Σw of the passed rays
    counters: list[dict]                                # [n]
    images: np.ndarray | None                           # [n, 256, 256] when asked for
    radial_hists: list[tuple] | None                    # [n] (bin edges, Σw, counts), as RayTracer.read_radial_hist
    spectra: list[Spectra] | None                       # [n]
    band_images: list[BandImages] | None                # [n]
    quantity_hists: list[list[QuantityHist]] | None     # [n] one QuantityHist per spec


def concat_scan_outputs(parts: list[ScanOutputs]) -> ScanOutputs:
    """The scan points of `parts` (consecutive blocks of one scan, e.g. one per GPU) as one ScanOutputs."""
    def cat(name):
        vals = [getattr(p, name) for p in parts]
        if any(v is None for v in vals):
            return None
        return np.concatenate(vals) if isinstance(vals[0], np.ndarray) else [x for v in vals for x in v]
    return ScanOutputs(*(cat(f) for f in ScanOutputs.__dataclass_fields__))


def angle_suffix(angle_deg: float) -> str:
    """File-name suffix of one point of an angular scan: `_angle{a:g}deg`."""
    return f"_angle{angle_deg:g}deg"


RADII_COLUMNS = ["Angle [deg]", "rSigma1", "rSigma2", "rSigma1W", "rSigma2W"]
MASS_COLUMN = "mAxion [eV]"   # first column of mass_scan_radii.csv


def write_scan_radii_csv(path: str | Path, angles, radii: list[ContainmentRadii], precision: int = 17,
                         first_column: str = RADII_COLUMNS[0]) -> Path:
    """The containment radii of every scan point (containment_radii_from_hist of its radial histogram, about the chip
    centre): columns `first_column` (the scan variable: `Angle [deg]` of an angular scan, MASS_COLUMN of a mass scan), then
    rSigma1, rSigma2, rSigma1W, rSigma2W [mm]."""
    a = np.asarray(angles, dtype=np.float64)
    if a.size != len(radii):
        raise ValueError(f"{len(radii)} radii for {a.size} scan points")
    cols = [a] + [np.array([getattr(r, f) for r in radii], dtype=np.float64) for f in RADII_COLUMNS[1:]]
    return _write_columns(path, [first_column] + RADII_COLUMNS[1:], cols, set(), precision)


def write_scan_outputs(scan: ScanOutputs, windowYear: int, outpath: str | Path, chipXMax: float = 14.0,
                       chipYMax: float = 14.0, precision: int = 17) -> list[Path]:
    """The files of an angular scan with accumulators: `angular_scan_telescope_y_radii.csv` (write_scan_radii_csv; with the
    radial histogram on), and for
    every scan point the spectra, band-image and quantity-histogram files of a fused run with the suffix `_angle{a:g}deg`
    (angle_suffix). The band images carry that point's own containment radii."""
    suffixes = [angle_suffix(float(a)) for a in scan.angles]
    if len(set(suffixes)) != len(suffixes):
        raise ValueError("two scan points share a file name (their angles agree to 6 significant digits)")
    paths: list[Path] = []
    radii = [None] * len(suffixes)
    if scan.radial_hists is not None:
        radii = [containment_radii_from_hist(*h) for h in scan.radial_hists]
        paths.append(write_scan_radii_csv(Path(outpath) / "angular_scan_telescope_y_radii.csv", scan.angles, radii, precision))
    for i, sfx in enumerate(suffixes):
        if scan.spectra is not None:
            paths.extend(write_spectra_csvs(scan.spectra[i], windowYear, outpath, suffix=sfx, precision=precision))
        if scan.band_images is not None:
            paths.extend(write_band_image_csvs(scan.band_images[i], windowYear, outpath, radii[i], chipXMax, chipYMax,
                                               precision, suffix=sfx))
        if scan.quantity_hists is not None:
            paths.extend(write_quantity_hist_csvs(scan.quantity_hists[i], windowYear, outpath, precision, suffix=sfx))
    return paths


def generateResultPlots(result, windowYear: int, outpath: str | Path, suffix: str = "",
                        radii: ContainmentRadii | None = None, chipXMax: float = 14.0, chipYMax: float = 14.0,
                        precision: int = 17, echo=print) -> Path:
    """generateResultPlots (rt:2246-2635) for a fused run: echoes the counters and writes
    `axion_image_{windowYear}{suffix}.csv` from the 256x256 image (heatmaptable2, rt:2629-2635). `result` is a
    raytracer.RunResult; `radii` comes from containment_radii(_from_hist)."""
    radii = radii or ContainmentRadii(0.0, 0.0, 0.0, 0.0)
    echo(result_summary(result.counters[0], radii, result.image[0]))
    year = WINDOW_YEAR_NAMES.get(windowYear, str(windowYear))
    return write_axion_image_csv(Path(outpath) / f"axion_image_{year}{suffix}.csv", result.image[0], radii.rSigma1W,
                                 radii.rSigma2W, chipXMax, chipYMax, precision)


def write_mass_scan_outputs(masses, radial_hists: list[tuple], band_images: list[BandImages] | None, windowYear: int,
                            outpath: str | Path, chipXMax: float = 14.0, chipYMax: float = 14.0,
                            precision: int = 17) -> list[Path]:
    """The per-mass radii and band images of a mass scan (RayTracer.read_mass_radial_hist / read_mass_band_images):
    `mass_scan_radii.csv` (write_scan_radii_csv with the masses in column MASS_COLUMN), and with `band_images` for every
    mass the write_band_image_csvs files `axion_image_{year}_E{lo:g}-{hi:g}keV_ma{m:.6g}eV.csv`, whose radius columns
    carry that mass's containment radii."""
    masses = [float(m) for m in masses]
    if len(radial_hists) != len(masses) or (band_images is not None and len(band_images) != len(masses)):
        raise ValueError(f"{len(radial_hists)} radial histograms and "
                         f"{'no' if band_images is None else len(band_images)} band images for {len(masses)} masses")
    suffixes = [mass_suffix(m) for m in masses]
    if len(set(suffixes)) != len(suffixes):
        raise ValueError("two masses of the scan share a file name (they agree to 6 significant digits)")
    radii = [containment_radii_from_hist(*h) for h in radial_hists]
    paths = [write_scan_radii_csv(Path(outpath) / "mass_scan_radii.csv", masses, radii, precision, MASS_COLUMN)]
    for k, sfx in enumerate(suffixes):
        if band_images is not None:
            paths.extend(write_band_image_csvs(band_images[k], windowYear, outpath, radii[k], chipXMax, chipYMax, precision,
                                               suffix=sfx))
    return paths
