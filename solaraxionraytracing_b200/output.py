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
