"""Host side of the angular scan with accumulators (no GPU): the ctypes mirror of sart_scan_out_t, the file names and
contents of output.write_scan_outputs, the containment-radii CSV and the joining of blocks of scan points."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from solaraxionraytracing_b200 import abi, output

ROOT = Path(__file__).resolve().parents[1]


def test_scan_out_mirrors_the_header():
    hdr = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "sart.h").read_text(), flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\} sart_scan_out_t;", hdr).group(1)
    fields = re.findall(r"(double|uint64_t)\*\s*(\w+)", body)
    assert [n for _, n in fields] == [n for n, _ in abi.ScanOut._fields_]
    want = {"double": C.POINTER(C.c_double), "uint64_t": C.POINTER(C.c_uint64)}
    assert [want[t] for t, _ in fields] == [t for _, t in abi.ScanOut._fields_]
    assert C.sizeof(abi.ScanOut) == len(fields) * C.sizeof(C.c_void_p)
    assert "sart_angular_scan_outputs" in abi.SIGNATURES


def test_angle_suffix():
    assert [output.angle_suffix(a) for a in np.linspace(-0.05, 0.05, 3)] == ["_angle-0.05deg", "_angle0deg", "_angle0.05deg"]
    assert output.angle_suffix(0.15000000000000002) == "_angle0.15deg"


def _scan(angles, rng, radial=True):
    n = len(angles)
    nb, nE = 32, 5
    edges = np.array([0.5, 2.0, 4.0])
    energies = np.array([0.01, 1.0, 3.0, 5.0, 7.0])

    def spectra():
        return output.Spectra(np.append(energies, np.nan), rng.random(nE + 1), rng.random(nE + 1),
                              rng.integers(0, 100, nE + 1).astype(np.uint64), rng.random(3),
                              rng.integers(0, 100, 3).astype(np.uint64))
    rad = [(np.linspace(0, 10, nb + 1), rng.random(nb), rng.integers(1, 50, nb).astype(np.uint64)) for _ in range(n)]
    bands = [output.BandImages(edges.copy(), rng.random((2, 256, 256)), rng.random((2, 256, 256)),
                               rng.integers(0, 9, 2).astype(np.uint64)) for _ in range(n)]
    qh = [[output.QuantityHist("reflect", output.quantity_hist_edges(4, 0.0, 1.0), rng.random(6), rng.random(6),
                               rng.integers(0, 9, 6).astype(np.uint64))] for _ in range(n)]
    return output.ScanOutputs(np.asarray(angles, dtype=np.float64), rng.random(n), [{"n_passed": k} for k in range(n)],
                              None, rad if radial else None, [spectra() for _ in range(n)], bands, qh)


def test_write_scan_outputs_names_and_contents(tmp_path):
    rng = np.random.default_rng(1)
    scan = _scan([-0.05, 0.0, 0.05], rng)
    paths = output.write_scan_outputs(scan, abi.WY_IAXO, tmp_path)
    names = sorted(p.name for p in paths)
    want = ["angular_scan_telescope_y_radii.csv"]
    for sfx in ("_angle-0.05deg", "_angle0deg", "_angle0.05deg"):
        want += [f"axion_energy_spectrum_BabyIAXO{sfx}.csv", f"axion_shell_flux_BabyIAXO{sfx}.csv",
                 f"axion_image_BabyIAXO_E0.5-2keV{sfx}.csv", f"axion_image_BabyIAXO_E2-4keV{sfx}.csv",
                 f"axion_hist_reflect_BabyIAXO{sfx}.csv"]
    assert names == sorted(want)
    radii = output.read_columns_csv(tmp_path / "angular_scan_telescope_y_radii.csv")
    assert list(radii) == output.RADII_COLUMNS == ["Angle [deg]", "rSigma1", "rSigma2", "rSigma1W", "rSigma2W"]
    assert np.array_equal(radii["Angle [deg]"], scan.angles)
    for i, sfx in enumerate(("_angle-0.05deg", "_angle0deg", "_angle0.05deg")):
        r = output.containment_radii_from_hist(*scan.radial_hists[i])
        assert [radii[f][i] for f in output.RADII_COLUMNS[1:]] == [r.rSigma1, r.rSigma2, r.rSigma1W, r.rSigma2W]
        sp = output.read_columns_csv(tmp_path / f"axion_energy_spectrum_BabyIAXO{sfx}.csv")
        assert np.array_equal(sp["flux"], scan.spectra[i].sum_w[:-1])
        img, cols = output.read_axion_image_csv(tmp_path / f"axion_image_BabyIAXO_E2-4keV{sfx}.csv")
        assert np.array_equal(img, scan.band_images[i].image[1])
        assert cols["yr0"][-1] == r.rSigma1W and cols["yr02"][-1] == r.rSigma2W   # the point's own radii
        h = output.read_columns_csv(tmp_path / f"axion_hist_reflect_BabyIAXO{sfx}.csv")
        assert np.array_equal(h["rays"].astype(np.uint64), scan.quantity_hists[i][0].counts)


def test_write_scan_outputs_without_radial_hist_and_clashing_angles(tmp_path):
    rng = np.random.default_rng(2)
    paths = output.write_scan_outputs(_scan([0.1, 0.2], rng, radial=False), abi.WY_2018, tmp_path)
    assert "angular_scan_telescope_y_radii.csv" not in {p.name for p in paths}
    _, cols = output.read_axion_image_csv(tmp_path / "axion_image_2018_E0.5-2keV_angle0.1deg.csv")
    assert cols["yr0"][-1] == 0.0
    with pytest.raises(ValueError, match="share a file name"):
        output.write_scan_outputs(_scan([0.1, 0.1000000001], rng), abi.WY_2018, tmp_path)


def test_write_scan_radii_csv(tmp_path):
    r = [output.ContainmentRadii(1.0, 2.0, 0.0, 2.5), output.ContainmentRadii(1.25, 2.125, 1.5, 3.0)]
    p = output.write_scan_radii_csv(tmp_path / "r.csv", [0.0, 0.3], r)
    assert p.read_text().splitlines() == ["Angle [deg],rSigma1,rSigma2,rSigma1W,rSigma2W", "0,1,2,0,2.5",
                                          "0.29999999999999999,1.25,2.125,1.5,3"]
    with pytest.raises(ValueError):
        output.write_scan_radii_csv(tmp_path / "r.csv", [0.0], r)


def test_concat_scan_outputs():
    rng = np.random.default_rng(3)
    a, b = _scan([0.0, 0.1], rng), _scan([0.2], rng)
    b.images = np.zeros((1, 256, 256))
    c = output.concat_scan_outputs([a, b])
    assert np.array_equal(c.angles, [0.0, 0.1, 0.2]) and np.array_equal(c.fluxes, np.concatenate([a.fluxes, b.fluxes]))
    assert c.counters == a.counters + b.counters
    assert c.images is None   # not every block has its images
    assert c.spectra == a.spectra + b.spectra and c.band_images[2] is b.band_images[0]
    assert c.quantity_hists[2] is b.quantity_hists[0] and c.radial_hists[1] is a.radial_hists[1]
