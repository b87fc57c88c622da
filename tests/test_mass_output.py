"""Host side of the per-mass radii and band images of a mass scan: the --massScanRadii / --massScanBands switches and their
refusals, write_mass_scan_outputs (file names, round trips) and write_scan_radii_csv with another first column."""
import re
from pathlib import Path

import numpy as np
import pytest

from solaraxionraytracing_b200 import __main__ as cli
from solaraxionraytracing_b200 import abi, config, output

ROOT = Path(__file__).resolve().parents[1]
NAMES = ("sart_enable_mass_radial_hist", "sart_read_mass_radial_hist", "sart_read_merged_mass_radial_hist",
         "sart_enable_mass_band_images", "sart_read_mass_band_images", "sart_read_merged_mass_band_images")


def test_command_line_arguments(capsys):
    a = cli.parse_args(["--massScanBands", "0.5,2,4,8", "--massScanRadii"])
    assert a.massScanBands == [0.5, 2.0, 4.0, 8.0] and a.massScanRadii
    a = cli.parse_args([])
    assert a.massScanBands is None and not a.massScanRadii
    with pytest.raises(SystemExit) as e:
        cli.parse_args(["--massScanBands", "4,2"])
    assert e.value.code == 2 and "--massScanBands" in capsys.readouterr().err


def _config(tmp_path, masses=None, extra=""):
    cfg = tmp_path / "c.toml"
    txt = config.DEFAULT_CONFIG.read_text()
    if masses is not None:
        txt += f"\n[Run]\nmAxion = {masses}\n"
    cfg.write_text(txt + extra)
    return cfg


@pytest.mark.parametrize("switch", [["--massScanRadii"], ["--massScanBands", "0.5,2,4,8"]])
def test_command_line_refuses_a_single_mass(tmp_path, capsys, switch):
    """Without a mass scan, and with a mass scan that is also an angular scan, the switches are argument errors that
    point to --energyBands, before any table is loaded."""
    with pytest.raises(SystemExit) as e:
        cli.main(["--config", str(_config(tmp_path)), *switch])
    err = capsys.readouterr().err
    assert e.value.code == 2 and switch[0] in err and "--energyBands" in err and "mass scan" in err
    with pytest.raises(SystemExit) as e:
        cli.main(["--config", str(_config(tmp_path, [0.01, 0.02])), "--angularScanMin", "0", "--angularScanMax", "0.1",
                  *switch])
    err = capsys.readouterr().err
    assert e.value.code == 2 and switch[0] in err and "angular scan" in err


def test_energy_bands_on_a_mass_scan_points_to_the_new_switch(tmp_path, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(["--config", str(_config(tmp_path, [0.01, 0.02])), "--energyBands", "0.5,2,4,8"])
    err = capsys.readouterr().err
    assert e.value.code == 2 and "single axion mass" in err and "--massScanBands" in err


def test_write_scan_radii_csv_first_column(tmp_path):
    radii = [output.ContainmentRadii(1.0, 2.0, 1.5, 2.5), output.ContainmentRadii(0.5, 1.25, 0.75, 1.75)]
    p = output.write_scan_radii_csv(tmp_path / "m.csv", [0.004, 0.02], radii, first_column=output.MASS_COLUMN)
    cols = output.read_columns_csv(p)
    assert list(cols) == [output.MASS_COLUMN, "rSigma1", "rSigma2", "rSigma1W", "rSigma2W"]
    assert np.array_equal(cols[output.MASS_COLUMN], [0.004, 0.02])
    assert np.array_equal(cols["rSigma2W"], [2.5, 1.75])
    # the default stays the angular scan's
    assert list(output.read_columns_csv(output.write_scan_radii_csv(tmp_path / "a.csv", [0.0, 0.1], radii))) == \
        output.RADII_COLUMNS


def _hist(rng, nbins=64, r_max=8.0):
    n = rng.integers(0, 50, nbins).astype(np.uint64)
    return np.linspace(0.0, r_max, nbins + 1), n * rng.random(nbins), n


def _bands(rng, edges, nb):
    img = rng.random((nb, abi.IMAGE_BINS, abi.IMAGE_BINS)) * (rng.random((nb, abi.IMAGE_BINS, abi.IMAGE_BINS)) < 0.002)
    return output.BandImages(np.asarray(edges), img, img * img, rng.integers(0, 1000, nb).astype(np.uint64))


def test_write_mass_scan_outputs_names_and_round_trip(tmp_path):
    rng = np.random.default_rng(3)
    masses = [0.004, 0.0082351, 0.02]
    edges = [0.5, 2.0, 4.0]
    hists = [_hist(rng) for _ in masses]
    bands = [_bands(rng, edges, 2) for _ in masses]
    paths = output.write_mass_scan_outputs(masses, hists, bands, 2, tmp_path)
    names = sorted(p.name for p in paths)
    want = ["mass_scan_radii.csv"] + [f"axion_image_BabyIAXO_E{lo:g}-{hi:g}keV_ma{m:.6g}eV.csv"
                                      for m in masses for lo, hi in zip(edges, edges[1:])]
    assert names == sorted(want) and sorted(p.name for p in tmp_path.iterdir()) == names
    radii = output.read_columns_csv(tmp_path / "mass_scan_radii.csv")
    for k, m in enumerate(masses):
        r = output.containment_radii_from_hist(*hists[k])
        assert radii[output.MASS_COLUMN][k] == m
        assert [radii[f][k] for f in output.RADII_COLUMNS[1:]] == [r.rSigma1, r.rSigma2, r.rSigma1W, r.rSigma2W]
        for j, (lo, hi) in enumerate(zip(edges, edges[1:])):
            img, cols = output.read_axion_image_csv(tmp_path / f"axion_image_BabyIAXO_E{lo:g}-{hi:g}keV_ma{m:.6g}eV.csv")
            assert np.array_equal(img, bands[k].image[j])
            assert np.nanmax(cols["yr0"]) == r.rSigma1W and np.nanmax(cols["yr02"]) == r.rSigma2W   # this mass's radii
    # radii only
    for p in tmp_path.iterdir():
        p.unlink()
    assert [p.name for p in output.write_mass_scan_outputs(masses, hists, None, 2, tmp_path)] == ["mass_scan_radii.csv"]


def test_write_mass_scan_outputs_refusals(tmp_path):
    rng = np.random.default_rng(4)
    with pytest.raises(ValueError, match="for 3 masses"):
        output.write_mass_scan_outputs([0.01, 0.02, 0.03], [_hist(rng)] * 2, None, 2, tmp_path)
    with pytest.raises(ValueError, match="for 2 masses"):
        output.write_mass_scan_outputs([0.01, 0.02], [_hist(rng)] * 2, [_bands(rng, [1.0, 2.0], 1)], 2, tmp_path)
    with pytest.raises(ValueError, match="share a file name"):
        output.write_mass_scan_outputs([0.01, 0.0100000001], [_hist(rng)] * 2, None, 2, tmp_path)
    assert not any(tmp_path.iterdir())


def test_header_and_abi_declare_the_entry_points():
    header = (ROOT / "include" / "sart.h").read_text()
    for name in NAMES:
        assert re.search(rf"\bint {name}\(", header), name
        assert name in abi.SIGNATURES, name


def test_library_exports_the_entry_points():
    from solaraxionraytracing_b200._lib import lib
    for name in NAMES:
        assert hasattr(lib, name), name
    assert lib.sart_enable_mass_radial_hist(None, 16, 1.0) == -1   # SART_ERR_ARG: no handle
    assert lib.sart_enable_mass_band_images(None, 0, None) == -1
    assert lib.sart_read_mass_radial_hist(None, None, None) == -1
    assert lib.sart_read_merged_mass_band_images(None, None, None, None) == -1
