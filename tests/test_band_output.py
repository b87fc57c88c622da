"""The band images of the command line and the C-ABI without a GPU: --energyBands parsing and its refusals (a mass scan
included), the file names and the round trip of output.write_band_image_csvs, and the new symbols in libsart and abi.py."""
import re
from pathlib import Path

import numpy as np
import pytest

from solaraxionraytracing_b200 import __main__ as cli
from solaraxionraytracing_b200 import abi, config, output

ROOT = Path(__file__).resolve().parents[1]


def test_parse_energy_bands():
    assert output.parse_energy_bands("0.5,2,4,8") == [0.5, 2.0, 4.0, 8.0]
    assert output.parse_energy_bands("0,15") == [0.0, 15.0]
    assert len(output.parse_energy_bands(",".join(str(k) for k in range(17)))) == 17


@pytest.mark.parametrize("text,match", [("1", "need 2 to 17"), (",".join(str(k) for k in range(18)), "need 2 to 17"),
                                        ("2,1", "ascending"), ("1,1", "ascending"), ("-1,2", ">= 0"),
                                        ("0,inf", "finite"), ("0,nan", "finite"), ("0;1", "comma-separated"),
                                        ("", "comma-separated")])
def test_parse_energy_bands_refusals(text, match):
    with pytest.raises(ValueError, match=match):
        output.parse_energy_bands(text)


def test_command_line_arguments(capsys):
    assert cli.parse_args(["--energyBands", "0.5,2,4,8"]).energyBands == [0.5, 2.0, 4.0, 8.0]
    assert cli.parse_args([]).energyBands is None
    with pytest.raises(SystemExit) as e:
        cli.parse_args(["--energyBands", "3"])
    assert e.value.code == 2 and "--energyBands" in capsys.readouterr().err


def test_command_line_refuses_a_mass_scan(tmp_path, capsys):
    """A configuration with several axion masses and --energyBands is an argument error, before any table is loaded."""
    cfg = tmp_path / "scan.toml"
    cfg.write_text(config.DEFAULT_CONFIG.read_text() + "\n[Run]\nmAxion = [0.01, 0.02]\n")
    with pytest.raises(SystemExit) as e:
        cli.main(["--config", str(cfg), "--energyBands", "0.5,2,4,8"])
    assert e.value.code == 2 and "single axion mass" in capsys.readouterr().err


def _bands(nb=3):
    rng = np.random.default_rng(7)
    img = rng.random((nb, abi.IMAGE_BINS, abi.IMAGE_BINS)) * (rng.random((nb, abi.IMAGE_BINS, abi.IMAGE_BINS)) < 0.01)
    return output.BandImages(edges=np.array([0.5, 2.0, 4.0, 8.0][:nb + 1]), image=img, image_w2=img * img,
                             counts=np.arange(1, nb + 1, dtype=np.uint64))


def test_writer_names_and_round_trip(tmp_path):
    b = _bands()
    radii = output.ContainmentRadii(1.0, 2.0, 1.5, 2.5)
    paths = output.write_band_image_csvs(b, abi.WY_IAXO, tmp_path / "out", radii)
    assert [p.name for p in paths] == ["axion_image_BabyIAXO_E0.5-2keV.csv", "axion_image_BabyIAXO_E2-4keV.csv",
                                       "axion_image_BabyIAXO_E4-8keV.csv"]
    whole = output.write_axion_image_csv(tmp_path / "whole.csv", b.image.sum(axis=0), radii.rSigma1W, radii.rSigma2W)
    _, wcols = output.read_axion_image_csv(whole)
    for k, p in enumerate(paths):
        img, cols = output.read_axion_image_csv(p)
        assert list(cols) == output.CSV_COLUMNS and len(cols["x"]) == abi.IMAGE_BINS ** 2
        assert np.array_equal(img, b.image[k])   # 17 significant digits round-trip f64
        for c in ("yr0", "yr02", "xr", "yr2"):      # the whole run's containment radii
            assert np.array_equal(np.nan_to_num(cols[c]), np.nan_to_num(wcols[c])), c


def test_writer_refusals(tmp_path):
    b = _bands()
    with pytest.raises(ValueError, match="edges for 3 band images"):
        output.write_band_image_csvs(output.BandImages(b.edges[:3], b.image, b.image_w2, b.counts), 2, tmp_path)
    same = output.BandImages(np.array([1.0, 1.0000001, 1.0000002]), b.image[:2], b.image_w2[:2], b.counts[:2])
    with pytest.raises(ValueError, match="share a file name"):
        output.write_band_image_csvs(same, 2, tmp_path)
    assert not any(tmp_path.iterdir())


def test_header_and_abi_declare_the_band_images():
    header = (ROOT / "include" / "sart.h").read_text()
    assert re.search(r"#define SART_MAX_BANDS (\d+)", header).group(1) == str(abi.MAX_BANDS)
    for name in ("sart_enable_band_images", "sart_read_band_images", "sart_read_merged_band_images"):
        assert re.search(rf"\bint {name}\(", header), name
        assert name in abi.SIGNATURES, name


def test_library_exports_the_band_images():
    from solaraxionraytracing_b200._lib import lib
    for name in ("sart_enable_band_images", "sart_read_band_images", "sart_read_merged_band_images"):
        assert hasattr(lib, name), name
    assert lib.sart_enable_band_images(None, 3, None) == -1   # SART_ERR_ARG: no handle
    assert lib.sart_read_band_images(None, None, None, None) == -1
