"""The per-mass spectra writer of a mass scan with --writeSpectra (output.write_mass_spectra_csvs)."""
import numpy as np
import pytest

from solaraxionraytracing_b200 import output


def _spectra(scale: float, n: int) -> output.Spectra:
    return output.Spectra(energies_keV=np.array([0.5, 1.5, np.nan]), sum_w=np.array([scale, 2.0 * scale, 0.0]),
                          sum_w2=np.array([scale ** 2, 4.0 * scale ** 2, 0.0]), counts=np.array([n, 2 * n, 0], dtype=np.uint64),
                          shell_sum_w=np.array([3.0 * scale, 0.0]), shell_counts=np.array([3 * n, 0], dtype=np.uint64))


def test_one_pair_of_files_per_mass(tmp_path):
    masses = [0.004, 0.008235101411623404, 0.02]
    spectra = [_spectra(10.0 ** -k, k + 1) for k in range(3)]
    paths = output.write_mass_spectra_csvs(spectra, masses, 2, tmp_path / "out")
    assert [p.name for p in paths] == [
        "axion_energy_spectrum_BabyIAXO_ma0.004eV.csv", "axion_shell_flux_BabyIAXO_ma0.004eV.csv",
        "axion_energy_spectrum_BabyIAXO_ma0.0082351eV.csv", "axion_shell_flux_BabyIAXO_ma0.0082351eV.csv",
        "axion_energy_spectrum_BabyIAXO_ma0.02eV.csv", "axion_shell_flux_BabyIAXO_ma0.02eV.csv"]
    for k in range(3):
        e = output.read_columns_csv(paths[2 * k])
        s = output.read_columns_csv(paths[2 * k + 1])
        assert e["Energy [keV]"].tolist() == [0.5, 1.5]   # no source row without an X-ray source
        assert e["flux"].tolist() == spectra[k].sum_w[:2].tolist() and e["rays"].tolist() == [k + 1, 2 * (k + 1)]
        assert s["flux"].tolist() == spectra[k].shell_sum_w.tolist() and s["rays"].tolist() == [3 * (k + 1), 0]
        assert e["rays"].sum() == s["rays"].sum() and e["flux"].sum() == s["flux"].sum()


def test_suffix_and_refusals(tmp_path):
    assert output.mass_suffix(0.0853) == "_ma0.0853eV" and output.mass_suffix(1e-6) == "_ma1e-06eV"
    with pytest.raises(ValueError, match="2 spectra for 1 masses"):
        output.write_mass_spectra_csvs([_spectra(1.0, 1)] * 2, [0.01], 2, tmp_path)
    with pytest.raises(ValueError, match="share a file name"):
        output.write_mass_spectra_csvs([_spectra(1.0, 1)] * 2, [0.01, 0.0100000001], 2, tmp_path)
    assert not any(tmp_path.iterdir())   # nothing written when the call is refused
