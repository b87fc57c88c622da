"""Host-side spectra of per-ray records (output.spectra_from_records) and the two CSV writers of --writeSpectra."""
import numpy as np
import pytest

from solaraxionraytracing_b200 import output


def test_spectra_from_records_bins_by_energy_index():
    energies = np.array([0.001, 0.011, 0.5, 1.0, 2.0])   # the first two both report 0.03 keV (rt:470-471)
    E = np.array([0.03, 0.5, 2.0, 2.0, 1.0, 0.5, 0.03])
    shell = np.array([0, 1, 2, 2, 0, 3, 1])
    w = np.array([0.5, 1.0, 2.0, 3.0, 0.0, 4.0, 0.25])      # w = 0: not passed (rt:2220), left out
    s = output.spectra_from_records(E, shell, w, energies, n_shells=4)
    assert s.energies_keV.size == 6 and np.isnan(s.energies_keV[-1])
    assert s.counts.tolist() == [2, 0, 2, 0, 2, 0]
    assert s.sum_w.tolist() == [0.75, 0.0, 5.0, 0.0, 5.0, 0.0]
    assert s.sum_w2.tolist() == [0.3125, 0.0, 17.0, 0.0, 13.0, 0.0]
    assert s.shell_counts.tolist() == [1, 2, 2, 1] and s.shell_sum_w.tolist() == [0.5, 1.25, 5.0, 4.0]
    with pytest.raises(ValueError, match="not tabulated"):
        output.spectra_from_records([0.7], [0], [1.0], energies)
    with pytest.raises(ValueError, match="shell"):
        output.spectra_from_records([0.5], [4], [1.0], energies, n_shells=4)


def test_spectra_from_records_xray_source_goes_to_the_last_bin():
    s = output.spectra_from_records([3.0, 3.0, 3.0], [0, 1, 1], [1.0, 0.0, 2.0], [1.0, 2.0], source_energy=3.0, n_shells=2)
    assert s.counts.tolist() == [0, 0, 2] and s.sum_w[-1] == 3.0 and s.energies_keV[-1] == 3.0


def test_spectrum_csv_round_trip(tmp_path):
    s = output.Spectra(energies_keV=np.array([0.5, 1.0 / 3.0, np.nan]), sum_w=np.array([1e-20, np.pi, 0.0]),
                       sum_w2=np.array([1e-40, 2.0, 0.0]), counts=np.array([3, 7, 0], dtype=np.uint64),
                       shell_sum_w=np.array([np.e, 0.0, 1.5]), shell_counts=np.array([4, 0, 6], dtype=np.uint64))
    pe, ps = output.write_spectra_csvs(s, 2, tmp_path / "out", suffix="_x")
    assert pe.name == "axion_energy_spectrum_BabyIAXO_x.csv" and ps.name == "axion_shell_flux_BabyIAXO_x.csv"
    assert pe.read_text().splitlines()[0] == "Energy [keV],flux,flux error,rays"
    e = output.read_columns_csv(pe)
    assert e["Energy [keV]"].tolist() == [0.5, 1.0 / 3.0]          # no source row without an X-ray source
    assert e["flux"].tolist() == [1e-20, np.pi] and e["flux error"].tolist() == [1e-20, np.sqrt(2.0)]
    assert e["rays"].tolist() == [3, 7]
    assert ps.read_text().splitlines()[1] == "0,2.7182818284590451,4"
    sh = output.read_columns_csv(ps)
    assert sh["shell"].tolist() == [0, 1, 2] and sh["flux"].tolist() == [np.e, 0.0, 1.5] and sh["rays"].tolist() == [4, 0, 6]
