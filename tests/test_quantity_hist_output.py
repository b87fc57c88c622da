"""Host side of the quantity histograms (sart_enable_quantity_hists): spec parsing and checks, the binning rule of
output.quantity_hists_from_records against a brute-force loop, and the CSV files of write_quantity_hist_csvs."""
import math

import numpy as np
import pytest

from solaraxionraytracing_b200 import abi, output


def test_parse_and_check_specs():
    assert output.parse_quantity_hist("transMagnet:256:0:1e-20") == ("transMagnet", 256, 0.0, 1e-20)
    assert output.parse_quantity_hist("yaw:1:-0.5:0.5") == ("yaw", 1, -0.5, 0.5)
    for bad in ("transMagnet:256:0", "bogus:4:0:1", "yaw:0:0:1", "yaw:513:0:1", "yaw:4.5:0:1", "yaw:4:1:1", "yaw:4:2:1",
                "yaw:4:nan:1", "yaw:4:0:inf", "yaw:x:0:1", "yaw:4:a:1", "yaw:4:0:1:2"):
        with pytest.raises(ValueError):
            output.parse_quantity_hist(bad)
    assert len(output.check_quantity_hist_specs([(q, 512, 0, 1) for q in abi.QUANTITIES])) == abi.N_QUANTITIES
    with pytest.raises(ValueError, match="twice"):
        output.check_quantity_hist_specs([("yaw", 4, 0, 1), ("yaw", 8, 0, 2)])
    with pytest.raises(ValueError):
        output.check_quantity_hist_specs([("yaw", 4, 0)])
    with pytest.raises(ValueError):
        output.check_quantity_hist_specs([("yaw", True, 0, 1)])


def test_command_line_parses_histograms():
    from solaraxionraytracing_b200.__main__ import parse_args
    a = parse_args(["--histogram", "reflect:20:0:1", "--histogram", "yaw:10:-0.5:0.5"])
    assert a.histogram == [("reflect", 20, 0.0, 1.0), ("yaw", 10, -0.5, 0.5)]
    assert parse_args([]).histogram is None
    for bad in (["--histogram", "reflect:20:0:1", "--histogram", "reflect:10:0:2"], ["--histogram", "bogus:4:0:1"],
                ["--histogram", "yaw:0:0:1"], ["--histogram", "yaw:4:1:0"]):
        with pytest.raises(SystemExit):
            parse_args(bad)


def _brute(v, nbins, lo, hi):
    inv = nbins / (hi - lo)
    if v < lo:
        return 0
    if not v < hi:
        return nbins + 1
    t = math.floor((v - lo) * inv)
    return 1 + int(min(t, nbins - 1))


@pytest.mark.parametrize("nbins,lo,hi", [(1, 0.0, 1.0), (7, -0.3, 0.45), (512, 1e-22, 3.3e-20), (10, -5.0, 5.0),
                                         (3, 0.1, 0.1000000000000001)])
def test_binning_against_a_brute_force_loop(nbins, lo, hi):
    rng = np.random.default_rng(nbins)
    span = hi - lo
    inner = lo + span * np.arange(nbins + 1) / nbins
    v = np.concatenate([rng.uniform(lo - span, hi + span, 5000), inner, np.nextafter(inner, -np.inf),
                        np.nextafter(inner, np.inf), [lo, hi, np.nextafter(hi, -np.inf), np.inf, -np.inf, np.nan, 0.0]])
    e = output.quantity_hist_entries(v, nbins, lo, hi)
    assert e.tolist() == [_brute(float(x), nbins, lo, hi) for x in v]
    assert output.quantity_hist_entries([lo], nbins, lo, hi)[0] == 1
    assert output.quantity_hist_entries([hi, np.inf, np.nan], nbins, lo, hi).tolist() == [nbins + 1] * 3
    assert output.quantity_hist_entries([-np.inf, np.nextafter(lo, -np.inf)], nbins, lo, hi).tolist() == [0, 0]


class _Records:
    def __init__(self, n, rng):
        self.w = np.where(rng.uniform(size=n) < 0.3, 0.0, rng.uniform(0.1, 2.0, size=n))
        for q in abi.QUANTITIES:
            setattr(self, q, rng.normal(size=n))
        self.yaw[:5] = [np.nan, np.inf, -np.inf, -1.0, 1.0]


def test_records_histograms_against_a_brute_force_loop():
    rng = np.random.default_rng(3)
    rec = _Records(3000, rng)
    specs = [("yaw", 5, -1.0, 1.0), ("reflect", 12, -2.0, 0.5)]
    hists = output.quantity_hists_from_records(rec, specs)
    for h, (name, nb, lo, hi) in zip(hists, specs):
        assert h.name == name and h.counts.dtype == np.uint64 and h.counts.size == nb + 2
        sw, sw2, n = np.zeros(nb + 2), np.zeros(nb + 2), np.zeros(nb + 2, dtype=np.uint64)
        for v, w in zip(getattr(rec, name), rec.w):
            if w == 0.0:
                continue
            k = _brute(float(v), nb, lo, hi)
            sw[k] += w; sw2[k] += w * w; n[k] += 1
        assert np.array_equal(h.counts, n)
        assert np.allclose(h.sum_w, sw, rtol=1e-13, atol=0) and np.allclose(h.sum_w2, sw2, rtol=1e-13, atol=0)
        assert int(h.counts.sum()) == int(np.count_nonzero(rec.w))
        assert h.edges[0] == lo and h.edges[-1] == hi and h.edges.size == nb + 1
    rec.pathCB = None
    with pytest.raises(ValueError, match="pathCB"):
        output.quantity_hists_from_records(rec, [("pathCB", 4, 0.0, 1.0)])


def test_csv_round_trip(tmp_path):
    rng = np.random.default_rng(5)
    hists = output.quantity_hists_from_records(_Records(2000, rng), [("transMagnet", 9, -1.5, 1.5), ("alpha2", 3, 0.0, 1.0)])
    paths = output.write_quantity_hist_csvs(hists, abi.WY_IAXO, tmp_path)
    assert [p.name for p in paths] == ["axion_hist_transMagnet_BabyIAXO.csv", "axion_hist_alpha2_BabyIAXO.csv"]
    for p, h in zip(paths, hists):
        c = output.read_columns_csv(p)
        assert list(c) == output.QUANTITY_HIST_COLUMNS
        assert c["lower edge"][0] == -np.inf and c["upper edge"][-1] == np.inf
        assert np.array_equal(c["lower edge"][1:], h.edges) and np.array_equal(c["upper edge"][:-1], h.edges)
        assert np.array_equal(c["flux"], h.sum_w) and np.array_equal(c["flux error"], np.sqrt(h.sum_w2))
        assert np.array_equal(c["rays"].astype(np.uint64), h.counts)
