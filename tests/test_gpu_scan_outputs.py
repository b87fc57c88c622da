"""sart_angular_scan_outputs / RayTracer.angular_scan_outputs: an angular scan that also fills, per scan point, a row of the
radial histogram, the spectra, the band images and the quantity histograms.

  * a row equals sart_update_setup (turned) + sart_reset_image + sart_trace_mc of the point's rays + the readers: exactly
    (counts identical, sums to 1e-12) in modes 0 and 1, in mode 2 at the handle's own angle and with the alias sampler; at
    other angles mode 2 keeps the handle's error budgets, so the rows agree as test_gpu_angular_scan.py explains;
  * the rows agree with each other and with the counters, mode 2 has mode 0's spectra and band counts, mode 0 has the
    oracle's spectra and quantity histograms;
  * the call leaves the handle's accumulators, image and counters as they were and gives sart_angular_scan's fluxes,
    counters and images; its refusals; the command line writes one set of files per scan point."""
import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import abi, output

pytestmark = pytest.mark.gpu
SEED = 299792458
EDGES = [0.5, 2.0, 4.0, 8.0]
ANGLES = np.array([0.0, 0.05, -0.05, 0.02])


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


def _turned(setup, angle):
    s = abi.Setup.from_buffer_copy(bytes(setup))
    s.telescope.telescope_turned_y = angle
    return s


def _specs(tr, n=100_000):
    """All eight quantities over the 2nd .. 98th percentile of the passed rays' values of n records."""
    rec = tr.traceAxionWrapper(n, SEED + 1)
    sel = rec.w != 0.0
    specs = []
    for k, name in enumerate(abi.QUANTITIES):
        v = np.asarray(getattr(rec, name))[sel]
        v = v[np.isfinite(v)]
        lo, hi = np.percentile(v, [2.0, 98.0]) if v.size else (0.0, 1.0)
        if not lo < hi:
            lo, hi = lo - 1.0 - abs(lo), hi + 1.0 + abs(hi)
        specs.append((name, 40 + 5 * k, float(lo), float(hi)))
    return specs


def _enable_all(tr, specs):
    tr.enable_radial_hist(4096)
    tr.enable_spectra()
    tr.enable_band_images(EDGES)
    tr.enable_quantity_hists(specs)


def _loop_point(tr, setup, mode, angle, first, n):
    tr.update_setup(_turned(setup, angle))
    tr.set_precision(mode)
    tr.reset_image()
    tr.trace_mc(n, SEED, first_ray=first)
    return (tr.read_image(), tr.read_radial_hist(), tr.read_spectra(), tr.read_band_images(), tr.read_quantity_hists())


def _close(a, b, rtol=1e-12):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.allclose(a, b, rtol=rtol, atol=1e-15 * max(float(np.abs(b).sum()), 1e-300))


def _assert_rows_equal(so, i, ref):
    """Row i of the scan equals the readers of a fused run: counts identical, sums within 1e-12."""
    _, (e, w, n), spec, bands, qh = ref
    re, rw, rn = so.radial_hists[i]
    assert np.array_equal(re, e) and np.array_equal(rn, n) and _close(rw, w)
    s = so.spectra[i]
    assert np.array_equal(s.counts, spec.counts) and np.array_equal(s.shell_counts, spec.shell_counts)
    assert _close(s.sum_w, spec.sum_w) and _close(s.sum_w2, spec.sum_w2) and _close(s.shell_sum_w, spec.shell_sum_w)
    b = so.band_images[i]
    assert np.array_equal(b.edges, bands.edges) and np.array_equal(b.counts, bands.counts)
    assert _close(b.image, bands.image) and _close(b.image_w2, bands.image_w2)
    for g, h in zip(so.quantity_hists[i], qh, strict=True):
        assert g.name == h.name and np.array_equal(g.edges, h.edges) and np.array_equal(g.counts, h.counts), g.name
        assert _close(g.sum_w, h.sum_w) and _close(g.sum_w2, h.sum_w2), g.name


def _l1(a, b):
    return float(np.abs(np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64)).sum())


def _assert_rows_close(so, i, ref):
    """Mode 2 at a turned angle (test_gpu_angular_scan.py: test_scan_equals_loop_of_runs): the same rays pass, so every
    count that depends on the energy or the shell only, and every total, is identical; what depends on a position or a
    record value may move a re-traced ray (at most 2.4e-3 of the rays) into a neighbouring bin."""
    _, (_, w, n), spec, bands, qh = ref
    _, rw, rn = so.radial_hists[i]
    assert int(rn.sum()) == int(n.sum()) and _l1(rn, n) <= 5e-3 * n.sum() and _l1(rw, w) <= 5e-3 * w.sum()
    s = so.spectra[i]
    assert np.array_equal(s.counts, spec.counts) and np.array_equal(s.shell_counts, spec.shell_counts)
    assert s.sum_w.sum() == pytest.approx(spec.sum_w.sum(), rel=1e-5)
    b = so.band_images[i]
    assert np.array_equal(b.counts, bands.counts)
    assert _l1(b.image, bands.image) <= 5e-3 * bands.image.sum()
    for g, h in zip(so.quantity_hists[i], qh, strict=True):
        assert int(g.counts.sum()) == int(h.counts.sum()), g.name
        assert _l1(g.counts, h.counts) <= 5e-3 * h.counts.sum() and _l1(g.sum_w, h.sum_w) <= 5e-3 * h.sum_w.sum(), g.name


def _assert_internal_sums(so):
    """Per row: Σ spectra counts = Σ radial counts = each histogram's Σ counts = n_passed, Σ energy Σw = the flux, and the
    band counts are the spectra counts summed over the energy bins whose reported energy lies in each band."""
    for i, c in enumerate(so.counters):
        s = so.spectra[i]
        assert int(s.counts.sum()) == int(so.radial_hists[i][2].sum()) == c["n_passed"]
        for h in so.quantity_hists[i]:
            assert int(h.counts.sum()) == c["n_passed"], h.name
        assert s.sum_w.sum() == pytest.approx(so.fluxes[i], rel=1e-12)
        e = np.maximum(s.energies_keV[:-1], 0.03)
        want = [int(s.counts[:-1][(e >= lo) & (e < hi)].sum()) for lo, hi in zip(EDGES, EDGES[1:])]
        assert so.band_images[i].counts.tolist() == want


@pytest.mark.parametrize("cfg", ["babyiaxo_xmm", "cast_llnl"])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_rows_equal_a_loop_of_fused_runs(rt, cfg, mode):
    setup, tb = make_config(cfg)
    n = 300_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        specs = _specs(tr)
        tr.set_precision(mode)
        _enable_all(tr, specs)
        so = tr.angular_scan_outputs(ANGLES, n, SEED, want_images=True, first_ray=3 * n)
        _assert_internal_sums(so)
        for i, a in enumerate(ANGLES):
            ref = _loop_point(tr, setup, mode, a, (3 + i) * n, n)
            c = ref[0].counters[0]
            assert c["n_exit"] == so.counters[i]["n_exit"] and c["n_passed"] == so.counters[i]["n_passed"]
            if mode == 2 and a != 0.0:
                _assert_rows_close(so, i, ref)
            else:
                _assert_rows_equal(so, i, ref)


def test_alias_sampler_rows_equal_the_loop(rt):
    """The alias sampler has no re-trace, so the error budgets play no part: every row equals the loop's at every angle."""
    setup, tb = make_config("babyiaxo_xmm")
    n = 300_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        specs = _specs(tr)
        tr.set_precision(2)
        tr.set_sampler(abi.SAMPLER_ALIAS)
        _enable_all(tr, specs)
        so = tr.angular_scan_outputs(ANGLES, n, SEED)
        _assert_internal_sums(so)
        for i, a in enumerate(ANGLES):
            _assert_rows_equal(so, i, _loop_point(tr, setup, 2, a, i * n, n))


@pytest.mark.parametrize("cfg", ["babyiaxo_xmm", "cast_llnl"])
@pytest.mark.parametrize("scale", [None, 12.0])
def test_mode2_has_the_spectra_and_band_counts_of_mode0(rt, cfg, scale):
    setup, tb = make_config(cfg)
    n = 500_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        _enable_all(tr, _specs(tr))
        tr.set_precision(0)
        s0 = tr.angular_scan_outputs(ANGLES, n, SEED)
        tr.set_precision(2)
        if scale is not None:
            tr.set_retrace(1, scale)
        s2 = tr.angular_scan_outputs(ANGLES, n, SEED)
    _assert_internal_sums(s2)
    for i in range(ANGLES.size):
        if scale is not None:
            assert s2.counters[i]["n_retraced"] > 0.01 * n
        assert s2.counters[i]["n_unresolved"] == 0
        assert np.array_equal(s2.spectra[i].counts, s0.spectra[i].counts)
        assert np.array_equal(s2.spectra[i].shell_counts, s0.spectra[i].shell_counts)
        assert np.array_equal(s2.band_images[i].counts, s0.band_images[i].counts)


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_mode0_rows_equal_the_oracle_records(rt, oracle, cfg):
    """Each row's spectra and quantity histograms are those of mode 0's per-ray records of the turned setup (exactly), and
    those of the oracle's records up to the rays whose exit code, weight or histogram entry libm moves (as in
    test_gpu_quantity_hists.py: test_mode0_equals_the_oracle_records)."""
    setup, tb = make_config(cfg)
    n = 200_000
    angles = np.array([0.0, 0.04])
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        specs = _specs(tr)
        tr.set_precision(0)
        tr.enable_spectra()
        tr.enable_quantity_hists(specs)
        so = tr.angular_scan_outputs(angles, n, SEED)
        for i, a in enumerate(angles):
            s = _turned(setup, a)
            tr.update_setup(s)
            gpu = tr.traceAxionWrapper(n, SEED, first_ray=i * n)
            ref = oracle.trace_mc_rays(s, tb, i * n, n, SEED)
            exact = output.spectra_from_records(gpu.energy, gpu.shell, gpu.w, tb.energies)
            assert np.array_equal(so.spectra[i].counts, exact.counts)
            assert np.array_equal(so.spectra[i].shell_counts[:s.telescope.nShells], exact.shell_counts[:s.telescope.nShells])
            assert _close(so.spectra[i].sum_w, exact.sum_w)
            for g, h in zip(so.quantity_hists[i], output.quantity_hists_from_records(gpu, specs), strict=True):
                assert np.array_equal(g.counts, h.counts) and _close(g.sum_w, h.sum_w), g.name
            odd = (gpu.code != ref.code) | (np.abs(gpu.w - ref.w) > 1e-10 * np.abs(ref.w))
            for name, nb, lo, hi in specs:
                odd |= output.quantity_hist_entries(getattr(gpu, name), nb, lo, hi) != \
                    output.quantity_hist_entries(getattr(ref, name), nb, lo, hi)
            print(cfg, a, "rays libm moves:", int(odd.sum()))
            assert odd.sum() <= n // 500
            orc = output.spectra_from_records(ref.energy, ref.shell, ref.w, tb.energies)
            assert _l1(so.spectra[i].counts, orc.counts) <= 2 * odd.sum()
            for g, h in zip(so.quantity_hists[i], output.quantity_hists_from_records(ref, specs)):
                assert _l1(g.counts, h.counts) <= 2 * odd.sum(), g.name


def _handle_state(tr):
    r = tr.read_image()
    parts = [r.image, r.image_w2]
    parts += list(tr.read_radial_hist()[1:])
    s = tr.read_spectra()
    parts += [s.sum_w, s.sum_w2, s.counts, s.shell_sum_w, s.shell_counts]
    b = tr.read_band_images()
    parts += [b.image, b.image_w2, b.counts]
    for h in tr.read_quantity_hists():
        parts += [h.sum_w, h.sum_w2, h.counts]
    return parts, r.counters


@pytest.mark.parametrize("mode", [0, 2])
def test_no_side_effects_and_the_scan_results_of_sart_angular_scan(rt, mode):
    setup, tb = make_config("babyiaxo_xmm")
    n = 300_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        fl, cnt, img = tr.angular_scan(ANGLES, n, SEED, want_images=True)
        _enable_all(tr, _specs(tr))
        tr.reset_image()
        tr.trace_mc(n, SEED, first_ray=10 * n)
        before, cnt_before = _handle_state(tr)
        so = tr.angular_scan_outputs(ANGLES, n, SEED, want_images=True)
        after, cnt_after = _handle_state(tr)
    assert cnt_before == cnt_after
    for x, y in zip(before, after, strict=True):
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()
    for i in range(ANGLES.size):
        c, d = dict(cnt[i]), dict(so.counters[i])
        for k in ("sum_w", "sum_w2", "sum_x", "sum_y", "sum_r"):
            assert d.pop(k) == pytest.approx(c.pop(k), rel=1e-12), k
        assert c == d
    assert np.allclose(so.fluxes, fl, rtol=1e-12, atol=0)
    assert np.allclose(so.images, img, rtol=1e-10, atol=1e-15 * img.sum())
    assert np.array_equal(so.angles, ANGLES)


def test_refusals(rt):
    from solaraxionraytracing_b200._lib import lib
    import ctypes as C
    setup, tb = make_config("babyiaxo_xmm")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        with pytest.raises(rt.SartError) as e:   # nothing on
            tr.angular_scan_outputs(ANGLES, 1000, SEED)
        assert e.value.code == -1
        tr.enable_spectra()
        a = np.ascontiguousarray(ANGLES)
        fl = np.empty(a.size)
        w = np.empty((a.size, 4096))
        out = abi.ScanOut()
        out.radial_sum_w = w.ctypes.data_as(abi.c_double_p)   # the radial histogram is off
        rc = lib.sart_angular_scan_outputs(tr._h, a.size, a.ctypes.data_as(abi.c_double_p), 0, 1000, SEED,
                                           fl.ctypes.data_as(abi.c_double_p), None, None, C.byref(out))
        assert rc == -1 and b"radial histogram" in lib.sart_last_error()
        # a failed allocation: 16 band images for 200 000 scan points are 3.2 TB
        tr.enable_band_images(np.linspace(0.5, 8.5, 17))
        big = np.zeros(200_000)
        flb = np.empty(big.size)
        rc = lib.sart_angular_scan_outputs(tr._h, big.size, big.ctypes.data_as(abi.c_double_p), 0, 1000, SEED,
                                           flb.ctypes.data_as(abi.c_double_p), None, None, None)
        assert rc == -4, lib.sart_last_error()
        so = tr.angular_scan_outputs(ANGLES, 100_000, SEED)   # and the handle still works
        assert so.spectra[0].counts.sum() == so.counters[0]["n_passed"] > 0
        tr.set_axion_masses([1e-3, 2e-3])
        with pytest.raises(rt.SartError) as e:
            tr.angular_scan_outputs(ANGLES, 1000, SEED)
        assert e.value.code == -1
        tr.set_axion_masses([1e-3])
        tr.enable_spectra(False)
        tr.enable_mass_spectra()
        with pytest.raises(rt.SartError) as e:
            tr.angular_scan_outputs(ANGLES, 1000, SEED)
        assert e.value.code == -3


def _cli(tmp_path, name, extra, monkeypatch=None, rt=None):
    from solaraxionraytracing_b200.__main__ import main
    from solaraxionraytracing_b200 import config
    cfg = tmp_path / f"{name}.toml"
    cfg.write_text(config.DEFAULT_CONFIG.read_text().replace('outputPath = "../out"', f'outputPath = "{tmp_path}/{name}"'))
    assert main(["--config", str(cfg), "--nRays", "200000", "--allowSynthetic", "--angularScanMin", "-0.05",
                 "--angularScanMax", "0.05", "--numAngularScanPoints", "3", "--writeSpectra", "--energyBands", "0.5,2,4,8",
                 "--histogram", "reflect:64:0:1"] + extra) == 0
    return tmp_path / name


def _files_equal_scan(out, so):
    """The files of the command line hold the rows of `so`, the scan it ran."""
    names = ["_angle-0.05deg", "_angle0deg", "_angle0.05deg"]
    assert [output.angle_suffix(float(a)) for a in so.angles] == names
    radii = output.read_columns_csv(out / "angular_scan_telescope_y_radii.csv")
    assert list(radii) == output.RADII_COLUMNS and np.array_equal(radii["Angle [deg]"], so.angles)
    for i, sfx in enumerate(names):
        r = output.containment_radii_from_hist(*so.radial_hists[i])
        for f in output.RADII_COLUMNS[1:]:
            assert radii[f][i] == getattr(r, f)
        sp = output.read_columns_csv(out / f"axion_energy_spectrum_BabyIAXO{sfx}.csv")
        keep = np.isfinite(so.spectra[i].energies_keV)
        assert np.array_equal(sp["rays"].astype(np.uint64), so.spectra[i].counts[keep])
        assert np.array_equal(sp["flux"], so.spectra[i].sum_w[keep])
        sh = output.read_columns_csv(out / f"axion_shell_flux_BabyIAXO{sfx}.csv")
        assert np.array_equal(sh["rays"].astype(np.uint64), so.spectra[i].shell_counts)
        for b, (lo, hi) in enumerate(zip([0.5, 2, 4], [2, 4, 8])):
            img, cols = output.read_axion_image_csv(out / f"axion_image_BabyIAXO{output.band_suffix(lo, hi)}{sfx}.csv")
            assert np.array_equal(img, so.band_images[i].image[b])
            assert cols["yr0"][-1] == r.rSigma1W
        h = output.read_columns_csv(out / f"axion_hist_reflect_BabyIAXO{sfx}.csv")
        assert np.array_equal(h["rays"].astype(np.uint64), so.quantity_hists[i][0].counts)
        assert np.array_equal(h["flux"], so.quantity_hists[i][0].sum_w)
    rel = np.loadtxt(out / "angular_scan_telescope_y.csv", delimiter=",", skiprows=1)
    assert np.array_equal(rel[:, 0], so.angles) and np.allclose(rel[:, 1], so.fluxes / so.fluxes.max(), rtol=1e-15)


def _scan_files(out):
    return {p.name: output.read_columns_csv(p) for p in sorted(out.glob("*.csv")) if not p.name.startswith("axion_image")}


def test_command_line_writes_one_set_of_files_per_scan_point(rt, tmp_path, monkeypatch):
    seen = []
    orig = rt.RayTracer.angular_scan_outputs

    def wrapper(self, *a, **k):
        r = orig(self, *a, **k)
        seen.append(r)
        return r
    monkeypatch.setattr(rt.RayTracer, "angular_scan_outputs", wrapper)
    one = _cli(tmp_path, "one", ["--device", "0"])
    (so,) = seen
    _files_equal_scan(one, so)
    devs = _cli(tmp_path, "devs", ["--devices", "0"])
    (_, so_d) = seen
    _files_equal_scan(devs, so_d)
    a, b = _scan_files(one), _scan_files(devs)
    assert a.keys() == b.keys()
    for name in a:
        for col in a[name]:
            assert np.allclose(a[name][col], b[name][col], rtol=1e-12, atol=0, equal_nan=True), (name, col)
    if rt.lib.sart_device_count() < 2:
        pytest.skip("a scan split over GPUs needs two of them")
    two = _cli(tmp_path, "two", ["--devices", "0,1"])
    c = _scan_files(two)
    assert c.keys() == a.keys()
    for name in a:
        for col in a[name]:
            assert np.allclose(a[name][col], c[name][col], rtol=1e-12, atol=0, equal_nan=True), (name, col)
    assert len(seen) == 4   # one block of scan points per device
