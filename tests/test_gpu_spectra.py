"""Energy spectrum and per-shell flux of the passed rays of a fused run (sart_enable_spectra / sart_read_spectra): the
reductions generateResultPlots (rt:2246-2635) makes over energiesAx, shellNumber and weights, against the oracle's
per-ray records (mode 0), against mode 0 (modes 1 and 2, the FP64 re-trace included), and against the per-ray records of
the same rays (mode 2)."""
import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import abi, output

pytestmark = pytest.mark.gpu
SEED = 299792458
BIG = dict(nR=1968, nE=1500, nAng=1000, nEn=1000)   # BASELINE-size tables


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


def _run(tr, n, seed=SEED, first=0):
    tr.reset_image()
    tr.trace_mc(n, seed, first_ray=first)
    res = tr.read_image()
    return res, tr.read_spectra()


def _invariants(c, s):
    assert int(s.counts.sum()) == int(s.shell_counts.sum()) == c["n_passed"]
    assert s.sum_w.sum() == pytest.approx(c["sum_w"], rel=1e-12)
    assert s.sum_w2.sum() == pytest.approx(c["sum_w2"], rel=1e-12)


def _same_counts(a, b):
    assert np.array_equal(a.counts, b.counts), np.nonzero(a.counts != b.counts)
    assert np.array_equal(a.shell_counts, b.shell_counts), (a.shell_counts, b.shell_counts)


def _records_spectra(rays, tb, setup):
    src = setup.testSource.energy if setup.testSource.active else None
    return output.spectra_from_records(rays.energy, rays.shell, rays.w, tb.energies, src, setup.telescope.nShells)


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_mode0_spectra_equal_the_oracle_records(rt, oracle, cfg):
    """2e6 rays: counts per energy and shell bin identical to the oracle's records. Σw per bin within 1e-6 over all rays,
    the per-ray weight agreement of Monte Carlo rays (test_gpu_parity.py: test_mc_rays_match_oracle): they are sampled
    with libm's sin / cos, which CUDA and glibc round differently for some arguments (DESIGN.md §3). Taking the rays whose
    exit code or weight (beyond 1e-10) that changes out of both sides by their records, Σw per bin agrees within 1e-10,
    mode 0's weight agreement on identical rays (measured: 0 such rays of CAST+LLNL, 1409 of BabyIAXO+XMM)."""
    setup, tb = make_config(cfg)
    n = 2_000_000
    ref = oracle.trace_mc_rays(setup, tb, 0, n, SEED)
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(0)
        tr.enable_spectra()
        res, s = _run(tr, n)
        gpu = tr.traceAxionWrapper(n, SEED)
    _invariants(res.counters[0], s)
    o = _records_spectra(ref, tb, setup)
    _same_counts(s, o)
    assert np.allclose(s.sum_w, o.sum_w, rtol=1e-6, atol=0)
    assert np.allclose(s.shell_sum_w, o.shell_sum_w, rtol=1e-6, atol=0)
    assert np.count_nonzero(gpu.code != ref.code) <= n // 5000
    odd = (gpu.code != ref.code) | (np.abs(gpu.w - ref.w) > 1e-10 * np.abs(ref.w))
    print(cfg, "rays with another exit code or weight than the oracle:", int(odd.sum()))
    if odd.any():   # take them out of both sides
        g_odd = output.spectra_from_records(gpu.energy[odd], gpu.shell[odd], gpu.w[odd], tb.energies, None, setup.telescope.nShells)
        o_odd = output.spectra_from_records(ref.energy[odd], ref.shell[odd], ref.w[odd], tb.energies, None, setup.telescope.nShells)
        for f in ("sum_w", "counts", "shell_sum_w", "shell_counts"):
            setattr(s, f, getattr(s, f) - getattr(g_odd, f))
            setattr(o, f, getattr(o, f) - getattr(o_odd, f))
    _same_counts(s, o)
    floor = 1e-15 * o.sum_w.sum()   # what the subtraction leaves of the rounding of a run's sums
    assert np.allclose(s.sum_w, o.sum_w, rtol=1e-10, atol=floor)
    assert np.allclose(s.shell_sum_w, o.shell_sum_w, rtol=1e-10, atol=floor)
    assert s.counts[-1] == 0 and np.isnan(s.energies_keV[-1])


@pytest.mark.parametrize("cfg,compact", [("cast_llnl", 0), ("babyiaxo_xmm", 0), ("babyiaxo_xmm", 1)])
def test_mode2_spectra_equal_mode0_on_1e9_rays(rt, cfg, compact):
    """1e9 rays, BASELINE-size tables: counts per bin identical to mode 0 (exit codes and sampling agree ray by ray),
    total Σw within 3e-4, Σw within 1e-3 in every bin with >= 1000 rays (measured on a B200: at most 7.3e-6 on CAST+LLNL,
    9.6e-7 on BabyIAXO+XMM); the counters identical with spectra on and off and the image the same to 1e-12."""
    setup, tb = make_config(cfg, **BIG)
    n = 1_000_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.enable_spectra()
        r0, s0 = _run(tr, n)
        tr.set_precision(2)
        tr.set_compaction(compact)
        r2, s2 = _run(tr, n)
        tr.enable_spectra(False)
        tr.reset_image()
        tr.trace_mc(n, SEED)
        off = tr.read_image()
        with pytest.raises(rt.SartError):
            tr.read_spectra()
    c0, c2 = r0.counters[0], r2.counters[0]
    _invariants(c0, s0)
    _invariants(c2, s2)
    assert c2["n_unresolved"] == 0
    _same_counts(s2, s0)
    assert abs(s2.sum_w.sum() / s0.sum_w.sum() - 1.0) < 3e-4
    big = s0.counts >= 1000
    assert big.sum() > 100
    rel = np.abs(s2.sum_w[big] / s0.sum_w[big] - 1.0)
    print(cfg, "compact", compact, "max per-bin Σw deviation from mode 0:", rel.max())
    assert rel.max() < 1e-3
    sh = s0.shell_counts >= 1000
    assert np.all(np.abs(s2.shell_sum_w[sh] / s0.shell_sum_w[sh] - 1.0) < 1e-3)
    co = off.counters[0]
    for k in c2:
        if k not in ("sum_w", "sum_w2", "sum_x", "sum_y", "sum_r"):
            assert c2[k] == co[k], k
    assert r2.image.sum() == pytest.approx(off.image.sum(), rel=1e-12)
    assert np.allclose(r2.image, off.image, rtol=1e-10, atol=0)   # per bin: only the order of the atomic adds differs
    assert c2["sum_w"] == pytest.approx(co["sum_w"], rel=1e-12)


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_retrace_fills_the_spectra(rt, cfg):
    """Error budgets scaled up 12x, so that percents of the rays go through the exact list-mode kernel: the counts still
    equal mode 0's, which they could not if the re-traced rays missed the spectra."""
    setup, tb = make_config(cfg, **BIG)
    n = 200_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.enable_spectra()
        r0, s0 = _run(tr, n, first=7)
        tr.set_precision(2)
        tr.set_retrace(1, 12.0)
        r2, s2 = _run(tr, n, first=7)
    c2 = r2.counters[0]
    frac = c2["n_retraced"] / n
    print(cfg, "re-traced fraction at budget scale 12:", frac)
    assert c2["n_unresolved"] == 0 and frac > 0.01
    _invariants(c2, s2)
    _same_counts(s2, s0)


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_mode2_spectra_equal_its_per_ray_records(rt, cfg):
    """5e6 rays in mode 2: the fused kernel's spectra against traceAxionWrapper's records of the same rays binned on the
    host — counts identical, Σw equal up to summation order (1e-12); mode 1 likewise."""
    setup, tb = make_config(cfg)
    n = 5_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.enable_spectra()
        for mode in (2, 1):
            tr.set_precision(mode)
            res, s = _run(tr, n)
            rays = tr.traceAxionWrapper(n, SEED)
            _invariants(res.counters[0], s)
            h = _records_spectra(rays, tb, setup)
            _same_counts(s, h)
            assert np.allclose(s.sum_w, h.sum_w, rtol=1e-12, atol=0), mode
            assert np.allclose(s.sum_w2, h.sum_w2, rtol=1e-12, atol=0), mode
            assert np.allclose(s.shell_sum_w, h.shell_sum_w, rtol=1e-12, atol=0), mode


def _other_setups():
    xs, xt = make_config("babyiaxo_xmm", flags=abi.CF_XRAY_TEST)
    xs.testSource.energy = 3.0
    gs, gt = make_config("babyiaxo_gas")
    ts, tt = make_config("cast_llnl")
    ts.telescope.telescope_turned_y = 0.08
    return {"xray": (xs, xt), "gas": (gs, gt), "turned": (ts, tt)}


@pytest.mark.parametrize("name", ["xray", "gas", "turned"])
def test_other_sources_and_setups(rt, name):
    """X-ray test source: every passed ray in bin nEnergies. Buffer gas (a generic-only stage) and a turned telescope:
    counts of mode 2 identical to mode 0 (mode 1: the invariants)."""
    setup, tb = _other_setups()[name]
    n = 20_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.enable_spectra()
        r0, s0 = _run(tr, n)
        _invariants(r0.counters[0], s0)
        for mode in (1, 2):
            tr.set_precision(mode)
            r, s = _run(tr, n)
            _invariants(r.counters[0], s)
            if mode == 2:   # exit codes of mode 0 ray by ray (re-trace); mode 1 has its own rounding
                _same_counts(s, s0)
            if name == "xray":
                assert s.counts[-1] == r.counters[0]["n_passed"] > 0 and s.energies_keV[-1] == 3.0
    if name == "xray":
        assert s0.counts[-1] == r0.counters[0]["n_passed"] > 0


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_alias_sampler_energy_spectrum(rt, cfg):
    """The alias sampler draws the same distributions as the inverse-CDF search: the two energy spectra agree in a
    two-sample chi^2 over the bins with enough rays."""
    setup, tb = make_config(cfg)
    n = 50_000_000
    h = {}
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.enable_spectra()
        for smp in (abi.SAMPLER_INVERSE_CDF, abi.SAMPLER_ALIAS):
            tr.set_sampler(smp)
            r, s = _run(tr, n, seed=99)
            _invariants(r.counters[0], s)
            h[smp] = s.counts.astype(np.float64)
    ha, hb = h[abi.SAMPLER_INVERSE_CDF], h[abi.SAMPLER_ALIAS]
    assert not np.array_equal(ha, hb)
    sel = (ha + hb) >= 50
    assert sel.sum() > 100
    sa, sb = ha[sel].sum(), hb[sel].sum()
    chi2 = (((ha[sel] / sa - hb[sel] / sb) ** 2) / (ha[sel] / sa ** 2 + hb[sel] / sb ** 2)).sum()
    ndf = int(sel.sum()) - 1
    assert abs(chi2 - ndf) / np.sqrt(2.0 * ndf) < 5.0, (chi2, ndf)


def test_lifecycle(rt):
    """reset_image clears the spectra; update_setup (its pilot launch) between enable and trace leaks nothing; reading
    after enable_spectra(False) raises; two masses refuse to run; angular_scan leaves the spectra as they were."""
    setup, tb = make_config("babyiaxo_xmm")
    n = 1_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        with pytest.raises(rt.SartError, match="no spectra"):
            tr.read_spectra()
        tr.enable_spectra()
        s = setup
        s.magnet.lengthColdbore += 1e-9      # a geometry change: sart_update_setup repeats the pilot launch
        tr.update_setup(s)
        tr.set_precision(2)
        tr.reset_image()
        tr.trace_mc(n, SEED)
        c = tr.read_image().counters[0]
        a = tr.read_spectra()
        _invariants(c, a)
        tr.angular_scan([0.0, 0.05], n, SEED)
        tr.traceAxionWrapper(10_000, SEED)
        tr.trace_passed(10_000, SEED)
        b = tr.read_spectra()
        for f in ("sum_w", "sum_w2", "counts", "shell_sum_w", "shell_counts"):
            assert np.array_equal(getattr(a, f), getattr(b, f)), f
        tr.reset_image()
        z = tr.read_spectra()
        assert z.counts.sum() == 0 and z.shell_counts.sum() == 0 and not z.sum_w.any()
        tr.set_axion_masses([0.01, 0.02])
        with pytest.raises(rt.SartError, match="single axion mass"):
            tr.trace_mc(1000, SEED)
        tr.set_axion_masses([setup.consts.mAxion])
        tr.trace_mc(1000, SEED)
        tr.enable_spectra(False)
        with pytest.raises(rt.SartError, match="no spectra"):
            tr.read_spectra()


def test_command_line_writes_the_spectra(rt, tmp_path, capsys):
    """--writeSpectra writes both CSV files next to the image; their `rays` columns add up to "Passed axions"."""
    from solaraxionraytracing_b200.__main__ import main
    from solaraxionraytracing_b200 import config
    cfg = tmp_path / "config.toml"
    cfg.write_text(config.DEFAULT_CONFIG.read_text().replace('outputPath = "../out"', f'outputPath = "{tmp_path}/out"'))
    assert main(["--config", str(cfg), "--nRays", "300000", "--allowSynthetic", "--writeSpectra"]) == 0
    out = capsys.readouterr().out
    passed = int(out.split("Passed axions ")[1].split()[0])
    spec = output.read_columns_csv(tmp_path / "out" / "axion_energy_spectrum_BabyIAXO.csv")
    shells = output.read_columns_csv(tmp_path / "out" / "axion_shell_flux_BabyIAXO.csv")
    assert list(spec) == output.SPECTRUM_COLUMNS and list(shells) == output.SHELL_FLUX_COLUMNS
    assert passed > 0 and int(spec["rays"].sum()) == passed == int(shells["rays"].sum())
    flux = float(out.split("The total flux arriving in the detector is: ")[1].split()[0])
    assert spec["flux"].sum() == pytest.approx(shells["flux"].sum(), rel=1e-12)
    assert 0 < flux <= spec["flux"].sum() * (1 + 1e-12)   # the image holds the passed rays that land in its bins
