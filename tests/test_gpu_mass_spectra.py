"""Energy spectrum and per-shell flux of every axion mass of a mass scan (sart_enable_mass_spectra /
sart_read_mass_spectra): per mass against single-mass runs of the same rays (mode 0, whose single-mass spectra
tests/test_gpu_spectra.py ties to the oracle), mode 2 against mode 0 (the FP64 re-trace included), the invariants against
the per-mass counters in every mode, the physics of the gas stage, the lifecycle and the command line."""
import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import abi, output

pytestmark = pytest.mark.gpu
SEED = 299792458
M_GAMMA = 0.008235101411623404   # m_gamma of the babyiaxo_gas setup: the resonance
MASSES = np.array([0.004, 0.008, M_GAMMA, 0.0085, 0.02])
FIELDS = ("sum_w", "sum_w2", "counts", "shell_sum_w", "shell_counts")
FLOATS = ("sum_w", "sum_w2", "sum_x", "sum_y", "sum_r")


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


def _run(tr, n, seed=SEED, first=0):
    tr.reset_image()
    tr.trace_mc(n, seed, first_ray=first)
    return tr.read_image(), tr.read_mass_spectra()


def _invariants(counters, spectra):
    assert len(counters) == len(spectra)
    for c, s in zip(counters, spectra):
        assert int(s.counts.sum()) == int(s.shell_counts.sum()) == c["n_passed"]
        assert s.sum_w.sum() == pytest.approx(c["sum_w"], rel=1e-12, abs=0)


def _same_counts(a, b, what=""):
    assert np.array_equal(a.counts, b.counts), (what, np.nonzero(a.counts != b.counts))
    assert np.array_equal(a.shell_counts, b.shell_counts), (what, a.shell_counts, b.shell_counts)


def _mean_energy(s):
    return float((s.energies_keV[:-1] * s.sum_w[:-1]).sum() / s.sum_w[:-1].sum())


@pytest.fixture(scope="module")
def gas_mode0(rt):
    """Mode 0 on 1e8 rays x MASSES of babyiaxo_gas: the reference the mode-2 tests compare to."""
    setup, tb = make_config("babyiaxo_gas")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_axion_masses(MASSES)
        tr.enable_mass_spectra()
        tr.set_precision(0)
        res, spec = _run(tr, 100_000_000)
    _invariants(res.counters, spec)
    return res, spec


def test_mode0_per_mass_equals_single_mass_runs(rt):
    """2e7 rays: slice m of the mass scan's spectra equals a single-mass run of m_k with sart_enable_spectra on the same
    rays: counts identical, Σw, Σw² and shell Σw per bin within 1e-12 (both compute the same per-ray weight; only the
    order of the atomic adds differs)."""
    setup, tb = make_config("babyiaxo_gas")
    n = 20_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(0)
        tr.set_axion_masses(MASSES)
        tr.enable_mass_spectra()
        res, scan = _run(tr, n)
        tr.enable_mass_spectra(False)
        single = []
        for m in MASSES:
            tr.set_axion_masses([m])
            tr.enable_spectra()
            tr.reset_image()
            tr.trace_mc(n, SEED)
            single.append((tr.read_image().counters[0], tr.read_spectra()))
            tr.enable_spectra(False)
    _invariants(res.counters, scan)
    for k, (c, s) in enumerate(single):
        assert res.counters[k]["n_passed"] == c["n_passed"] > 0
        _same_counts(scan[k], s, MASSES[k])
        for f in ("sum_w", "sum_w2", "shell_sum_w"):
            assert np.allclose(getattr(scan[k], f), getattr(s, f), rtol=1e-12, atol=0), (MASSES[k], f)
        assert np.array_equal(scan[k].energies_keV[:-1], s.energies_keV[:-1]) and np.isnan(scan[k].energies_keV[-1])


def test_mode2_equals_mode0_on_1e8_rays(rt, gas_mode0):
    """Every mass: counts identical bin by bin (exit codes and sampling agree ray by ray, the re-trace resolves the
    uncertain rays), no unresolved ray, Σw within 1e-3 in every bin with >= 1000 rays and in total within 2e-3, the
    per-mass flux tolerance of test_gpu_retrace.py: test_mass_scan_counters_equal_exact_on_1e8_rays."""
    r0, s0 = gas_mode0
    setup, tb = make_config("babyiaxo_gas")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_axion_masses(MASSES)
        tr.enable_mass_spectra()
        tr.set_precision(2)
        r2, s2 = _run(tr, 100_000_000)
    _invariants(r2.counters, s2)
    for k in range(MASSES.size):
        assert r2.counters[k]["n_unresolved"] == 0
        _same_counts(s2[k], s0[k], MASSES[k])
        big = s0[k].counts >= 1000
        assert big.sum() > 10
        rel = np.abs(s2[k].sum_w[big] / s0[k].sum_w[big] - 1.0)
        tot = abs(s2[k].sum_w.sum() / s0[k].sum_w.sum() - 1.0)
        print("mass", MASSES[k], "max per-bin Σw deviation from mode 0:", rel.max(), "total:", tot)
        assert rel.max() < 1e-3 and tot < 2e-3


def test_retrace_fills_the_mass_spectra(rt, gas_mode0):
    """Error budgets x 12, so that more than 1 % of the rays go through the exact list-mode kernel: the counts of every
    mass still equal mode 0's, which they could not if the re-traced rays missed the spectra."""
    r0, s0 = gas_mode0
    setup, tb = make_config("babyiaxo_gas")
    n = 100_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_axion_masses(MASSES)
        tr.enable_mass_spectra()
        tr.set_precision(2)
        tr.set_retrace(1, 12.0)
        r2, s2 = _run(tr, n)
    frac = r2.counters[0]["n_retraced"] / n
    print("re-traced fraction at budget scale 12:", frac)
    assert frac > 0.01
    _invariants(r2.counters, s2)
    for k in range(MASSES.size):
        assert r2.counters[k]["n_unresolved"] == 0
        _same_counts(s2[k], s0[k], MASSES[k])


@pytest.mark.parametrize("n_masses", [1, 5, 40])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_invariants_and_spectra_off_unchanged(rt, mode, n_masses):
    """Per mass: Σ energy counts == Σ shell counts == n_passed and Σ energy Σw == sum_w. With the spectra on and off the
    integer counters are identical and the images the same to 1e-10 per bin. M = 40 runs the two-masses-per-lane kernels
    of mode 2, M = 1 the mass-scan kernels at one mass (with the spectra off it runs the single-mass kernels)."""
    setup, tb = make_config("babyiaxo_gas")
    n = 3_000_000
    masses = MASSES if n_masses == 5 else (np.array([M_GAMMA]) if n_masses == 1 else np.linspace(0.002, 0.03, n_masses))
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        tr.set_axion_masses(masses)
        tr.enable_mass_spectra()
        on, spec = _run(tr, n, first=11)
        tr.enable_mass_spectra(False)
        tr.reset_image()
        tr.trace_mc(n, SEED, first_ray=11)
        off = tr.read_image()
    assert len(spec) == n_masses
    _invariants(on.counters, spec)
    for k in range(n_masses):
        a, b = on.counters[k], off.counters[k]
        assert a["n_passed"] > 0
        for f in a:
            # at M = 1 the spectra-off run takes the single-mass kernels, whose FP32 margin tests may queue other rays for
            # the exact re-trace than the mass-scan kernel's: how many were re-traced may differ, not what they gave
            if f not in FLOATS and not (n_masses == 1 and f == "n_retraced"):
                assert a[f] == b[f], (k, f, a[f], b[f])
        assert a["sum_w"] == pytest.approx(b["sum_w"], rel=1e-12)
    assert np.allclose(on.image, off.image, rtol=1e-10, atol=0)


@pytest.mark.parametrize("mode", [0, 2])
def test_off_resonance_spectrum_moves_to_high_energies(rt, mode):
    """Off the resonance the conversion probability grows with E^2 (q = |m_gamma^2 - m_a^2| / 2E), so the mean detected
    energy at m_a = 0.02 eV exceeds the one at m_a = m_gamma, where the spectrum follows the solar flux."""
    setup, tb = make_config("babyiaxo_gas")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        tr.set_axion_masses([M_GAMMA, 0.02])
        tr.enable_mass_spectra()
        _, (res, off) = _run(tr, 10_000_000)
    e_res, e_off = _mean_energy(res), _mean_energy(off)
    print(f"mode {mode}: mean detected energy {e_res:.4f} keV at m_gamma, {e_off:.4f} keV at 0.02 eV")
    assert e_off > e_res


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_vacuum_slices_are_identical(rt, mode):
    """In vacuum the conversion probability does not depend on the mass: every slice has the same counts and sums."""
    setup, tb = make_config("babyiaxo_xmm")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        tr.set_axion_masses([0.001, 0.01, 0.1])
        tr.enable_mass_spectra()
        res, spec = _run(tr, 3_000_000)
    _invariants(res.counters, spec)
    assert spec[0].counts.sum() > 0
    for s in spec[1:]:
        _same_counts(s, spec[0])
        for f in ("sum_w", "sum_w2", "shell_sum_w"):
            assert np.allclose(getattr(s, f), getattr(spec[0], f), rtol=1e-12, atol=0), f


def test_lifecycle(rt):
    """reset_image and a new number of masses clear the spectra; reading them while off raises; they refuse to be on
    together with the single-mass spectra (either way round) and to run with the alias sampler; angular_scan,
    traceAxionWrapper and trace_passed leave them as they were."""
    setup, tb = make_config("babyiaxo_xmm")
    n = 1_000_000
    zero = lambda spectra: all(not getattr(s, f).any() for s in spectra for f in FIELDS)   # noqa: E731
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        with pytest.raises(rt.SartError, match="no per-mass spectra"):
            tr.read_mass_spectra()
        tr.enable_mass_spectra()
        with pytest.raises(rt.SartError, match="per-mass spectra are on"):
            tr.enable_spectra()
        tr.enable_mass_spectra(False)
        tr.enable_spectra()
        with pytest.raises(rt.SartError, match="single-mass spectra are on"):
            tr.enable_mass_spectra()
        tr.enable_spectra(False)
        tr.enable_mass_spectra()
        tr.set_sampler(abi.SAMPLER_ALIAS)
        with pytest.raises(rt.SartError, match="inverse-CDF sampler"):
            tr.trace_mc(1000, SEED)
        tr.set_sampler(abi.SAMPLER_INVERSE_CDF)

        res, a = _run(tr, n)   # one mass: the mass-scan kernels at M = 1
        assert len(a) == 1 and a[0].counts.sum() > 0
        _invariants(res.counters, a)
        tr.angular_scan([0.0, 0.05], n, SEED)
        tr.traceAxionWrapper(10_000, SEED)
        tr.trace_passed(10_000, SEED)
        b = tr.read_mass_spectra()
        for f in FIELDS:
            assert np.array_equal(getattr(a[0], f), getattr(b[0], f)), f
        tr.reset_image()
        assert zero(tr.read_mass_spectra())

        tr.set_axion_masses([0.01, 0.02])
        tr.trace_mc(n, SEED)
        assert not zero(tr.read_mass_spectra())
        tr.set_axion_masses([0.03, 0.04])      # the same number of masses: the image and the spectra stay
        assert not zero(tr.read_mass_spectra())
        tr.set_axion_masses([0.01, 0.02, 0.03])   # another number: both are cleared
        assert len(tr.read_mass_spectra()) == 3 and zero(tr.read_mass_spectra())
        tr.enable_mass_spectra(False)
        with pytest.raises(rt.SartError, match="no per-mass spectra"):
            tr.read_mass_spectra()


def test_command_line_mass_scan_writes_the_spectra(rt, tmp_path, capsys):
    """A gas-stage mass scan with --writeSpectra writes one pair of CSV files per mass; per mass the `rays` columns add up
    to its passed count and the `flux` columns to its total flux. The images and stdout lines are those of a scan without."""
    from solaraxionraytracing_b200.__main__ import main
    from solaraxionraytracing_b200 import config
    masses = [0.006, 0.0082, 0.02]
    txt = config.DEFAULT_CONFIG.read_text().replace('outputPath = "../out"', f'outputPath = "{tmp_path}/out"')
    txt = txt.replace('stageSetup = "vacuum"', 'stageSetup = "gas"')
    txt += f'\n[Run]\nnRays = 300000\nseed = 3\nmAxion = {masses}\n'
    cfg = tmp_path / "config.toml"
    cfg.write_text(txt)
    assert main(["--config", str(cfg), "--allowSynthetic", "--writeSpectra"]) == 0
    out = capsys.readouterr().out
    lines = [line for line in out.splitlines() if line.startswith("m_a = ")]
    assert len(lines) == 3
    imgs = np.load(tmp_path / "out" / "axion_images_mass_scan.npy")
    for m, line in zip(masses, lines):
        passed = int(line.split("passed ")[1].split(",")[0])
        flux = float(line.split("total flux")[1])
        spec = output.read_columns_csv(tmp_path / "out" / f"axion_energy_spectrum_BabyIAXO_ma{m:.6g}eV.csv")
        shells = output.read_columns_csv(tmp_path / "out" / f"axion_shell_flux_BabyIAXO_ma{m:.6g}eV.csv")
        assert list(spec) == output.SPECTRUM_COLUMNS and list(shells) == output.SHELL_FLUX_COLUMNS
        assert passed > 0 and int(spec["rays"].sum()) == passed == int(shells["rays"].sum())
        assert spec["flux"].sum() == pytest.approx(flux, rel=1e-6)   # stdout prints 7 significant digits
        assert shells["flux"].sum() == pytest.approx(spec["flux"].sum(), rel=1e-12)
    assert len(list((tmp_path / "out").glob("axion_*_ma*eV.csv"))) == 6
    # the same scan without --writeSpectra: the same passed counts and fluxes and the same images (up to the order of the
    # sums), and no spectra files
    out_dir = tmp_path / "out"
    for p in out_dir.iterdir():
        p.unlink()
    assert main(["--config", str(cfg), "--allowSynthetic"]) == 0
    plain = [line for line in capsys.readouterr().out.splitlines() if line.startswith("m_a = ")]
    assert [x.split(",")[0] for x in plain] == [x.split(",")[0] for x in lines]
    assert np.allclose([float(x.split("total flux")[1]) for x in plain], [float(x.split("total flux")[1]) for x in lines],
                       rtol=1e-6, atol=0)
    assert np.allclose(np.load(out_dir / "axion_images_mass_scan.npy"), imgs, rtol=1e-10, atol=0)
    assert not list(out_dir.glob("axion_*_ma*eV.csv"))
