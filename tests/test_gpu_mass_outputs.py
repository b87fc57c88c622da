"""Containment radii and energy-band images of every axion mass of a mass scan (sart_enable_mass_radial_hist /
sart_enable_mass_band_images): per mass against single-mass runs of the same rays (mode 0), mode 2 against mode 0 (the FP64
re-trace included), the invariants against the per-mass counters, spectra and images in every mode, the vacuum, the
lifecycle and refusals, the merge over GPUs and the command line."""
import numpy as np
import pytest
# before libsart loads NCCL at its first communicator (see test_gpu_accumulators.py)
import torch

from helpers import make_config
from solaraxionraytracing_b200 import abi, multi_gpu, output

pytestmark = pytest.mark.gpu
SEED = 299792458
M_GAMMA = 0.008235101411623404   # m_gamma of the babyiaxo_gas setup: the resonance
MASSES = np.array([0.004, 0.008, M_GAMMA, 0.0085, 0.02])
EDGES = [0.0, 1.5, 3.0, 6.0, 1000.0]   # four bands that cover every tabulated energy
FLOATS = ("sum_w", "sum_w2", "sum_x", "sum_y", "sum_r")
NBINS = 4096


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


def _enable(tr, spectra=False):
    tr.enable_mass_radial_hist(NBINS)
    tr.enable_mass_band_images(EDGES)
    if spectra:
        tr.enable_mass_spectra()


def _run(tr, n, seed=SEED, first=0):
    tr.reset_image()
    tr.trace_mc(n, seed, first_ray=first)
    return tr.read_image(), tr.read_mass_radial_hist(), tr.read_mass_band_images()


def _radial_invariants(counters, rad):
    assert len(counters) == len(rad)
    for c, (_, w, n) in zip(counters, rad):
        assert int(n.sum()) == c["n_passed"]
        assert w.sum() == pytest.approx(c["sum_w"], rel=1e-12, abs=0)


def _radii_bins(a, b, binw):
    """The largest difference of the four containment radii of two radial histograms, in bins."""
    ra, rb = output.containment_radii_from_hist(*a), output.containment_radii_from_hist(*b)
    return max(abs(getattr(ra, f) - getattr(rb, f)) for f in ("rSigma1", "rSigma2", "rSigma1W", "rSigma2W")) / binw


@pytest.fixture(scope="module")
def gas_mode0(rt):
    """Mode 0 on 1e8 rays x MASSES of babyiaxo_gas: the reference the mode-2 tests compare to."""
    setup, tb = make_config("babyiaxo_gas")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_axion_masses(MASSES)
        _enable(tr)
        tr.set_precision(0)
        out = _run(tr, 100_000_000)
    _radial_invariants(out[0].counters, out[1])
    return out


def test_mode0_rows_equal_single_mass_runs(rt):
    """2e7 rays: row m of the per-mass radial histograms and band images equals a single-mass run of masses[m] with the
    radial histogram and the band images on, over the same rays: every count identical, Σw and Σw² per bin and pixel
    within 1e-12 (the same per-ray weights; only the order of the atomic adds differs)."""
    setup, tb = make_config("babyiaxo_gas")
    n = 20_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(0)
        tr.set_axion_masses(MASSES)
        _enable(tr)
        res, rad, bands = _run(tr, n)
        tr.enable_mass_radial_hist(0)
        tr.enable_mass_band_images(None)
        single = []
        for m in MASSES:
            tr.set_axion_masses([m])
            tr.enable_radial_hist(NBINS)
            tr.enable_band_images(EDGES)
            tr.reset_image()
            tr.trace_mc(n, SEED)
            single.append((tr.read_image().counters[0], tr.read_radial_hist(), tr.read_band_images()))
    _radial_invariants(res.counters, rad)
    for k, (c, r1, b1) in enumerate(single):
        assert res.counters[k]["n_passed"] == c["n_passed"] > 0
        assert np.array_equal(rad[k][0], r1[0])
        assert np.array_equal(rad[k][2], r1[2]), MASSES[k]
        assert np.allclose(rad[k][1], r1[1], rtol=1e-12, atol=0), MASSES[k]
        assert np.array_equal(bands[k].counts, b1.counts), (MASSES[k], bands[k].counts, b1.counts)
        assert np.array_equal(bands[k].edges, b1.edges)
        assert np.allclose(bands[k].image, b1.image, rtol=1e-12, atol=0), MASSES[k]
        assert np.allclose(bands[k].image_w2, b1.image_w2, rtol=1e-12, atol=0), MASSES[k]


def test_mode2_equals_mode0_on_1e8_rays(rt, gas_mode0):
    """Every mass: no unresolved ray, band counts identical, Σ radial counts = n_passed = mode 0's, each band plane within
    the mode-2 image tolerance of test_gpu_band_images.py (summed per-pixel deviation below 2e-2 of the plane's Σw), Σw per
    band within 3e-4 and the containment radii within two bins of mode 0's."""
    r0, rad0, b0 = gas_mode0
    setup, tb = make_config("babyiaxo_gas")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_axion_masses(MASSES)
        _enable(tr)
        tr.set_precision(2)
        r2, rad2, b2 = _run(tr, 100_000_000)
    _radial_invariants(r2.counters, rad2)
    binw = rad0[0][0][1] - rad0[0][0][0]
    for k in range(MASSES.size):
        assert r2.counters[k]["n_unresolved"] == 0
        assert r2.counters[k]["n_passed"] == r0.counters[k]["n_passed"]
        assert np.array_equal(b2[k].counts, b0[k].counts), (MASSES[k], b2[k].counts, b0[k].counts)
        for j in range(len(EDGES) - 1):
            tot = b0[k].image[j].sum()
            if b0[k].counts[j] < 1000:
                continue
            l1 = np.abs(b2[k].image[j] - b0[k].image[j]).sum() / tot
            dev = abs(b2[k].image[j].sum() / tot - 1.0)
            print(f"mass {MASSES[k]:.6g} band {j}: per-pixel L1 {l1:.3e}, Σw {dev:.3e}")
            assert l1 < 2e-2 and dev < 3e-4
        d = _radii_bins(rad2[k], rad0[k], binw)
        print(f"mass {MASSES[k]:.6g}: containment radii within {d:.3f} bins of mode 0")
        assert d <= 2.0


def test_retrace_fills_the_rows(rt, gas_mode0):
    """Error budgets x 12, so that more than 1 % of the rays go through the exact list-mode kernel: the band counts and
    the radial totals of every mass still equal mode 0's, which they could not if the re-traced rays missed the rows."""
    r0, rad0, b0 = gas_mode0
    setup, tb = make_config("babyiaxo_gas")
    n = 100_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_axion_masses(MASSES)
        _enable(tr)
        tr.set_precision(2)
        tr.set_retrace(1, 12.0)
        r2, rad2, b2 = _run(tr, n)
    frac = r2.counters[0]["n_retraced"] / n
    print("re-traced fraction at budget scale 12:", frac)
    assert frac > 0.01
    _radial_invariants(r2.counters, rad2)
    for k in range(MASSES.size):
        assert r2.counters[k]["n_unresolved"] == 0
        assert np.array_equal(b2[k].counts, b0[k].counts), MASSES[k]
        assert int(rad2[k][2].sum()) == int(rad0[k][2].sum())


def _band_of_energy_bins(spectra):
    """The band of every energy bin of a Spectra (the record energy max(0.03 keV, E); -1 for none)."""
    e = np.maximum(0.03, spectra.energies_keV[:-1])
    return np.searchsorted(np.asarray(EDGES), e, side="right") - 1


@pytest.mark.parametrize("n_masses", [1, 5, 40])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_invariants_and_off_unchanged(rt, mode, n_masses):
    """Per mass, with the per-mass spectra on as well: radial Σcounts = n_passed and ΣΣw = sum_w; each band's count is the
    spectra's counts summed over its energy bins; the bands cover every energy, so their planes add up to the mass's image.
    With the three accumulators on and off the integer counters are identical and the images the same to 1e-10. M = 40 runs
    the two-masses-per-lane kernels of mode 2, M = 1 the mass-scan kernels at one mass (off: the single-mass kernels)."""
    setup, tb = make_config("babyiaxo_gas")
    n = 3_000_000
    masses = MASSES if n_masses == 5 else (np.array([M_GAMMA]) if n_masses == 1 else np.linspace(0.002, 0.03, n_masses))
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        tr.set_axion_masses(masses)
        _enable(tr, spectra=True)
        on, rad, bands = _run(tr, n, first=11)
        spec = tr.read_mass_spectra()
        tr.enable_mass_radial_hist(0)
        tr.enable_mass_band_images(None)
        tr.enable_mass_spectra(False)
        tr.reset_image()
        tr.trace_mc(n, SEED, first_ray=11)
        off = tr.read_image()
    assert len(rad) == len(bands) == n_masses
    _radial_invariants(on.counters, rad)
    band = _band_of_energy_bins(spec[0])
    for k in range(n_masses):
        assert on.counters[k]["n_passed"] > 0
        want = [int(spec[k].counts[:-1][band == j].sum()) for j in range(len(EDGES) - 1)]
        assert bands[k].counts.tolist() == want, (k, bands[k].counts, want)
        assert int(bands[k].counts.sum()) == on.counters[k]["n_passed"]
        assert np.allclose(bands[k].image.sum(axis=0), on.image[k], rtol=1e-10, atol=1e-300)
        a, b = on.counters[k], off.counters[k]
        for f in a:
            if f not in FLOATS and not (n_masses == 1 and f == "n_retraced"):
                assert a[f] == b[f], (k, f, a[f], b[f])
        assert a["sum_w"] == pytest.approx(b["sum_w"], rel=1e-12)
    assert np.allclose(on.image, off.image, rtol=1e-10, atol=0)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_vacuum_rows_are_identical(rt, mode):
    """In vacuum the conversion probability does not depend on the mass: every row has the same counts and sums."""
    setup, tb = make_config("babyiaxo_xmm")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        tr.set_axion_masses([0.001, 0.01, 0.1])
        _enable(tr)
        res, rad, bands = _run(tr, 3_000_000)
    _radial_invariants(res.counters, rad)
    assert bands[0].counts.sum() > 0
    for r, b in zip(rad[1:], bands[1:]):
        assert np.array_equal(r[2], rad[0][2]) and np.array_equal(b.counts, bands[0].counts)
        assert np.allclose(r[1], rad[0][1], rtol=1e-12, atol=0)
        assert np.allclose(b.image, bands[0].image, rtol=1e-12, atol=0)
        assert np.allclose(b.image_w2, bands[0].image_w2, rtol=1e-12, atol=0)


def _arrays(tr, merged=False, kinds=("radial", "bands", "spectra")):
    """Every array of the per-mass radial histograms, band images and spectra (own or merged copy), as bytes."""
    out = {}
    if "radial" in kinds:
        rad = (tr.read_merged_mass_radial_hist if merged else tr.read_mass_radial_hist)()
        out["radial"] = [a.tobytes() for r in rad for a in r[1:]]
    if "bands" in kinds:
        bands = (tr.read_merged_mass_band_images if merged else tr.read_mass_band_images)()
        out["bands"] = [a.tobytes() for b in bands for a in (b.image, b.image_w2, b.counts)]
    if "spectra" in kinds:
        spec = (tr.read_merged_mass_spectra if merged else tr.read_mass_spectra)()
        out["spectra"] = [getattr(s, f).tobytes() for s in spec for f in ("sum_w", "sum_w2", "counts", "shell_sum_w")]
    return out


def _zero(arrays):
    return not any(np.frombuffer(b, dtype=np.uint8).any() for v in arrays.values() for b in v)


def test_lifecycle_and_refusals(rt):
    """Exclusion from the single-mass counterparts (either order) and the argument checks; the alias sampler, the quantity
    histograms, the single-mass spectra (in either order) and angular_scan_outputs are refused; angular_scan,
    traceAxionWrapper and trace_passed leave the rows alone; the merged copy of one handle is its own rows; switching one accumulator leaves the others and their merged copies
    bit-identical; reset_image clears the rows; a new number of masses clears them and invalidates their merged copies."""
    setup, tb = make_config("babyiaxo_gas")
    n = 1_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        with pytest.raises(rt.SartError, match="no per-mass radial"):
            tr.read_mass_radial_hist()
        with pytest.raises(rt.SartError, match="no per-mass band images"):
            tr.read_mass_band_images()
        tr.enable_mass_radial_hist(NBINS)
        with pytest.raises(rt.SartError, match="per-mass radial histograms are on"):
            tr.enable_radial_hist(NBINS)
        tr.enable_mass_radial_hist(0)
        tr.enable_radial_hist(NBINS)
        with pytest.raises(rt.SartError, match="single-mass radial histogram is on"):
            tr.enable_mass_radial_hist(NBINS)
        tr.enable_radial_hist(0)
        tr.enable_mass_band_images(EDGES)
        with pytest.raises(rt.SartError, match="per-mass band images are on"):
            tr.enable_band_images(EDGES)
        tr.enable_mass_band_images(None)
        tr.enable_band_images(EDGES)
        with pytest.raises(rt.SartError, match="single-mass band images are on"):
            tr.enable_mass_band_images(EDGES)
        tr.enable_band_images(None)
        for bad in ([1.0], [2.0, 1.0], [-1.0, 1.0], list(np.linspace(1, 2, abi.MAX_BANDS + 2))):
            with pytest.raises(rt.SartError, match="sart_enable_mass_band_images"):
                tr.enable_mass_band_images(bad)
        with pytest.raises(rt.SartError, match="bad argument"):
            tr.enable_mass_radial_hist(-1)

        _enable(tr)
        tr.set_sampler(abi.SAMPLER_ALIAS)
        with pytest.raises(rt.SartError, match="inverse-CDF sampler"):
            tr.trace_mc(1000, SEED)
        tr.set_sampler(abi.SAMPLER_INVERSE_CDF)
        tr.enable_quantity_hists([("reflect", 16, 0.0, 1.0)])
        with pytest.raises(rt.SartError, match="quantity histograms"):
            tr.trace_mc(1000, SEED)
        tr.enable_quantity_hists(None)
        # the single-mass spectra: the mass-scan kernels would leave them empty, so the run is refused (either order)
        tr.enable_spectra()
        with pytest.raises(rt.SartError, match="spectra need a single axion mass and the per-mass radial"):
            tr.trace_mc(1000, SEED)
        tr.enable_mass_radial_hist(0)
        tr.enable_mass_band_images(None)
        tr.reset_image()
        tr.trace_mc(1000, SEED)   # the spectra alone run
        assert tr.read_spectra().counts.sum() > 0
        tr.enable_mass_band_images(EDGES)
        with pytest.raises(rt.SartError, match="spectra need a single axion mass and the per-mass radial"):
            tr.trace_mc(1000, SEED)
        tr.enable_spectra(False)
        tr.enable_mass_radial_hist(NBINS)
        with pytest.raises(rt.SartError, match="per-mass radial histograms or band images are on"):
            tr.angular_scan_outputs([0.0], 1000, SEED)
        tr.enable_mass_spectra()

        _run(tr, n)   # one mass: the mass-scan kernels at M = 1
        multi_gpu.comm_init_all([tr])
        multi_gpu.allreduce_outputs([tr])
        own, merged = _arrays(tr), _arrays(tr, merged=True)
        assert own == merged and not _zero(own)   # one rank: the merged copy is the handle's own rows
        tr.angular_scan([0.0, 0.05], n, SEED)
        tr.traceAxionWrapper(10_000, SEED)
        tr.trace_passed(10_000, SEED)
        assert _arrays(tr) == own
        tr.enable_mass_radial_hist(NBINS)    # on again: cleared, everything else as it was
        assert _zero(_arrays(tr, kinds=("radial",)))
        assert _arrays(tr, kinds=("bands", "spectra")) == {k: own[k] for k in ("bands", "spectra")}
        assert _arrays(tr, True, ("bands", "spectra")) == {k: merged[k] for k in ("bands", "spectra")}
        with pytest.raises(rt.SartError, match="no merged per-mass radial"):
            tr.read_merged_mass_radial_hist()
        tr.enable_mass_band_images(EDGES[:3])
        assert _arrays(tr, kinds=("spectra",)) == {"spectra": own["spectra"]}
        assert _arrays(tr, True, ("spectra",)) == {"spectra": merged["spectra"]}

        tr.trace_mc(n, SEED)
        tr.reset_image()
        assert _zero(_arrays(tr))
        tr.set_axion_masses(MASSES[:2])
        tr.trace_mc(n, SEED)
        multi_gpu.allreduce_outputs([tr])
        tr.set_axion_masses(MASSES[2:4])      # the same number of masses: the rows and their merged copies stay
        assert not _zero(_arrays(tr, kinds=("bands",)))
        assert len(tr.read_merged_mass_band_images()) == 2
        tr.set_axion_masses(MASSES[:3])       # another number: cleared, the merged copies invalid
        assert len(tr.read_mass_band_images()) == 3 and len(tr.read_mass_radial_hist()) == 3
        assert _zero(_arrays(tr))
        with pytest.raises(rt.SartError, match="no merged per-mass band images"):
            tr.read_merged_mass_band_images()
        with pytest.raises(rt.SartError, match="no merged per-mass radial"):
            tr.read_merged_mass_radial_hist()


def test_create_and_destroy_returns_device_memory(rt):
    """20 handles, each with the per-mass radial histograms and band images on, traced, merged and destroyed: the device's
    free memory comes back to within 1 MiB. Measured after one such cycle, which loads the kernels and NCCL."""
    setup, tb = make_config("babyiaxo_gas")
    fs = rt.FullRaytraceSetup(setup, tb)

    def cycle():
        tr = rt.RayTracer(fs, 0)
        try:
            tr.set_precision(2)
            tr.set_axion_masses(MASSES)
            tr.enable_mass_radial_hist(NBINS)
            tr.enable_mass_band_images(EDGES[:2])
            tr.trace_mc(2_000_000, SEED)
            multi_gpu.comm_init_all([tr])
            multi_gpu.allreduce_outputs([tr])
            tr.read_merged_mass_band_images()
        finally:
            tr.close()

    cycle()
    torch.cuda.synchronize(0)
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(20):
        cycle()
    torch.cuda.synchronize(0)
    free1 = torch.cuda.mem_get_info(0)[0]
    assert abs(free1 - free0) <= 1 << 20, (free0, free1)


def test_merge_on_two_gpus(rt):
    """trace_on_devices over two GPUs equals one GPU tracing the same global rays (counts identical, sums within 1e-12);
    different band edges on the two ranks fail with SART_ERR_CONFIG."""
    if rt.lib.sart_device_count() < 2:
        pytest.skip("needs two GPUs")
    setup, tb = make_config("babyiaxo_gas")
    fs = rt.FullRaytraceSetup(setup, tb)
    n = 10_000_000
    with rt.RayTracer(fs, 0) as one:
        one.set_precision(2)
        one.set_axion_masses(MASSES)
        one.enable_mass_radial_hist()   # the default bins, as trace_on_devices
        one.enable_mass_band_images(EDGES)
        _, rad, bands = _run(one, n)
    r = multi_gpu.trace_on_devices(fs, [0, 1], n, SEED, precision=2, masses=MASSES, mass_radial_hist=True, mass_bands=EDGES)
    for k in range(MASSES.size):
        assert np.array_equal(r.mass_radial_hists[k][2], rad[k][2])
        assert np.allclose(r.mass_radial_hists[k][1], rad[k][1], rtol=1e-12, atol=1e-15 * rad[k][1].sum())
        assert np.array_equal(r.mass_band_images[k].counts, bands[k].counts)
        assert np.allclose(r.mass_band_images[k].image, bands[k].image, rtol=1e-12, atol=1e-15 * bands[k].image.sum())
    a, b = rt.RayTracer(fs, 0), rt.RayTracer(fs, 1)
    try:
        for t in (a, b):
            t.set_axion_masses(MASSES)
        a.enable_mass_band_images(EDGES)
        b.enable_mass_band_images(EDGES[:3])
        multi_gpu.comm_init_all([a, b])
        with pytest.raises(rt.SartError, match="band"):
            multi_gpu.allreduce_outputs([a, b])
    finally:
        a.close()
        b.close()


def _cli_config(tmp_path, masses, n=300_000):
    from solaraxionraytracing_b200 import config
    txt = config.DEFAULT_CONFIG.read_text().replace('outputPath = "../out"', f'outputPath = "{tmp_path}/out"')
    txt = txt.replace('stageSetup = "vacuum"', 'stageSetup = "gas"')
    txt += f'\n[Run]\nnRays = {n}\nseed = 3\nmAxion = {list(masses)}\n'
    cfg = tmp_path / "config.toml"
    cfg.write_text(txt)
    return cfg


def _direct_run(rt, cfg, masses, n, bands):
    """What the command line traces, run through RayTracer: the same setup, tables, precision, rays and accumulators."""
    from solaraxionraytracing_b200 import __main__ as cli, config as cfgmod, tables
    setup, res = cfgmod.setup_from_config(str(cfg), 0)
    tb = cli.load_tables(rt, tables, res, setup, 0, True)
    run = cfgmod.parseRun(cfgmod.load_config(str(cfg)))
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb), 0) as tr:
        rt.set_fastest_precision(tr, {"exact": 0, "fast": 1, "f32": 2}[run.precision], None)
        tr.set_axion_masses(masses)
        tr.enable_mass_radial_hist()
        tr.enable_mass_band_images(bands)
        tr.reset_image()
        tr.trace_mc(n, 3)
        return tr.read_mass_radial_hist(), tr.read_mass_band_images()


@pytest.mark.parametrize("devices", [None, "0"])
def test_command_line_writes_radii_and_band_images(rt, tmp_path, devices):
    """--massScanBands on a small gas-stage mass scan (one GPU, and through --devices): mass_scan_radii.csv and one band
    image CSV per band and mass, with the values of a direct RayTracer run and that mass's radii in the radius columns."""
    from solaraxionraytracing_b200.__main__ import main
    masses = [0.006, 0.0082, 0.02]
    bands = [0.5, 2.0, 4.0, 8.0]
    n = 300_000
    cfg = _cli_config(tmp_path, masses, n)
    extra = ["--devices", devices] if devices else []
    assert main(["--config", str(cfg), "--allowSynthetic", "--massScanBands", "0.5,2,4,8", *extra]) == 0
    out = tmp_path / "out"
    rad, bimg = _direct_run(rt, cfg, masses, n, bands)
    radii = output.read_columns_csv(out / "mass_scan_radii.csv")
    assert list(radii) == [output.MASS_COLUMN] + output.RADII_COLUMNS[1:]
    assert np.array_equal(radii[output.MASS_COLUMN], masses)
    for k, m in enumerate(masses):
        want = output.containment_radii_from_hist(*rad[k])
        for f in output.RADII_COLUMNS[1:]:
            assert radii[f][k] == pytest.approx(getattr(want, f), rel=1e-9, abs=1e-12), (m, f)
        for j, (lo, hi) in enumerate(zip(bands, bands[1:])):
            img, cols = output.read_axion_image_csv(out / f"axion_image_BabyIAXO{output.band_suffix(lo, hi)}"
                                                          f"{output.mass_suffix(m)}.csv")
            assert np.allclose(img, bimg[k].image[j], rtol=1e-9, atol=1e-300), (m, j)
            assert np.nanmax(cols["yr0"]) == pytest.approx(want.rSigma1W, rel=1e-9, abs=1e-12)
    assert len(list(out.glob("axion_image_*_ma*eV.csv"))) == 3 * 3


def test_command_line_file_lists(rt, tmp_path):
    """A mass scan with --writeSpectra writes the files it wrote before the new switches existed; --massScanRadii adds
    mass_scan_radii.csv and nothing else."""
    from solaraxionraytracing_b200.__main__ import main
    masses = [0.006, 0.0082, 0.02]
    cfg = _cli_config(tmp_path, masses, 100_000)
    out = tmp_path / "out"
    assert main(["--config", str(cfg), "--allowSynthetic", "--writeSpectra"]) == 0
    spectra_files = sorted(p.name for p in out.iterdir())
    want = ["axion_images_mass_scan.npy"] + [f"axion_{kind}_BabyIAXO{output.mass_suffix(m)}.csv"
                                             for kind in ("energy_spectrum", "shell_flux") for m in masses]
    assert spectra_files == sorted(want)
    for p in out.iterdir():
        p.unlink()
    assert main(["--config", str(cfg), "--allowSynthetic", "--massScanRadii"]) == 0
    assert sorted(p.name for p in out.iterdir()) == ["axion_images_mass_scan.npy", "mass_scan_radii.csv"]
