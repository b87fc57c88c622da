"""Detector images per energy band of the passed rays of a fused run (sart_enable_band_images / sart_read_band_images):
against the oracle's per-ray records binned by band (mode 0), against the run's own image, counters and spectra (modes 0,
1 and 2), against mode 0 on 1e9 rays (mode 2, the FP64 re-trace included), against the per-ray records of the same rays
(mode 2), for the X-ray source, next to the other accumulators, their lifecycle, several GPUs and the command line."""
import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import abi, output

pytestmark = pytest.mark.gpu
SEED = 299792458
BIG = dict(nR=1968, nE=1500, nAng=1000, nEn=1000)   # BASELINE-size tables
PLANE = abi.IMAGE_BINS * abi.IMAGE_BINS
EDGES3 = [0.5, 2.0, 4.0, 8.0]          # three bands with gaps below 0.5 keV and above 8 keV
ALL = [0.0, 2.0, 4.0, 1e6]             # three bands covering every energy


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


def _run(tr, n, seed=SEED, first=0):
    tr.reset_image()
    tr.trace_mc(n, seed, first_ray=first)
    return tr.read_image(), tr.read_band_images()


def _records_bands(x, y, w, energy, edges, chip=14.0, f32=False):
    """Band images of per-ray records binned on the host: rays with w != 0, band of the record's energy, the image bin of
    prepareHeatmap (rt:839-842) — with `f32` the bin as the FP32 kernels form it, from the position times the FP32 bin scale
    (trace_f32.cuh), so that rays next to a pixel edge land where the fused kernel put them."""
    x, y, w, e = (np.asarray(a, dtype=np.float64) for a in (x, y, w, energy))
    sel = w != 0.0
    x, y, w, e = x[sel], y[sel], w[sel], e[sel]
    edges = np.asarray(edges, dtype=np.float64)
    nb = edges.size - 1
    band = np.searchsorted(edges, e, side="right") - 1
    inb = (band >= 0) & (band < nb)
    if f32:
        inv = np.float32(abi.IMAGE_BINS / chip)
        cx, cy = (np.floor(a.astype(np.float32) * inv).astype(np.float64) for a in (x, y))
    else:
        step = chip / abi.IMAGE_BINS
        cx, cy = np.floor(x / step), np.floor(y / step)
    onchip = (cx >= 0) & (cx < abi.IMAGE_BINS) & (cy >= 0) & (cy < abi.IMAGE_BINS)
    counts = np.bincount(band[inb], minlength=nb).astype(np.uint64)
    k = inb & onchip
    flat = band[k] * PLANE + cy[k].astype(np.int64) * abi.IMAGE_BINS + cx[k].astype(np.int64)
    img = np.bincount(flat, weights=w[k], minlength=nb * PLANE).reshape(nb, abi.IMAGE_BINS, abi.IMAGE_BINS)
    return counts, img


def _cover_everything(res, b):
    """Bands covering every energy: the planes add up to the image, the counts to n_passed."""
    c = res.counters[0]
    assert int(b.counts.sum()) == c["n_passed"]
    floor = 1e-15 * res.image[0].sum()
    assert np.allclose(b.image.sum(axis=0), res.image[0], rtol=1e-12, atol=floor)
    assert np.allclose(b.image_w2.sum(axis=0), res.image_w2[0], rtol=1e-12, atol=1e-15 * res.image_w2[0].sum())


def _band_counts_from_spectra(s, edges):
    e = np.maximum(s.energies_keV[:-1], 0.03)
    out = []
    for lo, hi in zip(edges, edges[1:]):
        out.append(int(s.counts[:-1][(e >= lo) & (e < hi)].sum()))
    return np.array(out, dtype=np.uint64)


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_mode0_band_images_equal_the_oracle_records(rt, oracle, cfg):
    """2e6 rays, three bands: counts per band and Σw per band and pixel equal the oracle's records binned by band, after the
    rays whose exit code or weight differs because of libm's sin / cos are taken out of both sides (as in
    test_gpu_spectra.py: test_mode0_spectra_equal_the_oracle_records)."""
    setup, tb = make_config(cfg)
    n = 2_000_000
    ref = oracle.trace_mc_rays(setup, tb, 0, n, SEED)
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(0)
        tr.enable_band_images(EDGES3)
        res, b = _run(tr, n)
        gpu = tr.traceAxionWrapper(n, SEED)
    assert np.count_nonzero(gpu.code != ref.code) <= n // 5000
    odd = (gpu.code != ref.code) | (np.abs(gpu.w - ref.w) > 1e-10 * np.abs(ref.w))
    keep = ~odd
    g_n, g_img = _records_bands(gpu.x[odd], gpu.y[odd], gpu.w[odd], gpu.energy[odd], EDGES3)
    o_n, o_img = _records_bands(ref.x[keep], ref.y[keep], ref.w[keep], ref.energy[keep], EDGES3)
    counts = b.counts - g_n
    img = b.image - g_img
    assert np.array_equal(counts, o_n), (counts, o_n)
    floor = 1e-15 * o_img.sum()
    assert np.allclose(img, o_img, rtol=1e-10, atol=floor)
    assert counts.sum() > 0


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_band_images_against_image_counters_and_spectra(rt, cfg):
    """Modes 0, 1, 2: bands covering every energy add up to the image and to n_passed; bands with gaps, with the spectra
    on, count exactly the spectra's rays of the energy bins inside them."""
    setup, tb = make_config(cfg)
    n = 20_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        for mode in (0, 1, 2):
            tr.set_precision(mode)
            tr.enable_spectra(False)
            tr.enable_band_images(ALL)
            res, b = _run(tr, n)
            _cover_everything(res, b)
            tr.enable_spectra()
            tr.enable_band_images(EDGES3)
            res, b = _run(tr, n)
            s = tr.read_spectra()
            assert np.array_equal(b.counts, _band_counts_from_spectra(s, EDGES3)), mode
            assert int(b.counts.sum()) < res.counters[0]["n_passed"]


def _mode2_vs_mode0(rt, cfg, n, compact=None, scale=None, first=0):
    setup, tb = make_config(cfg, **BIG)
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.enable_band_images(EDGES3)
        r0, b0 = _run(tr, n, first=first)
        tr.set_precision(2)
        if compact is not None:
            tr.set_compaction(compact)
        if scale is not None:
            tr.set_retrace(1, scale)
        r2, b2 = _run(tr, n, first=first)
    c2 = r2.counters[0]
    assert c2["n_unresolved"] == 0
    assert np.array_equal(b2.counts, b0.counts), (b2.counts, b0.counts)
    assert b2.image.sum() == pytest.approx(b0.image.sum(), rel=3e-4)
    return c2, b0, b2


@pytest.mark.parametrize("cfg,compact", [("cast_llnl", 0), ("babyiaxo_xmm", 0), ("babyiaxo_xmm", 1)])
def test_mode2_band_images_equal_mode0_on_1e9_rays(rt, cfg, compact):
    """1e9 rays, BASELINE-size tables: counts per band identical to mode 0, Σw per band within 3e-4, and each plane within
    the tolerance of the mode-2 image against mode 0 (test_gpu_f32.py, test_gpu_fast.py): the summed absolute difference per
    pixel below 2e-2 of the plane's Σw — FP32 positions move the rays next to a pixel edge into the neighbouring pixel."""
    _, b0, b2 = _mode2_vs_mode0(rt, cfg, 1_000_000_000, compact=compact)
    for k in range(b0.counts.size):
        assert abs(b2.image[k].sum() / b0.image[k].sum() - 1.0) < 3e-4
        l1 = np.abs(b2.image[k] - b0.image[k]).sum() / b0.image[k].sum()
        print(cfg, "compact", compact, "band", k, "summed per-pixel deviation from mode 0:", l1)
        assert l1 < 2e-2


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_retrace_fills_the_band_images(rt, cfg):
    """Error budgets scaled up 12x, so that percents of the rays go through the exact list-mode kernel: the counts still
    equal mode 0's."""
    c2, _, _ = _mode2_vs_mode0(rt, cfg, 200_000_000, scale=12.0, first=7)
    assert c2["n_retraced"] / 200_000_000 > 0.01


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_mode2_band_images_equal_its_per_ray_records(rt, cfg):
    """5e6 rays in mode 2: the band images against traceAxionWrapper's records of the same rays binned on the host — counts
    identical, Σw per pixel equal up to summation order."""
    setup, tb = make_config(cfg)
    n = 5_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.enable_band_images(EDGES3)
        res, b = _run(tr, n)
        rays = tr.traceAxionWrapper(n, SEED)
    counts, img = _records_bands(rays.x, rays.y, rays.w, rays.energy, EDGES3, setup.consts.chipXMax, f32=True)
    assert np.array_equal(b.counts, counts)
    assert np.allclose(b.image, img, rtol=1e-12, atol=1e-15 * img.sum())


def test_xray_source(rt):
    """Every passed ray of the X-ray source lands in the band of its energy; after update_setup with a source energy in
    another band the new rays land there."""
    setup, tb = make_config("babyiaxo_xmm", flags=abi.CF_XRAY_TEST)
    setup.testSource.energy = 3.0
    n = 5_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        for mode in (0, 2):
            tr.set_precision(mode)
            tr.enable_band_images(EDGES3)
            res, b = _run(tr, n)
            assert b.counts.tolist() == [0, res.counters[0]["n_passed"], 0] and b.counts[1] > 0
            s = setup
            s.testSource.energy = 5.0
            tr.update_setup(s)
            tr.set_precision(mode)
            res, b = _run(tr, n)
            assert b.counts.tolist() == [0, 0, res.counters[0]["n_passed"]] and b.counts[2] > 0
            s.testSource.energy = 3.0
            tr.update_setup(s)


def test_other_accumulators_unaffected(rt):
    """Radial histogram and spectra on: identical with and without the band images."""
    setup, tb = make_config("babyiaxo_xmm")
    n = 20_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.enable_radial_hist()
        tr.enable_spectra()
        out = {}
        for on in (False, True):
            tr.enable_band_images(EDGES3 if on else None)
            tr.reset_image()
            tr.trace_mc(n, SEED)
            out[on] = (tr.read_image(), tr.read_radial_hist(), tr.read_spectra())
    (r0, h0, s0), (r1, h1, s1) = out[False], out[True]
    assert np.array_equal(h0[2], h1[2]) and np.allclose(h0[1], h1[1], rtol=1e-12, atol=0)
    assert np.array_equal(s0.counts, s1.counts) and np.array_equal(s0.shell_counts, s1.shell_counts)
    assert np.allclose(s0.sum_w, s1.sum_w, rtol=1e-12, atol=0)
    assert r0.counters[0]["n_passed"] == r1.counters[0]["n_passed"]
    assert np.allclose(r0.image, r1.image, rtol=1e-10, atol=0)


def test_alias_sampler(rt):
    """The alias sampler is supported: its band images cover every passed ray and add up to its image."""
    setup, tb = make_config("cast_llnl")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.set_sampler(abi.SAMPLER_ALIAS)
        tr.enable_band_images(ALL)
        res, b = _run(tr, 20_000_000, seed=99)
        _cover_everything(res, b)


def test_lifecycle_and_errors(rt):
    setup, tb = make_config("babyiaxo_xmm")
    n = 1_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        with pytest.raises(rt.SartError, match="no band images"):
            tr.read_band_images()
        for bad in ([1.0], [2.0, 1.0], [1.0, 1.0], [-1.0, 2.0], [0.0, np.inf], [0.0, np.nan], list(range(18))):
            with pytest.raises(rt.SartError, match="sart_enable_band_images"):
                tr.enable_band_images(bad)
        e = np.array(EDGES3)
        assert rt.lib.sart_enable_band_images(tr._h, 17, None) == -1            # SART_ERR_ARG
        assert rt.lib.sart_enable_band_images(tr._h, -1, e.ctypes.data_as(abi.c_double_p)) == -1
        tr.enable_band_images(list(range(17)))   # 16 bands: the most there are
        tr.enable_band_images(EDGES3)
        _, a = _run(tr, n)
        assert a.counts.sum() > 0
        tr.angular_scan([0.0, 0.05], n, SEED)
        tr.traceAxionWrapper(10_000, SEED)
        tr.trace_passed(10_000, SEED)
        tr.trace_presampled(np.zeros((3, 4)), np.zeros((2, 4)), np.full(4, 3.0))
        w = np.random.default_rng(1).integers(0, 2 ** 32, size=(6, 1000), dtype=np.uint32)
        tr.trace_words(w)
        b = tr.read_band_images()
        for f in ("image", "image_w2", "counts"):
            assert np.array_equal(getattr(a, f), getattr(b, f)), f
        tr.reset_image()
        z = tr.read_band_images()
        assert z.counts.sum() == 0 and not z.image.any()
        tr.trace_mc(n, SEED)
        tr.enable_band_images([1.0, 3.0])
        z = tr.read_band_images()
        assert z.counts.tolist() == [0] and not z.image.any() and z.edges.tolist() == [1.0, 3.0]
        tr.set_axion_masses([0.01, 0.02])
        with pytest.raises(rt.SartError, match="single axion mass"):
            tr.trace_mc(1000, SEED)
        tr.set_axion_masses([setup.consts.mAxion])
        tr.enable_band_images(None)
        tr.enable_mass_spectra()
        tr.enable_band_images(EDGES3)
        with pytest.raises(rt.SartError, match="per-mass spectra"):
            tr.trace_mc(1000, SEED)
        tr.enable_band_images(None)
        with pytest.raises(rt.SartError, match="no band images"):
            tr.read_band_images()


def test_merge_one_rank_and_refusals(rt):
    """sart_allreduce_outputs over one handle: the merged band images equal the handle's own."""
    from solaraxionraytracing_b200 import multi_gpu
    setup, tb = make_config("cast_llnl")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.enable_band_images(EDGES3)
        _, b = _run(tr, 2_000_000)
        multi_gpu.comm_init_all([tr])
        multi_gpu.allreduce_outputs([tr])
        m = tr.read_merged_band_images()
        assert np.array_equal(m.counts, b.counts) and np.array_equal(m.image, b.image)
        tr.enable_band_images([1.0, 2.0])
        with pytest.raises(rt.SartError, match="no merged band images"):
            tr.read_merged_band_images()


def _two_gpus(rt):
    if rt.lib.sart_device_count() < 2:
        pytest.skip("needs two GPUs")


def test_merge_on_two_gpus(rt):
    """Two handles through sart_comm_init_all: merged band images equal one GPU tracing the same global rays; different
    edges on the two handles are refused."""
    _two_gpus(rt)
    from solaraxionraytracing_b200 import multi_gpu
    setup, tb = make_config("babyiaxo_xmm")
    fs = rt.FullRaytraceSetup(setup, tb)
    n = 10_000_000
    with rt.RayTracer(fs, 0) as one:
        one.set_precision(2)
        one.enable_band_images(EDGES3)
        _, ref = _run(one, n)
    r = multi_gpu.trace_on_devices(fs, [0, 1], n, SEED, precision=2, bands=EDGES3)
    assert np.array_equal(r.band_images.counts, ref.counts)
    assert np.allclose(r.band_images.image, ref.image, rtol=1e-12, atol=1e-15 * ref.image.sum())
    a, b = rt.RayTracer(fs, 0), rt.RayTracer(fs, 1)
    try:
        a.enable_band_images(EDGES3)
        b.enable_band_images([0.5, 2.0, 4.0, 9.0])
        multi_gpu.comm_init_all([a, b])
        with pytest.raises(rt.SartError, match="band"):
            multi_gpu.allreduce_outputs([a, b])
    finally:
        a.close()
        b.close()


def _cli(tmp_path, name, extra):
    from solaraxionraytracing_b200.__main__ import main
    from solaraxionraytracing_b200 import config
    cfg = tmp_path / f"{name}.toml"
    cfg.write_text(config.DEFAULT_CONFIG.read_text().replace('outputPath = "../out"', f'outputPath = "{tmp_path}/{name}"'))
    assert main(["--config", str(cfg), "--nRays", "300000", "--allowSynthetic", "--energyBands", "0,2,4,1000"] + extra) == 0
    return tmp_path / name


def test_command_line_writes_the_band_images(rt, tmp_path):
    """--energyBands writes one 13-column image file per band; bands covering everything add up to the image."""
    out = _cli(tmp_path, "one", [])
    img, cols = output.read_axion_image_csv(out / "axion_image_BabyIAXO.csv")
    names = ["axion_image_BabyIAXO_E0-2keV.csv", "axion_image_BabyIAXO_E2-4keV.csv", "axion_image_BabyIAXO_E4-1000keV.csv"]
    total = np.zeros_like(img)
    for nm in names:
        b, bc = output.read_axion_image_csv(out / nm)
        assert list(bc) == output.CSV_COLUMNS
        assert np.array_equal(bc["yr0"], cols["yr0"])   # the whole run's containment radii
        total += b
    assert img.sum() > 0 and np.allclose(total, img, rtol=1e-12, atol=1e-15 * img.sum())
    if rt.lib.sart_device_count() >= 2:
        multi = _cli(tmp_path, "multi", ["--devices", "0,1"])
        for nm in names:
            a, _ = output.read_axion_image_csv(out / nm)
            b, _ = output.read_axion_image_csv(multi / nm)
            assert np.allclose(a, b, rtol=1e-12, atol=1e-15 * img.sum())
