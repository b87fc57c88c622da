"""Weighted histograms of per-ray record quantities of the passed rays of a fused run (sart_enable_quantity_hists /
sart_read_quantity_hists): against the oracle's records (mode 0), against the per-ray records of the same rays in the same
mode (modes 0, 1, 2; compaction, the alias sampler, a forced re-trace), row totals against mode 0 on 1e9 rays, next to the
other accumulators, for the X-ray source, their lifecycle and refusals, merging over ranks and the command line."""
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


def _specs_from(records, nbins=64):
    """All eight quantities, each over the 2nd .. 98th percentile of its passed rays' values (so that under- and overflow,
    and the regular bins, all see rays); a quantity with a single value gets a range around it."""
    sel = np.asarray(records.w) != 0.0
    specs = []
    for k, name in enumerate(abi.QUANTITIES):
        v = np.asarray(getattr(records, name))[sel]
        v = v[np.isfinite(v)]
        lo, hi = (np.percentile(v, [2.0, 98.0]) if v.size else (0.0, 1.0))
        if not lo < hi:
            lo, hi = lo - 1.0 - abs(lo), hi + 1.0 + abs(hi)
        specs.append((name, nbins + 7 * k, float(lo), float(hi)))
    return specs


def _assert_equal_hists(got, want, rtol=1e-12):
    assert [h.name for h in got] == [h.name for h in want]
    for g, w in zip(got, want):
        assert np.array_equal(g.counts, w.counts), (g.name, g.counts, w.counts)
        floor = 1e-15 * max(w.sum_w.sum(), 1e-300)
        assert np.allclose(g.sum_w, w.sum_w, rtol=rtol, atol=floor), g.name
        assert np.allclose(g.sum_w2, w.sum_w2, rtol=rtol, atol=1e-15 * max(w.sum_w2.sum(), 1e-300)), g.name
        assert np.array_equal(g.edges, w.edges)


def _fused(tr, n, specs, seed=SEED, first=0):
    tr.enable_quantity_hists(specs)
    tr.reset_image()
    tr.trace_mc(n, seed, first_ray=first)
    return tr.read_image(), tr.read_quantity_hists()


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_mode0_equals_the_oracle_records(rt, oracle, cfg):
    """2e6 rays, all eight quantities: counts equal and Σw within 1e-10 of the oracle's records binned on the host, after
    the rays whose exit code, weight or histogram entry differs because of libm are taken out of both sides (as in
    test_gpu_band_images.py: test_mode0_band_images_equal_the_oracle_records)."""
    setup, tb = make_config(cfg)
    n = 2_000_000
    ref = oracle.trace_mc_rays(setup, tb, 0, n, SEED)
    specs = _specs_from(ref)
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(0)
        _, got = _fused(tr, n, specs)
        gpu = tr.traceAxionWrapper(n, SEED)
    assert np.count_nonzero(gpu.code != ref.code) <= n // 5000
    odd = (gpu.code != ref.code) | (np.abs(gpu.w - ref.w) > 1e-10 * np.abs(ref.w))
    print(cfg, "rays with another exit code or weight:", int(odd.sum()))
    for name, nb, lo, hi in specs:
        moved = output.quantity_hist_entries(getattr(gpu, name), nb, lo, hi) != \
            output.quantity_hist_entries(getattr(ref, name), nb, lo, hi)
        print(cfg, name, "rays in another entry:", int(moved.sum()))
        odd |= moved
    assert odd.sum() <= n // 500

    class Sub:
        def __init__(self, rec, sel):
            self.w = rec.w[sel]
            for q in abi.QUANTITIES:
                setattr(self, q, getattr(rec, q)[sel])

    g_odd = output.quantity_hists_from_records(Sub(gpu, odd), specs)
    o_keep = output.quantity_hists_from_records(Sub(ref, ~odd), specs)
    for g, go, o in zip(got, g_odd, o_keep):
        assert np.array_equal(g.counts - go.counts, o.counts), g.name
        assert np.allclose(g.sum_w - go.sum_w, o.sum_w, rtol=1e-10, atol=1e-15 * o.sum_w.sum()), g.name
        assert o.counts[1:-1].sum() > 0


CASES = [("cast_llnl", 0, None, False, None, False), ("babyiaxo_xmm", 0, None, False, None, False)] + [
    (cfg, mode, compact, False, None, smem) for cfg in ("cast_llnl", "babyiaxo_xmm") for mode in (1, 2) for compact in (0, 1)
    for smem in (False, True)] + [
    ("cast_llnl", 2, None, True, None, False), ("babyiaxo_xmm", 2, None, True, None, False),
    ("cast_llnl", 2, None, False, 12.0, False), ("babyiaxo_xmm", 2, None, False, 12.0, False)]


@pytest.mark.parametrize("cfg,mode,compact,alias,scale,smem", CASES)
def test_fused_equals_the_same_modes_records(rt, monkeypatch, cfg, mode, compact, alias, scale, smem):
    """4e6 rays: counts identical and Σw, Σw² within 1e-12 of quantity_hists_from_records on traceAxionWrapper's records of
    the same rays in the same mode (compaction on and off; the blocks' sums in their replicas or, with SART_QHIST_SMEM, in
    shared memory; error budgets x12, so that percents of the rays go through the FP64 re-trace). The alias sampler: the fused kernel runs without the margin tests (it has no re-trace), the record
    kernel with them, and the two give slightly different values to about 1e-5 of the passed rays (measured on B200:
    at most 38 of 3.5e6 rays in another bin, Σw 1.4e-7 apart) — every row counts n_passed, at most 1e-4 of the passed rays
    sit in another bin, and the sums agree to 1e-6."""
    if smem:
        monkeypatch.setenv("SART_QHIST_SMEM", "1")
    setup, tb = make_config(cfg)
    n = 4_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        if compact is not None:
            tr.set_compaction(compact)
        if alias:
            tr.set_sampler(abi.SAMPLER_ALIAS)
        if scale is not None:
            tr.set_retrace(1, scale)
        rays = tr.traceAxionWrapper(n, SEED)
        specs = _specs_from(rays)
        res, got = _fused(tr, n, specs)
    c = res.counters[0]
    if scale is not None:
        assert c["n_retraced"] / n > 0.01
    assert c["n_unresolved"] == 0
    want = output.quantity_hists_from_records(rays, specs)
    for h in got:
        assert int(h.counts.sum()) == c["n_passed"]
    if not alias:
        _assert_equal_hists(got, want)
        return
    for g, w in zip(got, want):
        moved = int(np.abs(g.counts.astype(np.int64) - w.counts.astype(np.int64)).sum())
        print(cfg, g.name, "rays in another bin:", moved)
        assert moved <= max(10, c["n_passed"] // 10_000), g.name
        assert g.sum_w.sum() == pytest.approx(w.sum_w.sum(), rel=1e-6)
        assert np.abs(g.sum_w - w.sum_w).sum() <= 1e-4 * w.sum_w.sum()


def test_row_totals_on_1e9_rays(rt):
    """1e9 rays, mode 2 with the re-trace, all eight quantities at 256 bins: every row counts n_passed rays, which equals
    mode 0's, and sums to the run's Σw."""
    setup, tb = make_config("cast_llnl", **BIG)
    n = 1_000_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        rays = tr.traceAxionWrapper(1_000_000, SEED)
        specs = [(name, 256, lo, hi) for name, _, lo, hi in _specs_from(rays)]
        r0, _ = _fused(tr, n, specs)
        tr.set_precision(2)
        r2, got = _fused(tr, n, specs)
    c0, c2 = r0.counters[0], r2.counters[0]
    assert c2["n_unresolved"] == 0 and c2["n_passed"] == c0["n_passed"]
    for h in got:
        assert int(h.counts.sum()) == c2["n_passed"], h.name
        assert h.sum_w.sum() == pytest.approx(c2["sum_w"], rel=1e-12), h.name
        assert h.sum_w2.sum() == pytest.approx(c2["sum_w2"], rel=1e-12), h.name


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_other_accumulators_unaffected(rt, mode):
    """Image, counters, radial histogram, spectra and band images are the same with and without the quantity histograms."""
    setup, tb = make_config("babyiaxo_xmm")
    n = 10_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        specs = _specs_from(tr.traceAxionWrapper(200_000, SEED))
        tr.enable_radial_hist()
        tr.enable_spectra()
        tr.enable_band_images([0.5, 2.0, 4.0, 8.0])
        out = {}
        for on in (False, True):
            tr.enable_quantity_hists(specs if on else None)
            tr.reset_image()
            tr.trace_mc(n, SEED)
            out[on] = (tr.read_image(), tr.read_radial_hist(), tr.read_spectra(), tr.read_band_images())
    (r0, h0, s0, b0), (r1, h1, s1, b1) = out[False], out[True]
    c0, c1 = r0.counters[0], r1.counters[0]
    for k in c0:
        if k.startswith("sum_"):
            assert c1[k] == pytest.approx(c0[k], rel=1e-12, abs=0), k
        else:
            assert c1[k] == c0[k], k
    assert np.allclose(r1.image, r0.image, rtol=1e-12, atol=1e-15 * r0.image.sum())
    assert np.array_equal(h0[2], h1[2]) and np.allclose(h0[1], h1[1], rtol=1e-12, atol=0)
    assert np.array_equal(s0.counts, s1.counts) and np.array_equal(s0.shell_counts, s1.shell_counts)
    assert np.allclose(s0.sum_w, s1.sum_w, rtol=1e-12, atol=0)
    assert np.array_equal(b0.counts, b1.counts)
    assert np.allclose(b0.image, b1.image, rtol=1e-12, atol=1e-15 * b0.image.sum())


def test_xray_source(rt):
    """The X-ray source in modes 0 and 2: the histograms equal those of the same rays' records."""
    setup, tb = make_config("babyiaxo_xmm", flags=abi.CF_XRAY_TEST)
    setup.testSource.energy = 3.0
    n = 2_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        for mode in (0, 2):
            tr.set_precision(mode)
            rays = tr.traceAxionWrapper(n, SEED)
            specs = _specs_from(rays)
            res, got = _fused(tr, n, specs)
            assert res.counters[0]["n_passed"] > 0
            _assert_equal_hists(got, output.quantity_hists_from_records(rays, specs))


def test_lifecycle_and_refusals(rt):
    setup, tb = make_config("babyiaxo_xmm")
    n = 1_000_000
    specs = [("reflect", 16, 0.0, 1.0), ("yaw", 8, -1.0, 1.0)]
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        with pytest.raises(rt.SartError, match="no quantity histograms"):
            tr.read_quantity_hists()
        h = tr._h
        Spec = abi.QuantityHistSpec

        def enable(*s):
            arr = (Spec * max(len(s), 1))(*s)
            return rt.lib.sart_enable_quantity_hists(h, len(s), arr)

        for bad in ([Spec(8, 4, 0.0, 1.0)], [Spec(-1, 4, 0.0, 1.0)], [Spec(0, 0, 0.0, 1.0)], [Spec(0, 513, 0.0, 1.0)],
                    [Spec(0, 4, 1.0, 1.0)], [Spec(0, 4, 2.0, 1.0)], [Spec(0, 4, np.nan, 1.0)], [Spec(0, 4, 0.0, np.inf)],
                    [Spec(0, 4, -np.inf, 0.0)], [Spec(0, 4, 0.0, 1.0), Spec(0, 8, 0.0, 2.0)]):
            assert enable(*bad) == -1, bad                                             # SART_ERR_ARG
        assert rt.lib.sart_enable_quantity_hists(h, 9, (Spec * 9)()) == -1
        assert rt.lib.sart_enable_quantity_hists(h, -1, None) == -1
        assert rt.lib.sart_enable_quantity_hists(h, 2, None) == -1
        assert enable(*[Spec(q, 512, 0.0, 1.0) for q in range(8)]) == 0               # the largest there is
        with pytest.raises(ValueError):
            tr.enable_quantity_hists([("bogus", 4, 0.0, 1.0)])
        tr.enable_quantity_hists(specs)
        _, a = _fused(tr, n, specs)
        assert sum(int(x.counts.sum()) for x in a) > 0
        tr.trace_mc(n, SEED, first_ray=n)        # accumulates (+=)
        acc = tr.read_quantity_hists()
        assert all(int(y.counts.sum()) > int(x.counts.sum()) for x, y in zip(a, acc))
        tr.angular_scan([0.0, 0.05], n, SEED)
        tr.traceAxionWrapper(10_000, SEED)
        tr.trace_passed(10_000, SEED)
        tr.trace_presampled(np.zeros((3, 4)), np.zeros((2, 4)), np.full(4, 3.0))
        w = np.random.default_rng(1).integers(0, 2 ** 32, size=(6, 1000), dtype=np.uint32)
        tr.trace_words(w)
        b = tr.read_quantity_hists()
        for x, y in zip(acc, b):
            assert np.array_equal(x.counts, y.counts) and np.array_equal(x.sum_w, y.sum_w)
        tr.reset_image()
        assert all(not z.counts.any() and not z.sum_w.any() for z in tr.read_quantity_hists())
        tr.trace_mc(n, SEED)
        tr.enable_quantity_hists([("pathCB", 4, 0.0, 1e4)])    # other specs: cleared, new shape
        (z,) = tr.read_quantity_hists()
        assert z.name == "pathCB" and z.counts.size == 6 and not z.counts.any()
        tr.set_axion_masses([0.01, 0.02])
        with pytest.raises(rt.SartError, match="single axion mass"):
            tr.trace_mc(1000, SEED)
        tr.set_axion_masses([setup.consts.mAxion])
        tr.enable_quantity_hists(None)
        tr.enable_mass_spectra()
        tr.enable_quantity_hists(specs)
        with pytest.raises(rt.SartError, match="per-mass spectra"):
            tr.trace_mc(1000, SEED)
        tr.enable_mass_spectra(False)
        tr.enable_quantity_hists([])
        with pytest.raises(rt.SartError, match="no quantity histograms"):
            tr.read_quantity_hists()


def test_merge_one_rank(rt):
    """sart_allreduce_outputs over one handle: the merged histograms equal the handle's own; new specs drop the merged copy."""
    from solaraxionraytracing_b200 import multi_gpu
    setup, tb = make_config("cast_llnl")
    specs = [("alpha1", 32, 0.0, 1.0), ("transProbArgon", 16, 0.0, 1.0)]
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        _, a = _fused(tr, 2_000_000, specs)
        multi_gpu.comm_init_all([tr])
        multi_gpu.allreduce_outputs([tr])
        m = tr.read_merged_quantity_hists()
        for x, y in zip(a, m):
            assert np.array_equal(x.counts, y.counts) and np.array_equal(x.sum_w, y.sum_w)
        tr.enable_quantity_hists(specs[:1])
        with pytest.raises(rt.SartError, match="no merged quantity histograms"):
            tr.read_merged_quantity_hists()


def test_merge_on_two_gpus(rt):
    """Two handles through sart_comm_init_all: the merged histograms equal one GPU tracing the same global rays; handles
    with different specs (another range, the same number of entries) are refused before any collective."""
    if rt.lib.sart_device_count() < 2:
        pytest.skip("needs two GPUs")
    from solaraxionraytracing_b200 import multi_gpu
    setup, tb = make_config("babyiaxo_xmm")
    fs = rt.FullRaytraceSetup(setup, tb)
    n = 10_000_000
    specs = [("reflect", 32, 0.0, 1.0), ("deviationDet", 32, 0.0, 1.0)]
    with rt.RayTracer(fs, 0) as one:
        one.set_precision(2)
        _, ref = _fused(one, n, specs)
    r = multi_gpu.trace_on_devices(fs, [0, 1], n, SEED, precision=2, quantity_hists=specs)
    for x, y in zip(r.quantity_hists, ref):
        assert np.array_equal(x.counts, y.counts)
        assert np.allclose(x.sum_w, y.sum_w, rtol=1e-12, atol=1e-15 * y.sum_w.sum())
    a, b = rt.RayTracer(fs, 0), rt.RayTracer(fs, 1)
    try:
        a.enable_quantity_hists(specs)
        b.enable_quantity_hists([("reflect", 32, 0.0, 2.0), specs[1]])
        multi_gpu.comm_init_all([a, b])
        with pytest.raises(rt.SartError, match="quantity histograms"):
            multi_gpu.allreduce_outputs([a, b])
    finally:
        a.close()
        b.close()


def _cli(tmp_path, name, extra):
    from solaraxionraytracing_b200.__main__ import main
    from solaraxionraytracing_b200 import config
    cfg = tmp_path / f"{name}.toml"
    cfg.write_text(config.DEFAULT_CONFIG.read_text().replace('outputPath = "../out"', f'outputPath = "{tmp_path}/{name}"'))
    assert main(["--config", str(cfg), "--nRays", "300000", "--allowSynthetic", "--histogram", "reflect:20:0:1",
                 "--histogram", "yaw:10:-0.5:0.5"] + extra) == 0
    return tmp_path / name


def _captured(monkeypatch, rt, method):
    """Wraps RayTracer.<method> so that the test sees the histograms the command line read."""
    seen = []
    orig = getattr(rt.RayTracer, method)

    def wrapper(self):
        r = orig(self)
        seen.append(r)
        return r
    monkeypatch.setattr(rt.RayTracer, method, wrapper)
    return seen


def _rows_equal(path, h):
    c = output.read_columns_csv(path)
    assert list(c) == output.QUANTITY_HIST_COLUMNS
    assert c["lower edge"][0] == -np.inf and c["upper edge"][-1] == np.inf
    assert np.array_equal(c["lower edge"][1:], h.edges) and np.array_equal(c["upper edge"][:-1], h.edges)
    assert np.array_equal(c["rays"].astype(np.uint64), h.counts)
    assert np.array_equal(c["flux"], h.sum_w) and np.array_equal(c["flux error"], np.sqrt(h.sum_w2))
    return c


def test_command_line_writes_the_histograms(rt, tmp_path, monkeypatch):
    """--histogram writes one file per histogram whose rows are the histograms the run read (read_quantity_hists on one
    GPU, read_merged_quantity_hists with --devices)."""
    seen = _captured(monkeypatch, rt, "read_quantity_hists")
    out = _cli(tmp_path, "one", [])
    (hists,) = seen
    assert [h.name for h in hists] == ["reflect", "yaw"]
    for h in hists:
        c = _rows_equal(out / f"axion_hist_{h.name}_BabyIAXO.csv", h)
        assert c["rays"].sum() > 0
    if rt.lib.sart_device_count() >= 2:
        seen_m = _captured(monkeypatch, rt, "read_merged_quantity_hists")
        multi = _cli(tmp_path, "multi", ["--devices", "0,1"])
        (mh,) = seen_m
        for h, m in zip(hists, mh):
            _rows_equal(multi / f"axion_hist_{m.name}_BabyIAXO.csv", m)
            assert np.array_equal(m.counts, h.counts)
