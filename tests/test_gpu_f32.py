"""The single-precision pipeline (precision mode 2: FP32 geometry on (point, slopes), FP32 weight factors, FP64 sums)
against the exact pipeline, a 60-digit evaluation of the reference's formulas, and the CPU oracle (statistically).

Stated tolerances (north_star tier (a): "(x, y, weight) within a stated FP32 tolerance"):
  * sampling is integer work shared with mode 1: every ray has the SAME emission shell / energy / exit-disc point as in
    the exact pipeline (energies compared bit for bit on the rays both pipelines pass);
  * vs 60-digit arithmetic on the same ray: |d| <= 2e-4 mm (LLNL, 1.5 m to the detector; measured median 9e-6, max
    4e-5) / 5e-4 mm (XMM, 7.5 m; measured median 2.4e-5, max 1.1e-4) on every tested ray — the rounding noise of the
    reference's own f64 formulation is 5.6e-5 mm median, 4e-4 mm at the 99th percentile with outliers to 0.1 mm
    (DESIGN.md §3), so FP32 on (point, slopes) is closer to exact arithmetic than the reference's FP64 on point pairs;
  * vs the exact pipeline on the same Philox rays: exit codes equal for all but <= 1e-4 of the rays (measured 1e-5),
    detector positions median <= 2e-4 mm / 99 % <= 1.5e-3 mm (measured 1.3e-5 / 5.5e-5 LLNL, 6e-5 / 2.8e-4 XMM — the
    reference's noise, which the exact pipeline reproduces), weights 99 % |dw/w| <= 2e-4 (5e-3 with the buffer gas);
  * vs the CPU oracle with an independent seed: per-bin chi^2 of the 256x256 image consistent with 1.
"""
import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import abi
from test_gpu_fast import _chi2

pytestmark = pytest.mark.gpu
SEED = 299792458


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    assert raytracer.lib.sart_has_precision(2) == 1
    return raytracer


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm", "cast_abrixas", "babyiaxo_gas"])
def test_f32_rays_vs_exact(rt, cfg):
    setup, tb = make_config(cfg)
    n = 1_000_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        ex = tr.traceAxionWrapper(n, SEED, optional=True)
        tr.set_precision(2)
        fa = tr.traceAxionWrapper(n, SEED, optional=True)
    mism = ex.exit_code != fa.exit_code
    print(cfg, "exit-code mismatch rate", mism.mean())
    assert mism.mean() <= 1e-4, f"exit-code mismatch rate {mism.mean():.2e}"
    both = (~mism) & (ex.exit_code == abi.EXIT_PASSED)
    assert both.sum() > n // 10
    assert np.array_equal(ex.shell[both], fa.shell[both])
    assert np.array_equal(ex.energy[both].astype(np.float32), fa.energy[both].astype(np.float32))   # same sampled energy
    d = np.hypot(ex.x[both] - fa.x[both], ex.y[both] - fa.y[both])
    print(cfg, "position diff median / 99% / max", np.median(d), np.quantile(d, 0.99), d.max())
    assert np.median(d) <= 2e-4 and np.quantile(d, 0.99) <= 1.5e-3, (np.median(d), np.quantile(d, 0.99))
    dw = np.abs(fa.w[both] / ex.w[both] - 1.0)
    print(cfg, "weight diff 99%", np.quantile(dw, 0.99))
    tol = 5e-3 if cfg == "babyiaxo_gas" else 2e-4
    assert np.quantile(dw, 0.99) <= tol, np.quantile(dw, 0.99)


@pytest.mark.parametrize("cfg,tol", [("cast_llnl", 2e-4), ("babyiaxo_xmm", 5e-4)])
def test_f32_rays_vs_high_precision(rt, oracle, cfg, tol):
    import hp_trace
    setup, tb = make_config(cfg)
    n = 3000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        fa = tr.traceAxionWrapper(n, SEED, optional=False)
    origin, exit_xy, _ = oracle.sample_rays(setup, tb, 0, n, SEED)
    idx = np.flatnonzero(fa.exit_code == abi.EXIT_PASSED)[:250]
    errs = []
    for i in idx:
        hp = hp_trace.trace(setup, origin[:, i], exit_xy[:, i])
        if hp is None:      # a boundary ray: FP32 and exact arithmetic may classify it differently
            continue
        assert hp[2] == fa.shell[i]
        errs.append(float(np.hypot(hp[0] - fa.x[i], hp[1] - fa.y[i])))
    errs = np.array(errs)
    print(cfg, "vs 60-digit: median / max", np.median(errs), errs.max(), "n", errs.size)
    assert errs.size >= 240
    assert errs.max() <= tol, errs.max()


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_f32_counters_and_compaction(rt, cfg):
    setup, tb = make_config(cfg)
    n = 3_000_001
    out = {}
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.trace_mc(n, SEED, first_ray=17); e = tr.read_image()
        tr.set_precision(2)
        for mode in (0, 1):
            tr.set_compaction(mode)
            tr.reset_image()
            tr.trace_mc(n, SEED, first_ray=17)
            out[mode] = tr.read_image()
    a, b = out[0].counters[0], out[1].counters[0]
    assert a["n_exit"] == b["n_exit"] and a["n_rays"] == b["n_rays"] == n
    assert np.allclose(out[0].image, out[1].image, rtol=1e-10, atol=0)
    ce = e.counters[0]
    for k, v in ce["n_exit"].items():
        assert abs(a["n_exit"][k] - v) <= max(30, n // 2000), (k, a["n_exit"][k], v)
    assert abs(a["sum_w"] / ce["sum_w"] - 1.0) < 3e-4
    assert abs(out[0].image.sum() / a["sum_w"] - 1.0) < 1e-9


@pytest.mark.parametrize("sampler", [abi.SAMPLER_INVERSE_CDF, abi.SAMPLER_ALIAS])
def test_f32_image_statistically_equal_to_oracle(rt, oracle, sampler):
    """Tier (b) for both samplers of the FP32 pipeline: the inverse-CDF search (the reference's lowerBound) and the alias
    tables of the same distributions."""
    setup, tb = make_config("cast_llnl")
    n_gpu, n_cpu = 20_000_000, 2_000_000
    img_o, img2_o, cnt_o = oracle.trace_mc(setup, tb, 0, n_cpu, 12345)
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.set_sampler(sampler)
        tr.trace_mc(n_gpu, 777)
        res = tr.read_image()
    a, va = res.image[0] / n_gpu, res.image_w2[0] / n_gpu ** 2
    b, vb = img_o[0] / n_cpu, img2_o[0] / n_cpu ** 2
    chi2, ndf = _chi2(a, va, b, vb)
    assert ndf > 100
    z = (chi2 - ndf) / np.sqrt(2.0 * ndf)
    assert abs(z) < 5.0, (chi2, ndf, z)
    sig = np.sqrt(va.sum() + vb.sum())
    assert abs(a.sum() - b.sum()) < 4.0 * sig
    pa, pb = res.counters[0]["n_passed"] / n_gpu, cnt_o[0]["n_passed"] / n_cpu
    assert abs(pa - pb) < 5.0 * np.sqrt(pb * (1 - pb) * (1 / n_gpu + 1 / n_cpu))


def test_f32_xray_source_and_scan(rt):
    """The X-ray test source and the batched angular scan run in mode 2 and agree with mode 1 to Monte Carlo noise-free
    precision (same rays): relative fluxes within 2e-3."""
    flags = rt.flags_from_cli(xrayTest=True, ignoreDetWindow=True, ignoreGasAbs=True, ignoreConvProb=True)
    setup, tb = make_config("babyiaxo_xmm", flags=flags)
    setup.testSource.parallel = 1
    setup.consts.chipXMax = setup.consts.chipYMax = 100.0
    angles = np.array([0.0, 0.05, 0.15, 0.3])
    fl = {}
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        for mode in (1, 2):
            tr.set_precision(mode)
            fl[mode], cnt, _ = tr.angular_scan(angles, 1_000_000, SEED)
            assert all(c["n_rays"] == 1_000_000 for c in cnt)
    assert np.allclose(fl[2], fl[1], rtol=2e-3)
    assert fl[2][0] > fl[2][1] > fl[2][2] > fl[2][3] > 0


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm", "babyiaxo_gas"])
def test_f32_presampled_vs_oracle(rt, oracle, cfg):
    """Tier (a) for the FP32 pipeline: the CPU oracle and sart_trace_presampled (precision 2) fed identical pre-sampled
    emission points, exit-disc points and energies. Hit/miss classification equal for all but <= 1e-4 of the rays (rays
    within the reference's own rounding noise of an aperture edge), positions within 1.5e-3 mm (99 %), weights within
    2e-4 relative (99 %; 5e-3 with the buffer gas)."""
    setup, tb = make_config(cfg)
    n = 400_000
    origin, exit_xy, energy = oracle.sample_rays(setup, tb, 0, n, SEED)
    ref = oracle.trace_presampled(setup, tb, origin, exit_xy, energy)
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        gpu = tr.trace_presampled(origin, exit_xy, energy)
    assert not np.any(gpu.code & abi.FLAG_INTERP_CLAMPED & ~(ref.code & abi.FLAG_INTERP_CLAMPED)), "energies are table values"
    mism = (gpu.code & abi.CODE_MASK) != (ref.code & abi.CODE_MASK)
    assert mism.mean() <= 1e-4, mism.mean()
    both = (~mism) & ((ref.code & abi.CODE_MASK) == abi.EXIT_PASSED)
    assert both.sum() > n // 10
    assert np.array_equal(gpu.shell[both], ref.shell[both])
    d = np.hypot(gpu.x[both] - ref.x[both], gpu.y[both] - ref.y[both])
    assert np.median(d) <= 2e-4 and np.quantile(d, 0.99) <= 1.5e-3, (np.median(d), np.quantile(d, 0.99))
    dw = np.abs(gpu.w[both] / ref.w[both] - 1.0)
    assert np.quantile(dw, 0.99) <= (5e-3 if cfg == "babyiaxo_gas" else 2e-4), np.quantile(dw, 0.99)
    assert np.allclose(gpu.energy[both], ref.energy[both], rtol=0, atol=0)


def test_f32_presampled_off_grid_energy_is_flagged(rt, oracle):
    setup, tb = make_config("cast_llnl")
    n = 1000
    origin, exit_xy, energy = oracle.sample_rays(setup, tb, 0, n, SEED)
    shifted = energy + 0.37 * (tb.energies[1] - tb.energies[0])
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.set_retrace(0)     # a re-traced ray would go through the exact pipeline, which interpolates at the shifted energy
        a = tr.trace_presampled(origin, exit_xy, energy, optional=False)
        b = tr.trace_presampled(origin, exit_xy, shifted, optional=False)
    reached = (a.code & abi.CODE_MASK).astype(int)
    tail = np.isin(reached, [abi.EXIT_PASSED, abi.EXIT_ZERO_WEIGHT, abi.EXIT_WINDOW_APERTURE])
    assert tail.sum() > 100
    assert np.all((b.code[tail] & abi.FLAG_INTERP_CLAMPED) != 0) and not np.any(a.code[tail] & abi.FLAG_INTERP_CLAMPED)
    assert np.array_equal(a.x, b.x) and np.array_equal(a.w, b.w)      # traced at the nearest tabulated energy


def test_f32_mass_scan_vs_exact(rt):
    """BASELINE config 4 with FP32 tracing: 64 axion masses sharing one traced ray, against the exact pipeline."""
    setup, tb = make_config("babyiaxo_gas")
    n = 400_000
    masses = np.concatenate([np.linspace(0.004, 0.012, 40), np.linspace(0.02, 0.4, 24)])
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_axion_masses(masses)
        tr.trace_mc(n, 3)
        e = tr.read_image()
        tr.set_precision(2)
        tr.reset_image()
        tr.trace_mc(n // 3, 3); tr.trace_mc(n - n // 3, 3, first_ray=n // 3)     # two launches: the accumulators fold twice
        f = tr.read_image()
    assert f.image.shape == (64, 256, 256)
    for m in range(64):
        ce, cf = e.counters[m], f.counters[m]
        assert cf["n_rays"] == n
        assert abs(cf["n_passed"] - ce["n_passed"]) <= 20, m
        for k, v in ce["n_exit"].items():
            assert abs(cf["n_exit"][k] - v) <= 20, (m, k)
        assert abs(cf["sum_w"] / ce["sum_w"] - 1.0) < 2e-3, (m, cf["sum_w"], ce["sum_w"])
        assert abs(f.image[m].sum() / cf["sum_w"] - 1.0) < 1e-9
        assert abs(f.image_w2[m].sum() / cf["sum_w2"] - 1.0) < 1e-9
    assert np.abs(f.image - e.image).sum() / e.image.sum() < 2e-2


def _weighted_ks(a, wa, b, wb):
    """Two-sample Kolmogorov-Smirnov distance of weighted samples and its effective sizes (Sum w)^2 / Sum w^2."""
    ia, ib = np.argsort(a), np.argsort(b)
    a, wa, b, wb = a[ia], wa[ia], b[ib], wb[ib]
    grid = np.concatenate([a, b])
    grid.sort()
    Fa = np.searchsorted(a, grid, side="right")
    Fb = np.searchsorted(b, grid, side="right")
    ca, cb = np.concatenate([[0.0], np.cumsum(wa)]) / wa.sum(), np.concatenate([[0.0], np.cumsum(wb)]) / wb.sum()
    d = float(np.max(np.abs(ca[Fa] - cb[Fb])))
    return d, wa.sum() ** 2 / (wa ** 2).sum(), wb.sum() ** 2 / (wb ** 2).sum()


@pytest.mark.parametrize("sampler", [abi.SAMPLER_INVERSE_CDF, abi.SAMPLER_ALIAS])
@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_f32_ks_against_oracle(rt, oracle, cfg, sampler):
    """Tier (b), Kolmogorov-Smirnov: the weighted distributions of x, y, r and energy of the passed rays, GPU (seed A)
    against the CPU oracle (independent seed B), agree at the 0.1 % level (c(alpha) = 1.95)."""
    setup, tb = make_config(cfg)
    n_gpu, n_cpu = 3_000_000, 600_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        tr.set_sampler(sampler)
        g = tr.traceAxionWrapper(n_gpu, 4242)
    o = oracle.trace_mc_rays(setup, tb, 0, n_cpu, 987654321)
    pg, po = g.passed, (o.code & abi.CODE_MASK) == abi.EXIT_PASSED
    assert pg.sum() > 1000 and po.sum() > 1000
    for name in ("x", "y", "r", "energy"):
        va, vb = getattr(g, name)[pg], getattr(o, name)[po]
        if name == "energy":     # a discrete distribution: the FP32 pipeline returns the table energy rounded to f32, so
            va, vb = va.astype(np.float32), vb.astype(np.float32)   # compare the atoms at equal values
        d, na, nb = _weighted_ks(va, g.w[pg], vb, o.w[po])
        crit = 1.95 * np.sqrt((na + nb) / (na * nb))
        assert d < crit, (name, d, crit, na, nb)


def test_f32_presampled_edge_inputs(rt, oracle):
    """Empty batch, a far-off-axis ray, NaN inputs and an energy outside the tabulated range in the FP32 pre-sampled
    kernel: no crash, the geometric classification of the well-defined rays equals the oracle's, the NaN ray and the
    out-of-range energy end in a defined exit code / the clamped flag."""
    setup, tb = make_config("cast_llnl")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        out = tr.trace_presampled(np.zeros((3, 0)), np.zeros((2, 0)), np.zeros(0))
        assert out.n == 0
        origin = np.array([[0.0, 1e13, np.nan, 3e11], [0.0, 0.0, 0.0, -2e11], [-1.5e14, -1.5e14, -1.5e14, -1.4999e14]])
        exit_xy = np.array([[0.0, 0.0, 1.0, 21.49], [0.0, 0.0, 1.0, 0.0]])
        energy = np.array([float(tb.energies[40]), float(tb.energies[40]), float(tb.energies[40]), 20.0])
        ref = oracle.trace_presampled(setup, tb, origin, exit_xy, energy)
        gpu = tr.trace_presampled(origin, exit_xy, energy)
    for i in (0, 1, 3):
        assert (gpu.code[i] & abi.CODE_MASK) == (ref.code[i] & abi.CODE_MASK), (i, gpu.code[i], ref.code[i])
    assert 0 < (gpu.code[2] & abi.CODE_MASK) < abi.N_EXIT_CODES and gpu.w[2] == 0.0      # NaN origin: never "passed"
    assert np.all(np.isfinite(gpu.x)) and np.all(np.isfinite(gpu.w))


@pytest.mark.parametrize("mode", [2, 0])
def test_presampled_host_path_chunks(rt, oracle, mode):
    """sart_trace_presampled with host buffers streams chunks of 1 Mi rays through two device buffers on three streams;
    the records are bit-identical to tracing the same rays slice by slice (one chunk per call)."""
    setup, tb = make_config("cast_llnl")
    n = 2_300_007 if mode == 2 else 1_200_003
    origin, exit_xy, energy = oracle.sample_rays(setup, tb, 0, n, 77)
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        whole = tr.trace_presampled(origin, exit_xy, energy, optional=True)
        parts = []
        for a in range(0, n, 700_000):
            b = min(n, a + 700_000)
            parts.append(tr.trace_presampled(origin[:, a:b], exit_xy[:, a:b], energy[a:b], optional=True))
    for name in ("x", "y", "w", "code", "shell", "energy", "r"):
        assert np.array_equal(getattr(whole, name), np.concatenate([getattr(p, name) for p in parts])), name
    assert (whole.exit_code == abi.EXIT_PASSED).mean() > 0.8


def test_f32_refuses_shells_its_radial_table_cannot_resolve(rt):
    """A glass 1e-5 mm thick puts two boundaries of the shell search into one bucket of the radial table (at most 4000
    buckets): the FP32 pipeline refuses the setup with a message, modes 1 and 0 (their own shell scans) trace it, and the
    CPU-side helper reports the same condition."""
    import ctypes as C
    setup, tb = make_config("cast_llnl")
    setup.telescope.allThickness[3] = 1e-5
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        with pytest.raises(rt.SartError, match="radial lookup table"):
            tr.set_precision(2)
        out = {}
        for mode in (1, 0):
            tr.set_precision(mode); tr.reset_image()
            tr.trace_mc(200_000, 3)
            out[mode] = tr.read_image().counters[0]
    assert out[1]["n_rays"] == out[0]["n_rays"] == 200_000
    assert sum(abs(out[1]["n_exit"][k] - out[0]["n_exit"][k]) for k in out[0]["n_exit"]) <= 4
    rho = np.array([70.0], dtype=np.float32); a = np.zeros(1, dtype=np.int32); b = np.zeros(1, dtype=np.int32)
    rc = rt.lib.sart_shell_lookup(C.byref(setup), 1, rho.ctypes.data_as(C.POINTER(C.c_float)),
                                  a.ctypes.data_as(C.POINTER(C.c_int32)), b.ctypes.data_as(C.POINTER(C.c_int32)))
    assert rc != 0


@pytest.mark.parametrize("cfg", ["cast_llnl", "babyiaxo_xmm"])
def test_alias_sampler_draws_the_same_distributions(rt, cfg):
    """sart_set_sampler(ALIAS) against the inverse-CDF search on the same kernels: the energies of the rays that reach the
    mirrors (a discrete distribution over the table energies, mixed over the emission shells) in a two-sample chi^2 over
    the atoms; the exit-code histogram (which depends on the emission radius through the ray directions) within
    binomial errors; the images (fused kernel, with warp compaction on BabyIAXO+XMM) in the per-bin chi^2 of tier (b).
    The two samplers map the same random words to different rays, so the two runs are independent samples."""
    setup, tb = make_config(cfg)
    n = 6_000_000
    recs, imgs = {}, {}
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(2)
        for smp in (abi.SAMPLER_INVERSE_CDF, abi.SAMPLER_ALIAS):
            tr.set_sampler(smp)
            recs[smp] = tr.traceAxionWrapper(n, 31337)
            tr.reset_image()
            tr.trace_mc(4 * n, 99)
            imgs[smp] = tr.read_image()
        tr.set_sampler(abi.SAMPLER_ALIAS)
        tr.set_precision(1)
        with pytest.raises(rt.SartError, match="alias sampler"):
            tr.trace_mc(1000, 1)
    a, b = recs[abi.SAMPLER_INVERSE_CDF], recs[abi.SAMPLER_ALIAS]
    assert not np.array_equal(a.code, b.code)                       # different rays ...
    # ... same statistics. Exit codes: every code within 5 sigma (two binomial samples)
    for code in range(16):
        ka, kb = int(((a.code & abi.CODE_MASK) == code).sum()), int(((b.code & abi.CODE_MASK) == code).sum())
        p = (ka + kb) / (2 * n)
        assert abs(ka - kb) <= 5.0 * np.sqrt(2 * n * p * (1 - p)) + 1, (code, ka, kb)
    # energies of the rays with an energy (stage B reached): chi^2 over the atoms with enough entries
    ea, eb = a.energy[a.energy > 0].astype(np.float32), b.energy[b.energy > 0].astype(np.float32)
    atoms = np.union1d(ea, eb)
    ha = np.bincount(np.searchsorted(atoms, ea), minlength=atoms.size).astype(np.float64)
    hb = np.bincount(np.searchsorted(atoms, eb), minlength=atoms.size).astype(np.float64)
    sel = (ha + hb) >= 50
    assert sel.sum() > 100
    sa, sb = ha[sel].sum(), hb[sel].sum()
    chi2 = (((ha[sel] / sa - hb[sel] / sb) ** 2) / (ha[sel] / sa ** 2 + hb[sel] / sb ** 2)).sum()
    ndf = int(sel.sum()) - 1
    assert abs(chi2 - ndf) / np.sqrt(2.0 * ndf) < 5.0, (chi2, ndf)
    # images of the fused kernels
    ia, ib = imgs[abi.SAMPLER_INVERSE_CDF], imgs[abi.SAMPLER_ALIAS]
    m = 4 * n
    chi2, ndf = _chi2(ia.image[0] / m, ia.image_w2[0] / m ** 2, ib.image[0] / m, ib.image_w2[0] / m ** 2)
    assert ndf > 50
    assert abs(chi2 - ndf) / np.sqrt(2.0 * ndf) < 5.0, (chi2, ndf)
    ca, cb = ia.counters[0], ib.counters[0]
    assert abs(ca["sum_w"] - cb["sum_w"]) < 5.0 * np.sqrt(ca["sum_w2"] + cb["sum_w2"])
    assert ca["n_rays"] == cb["n_rays"] == m and sum(cb["n_exit"].values()) == m

