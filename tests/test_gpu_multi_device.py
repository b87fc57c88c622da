"""Merging the optional accumulators of a fused run over GPUs (sart_allreduce_outputs and the sart_read_merged_* readers)
and the command line's --devices: a one-rank merge is a copy of the handle's own accumulators, a run sharded over the
visible GPUs (up to 8) equals one GPU tracing the same global rays, and --devices writes the files --device 0 writes."""
import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import multi_gpu, output

pytestmark = pytest.mark.gpu
SEED = 299792458
MASSES = np.array([0.004, 0.008, 0.0082, 0.0085, 0.02])
SPECTRA_FIELDS = ("sum_w", "sum_w2", "counts", "shell_sum_w", "shell_counts")
ERR_ARG, ERR_CONFIG = -1, -3


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


def _gpus(rt):
    n = min(8, rt.lib.sart_device_count())
    if n < 2:
        pytest.skip(f"needs at least 2 GPUs, {n} visible")
    return n


def _spectra_equal(a, b):
    for f in SPECTRA_FIELDS:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f


def _hist_equal(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_one_rank_merge_is_a_copy(rt):
    """One handle, its own communicator: the merged radial histogram and spectra equal the handle's own; a second merge
    without a reset gives the same (the handle's accumulators are untouched), and so does one after sart_reset_image."""
    setup, tb = make_config("cast_llnl")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb), 0) as tr:
        tr.set_precision(2)
        tr.enable_radial_hist()
        tr.enable_spectra()
        multi_gpu.comm_init_all([tr])
        tr.reset_image()
        tr.trace_mc(3_000_000, SEED)
        for read in (tr.read_merged_radial_hist, tr.read_merged_spectra):   # before any merge
            with pytest.raises(rt.SartError) as e:
                read()
            assert e.value.code == ERR_ARG
        multi_gpu.allreduce_outputs([tr])
        hist, spec = tr.read_radial_hist(), tr.read_spectra()
        assert spec.counts.sum() > 0 and hist[2].sum() > 0
        _hist_equal(tr.read_merged_radial_hist(), hist)
        _spectra_equal(tr.read_merged_spectra(), spec)
        tr.allreduce_outputs()   # the per-rank form, again without a reset
        _hist_equal(tr.read_merged_radial_hist(), hist)
        _spectra_equal(tr.read_merged_spectra(), spec)
        tr.reset_image()         # leaves the merged copies readable
        _spectra_equal(tr.read_merged_spectra(), spec)
        tr.enable_spectra()      # switching on again invalidates the merged spectra, not the merged histogram
        with pytest.raises(rt.SartError, match="no merged spectra") as e:
            tr.read_merged_spectra()
        assert e.value.code == ERR_ARG
        _hist_equal(tr.read_merged_radial_hist(), hist)
        tr.enable_spectra(False)
        tr.enable_radial_hist(0)
        with pytest.raises(rt.SartError, match="no radial histogram, spectra or per-mass spectra") as e:
            tr.allreduce_outputs()
        assert e.value.code == ERR_ARG
        with pytest.raises(rt.SartError):
            tr.read_merged_radial_hist()


def test_one_rank_merge_of_mass_spectra(rt):
    """The same with 5 masses and the per-mass spectra."""
    setup, tb = make_config("cast_llnl")
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb), 0) as tr:
        tr.set_precision(2)
        tr.set_axion_masses(MASSES)
        tr.enable_mass_spectra()
        multi_gpu.comm_init_all([tr])
        tr.reset_image()
        tr.trace_mc(3_000_000, SEED)
        with pytest.raises(rt.SartError) as e:
            tr.read_merged_mass_spectra()
        assert e.value.code == ERR_ARG
        own = tr.read_mass_spectra()
        assert len(own) == 5 and all(s.counts.sum() > 0 for s in own)
        for _ in range(2):
            multi_gpu.allreduce_outputs([tr])
            merged = tr.read_merged_mass_spectra()
            assert len(merged) == 5
            for a, b in zip(merged, own):
                _spectra_equal(a, b)
        tr.set_axion_masses(MASSES[:3])   # another number of masses invalidates the merged rows
        with pytest.raises(rt.SartError) as e:
            tr.read_merged_mass_spectra()
        assert e.value.code == ERR_ARG


def _single_gpu(rt, fs, n, mode, masses=None):
    """The reference: one GPU traces all n rays."""
    with rt.RayTracer(fs, 0) as tr:
        tr.set_precision(mode)
        if masses is not None:
            tr.set_axion_masses(masses)
            tr.enable_mass_spectra()
        else:
            tr.enable_radial_hist()
            tr.enable_spectra()
        tr.reset_image()
        tr.trace_mc(n, SEED)
        res = tr.read_image()
        if masses is not None:
            return res, None, tr.read_mass_spectra()
        return res, tr.read_radial_hist(), tr.read_spectra()


def _close(a, b):
    assert np.allclose(a, b, rtol=1e-12, atol=0), np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


def _same_run(multi, single):
    res, hist, spec = single
    for cm, cs in zip(multi.result.counters, res.counters):
        for k, v in cs.items():
            if isinstance(v, float):
                assert cm[k] == pytest.approx(v, rel=1e-12), k
            else:
                assert cm[k] == v, k
    assert np.allclose(multi.result.image, res.image, rtol=1e-10, atol=0)   # per bin: only the order of the adds differs
    if hist is not None:
        assert np.array_equal(multi.radial_hist[2], hist[2])
        _close(multi.radial_hist[1], hist[1])
    for m, s in zip(multi.spectra if isinstance(spec, list) else [multi.spectra], spec if isinstance(spec, list) else [spec]):
        assert np.array_equal(m.counts, s.counts) and np.array_equal(m.shell_counts, s.shell_counts)
        for f in ("sum_w", "sum_w2", "shell_sum_w"):
            _close(getattr(m, f), getattr(s, f))


@pytest.mark.parametrize("mode,n", [(2, 100_000_000), (0, 1_000_000)])
def test_sharded_run_equals_one_gpu(rt, mode, n):
    """Radial histogram + spectra of a run sharded over the GPUs: every count identical to one GPU tracing the same
    global rays, every sum within 1e-12 (only the order of summation differs)."""
    ng = _gpus(rt)
    setup, tb = make_config("cast_llnl")
    fs = rt.FullRaytraceSetup(setup, tb)
    multi = multi_gpu.trace_on_devices(fs, list(range(ng)), n, SEED, precision=mode, radial_hist=True, spectra=True)
    assert multi.precision == mode and multi.result.counters[0]["n_rays"] == n
    _same_run(multi, _single_gpu(rt, fs, n, mode))


@pytest.mark.parametrize("mode,n", [(2, 100_000_000), (0, 1_000_000)])
def test_sharded_mass_scan_equals_one_gpu(rt, mode, n):
    """The same for 5 masses and the per-mass spectra."""
    ng = _gpus(rt)
    setup, tb = make_config("cast_llnl")
    fs = rt.FullRaytraceSetup(setup, tb)
    multi = multi_gpu.trace_on_devices(fs, list(range(ng)), n, SEED, precision=mode, masses=MASSES, spectra=True)
    assert len(multi.spectra) == 5 and multi.radial_hist is None
    _same_run(multi, _single_gpu(rt, fs, n, mode, MASSES))


def test_in_process_mismatch_is_refused_on_the_host(rt):
    """Spectra on for handle 0 and off for handle 1: SART_ERR_CONFIG before any collective, after which an agreeing call
    goes through (nothing was left waiting in NCCL)."""
    _gpus(rt)
    setup, tb = make_config("cast_llnl")
    fs = rt.FullRaytraceSetup(setup, tb)
    with rt.RayTracer(fs, 0) as t0, rt.RayTracer(fs, 1) as t1:
        multi_gpu.comm_init_all([t0, t1])
        t0.enable_spectra()
        with pytest.raises(rt.SartError, match="differ") as e:
            multi_gpu.allreduce_outputs([t0, t1])
        assert e.value.code == ERR_CONFIG
        t1.enable_spectra()
        for k, t in enumerate((t0, t1)):
            t.trace_mc(1_000_000, SEED, first_ray=k * 1_000_000)
        multi_gpu.allreduce_outputs([t0, t1])
        a, b = t0.read_spectra(), t1.read_spectra()
        m = t1.read_merged_spectra()
        assert np.array_equal(m.counts, a.counts + b.counts)


# -- the command line


def _cli(tmp_path, name, args, cfg):
    from solaraxionraytracing_b200.__main__ import main
    out = tmp_path / name
    assert main(["--config", str(cfg), "--outputPath", str(out), "--allowSynthetic", "--seed", "11", *args]) == 0
    return out


def _config(tmp_path, extra=""):
    from solaraxionraytracing_b200 import config
    cfg = tmp_path / "config.toml"
    txt = config.DEFAULT_CONFIG.read_text()
    if extra:
        txt = txt.replace('stageSetup = "vacuum"', 'stageSetup = "gas"') + extra
    cfg.write_text(txt)
    return cfg


def _same_csv(a, b, ints):
    ca, cb = output.read_columns_csv(a), output.read_columns_csv(b)
    assert list(ca) == list(cb)
    for name in ca:
        if name in ints:
            assert np.array_equal(ca[name], cb[name]), (a.name, name)
        else:
            scale = np.nanmax(np.abs(cb[name])) if np.isfinite(cb[name]).any() else 0.0
            assert np.allclose(ca[name], cb[name], rtol=1e-12, atol=1e-12 * scale, equal_nan=True), (a.name, name)


def _same_files(multi, single):
    names = sorted(p.name for p in single.iterdir())
    assert names == sorted(p.name for p in multi.iterdir())
    for name in names:
        if name.endswith(".npy"):
            assert np.allclose(np.load(multi / name), np.load(single / name), rtol=1e-12, atol=0)
        elif name.startswith("axion_image_"):
            _same_csv(multi / name, single / name, {"x", "y"})
        else:
            _same_csv(multi / name, single / name, {"rays", "shell"})
    return names


@pytest.mark.parametrize("devices", ["all", "0"])
def test_command_line_devices_single_mass(rt, tmp_path, devices):
    """--devices writes the image CSV (radii from the merged radial histogram) and the spectra CSVs of --device 0."""
    cfg = _config(tmp_path)
    args = ["--nRays", "3000000", "--writeSpectra"]
    single = _cli(tmp_path, "single", args, cfg)
    multi = _cli(tmp_path, "multi", [*args, "--devices", devices], cfg)
    names = _same_files(multi, single)
    assert len(names) == 3 and any(n.startswith("axion_image_") for n in names)


def test_command_line_devices_mass_scan(rt, tmp_path):
    """A 3-mass scan from a config file: the per-mass images and per-mass spectra CSVs of --device 0."""
    cfg = _config(tmp_path, "\n[Run]\nmAxion = [0.006, 0.0082, 0.02]\n")
    args = ["--nRays", "3000000", "--writeSpectra"]
    single = _cli(tmp_path, "single", args, cfg)
    multi = _cli(tmp_path, "multi", [*args, "--devices", "all"], cfg)
    names = _same_files(multi, single)
    assert "axion_images_mass_scan.npy" in names and len(names) == 7


def test_command_line_devices_angular_scan(rt, tmp_path):
    """An angular scan dealt over the devices gives the relative fluxes of --device 0 to 1e-12 per point."""
    cfg = _config(tmp_path)
    args = ["--nRays", "500000", "--angularScanMin", "0", "--angularScanMax", "0.1", "--numAngularScanPoints", "7"]
    single = _cli(tmp_path, "single", args, cfg)
    multi = _cli(tmp_path, "multi", [*args, "--devices", "all"], cfg)
    a = np.loadtxt(multi / "angular_scan_telescope_y.csv", delimiter=",", skiprows=1)
    b = np.loadtxt(single / "angular_scan_telescope_y.csv", delimiter=",", skiprows=1)
    assert a.shape == b.shape == (7, 2)
    assert np.array_equal(a[:, 0], b[:, 0])
    assert np.allclose(a[:, 1], b[:, 1], rtol=1e-12, atol=0)
