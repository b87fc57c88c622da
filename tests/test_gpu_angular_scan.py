"""sart_angular_scan / performAngularScan (src/raytracer.nim:2778-2815): batched scan of telescope_turned_y.

  * the batched scan equals a loop of sart_update_setup + sart_trace_mc over the same global rays (counters identical,
    fluxes to 1e-12: only the order of the atomic f64 additions differs);
  * in exact mode every scan point has the oracle's exit-code histogram for the rotated setup (bit-exact classification);
  * the vignetting curve of the XMM optic agrees with the McXtrace simulation the reference overlays on its own scan
    (resources/McXtrace_angular_xmm.csv, the only externally pinned full-run curve): |relative flux - McXtrace| <= 0.09
    at each of its 14 angles, 1.000 at 0 deg falling to ~0.5 at 0.3 deg. The chip is enlarged to 100 mm for this
    comparison: on the reference's 14 mm chip the focal spot (7500 mm focal length) leaves the chip beyond 0.05 deg."""
import copy
from pathlib import Path

import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import abi, tables

pytestmark = pytest.mark.gpu
SEED = 299792458
GOLDEN = Path(__file__).resolve().parent / "golden"


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


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_scan_equals_loop_of_runs(rt, mode):
    """Mode 2: a scan point keeps the handle's error budgets (latA / detA doubled for a turned frame), sart_update_setup
    derives them for the turned setup, so a few rays are re-traced in FP64 in one run and kept in FP32 in the other. Their
    classification is the same either way (DESIGN.md section 3b), so the integer counters are identical. What such a ray
    adds differs by the FP32 / FP64 agreement of section 3b: weights 99 % within 2e-4 relative, positions ~1e-4 mm, which
    can move a ray into the neighbouring image bin. At most the 2.4e-3 of the rays that are re-traced on BabyIAXO+XMM
    differ: 2.4e-3 x 2e-4 ~ 5e-7 of the flux, checked at 1e-5; a ray in another bin counts twice its weight in the L1
    distance of the images, at most 2 x 2.4e-3 of the image's sum, checked at 5e-3."""
    setup, tb = make_config("babyiaxo_xmm")
    angles = np.array([0.0, 0.02, 0.05, -0.03])
    n = 400_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(mode)
        fl, cnt, img = tr.angular_scan(angles, n, SEED, want_images=True, first_ray=7 * n)
        for i, a in enumerate(angles):
            tr.update_setup(_turned(setup, a))
            tr.set_precision(mode)
            tr.reset_image()
            tr.trace_mc(n, SEED, first_ray=(7 + i) * n)
            res = tr.read_image()
            c = res.counters[0]
            assert c["n_exit"] == cnt[i]["n_exit"] and c["n_passed"] == cnt[i]["n_passed"]
            if mode == 2:
                assert c["n_passed_till_window"] == cnt[i]["n_passed_till_window"]
                assert c["sum_w"] == pytest.approx(fl[i], rel=1e-5)
                assert np.abs(res.image[0] - img[i]).sum() <= 5e-3 * img[i].sum()
            else:
                assert c["sum_w"] == pytest.approx(fl[i], rel=1e-12)
                assert np.allclose(res.image[0], img[i], rtol=1e-10, atol=0)
    assert fl[0] > fl[2] > 0


def test_exact_scan_points_match_oracle(rt, oracle):
    setup, tb = make_config("babyiaxo_xmm")
    angles = np.array([0.0, 0.04, 0.1])
    n = 30_000
    with rt.RayTracer(rt.FullRaytraceSetup(setup, tb)) as tr:
        tr.set_precision(0)
        fl, cnt, _ = tr.angular_scan(angles, n, SEED)
    for i, a in enumerate(angles):
        _, _, oc = oracle.trace_mc(_turned(setup, a), tb, i * n, n, SEED)
        assert cnt[i]["n_exit"] == oc[0]["n_exit"], (a, cnt[i]["n_exit"], oc[0]["n_exit"])
        assert fl[i] == pytest.approx(oc[0]["sum_w"], rel=1e-9)


def test_xmm_vignetting_against_mcxtrace(rt):
    curves = np.load(GOLDEN / "angular_scan_reference_curves.npz")
    angles, mcx = curves["mcxtrace_angle_deg"], curves["mcxtrace_rel"]
    assert angles[0] == 0.0 and mcx[0] == 1.0 and mcx[-1] == pytest.approx(0.5477)
    flags = rt.flags_from_cli(xrayTest=True, ignoreDetWindow=True, ignoreGasAbs=True, ignoreConvProb=True)
    setup = rt.newExperimentSetup("BabyIAXO", "InGridIAXO", "vacuum", "XMM", flags)
    setup.testSource.parallel = 1
    setup.consts.chipXMax = setup.consts.chipYMax = 100.0
    em = tables.synthetic_emission(64, 64, "primakoff")     # unused by the X-ray source, required by the table struct
    rc, dc = rt.buildCdfs(em)
    tb = tables.TableSet(energies=em.energies, fluxRadiusCDF=rc, diffFluxCDFs=dc,
                         reflectivity=tables.gold_reflectivity_packaged(), **tables.detector_tables_packaged())
    fs = rt.FullRaytraceSetup(setup, tb)
    out = {}
    for mode in (1, 0):
        with rt.RayTracer(fs) as tr:
            tr.set_precision(mode)
            _, rel, _ = rt.performAngularScan(fs, 0.0, 0.3, 14, nRays=2_000_000, tracer=tr)
            fl, _, _ = tr.angular_scan(angles, 2_000_000, SEED)
        rel_m = fl / fl.max()
        out[mode] = rel_m
        assert rel_m[0] == 1.0
        assert np.all(np.diff(rel_m) < 0), rel_m                      # vignetting grows monotonically
        assert np.max(np.abs(rel_m - mcx)) <= 0.09, np.abs(rel_m - mcx).max()
        assert 0.42 < rel_m[-1] < 0.55
        assert rel[0] == 1.0 and 0.42 < rel[-1] < 0.55                 # the linspace(0, 0.3, 14) driver
    assert np.max(np.abs(out[0] - out[1])) < 5e-3                      # fast vs exact: Monte Carlo noise only
