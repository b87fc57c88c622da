"""sart_update_setup against a fresh handle: a handle created with setup A and moved to setup B traces what a handle created
with B traces, in every precision mode. The update keeps the tables of sart_create and rewrites in place what depends on
the setup: the shell records (a detector position change moves the shells' focal plane) and, of the reflectivity table
of the throughput pipelines, only the X-ray source's row (a source energy change).

Both handles trace the same global rays with the same compaction, so the integer counters are identical; the image and
the sums agree to 1e-12 relative (only the order of the atomic f64 additions differs)."""
import numpy as np
import pytest

from helpers import make_config
from solaraxionraytracing_b200 import abi

pytestmark = pytest.mark.gpu
SEED = 299792458
N = 2_000_000
INT_KEYS = ("n_rays", "n_passed", "n_passed_till_window", "n_hit_nickel", "n_interp_clamped", "n_retraced", "n_unresolved",
            "n_exit")


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


def _copy(setup):
    return abi.Setup.from_buffer_copy(bytes(setup))


def _case(name):
    """(setup A, setup B, tables, compaction)"""
    if name == "detector_distance":
        a, tb = make_config("cast_llnl")
        b = _copy(a)
        b.detectorInstall.distanceDetectorXRT += 5.0   # mm: defocuses the spot
        return a, b, tb, 0
    a, tb = make_config("babyiaxo_xmm", flags=abi.CF_XRAY_TEST)
    a.testSource.energy = 3.0
    b = _copy(a)
    b.testSource.energy = 5.0
    return a, b, tb, 1


def _run(tr, mode, compact):
    tr.set_precision(mode)
    tr.set_compaction(compact)
    tr.reset_image()
    tr.trace_mc(N, SEED)
    return tr.read_image()


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("case", ["detector_distance", "xray_energy"])
def test_updated_handle_traces_like_fresh_one(rt, case, mode):
    a, b, tb, compact = _case(case)
    with rt.RayTracer(rt.FullRaytraceSetup(a, tb)) as upd, rt.RayTracer(rt.FullRaytraceSetup(b, tb)) as fresh:
        before = _run(upd, mode, compact)
        upd.update_setup(b)
        ru, rf = _run(upd, mode, compact), _run(fresh, mode, compact)
    cu, cf = ru.counters[0], rf.counters[0]
    assert cf["n_passed"] > 0
    # the change matters: setup A traced on the same rays gives another image
    assert not np.allclose(before.image, rf.image, rtol=1e-6, atol=0)
    for k in INT_KEYS:
        assert cu[k] == cf[k], (k, cu[k], cf[k])
    # sum_x and sum_y are signed: their rounding is bounded by that of the sum of the radii
    scale = 1e-12 * cf["sum_r"]
    for k in ("sum_w", "sum_w2", "sum_r", "sum_x", "sum_y"):
        assert cu[k] == pytest.approx(cf[k], rel=1e-12, abs=scale if k in ("sum_x", "sum_y") else 0), k
    assert np.allclose(ru.image, rf.image, rtol=1e-12, atol=0)
    assert np.allclose(ru.image_w2, rf.image_w2, rtol=1e-12, atol=0)
