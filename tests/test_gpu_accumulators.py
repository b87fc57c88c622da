"""Lifecycle of a handle's optional accumulators (the radial histogram, the spectra and the per-mass spectra) and of their
merged copies (sart_allreduce_outputs on a one-rank communicator): switching one of them on again, off or to another size
leaves the others and their merged copies bit for bit as they were, sart_reset_image clears every accumulator of the
handle and no merged copy, and a handle with its accumulators on and merged gives its device memory back when destroyed."""
import numpy as np
import pytest
# before libsart loads NCCL at its first communicator: then both use torch's copy (csrc/comm.cu), while another NCCL
# loaded first can keep torch from importing in this process, here and in every later test module
import torch

from helpers import make_config
from solaraxionraytracing_b200 import multi_gpu

pytestmark = pytest.mark.gpu
SEED = 299792458
MASSES = np.array([0.004, 0.0082, 0.02])
SPECTRA_FIELDS = ("sum_w", "sum_w2", "counts", "shell_sum_w", "shell_counts")
ERR_ARG = -1


@pytest.fixture(scope="module")
def rt():
    from solaraxionraytracing_b200 import raytracer
    if raytracer.lib.sart_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu-marked tests need a B200")
    return raytracer


@pytest.fixture(scope="module")
def fs(rt):
    setup, tb = make_config("cast_llnl")
    return rt.FullRaytraceSetup(setup, tb)


def _read(tr, kind, merged):
    """The arrays of one accumulator, the handle's own or its merged copy, as a list of numpy arrays."""
    if kind == "radial":
        return list((tr.read_merged_radial_hist if merged else tr.read_radial_hist)()[1:])
    if kind == "spectra":
        spectra = [(tr.read_merged_spectra if merged else tr.read_spectra)()]
    else:
        spectra = (tr.read_merged_mass_spectra if merged else tr.read_mass_spectra)()
    return [getattr(s, f) for s in spectra for f in SPECTRA_FIELDS]


def _bits(arrays):
    return [a.tobytes() for a in arrays]


def _traced_and_merged(rt, fs, kinds):
    """A handle with the radial histogram and the spectra (one mass) or the per-mass spectra (MASSES) on, after a traced
    run and a merge."""
    tr = rt.RayTracer(fs, 0)
    tr.set_precision(2)
    if "mass" in kinds:
        tr.set_axion_masses(MASSES)
        tr.enable_mass_spectra()
    else:
        tr.enable_spectra()
    tr.enable_radial_hist()
    multi_gpu.comm_init_all([tr])
    tr.reset_image()
    tr.trace_mc(2_000_000, SEED)
    multi_gpu.allreduce_outputs([tr])
    for k in kinds:
        assert any(a.any() for a in _read(tr, k, False)), k
    return tr


SWITCHES = {   # (accumulator switched, what is done to it) -> the call
    ("radial", "resize"): lambda tr: tr.enable_radial_hist(8192),
    ("radial", "off"): lambda tr: tr.enable_radial_hist(0),
    ("spectra", "again"): lambda tr: tr.enable_spectra(),
    ("spectra", "off"): lambda tr: tr.enable_spectra(False),
    ("mass", "again"): lambda tr: tr.enable_mass_spectra(),
    ("mass", "off"): lambda tr: tr.enable_mass_spectra(False),
}


@pytest.mark.parametrize("others", [("spectra",), ("mass",)], ids=["one-mass", "3-masses"])
@pytest.mark.parametrize("switched,how", [("radial", "resize"), ("radial", "off"), ("spectra", "again"),
                                          ("spectra", "off")])
def test_switching_one_accumulator_leaves_the_others(rt, fs, others, switched, how):
    """After a merge, one accumulator is switched: the other one and its merged copy read back bit-identical, the switched
    one has no merged copy (SART_ERR_ARG), and switched on it starts from zero. In the 3-mass run the per-mass spectra
    take the place of the spectra."""
    if switched == "spectra":
        switched = others[0]
    kinds = ("radial",) + others
    tr = _traced_and_merged(rt, fs, kinds)
    try:
        kept = [k for k in kinds if k != switched]
        before = {(k, m): _bits(_read(tr, k, m)) for k in kept for m in (False, True)}
        SWITCHES[(switched, how)](tr)
        for key, bits in before.items():
            assert _bits(_read(tr, *key)) == bits, key
        with pytest.raises(rt.SartError) as e:
            _read(tr, switched, True)
        assert e.value.code == ERR_ARG
        if how != "off":
            own = _read(tr, switched, False)
            assert own and not any(a.any() for a in own)
            if switched == "radial":
                assert own[0].size == 8192
        else:
            with pytest.raises(rt.SartError) as e:
                _read(tr, switched, False)
            assert e.value.code == ERR_ARG
    finally:
        tr.close()


@pytest.mark.parametrize("others", [("spectra",), ("mass",)], ids=["one-mass", "3-masses"])
def test_reset_image_clears_own_accumulators_not_merged_copies(rt, fs, others):
    kinds = ("radial",) + others
    tr = _traced_and_merged(rt, fs, kinds)
    try:
        merged = {k: _bits(_read(tr, k, True)) for k in kinds}
        tr.reset_image()
        for k in kinds:
            assert not any(a.any() for a in _read(tr, k, False)), k
            assert _bits(_read(tr, k, True)) == merged[k], k
    finally:
        tr.close()


def test_create_and_destroy_returns_device_memory(rt, fs):
    """20 handles, each with the radial histogram and the spectra on, merged, then the spectra off and the per-mass spectra
    of 3 masses on, merged again, then destroyed: the device's free memory comes back to within 1 MiB. Measured after one
    such cycle, which loads the kernels and whatever NCCL sets up once per process."""
    def cycle():
        tr = _traced_and_merged(rt, fs, ("radial", "spectra"))
        try:
            tr.enable_spectra(False)
            tr.set_axion_masses(MASSES)
            tr.enable_mass_spectra()
            tr.trace_mc(2_000_000, SEED)
            multi_gpu.allreduce_outputs([tr])
            assert len(tr.read_merged_mass_spectra()) == MASSES.size
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
