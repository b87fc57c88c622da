"""Sharding of one Monte Carlo run over the GPUs of a box: one process per GPU, torch.distributed for the plumbing.

Rays are independent and ray i depends only on (seed, i) (Philox counter = global ray index), so the run is cut into
contiguous index ranges, one per rank, with no data-path exchange; the only collective is the final sum of the
detector image, the sum-of-squares image and the counters (512 KiB + 512 KiB + 224 B per axion mass) — one
all-reduce over NVLink (NCCL) on the device buffers libsart exposes. The reference's only parallel construct is the
Weave parallelFor over rays inside one process (src/raytracer.nim:2234-2244).

One process can also drive several GPUs itself (trace_on_devices, angular_scan_on_devices, angular_scan_outputs_on_devices):
one RayTracer per device,
one NCCL communicator over all of them (sart_comm_init_all), and the same collectives behind the C-ABI, which then take
every handle of the process in one call.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass

import numpy as np

from . import abi
from ._lib import check, lib
from .output import BandImages, QuantityHist, ScanOutputs, Spectra, concat_scan_outputs


def shard(n_rays: int, rank: int, world: int, first_ray: int = 0) -> tuple[int, int]:
    """Contiguous, balanced partition of [first_ray, first_ray + n_rays): returns (first, count) of `rank`."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, rem = divmod(n_rays, world)
    count = base + (1 if rank < rem else 0)
    first = first_ray + rank * base + min(rank, rem)
    return first, count


N_COUNTER_WORDS = C.sizeof(abi.Counters) // 8
N_COUNTER_INTS = abi.Counters.sum_w.offset // 8     # the leading u64 fields; the rest are f64 sums


def counters_to_arrays(counters: list[dict]) -> tuple[np.ndarray, np.ndarray]:
    """Counter dicts (one per axion mass) -> (int64 [M, n_int], float64 [M, n_float]) in struct order."""
    ints, flts = [], []
    for c in counters:
        ex = [c["n_exit"].get(name, 0) for name in abi.EXIT_NAMES] + [0] * (16 - abi.N_EXIT_CODES)
        ints.append([c["n_rays"], *ex, c["n_passed"], c["n_passed_till_window"], c["n_hit_nickel"],
                     c["n_interp_clamped"], c.get("n_retraced", 0), c.get("n_unresolved", 0)])
        flts.append([c["sum_w"], c["sum_w2"], c["sum_x"], c["sum_y"], c["sum_r"]])
    return np.asarray(ints, dtype=np.int64), np.asarray(flts, dtype=np.float64)


def arrays_to_counters(ints: np.ndarray, flts: np.ndarray) -> list[dict]:
    out = []
    for i, f in zip(ints, flts):
        d = {"n_rays": int(i[0]), "n_exit": {name: int(i[1 + k]) for k, name in enumerate(abi.EXIT_NAMES)},
             "n_passed": int(i[17]), "n_passed_till_window": int(i[18]), "n_hit_nickel": int(i[19]),
             "n_interp_clamped": int(i[20]), "n_retraced": int(i[21]), "n_unresolved": int(i[22]), "sum_w": float(f[0]), "sum_w2": float(f[1]), "sum_x": float(f[2]),
             "sum_y": float(f[3]), "sum_r": float(f[4])}
        out.append(d)
    return out


def merge_host(image: np.ndarray, image_w2: np.ndarray, counters: list[dict], group=None):
    """All-reduce(sum) of host-side results over `group` (any torch.distributed backend; gloo on CPU).
    Returns (image, image_w2, counters) holding the whole run on every rank."""
    import torch
    import torch.distributed as dist
    ints, flts = counters_to_arrays(counters)
    t_img, t_img2 = torch.from_numpy(np.ascontiguousarray(image)), torch.from_numpy(np.ascontiguousarray(image_w2))
    t_i, t_f = torch.from_numpy(ints), torch.from_numpy(flts)
    for t in (t_img, t_img2, t_i, t_f):
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t_img.numpy(), t_img2.numpy(), arrays_to_counters(t_i.numpy(), t_f.numpy())


def comm_init(tracer, rank: int, world: int, device: int, group=None):
    """Gives `tracer` its NCCL communicator (sart_comm_init_rank): rank 0 draws the 128-byte NCCL id and broadcasts it
    over the already initialised torch.distributed group — the only thing torch ships; the collective itself is
    sart_allreduce behind the C-ABI."""
    import torch
    import torch.distributed as dist
    uid = torch.zeros(abi.COMM_ID_BYTES, dtype=torch.uint8)
    if rank == 0:
        uid = torch.frombuffer(bytearray(tracer.comm_unique_id()), dtype=torch.uint8).clone()
    if dist.get_backend(group) == "nccl":
        uid = uid.to(f"cuda:{device}")
    dist.broadcast(uid, src=0, group=group)
    tracer.comm_init_rank(world, rank, bytes(uid.cpu().numpy().tobytes()))


class _DevArray:
    def __init__(self, ptr: int, n: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def device_views(tracer, device: int):
    """Zero-copy torch views of a RayTracer's device-resident image, w^2 image and counters (ints, floats)."""
    import torch
    img, img2, n = tracer.image_dev()
    m = tracer.n_masses
    dev = f"cuda:{device}"
    cnt = tracer.counters_dev()
    views = [torch.as_tensor(_DevArray(img, n, "<f8"), device=dev), torch.as_tensor(_DevArray(img2, n, "<f8"), device=dev)]
    if m == 1:
        views.append(torch.as_tensor(_DevArray(cnt, N_COUNTER_INTS, "<i8"), device=dev))
        views.append(torch.as_tensor(_DevArray(cnt + 8 * N_COUNTER_INTS, N_COUNTER_WORDS - N_COUNTER_INTS, "<f8"), device=dev))
    else:
        # interleaved int/float words per mass: reduce each mass record's two halves separately
        for k in range(m):
            base = cnt + k * 8 * N_COUNTER_WORDS
            views.append(torch.as_tensor(_DevArray(base, N_COUNTER_INTS, "<i8"), device=dev))
            views.append(torch.as_tensor(_DevArray(base + 8 * N_COUNTER_INTS, N_COUNTER_WORDS - N_COUNTER_INTS, "<f8"), device=dev))
    return views


def allreduce_device(tracer, device: int, group=None, views=None):
    """One NCCL all-reduce(sum) per buffer on the tracer's stream (call inside `torch.cuda.stream(ext_stream)`)."""
    import torch.distributed as dist
    for t in (views or device_views(tracer, device)):
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


def calculateFluxFractionsSharded(raytraceSetup, nRays: int, seed: int = 299792458, device: int | None = None,
                                  group=None):
    """calculateFluxFractions (rt:2755-2776) over all ranks of an initialised torch.distributed NCCL group: every
    rank traces its shard on its GPU, the images are summed with one all-reduce, every rank returns the full result."""
    import torch
    import torch.distributed as dist
    from . import raytracer as rt
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    device = torch.cuda.current_device() if device is None else device
    first, count = shard(nRays, rank, world)
    with rt.RayTracer(raytraceSetup, device) as tr:
        for mode in (2, 1):      # the fastest pipeline this setup supports; precision 0 otherwise
            try:
                tr.set_precision(mode)
                break
            except rt.SartError:
                pass
        comm_init(tr, rank, world, device, group)
        tr.reset_image()
        tr.trace_mc(count, seed, first_ray=first)
        tr.allreduce()
        return tr.read_merged()


# -- one process, n GPUs: NCCL needs every handle of the process in one call (RayTracer.allreduce is the per-rank form)
def _handles(tracers):
    return (abi.H * len(tracers))(*[t._h for t in tracers])


def comm_init_all(tracers):
    """One NCCL communicator over `tracers`, each on its own device (sart_comm_init_all); rank i = tracers[i]."""
    check(lib.sart_comm_init_all(_handles(tracers), len(tracers)))


def allreduce(tracers):
    """sart_allreduce over every tracer of comm_init_all: image, w^2 image and counters into each one's read_merged()."""
    check(lib.sart_allreduce(_handles(tracers), len(tracers)))


def allreduce_outputs(tracers):
    """sart_allreduce_outputs over every tracer of comm_init_all: the accumulators that are on (radial histogram, spectra,
    band images, quantity histograms and their per-mass forms), into each one's read_merged_* readers. Synchronises."""
    check(lib.sart_allreduce_outputs(_handles(tracers), len(tracers)))


@dataclass
class DevicesResult:
    """A fused run traced on several GPUs and merged over them."""
    result: object                          # raytracer.RunResult: image, w^2 image and counters of the whole run
    radial_hist: tuple | None               # (bin edges, sum of weights, counts) as RayTracer.read_radial_hist
    spectra: Spectra | list[Spectra] | None  # one Spectra (at most one mass) or one per mass (a mass scan)
    precision: int                           # the precision mode the run took
    band_images: BandImages | None = None    # the band images of `bands` (RayTracer.read_band_images)
    quantity_hists: list[QuantityHist] | None = None   # the histograms of `quantity_hists` (RayTracer.read_quantity_hists)
    mass_radial_hists: list[tuple] | None = None        # per mass, as RayTracer.read_mass_radial_hist
    mass_band_images: list[BandImages] | None = None    # per mass, the band images of `mass_bands`


def _open_tracers(fullSetup, devices, precision: int, sampler, masses, warn):
    """One RayTracer per device, configured as the command line configures one: the fastest precision mode up to
    `precision` the setup supports (decided on the first device), the sampler and the axion masses."""
    from . import raytracer as rt
    if not devices or len(set(devices)) != len(devices):
        raise ValueError(f"need distinct devices, got {list(devices)}")
    tracers = []
    try:
        for d in devices:
            tracers.append(rt.RayTracer(fullSetup, d))
        mode = rt.set_fastest_precision(tracers[0], precision, warn)
        for t in tracers:
            t.set_precision(mode)
            if sampler is not None:
                t.set_sampler(sampler)
            if masses is not None and len(masses):
                t.set_axion_masses(masses)
    except BaseException:
        for t in tracers:
            t.close()
        raise
    return tracers, mode


def trace_on_devices(fullSetup, devices, nRays: int, seed: int = 299792458, *, precision: int = 2, sampler=None,
                     masses=None, radial_hist: bool = False, spectra: bool = False, bands=None, quantity_hists=None,
                     mass_radial_hist: bool = False, mass_bands=None, warn=None) -> DevicesResult:
    """The fused run of `nRays` rays over `devices`, one process: device k traces shard(nRays, k, n) of the global rays,
    so the result is that of one GPU tracing all of them, up to the order of the floating-point sums. The shards run
    concurrently (trace_mc only queues work); then sart_allreduce and, with `radial_hist` or `spectra`,
    sart_allreduce_outputs merge them. `spectra` means the single-mass spectra for at most one axion mass and the per-mass
    spectra for a mass scan. `bands`: the edges of the band images (RayTracer.enable_band_images; at most one axion
    mass). `quantity_hists`: the specs of the quantity histograms (RayTracer.enable_quantity_hists; at most one axion mass).
    `mass_radial_hist` / `mass_bands` (band edges): the per-mass radial histograms and band images
    (RayTracer.enable_mass_radial_hist / enable_mass_band_images) of a mass scan. `warn` receives the precision fall-back messages (see raytracer.set_fastest_precision)."""
    tracers, mode = _open_tracers(fullSetup, devices, precision, sampler, masses, warn)
    try:
        scan = masses is not None and len(masses) > 1
        for t in tracers:
            if radial_hist:
                t.enable_radial_hist()
            if spectra:
                t.enable_mass_spectra() if scan else t.enable_spectra()
            if bands is not None:
                t.enable_band_images(bands)
            if quantity_hists:
                t.enable_quantity_hists(quantity_hists)
            if mass_radial_hist:
                t.enable_mass_radial_hist()
            if mass_bands is not None:
                t.enable_mass_band_images(mass_bands)
            t.reset_image()
        comm_init_all(tracers)
        for rank, t in enumerate(tracers):
            first, count = shard(nRays, rank, len(tracers))
            if count:
                t.trace_mc(count, seed, first_ray=first)
        allreduce(tracers)
        if radial_hist or spectra or bands is not None or quantity_hists or mass_radial_hist or mass_bands is not None:
            allreduce_outputs(tracers)
        t0 = tracers[0]
        merged_spectra = None
        if spectra:
            merged_spectra = t0.read_merged_mass_spectra() if scan else t0.read_merged_spectra()
        return DevicesResult(t0.read_merged(), t0.read_merged_radial_hist() if radial_hist else None, merged_spectra, mode,
                             t0.read_merged_band_images() if bands is not None else None,
                             t0.read_merged_quantity_hists() if quantity_hists else None,
                             t0.read_merged_mass_radial_hist() if mass_radial_hist else None,
                             t0.read_merged_mass_band_images() if mass_bands is not None else None)
    finally:
        for t in tracers:
            t.close()


def angular_scan_on_devices(fullSetup, devices, angularScanMin: float, angularScanMax: float,
                            numAngularScanPoints: int = 50, nRays: int = 1_000_000, seed: int = 299792458, *,
                            precision: int = 2, sampler=None, masses=None, warn=None):
    """performAngularScan over `devices` in one process: device k takes the contiguous block shard(points, k, n) of the
    scan points, and scan point i traces the global rays [i*nRays, (i+1)*nRays) as on one GPU. sart_angular_scan blocks,
    so each device runs in its own thread; the fluxes are put together on the host. Returns (angles [deg],
    flux / max flux, fluxes)."""
    angles = np.linspace(angularScanMin, angularScanMax, numAngularScanPoints)
    fluxes = np.zeros(numAngularScanPoints)
    tracers, _ = _open_tracers(fullSetup, devices, precision, sampler, masses, warn)
    errors = []

    def scan(rank, t):
        lo, cnt = shard(numAngularScanPoints, rank, len(tracers))
        try:
            if cnt:
                fluxes[lo:lo + cnt] = t.angular_scan(angles[lo:lo + cnt], nRays, seed, first_ray=lo * nRays)[0]
        except BaseException as e:   # re-raised in the calling thread
            errors.append(e)

    try:
        threads = [threading.Thread(target=scan, args=(k, t)) for k, t in enumerate(tracers)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
    finally:
        for t in tracers:
            t.close()
    if errors:
        raise errors[0]
    return angles, fluxes / fluxes.max(), fluxes


def angular_scan_outputs_on_devices(fullSetup, devices, angularScanMin: float, angularScanMax: float,
                                    numAngularScanPoints: int = 50, nRays: int = 1_000_000, seed: int = 299792458, *,
                                    precision: int = 2, sampler=None, masses=None, radial_hist: bool = True,
                                    spectra: bool = False, bands=None, quantity_hists=None, want_images: bool = False,
                                    warn=None) -> ScanOutputs:
    """RayTracer.angular_scan_outputs over `devices` in one process, scan points dealt as in angular_scan_on_devices
    (device k takes the contiguous block shard(points, k, n), scan point i traces the global rays [i*nRays, (i+1)*nRays)).
    The accumulators `radial_hist`, `spectra` (single-mass), `bands` (band edges) and `quantity_hists` (specs) are switched
    on every device; the blocks of scan points are put together on the host, so the result is that of one GPU."""
    angles = np.linspace(angularScanMin, angularScanMax, numAngularScanPoints)
    tracers, _ = _open_tracers(fullSetup, devices, precision, sampler, masses, warn)
    parts: list[ScanOutputs | None] = [None] * len(tracers)
    errors = []

    def scan(rank, t):
        lo, cnt = shard(numAngularScanPoints, rank, len(tracers))
        try:
            if cnt:
                parts[rank] = t.angular_scan_outputs(angles[lo:lo + cnt], nRays, seed, want_images, first_ray=lo * nRays)
        except BaseException as e:   # re-raised in the calling thread
            errors.append(e)

    try:
        for t in tracers:
            if radial_hist:
                t.enable_radial_hist()
            if spectra:
                t.enable_spectra()
            if bands is not None:
                t.enable_band_images(bands)
            if quantity_hists:
                t.enable_quantity_hists(quantity_hists)
        threads = [threading.Thread(target=scan, args=(k, t)) for k, t in enumerate(tracers)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
    finally:
        for t in tracers:
            t.close()
    if errors:
        raise errors[0]
    return concat_scan_outputs([p for p in parts if p is not None])
