#!/usr/bin/env python
"""bench.py — traced rays/s of the per-ray pipeline on N B200s (BASELINE.json's metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--rays-per-step R] [--precision exact|fast]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...     # the reference's CPU algorithm (restated oracle) on the host cores
  python bench.py ... --dump-outputs DIR   # also writes the last timed step's image and counters as DIR/<name>.npy

Workload (config.workload): BASELINE config "CAST magnet + LLNL telescope, detector chain active
(Si3N4/Al window + Ar), 1e9 rays" — the largest single-GPU configuration of the setup the north-star target is
quoted on. Tables have the reference's shapes (1968x1500 solar model, 4x1000x1000 reflectivity) with synthetic
content (three of the reference's input files are not shipped), detector-chain tables are the reference's own.

A "step" is one fused Monte Carlo pass (Philox sampling -> trace -> weighted 256x256 histogram) over
--rays-per-step rays PER GPU (weak scaling); with N > 1 each step ends with one NCCL all-reduce of the image and the
counters. `value` counts launched rays of all ranks / max-over-ranks device time.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import signal
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SEED = 299792458  # randomize(299792458), raytracer.nim:276
# Algorithmic work per launched ray (SURVEY.md §8a tally x measured stage-reach probabilities, DESIGN.md §5):
# 230 (sampling + bore/pipes + frame) + 70*0.997 (shell scan) + 370*0.936 (two mirror solves + reflections)
# + 223*0.91 (detector plane, angles, weights, histogram) for CAST+LLNL.
F_RAY_LLNL = 850.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rays-per-step", type=float, default=1e9)
    ap.add_argument("--precision", choices=["exact", "fast", "f32"], default=None)
    ap.add_argument("--sampler", choices=["inverse_cdf", "alias"], default="inverse_cdf",
                    help="inverse_cdf: the reference's lowerBound(cdf, u), the same rays as the CPU oracle (default, the "
                         "headline); alias: the same distributions through alias tables (statistical parity only)")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-presampled", action="store_true", help="skip the tier-(a) pre-sampled kernel measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations (2, 4, 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (image, w^2 image, counters) "
                         "as DIR/<name>.npy in float64, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours (the reference arm sizes its steps by its own speed)")
    return args


# ---------------------------------------------------------------------------------------------------------------
def workload_tables(rt, tables, device):
    """Full-size tables of the CAST+LLNL workload; CDFs built on the GPU (sart_build_cdfs)."""
    em = tables.synthetic_emission(1968, 1500, "abc")
    rc, dc = rt.buildCdfs(em, device)
    refl = tables.synthetic_reflectivity(4, 1000, 1000)
    return tables.TableSet(energies=em.energies, fluxRadiusCDF=rc, diffFluxCDFs=dc, reflectivity=refl,
                           **tables.detector_tables_packaged())


def workload_tables_cpu(orc, tables):
    em = tables.synthetic_emission(1968, 1500, "abc")
    rc, dc = orc.build_cdfs(em.radii, em.energies, em.emRates)
    refl = tables.synthetic_reflectivity(4, 1000, 1000)
    return tables.TableSet(energies=em.energies, fluxRadiusCDF=rc, diffFluxCDFs=dc, reflectivity=refl,
                           **tables.detector_tables_packaged())


WORKLOAD = "CAST+LLNL vacuum, InGrid2018 window+Ar chain, solar table 1968x1500, reflectivity 4x1000x1000"


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def cpu_leg(seconds: float, threads: int | None = None):
    """Times the restated CPU oracle (the reference's algorithm; the Nim binary cannot be built in this image) on
    a bounded sample of the same workload. Returns (rays/s, cores, sample description)."""
    from oracle import oracle as orc
    from oracle import ref_setup
    from solaraxionraytracing_b200 import abi, tables
    orc.lib()
    # torchrun exports OMP_NUM_THREADS=1 to every rank: ask for the host's cores explicitly
    cores = threads or host_cores()
    orc.lib().oracle_set_num_threads(cores)
    setup = ref_setup.make_setup(abi.ES_CAST, abi.DK_INGRID2018, abi.SK_VACUUM, abi.TK_LLNL, 0)
    tb = workload_tables_cpu(orc, tables)
    n0 = 200_000
    t0 = time.perf_counter()
    orc.trace_mc(setup, tb, 0, n0, SEED)
    rate = n0 / (time.perf_counter() - t0)
    n = int(max(n0, min(rate * seconds, 5e7)))
    t0 = time.perf_counter()
    _, _, cnt = orc.trace_mc(setup, tb, n0, n, SEED)
    dt = time.perf_counter() - t0
    return n / dt, cores, f"{n} rays of the same workload, OpenMP {cores} threads, {dt:.1f} s", cnt[0], n0, n


def parity_leg(tr, first: int, n: int, cnt_cpu: dict | None = None):
    """bench.py checks what it times: the fused kernel on the global rays [first, first + n) of the workload against the
    CPU oracle on the very same rays (Philox is keyed on the global ray index): exit-code histogram within n/5000 per
    code, total flux within 1e-3. `cnt_cpu`: the oracle's counters if the cpu_baseline leg already traced that range."""
    if cnt_cpu is None:
        from oracle import oracle as orc
        from oracle import ref_setup
        from solaraxionraytracing_b200 import abi, tables
        orc.lib().oracle_set_num_threads(host_cores())
        setup = ref_setup.make_setup(abi.ES_CAST, abi.DK_INGRID2018, abi.SK_VACUUM, abi.TK_LLNL, 0)
        cnt_cpu = orc.trace_mc(setup, workload_tables_cpu(orc, tables), first, n, SEED)[2][0]
    tr.reset_image()
    tr.trace_mc(n, SEED, first_ray=first)
    cg = tr.read_image().counters[0]
    tr.reset_image()
    diff = {k: cg["n_exit"][k] - v for k, v in cnt_cpu["n_exit"].items()}
    tol = max(1, n // 5000)
    flux = abs(cg["sum_w"] / cnt_cpu["sum_w"] - 1.0) if cnt_cpu["sum_w"] else None
    ok = cg["n_rays"] == cnt_cpu["n_rays"] == n and all(abs(d) <= tol for d in diff.values()) and (flux is None or flux < 1e-3)
    return {"ok": bool(ok), "rays": n, "first_ray": first, "tolerance_per_code": tol,
            "exit_code_diff_gpu_minus_cpu": {k: d for k, d in diff.items() if d}, "max_abs_diff": max(abs(d) for d in diff.values()),
            "sum_w_rel_diff": flux, "passed_gpu": cg["n_passed"], "passed_cpu": cnt_cpu["n_passed"],
            "retraced_fp64": cg.get("n_retraced"), "unresolved": cg.get("n_unresolved"),
            "against": "restated CPU oracle on the same Philox rays (not the Nim executable)"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the line-faithful oracle port (kind
    "port"), all host threads, each step a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    from oracle import ref_setup
    from solaraxionraytracing_b200 import abi, tables
    orc.lib()
    # all the host threads the box has: under torchrun (N > 1) every rank inherits OMP_NUM_THREADS=1, which would time
    # the CPU arm on one core
    cores = host_cores()
    orc.lib().oracle_set_num_threads(cores)
    cores = orc.lib().oracle_num_threads()
    setup = ref_setup.make_setup(abi.ES_CAST, abi.DK_INGRID2018, abi.SK_VACUUM, abi.TK_LLNL, 0)
    tb = workload_tables_cpu(orc, tables)
    t0 = time.perf_counter()
    orc.trace_mc(setup, tb, 0, 100_000, SEED)
    rate = 100_000 / (time.perf_counter() - t0)
    total = args.steps + args.warmup
    per_step = int(max(50_000, min(rate * (90.0 / max(1, total)), 2e7)))  # whole run within ~1.5 min
    for w in range(args.warmup):
        orc.trace_mc(setup, tb, w * per_step, per_step, SEED)
    t0 = time.perf_counter()
    for k in range(args.steps):
        orc.trace_mc(setup, tb, (args.warmup + k) * per_step, per_step, SEED)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = f"{per_step} rays/step of the same workload on {cores} host threads (restated oracle, not the Nim executable)"
    print(json.dumps({
        "impl": "reference", "metric": "traced rays/s", "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rays_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        # PR_SET_PDEATHSIG: the sampler gets SIGTERM when bench.py exits, also when it dies before stop()
        libc = C.CDLL(None, use_errno=True)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL,
                                      preexec_fn=lambda: libc.prctl(1, signal.SIGTERM))
        except OSError:
            self.p = None

    def mark(self, name: str):
        """Wall-clock marks ("t0"/"t1") of the timed region, to pick the samples taken inside it."""
        setattr(self, name, time.time())

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        import datetime
        rows = []
        for line in self.f.read().splitlines():
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(p[1]), float(p[2]), p[5:9]))
            except ValueError:
                continue
        os.unlink(self.f.name)
        t0, t1 = getattr(self, "t0", None), getattr(self, "t1", None)
        inside = [r for r in rows if t0 is not None and t1 is not None and t0 - 0.05 <= r[0] <= t1 + 0.05]
        where = "timed region"
        if not inside:
            # region shorter than the sampling period: fall back to the samples under load (upper half by SM clock)
            inside = sorted(rows, key=lambda r: r[1])[len(rows) // 2:]
            where = "whole run, upper half by SM clock (timed region shorter than the 100 ms sampling period)"
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm = [r[1] for r in inside]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max((r[2] for r in rows), default=None),
                "samples": len(inside), "window": where, "reasons": sorted(reasons)}


def alias_leg(tr, torch, stream, flush, R: int, peak_tflops: float, steps: int = 5, warmup: int = 3):
    """The same fused kernel with sart_set_sampler(SART_SAMPLER_ALIAS): emission shell and energy drawn from alias
    tables of the same discrete distributions (one lookup each) instead of the inverse-CDF search. Reported next to the
    headline, not as the headline: its runs agree with the reference statistically (tier b: tests/test_gpu_f32.py), but
    a (seed, index) pair no longer denotes the ray it denotes in the CPU oracle."""
    from solaraxionraytracing_b200 import abi
    tr.set_sampler(abi.SAMPLER_ALIAS)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with torch.cuda.stream(stream):
        tr.reset_image()
        for k in range(warmup + steps):
            flush.zero_()
            if k >= warmup:
                ev[k - warmup][0].record(stream)
            tr.trace_mc(R, SEED, first_ray=k * R)
            if k >= warmup:
                ev[k - warmup][1].record(stream)
        torch.cuda.synchronize()
    ms = statistics.mean(a.elapsed_time(b) for a, b in ev)
    c = tr.read_image().counters[0]
    tr.set_sampler(abi.SAMPLER_INVERSE_CDF)
    tr.reset_image()
    achieved = F_RAY_LLNL * R / (ms * 1e-3) / 1e12
    return {"value": R / (ms * 1e-3), "unit": "rays/s", "kernel_ms": ms, "steps": steps, "warmup": warmup,
            "passed_fraction": c["n_passed"] / max(1, c["n_rays"]),
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s",
                         "frac": achieved / peak_tflops if peak_tflops else None},
            "note": "sart_set_sampler(SART_SAMPLER_ALIAS): same distributions, one table lookup per draw; statistical "
                    "parity only (not the headline)"}


def pure_fp32_leg(tr, torch, stream, flush, R: int, peak_tflops: float, steps: int = 5, warmup: int = 3):
    """The same fused kernel with sart_set_retrace(h, 0, ...): the kernel variant without the margin tests and without the
    FP64 re-trace of uncertain rays. About 1e-5 of the rays then differ from the exact pipeline in their exit code, so it is
    reported next to the headline, not as the headline: what bit-exact classification costs."""
    tr.set_retrace(0, 1.0)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with torch.cuda.stream(stream):
        tr.reset_image()
        for k in range(warmup + steps):
            flush.zero_()
            if k >= warmup:
                ev[k - warmup][0].record(stream)
            tr.trace_mc(R, SEED, first_ray=k * R)
            if k >= warmup:
                ev[k - warmup][1].record(stream)
        torch.cuda.synchronize()
    ms = statistics.mean(a.elapsed_time(b) for a, b in ev)
    tr.set_retrace(1, 1.0)
    tr.reset_image()
    achieved = F_RAY_LLNL * R / (ms * 1e-3) / 1e12
    return {"value": R / (ms * 1e-3), "unit": "rays/s", "kernel_ms": ms, "steps": steps, "warmup": warmup,
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s",
                         "frac": achieved / peak_tflops if peak_tflops else None},
            "note": "sart_set_retrace(h, 0, 1): pure FP32, no margin tests, no FP64 re-trace; ~1e-5 of the rays differ from the "
                    "exact pipeline in their exit code (not the headline)"}


def presampled_leg(tr, torch, device, n_unique: int = 1 << 20, repeat: int = 16, host_repeat: int = 8):
    """Tier-(a) kernel (k_trace_presampled, exact FP64 mode): SoA rays in HBM -> SoA records in HBM, 80 B/ray
    (48 in: origin xyz, exit xy, energy; 32 out: x, y, w f64 + code, shell i32), plus the same through host buffers.
    Inputs are real Philox rays of the workload (sampled once through the C-ABI), tiled `repeat` times on the device."""
    import numpy as np
    from solaraxionraytracing_b200 import abi
    # sample inputs with the product itself: trace n_unique MC rays and keep... the C-ABI returns no emission points,
    # so draw them from the same distributions on the host (uniform disc; solar shell radius from the radius CDF)
    rng = np.random.default_rng(12345)
    tb = tr.fullSetup.tables
    s = tr.fullSetup.expSetup
    ridx = np.searchsorted(tb.fluxRadiusCDF, rng.random(n_unique), side="left")
    r = (0.0015 + 0.0005 * ridx) * s.consts.radiusSun
    a1, a2 = 2 * np.pi * rng.random(n_unique), np.pi * rng.random(n_unique)
    origin = np.stack([np.cos(a1) * np.sin(a2) * r, np.sin(a1) * np.sin(a2) * r, np.cos(a2) * r - s.consts.distanceSunEarth])
    rd, ad = s.magnet.radiusCB * np.sqrt(rng.random(n_unique)), 2 * np.pi * rng.random(n_unique)
    exit_xy = np.stack([np.cos(ad) * rd, np.sin(ad) * rd])
    eidx = np.array([np.searchsorted(tb.diffFluxCDFs[i], u) for i, u in zip(ridx[:4096], rng.random(4096))])
    energy = np.maximum(0.03, tb.energies[np.minimum(eidx, tb.energies.size - 1)])
    energy = np.resize(energy, n_unique)
    n = n_unique * repeat
    dev = f"cuda:{device}"
    d_o = torch.from_numpy(np.ascontiguousarray(origin)).to(dev).repeat(1, repeat).contiguous()
    d_e = torch.from_numpy(np.ascontiguousarray(exit_xy)).to(dev).repeat(1, repeat).contiguous()
    d_en = torch.from_numpy(energy).to(dev).repeat(repeat).contiguous()
    ox, oy, ow = (torch.empty(n, dtype=torch.float64, device=dev) for _ in range(3))
    oc, osh = (torch.empty(n, dtype=torch.int32, device=dev) for _ in range(2))
    ro = abi.RayOut()
    import ctypes as C
    ro.x, ro.y, ro.w = (C.cast(t.data_ptr(), abi.c_double_p) for t in (ox, oy, ow))
    ro.code, ro.shell = (C.cast(t.data_ptr(), abi.c_int32_p) for t in (oc, osh))
    stream = torch.cuda.ExternalStream(tr.stream, device=device)
    ms_by_mode = {}
    for mode in (0, 2):
        tr.set_precision(mode)
        with torch.cuda.stream(stream):
            for _ in range(2):
                tr.trace_presampled_dev(n, d_o.data_ptr(), d_e.data_ptr(), d_en.data_ptr(), ro)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            reps = 3
            for _ in range(reps):
                tr.trace_presampled_dev(n, d_o.data_ptr(), d_e.data_ptr(), d_en.data_ptr(), ro)
            e1.record(stream)
            torch.cuda.synchronize()
        ms_by_mode[mode] = e0.elapsed_time(e1) / reps
    ms = ms_by_mode[2]
    passed = float((oc.bitwise_and(0xff) == 0).double().mean().item())
    # end to end with host (pinned) buffers through sart_trace_presampled: 8 Mi rays, i.e. eight 1 Mi-ray chunks whose
    # H2D copies, kernels and D2H copies overlap inside the call
    n_host = n_unique * host_repeat
    h_o = torch.from_numpy(np.ascontiguousarray(np.tile(origin, (1, host_repeat)))).pin_memory()
    h_e = torch.from_numpy(np.ascontiguousarray(np.tile(exit_xy, (1, host_repeat)))).pin_memory()
    h_en = torch.from_numpy(np.tile(energy, host_repeat)).pin_memory()
    hx, hy, hw = (torch.empty(n_host, dtype=torch.float64).pin_memory() for _ in range(3))
    hc, hs = (torch.empty(n_host, dtype=torch.int32).pin_memory() for _ in range(2))
    hro = abi.RayOut()
    hro.x, hro.y, hro.w = (C.cast(t.data_ptr(), abi.c_double_p) for t in (hx, hy, hw))
    hro.code, hro.shell = (C.cast(t.data_ptr(), abi.c_int32_p) for t in (hc, hs))
    from solaraxionraytracing_b200._lib import check, lib
    call = lambda: check(lib.sart_trace_presampled(tr._h, n_host, C.cast(h_o.data_ptr(), abi.c_double_p),
                                                   C.cast(h_e.data_ptr(), abi.c_double_p),
                                                   C.cast(h_en.data_ptr(), abi.c_double_p), C.byref(hro)))
    call()
    t0 = time.perf_counter()
    for _ in range(3):
        call()
    e2e = 3 * n_host / (time.perf_counter() - t0)
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except (OSError, ValueError):
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    rate = n / (ms * 1e-3)
    return {"kernel": "k_trace_presampled_f32", "rays": n, "rays_per_s": rate, "passed_fraction": passed,
            "exact_fp64_kernel_rays_per_s": n / (ms_by_mode[0] * 1e-3),
            "bytes_per_ray": 80, "e2e_rays_per_s": e2e, "e2e_rays_per_call": n_host, "e2e_h2d_bytes": 48 * n_host, "e2e_d2h_bytes": 32 * n_host,
            "roofline": {"bound": "hbm", "achieved": rate * 80 / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": rate * 80 / 1e9 / hbm, "traffic": ncu_traffic("k_trace_presampled_f32"),
                         "algorithmic_bytes": 80 * n,
                         "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                         "note": "80 B of HBM traffic per ray (48 in, 32 out); the rest of the time is the per-ray "
                                 "arithmetic and table gathers of the fused kernel"}}


def records_leg(tr, torch, n: int = 1 << 24, reps: int = 3):
    """The literal traceAxionWrapper drop-in (sart_trace_mc_rays): Philox sampling + trace on the GPU, one record per
    ray (x, y, w f64 + code, shell i32 = 32 B) copied into the caller's pinned host arrays inside the call."""
    import ctypes as C
    from solaraxionraytracing_b200 import abi
    from solaraxionraytracing_b200._lib import check, lib
    hx, hy, hw = (torch.empty(n, dtype=torch.float64).pin_memory() for _ in range(3))
    hc, hs = (torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(2))
    ro = abi.RayOut()
    ro.x, ro.y, ro.w = (C.cast(t.data_ptr(), abi.c_double_p) for t in (hx, hy, hw))
    ro.code, ro.shell = (C.cast(t.data_ptr(), abi.c_int32_p) for t in (hc, hs))
    tr.set_precision(2)
    call = lambda k: check(lib.sart_trace_mc_rays(tr._h, k * n, n, SEED, C.byref(ro)))
    call(0)
    t0 = time.perf_counter()
    for k in range(reps):
        call(1 + k)
    dt = (time.perf_counter() - t0) / reps
    return {"api": "sart_trace_mc_rays (traceAxionWrapper, per-ray records to host)", "precision": "f32", "rays_per_call": n,
            "value": n / dt, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 32 * n,
            "d2h_GBps": 32 * n / dt / 1e9, "passed_fraction": float((hc.bitwise_and(0xff) == 0).double().mean())}


# Algorithmic work per launched ray of the other BASELINE configurations (DESIGN.md section 5; SURVEY.md section 8d tally x measured
# stage-reach probabilities): BabyIAXO + XMM 565 FLOP (23 % of the rays pass, 2/3 never reach a mirror); the buffer-gas
# mass scan adds 100 FLOP per mass for the rays that reach the weight stage (0.25 of them).
F_RAY_XMM = 565.0
F_MASS = 100.0


def other_configs_leg(rt, tables, torch, device, peak_tflops, rank=0, world=1, rays5=None):
    """BASELINE configs 2, 4 and 5 next to the headline (config 1/3), each a few launches, device-timed on its handle's
    stream. With world > 1 only config 5 runs: its rays are sharded over the ranks by global ray index and merged with
    sart_allreduce, as BASELINE.json describes it (1e11 rays over 8 GPUs)."""
    import numpy as np
    from solaraxionraytracing_b200 import multi_gpu
    em = tables.synthetic_emission(1968, 1500, "primakoff")
    rc, dc = rt.buildCdfs(em, device)
    tb = tables.TableSet(energies=em.energies, fluxRadiusCDF=rc, diffFluxCDFs=dc,
                         reflectivity=tables.synthetic_reflectivity(1, 1000, 1000), **tables.detector_tables_packaged())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{device}")

    def timed(tr, n, first=0, reps=3, merge=False):
        stream = torch.cuda.ExternalStream(tr.stream, device=device)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        with torch.cuda.stream(stream):
            tr.reset_image()
            tr.trace_mc(max(1, n // 10), SEED, first_ray=first)   # warm-up (a full-size launch: the re-trace queue gets its final size)
            tr.reset_image()
            tr.trace_mc(n, SEED, first_ray=first)
            if merge:
                tr.allreduce()   # the first collective of a new communicator sets up its connections
            tr.reset_image()
            for a, b in ev:
                flush.zero_()
                a.record(stream)
                tr.trace_mc(n, SEED, first_ray=first)
                if merge:
                    tr.allreduce()
                b.record(stream)
            torch.cuda.synchronize()
        return statistics.mean(a.elapsed_time(b) for a, b in ev), reps

    out = {}
    if world == 1:
        # config 2: CAST magnet + XMM optic. With the reference's own geometry the CAST bore (r = 21.5 mm) lies inside XMM's
        # central blocker (<= 64.7 mm, rt:1674): every ray that leaves the bore ends as `opaque` (kept as a parity case)
        with rt.RayTracer(rt.FullRaytraceSetup(rt.newExperimentSetup("CAST", "InGrid2018", "vacuum", "XMM", 0), tb), device) as tr:
            tr.set_precision(2)
            n = 10**8
            ms, reps = timed(tr, n)
            c = tr.read_image().counters[0]
            out["2_cast_xmm"] = {"rays": n, "value": n / (ms * 1e-3), "unit": "rays/s", "kernel_ms": ms,
                                 "passed_fraction": c["n_passed"] / c["n_rays"], "opaque_fraction": c["n_exit"]["opaque"] / c["n_rays"],
                                 "note": "the CAST bore lies inside XMM's central blocker: no ray reaches the mirrors (rt:1674)"}
        # config 4: BabyIAXO, buffer gas, 64 axion masses around m_gamma sharing every traced ray, 1e8 rays per mass
        setup4 = rt.newExperimentSetup("BabyIAXO", "InGridIAXO", "gas", "XMM", 0)
        with rt.RayTracer(rt.FullRaytraceSetup(setup4, tb), device) as tr:
            tr.set_precision(2)
            mag, k = setup4.magnet, setup4.consts
            p_gas = mag.pGasRoom / k.roomTemp * mag.tGas                      # rt:1601 (bar, consumed as mbar: quirk Q4)
            ne = 2.0 * 6.022e23 * ((p_gas * 1e2) / (8.314 * mag.tGas))       # am:51-61
            m_gamma = float(np.sqrt(1.97e-7 ** 3 * 4.0 * np.pi * (1.0 / 137.0) * ne / 511e3))
            masses = np.linspace(0.5 * m_gamma, 1.5 * m_gamma, 64)
            tr.set_axion_masses(masses)
            n = 10**8
            ms, reps = timed(tr, n)
            cs = tr.read_image().counters
            reach = (cs[0]["n_passed"] + cs[0]["n_exit"]["zero_weight"] + cs[0]["n_exit"]["window_aperture"]) / cs[0]["n_rays"]
            flop = F_RAY_XMM + 64 * F_MASS * reach
            ach = flop * n / (ms * 1e-3) / 1e12
            out["4_mass_scan"] = {"rays_per_mass": n, "masses": 64, "m_gamma_eV": m_gamma, "value": n / (ms * 1e-3), "unit": "rays/s",
                                  "ray_masses_per_s": 64 * n / (ms * 1e-3), "kernel_ms": ms, "flop_per_ray": flop,
                                  "roofline": {"bound": "fp32", "achieved": ach, "peak": peak_tflops, "unit": "TFLOP/s",
                                               "frac": ach / peak_tflops if peak_tflops else None},
                                  "passed_fraction_first_mass": cs[0]["n_passed"] / cs[0]["n_rays"],
                                  "retraced_fp64_fraction": cs[0]["n_retraced"] / cs[0]["n_rays"]}
    # config 5: BabyIAXO / InGridIAXO / vacuum / XMM = config_default.toml as shipped
    with rt.RayTracer(rt.FullRaytraceSetup(rt.newExperimentSetup("BabyIAXO", "InGridIAXO", "vacuum", "XMM", 0), tb), device) as tr:
        tr.set_precision(2)
        total = int(rays5 or (10**9 if world == 1 else 10**11))
        first, count = multi_gpu.shard(total, rank, world)
        if world > 1:
            multi_gpu.comm_init(tr, rank, world, device)
        ms, reps = timed(tr, count, first=first, reps=2 if world > 1 else 3, merge=world > 1)
        t = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{device}")
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        c = (tr.read_merged() if world > 1 else tr.read_image()).counters[0]
        assert c["n_rays"] == total * reps, (c["n_rays"], total, reps)
        ach = F_RAY_XMM * (total / world) / (ms * 1e-3) / 1e12
        out["5_babyiaxo_xmm"] = {"rays": total, "n_gpus": world, "value": total / (ms * 1e-3), "unit": "rays/s", "ms": ms,
                                 "flop_per_ray": F_RAY_XMM,
                                 "roofline": {"bound": "fp32", "achieved": ach, "peak": peak_tflops, "unit": "TFLOP/s",
                                              "frac": ach / peak_tflops if peak_tflops else None, "per": "GPU"},
                                 "passed_fraction": c["n_passed"] / c["n_rays"],
                                 "retraced_fp64_fraction": c["n_retraced"] / c["n_rays"], "unresolved": c["n_unresolved"],
                                 "timed": "trace of this rank's shard + sart_allreduce, max over ranks" if world > 1 else "fused launch"}
    return out


def passed_leg(tr, torch, n: int = 1 << 26, reps: int = 3):
    """sart_trace_mc_passed: the drop-in for consumers that filter `passed` first (generateResultPlots does, rt:2252-2289) —
    only the passed rays cross PCIe, as f32 records compacted on the GPU (ray offset, x, y, w, shell = 17 B per passed
    ray), in 2^24-ray chunks whose copies overlap the next chunk's kernels. Pinned host arrays."""
    import numpy as np
    from solaraxionraytracing_b200 import abi
    tr.set_precision(2)
    dt = {name: np.dtype(t) for name, t in abi.PASSED_OUT_FIELDS}
    fields = ("ray", "x", "y", "w", "shell")
    torch_dt = {"ray": torch.int32, "x": torch.float32, "y": torch.float32, "w": torch.float32, "shell": torch.uint8}
    pinned = {f: torch.empty(n, dtype=torch_dt[f]).pin_memory() for f in fields}
    bufs = {f: pinned[f].numpy().view(dt[f]) for f in fields}
    rec, cnt = tr.trace_passed(n, SEED, first_ray=0, fields=fields, buffers=bufs)
    t0 = time.perf_counter()
    for k in range(reps):
        rec, cnt = tr.trace_passed(n, SEED, first_ray=(1 + k) * n, fields=fields, buffers=bufs)
    dtm = (time.perf_counter() - t0) / reps
    n_pass = int(rec["ray"].size)
    bytes_per = sum(dt[f].itemsize for f in fields)
    return {"api": "sart_trace_mc_passed (records of the passed rays only, compacted, f32)", "rays_per_call": n, "value": n / dtm,
            "unit": "rays/s", "passed_fraction": n_pass / n, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": bytes_per * n_pass,
            "d2h_GBps": bytes_per * n_pass / dtm / 1e9, "bytes_per_passed_ray": bytes_per,
            "retraced_fp64_fraction": cnt["n_retraced"] / n}


def dump_outputs(res, out_dir: str):
    """Writes a step's outputs as out_dir/<name>.npy, float64: `image` and `image_w2` [M, 256, 256], every counter per
    mass [M] and `n_exit` [M, 13] (columns in abi.EXIT_NAMES order), M = number of axion masses. n_retraced and
    n_unresolved are left out: they tell how the FP32 pipeline reached its result, not what the result is."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    arrays = {"image": res.image, "image_w2": res.image_w2, "n_exit": [list(c["n_exit"].values()) for c in res.counters]}
    for name in res.counters[0]:
        if name not in ("n_exit", "n_retraced", "n_unresolved"):
            arrays[name] = [c[name] for c in res.counters]
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", np.asarray(a, dtype=np.float64))


def ncu_traffic(kernel: str):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/ncu_traffic.json), or None."""
    try:
        return json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())[kernel]["dram_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        return None


def run_ours(args):
    import torch
    from solaraxionraytracing_b200 import abi, multi_gpu, raytracer as rt, tables

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the ray-tracing path)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_gpus = world
    R = int(args.rays_per_step)
    K, W = args.steps, args.warmup
    precision = args.precision or ("f32" if rt.lib.sart_has_precision(2) else "fast")

    t0 = time.perf_counter()
    tb = workload_tables(rt, tables, local)
    setup = rt.newExperimentSetup("CAST", "InGrid2018", "vacuum", "LLNL", 0)
    fs = rt.FullRaytraceSetup(setup, tb)
    tr = rt.RayTracer(fs, local)
    tr.set_precision({"exact": 0, "fast": 1, "f32": 2}[precision])
    if args.sampler == "alias":
        tr.set_sampler(abi.SAMPLER_ALIAS)
    table_upload_s = time.perf_counter() - t0

    stream = torch.cuda.ExternalStream(tr.stream, device=local)
    _, _, img_len = tr.image_dev()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}")  # > 126 MB L2
    if dist is not None:
        # the path's one collective lives behind the C-ABI (sart_allreduce: ONE ncclAllReduce over image | w^2 image |
        # counters into a separate merged buffer); torch.distributed only ships the 128-byte NCCL id and the timings
        multi_gpu.comm_init(tr, rank, world, local)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step(k: int, ev=None):
        """One step: flush L2, trace R rays of this rank's shard, merge images across ranks."""
        first = (k * n_gpus + rank) * R
        flush.zero_()
        if ev is not None:
            ev[0].record(stream)
        tr.trace_mc(R, SEED, first_ray=first)
        if ev is not None:
            ev[1].record(stream)
        if dist is not None:
            tr.allreduce()   # the ranks' own images keep accumulating; the sum over ranks lands in the merged buffer

    smi_index = local
    try:
        smi_index = int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local])
    except (KeyError, ValueError, IndexError):
        pass
    sampler = ClockSampler(smi_index)
    if rank == 0:
        sampler.start()   # started before the warm-up: nvidia-smi needs up to a second to deliver its first sample
    with torch.cuda.stream(stream):
        tr.reset_image()
        for w in range(W):
            step(w)
        barrier()
        tr.reset_image()
        barrier()
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        sampler.mark("t0")
        e0.record(stream)
        for k in range(K):
            step(W + k, kev[k])
        e1.record(stream)
        barrier()
        sampler.mark("t1")
        clocks = sampler.stop() if rank == 0 else None
        ms_total = e0.elapsed_time(e1)
        kernel_ms = [a.elapsed_time(b) for a, b in kev]
    res = tr.read_merged() if dist is not None else tr.read_image()
    if args.dump_outputs:
        # the image accumulates over the timed steps: trace the last one again into a cleared image. These are the same
        # rays (Philox is keyed on the global ray index), and the timed window stays free of host reads.
        with torch.cuda.stream(stream):
            tr.reset_image()
            step(W + K - 1)
        barrier()
        last = tr.read_merged() if dist is not None else tr.read_image()
        if rank == 0:
            dump_outputs(last, args.dump_outputs)
    # per-rank kernel times: a straggler rank must be visible
    t_k = torch.tensor(kernel_ms, dtype=torch.float64, device=f"cuda:{local}")
    all_k = [torch.empty_like(t_k) for _ in range(world)]
    if dist is not None:
        dist.all_gather(all_k, t_k)
    else:
        all_k = [t_k]
    rank_kernel_ms = [float(t.mean().item()) for t in all_k]

    t_ms = torch.tensor([ms_total], dtype=torch.float64, device=f"cuda:{local}")
    if dist is not None:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_total = float(t_ms.item())
    value = n_gpus * R * K / (ms_total * 1e-3)

    # ---- end to end through the C-ABI with host buffers: reset + trace + read image/counters back to the host
    def e2e_step(k):
        first = ((W + K + k) * n_gpus + rank) * R
        tr.reset_image()
        tr.trace_mc(R, SEED, first_ray=first)
        if dist is not None:
            tr.allreduce()
            return tr.read_merged()   # D2H of the merged image, w2 image and counters, synchronises
        return tr.read_image()   # D2H of image, w2 image and counters, synchronises
    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        e2e_step(1 + k)
    barrier()
    e2e_s = time.perf_counter() - t0
    t_e = torch.tensor([e2e_s], dtype=torch.float64, device=f"cuda:{local}")
    if dist is not None:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = n_gpus * R * K / float(t_e.item())
    d2h = 2 * img_len * 8 + C.sizeof(abi.Counters) * tr.n_masses

    fp64 = precision == "exact"
    peak = C.c_double(0.0)
    rt.check(rt.lib.sart_measure_fma_peak(local, 1 if fp64 else 0, C.byref(peak)))
    other = None
    if not args.no_configs and precision == "f32":
        other = other_configs_leg(rt, tables, torch, local, peak.value, rank, world)   # collective for N > 1
    if rank == 0:
        c = res.counters[0]
        k_ms = statistics.mean(kernel_ms)
        assert c["n_rays"] == n_gpus * R * K, (c["n_rays"], n_gpus, R, K)   # every rank's shard is in the merged counters
        achieved = F_RAY_LLNL * R / (k_ms * 1e-3) / 1e12
        out = {
            "metric": "traced rays/s", "value": value, "unit": "rays/s", "n_gpus": n_gpus, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"exact": "f64", "fast": "f64 geometry + f32 weights", "f32": "f32"}[precision], "data": "synthetic",
            "config": {"workload": WORKLOAD, "rays_per_step_per_gpu": R, "precision": precision, "sampler": args.sampler,
                       "l2": "256 MiB buffer written between steps (L2 flush)", "seed": SEED,
                       "table_upload_s": round(table_upload_s, 3),
                       "passed_fraction": c["n_passed"] / max(1, c["n_rays"]),
                       "retraced_fp64_fraction": c["n_retraced"] / max(1, c["n_rays"]), "unresolved": c["n_unresolved"],
                       "collective": None if dist is None else "sart_allreduce: one ncclAllReduce(f64 sum) of image | w^2 image | counters per step"},
            "kernel_ms_over_ranks": {"min": min(rank_kernel_ms), "median": statistics.median(rank_kernel_ms),
                                     "max": max(rank_kernel_ms)},
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h,
                    "note": "sart_reset_image + sart_trace_mc (+ sart_allreduce) + sart_read_image/_merged per step through the C-ABI; the path "
                            "has no per-step host inputs (rays are generated in-kernel from Philox), tables are "
                            "resident per run (config.table_upload_s)"},
            # per step: fused trace kernel + FP64 re-trace of its uncertain rays + image-replica fold (+ counter pack before the all-reduce)
            "gpu_launches": K * ((3 if precision == "f32" else 2 if precision == "fast" else 1) + (1 if dist is not None else 0)),
            "clocks": clocks,
            "roofline": {"bound": "fp64" if fp64 else "fp32", "achieved": achieved, "peak": peak.value,
                         "unit": "TFLOP/s", "frac": achieved / peak.value if peak.value else None,
                         "traffic": ncu_traffic({"exact": "k_trace_mc_image", "fast": "k_trace_mc_fast",
                                                 "f32": "k_trace_mc_f32"}[precision]) if R == 10**9 else None,
                         "traffic_note": "DRAM bytes per 1e9-ray launch from the committed ncu capture: the tables' "
                                         "cold misses; the path has no per-ray HBM traffic",
                         "kernel": {"exact": "k_trace_mc_image", "fast": "k_trace_mc_fast", "f32": "k_trace_mc_f32"}[precision],
                         "kernel_ms": k_ms, "flop_per_ray": F_RAY_LLNL,
                         "peak_source": "sart_measure_fma_peak in this run (MEASURED_PEAKS.json has no CUDA-core "
                                        "figure); the kernel moves ~0 HBM bytes per ray"},
        }
        if n_gpus == 1 and not args.no_presampled and precision == "f32" and args.sampler == "inverse_cdf":
            out["pure_fp32"] = pure_fp32_leg(tr, torch, stream, flush, R, peak.value)
            out["alias_sampler"] = alias_leg(tr, torch, stream, flush, R, peak.value)
        if n_gpus == 1 and not args.no_presampled:
            out["presampled"] = presampled_leg(tr, torch, local)
            out["e2e_records"] = records_leg(tr, torch)
            out["e2e_passed"] = passed_leg(tr, torch)
        if other is not None:
            out["configs"] = other
        tr.set_precision({"exact": 0, "fast": 1, "f32": 2}[precision])
        if n_gpus == 1 and not args.no_cpu_baseline:
            v, cores, sample, cnt_cpu, n0, n_cpu = cpu_leg(args.cpu_seconds)
            out["cpu_baseline"] = {"value": v, "unit": "rays/s", "cores": cores, "kind": "port",
                                   "sample": sample + " (restated oracle, not the Nim executable)"}
            v1, _, sample1, _, _, _ = cpu_leg(min(args.cpu_seconds, 3.0), threads=1)   # BASELINE.md: 1 thread next to all threads
            out["cpu_baseline"]["one_thread"] = {"value": v1, "unit": "rays/s", "cores": 1, "sample": sample1}
            out["parity_check"] = parity_leg(tr, n0, n_cpu, cnt_cpu)
        else:
            out["parity_check"] = parity_leg(tr, 0, 1_000_000)
        print(json.dumps(out), flush=True)
        if not out["parity_check"]["ok"]:
            tr.close()
            raise SystemExit("bench.py: the timed kernel disagrees with the CPU oracle on the same rays: %r" % (out["parity_check"],))
    tr.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    # The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner to stdout when a
    # communicator is created): send file descriptor 1 to stderr for the whole run and keep the real stdout for the line.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
