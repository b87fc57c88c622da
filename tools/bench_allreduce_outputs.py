#!/usr/bin/env python
"""What sart_allreduce_outputs costs: one handle per visible GPU in this process (sart_comm_init_all), each after a small
fused run, and the host time of the call, which ends in synchronised streams (the agreement step synchronises, then the
payload is queued; a sart_synchronize of every handle closes the timed window). Two cases, each the median of repeated
calls after warm-up calls:
  radial: the radial histogram (16384 bins) + the spectra of the BabyIAXO+XMM default setup (nE = 1500): ~0.3 MB per GPU;
  masses: the per-mass spectra of 64 masses at nE = 1500: the first 64 rows of ~2.4 MB per GPU.
The sart_allreduce of the image is timed the same way for comparison. Prints one JSON line with the medians, the GPU count
and the device name and power limit (a query of nvidia-smi in the same run).

  python tools/bench_allreduce_outputs.py [--calls 50]"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ap = argparse.ArgumentParser()
ap.add_argument("--calls", type=int, default=50)
a = ap.parse_args()
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import numpy as np  # noqa: E402

from solaraxionraytracing_b200 import multi_gpu, raytracer as rt  # noqa: E402

ng = rt.lib.sart_device_count()
if ng < 1:
    raise SystemExit("bench_allreduce_outputs needs a CUDA device")
fs = rt.initFullSetup("BabyIAXO", "InGridIAXO", "vacuum", "XMM")
out = {"gpus": ng, "calls": a.calls, "nE": int(fs.tables.energies.size)}


def timed(fn, tracers):
    for _ in range(5):   # warm-up: NCCL's first calls set up its channels; the merged copies are allocated
        fn(tracers)
        for t in tracers:
            t.synchronize()
    ms = []
    for _ in range(a.calls):
        t0 = time.perf_counter()
        fn(tracers)
        for t in tracers:
            t.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": round(statistics.median(ms), 4), "min_ms": round(min(ms), 4), "max_ms": round(max(ms), 4)}


tracers = [rt.RayTracer(fs, d) for d in range(ng)]
try:
    multi_gpu.comm_init_all(tracers)
    for k, t in enumerate(tracers):
        t.set_precision(2)
        t.enable_radial_hist(16384)
        t.enable_spectra()
        t.trace_mc(1_000_000, 299792458, first_ray=k * 1_000_000)
    out["radial_hist_and_spectra"] = timed(multi_gpu.allreduce_outputs, tracers)
    out["allreduce_image"] = timed(multi_gpu.allreduce, tracers)
    masses = np.linspace(0.004, 0.02, 64)
    for k, t in enumerate(tracers):
        t.enable_radial_hist(0)
        t.enable_spectra(False)
        t.set_axion_masses(masses)
        t.enable_mass_spectra()
        t.trace_mc(1_000_000, 299792458, first_ray=k * 1_000_000)
    out["mass_spectra_64"] = timed(multi_gpu.allreduce_outputs, tracers)
finally:
    for t in tracers:
        t.close()
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
out["nvidia_smi"] = q.stdout.strip().splitlines() if q.returncode == 0 and q.stdout.strip() else None
print(json.dumps(out))
