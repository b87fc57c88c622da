#!/usr/bin/env python
"""What the band images of sart_enable_band_images cost in the fused FP32 run (precision 2, re-trace on), on CAST+LLNL and
BabyIAXO+XMM with the full-size tables of initFullSetup, 1e9 rays per launch. Variants, alternating launch by launch:
  off      the plain kernel variant (nothing optional)
  rad      the generic variant with the radial histogram on (what the spectra's cost was measured against, tools/bench_spectra.py)
  B:R      B band images (B = 4: 0.5,2,4,8,15 keV; B = 16: 16 equal bands over 0..15 keV), R replicas (SART_BAND_REPLICAS)
  rad+B:R  the same with the radial histogram on
Every launch is timed with CUDA events on the handle's stream and preceded by a 512 MB memset that evicts the 126 MB L2;
each variant's figure is the median of its launches. Prints one JSON line (device name and power limit read with a query
of nvidia-smi in the same run).

  python tools/bench_band_images.py [--launches 5] [--variants off 4:8 16:8 ...]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from pathlib import Path

ap = argparse.ArgumentParser()
ap.add_argument("--launches", type=int, default=5)
ap.add_argument("--rays", type=float, default=1e9)
ap.add_argument("--variants", nargs="*", default=["off", "rad", "4:8", "rad+4:8", "16:8"], help="off, rad, [rad+]bands:replicas")
a = ap.parse_args()
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from solaraxionraytracing_b200 import raytracer as rt  # noqa: E402

if rt.lib.sart_device_count() < 1:
    raise SystemExit("bench_band_images needs a CUDA device")
EDGES = {4: [0.5, 2.0, 4.0, 8.0, 15.0], 16: list(np.linspace(0.0, 15.0, 17))}
n = int(a.rays)
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
out = {"rays": n, "launches": a.launches, "configs": {}}
for name, args in (("cast_llnl", ("CAST", "InGrid2018", "vacuum", "LLNL")),
                   ("babyiaxo_xmm", ("BabyIAXO", "InGridIAXO", "vacuum", "XMM"))):
    fs = rt.initFullSetup(*args)
    with rt.RayTracer(fs) as tr:
        tr.set_precision(2)
        stream = torch.cuda.ExternalStream(tr.stream)

        def select(v):
            tr.enable_radial_hist(16384) if v.startswith("rad") else tr.enable_radial_hist(0, 1.0)
            v = v.split("+")[-1]
            if v in ("off", "rad"):
                tr.enable_band_images(None)
                return
            b, r = v.split(":")
            os.environ["SART_BAND_REPLICAS"] = r
            tr.enable_band_images(EDGES[int(b)])

        def launch():
            flush.zero_()
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(stream)
            tr.trace_mc(n, 299792458)
            t1.record(stream)
            t1.synchronize()
            return t0.elapsed_time(t1)

        ms = {v: [] for v in a.variants}
        passed = {}
        for v in a.variants:   # warm-up: module load, shared-memory carve-out, replica buffers
            select(v)
            tr.reset_image()
            launch()
        for _ in range(a.launches):
            for v in a.variants:
                select(v)
                tr.reset_image()
                ms[v].append(launch())
                passed[v] = tr.read_image(want_w2=False).counters[0]["n_passed"]
        res = {v: {"ms": [round(x, 3) for x in t], "median_ms": round(statistics.median(t), 3)} for v, t in ms.items()}
        for base in ("off", "rad"):
            for v in a.variants:
                if base in res and v != base and v.startswith("rad") == (base == "rad"):
                    res[v][f"vs_{base}"] = round(res[v]["median_ms"] / res[base]["median_ms"] - 1.0, 4)
        res["n_passed"] = passed[a.variants[0]]
        assert len(set(passed.values())) == 1, passed   # every variant traces the same rays to the same outcome
        out["configs"][name] = res
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
out["device"] = torch.cuda.get_device_name(0)
out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
print(json.dumps(out))
