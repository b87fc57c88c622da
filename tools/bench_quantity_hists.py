#!/usr/bin/env python
"""What the quantity histograms of sart_enable_quantity_hists cost in the fused FP32 run (precision 2, re-trace on), on
CAST+LLNL and BabyIAXO+XMM with the full-size tables of initFullSetup, 1e9 rays per launch. Variants, alternating launch by
launch:
  off        the plain kernel variant (nothing optional)
  rad        the generic variant with the radial histogram on (what the spectra's cost was measured against)
  rad+K      the same with K histograms at 256 bins (K = 2: reflect and transMagnet; K = 8: all eight quantities), the
             block's sums in shared memory (SART_QHIST_SMEM) where the block has room for them
  rad+Kg     the same with the sums in 8 block replicas in global memory (the default), folded after the launch
The ranges are the 2nd .. 98th percentiles of each quantity over 1e6 rays of the same run. Every launch is timed with CUDA
events on the handle's stream and preceded by a 512 MB memset that evicts the 126 MB L2; each variant's figure is the median
of its launches. Prints one JSON line (device name and power limit read with a query of nvidia-smi in the same run).

  python tools/bench_quantity_hists.py [--launches 5] [--variants off rad rad+2 rad+8 rad+8g ...]"""
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
ap.add_argument("--variants", nargs="*", default=["off", "rad", "rad+2", "rad+8", "rad+2g", "rad+8g"],
                help="off, rad, rad+K or rad+Kg with K = 2 or 8")
a = ap.parse_args()
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from solaraxionraytracing_b200 import abi, raytracer as rt  # noqa: E402

if rt.lib.sart_device_count() < 1:
    raise SystemExit("bench_quantity_hists needs a CUDA device")
n = int(a.rays)
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
out = {"rays": n, "launches": a.launches, "configs": {}}
for name, args in (("cast_llnl", ("CAST", "InGrid2018", "vacuum", "LLNL")),
                   ("babyiaxo_xmm", ("BabyIAXO", "InGridIAXO", "vacuum", "XMM"))):
    fs = rt.initFullSetup(*args)
    with rt.RayTracer(fs) as tr:
        tr.set_precision(2)
        stream = torch.cuda.ExternalStream(tr.stream)
        rays = tr.traceAxionWrapper(1_000_000, 299792458)
        sel = rays.w != 0.0
        specs = []
        for q in abi.QUANTITIES:
            v = getattr(rays, q)[sel]
            lo, hi = np.percentile(v[np.isfinite(v)], [2.0, 98.0])
            specs.append((q, 256, float(lo), float(hi) if hi > lo else float(lo) + 1.0))
        sets = {"2": specs[:2], "8": specs}

        def select(v):
            tr.enable_radial_hist(16384) if v.startswith("rad") else tr.enable_radial_hist(0, 1.0)
            v = v.split("+")[-1]
            if v in ("off", "rad"):
                tr.enable_quantity_hists(None)
                return
            if v.endswith("g"):
                os.environ.pop("SART_QHIST_SMEM", None)
            else:
                os.environ["SART_QHIST_SMEM"] = "1"
            tr.enable_quantity_hists(sets[v.rstrip("g")])

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
        os.environ.pop("SART_QHIST_SMEM", None)
        res = {v: {"ms": [round(x, 3) for x in t], "median_ms": round(statistics.median(t), 3)} for v, t in ms.items()}
        for base in ("off", "rad"):
            for v in a.variants:
                if base in res and v != base and v.startswith("rad") == (base == "rad"):
                    res[v][f"vs_{base}"] = round(res[v]["median_ms"] / res[base]["median_ms"] - 1.0, 4)
        res["n_passed"] = passed[a.variants[0]]
        res["compaction"] = tr.compaction if hasattr(tr, "compaction") else None
        assert len(set(passed.values())) == 1, passed   # every variant traces the same rays to the same outcome
        out["configs"][name] = res
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
out["device"] = torch.cuda.get_device_name(0)
out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
print(json.dumps(out))
