#!/usr/bin/env python
"""What the spectra of sart_enable_spectra cost in the fused FP32 run (precision 2, re-trace on), on CAST+LLNL and
BabyIAXO+XMM with the full-size tables of initFullSetup, 1e9 rays per launch. Variants, alternating launch by launch:
  a        the plain kernel variant (nothing optional)
  b        the generic variant with the radial histogram on (sart_enable_radial_hist), spectra off
  c:E,S    b with the spectra on, E energy and S shell replicas (SART_SPEC_E_REPLICAS / SART_SPEC_S_REPLICAS)
Every launch is timed with CUDA events on the handle's stream and preceded by a 512 MB memset that evicts the 126 MB L2.
Prints one JSON line (device name and power limit read with a query of nvidia-smi).

  python tools/bench_spectra.py [--repo DIR] [--launches 5] [--replicas 32,1024 ...]

--repo runs another checkout's package (e.g. the parent commit's build, to compare variants a and b across builds in one
GPU session); variant c is skipped when that package has no spectra."""
import argparse
import json
import os
import statistics
import subprocess
import sys
from pathlib import Path

ap = argparse.ArgumentParser()
ap.add_argument("--repo", default=str(Path(__file__).resolve().parents[1]))
ap.add_argument("--launches", type=int, default=5)
ap.add_argument("--rays", type=float, default=1e9)
ap.add_argument("--replicas", nargs="*", default=["32,1024"], help="E,S replica pairs of variant c")
a = ap.parse_args()
sys.path.insert(0, a.repo)

import torch  # noqa: E402

from solaraxionraytracing_b200 import raytracer as rt  # noqa: E402

if rt.lib.sart_device_count() < 1:
    raise SystemExit("bench_spectra needs a CUDA device")
has_spectra = hasattr(rt.RayTracer, "enable_spectra")
n = int(a.rays)
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
variants = ["a", "b"] + ([f"c:{r}" for r in a.replicas] if has_spectra else [])
out = {"repo": a.repo, "rays": n, "launches": a.launches, "configs": {}}
for name, args in (("cast_llnl", ("CAST", "InGrid2018", "vacuum", "LLNL")),
                   ("babyiaxo_xmm", ("BabyIAXO", "InGridIAXO", "vacuum", "XMM"))):
    fs = rt.initFullSetup(*args)
    with rt.RayTracer(fs) as tr:
        tr.set_precision(2)
        stream = torch.cuda.ExternalStream(tr.stream)

        def select(v):
            if has_spectra:
                tr.enable_spectra(False)
            tr.enable_radial_hist(0, 1.0) if v == "a" else tr.enable_radial_hist(16384)
            if v.startswith("c:"):
                e, s = v[2:].split(",")
                os.environ["SART_SPEC_E_REPLICAS"], os.environ["SART_SPEC_S_REPLICAS"] = e, s
                tr.enable_spectra()

        def launch():
            flush.zero_()
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(stream)
            tr.trace_mc(n, 299792458)
            t1.record(stream)
            t1.synchronize()
            return t0.elapsed_time(t1)

        ms = {v: [] for v in variants}
        sums = {}
        for v in variants:   # warm-up: module load, shared-memory carve-out, replica buffers
            select(v)
            tr.reset_image()
            launch()
        for _ in range(a.launches):
            for v in variants:
                select(v)
                tr.reset_image()
                ms[v].append(launch())
                c = tr.read_image(want_w2=False).counters[0]
                sums[v] = (c["n_passed"], c["sum_w"])
        res = {v: {"ms": [round(x, 3) for x in t], "median_ms": round(statistics.median(t), 3)} for v, t in ms.items()}
        for v in variants[1:]:
            res[v]["vs_a"] = round(res[v]["median_ms"] / res["a"]["median_ms"] - 1.0, 4)
            if v.startswith("c:"):
                res[v]["vs_b"] = round(res[v]["median_ms"] / res["b"]["median_ms"] - 1.0, 4)
        res["n_passed"] = sums["a"][0]
        assert len({s[0] for s in sums.values()}) == 1, sums   # every variant traces the same rays to the same outcome
        out["configs"][name] = res
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
out["device"] = torch.cuda.get_device_name(0)
out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
print(json.dumps(out))
