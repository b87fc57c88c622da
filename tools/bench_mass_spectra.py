#!/usr/bin/env python
"""What the per-mass spectra of sart_enable_mass_spectra cost in a buffer-gas mass scan: BASELINE config 4 (BabyIAXO,
InGridIAXO, gas stage, XMM, the full-size tables of initFullSetup, 64 axion masses from 0.5 to 1.5 m_gamma, precision 2,
re-trace on), 1e8 rays per launch, with the per-mass spectra off and on, alternating launch by launch. Every launch is
timed with CUDA events on the handle's stream (the trace kernel, the FP64 re-trace and the folds) and preceded by a 512 MB
memset that evicts the 126 MB L2. Prints one JSON line with the medians (device name and power limit read with a query of
nvidia-smi).

  python tools/bench_mass_spectra.py [--launches 5] [--rays 1e8] [--masses 64]"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ap = argparse.ArgumentParser()
ap.add_argument("--launches", type=int, default=5)
ap.add_argument("--rays", type=float, default=1e8)
ap.add_argument("--masses", type=int, default=64)
a = ap.parse_args()
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from solaraxionraytracing_b200 import raytracer as rt  # noqa: E402

if rt.lib.sart_device_count() < 1:
    raise SystemExit("bench_mass_spectra needs a CUDA device")
n = int(a.rays)
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
fs = rt.initFullSetup("BabyIAXO", "InGridIAXO", "gas", "XMM")
mag, k = fs.expSetup.magnet, fs.expSetup.consts
p_gas = mag.pGasRoom / k.roomTemp * mag.tGas                      # as bench.py config 4
ne = 2.0 * 6.022e23 * ((p_gas * 1e2) / (8.314 * mag.tGas))
m_gamma = float(np.sqrt(1.97e-7 ** 3 * 4.0 * np.pi * (1.0 / 137.0) * ne / 511e3))
masses = np.linspace(0.5 * m_gamma, 1.5 * m_gamma, a.masses)
out = {"config": "4_mass_scan", "rays": n, "masses": a.masses, "m_gamma_eV": m_gamma, "launches": a.launches}
with rt.RayTracer(fs) as tr:
    tr.set_precision(2)
    tr.set_axion_masses(masses)
    stream = torch.cuda.ExternalStream(tr.stream)

    def launch():
        tr.reset_image()
        flush.zero_()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        tr.trace_mc(n, 299792458)
        t1.record(stream)
        t1.synchronize()
        return t0.elapsed_time(t1)

    ms = {"off": [], "on": []}
    counts = {}
    for v in ("off", "on", "off", "on"):   # warm-up: module load, shared-memory carve-out, accumulators
        tr.enable_mass_spectra(v == "on")
        launch()
    for _ in range(a.launches):
        for v in ("off", "on"):
            tr.enable_mass_spectra(v == "on")
            ms[v].append(launch())
            cs = tr.read_image(want_w2=False).counters
            counts[v] = [c["n_passed"] for c in cs]
            if v == "on":
                s = tr.read_mass_spectra()
                assert [int(x.counts.sum()) for x in s] == counts[v]
    assert counts["off"] == counts["on"], "the spectra changed what the scan computes"
    res = {v: {"ms": [round(x, 3) for x in t], "median_ms": round(statistics.median(t), 3)} for v, t in ms.items()}
    res["on_over_off"] = round(res["on"]["median_ms"] / res["off"]["median_ms"], 4)
    res["n_passed_first_mass"] = counts["on"][0]
    res["retraced_fraction"] = cs[0]["n_retraced"] / cs[0]["n_rays"]
    out.update(res)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
out["device"] = torch.cuda.get_device_name(0)
out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
print(json.dumps(out))
