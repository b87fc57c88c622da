#!/usr/bin/env python
"""What the per-mass radial histograms and band images (sart_enable_mass_radial_hist, sart_enable_mass_band_images) cost in
a buffer-gas mass scan, and the host loop they replace. BASELINE config 4 (BabyIAXO, InGridIAXO, gas stage, XMM, the
full-size tables of initFullSetup, 64 axion masses from 0.5 to 1.5 m_gamma, precision 2, re-trace on), 1e8 rays per launch.

Variants of one batched scan, alternated launch by launch: plain; the per-mass spectra alone (their own compile-time
kernel); the per-mass radii (16384 bins); 4 per-mass bands; radii and bands; radii, bands and the per-mass spectra (their
increment over radii and bands is reported next to their increment over the plain scan). The
baseline is the host loop of 64 single-mass runs of the same rays with the radial histogram and 4 band images on: each
run is set_axion_masses([m]), reset_image, trace_mc, timed as a whole without its read-outs (which would add host
synchronisation: the loop's figure is a lower bound). Every launch (and the whole loop) is timed with CUDA events on the
handle's stream and preceded by a 512 MB memset that evicts the 126 MB L2. Prints one JSON line with the medians (device
name and power limit read with a query of nvidia-smi).

  python tools/bench_mass_outputs.py [--launches 5] [--rays 1e8] [--masses 64]"""
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
    raise SystemExit("bench_mass_outputs needs a CUDA device")
n = int(a.rays)
SEED = 299792458
EDGES = [0.0, 2.0, 4.0, 7.0, 1000.0]   # 4 bands over every energy
VARIANTS = {"plain": (), "spectra": ("spectra",), "radii": ("radii",), "bands": ("bands",), "radii+bands": ("radii", "bands"),
            "all": ("radii", "bands", "spectra")}
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:0")
fs = rt.initFullSetup("BabyIAXO", "InGridIAXO", "gas", "XMM")
mag, k = fs.expSetup.magnet, fs.expSetup.consts
p_gas = mag.pGasRoom / k.roomTemp * mag.tGas                      # as bench.py config 4
ne = 2.0 * 6.022e23 * ((p_gas * 1e2) / (8.314 * mag.tGas))
m_gamma = float(np.sqrt(1.97e-7 ** 3 * 4.0 * np.pi * (1.0 / 137.0) * ne / 511e3))
masses = np.linspace(0.5 * m_gamma, 1.5 * m_gamma, a.masses)
out = {"config": "4_mass_scan", "rays": n, "masses": a.masses, "m_gamma_eV": m_gamma, "launches": a.launches,
       "bands": EDGES}


def timed(tr, body):
    stream = torch.cuda.ExternalStream(tr.stream)
    flush.zero_()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    body()
    t1.record(stream)
    t1.synchronize()
    return t0.elapsed_time(t1)


def configure(tr, v):
    on = VARIANTS[v]
    tr.enable_mass_spectra("spectra" in on)
    tr.enable_mass_radial_hist(16384 if "radii" in on else 0)
    tr.enable_mass_band_images(EDGES if "bands" in on else None)


with rt.RayTracer(fs) as tr, rt.RayTracer(fs) as single:
    tr.set_precision(2)
    tr.set_axion_masses(masses)
    single.set_precision(2)
    single.set_axion_masses(masses[:1])
    single.enable_radial_hist(16384)
    single.enable_band_images(EDGES)

    def scan():
        tr.reset_image()
        tr.trace_mc(n, SEED)

    def loop():
        for m in masses:
            single.set_axion_masses([m])
            single.reset_image()
            single.trace_mc(n, SEED)

    ms = {v: [] for v in VARIANTS}
    ms["loop"] = []
    passed = {}
    for v in VARIANTS:   # warm-up: module load, shared-memory carve-out, accumulators
        configure(tr, v)
        timed(tr, scan)
    timed(single, loop)
    for _ in range(a.launches):
        for v in VARIANTS:
            configure(tr, v)
            ms[v].append(timed(tr, scan))
            passed[v] = [c["n_passed"] for c in tr.read_image(want_w2=False).counters]
            if "radii" in VARIANTS[v]:
                assert [int(h[2].sum()) for h in tr.read_mass_radial_hist()] == passed[v]
            if "bands" in VARIANTS[v]:
                assert [int(b.counts.sum()) for b in tr.read_mass_band_images()] == passed[v]
        ms["loop"].append(timed(single, loop))
    assert all(p == passed["plain"] for p in passed.values()), "an accumulator changed what the scan computes"
    res_loop_passed = single.read_image(want_w2=False).counters[0]["n_passed"]
    res = {v: {"ms": [round(x, 3) for x in t], "median_ms": round(statistics.median(t), 3)} for v, t in ms.items()}
    med = {v: r["median_ms"] for v, r in res.items()}
    res["over_plain"] = {v: round(med[v] / med["plain"], 4) for v in VARIANTS}
    res["loop_over_all"] = round(med["loop"] / med["all"], 3)
    res["spectra_increment_ms"] = {"own_kernel": round(med["spectra"] - med["plain"], 3),
                                   "rows_kernel": round(med["all"] - med["radii+bands"], 3)}
    cs = tr.read_image(want_w2=False).counters
    res["retraced_fraction"] = cs[0]["n_retraced"] / cs[0]["n_rays"]
    res["loop_last_mass_passed_as_scan"] = res_loop_passed == passed["plain"][-1]
    out.update(res)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
out["device"] = torch.cuda.get_device_name(0)
out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
print(json.dumps(out))
