#!/usr/bin/env python
"""What an angular scan with accumulators costs (sart_angular_scan_outputs), against the plain scan and against the host loop
it replaces: a 14-point scan of telescope_turned_y over [-0.3, 0.3] deg, 1e8 rays per point, precision 2 with the re-trace,
CAST+LLNL and BabyIAXO+XMM with the full-size tables of initFullSetup. Cases, alternating round by round:
  scan       sart_angular_scan (no accumulators)
  rad, spec, bands, qh, all
             sart_angular_scan_outputs with the radial histogram (16384 bins), the spectra, 3 band images (0.5-2-4-8 keV),
             2 quantity histograms at 256 bins (reflect, transMagnet), or all four together
  loop       what a caller without it writes, with all four on: per point sart_update_setup (turned), sart_reset_image,
             sart_trace_mc and the five readers
Each figure is the host time of one whole scan (the calls synchronise), median over the rounds; the L2 is not flushed between
scans (1.4e9 rays per scan). With --repo DIR the plain scan of another checkout (e.g. the parent commit, built) is timed in
subprocesses that alternate with subprocesses timing this checkout's, so that the two builds are compared under the same
conditions. Prints one JSON line with the device name and power limit (nvidia-smi, same run).

  python tools/bench_scan_outputs.py [--rounds 5] [--rays 1e8] [--points 14] [--repo DIR [--pairs 3]]"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--rays", type=float, default=1e8)
ap.add_argument("--points", type=int, default=14)
ap.add_argument("--repo", default=None, help="another checkout whose plain sart_angular_scan is timed beside this one's")
ap.add_argument("--pairs", type=int, default=3, help="subprocess pairs (other checkout, this checkout) with --repo")
ap.add_argument("--scan-only", default=None, help=argparse.SUPPRESS)   # a subprocess: time the plain scan of this checkout
a = ap.parse_args()
ROOT = Path(a.scan_only or Path(__file__).resolve().parents[1])
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

from solaraxionraytracing_b200 import abi, raytracer as rt  # noqa: E402

CONFIGS = {"cast_llnl": ("CAST", "InGrid2018", "vacuum", "LLNL"), "babyiaxo_xmm": ("BabyIAXO", "InGridIAXO", "vacuum", "XMM")}
SEED = 299792458
if rt.lib.sart_device_count() < 1:
    raise SystemExit("bench_scan_outputs needs a CUDA device")
n = int(a.rays)
angles = np.linspace(-0.3, 0.3, a.points)


def timed(f):
    t0 = time.perf_counter()
    f()
    return (time.perf_counter() - t0) * 1e3


def open_tracer(name):
    fs = rt.initFullSetup(*CONFIGS[name])
    tr = rt.RayTracer(fs)
    tr.set_precision(2)
    return fs, tr


if a.scan_only:   # one subprocess of --repo: warm-up, then `rounds` plain scans per configuration
    res = {}
    for name in CONFIGS:
        _, tr = open_tracer(name)
        with tr:
            tr.angular_scan(angles, n, SEED)
            res[name] = statistics.median(timed(lambda: tr.angular_scan(angles, n, SEED)) for _ in range(a.rounds))
    print(json.dumps(res))
    sys.exit(0)

out = {"rays_per_point": n, "points": a.points, "rounds": a.rounds, "configs": {}}
for name in CONFIGS:
    fs, tr = open_tracer(name)
    with tr:
        setup = abi.Setup.from_buffer_copy(bytes(fs.expSetup))
        rays = tr.traceAxionWrapper(1_000_000, SEED)
        sel = rays.w != 0.0
        specs = []
        for q in ("reflect", "transMagnet"):
            v = getattr(rays, q)[sel]
            lo, hi = np.percentile(v[np.isfinite(v)], [2.0, 98.0])
            specs.append((q, 256, float(lo), float(hi) if hi > lo else float(lo) + 1.0))

        def select(case):
            on = {"rad", "spec", "bands", "qh"} if case in ("all", "loop") else {case}
            tr.enable_radial_hist(16384) if "rad" in on else tr.enable_radial_hist(0, 1.0)
            tr.enable_spectra("spec" in on)
            tr.enable_band_images([0.5, 2.0, 4.0, 8.0] if "bands" in on else None)
            tr.enable_quantity_hists(specs if "qh" in on else None)

        def loop():
            for i, ang in enumerate(angles):
                s = abi.Setup.from_buffer_copy(bytes(setup))
                s.telescope.telescope_turned_y = ang
                tr.update_setup(s)
                tr.set_precision(2)
                tr.reset_image()
                tr.trace_mc(n, SEED, first_ray=i * n)
                tr.read_image(want_w2=False)
                tr.read_radial_hist(), tr.read_spectra(), tr.read_band_images(), tr.read_quantity_hists()
            tr.update_setup(setup)
            tr.set_precision(2)

        def outputs(case):
            passed[case] = tr.angular_scan_outputs(angles, n, SEED).counters[0]["n_passed"]

        run = {"scan": lambda: tr.angular_scan(angles, n, SEED), "loop": loop}
        cases = ["scan", "rad", "spec", "bands", "qh", "all", "loop"]
        ms = {c: [] for c in cases}
        passed = {}
        for r in range(a.rounds + 1):   # round 0: warm-up (module loads, replica and stage buffers)
            for c in cases:
                select(c)
                t = timed(run[c] if c in run else lambda: outputs(c))
                if r:
                    ms[c].append(t)
        res = {c: {"ms": [round(x, 2) for x in t], "median_ms": round(statistics.median(t), 2)} for c, t in ms.items()}
        for c in cases[1:]:
            res[c]["vs_scan"] = round(res[c]["median_ms"] / res["scan"]["median_ms"] - 1.0, 4)
        res["all"]["vs_loop"] = round(res["all"]["median_ms"] / res["loop"]["median_ms"] - 1.0, 4)
        assert len(set(passed.values())) == 1, passed   # every accumulator set traces the same rays to the same outcome
        out["configs"][name] = res
if a.repo:
    other = Path(a.repo).resolve()
    runs = {"other": [], "this": []}
    for _ in range(a.pairs):
        for who, root in (("other", other), ("this", Path(__file__).resolve().parents[1])):
            p = subprocess.run([sys.executable, __file__, "--scan-only", str(root), "--rounds", str(a.rounds), "--rays",
                                str(a.rays), "--points", str(a.points)], capture_output=True, text=True, check=True)
            runs[who].append(json.loads(p.stdout.strip().splitlines()[-1]))
    out["plain_scan_vs_repo"] = {
        name: {who: {"ms": [round(r[name], 2) for r in rs], "median_ms": round(statistics.median(r[name] for r in rs), 2)}
               for who, rs in runs.items()} for name in CONFIGS}
    out["repo"] = str(other)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
out["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
print(json.dumps(out))
