#!/usr/bin/env python
"""Cost of sub-grid fit peaks (DESIGN.md section 17) on the C3 workload (4096^2 seed-2 DEM, Scarp 100, 30
log-spaced ages x 181 orientations); the card's name and power limit are read in the same process.
Writes ``<out>/peak_bench.json``:

* device time, CUDA events on one stream, steps alternated over the rounds: ``match``'s sweep
  (reset + sweep) and the peak pass on the same plan (``sb_peak_sweep``: table upload, code plane,
  plane clear, sweep), and ``sb_peak_finalize`` (decode and download);
* per-kernel device time of both sweeps (the plan's profile counters, an event pair around every
  launch, a run of its own);
* ``core.fit_peak`` against ``core.match`` and ``core.fit_region`` end to end (DEM upload, sweeps,
  decode, download), host clock, in blocks (the first call of a block re-sizes the cached plan and is
  reported apart).

    python scratch/peak_bench.py --out DIR [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0]
    except Exception as e:          # noqa: BLE001 -- recorded, not fatal
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for peak_bench.json")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import __graft_entry__
    __graft_entry__.build()
    import scarplet_b200 as sl
    from scarplet_b200 import params as P, templates as T
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem

    if not torch.cuda.is_available():
        raise SystemExit("peak_bench.py: no CUDA device")
    n = 4096
    ratio = 0.9
    z = synthetic_dem(n, seed=2, relief=30.0)
    ages = np.logspace(0, 3.5, 30)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    tables = P.region_tables(ages, angles)
    spec = T.Scarp._sb_spec
    stream = torch.cuda.Stream()
    doc = {"card": card(),
           "config": "C3: 4096^2 seed-2 synthetic DEM, Scarp 100, 30 log-spaced ages (10^0-10^3.5) x 181 "
                     "orientations = 5430 templates"}

    # ---- device time: match sweep and peak pass, alternated -------------------------------------------
    plan = Plan(n, n, 1.0, 1.0, stream=stream.cuda_stream)
    plan.set_dem(z)
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, 100.0, ages, angles, "age_major")

    def match_sweep():
        plan.reset()
        plan.sweep(a_rec, t_rec)

    def peak_sweep():
        plan.peak_sweep(a_rec, t_rec, tables)

    steps = {"match_sweep": match_sweep, "peak_sweep": peak_sweep}
    for name in steps:                                   # warm-up: modules, twiddles, workspace
        steps[name]()
    stream.synchronize()
    bytes_before = plan.device_bytes
    ms = {name: [] for name in steps}
    launches = {}
    for _ in range(args.rounds):
        # the peak pass follows a match sweep: best state 0 holds the winners whose neighbours it records
        for name in ("match_sweep", "peak_sweep"):
            l0 = plan.launches
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            steps[name]()
            e1.record(stream)
            e1.synchronize()
            ms[name].append(e0.elapsed_time(e1))
            launches[name] = plan.launches - l0
    med = {k: float(np.median(v)) for k, v in ms.items()}
    doc["device_ms"] = ms
    doc["device_ms_median"] = med
    doc["peak_sweep_over_match_sweep"] = med["peak_sweep"] / med["match_sweep"]
    doc["launches"] = launches
    doc["plan_device_bytes"] = bytes_before
    doc["peak_planes_bytes"] = 20 * n * n
    fin = []
    for _ in range(args.rounds):
        t0 = time.perf_counter()
        plan.peak_finalize(age_of, angle_of, tables)
        fin.append((time.perf_counter() - t0) * 1e3)
    doc["peak_finalize_ms_host_clock"] = fin

    # ---- per-kernel device time (event pair around every launch, a run of its own) -----------------
    prof = {}
    for name in ("match_sweep", "peak_sweep"):
        plan.set_option("profile", 1)
        plan.profile(reset=True)
        steps[name]()
        stream.synchronize()
        prof[name] = {k: v[0] for k, v in plan.profile(reset=True).items()}
        plan.set_option("profile", 0)
    doc["kernel_ms_profiled"] = prof
    doc["fit_kernel_share"] = {k: v["k_fit_rows"] / sum(v.values()) for k, v in prof.items()}
    plan.close()
    torch.cuda.empty_cache()

    # ---- end to end through the public API -----------------------------------------------------------
    grid = sl.DEMGrid(z, 1.0)

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        return time.perf_counter() - t0, r

    calls = {"fit_peak": lambda: sl.fit_peak(grid, T.Scarp, 100.0, ages=ages),
             "fit_region": lambda: sl.fit_region(grid, T.Scarp, 100.0, ratio, ages=ages),
             "match": lambda: sl.match(grid, T.Scarp, scale=100.0, ages=ages)}
    e2e = {k: [] for k in calls}
    first = {k: [] for k in calls}
    for order in (("fit_peak", "fit_region", "match"), ("match", "fit_region", "fit_peak")):
        for name in order:
            for k in range(1 + args.rounds):
                s, r = timed(calls[name])
                (first if k == 0 else e2e)[name].append(s * 1e3)
                del r
    doc["e2e_ms"] = e2e
    doc["e2e_ms_median"] = {k: float(np.median(v)) for k, v in e2e.items()}
    doc["e2e_first_call_of_block_ms"] = first
    sl.release()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "peak_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
