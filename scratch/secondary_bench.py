#!/usr/bin/env python
"""Cost of secondary fits (DESIGN.md section 16) on the C3 workload (4096^2 seed-2 DEM, Scarp 100, 30
log-spaced ages x 181 orientations, min_separation 10 degrees); the card's name and power limit are
read in the same process.  Writes ``<out>/secondary_bench.json``:

* device time, CUDA events on one stream, steps alternated over the rounds: ``match``'s sweep
  (reset + sweep) and the secondary sweep on the same 2-state plan (``sb_secondary_sweep``: table
  upload, position plane, state 1 reset, sweep);
* per-kernel device time of both (the plan's profile counters, an event pair around every launch, a
  run of its own);
* ``core.secondary_fit`` against ``core.match`` and ``core.fit_region`` end to end (DEM upload,
  sweeps, decode, download), host clock, in blocks (the first call of a block re-sizes the cached
  plan and is reported apart).

    python scratch/secondary_bench.py --out DIR [--rounds 3]
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
    ap.add_argument("--out", required=True, help="directory for secondary_bench.json")
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
        raise SystemExit("secondary_bench.py: no CUDA device")
    n = 4096
    sep = np.radians(10.0)
    ratio = 0.9
    z = synthetic_dem(n, seed=2, relief=30.0)
    ages = np.logspace(0, 3.5, 30)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    tables = P.region_tables(ages, angles)
    m = P.separation_positions(sep, angles)
    spec = T.Scarp._sb_spec
    stream = torch.cuda.Stream()
    doc = {"card": card(),
           "config": "C3: 4096^2 seed-2 synthetic DEM, Scarp 100, 30 log-spaced ages (10^0-10^3.5) x 181 "
                     "orientations = 5430 templates, min_separation 10 deg = %d positions" % m}

    # ---- device time: match sweep and secondary sweep, alternated ------------------------------------
    plan = Plan(n, n, 1.0, 1.0, stream=stream.cuda_stream, states=2)
    plan.set_dem(z)
    a_rec, t_rec, _, _ = plan.build_sweep(spec, 100.0, ages, angles, "age_major")

    def match_sweep():
        plan.reset()
        plan.sweep(a_rec, t_rec)

    def secondary_sweep():
        plan.secondary_sweep(a_rec, t_rec, tables, m)

    steps = {"match_sweep": match_sweep, "secondary_sweep": secondary_sweep}
    for name in steps:                                   # warm-up: modules, twiddles, workspace
        steps[name]()
    stream.synchronize()
    bytes_before = plan.device_bytes
    ms = {name: [] for name in steps}
    launches = {}
    for _ in range(args.rounds):
        # the secondary sweep follows a match sweep: best state 0 holds the winners it separates from
        for name in ("match_sweep", "secondary_sweep"):
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
    doc["secondary_sweep_over_match_sweep"] = med["secondary_sweep"] / med["match_sweep"]
    doc["launches"] = launches
    doc["plan_device_bytes_2_states"] = bytes_before
    doc["state1_and_position_plane_bytes"] = 14 * n * n

    # ---- per-kernel device time (event pair around every launch, a run of its own) -----------------
    prof = {}
    for name in ("match_sweep", "secondary_sweep"):
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

    calls = {"secondary_fit": lambda: sl.secondary_fit(grid, T.Scarp, 100.0, sep, ages=ages),
             "fit_region": lambda: sl.fit_region(grid, T.Scarp, 100.0, ratio, ages=ages),
             "match": lambda: sl.match(grid, T.Scarp, scale=100.0, ages=ages)}
    e2e = {k: [] for k in calls}
    first = {k: [] for k in calls}
    for order in (("secondary_fit", "fit_region", "match"), ("match", "fit_region", "secondary_fit")):
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
    with open(os.path.join(args.out, "secondary_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
