#!/usr/bin/env python
"""Cost of fit confidence regions (DESIGN.md section 14) on the C3 workload (4096^2 seed-2 DEM, Scarp
100, 30 log-spaced ages x 181 orientations); the card's name and power limit are read in the same
process.  Writes ``<out>/region_bench.json``:

* device time, CUDA events on one stream, steps alternated: ``match``'s sweep (reset + sweep), the
  region pass on the same plan (``sb_region_sweep``: plane clearing, table upload, sweep), and
  ``age_range``'s per-age sweep (30 best states);
* per-kernel device time of the match sweep and of the region pass (the plan's profile counters, an
  event pair around every launch, a run of its own);
* ``k_region_finalize`` alone (``sb_region_finalize`` into device memory);
* ``core.fit_region`` against ``core.age_range`` and ``core.match`` end to end (DEM upload, sweeps,
  decode, download), host clock, in blocks (the first call of a block re-sizes the cached plan and
  is reported apart).

    python scratch/region_bench.py --out DIR [--rounds 3]
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
    ap.add_argument("--out", required=True, help="directory for region_bench.json")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import __graft_entry__
    __graft_entry__.build()
    import scarplet_b200 as sl
    from scarplet_b200 import params as P, templates as T
    from scarplet_b200._lib import check
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem

    if not torch.cuda.is_available():
        raise SystemExit("region_bench.py: no CUDA device")
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
                     "orientations = 5430 templates, snr_ratio %g" % ratio}

    # ---- device time: match sweep, region pass, per-age sweep, alternated ----------------------------
    single = Plan(n, n, 1.0, 1.0, stream=stream.cuda_stream)
    per_age = Plan(n, n, 1.0, 1.0, stream=stream.cuda_stream, states=len(ages))
    single.set_dem(z)
    per_age.set_dem(z)
    s_rec = single.build_sweep(spec, 100.0, ages, angles, "age_major")
    p_rec = per_age.build_sweep(spec, 100.0, ages, angles, "age_major", state_per_age=True)

    def match_sweep():
        single.reset()
        single.sweep(s_rec[0], s_rec[1])

    def region_pass():
        single.region_sweep(s_rec[0], s_rec[1], ratio, tables)

    def age_sweep():
        per_age.reset()
        per_age.sweep(p_rec[0], p_rec[1])

    steps = {"match_sweep": match_sweep, "region_pass": region_pass, "age_range_sweep": age_sweep}
    for name in ("match_sweep", "region_pass", "age_range_sweep"):      # warm-up: modules, twiddles, workspace
        steps[name]()
    stream.synchronize()
    ms = {name: [] for name in steps}
    launches = {}
    for _ in range(args.rounds):
        # the region pass follows a match sweep: best state 0 holds the search it thresholds against
        for name in ("match_sweep", "region_pass", "age_range_sweep"):
            plan = per_age if name == "age_range_sweep" else single
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
    doc["region_pass_over_match_sweep"] = med["region_pass"] / med["match_sweep"]
    doc["fit_region_sweeps_over_age_range_sweep"] = (med["match_sweep"] + med["region_pass"]) / med["age_range_sweep"]
    doc["launches"] = launches
    doc["region_plane_bytes"] = 4 * (3 + -(-len(tables.pos_angle) // 32)) * n * n
    doc["per_age_best_state_bytes"] = 12 * n * n * len(ages)

    # ---- per-kernel device time (event pair around every launch, a run of its own) -----------------
    prof = {}
    for name in ("match_sweep", "region_pass"):
        single.set_option("profile", 1)
        single.profile(reset=True)
        steps[name]()
        stream.synchronize()
        prof[name] = {k: v[0] for k, v in single.profile(reset=True).items()}
        single.set_option("profile", 0)
    doc["kernel_ms_profiled"] = prof

    # ---- k_region_finalize alone ---------------------------------------------------------------------
    out = torch.empty((9, n, n), dtype=torch.float64, device="cuda")
    age_of, angle_of = np.ascontiguousarray(s_rec[2]), np.ascontiguousarray(s_rec[3])
    rank_age, pos_angle = np.ascontiguousarray(tables.rank_age), np.ascontiguousarray(tables.pos_angle)

    def decode():
        check(single.lib, single.lib.sb_region_finalize(single._h, 0, n, age_of.ctypes.data, angle_of.ctypes.data,
                                                        len(age_of), rank_age.ctypes.data, len(rank_age),
                                                        pos_angle.ctypes.data, len(pos_angle), int(tables.periodic),
                                                        out.data_ptr(), 1))
    decode()
    k_ms = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        decode()                                        # includes the small table uploads
        e1.record(stream)
        e1.synchronize()
        k_ms.append(e0.elapsed_time(e1))
    doc["k_region_finalize_ms"] = k_ms
    doc["k_region_finalize_ms_median"] = float(np.median(k_ms))
    del out
    single.close()
    per_age.close()
    torch.cuda.empty_cache()

    # ---- end to end through the public API -----------------------------------------------------------
    grid = sl.DEMGrid(z, 1.0)

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        return time.perf_counter() - t0, r

    calls = {"fit_region": lambda: sl.fit_region(grid, T.Scarp, 100.0, ratio, ages=ages),
             "age_range": lambda: sl.age_range(grid, T.Scarp, 100.0, ratio, ages=ages),
             "match": lambda: sl.match(grid, T.Scarp, scale=100.0, ages=ages)}
    e2e = {k: [] for k in calls}
    first = {k: [] for k in calls}
    for order in (("fit_region", "age_range", "match"), ("match", "age_range", "fit_region")):
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
    with open(os.path.join(args.out, "region_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
