#!/usr/bin/env python
"""Cost of the age-resolved search (DESIGN.md section 13) on the C3 workload (4096^2 seed-2 DEM,
Scarp 100, 30 log-spaced ages x 181 orientations); the card's name and power limit are read in the
same process.  Writes ``<out>/ages_bench.json``:

* device time of one sweep with one best state per age against ``match``'s single-state sweep:
  two plans on one stream, steps alternated, CUDA events around each step (reset + sweep);
* ``k_age_range`` alone (``sb_age_range`` into device memory), CUDA events, after a warm-up;
* ``core.age_range`` against ``core.match`` end to end (DEM upload, sweep, decode, download),
  host clock, in blocks (the first call of a block also re-sizes the cached plan's best states
  and is reported apart);
* ``core.match_ages`` against 30 separate ``calculate_best_fit_parameters(age=a)`` calls.

    python scratch/ages_bench.py --out DIR [--rounds 3]
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
    ap.add_argument("--out", required=True, help="directory for ages_bench.json")
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
        raise SystemExit("ages_bench.py: no CUDA device")
    n = 4096
    z = synthetic_dem(n, seed=2, relief=30.0)
    ages = np.logspace(0, 3.5, 30)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    spec = T.Scarp._sb_spec
    stream = torch.cuda.Stream()
    doc = {"card": card(),
           "config": "C3: 4096^2 seed-2 synthetic DEM, Scarp 100, 30 log-spaced ages (10^0-10^3.5) x 181 "
                     "orientations = 5430 templates"}

    # ---- device time: per-age sweep (30 states) against match's sweep (1 state), alternated ----------
    single = Plan(n, n, 1.0, 1.0, stream=stream.cuda_stream)
    per_age = Plan(n, n, 1.0, 1.0, stream=stream.cuda_stream, states=len(ages))
    runs = {}
    for name, plan, kw in (("match", single, {}), ("per_age", per_age, {"state_per_age": True})):
        plan.set_dem(z)
        runs[name] = (plan,) + plan.build_sweep(spec, 100.0, ages, angles, "age_major", **kw)

    def step(name):
        plan, a_rec, t_rec, _, _ = runs[name]
        plan.reset()
        plan.sweep(a_rec, t_rec)

    for name in runs:                                   # warm-up: modules, twiddles, workspace
        step(name)
    stream.synchronize()
    ms = {name: [] for name in runs}
    launches = {}
    for _ in range(args.rounds):
        for name in ("match", "per_age"):
            plan = runs[name][0]
            l0 = plan.launches
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            step(name)
            e1.record(stream)
            e1.synchronize()
            ms[name].append(e0.elapsed_time(e1))
            launches[name] = plan.launches - l0
    doc["sweep_device_ms"] = ms
    doc["sweep_device_ms_median"] = {k: float(np.median(v)) for k, v in ms.items()}
    doc["sweep_ratio_per_age_over_match"] = doc["sweep_device_ms_median"]["per_age"] / doc["sweep_device_ms_median"]["match"]
    doc["sweep_launches"] = launches
    doc["best_state_bytes_per_age_sweep"] = 12 * n * n * len(ages)

    # ---- per-kernel device time of each sweep (event pair around every launch, a run of its own) -----
    prof = {}
    for name in ("match", "per_age"):
        plan = runs[name][0]
        plan.set_option("profile", 1)
        plan.profile(reset=True)
        step(name)
        stream.synchronize()
        prof[name] = {k: v[0] for k, v in plan.profile(reset=True).items()}
        plan.set_option("profile", 0)
    doc["sweep_kernel_ms_profiled"] = prof

    # ---- k_age_range alone ---------------------------------------------------------------------
    step("per_age")
    plan, _, _, age_of, angle_of = runs["per_age"]
    out = torch.empty((6, n, n), dtype=torch.float64, device="cuda")
    age_of, angle_of = np.ascontiguousarray(age_of), np.ascontiguousarray(angle_of)

    def reduce():
        from scarplet_b200._lib import check
        check(plan.lib, plan.lib.sb_age_range(plan._h, len(ages), 0, n, 0.9, age_of.ctypes.data, angle_of.ctypes.data,
                                              len(age_of), out.data_ptr(), 1))
    reduce()
    k_ms = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        reduce()                                        # includes the 2 x 5430 x 8 B table upload
        e1.record(stream)
        e1.synchronize()
        k_ms.append(e0.elapsed_time(e1))
    doc["k_age_range_ms"] = k_ms
    doc["k_age_range_ms_median"] = float(np.median(k_ms))
    # bytes the reduction must move at least: 30 SNR planes (4 B) in, 6 float64 planes out
    need = n * n * (4 * len(ages) + 6 * 8)
    doc["k_age_range_min_bytes"] = need
    doc["k_age_range_bytes_per_s_at_min_bytes"] = need / (doc["k_age_range_ms_median"] * 1e-3)
    del out
    single.close()
    per_age.close()
    runs.clear()
    torch.cuda.empty_cache()

    # ---- end to end through the public API ---------------------------------------------------------
    grid = sl.DEMGrid(z, 1.0)

    def timed(fn):
        t0 = time.perf_counter()
        r = fn()
        return time.perf_counter() - t0, r

    e2e = {"age_range": [], "match": []}
    first = {"age_range": [], "match": []}
    calls = {"age_range": lambda: sl.age_range(grid, T.Scarp, 100.0, 0.9, ages=ages),
             "match": lambda: sl.match(grid, T.Scarp, scale=100.0, ages=ages)}
    for order in (("age_range", "match"), ("match", "age_range")):
        for name in order:
            for k in range(1 + args.rounds):
                s, r = timed(calls[name])
                (first if k == 0 else e2e)[name].append(s * 1e3)
                del r
    doc["e2e_ms"] = e2e
    doc["e2e_ms_median"] = {k: float(np.median(v)) for k, v in e2e.items()}
    doc["e2e_first_call_of_block_ms"] = first

    m_ages, loop = [], []
    s, r = timed(lambda: sl.match_ages(grid, T.Scarp, 100.0, ages=ages))           # warm-up
    del r
    for _ in range(2):
        s, r = timed(lambda: sl.match_ages(grid, T.Scarp, 100.0, ages=ages))
        m_ages.append(s * 1e3)
        del r
        s, r = timed(lambda: [sl.calculate_best_fit_parameters(grid, T.Scarp, 100.0, a) for a in ages])
        loop.append(s * 1e3)
        del r
    doc["match_ages_e2e_ms"] = m_ages
    doc["thirty_calculate_best_fit_parameters_e2e_ms"] = loop
    sl.release()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "ages_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
