#!/usr/bin/env python
"""Device-resident C3 steps (4096^2, Scarp 100, 30 ages x 181 angles) in one process, three
plans timed in alternation: unmasked, nodata="mask" on a DEM without nodata, and nodata="mask"
with about 10 % nodata in an irregular footprint border.  Records the card's name and power
limit next to the times; writes ``<out>/masked_bench.json``.

    python scratch/masked_bench.py --out DIR --rounds 3
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


def footprint(z, frac_target=0.10, seed=0):
    """``z`` with NaN outside an irregular footprint covering about 1 - frac_target of it."""
    rng = np.random.default_rng(seed)
    ny, nx = z.shape
    yy, xx = np.mgrid[0:ny, 0:nx]
    ry, rx = (yy - ny / 2) / (ny / 2), (xx - nx / 2) / (nx / 2)
    r = np.maximum(np.abs(ry), np.abs(rx)) * (1.0 + 0.03 * np.sin(7 * np.arctan2(ry, rx)))
    r += 0.004 * rng.standard_normal((ny, nx))
    cut = np.quantile(r, 1.0 - frac_target)
    out = z.copy()
    out[r > cut] = np.nan
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0]
    except Exception as e:          # noqa: BLE001 -- recorded, not fatal
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for masked_bench.json")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import __graft_entry__
    __graft_entry__.build()
    from scarplet_b200 import params as P, templates as T
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from tests.parity import stack_report

    n = 4096
    z = synthetic_dem(n, seed=2)
    zh = footprint(z)
    ages = np.logspace(0, 3.5, 30)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    spec = T.Scarp._sb_spec
    runs = {"unmasked": ("propagate", z), "masked_no_nodata": ("mask", z), "masked_10pct_border": ("mask", zh)}
    plans, recs, outs = {}, {}, {}
    for name, (mode, dem) in runs.items():
        plan = Plan(n, n, 1.0, 1.0, nodata=mode, workspace_mb=20000)
        plan.set_dem(dem)
        recs[name] = plan.build_sweep(spec, 100.0, ages, angles)
        plans[name] = plan
    times = {k: [] for k in runs}
    for r in range(args.rounds + 1):                   # round 0 warms every plan up
        for name, plan in plans.items():
            a, t, age_of, angle_of = recs[name]
            plan.sync()
            t0 = time.perf_counter()
            plan.reset()
            plan.sweep(a, t)
            plan.sync()
            dt = time.perf_counter() - t0
            if r > 0:
                times[name].append(dt * 1e3)
            if r == args.rounds:
                outs[name] = plan.finalize(age_of, angle_of)
            print("round %d %-22s %.1f ms" % (r, name, dt * 1e3), flush=True)
    evals = float(n) * n * len(ages) * len(angles)
    rep = stack_report(outs["masked_no_nodata"], outs["unmasked"])
    doc = {
        "card": card(),
        "config": "C3 4096^2 Scarp 100, 30 ages x 181 angles, one process, device-resident, host clock "
                  "around reset + sweep + synchronise, %d alternating rounds after one warm-up round" % args.rounds,
        "nodata_fraction_border": float(np.isnan(zh).mean()),
        "ms": times,
        "ms_median": {k: float(np.median(v)) for k, v in times.items()},
        "gpx_evals_per_s_median": {k: evals / np.median(v) / 1e6 for k, v in times.items()},
        "masked_no_nodata_vs_unmasked": {k: rep[k] for k in ("mask_equal", "index_agreement", "snr_rel_max_strong",
                                                              "amp_rel_max_strong", "snr_rel_max")},
        "masked_no_nodata_bit_identical": bool(np.array_equal(outs["masked_no_nodata"], outs["unmasked"])),
        "nodata_pixels_zero": bool((outs["masked_10pct_border"][:, np.isnan(zh)] == 0).all()),
    }
    for p in plans.values():
        p.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "masked_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc, indent=1))


if __name__ == "__main__":
    main()
