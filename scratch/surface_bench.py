#!/usr/bin/env python
"""Device time of ``Plan.fit_surface`` (DESIGN.md section 12): 1024 seeded pixels x the C3 template
set (Scarp 100, 30 ages x 181 angles = 5430 templates) on the C3 DEM (4096^2, seed 2).  CUDA events
on the plan's stream around each call (records in, results out to host memory included), after a
warm-up call, several repeats; the card's name and power limit are read in the same process.
Writes ``<out>/surface_bench.json``.

    python scratch/surface_bench.py --out DIR [--pixels 1024] [--repeats 5]
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
    ap.add_argument("--out", required=True, help="directory for surface_bench.json")
    ap.add_argument("--pixels", type=int, default=1024)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    import torch
    import __graft_entry__
    __graft_entry__.build()
    from scarplet_b200 import params as P, templates as T
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem

    n = 4096
    z = synthetic_dem(n, seed=2)
    ages = np.logspace(0, 3.5, 30)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    spec = T.Scarp._sb_spec
    rng = np.random.default_rng(0)
    rows, cols = rng.integers(0, n, args.pixels), rng.integers(0, n, args.pixels)
    stream = torch.cuda.Stream()
    plan = Plan(n, n, 1.0, 1.0, stream=stream.cuda_stream)
    plan.set_dem(z)
    # counts from the shapes: support-box cells of every template (what the kernel walks)
    recs = P.template_records(spec, 100.0, ages, angles, n, n, 1.0, plan.x, plan.y,
                              np.arange(len(angles)), np.zeros((len(angles), len(ages)), dtype=np.int64))
    box_cells = ((recs["sy_hi"] - recs["sy_lo"] + 1).astype(np.int64) * (recs["sx_hi"] - recs["sx_lo"] + 1)).sum()
    products = int(box_cells) * args.pixels

    plan.fit_surface(spec, 100.0, ages, angles, rows, cols)            # warm-up: module load, float64 planes
    ms, wall = [], []
    for _ in range(args.repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream.synchronize()
        t0 = time.perf_counter()
        a.record(stream)
        amp, snr = plan.fit_surface(spec, 100.0, ages, angles, rows, cols)
        b.record(stream)
        b.synchronize()
        wall.append(1e3 * (time.perf_counter() - t0))
        ms.append(a.elapsed_time(b))
    med = float(np.median(ms))
    doc = {
        "card": card(),
        "config": "fit_surface: %d seeded pixels x Scarp 100, 30 ages x 181 angles (5430 templates) on the "
                  "4096^2 seed-2 synthetic DEM; CUDA events on the plan's stream around each call after one "
                  "warm-up call" % args.pixels,
        "ms_per_call": ms,
        "ms_median": med,
        "host_wall_ms": wall,
        "support_box_cells": int(box_cells),
        "pixel_cell_products": products,
        "products_per_s": products / (med * 1e-3),
        "float64_flops_per_s_two_per_product": 2 * products / (med * 1e-3),
        "snr_positive_share": float((snr > 0).mean()),
    }
    plan.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "surface_bench.json"), "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
