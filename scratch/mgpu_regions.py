"""Age ranges and fit confidence regions on several GPUs (DESIGN.md section 15), one rank per GPU under
torchrun, NCCL.  Rank 0 writes ``<out>/r08_mgpu_regions.json``; the card's name and power limit are
read in the same run.

* Equality on C3 (4096^2 seed 2, Scarp 100, 30 ages x 181 orientations, snr_ratio 0.9): every rank's
  band of ``sharded_fit_region`` / ``sharded_age_range`` must equal the same rows of a single-GPU
  ``core.fit_region`` / ``core.age_range`` (computed by that rank on its own GPU) bit for bit; the
  row-band drivers must equal a fresh slab plan with the shared curvature statistics bit for bit, and
  the whole raster as ``spatial_search`` does (planes 0..3 within the stack_report bound, the rest
  equal on >= 99 % of the valid pixels).
* Times, maximum over ranks, median of ``--rounds`` rounds after one warm-up: C3 split into phases
  (CUDA events on the stream the plan and NCCL share: sweep, best merge, region pass, region merge =
  all-to-all + k_region_merge, finalize), and the drivers end to end (host clock, synchronised).
* North-star 16384^2 (bench.py's device-generated DEM, seed 4): ``sharded_fit_region``,
  ``sharded_age_range`` (97 GB of per-age states per rank: timed if it fits, its failure reported if
  not) and ``spatial_age_range``, with each plan's device bytes.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29513 scratch/mgpu_regions.py --out profiles
"""
import argparse
import json
import os
import subprocess
import sys
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

RATIO = 0.9
AGES = np.logspace(0, 3.5, 30)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=30).stdout.strip()
    except Exception as e:          # noqa: BLE001 -- recorded, not fatal
        return "unknown (%s)" % e


def reduce_max(values, device):
    t = torch.tensor(values, dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def all_true(flag, device):
    t = torch.tensor([1 if flag else 0], device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


class Phases(object):
    """CUDA events on one stream, one per phase boundary."""

    def __init__(self, stream):
        self.stream, self.marks = stream, []

    def mark(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record(self.stream)
        self.marks.append((name, e))

    def ms(self):
        self.marks[-1][1].synchronize()
        return {b[0]: a[1].elapsed_time(b[1]) for a, b in zip(self.marks, self.marks[1:])}


def region_phases(plan, spec, scale, angles, device, stream, rank, world):
    """sharded_fit_region's steps, with an event between each (and between the all-to-all and the fold)."""
    from scarplet_b200 import distributed as D
    from scarplet_b200 import params as P
    ph = Phases(stream)
    tables = P.region_tables(AGES, angles)
    a, t, age_of, angle_of = plan.build_sweep(spec, scale, AGES, angles, "age_major", template_share=(rank, world))
    ph.mark("start")
    plan.reset()
    plan.sweep(a, t)
    ph.mark("sweep")
    D.merge_best_state(plan, device)
    ph.mark("best_merge")
    plan.region_sweep(a, t, RATIO, tables)
    ph.mark("region_pass")
    ny, nx = plan.ny, plan.nx
    bands = [D.shard_bounds(ny, world, r) for r in range(world)]
    lo, hi = bands[rank]
    ptr, n_planes = plan.region_planes()
    src = D._as_tensor(ptr, n_planes * ny * nx, "i4", device).view(n_planes, ny * nx)
    dst = torch.empty((n_planes, world * nx * (hi - lo)), dtype=torch.int32, device=device)
    for p in range(n_planes):
        dist.all_to_all_single(dst[p], src[p], output_split_sizes=[nx * (hi - lo)] * world,
                               input_split_sizes=[nx * (b - a_) for a_, b in bands])
    ph.mark("region_all_to_all")
    plan.region_merge((lo, hi), world, dst.data_ptr())
    ph.mark("k_region_merge")
    out = plan.region_finalize(age_of, angle_of, tables, rows=(lo, hi))
    ph.mark("finalize")
    return ph.ms(), (lo, hi, out)


def range_phases(plan, spec, scale, angles, device, stream, rank, world):
    from scarplet_b200 import distributed as D
    ph = Phases(stream)
    a, t, age_of, angle_of = plan.build_sweep(spec, scale, AGES, angles, "age_major", template_share=(rank, world),
                                              state_per_age=True)
    ph.mark("start")
    plan.reset()
    plan.sweep(a, t)
    ph.mark("sweep")
    for s in range(len(AGES)):
        band = D.merge_best_bands(plan, device, state=s)
    ph.mark("best_merge_bands")
    out = plan.age_range(age_of, angle_of, RATIO, rows=band)
    ph.mark("finalize")
    return ph.ms(), band + (out,)


def timed(fn, stream, rounds):
    """Host seconds of ``fn()`` ending in a synchronise, per round after one warm-up (maximum over ranks)."""
    times = []
    for k in range(1 + rounds):
        stream.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        r = fn()
        stream.synchronize()
        dt = time.perf_counter() - t0
        del r
        if k:
            times.append(dt)
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--skip-ns", action="store_true")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=device)
    import scarplet_b200 as sl
    from parity import stack_report
    from scarplet_b200 import distributed as D
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from scarplet_b200.templates import Scarp
    from bench import device_dem_rows
    spec = Scarp._sb_spec
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    stream = torch.cuda.Stream(device=device)
    doc = {"card": card() if rank == 0 else None, "world": world, "snr_ratio": RATIO, "rounds": args.rounds}
    ok = True
    with torch.cuda.stream(stream):
        # ---- C3: equality ---------------------------------------------------------------------------
        n = 4096
        z = synthetic_dem(n, seed=2, relief=30.0)
        grid = sl.DEMGrid(z, 1.0)
        want_region = sl.fit_region(grid, Scarp, 100.0, RATIO, ages=AGES)
        want_range = sl.age_range(grid, Scarp, 100.0, RATIO, ages=AGES)
        sl.release()
        eq = {}
        with Plan(n, n, 1.0, 1.0, device=local, stream=stream.cuda_stream) as plan:
            D.set_dem_sharded(plan, z, device)
            lo, hi, got = D.sharded_fit_region(plan, spec, 100.0, AGES, angles, RATIO, device=device)
            eq["sharded_fit_region"] = bool(np.array_equal(got, want_region[:, lo:hi], equal_nan=True))
            lo, hi, got = D.sharded_age_range(plan, spec, 100.0, AGES, angles, RATIO, device=device)
            eq["sharded_age_range"] = bool(np.array_equal(got, want_range[:, lo:hi], equal_nan=True))
            ms_region = [region_phases(plan, spec, 100.0, angles, device, stream, rank, world) for _ in range(1 + args.rounds)]
            eq["phased_fit_region"] = bool(np.array_equal(ms_region[-1][1][2], want_region[:, lo:hi], equal_nan=True))
            ms_range = [range_phases(plan, spec, 100.0, angles, device, stream, rank, world) for _ in range(1 + args.rounds)]
            e2e = {"sharded_fit_region": timed(lambda: D.sharded_fit_region(plan, spec, 100.0, AGES, angles, RATIO,
                                                                           device=device), stream, args.rounds),
                   "sharded_age_range": timed(lambda: D.sharded_age_range(plan, spec, 100.0, AGES, angles, RATIO,
                                                                         device=device), stream, args.rounds)}
        # row bands
        plan, (lo, hi) = D.spatial_plan(n, n, 1.0, 1.0, spec, 100.0, AGES, angles, device=local,
                                        stream=stream.cuda_stream, states=len(AGES))
        halo = D.slab_halo(spec, 100.0, AGES, angles, n, n, 1.0)
        with plan, Plan(n, n, 1.0, 1.0, device=local, stream=stream.cuda_stream, slab=(lo, hi, halo)) as fresh:
            plan.set_dem(z)
            D.share_dem_stats(plan, device=device)
            fresh.set_dem(z)
            D.share_dem_stats(fresh, device=device)
            sp = {"spatial_age_range": D.spatial_age_range(plan, spec, 100.0, AGES, angles, RATIO)[2],
                  "spatial_fit_region": D.spatial_fit_region(plan, spec, 100.0, AGES, angles, RATIO)[2]}
            eq["spatial_age_range_vs_slab_plan"] = bool(np.array_equal(
                sp["spatial_age_range"], D.spatial_age_range(fresh, spec, 100.0, AGES, angles, RATIO)[2], equal_nan=True))
            eq["spatial_fit_region_vs_slab_plan"] = bool(np.array_equal(
                sp["spatial_fit_region"], D.spatial_fit_region(fresh, spec, 100.0, AGES, angles, RATIO)[2], equal_nan=True))
            e2e["spatial_fit_region"] = timed(lambda: D.spatial_fit_region(plan, spec, 100.0, AGES, angles, RATIO),
                                              stream, args.rounds)
            e2e["spatial_age_range"] = timed(lambda: D.spatial_age_range(plan, spec, 100.0, AGES, angles, RATIO),
                                             stream, args.rounds)
        whole = {}
        for name, want in (("spatial_fit_region", want_region), ("spatial_age_range", want_range)):
            got, ref = sp[name], want[:, lo:hi]
            rep = stack_report(got[:4], ref[:4])
            fit = ref[3] > 0
            agree = float((got[4:] == ref[4:]).all(axis=0)[fit].mean())
            good = rep["mask_equal"] and rep["index_agreement"] >= 0.999 and rep["snr_rel_max_strong"] < 5e-5 and agree >= 0.99
            whole[name] = {"rank": rank, "ok": bool(good), "index_agreement": rep["index_agreement"],
                           "snr_rel_max_strong": rep["snr_rel_max_strong"], "planes_4_up_agree": agree}
            eq[name + "_vs_whole_bound"] = bool(good)
        del want_region, want_range
        ok = all(eq.values())
        doc["c3_equal_all_ranks"] = {k: all_true(v, device) for k, v in eq.items()}
        worst = [min(whole[k]["index_agreement"] for k in whole), max(whole[k]["snr_rel_max_strong"] for k in whole),
                 min(whole[k]["planes_4_up_agree"] for k in whole)]
        w = reduce_max([-worst[0], worst[1], -worst[2]], device)
        doc["c3_spatial_vs_whole_worst_rank"] = {"index_agreement_min": -w[0], "snr_rel_max_strong_max": w[1],
                                                 "planes_4_up_agree_min": -w[2]}

        def phase_med(runs):
            keys = list(runs[1][0].keys())
            per_round = [reduce_max([r[0][k] for k in keys], device) for r in runs[1:]]
            return {k: float(np.median([pr[i] for pr in per_round])) for i, k in enumerate(keys)}
        doc["c3_phases_ms_max_over_ranks_median"] = {"sharded_fit_region": phase_med(ms_region),
                                                     "sharded_age_range": phase_med(ms_range)}
        doc["c3_e2e_s_max_over_ranks"] = {k: reduce_max(v, device) for k, v in e2e.items()}
        doc["c3_e2e_s_median"] = {k: float(np.median(v)) for k, v in doc["c3_e2e_s_max_over_ranks"].items()}
        torch.cuda.empty_cache()

        # ---- north-star 16384^2 ------------------------------------------------------------------------
        if not args.skip_ns:
            n = 16384
            ns = {}
            zd = device_dem_rows(n, 4, 0, n, device)
            stream.synchronize()
            torch.cuda.synchronize()
            for name, states in (("sharded_fit_region", 1), ("sharded_age_range", len(AGES))):
                res = {}
                try:
                    with Plan(n, n, 1.0, 1.0, device=local, stream=stream.cuda_stream) as plan:
                        plan.set_dem_device(zd.data_ptr())
                        fits = True
                        try:
                            plan.set_states(states)
                        except Exception as e:            # noqa: BLE001 -- reported
                            fits, res["failure"] = False, "rank %d: %s" % (rank, e)
                        if all_true(fits, device):
                            fn = getattr(D, name)
                            res["s_max_over_ranks"] = reduce_max(timed(lambda: fn(plan, spec, 100.0, AGES, angles, RATIO,
                                                                                  device=device), stream, args.rounds), device)
                            res["s_median"] = float(np.median(res["s_max_over_ranks"]))
                            res["device_bytes_max_over_ranks"] = reduce_max([plan.device_bytes], device)[0]
                            res["torch_peak_bytes_max_over_ranks"] = reduce_max([torch.cuda.max_memory_allocated(device)],
                                                                                device)[0]
                except Exception:                         # noqa: BLE001 -- reported (the ranks fail alike: same sizes)
                    res["failure"] = "rank %d: %s" % (rank, traceback.format_exc(limit=3))
                ns[name] = res
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats(device)
            del zd
            torch.cuda.empty_cache()
            plan, (lo, hi) = D.spatial_plan(n, n, 1.0, 1.0, spec, 100.0, AGES, angles, device=local,
                                            stream=stream.cuda_stream, states=len(AGES))
            with plan:
                r0, nrows = plan.dem_rows()
                zb = device_dem_rows(n, 4, r0, nrows, device)
                stream.synchronize()
                plan.set_dem_device(zb.data_ptr())
                D.share_dem_stats(plan, device=device)
                t = timed(lambda: D.spatial_age_range(plan, spec, 100.0, AGES, angles, RATIO), stream, args.rounds)
                ns["spatial_age_range"] = {"s_max_over_ranks": reduce_max(t, device),
                                           "device_bytes_max_over_ranks": reduce_max([plan.device_bytes], device)[0]}
                ns["spatial_age_range"]["s_median"] = float(np.median(ns["spatial_age_range"]["s_max_over_ranks"]))
            doc["north_star"] = ns
    doc["config"] = ("C3: 4096^2 seed-2 synthetic DEM (relief 30); north-star: 16384^2 bench.py device DEM seed 4; "
                     "Scarp 100, 30 log-spaced ages (10^0-10^3.5) x 181 orientations, snr_ratio %g; one rank per "
                     "GPU, NCCL; plans on the stream NCCL uses" % RATIO)
    all_ok = all_true(ok, device)
    doc["all_ok"] = all_ok
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r08_mgpu_regions.json"), "w") as f:
            json.dump(doc, f, indent=1)
        print(json.dumps(doc), flush=True)
    dist.destroy_process_group()
    sys.exit(0 if all_ok else 1)


if __name__ == "__main__":
    main()
