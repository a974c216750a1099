"""Nodata-aware template search (``nodata="mask"``, ``sb_plan_set_nodata``): each fit uses only
the template cells whose curvature is defined.  The masked oracle (tests/masked_oracle.py) is
pinned against the reference's own fit on filled DEMs; the device is checked against it through
the CPU emulator build of the kernels (tests/emu), and on the B200 with the ``gpu`` tests."""
import os
import sys

import numpy as np
import pytest

from oracle import scarplet_oracle as O
from tests import masked_oracle as MO
from tests.parity import assert_parity, save_report, stack_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _holes(z, kind, seed=0):
    """A copy of ``z`` with nodata: scattered single cells (one of them +Inf), a block, or an
    irregular footprint border (what a survey tile padded out to a rectangle looks like)."""
    rng = np.random.default_rng(seed)
    z = np.array(z, dtype=np.float64)
    ny, nx = z.shape
    if kind in ("cells", "border+cells"):
        idx = rng.choice(ny * nx, size=max(4, ny * nx // 300), replace=False)
        z.flat[idx] = np.nan
        z.flat[idx[0]] = np.inf
    if kind == "block":
        z[ny // 3:ny // 3 + 7, nx // 2:nx // 2 + 11] = np.nan
    if kind in ("border", "border+cells"):
        yy, xx = np.mgrid[0:ny, 0:nx]
        ry, rx = (yy - ny / 2) / (ny / 2), (xx - nx / 2) / (nx / 2)
        edge = 0.93 + 0.05 * np.sin(5 * np.arctan2(ry, rx)) + 0.02 * rng.standard_normal((ny, nx))
        z[np.hypot(ry, rx) > edge] = np.nan
    return z


def _assert_small_parity(rep):
    """assert_parity's bounds as the emulator tests of small rasters apply them: masks (here: every
    coverage decision) exact, indices, and the relative error of the pixels at or above the median
    SNR.  (A raster of 10^4 pixels holds a few whose best SNR is ~1e-6 of the median; their share
    exceeds assert_parity's 5e-5, a bound set for megapixel rasters.)"""
    assert rep["mask_mismatch_unexplained"] == 0, rep
    assert rep["index_agreement"] >= 0.999 and rep["disagree_unexplained"] == 0, rep
    assert rep["snr_rel_max_strong"] <= 1e-4 and rep["amp_rel_max_strong"] <= 1e-4, rep


def _search(plan, z, spec, scale, ages, angles):
    plan.set_dem(z)
    a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
    plan.reset()
    plan.sweep(a, t)
    return plan.finalize(age_of, angle_of)


# ---------------------------------------------------------------------------
# the oracle, pinned independently of the device
# ---------------------------------------------------------------------------
def test_masked_oracle_equals_reference_on_filled_dems():
    """min_coverage = 1: every candidate equals the reference's fit on the DEM with its holes
    filled -- whatever they are filled with; without nodata the masked fit IS the reference's."""
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(90, seed=4, nx=110)
    holes = _holes(z, "block")
    holes[60, 20:23] = np.nan
    fills = [np.where(np.isfinite(holes), holes, 0.0),
             np.where(np.isfinite(holes), holes, z + np.random.default_rng(1).standard_normal(z.shape) * 5.0)]
    for angle in (-1.2, 0.3, np.pi / 2):
        amp, _, _, snr = MO.match_template_masked(holes, 1.0, 1.0, O.SCARP, 9, 4.0, angle)
        cand = snr > 0
        assert cand.sum() > 2000
        for filled in fills:
            ramp, _, _, rsnr = O.match_template(filled, 1.0, 1.0, O.SCARP, 9, 4.0, angle)
            assert np.allclose(snr[cand], rsnr[cand], rtol=1e-9, atol=0)
            assert np.allclose(amp[cand], ramp[cand], rtol=1e-9, atol=1e-12 * np.abs(ramp).max())
            # every pixel the mask drops has a missing cell under the template (or is one)
            assert not (cand & (rsnr == 0)).any()
        amp0, _, _, snr0 = MO.match_template_masked(z, 1.0, 1.0, O.SCARP, 9, 4.0, angle)
        ramp, _, _, rsnr = O.match_template(z, 1.0, 1.0, O.SCARP, 9, 4.0, angle)
        assert np.allclose(snr0, rsnr, rtol=1e-12, atol=0) and np.allclose(amp0, ramp, rtol=1e-12, atol=0)
    # lower coverage admits more pixels, never fewer
    _, _, _, s6 = MO.match_template_masked(holes, 1.0, 1.0, O.SCARP, 9, 4.0, 0.3, min_coverage=0.6)
    _, _, _, s1 = MO.match_template_masked(holes, 1.0, 1.0, O.SCARP, 9, 4.0, 0.3)
    assert ((s1 > 0) <= (s6 > 0)).all() and (s6 > 0).sum() > (s1 > 0).sum()


# ---------------------------------------------------------------------------
# the device (CPU emulator build) against the oracle
# ---------------------------------------------------------------------------
CASES = [
    # template, shape, holes, min_coverage
    ("Scarp", (150, 170), "cells", 1.0),               # padded FFT domain
    ("Scarp", (128, 128), "block", 0.6),               # periodic domain, partial windows
    ("Scarp", (128, 128), "border", 1.0),
    ("Channel", (96, 100), "border", 0.6),             # no edge mask: the wrap-around is live output
    ("RightFacingUpperBreakScarp", (96, 128), "border+cells", 0.6),   # get_err_mask
]
KINDS = {"Scarp": O.SCARP, "Channel": O.RICKER, "RightFacingUpperBreakScarp": O.RIGHT_UPPER}


def _case_params(tmpl):
    from scarplet_b200 import params as P
    angles = P.search_angles(-np.pi / 2, np.pi / 2)[2::25]
    if tmpl == "Channel":
        return 5, [0.2], angles
    return 10, [2.0, 20.0], angles


@pytest.mark.parametrize("tmpl,shape,holes,min_cov", CASES)
def test_masked_search_matches_oracle(emu_lib, tmpl, shape, holes, min_cov):
    from scarplet_b200 import templates as T
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    ny, nx = shape
    z = _holes(synthetic_dem(ny, seed=11, nx=nx), holes, seed=ny)
    keep = z.copy()
    scale, ages, angles = _case_params(tmpl)
    with Plan(ny, nx, 1.0, 1.0, nodata="mask", min_coverage=min_cov) as plan:
        got = _search(plan, z, getattr(T, tmpl)._sb_spec, scale, ages, angles)
    assert np.array_equal(z, keep, equal_nan=True)                  # the caller's DEM is untouched
    assert np.isfinite(got).all()
    assert (got[:, ~np.isfinite(z)] == 0).all()                     # nodata cells: no result
    ref = MO.search_masked(z, 1.0, 1.0, KINDS[tmpl], scale, ages, angles, min_cov)
    rep = stack_report(got, ref, odd_template=(tmpl != "Channel"))
    assert rep["valid"] > 1000, rep
    _assert_small_parity(rep)


def test_masked_without_nodata_equals_unmasked(emu_lib):
    """On a DEM without nodata every window is fully covered: the masked fit takes the unmasked
    arithmetic (the template's own constants).  Reported: whether the results are bit-identical."""
    from scarplet_b200 import templates as T
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(150, seed=11, nx=170)
    scale, ages, angles = _case_params("Scarp")
    outs = {}
    for mode in ("propagate", "mask"):
        with Plan(150, 170, 1.0, 1.0, nodata=mode) as plan:
            outs[mode] = _search(plan, z, T.Scarp._sb_spec, scale, ages, angles)
    rep = stack_report(outs["mask"], outs["propagate"])
    rep["bit_identical"] = bool(np.array_equal(outs["mask"], outs["propagate"]))
    print("masked vs unmasked on a DEM without nodata:", rep)
    assert rep["mask_equal"] and rep["index_agreement"] >= 0.999, rep
    assert rep["snr_rel_max_strong"] <= 1e-5 and rep["amp_rel_max_strong"] <= 1e-5, rep


def test_masked_row_slabs_equal_whole_raster(emu_lib):
    """Row bands of a masked plan (spatial sharding) give the whole-raster masked search; the
    curvature statistics of the bands add up and carry no NaN."""
    from scarplet_b200 import distributed as D, templates as T
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    ny, nx = 150, 170
    z = _holes(synthetic_dem(ny, seed=11, nx=nx), "border+cells", seed=3)
    spec = T.Scarp._sb_spec
    scale, ages, angles = _case_params("Scarp")
    with Plan(ny, nx, 1.0, 1.0, nodata="mask") as plan:
        whole = _search(plan, z, spec, scale, ages, angles)
        s_all, n_all = plan.curv_stats()
    assert np.isfinite(s_all)
    halo = D.slab_halo(spec, scale, ages, angles, nx, ny, 1.0)
    parts, stats = [], []
    for r in range(3):
        lo, hi = D.shard_bounds(ny, 3, r)
        with Plan(ny, nx, 1.0, 1.0, slab=(lo, hi, halo), nodata="mask") as plan:
            plan.set_dem(z)
            stats.append(plan.curv_stats())
            plan.set_curv_stats(s_all, n_all)
            a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
            plan.reset()
            plan.sweep(a, t)
            parts.append(plan.finalize(age_of, angle_of))
    got = np.concatenate(parts, axis=1)
    assert np.isclose(sum(s for s, _ in stats), s_all, rtol=1e-12) and sum(n for _, n in stats) == n_all
    rep = stack_report(got, whole)
    assert rep["mask_equal"] and rep["index_agreement"] >= 0.999 and rep["snr_rel_max_strong"] < 2e-5, rep
    ref = MO.search_masked(z, 1.0, 1.0, O.SCARP, scale, ages, angles)
    _assert_small_parity(stack_report(got, ref))


def test_core_entry_points_take_nodata(emu_lib):
    """core.match / calculate_best_fit_parameters / match_scales take nodata= and min_coverage=;
    the plan cache keeps masked and unmasked plans apart; plugin classes refuse the mask."""
    import scarplet_b200 as sl
    from scarplet_b200 import core, templates as T
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from tests.plugin_templates import ShiftedRidge
    z = _holes(synthetic_dem(96, seed=2, nx=112), "block")
    grid = sl.DEMGrid(z, 1.0)
    kw = dict(ang_min=-0.3, ang_max=0.3)
    plain = sl.calculate_best_fit_parameters(grid, T.Scarp, 10, 3.0, **kw)
    assert np.isnan(plain[3]).any()                                 # the reference's NaN semantics
    masked = sl.calculate_best_fit_parameters(grid, T.Scarp, 10, 3.0, nodata="mask", min_coverage=0.7, **kw)
    assert np.isfinite(masked).all() and (masked[3] > 0).sum() > 3000
    with Plan(96, 112, 1.0, 1.0, nodata="mask", min_coverage=0.7) as plan:
        direct = _search(plan, z, T.Scarp._sb_spec, 10, [3.0], sl.params.search_angles(-0.3, 0.3))
    assert np.array_equal(masked, direct)
    assert np.array_equal(sl.match(grid, T.Scarp, scale=10, age=3.0, nodata="mask", min_coverage=0.7, **kw), direct)
    many = sl.match(grid, T.Scarp, scale=10, ages=[3.0], nodata="mask", min_coverage=0.7, **kw)
    assert np.array_equal(np.stack(many), direct)
    by_scale = core.match_scales(grid, T.Scarp, [10], age=3.0, nodata="mask", min_coverage=0.7, **kw)
    assert np.array_equal(by_scale[10], direct)
    assert np.array_equal(sl.calculate_best_fit_parameters(grid, T.Scarp, 10, 3.0, **kw), plain, equal_nan=True)
    with pytest.raises(ValueError):
        sl.calculate_best_fit_parameters(grid, ShiftedRidge, 10, 3.0, nodata="mask", **kw)
    sl.release()


def test_nodata_errors(emu_lib):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P, templates as T
    from scarplet_b200._lib import SbError
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(64, seed=1, nx=80)
    for cov in (0.0, -0.5, 1.5, float("nan")):
        with pytest.raises(SbError, match="min_coverage"):
            Plan(64, 80, 1.0, 1.0, nodata="mask", min_coverage=cov)
    with pytest.raises(ValueError):
        Plan(64, 80, 1.0, 1.0, nodata="fill")
    with pytest.raises(SbError, match="precision 32"):
        Plan(64, 80, 1.0, 1.0, precision=64, nodata="mask")
    with Plan(64, 80, 1.0, 1.0) as plan:
        plan.set_option("fast", 0)
        with pytest.raises(SbError, match="fast"):
            plan.set_nodata("mask")
    angles = P.search_angles(-0.1, 0.1)
    with Plan(64, 80, 1.0, 1.0, nodata="mask") as plan:
        plan.set_dem(z)
        with pytest.raises(SbError, match="match_template"):
            plan.match_template(T.Scarp._sb_spec, 8, 3.0, 0.1)
        with pytest.raises(SbError, match="match_template"):
            plan.match_template_raster(plan.render_template(T.Scarp._sb_spec, 8, 3.0, 0.1), 0.1)
        a, t, _, _ = plan.build_sweep(T.Scarp._sb_spec, 8, [3.0], angles)
        for key, value in (("fast", 0), ("precision", 64)):
            plan.set_option(key, value)
            plan.reset()
            with pytest.raises(SbError, match="nodata mask"):
                plan.sweep(a, t)
            plan.set_option(key, {"fast": 1, "precision": 32}[key])
    with pytest.raises(ValueError):
        sl.match(sl.DEMGrid(z, 1.0), T.Scarp, scale=8, age=3.0, nodata="bogus")
    sl.release()


# ---------------------------------------------------------------------------
# orientation shards over two ranks (gloo, emulator build)
# ---------------------------------------------------------------------------
SHAPE = (96, 128)
SCALE, AGES = 8, [2.0, 9.0]


def _gloo_inputs():
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    z = _holes(synthetic_dem(SHAPE[0], seed=7, nx=SHAPE[1], relief=3.0), "border+cells", seed=5)
    return z, P.search_angles(-np.pi / 2, np.pi / 2)[::9]


def _gloo_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), SB_EMU_WORKERS="2")
    import torch
    import torch.distributed as dist
    from tests.emu.build_emu import build
    from scarplet_b200 import _lib
    _lib._use_library(_lib.open_library(build()))
    from scarplet_b200 import distributed as D
    from scarplet_b200.engine import Plan
    from scarplet_b200.templates import Scarp
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cpu = torch.device("cpu")
    z, angles = _gloo_inputs()
    ny, nx = SHAPE
    with Plan(ny, nx, 1.0, 1.0, nodata="mask", min_coverage=0.8) as plan:
        D.set_dem_sharded(plan, z, cpu)
        out = D.sharded_search(plan, Scarp._sb_spec, SCALE, AGES, angles, "age_major", device=cpu)
        np.save(os.path.join(out_dir, "replicated%d.npy" % rank), out)
        lo, hi, band = D.sharded_search(plan, Scarp._sb_spec, SCALE, AGES, angles, "age_major", device=cpu,
                                        merge="bands")
        np.save(os.path.join(out_dir, "bands%d.npy" % rank), band)
    plan, (lo, hi) = D.spatial_plan(ny, nx, 1.0, 1.0, Scarp._sb_spec, SCALE, AGES, angles,
                                    nodata="mask", min_coverage=0.8)
    with plan:
        plan.set_dem(z)
        D.share_dem_stats(plan, device=cpu)
        _, _, band = D.spatial_search(plan, Scarp._sb_spec, SCALE, AGES, angles)
        np.save(os.path.join(out_dir, "spatial%d.npy" % rank), band)
    dist.destroy_process_group()


def test_masked_sharded_search_equals_single_rank(tmp_path, emu_lib):
    """Orientation shards of a masked search merge (replicated and banded) to the single-rank
    masked search bit for bit; the row-band split matches it to rounding."""
    import torch.multiprocessing as mp
    from scarplet_b200.engine import Plan
    from scarplet_b200.templates import Scarp
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    z, angles = _gloo_inputs()
    with Plan(SHAPE[0], SHAPE[1], 1.0, 1.0, nodata="mask", min_coverage=0.8) as plan:
        single = _search(plan, z, Scarp._sb_spec, SCALE, AGES, angles)
    assert (single[3] > 0).sum() > 1000 and np.isfinite(single).all()
    r0, r1 = np.load(tmp_path / "replicated0.npy"), np.load(tmp_path / "replicated1.npy")
    assert np.array_equal(r0, r1) and np.array_equal(r0, single)
    bands = np.concatenate([np.load(tmp_path / ("bands%d.npy" % r)) for r in range(2)], axis=1)
    assert np.array_equal(bands, single)
    spatial = np.concatenate([np.load(tmp_path / ("spatial%d.npy" % r)) for r in range(2)], axis=1)
    rep = stack_report(spatial, single)
    assert rep["mask_equal"] and rep["index_agreement"] >= 0.999 and rep["snr_rel_max_strong"] < 2e-5, rep


# ---------------------------------------------------------------------------
# on the B200
# ---------------------------------------------------------------------------
CORES = 16


def _masked_angle_stack(args):
    z, kind, scale, age, angle, min_cov = args
    return MO.match_template_masked(z, 1.0, 1.0, kind, scale, age, angle, min_cov)


def _oracle_masked(z, kind, scale, ages, angles, min_cov=1.0):
    """match()'s hierarchical reduce (core.py:285-292) of the masked fit: the result and the
    per-age stacks (which explain the reference's exact-tie resets, tests/parity.py)."""
    import multiprocessing as mp
    ny, nx = z.shape
    with mp.Pool(CORES) as pool:
        stacks = [np.stack(O.compare(pool.imap(_masked_angle_stack, [(z, kind, scale, a, ang, min_cov)
                                                                     for ang in angles]), ny, nx))
                  for a in ages]
    if len(ages) == 1:
        return stacks[0], np.stack(stacks)
    return np.stack(O.compare(stacks, ny, nx)), np.stack(stacks)


def _gpu_holes(z, seed, lake=None):
    """Nodata at B200 sizes: an irregular footprint border (about 10 % of the raster), one
    scattered cell in 20 000 (large templates cover thousands of cells) and optionally a lake
    ``(row, col, radius)``."""
    rng = np.random.default_rng(seed)
    z = np.array(z, dtype=np.float64)
    ny, nx = z.shape
    yy, xx = np.mgrid[0:ny, 0:nx]
    ry, rx = (yy - ny / 2) / (ny / 2), (xx - nx / 2) / (nx / 2)
    r = np.maximum(np.abs(ry), np.abs(rx)) * (1.0 + 0.03 * np.sin(7 * np.arctan2(ry, rx)))
    r += 0.004 * rng.standard_normal((ny, nx))
    z[r > np.quantile(r, 0.9)] = np.nan
    z.flat[rng.choice(ny * nx, size=ny * nx // 20000, replace=False)] = np.nan
    if lake is not None:
        cy, cx, rad = lake
        ang = np.arctan2(yy - cy, xx - cx)
        z[np.hypot(yy - cy, xx - cx) < rad * (1.0 + 0.1 * np.sin(5 * ang))] = np.nan
    return z


def _save(name, rep, config):
    save_report("masked_" + name, rep, {"config": config})


@pytest.mark.gpu
def test_c1_masked_full_raster(cuda_lib):
    """C1 size with a footprint border and scattered holes: the whole raster against the oracle."""
    import scarplet_b200 as sl
    from scarplet_b200.WindowedTemplate import Scarp
    from scarplet_b200.synth import synthetic_dem
    z = _gpu_holes(synthetic_dem(1024, seed=0), seed=1)
    res = sl.match(sl.DEMGrid(z, 1.0), Scarp, scale=100, age=10, nodata="mask")
    ref, _ = _oracle_masked(z, O.SCARP, 100, [10.0], O.search_angles())
    rep = stack_report(res, ref)
    rep["nodata_fraction"] = float((~np.isfinite(z)).mean())
    _save("c1_full_raster", rep, "C1 1024^2 Scarp 100 age 10, 181 angles, footprint border (10 %) + "
                                        "scattered cells, nodata='mask', min_coverage 1, full raster")
    assert (res[:, ~np.isfinite(z)] == 0).all()
    assert rep["valid"] > 500000
    assert_parity(rep)


@pytest.mark.gpu
def test_c3_masked_six_ages_crop(cuda_lib):
    """4096^2 with a footprint border, scattered holes and a lake, 6 ages (kt 1 ... 3162) x 181
    angles, min_coverage 0.7: a crop that reaches into the lake against the oracle."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200.WindowedTemplate import Scarp
    from scarplet_b200.synth import synthetic_dem
    n = 4096
    z = _gpu_holes(synthetic_dem(n, seed=2), seed=2, lake=(2200, 1900, 300))
    ages = np.logspace(0, 3.5, 30)[[0, 6, 12, 18, 24, 29]]
    res = np.stack(sl.match(sl.DEMGrid(z, 1.0), Scarp, scale=100, ages=ages, nodata="mask", min_coverage=0.7))
    m = int(1.4143 * 100 + 2 * P.scarp_halfwidth(ages.max()) + 16)
    size, c0 = 2 * m + 260, 1700                     # the inner crop reaches into the lake
    ref, stacks = _oracle_masked(z[c0:c0 + size, c0:c0 + size], O.SCARP, 100, ages, O.search_angles(), 0.7)
    inner = (slice(None), slice(m, size - m), slice(m, size - m))
    crop = res[:, c0 + m:c0 + size - m, c0 + m:c0 + size - m]
    rep = stack_report(crop, ref[inner], ref_age_stacks=stacks[(slice(None),) + inner], ages=ages)
    rep["nodata_fraction_crop"] = float((~np.isfinite(z[c0 + m:c0 + size - m, c0 + m:c0 + size - m])).mean())
    _save("c3_six_ages_crop", rep, "4096^2 Scarp 100, 6 ages x 181 angles, footprint border, scattered cells, "
                                          "a lake, "
                                          "min_coverage 0.7, %d^2 crop at %d, margin %d" % (size, c0, m))
    assert rep["valid"] > 20000
    assert_parity(rep)
