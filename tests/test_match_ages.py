"""Age-resolved search (``sb_age_range``, ``core.match_ages``, ``core.age_range``, DESIGN.md section
13): one best state per age in one sweep.  The per-age slices are checked against the float64
oracle, the fold over the states against ``match`` bit for bit, and the age range against a NumPy
restatement of its contract; the CPU cases run the emulator build of the kernels (tests/emu), the
``gpu`` cases the B200."""
import numpy as np
import pytest

from oracle import scarplet_oracle as O
from tests.parity import assert_parity, save_report, stack_report
from tests.test_nodata_mask import _assert_small_parity, _gpu_holes, _holes

KINDS = {"Scarp": O.SCARP, "Channel": O.RICKER, "RightFacingUpperBreakScarp": O.RIGHT_UPPER}


def _template(name):
    from scarplet_b200 import templates as T
    return getattr(T, name)


def _grid(z):
    import scarplet_b200 as sl
    return sl.DEMGrid(z, 1.0)


def restated_range(stacks, fold_snr, ratio):
    """Planes 4 and 5 of ``age_range`` from the per-age stacks [G, 4, ny, nx], as the contract states
    them: the smallest / largest decoded age over the ages with snr > 0 and snr >= ratio * best
    (float64), 0 where the fold has no fit."""
    snr, age = stacks[:, 3], stacks[:, 1]
    ok = (snr > 0) & (snr >= ratio * fold_snr[None])
    lo = np.where(ok, age, np.inf).min(axis=0)
    hi = np.where(ok, age, -np.inf).max(axis=0)
    fit = fold_snr > 0
    return np.where(fit, lo, 0.0), np.where(fit, hi, 0.0)


def _stacks(by_age, ages):
    return np.stack([by_age[float(a)] for a in ages])


def _assert_structure(stacks, fold, ages, min_fit=100):
    """Entry s decodes age ages[s] wherever it has a fit; no entry beats the fold, and the entry at
    the fold's age equals its SNR."""
    fold_snr = fold[3]
    fit = fold_snr > 0
    for s, a in enumerate(ages):
        hit = stacks[s, 3] > 0
        assert (stacks[s, 1][hit] == a).all() and (stacks[s, 1][~hit] == 0).all()
        finite = np.isfinite(stacks[s, 3]) & np.isfinite(fold_snr)
        assert (stacks[s, 3][finite] <= fold_snr[finite]).all()
        at = fit & (fold[1] == a)
        assert np.array_equal(stacks[s, 3][at], fold_snr[at])
    assert fit.sum() >= min_fit


# ---------------------------------------------------------------------------
# CPU (emulator build of the kernels)
# ---------------------------------------------------------------------------
ORACLE_CASES = [
    # (template, (ny, nx), scale, ages, (ang_min, ang_max))
    ("Scarp", (97, 130), 10, [2.0, 6.0, 20.0], (-0.4, 0.4)),                    # odd raster
    ("Channel", (96, 100), 5, [0.15, 0.2, 0.3], (-0.3, 0.3)),                   # no edge mask: wrap-around live
    ("RightFacingUpperBreakScarp", (96, 128), 10, [2.0, 6.0, 20.0], (-0.4, 0.4)),   # get_err_mask
]


@pytest.mark.parametrize("tmpl,shape,scale,ages,span", ORACLE_CASES)
def test_per_age_slices_match_oracle(emu_lib, tmpl, shape, scale, ages, span):
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    ny, nx = shape
    z = synthetic_dem(ny, seed=4, nx=nx)
    by_age = sl.match_ages(_grid(z), _template(tmpl), scale, ages=ages, ang_min=span[0], ang_max=span[1])
    assert sorted(by_age) == sorted(ages)
    for a in ages:
        assert by_age[a].shape == (4, ny, nx) and by_age[a].dtype == np.float64
        ref = O.calculate_best_fit_parameters(z, 1.0, 1.0, KINDS[tmpl], scale, a, ang_max=span[1], ang_min=span[0],
                                              processes=2)
        rep = stack_report(by_age[a], ref)
        assert rep["valid"] > 1000, rep
        _assert_small_parity(rep)
    sl.release()


def _fold_cases():
    from scarplet_b200.synth import synthetic_dem
    clean = synthetic_dem(80, seed=9, nx=104)
    nan = clean.copy()
    nan[33, 61] = np.nan
    return {"propagate": (clean, {}), "propagate_nan": (nan, {}),
            "mask_holes": (_holes(clean, "border+cells", seed=2), dict(nodata="mask", min_coverage=0.6))}


@pytest.mark.parametrize("case", ["propagate", "propagate_nan", "mask_holes"])
def test_fold_equals_match(emu_lib, case):
    import scarplet_b200 as sl
    z, masking = _fold_cases()[case]
    Scarp = _template("Scarp")
    ages, kw = [1.5, 4.0, 12.0, 30.0], dict(ang_min=-0.5, ang_max=0.5)
    grid = _grid(z)
    ref = np.stack(sl.match(grid, Scarp, scale=9, ages=ages, **kw, **masking))
    for ratio in (0.5, 0.9, 1.0):
        got = sl.age_range(grid, Scarp, 9, ratio, ages=ages, **kw, **masking)
        assert got.shape == (6,) + z.shape
        assert np.array_equal(got[:4], ref, equal_nan=True), ratio
    if case == "propagate_nan":
        assert np.isnan(ref[3]).any() and (ref[3] == 0).any()
        assert (got[4:][:, np.isnan(ref[3])] == 0).all()
    if case == "mask_holes":
        assert (ref[3][~np.isfinite(z)] == 0).all() and (ref[3] > 0).sum() > 1000
    stacks = _stacks(sl.match_ages(grid, Scarp, 9, ages=ages, **kw, **masking), ages)
    _assert_structure(stacks, ref, ages, min_fit=0 if case == "propagate_nan" else 100)
    sl.release()


def _plan_results(z, spec, scale, ages, angles, substreams=None, slab=None, curv=None, sub_rows=None):
    """On one plan: match's stack (one best state), then the per-age sweep's ``age_range`` planes
    and per-age stacks, the plan's device bytes, and its curvature statistics (a row slab: ``curv``,
    the whole raster's, as ``distributed.share_dem_stats`` hands them out) or ``age_range`` of the
    rows ``sub_rows``."""
    from scarplet_b200.engine import Plan
    ny, nx = z.shape
    with Plan(ny, nx, 1.0, 1.0, slab=slab) as plan:
        if substreams is not None:
            plan.set_option("fit_substreams", substreams)
        plan.set_dem(z)
        if curv is not None:
            plan.set_curv_stats(*curv)
        a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        single = plan.finalize(age_of, angle_of).copy()
        plan.set_states(len(ages))
        a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, state_per_age=True)
        plan.reset()
        plan.sweep(a, t)
        rng = plan.age_range(age_of, angle_of, 0.8)
        stacks = np.stack([plan.finalize(age_of, angle_of, state=s).copy() for s in range(len(ages))])
        extra = plan.curv_stats() if sub_rows is None else plan.age_range(age_of, angle_of, 0.8, rows=sub_rows)
        return single, rng, stacks, plan.device_bytes, extra


def test_fold_with_and_without_fit_substreams(emu_lib):
    """A raster this small deals the fit kernel's templates to sub-streams, each with its own copy
    of every best state (folded after the sweep); ``fit_substreams=1`` keeps one copy.  The fold
    equals match either way."""
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(64, seed=13, nx=72)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-0.6, 0.6)
    spec = _template("Scarp")._sb_spec
    auto = _plan_results(z, spec, 7, ages, angles)
    one = _plan_results(z, spec, 7, ages, angles, substreams=1)
    # the copies are visible in the plan's device memory: 12 B per pixel, state and copy
    assert auto[3] - one[3] >= 12 * z.size * len(ages)
    for single, rng, stacks, _, _ in (auto, one):
        assert np.array_equal(rng[:4], single)
        _assert_structure(stacks, single, ages)
    assert np.array_equal(auto[1], one[1]) and np.array_equal(auto[2], one[2])


@pytest.mark.parametrize("ratio", [0.5, 0.9, 1.0])
def test_age_range_restated(emu_lib, ratio):
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(80, seed=17, nx=96)
    grid, Scarp = _grid(z), _template("Scarp")
    ages, kw = [1.0, 2.5, 6.0, 15.0, 40.0], dict(ang_min=-0.5, ang_max=0.5)
    got = sl.age_range(grid, Scarp, 9, ratio, ages=ages, **kw)
    stacks = _stacks(sl.match_ages(grid, Scarp, 9, ages=ages, **kw), ages)
    lo, hi = restated_range(stacks, got[3], ratio)
    assert np.array_equal(got[4], lo) and np.array_equal(got[5], hi)
    fit = got[3] > 0
    assert (lo[fit] <= got[1][fit]).all() and (got[1][fit] <= hi[fit]).all()
    if ratio == 1.0:
        assert np.array_equal(lo[fit], got[1][fit]) or (lo[fit] < hi[fit]).sum() < 0.01 * fit.sum()
    else:
        assert (lo[fit] < hi[fit]).sum() > 100          # a range, not just the best age
    sl.release()


def test_row_slabs(emu_lib):
    """Row bands (``distributed.spatial_search``'s plans: slab, halo, shared curvature statistics)
    with per-age states: on each band the fold is bit for bit that band's ``match``, ``age_range``
    of a sub-band is bit for bit the band's rows, and the bands put together agree with the
    whole-raster plan to float32 rounding (their FFT domains differ, as for ``match``)."""
    from scarplet_b200 import distributed as D, params as P
    from scarplet_b200.synth import synthetic_dem
    ny, nx = 90, 76
    z = synthetic_dem(ny, seed=19, nx=nx)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-0.4, 0.4)
    spec = _template("Scarp")._sb_spec
    whole = _plan_results(z, spec, 8, ages, angles)
    halo = D.slab_halo(spec, 8, ages, angles, nx, ny, 1.0)
    parts = []
    for lo, hi in ((0, 41), (41, ny)):
        single, rng, stacks, _, sub = _plan_results(z, spec, 8, ages, angles, slab=(lo, hi, halo), curv=whole[4],
                                                    sub_rows=(lo + 5, lo + 20))
        assert rng.shape == (6, hi - lo, nx) and stacks.shape == (len(ages), 4, hi - lo, nx)
        assert np.array_equal(rng[:4], single)
        assert np.array_equal(sub, rng[:, 5:20])
        _assert_structure(stacks, single, ages)
        lo_r, hi_r = restated_range(stacks, rng[3], 0.8)
        assert np.array_equal(rng[4], lo_r) and np.array_equal(rng[5], hi_r)
        parts.append((rng, stacks))
    rng = np.concatenate([p[0] for p in parts], axis=1)
    stacks = np.concatenate([p[1] for p in parts], axis=2)
    for got, ref in [(rng[:4], whole[1][:4])] + [(stacks[s], whole[2][s]) for s in range(len(ages))]:
        rep = stack_report(got, ref)
        assert rep["mask_equal"] and rep["index_agreement"] >= 0.999 and rep["snr_rel_max_strong"] < 2e-5, rep


def test_refusals(emu_lib):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200._lib import SbError
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from tests.plugin_templates import ShiftedRidge
    ny, nx = 48, 56
    z = synthetic_dem(ny, seed=1, nx=nx)
    grid, Scarp = _grid(z), _template("Scarp")
    kw = dict(ang_min=-0.1, ang_max=0.1)
    for fn, extra in ((sl.match_ages, ()), (sl.age_range, (0.5,))):
        for bad in (dict(ages=[2.0]), ):
            with pytest.raises(ValueError, match="built-in"):
                fn(grid, ShiftedRidge, 8, *extra, **bad, **kw)
        with pytest.raises(ValueError, match="keyword"):
            fn(grid, Scarp, 8, *extra, ages=[2.0], shift=1, **kw)
        with pytest.raises(ValueError, match="64"):
            fn(grid, Scarp, 8, *extra, ages=np.linspace(1.0, 50.0, 65), **kw)
        with pytest.raises(ValueError, match="64"):
            fn(grid, Scarp, 8, *extra, ages=[], **kw)
        with pytest.raises(ValueError, match="duplicate"):
            fn(grid, Scarp, 8, *extra, ages=[2.0, 3.0, 2.0], **kw)
    for ratio in (0.0, -0.5, 1.0 + 1e-12, 1.5, np.nan, np.inf):
        with pytest.raises(ValueError, match="snr_ratio"):
            sl.age_range(grid, Scarp, 8, ratio, ages=[2.0], **kw)
    spec = Scarp._sb_spec
    angles = P.search_angles(-0.1, 0.1)
    with Plan(ny, nx, 1.0, 1.0) as plan:
        for args in (dict(scale=[8, 9]), dict(order="angle_major"), dict(ages=np.linspace(1.0, 50.0, 65))):
            call = dict(scale=8, ages=[2.0, 3.0], order="age_major")
            call.update(args)
            with pytest.raises(ValueError, match="state_per_age"):
                plan.build_sweep(spec, call["scale"], call["ages"], angles, call["order"], state_per_age=True)
    with Plan(ny, nx, 1.0, 1.0, slab=(10, 30, 20), states=2) as plan:
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(spec, 8, [2.0, 3.0], angles, state_per_age=True)
        plan.reset()
        plan.sweep(a, t)
        assert plan.age_range(age_of, angle_of, 1.0).shape == (6, 20, nx)
        out = np.empty(6 * nx * 20)

        def raw(n_states=2, lo=10, hi=30, ratio=0.5, n_idx=len(age_of)):
            from scarplet_b200._lib import check
            check(plan.lib, plan.lib.sb_age_range(plan._h, n_states, lo, hi, ratio, age_of.ctypes.data,
                                                  angle_of.ctypes.data, n_idx, out.ctypes.data, 0))
        raw()
        for bad in (dict(ratio=0.0), dict(ratio=1.5), dict(ratio=float("nan"))):
            with pytest.raises(SbError, match="snr_ratio"):
                raw(**bad)
        for bad in (dict(n_states=0), dict(n_states=3)):
            with pytest.raises(SbError, match="n_states"):
                raw(**bad)
        for bad in (dict(lo=9), dict(hi=31), dict(lo=20, hi=20)):
            with pytest.raises(SbError, match="rows outside"):
                raw(**bad)
        with pytest.raises(SbError, match="bad arguments"):
            raw(n_idx=0)
    assert np.array_equal(z, synthetic_dem(ny, seed=1, nx=nx))
    sl.release()


# ---------------------------------------------------------------------------
# on the B200
# ---------------------------------------------------------------------------
C3_AGES = np.logspace(0, 3.5, 30)


@pytest.mark.gpu
def test_gpu_c3_fold_equals_match(cuda_lib):
    """C3 (4096^2 seed 2, Scarp 100, 30 ages x 181 orientations): the age-resolved fold is match."""
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(4096, seed=2)
    grid, Scarp = _grid(z), _template("Scarp")
    got = sl.age_range(grid, Scarp, 100.0, 0.9, ages=C3_AGES)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=C3_AGES))
    equal = bool(np.array_equal(got[:4], ref, equal_nan=True))
    fit = ref[3] > 0
    save_report("c3_fold_vs_match", {"planes_0_3_array_equal": equal, "valid": int(fit.sum()),
                                     "range_width_gt0_share": float((got[5][fit] > got[4][fit]).mean())},
                {"config": "C3 4096^2 seed 2, Scarp 100, 30 ages x 181 orientations, snr_ratio 0.9"})
    assert equal
    sl.release()


@pytest.mark.gpu
def test_gpu_1024_slices_range_and_mask(cuda_lib):
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    n = 1024
    z = synthetic_dem(n, seed=6)
    grid, Scarp = _grid(z), _template("Scarp")
    by_age = sl.match_ages(grid, Scarp, 100.0, ages=C3_AGES)
    stacks = _stacks(by_age, C3_AGES)
    for s in (3, 15, 27):
        a = float(C3_AGES[s])
        ref = O.calculate_best_fit_parameters(z, 1.0, 1.0, O.SCARP, 100.0, a, processes=8)
        rep = stack_report(by_age[a], ref)
        save_report("slice_1024_age_%d" % s, rep, {"config": "1024^2 seed 6, Scarp 100, match_ages over 30 ages x "
                                                             "181 orientations; the slice of age %r against the "
                                                             "float64 oracle" % a})
        assert rep["valid"] > 100000, rep
        assert_parity(rep)
    for ratio in (0.5, 0.9, 1.0):
        got = sl.age_range(grid, Scarp, 100.0, ratio, ages=C3_AGES)
        lo, hi = restated_range(stacks, got[3], ratio)
        assert np.array_equal(got[4], lo) and np.array_equal(got[5], hi), ratio
    _assert_structure(stacks, got[:4], C3_AGES)
    holes = _gpu_holes(z, seed=6)
    assert 0.09 < np.mean(~np.isfinite(holes)) < 0.12
    masked = dict(nodata="mask", min_coverage=0.7)
    got = sl.age_range(_grid(holes), Scarp, 100.0, 0.9, ages=C3_AGES, **masked)
    ref = np.stack(sl.match(_grid(holes), Scarp, scale=100.0, ages=C3_AGES, **masked))
    save_report("masked_1024_fold_vs_match", {"planes_0_3_array_equal": bool(np.array_equal(got[:4], ref, equal_nan=True)),
                                              "valid": int((ref[3] > 0).sum()),
                                              "nodata_share": float(np.mean(~np.isfinite(holes)))},
                {"config": "1024^2 seed 6, ~10 % nodata (border + cells), Scarp 100, 30 ages x 181, "
                           "min_coverage 0.7"})
    assert np.array_equal(got[:4], ref, equal_nan=True)
    sl.release()
