"""Fit surfaces at chosen pixels (``sb_fit_surface``, ``core.fit_surface``, DESIGN.md section 12):
the post-mask amplitude and SNR of every (age, orientation) template at a list of pixels, by
direct float64 correlation.  Checked against the float64 oracle (whole-raster FFT fits), the
masked oracle, and the float32 sweep; the CPU cases run the emulator build of the kernels
(tests/emu), the ``gpu`` cases the B200."""
import numpy as np
import pytest

from oracle import scarplet_oracle as O
from tests import masked_oracle as MO
from tests.parity import save_report
from tests.test_nodata_mask import _gpu_holes, _holes

KINDS = {"Scarp": O.SCARP, "Channel": O.RICKER, "RightFacingUpperBreakScarp": O.RIGHT_UPPER}


def _angles(n=8):
    from scarplet_b200 import params as P
    return P.search_angles(-np.pi / 2, np.pi / 2)[2::180 // n][:n]


def _pixels(ny, nx, seed, n=24, border=False):
    """Corners and edge midpoints, then seeded pixels: near the raster border (``border``: the
    wrap-around rows / columns of a template without edge mask) or anywhere."""
    rng = np.random.default_rng(seed)
    fixed = [(0, 0), (0, nx - 1), (ny - 1, 0), (ny - 1, nx - 1), (0, nx // 2), (ny // 2, 0), (ny - 1, nx // 2),
             (ny // 2, nx - 1)]
    out = list(fixed)
    while len(out) < n:
        if border:
            r = int(rng.choice([rng.integers(0, 3), rng.integers(ny - 3, ny), rng.integers(0, ny)]))
            c = int(rng.choice([rng.integers(0, 3), rng.integers(nx - 3, nx), rng.integers(0, nx)]))
        else:
            r, c = int(rng.integers(0, ny)), int(rng.integers(0, nx))
        out.append((r, c))
    return np.array(out, dtype=np.int64)


def _oracle_planes(z, kind, scale, ages, angles, masked=None):
    """[G, A, ny, nx] amp and snr of the whole-raster oracle fits."""
    fit = (lambda age, a: O.match_template(z, 1.0, 1.0, kind, scale, age, a)) if masked is None else \
        (lambda age, a: MO.match_template_masked(z, 1.0, 1.0, kind, scale, age, a, masked))
    amp = np.empty((len(ages), len(angles)) + z.shape)
    snr = np.empty_like(amp)
    for g, age in enumerate(ages):
        for a, angle in enumerate(angles):
            r = fit(age, angle)
            amp[g, a], snr[g, a] = r[0], r[3]
    return amp, snr


def _at(planes, pixels):
    """[n_pix, G, A] samples of [G, A, ny, nx] planes."""
    return np.moveaxis(planes[:, :, pixels[:, 0], pixels[:, 1]], -1, 0)


def assert_surface_close(amp, snr, ref_amp_planes, ref_snr_planes, pixels):
    """Zero entries exact; amp to rtol 1e-9 (atol 1e-12 max|amp|); snr to rtol 1e-9 where the
    reference is at least 1e-6 of its maximum, atol 1e-9 max below."""
    ramp, rsnr = _at(ref_amp_planes, pixels), _at(ref_snr_planes, pixels)
    assert np.array_equal(amp == 0, ramp == 0) and np.array_equal(snr == 0, rsnr == 0)
    amax, smax = np.abs(ref_amp_planes).max(), np.abs(ref_snr_planes).max()
    np.testing.assert_allclose(amp, ramp, rtol=1e-9, atol=1e-12 * amax)
    strong = np.abs(rsnr) >= 1e-6 * smax
    np.testing.assert_allclose(snr[strong], rsnr[strong], rtol=1e-9, atol=0)
    np.testing.assert_allclose(snr[~strong], rsnr[~strong], rtol=0, atol=1e-9 * smax)


def _grid(z):
    import scarplet_b200 as sl
    return sl.DEMGrid(z, 1.0)


def _template(name):
    from scarplet_b200 import templates as T
    return getattr(T, name)


# ---------------------------------------------------------------------------
# CPU (emulator build of the kernels)
# ---------------------------------------------------------------------------
ORACLE_CASES = [
    # (template, (ny, nx), scale, ages, wrap-around border pixels)
    ("Scarp", (97, 130), 10, [2.0, 20.0], False),                      # odd raster: index convention
    ("Channel", (96, 100), 5, [0.2], True),                             # no edge mask: wrap-around is live
    ("RightFacingUpperBreakScarp", (96, 128), 10, [2.0, 20.0], False),  # get_err_mask
]


def _plan_surface(plan, z, tmpl, scale, ages, angles, pixels):
    plan.set_dem(z)
    return plan.fit_surface(_template(tmpl)._sb_spec, scale, ages, angles, pixels[:, 0], pixels[:, 1])


@pytest.mark.parametrize("tmpl,shape,scale,ages,border", ORACLE_CASES)
def test_surface_matches_oracle(emu_lib, tmpl, shape, scale, ages, border):
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    ny, nx = shape
    z = synthetic_dem(ny, seed=5, nx=nx)
    angles = _angles()
    pixels = _pixels(ny, nx, seed=ny + nx, border=border)
    with Plan(ny, nx, 1.0, 1.0) as plan:
        amp, snr = _plan_surface(plan, z, tmpl, scale, ages, angles, pixels)
    assert amp.shape == snr.shape == (len(pixels), len(ages), len(angles))
    ref_amp, ref_snr = _oracle_planes(z, KINDS[tmpl], scale, ages, angles)
    at = _at(ref_snr, pixels)
    assert (at > 0).sum() > 50 and ((at == 0).any() or tmpl == "Channel")   # Channel: no edge mask
    assert_surface_close(amp, snr, ref_amp, ref_snr, pixels)


@pytest.mark.parametrize("tmpl,holes,min_cov", [("Scarp", "border+cells", 1.0), ("Scarp", "block", 0.6),
                                                ("RightFacingUpperBreakScarp", "border+cells", 0.6)])
def test_masked_surface_matches_oracle(emu_lib, tmpl, holes, min_cov):
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    ny, nx = 97, 130
    z = _holes(synthetic_dem(ny, seed=11, nx=nx), holes, seed=ny)
    bad = np.argwhere(~np.isfinite(z))[:4]
    pixels = np.concatenate([_pixels(ny, nx, seed=3, n=20), bad])
    scale, ages, angles = 10, [2.0, 20.0], _angles()
    with Plan(ny, nx, 1.0, 1.0, nodata="mask", min_coverage=min_cov) as plan:
        amp, snr = _plan_surface(plan, z, tmpl, scale, ages, angles, pixels)
    ref_amp, ref_snr = _oracle_planes(z, KINDS[tmpl], scale, ages, angles, masked=min_cov)
    assert (amp[-len(bad):] == 0).all() and (snr[-len(bad):] == 0).all()     # nodata pixels: no result
    assert (snr > 0).sum() > 20
    assert np.array_equal(amp != 0, _at(ref_amp, pixels) != 0)               # the candidate pattern
    assert_surface_close(amp, snr, ref_amp, ref_snr, pixels)


def test_nan_in_propagate_dem(emu_lib):
    """The reference's whole-raster fft2 spreads one NaN to every entry the masks leave."""
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    ny, nx = 97, 130
    z = synthetic_dem(ny, seed=5, nx=nx)
    z[40, 77] = np.nan
    keep = z.copy()
    pixels = _pixels(ny, nx, seed=9)
    ages, angles = [2.0, 20.0], _angles()
    with Plan(ny, nx, 1.0, 1.0) as plan:
        amp, snr = _plan_surface(plan, z, "RightFacingUpperBreakScarp", 10, ages, angles, pixels)
    assert np.array_equal(z, keep, equal_nan=True)                        # the caller's DEM is untouched
    ref_amp, ref_snr = _oracle_planes(z, O.RIGHT_UPPER, 10, ages, angles)
    for got, ref in ((amp, _at(ref_amp, pixels)), (snr, _at(ref_snr, pixels))):
        assert np.isnan(got).any() and (got == 0).any()
        assert np.array_equal(np.isnan(got), np.isnan(ref)) and np.array_equal(got == 0, ref == 0)


def check_against_sweep(amp, snr, stack, ages, angles, pixels, oracle_snr=None):
    """Case by case against the float32 sweep ``stack`` (the whole raster's [amp, age, angle, snr]):
    the surface maximum is the sweep's best SNR within 1e-4; its first maximum is the sweep's flat
    index, or the sweep's pick is within 1e-4 of it (a float32 near-tie), or the two are the
    +-90 degree pair (DESIGN.md section 5); the decoded age / angle of an agreeing pixel are the
    sweep's.  Below the median SNR of the sweep's valid pixels the float32 pipeline does not
    resolve 1e-4 relative (DESIGN.md section 4 bounds it above the median only): a pixel there
    that misses these properties is explained when ``oracle_snr(i, j, [k, ...])`` -- the float64
    whole-raster fit of templates k -- equals the surface at both its maximum and the sweep's pick
    to 1e-9.  Returns a report; ``unexplained`` counts every pixel left over."""
    A = len(angles)
    flat = snr.reshape(len(pixels), -1)
    floor = float(np.median(stack[3][stack[3] > 0]))
    rep = dict(pixels=len(pixels), valid=0, index_equal=0, near_tie=0, pm90_pair=0, weak_vs_float64=0,
               unexplained=0, unexplained_pixels=[], snr_rel_max=0.0, snr_rel_max_strong=0.0, all_masked_zero=0,
               median_sweep_snr=floor)
    for q, (i, j) in enumerate(pixels):
        s_amp, s_age, s_ang, s_snr = stack[:, i, j]
        if s_snr == 0:
            assert flat[q].max() == 0, (i, j)
            rep["all_masked_zero"] += 1
            continue
        rep["valid"] += 1
        best = int(np.argmax(flat[q]))
        smax = flat[q, best]
        rel = float(abs(s_snr - smax) / smax)
        rep["snr_rel_max"] = max(rep["snr_rel_max"], rel)
        if s_snr >= floor:
            rep["snr_rel_max_strong"] = max(rep["snr_rel_max_strong"], rel)
        g = int(np.flatnonzero(ages == s_age)[0])
        a = int(np.flatnonzero(angles == s_ang)[0])
        pick = g * A + a
        kind = None
        if rel <= 1e-4:
            if pick == best:
                kind = "index_equal"
                assert ages[best // A] == s_age and angles[best % A] == s_ang
            elif flat[q, pick] >= (1 - 1e-4) * smax:
                kind = "near_tie"
            elif best // A == g and {best % A, a} == {0, A - 1}:
                kind = "pm90_pair"
        if kind is None and s_snr < floor and oracle_snr is not None:
            ks = [best, pick]
            if np.allclose(flat[q, ks], oracle_snr(int(i), int(j), ks), rtol=1e-9, atol=0):
                kind = "weak_vs_float64"
        if kind is None:
            rep["unexplained"] += 1
            rep["unexplained_pixels"].append([int(i), int(j), float(s_snr), float(smax)])
        else:
            rep[kind] += 1
    return rep


def _oracle_snr(fit, ages, angles):
    """``oracle_snr`` for ``check_against_sweep``: ``fit(age, angle)`` -> the whole-raster snr plane."""
    A, cache = len(angles), {}

    def at(i, j, ks):
        for k in ks:
            if k not in cache:
                cache[k] = fit(ages[k // A], angles[k % A])
        return np.array([cache[k][i, j] for k in ks])
    return at


def _sweep(plan, spec, scale, ages, angles):
    a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
    plan.reset()
    plan.sweep(a, t)
    return plan.finalize(age_of, angle_of)


def test_surface_agrees_with_sweep(emu_lib):
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    ny, nx = 97, 130
    z = synthetic_dem(ny, seed=6, nx=nx)
    ages, angles = np.array([2.0, 20.0]), P.search_angles(-np.pi / 2, np.pi / 2)[::24]
    pixels = _pixels(ny, nx, seed=1)
    spec = _template("Scarp")._sb_spec
    with Plan(ny, nx, 1.0, 1.0) as plan:
        amp, snr = _plan_surface(plan, z, "Scarp", 10, ages, angles, pixels)
        stack = _sweep(plan, spec, 10, ages, angles)
    rep = check_against_sweep(amp, snr, stack, ages, angles, pixels)
    assert rep["valid"] >= 12 and rep["unexplained"] == 0, rep


def test_bit_identical_under_batching_and_plan_options(emu_lib):
    """A pixel's values do not depend on the other pixels of the call, their order, duplicates,
    the split into calls, precision, fast, or a row slab."""
    from scarplet_b200 import distributed as D
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    ny, nx = 97, 130
    z = synthetic_dem(ny, seed=7, nx=nx)
    ages, angles = [2.0, 20.0], _angles()
    pixels = _pixels(ny, nx, seed=2)
    spec = _template("Scarp")._sb_spec
    with Plan(ny, nx, 1.0, 1.0) as plan:
        amp, snr = _plan_surface(plan, z, "Scarp", 10, ages, angles, pixels)
        perm = np.random.default_rng(0).permutation(len(pixels))
        pa, ps = plan.fit_surface(spec, 10, ages, angles, pixels[perm, 0], pixels[perm, 1])
        assert np.array_equal(pa, amp[perm]) and np.array_equal(ps, snr[perm])
        h = len(pixels) // 3
        parts = [plan.fit_surface(spec, 10, ages, angles, pixels[s, 0], pixels[s, 1])
                 for s in (slice(0, h), slice(h, None))]
        assert np.array_equal(np.concatenate([p[0] for p in parts]), amp)
        assert np.array_equal(np.concatenate([p[1] for p in parts]), snr)
        dup = np.concatenate([pixels[5:8], pixels[5:8], pixels[:1]])
        da, dsn = plan.fit_surface(spec, 10, ages, angles, dup[:, 0], dup[:, 1])
        assert np.array_equal(da, np.concatenate([amp[5:8], amp[5:8], amp[:1]]))
        assert np.array_equal(dsn, np.concatenate([snr[5:8], snr[5:8], snr[:1]]))
    for opts in (dict(precision=64), dict(fast=0)):
        with Plan(ny, nx, 1.0, 1.0, precision=opts.get("precision")) as plan:
            if "fast" in opts:
                plan.set_option("fast", opts["fast"])
            oa, osn = _plan_surface(plan, z, "Scarp", 10, ages, angles, pixels)
        assert np.array_equal(oa, amp) and np.array_equal(osn, snr), opts
    halo = D.slab_halo(spec, 10, ages, angles, nx, ny, 1.0)
    lo, hi = 30, 70
    inside = (pixels[:, 0] >= lo) & (pixels[:, 0] < hi)
    assert inside.sum() >= 5
    with Plan(ny, nx, 1.0, 1.0, slab=(lo, hi, halo)) as plan:
        sa, ss = _plan_surface(plan, z, "Scarp", 10, ages, angles, pixels[inside])
    assert np.array_equal(sa, amp[inside]) and np.array_equal(ss, snr[inside])


def test_fit_surface_errors(emu_lib):
    import scarplet_b200 as sl
    from scarplet_b200._lib import SbError
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from tests.plugin_templates import ShiftedRidge
    ny, nx = 64, 80
    z = synthetic_dem(ny, seed=1, nx=nx)
    keep = z.copy()
    grid = _grid(z)
    Scarp = _template("Scarp")
    kw = dict(ages=[3.0], ang_min=-0.1, ang_max=0.1)
    for bad in ([(0, nx)], [(-1, 0)], [(ny, 3)], [(0.5, 2)], np.array([[1.0, 2.0]]), [(1, 2, 3)], [[True, False]]):
        with pytest.raises(ValueError):
            sl.fit_surface(grid, Scarp, 8, bad, **kw)
    empty = sl.fit_surface(grid, Scarp, 8, [], **kw)
    assert empty.amp.shape == empty.snr.shape == (0, 1, len(empty.angles)) == (0, 1, 12)
    assert sl.fit_surface(grid, Scarp, 8, np.zeros((0, 2), dtype=np.int32), **kw).snr.shape == (0, 1, 12)
    with pytest.raises(ValueError):
        sl.fit_surface(grid, ShiftedRidge, 8, [(3, 4)], **kw)
    with pytest.raises(ValueError):
        sl.fit_surface(grid, Scarp, 8, [(3, 4)], shift=1, **kw)
    fs = sl.fit_surface(grid, Scarp, 8, [(30, 40)], **kw)
    assert fs.amp.shape == (1, 1, 12) and np.array_equal(fs.ages, [3.0]) and (fs.snr > 0).any()
    assert len(sl.fit_surface(grid, Scarp, 8, [(30, 40)], ang_min=-0.1, ang_max=0.1).ages) == 35
    assert np.array_equal(z, keep)
    spec = Scarp._sb_spec
    with Plan(ny, nx, 1.0, 1.0) as plan:
        with pytest.raises(SbError, match="no DEM"):
            plan.fit_surface(spec, 8, [3.0], [0.0], [3], [4])
    with Plan(ny, nx, 1.0, 1.0) as plan:
        from ctypes import byref
        from scarplet_b200 import params as P
        from scarplet_b200._lib import check
        plan.set_dem(z)
        rec = P.template_record(spec, 8, 3.0, 0.0, nx, ny, 1.0, plan.x, plan.y, 0, 0)
        rec.kind = 2                                                     # SB_KIND_RASTER
        out = np.empty(2)
        rows, cols = np.array([3], dtype=np.int32), np.array([4], dtype=np.int32)
        with pytest.raises(SbError, match="raster"):
            check(plan.lib, plan.lib.sb_fit_surface(plan._h, byref(P.angle_record(0.0)), 1, byref(rec), 1,
                                                    rows.ctypes.data, cols.ctypes.data, 1, out.ctypes.data,
                                                    out[1:].ctypes.data, 0))
    with Plan(ny, nx, 1.0, 1.0, slab=(20, 40, 30)) as plan:
        plan.set_dem(z)
        with pytest.raises(SbError, match="outside rows"):
            plan.fit_surface(spec, 8, [3.0], [0.0], [19], [4])
        amp, snr = plan.fit_surface(spec, 8, [3.0], [0.0], [20, 39], [4, 5])
        assert amp.shape == (2, 1, 1)
    with Plan(ny, nx, 1.0, 1.0, slab=(20, 40, 3)) as plan:
        plan.set_dem(z)
        with pytest.raises(SbError, match="halo too small"):
            plan.fit_surface(spec, 8, [3.0], [0.0], [25], [4])
    sl.release()


# ---------------------------------------------------------------------------
# on the B200
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_surface_matches_oracle(cuda_lib):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    ny, nx = 300, 257
    z = synthetic_dem(ny, seed=21, nx=nx)
    ages = [1.5, 8.0, 40.0]
    angles = P.search_angles(-np.pi / 2, np.pi / 2)[::10]                 # 19 orientations, both ends
    pixels = _pixels(ny, nx, seed=4, n=64)
    fs = sl.fit_surface(_grid(z), _template("Scarp"), 20, pixels, ages=ages)
    sel = np.arange(0, 181, 10)
    assert np.array_equal(fs.angles[sel], angles)
    ref_amp, ref_snr = _oracle_planes(z, O.SCARP, 20, ages, angles)
    assert_surface_close(fs.amp[:, :, sel], fs.snr[:, :, sel], ref_amp, ref_snr, pixels)
    sl.release()


def _c3_pixels(stack, ages, angles, rng, n=256):
    """Seeded interior pixels, pixels next to the edge of the window limits (the un-masked
    rectangle of some templates ends there), and pixels whose sweep pick is an orientation at
    the +-90 degree seam or whose best SNR is low (where neighbours nearly tie)."""
    ny, nx = stack.shape[1:]
    snr, ang = stack[3], stack[2]
    out = [(int(r), int(c)) for r, c in zip(rng.integers(0, ny, 96), rng.integers(0, nx, 96))]
    valid_rows = np.flatnonzero((snr > 0).any(axis=1))
    r0, r1 = int(valid_rows[0]), int(valid_rows[-1])
    for r in (r0 - 1, r0, r0 + 1, r1 - 1, r1, r1 + 1):
        out += [(r, int(c)) for c in rng.integers(0, nx, 8)]
    seam = np.argwhere((snr > 0) & (np.abs(np.abs(ang) - np.pi / 2) < 1e-9))
    weak = np.argwhere((snr > 0) & (snr < np.quantile(snr[snr > 0], 0.02)))
    for cand in (seam, weak):
        if len(cand):
            out += [tuple(int(v) for v in cand[k]) for k in rng.choice(len(cand), min(len(cand), 56), replace=False)]
    return np.array(out[:n], dtype=np.int64)


@pytest.mark.gpu
def test_gpu_c3_surface_agrees_with_sweep(cuda_lib):
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    n = 4096
    z = synthetic_dem(n, seed=2)
    ages, angles = np.logspace(0, 3.5, 30), P.search_angles(-np.pi / 2, np.pi / 2)
    spec = _template("Scarp")._sb_spec
    with Plan(n, n, 1.0, 1.0) as plan:
        plan.set_dem(z)
        stack = _sweep(plan, spec, 100.0, ages, angles)
        pixels = _c3_pixels(stack, ages, angles, np.random.default_rng(8))
        amp, snr = plan.fit_surface(spec, 100.0, ages, angles, pixels[:, 0], pixels[:, 1])
    rep = check_against_sweep(amp, snr, stack, ages, angles, pixels,
                              _oracle_snr(lambda g, a: O.match_template(z, 1.0, 1.0, O.SCARP, 100.0, g, a)[3], ages, angles))
    save_report("surface_c3_vs_sweep", rep, {"config": "C3 4096^2 seed 2, Scarp 100, 30 ages x 181 angles, "
                                                       "%d pixels (interior, window-limit edge, +-90 seam, weak)"
                                                       % len(pixels)})
    assert rep["pixels"] == 256 and rep["valid"] > 150 and rep["unexplained"] == 0, rep


@pytest.mark.gpu
def test_gpu_masked_surface_agrees_with_sweep(cuda_lib):
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    n = 1024
    z = _gpu_holes(synthetic_dem(n, seed=3), seed=3, lake=(600, 420, 90))
    ages, angles = np.array([3.0, 30.0]), P.search_angles(-np.pi / 2, np.pi / 2)
    spec = _template("Scarp")._sb_spec
    with Plan(n, n, 1.0, 1.0, nodata="mask", min_coverage=0.7) as plan:
        plan.set_dem(z)
        stack = _sweep(plan, spec, 50.0, ages, angles)
        pixels = _c3_pixels(stack, ages, angles, np.random.default_rng(9))
        amp, snr = plan.fit_surface(spec, 50.0, ages, angles, pixels[:, 0], pixels[:, 1])
    rep = check_against_sweep(amp, snr, stack, ages, angles, pixels,
                              _oracle_snr(lambda g, a: MO.match_template_masked(z, 1.0, 1.0, O.SCARP, 50.0, g, a, 0.7)[3],
                                          ages, angles))
    bad = ~np.isfinite(z[pixels[:, 0], pixels[:, 1]])
    assert (snr[bad] == 0).all() and (amp[bad] == 0).all()
    save_report("surface_masked_1024_vs_sweep", rep, {"config": "1024^2 seed 3, border + cells + lake, Scarp 50, "
                                                                "2 ages x 181 angles, min_coverage 0.7"})
    assert rep["valid"] > 150 and rep["unexplained"] == 0, rep
