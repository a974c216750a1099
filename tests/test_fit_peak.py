"""Sub-grid fit peaks (``sb_peak_sweep``, ``sb_peak_finalize``, ``core.fit_peak``, DESIGN.md section 17):
each pixel's age and orientation between the grid points, from the SNR of the templates one age rank and
one orientation position either side of its winner, recorded by a second sweep of the same records.

Planes 0..3 must equal ``match`` bit for bit.  The four neighbour planes (``Plan.peak_planes``) are
checked exactly against a restatement built from every template's float32 SNR plane, taken from
one-orientation shares of the same search (``tests.parity.template_shares``); planes 5..7
against a NumPy float64 restatement of the formulas on those neighbours, bit for bit, and plane 4 (the
one ``exp10``) within 2 ulp.  The CPU cases run the emulator build of the kernels (tests/emu), the
``gpu`` cases the B200."""
import numpy as np
import pytest

from tests.parity import save_report, template_shares
from tests.test_nodata_mask import _gpu_holes, _holes
from tests.test_secondary_fit import positions_of


def _template(name):
    from scarplet_b200 import templates as T
    return getattr(T, name)


def _grid(z):
    import scarplet_b200 as sl
    return sl.DEMGrid(z, 1.0)


def _dem(shape, seed):
    from scarplet_b200.synth import synthetic_dem
    return synthetic_dem(shape[0], seed=seed, nx=shape[1])


# ---------------------------------------------------------------------------
# the contract, restated
# ---------------------------------------------------------------------------
class Winner(object):
    """Age rank ``r`` and orientation position ``p`` of each pixel's winner (planes 0..3 ``ref``), -1
    where the pixel has no fit."""

    def __init__(self, ref, ages, angles):
        from scarplet_b200 import params as P
        t = P.region_tables(ages, angles)
        self.tables, self.n_pos, self.periodic = t, len(t.pos_angle), t.periodic
        self.fit = ref[3] > 0
        self.nan = np.isnan(ref[3])
        self.r = np.where(self.fit, np.searchsorted(t.rank_age, np.where(self.fit, ref[1], t.rank_age[0])), -1)
        assert np.array_equal(t.rank_age[self.r[self.fit]], ref[1][self.fit])
        self.p = np.where(self.fit, positions_of(np.where(self.fit, ref[2], angles[0]), np.asarray(angles)), -1)

    def targets(self):
        """(rank, position) of the four neighbours [age-, age+, ang-, ang+] per pixel (-1: none)."""
        r, p, n = self.r, self.p, self.n_pos
        if self.periodic:
            pm, pp = (p - 1) % n, (p + 1) % n
        else:
            pm, pp = np.where(p > 0, p - 1, -1), np.where(p < n - 1, p + 1, -1)
        pm, pp = np.where(self.fit, pm, -1), np.where(self.fit, pp, -1)
        return [(r - 1, p), (r + 1, p), (r, pm), (r, pp)]


def restated_neighbours(z, spec, scale, ages, angles, ref, device=None, **plan_kw):
    """The four neighbour planes (float32 [4, rows, nx]) as the contract states them: per pixel with a fit,
    the largest candidate SNR > 0 among the templates at (r -+ 1, p) and (r, p -+ 1); 0 elsewhere.  More
    than 64 ages (one best state each in the shares) go in runs of at most 64."""
    import torch
    w = Winner(ref, ages, angles)
    ages = np.asarray(ages, dtype=np.float64)
    rank = np.argsort(np.argsort(ages, kind="stable"), kind="stable")
    tg = [(torch.as_tensor(tr, device=device), torch.as_tensor(tp, device=device)) for tr, tp in w.targets()]
    fit = torch.as_tensor(w.fit, device=device)
    out = torch.zeros((4,) + ref.shape[1:], dtype=torch.float32, device=device)
    for g0 in range(0, len(ages), 64):
        run = slice(g0, g0 + 64)
        shares = (template_shares(z, spec, scale, ages, angles, device, **plan_kw) if len(ages) <= 64 else
                  template_shares(z, spec, scale, ages, angles, run=run, **plan_kw))
        for i, snr, _ in shares:
            pos = i % w.n_pos
            for g, rk in enumerate(rank[run]):
                s = snr[g]
                for j, (tr, tp) in enumerate(tg):
                    q = fit & (tr == int(rk)) & (tp == pos) & (s > out[j])
                    out[j] = torch.where(q, s, out[j])
    return out.cpu().numpy()


def restated_peak(ref, nb, ages, angles):
    """Planes 4..7 of ``fit_peak`` from planes 0..3 ``ref`` and the neighbour planes ``nb``, in NumPy
    float64 with the kernel's operation order."""
    w = Winner(ref, ages, angles)
    G, n = len(ages), w.n_pos
    x = np.log10(w.tables.rank_age)
    step = angles[1] - angles[0] if len(angles) > 1 else 0.0
    fit, s0 = w.fit, np.where(w.fit, ref[3], 0.0)
    am, ap, gm, gp = (np.asarray(v, dtype=np.float64) for v in nb)
    age_pk, ang_pk = np.where(fit, ref[1], 0.0), np.where(fit, ref[2], 0.0)
    g_age, g_ang, refined = np.zeros_like(s0), np.zeros_like(s0), np.zeros_like(s0)
    with np.errstate(divide="ignore", invalid="ignore"):
        dm, dp = s0 - am, s0 - ap
        ok = fit & (w.r > 0) & (w.r < G - 1) & (am > 0) & (ap > 0) & (dm + dp > 0)
        if ok.any():
            r = np.clip(w.r, 1, G - 2)
            hm, hp = x[r] - x[r - 1], x[r + 1] - x[r]
            num = dm * (hp * hp) - dp * (hm * hm)
            u = num / (2.0 * (dm * hp + dp * hm))
            age_pk = np.where(ok, 10 ** (x[r] + u), age_pk)
            g_age = np.where(ok, u * num / (2.0 * hm * hp * (hm + hp)), 0.0)
            refined += ok
        dm, dp = s0 - gm, s0 - gp
        has = (n >= 3) if w.periodic else ((w.p > 0) & (w.p < n - 1))
        ok = fit & has & (gm > 0) & (gp > 0) & (dm + dp > 0)
        t, sm = dm - dp, dm + dp
        ang_pk = np.where(ok, ref[2] + (t / (2.0 * sm)) * step, ang_pk)
        g_ang = np.where(ok, (t * t) / (8.0 * sm), 0.0)
        refined += 2.0 * ok
    out = np.stack([age_pk, ang_pk, s0 + g_age + g_ang, refined])
    out[:, ~fit] = 0.0
    out[2][w.nan] = np.nan
    return out


def _ulp_close(a, b, n):
    return np.all(np.abs(a - b) <= n * np.spacing(np.maximum(np.abs(a), np.abs(b))))


def check_peak(got, ref, nb, ages, angles):
    """Planes 0..3 are ``ref``; planes 5..7 the restatement bit for bit, plane 4 within 2 ulp; the
    properties of the contract."""
    want = restated_peak(ref, nb, ages, angles)
    assert np.array_equal(got[:4], ref, equal_nan=True)
    assert np.array_equal(got[5:], want[1:], equal_nan=True)
    assert _ulp_close(got[4], want[0], 2)
    w = Winner(ref, ages, angles)
    fit, rf = w.fit, got[7].astype(int)
    assert (nb >= 0).all() and (nb[:, ~fit] == 0).all()
    assert (nb[:, fit] <= got[3][fit].astype(np.float32)).all()        # neighbours never beat the winner
    assert (got[4:][:, ~fit & ~w.nan] == 0).all()
    assert (got[6][fit] >= got[3][fit]).all()
    a, o = fit & (rf & 1 > 0), fit & (rf & 2 > 0)
    x = np.log10(w.tables.rank_age)
    if a.any():
        du = np.log10(got[4][a]) - np.log10(got[1][a])
        r = w.r[a]
        assert (du >= -(x[r] - x[r - 1]) / 2 - 1e-12).all() and (du <= (x[r + 1] - x[r]) / 2 + 1e-12).all()
    assert np.array_equal(got[4][fit & ~a], got[1][fit & ~a])
    assert np.array_equal(got[5][fit & ~o], got[2][fit & ~o])
    if len(angles) > 1:
        assert (np.abs(got[5][o] - got[2][o]) <= (angles[1] - angles[0]) / 2 * (1 + 1e-12)).all()
    # an axis without a neighbour is never refined
    G = len(ages)
    assert not (a & ((w.r == 0) | (w.r == G - 1) | (nb[0] == 0) | (nb[1] == 0))).any()
    if not w.periodic:
        assert not (o & ((w.p == 0) | (w.p == w.n_pos - 1))).any()
    assert not (o & ((nb[2] == 0) | (nb[3] == 0))).any()
    return a, o


def _two_pass(z, spec, scale, ages, angles, substreams=None, slab=None, curv=None, rows=None, **nodata):
    """On one plan: state 0's raw planes after match's sweep and after the peak pass, the neighbour
    planes (float32 [4, rows, nx]), ``peak_finalize``, its band ``rows`` and the curvature statistics."""
    from scarplet_b200 import params as P
    from scarplet_b200.distributed import _as_tensor
    from scarplet_b200.engine import Plan
    ny, nx = z.shape
    tables = P.region_tables(ages, angles)
    with Plan(ny, nx, 1.0, 1.0, slab=slab, **nodata) as plan:
        if substreams is not None:
            plan.set_option("fit_substreams", substreams)
        plan.set_dem(z)
        if curv is not None:
            plan.set_curv_stats(*curv)
        rows_n = plan.row_hi - plan.row_lo
        n = rows_n * nx

        def raw0():
            plan.sync()
            ps, pa, pi = plan.best_state_pointers(0)
            return [_as_tensor(p, n, k, None).numpy().tobytes() for p, k in ((ps, "f4"), (pa, "f4"), (pi, "i4"))]
        a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        before = raw0()
        plan.peak_sweep(a, t, tables)
        after = raw0()
        nb = _as_tensor(plan.peak_planes(), 4 * n, "f4", None).numpy().reshape(4, rows_n, nx).copy()
        out = plan.peak_finalize(age_of, angle_of, tables)
        band = None if rows is None else plan.peak_finalize(age_of, angle_of, tables, rows=rows)
        return before, after, nb, out, band, plan.curv_stats()


# ---------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------
def _scarp_dem(ny, nx, log_kt, strike, noise, seed):
    """A planar ramp plus one erf scarp of diffusion age kt = 10 ** log_kt whose profile runs along
    xr = x cos(strike) + y sin(strike), with white noise of ``noise`` m."""
    from scipy.special import erf
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:ny, 0:nx].astype(np.float64)
    xr = (x - x.mean()) * np.cos(strike) + (y - y.mean()) * np.sin(strike)
    z = 100.0 + 0.02 * x - 0.01 * y + 1.5 * erf(xr / (2.0 * np.sqrt(10.0 ** log_kt)))
    return z + noise * rng.standard_normal((ny, nx)), xr


def _cases():
    nan = _dem((64, 72), 21)
    nan[30, 41] = np.nan
    return {
        # name: (template, dem, scale, ages, (ang_min, ang_max), nodata kwargs)
        "scarp_odd": ("Scarp", _dem((73, 90), 4), 9, [2.0, 6.0, 20.0, 50.0], (-0.4, 0.4), {}),
        "channel_wrap": ("Channel", _dem((64, 70), 5), 5, [0.1, 0.15, 0.2, 0.3], (-0.3, 0.3), {}),  # no edge mask
        "upper_break": ("RightFacingUpperBreakScarp", _dem((64, 80), 6), 9, [2.0, 6.0, 20.0], (-0.4, 0.4),
                        {}),                                                                       # get_err_mask
        "mask_holes": ("Scarp", _holes(_dem((72, 80), 2), "border+cells", seed=2), 9, [1.5, 4.0, 12.0], (-0.4, 0.4),
                       dict(nodata="mask", min_coverage=0.6)),
        "propagate_nan": ("Scarp", nan, 9, [2.0, 6.0, 15.0], (-0.3, 0.3), {}),
        # a scarp facing along y: winners at and next to +-90 degrees
        "periodic": ("Scarp", _scarp_dem(40, 44, 0.7, np.pi / 2, 2e-3, 8)[0], 6, [2.0, 5.0, 12.0],
                     (-np.pi / 2, np.pi / 2), {}),
        "linear_ends": ("Scarp", _dem((48, 52), 9), 6, [2.0, 5.0, 12.0], (-np.pi / 4, np.pi / 4), {}),
        "unsorted_ages": ("Scarp", _dem((56, 60), 10), 8, [20.0, 2.0, 50.0, 6.0], (-0.3, 0.3), {}),
        "single_age": ("Scarp", _dem((56, 60), 11), 8, [6.0], (-0.3, 0.3), {}),
        "ages_70": ("Scarp", _dem((40, 48), 12), 6, list(np.linspace(1.0, 60.0, 70)), (-0.05, 0.05), {}),
    }


@pytest.mark.parametrize("case", list(_cases()))
def test_peak_restated(emu_lib, case):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    tmpl, z, scale, ages, span, masking = _cases()[case]
    Template = _template(tmpl)
    kw = dict(ang_min=span[0], ang_max=span[1], **masking)
    angles = P.search_angles(*span)
    ref = np.stack(sl.match(_grid(z), Template, scale=scale, ages=ages, **kw))
    got = sl.fit_peak(_grid(z), Template, scale, ages=ages, **kw)
    assert got.shape == (8,) + z.shape and got.dtype == np.float64
    before, after, nb, out, _, _ = _two_pass(z, Template._sb_spec, scale, ages, angles, **masking)
    assert before == after                                   # state 0 byte for byte
    assert np.array_equal(out, got, equal_nan=True)
    want = restated_neighbours(z, Template._sb_spec, scale, ages, angles, ref, **masking)
    assert np.array_equal(nb, want)
    a, o = check_peak(got, ref, nb, ages, angles)
    w = Winner(ref, ages, angles)
    if case == "single_age":
        assert not a.any() and o.sum() > 100
    elif case == "ages_70":
        assert a.sum() > 100
    elif case != "propagate_nan":             # (the NaN's windows cover most of this raster)
        assert a.sum() > 5 and o.sum() > 100, (a.sum(), o.sum())
    if case == "propagate_nan":
        nan = np.isnan(ref[3])
        assert nan.any() and np.isnan(got[6][nan]).all() and (got[[4, 5, 7]][:, nan] == 0).all()
    if case == "periodic":
        # winners at +-90 degrees (position 0), whose orientation- neighbour wraps round to n_pos - 1,
        # and winners at positions 1 and n_pos - 1, whose neighbour at position 0 is the twin pair
        assert (o & (w.p == 0)).sum() > 0
        assert (o & ((w.p == 1) | (w.p == w.n_pos - 1))).sum() > 0
        assert (got[2] == angles[-1]).sum() > 0                 # a +90 degree winner: position 0 too
    if case == "linear_ends":
        assert (w.fit & (w.p == 0)).sum() > 0 and (w.fit & (w.p == w.n_pos - 1)).sum() > 0
    if case == "mask_holes":
        assert (got[:, ~np.isfinite(z)] == 0).all()
    sl.release()


def test_neighbours_below_match_ages(emu_lib):
    """Each age neighbour is at most the best SNR over every orientation at its age (``match_ages``)."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    z = _dem((56, 64), 14)
    ages, span = [1.5, 4.0, 10.0, 25.0], (-0.4, 0.4)
    angles = P.search_angles(*span)
    spec = _template("Scarp")._sb_spec
    per_age = sl.match_ages(_grid(z), _template("Scarp"), 8, ages=ages, ang_min=span[0], ang_max=span[1])
    _, _, nb, out, _, _ = _two_pass(z, spec, 8, ages, angles)
    w = Winner(out[:4], ages, angles)
    srt = np.sort(ages)
    for j, dr in ((0, -1), (1, 1)):
        has = w.fit & (w.r + dr >= 0) & (w.r + dr < len(ages)) & (nb[j] > 0)
        assert has.sum() > 100
        best = np.stack([per_age[float(a)][3] for a in srt])          # [rank, ny, nx]
        at = best[np.clip(w.r + dr, 0, len(ages) - 1), np.arange(z.shape[0])[:, None], np.arange(z.shape[1])]
        assert (nb[j][has] <= at[has]).all()
    sl.release()


@pytest.mark.parametrize("masking", [{}, dict(nodata="mask", min_coverage=0.6)])
def test_substreams(emu_lib, masking):
    """A raster this small deals the fit kernel's templates to sub-streams: the neighbour planes and the
    result are the same with one."""
    from scarplet_b200 import params as P
    z = _dem((64, 72), 13)
    if masking:
        z = _holes(z, "border+cells", seed=13)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-np.pi / 2, np.pi / 2)[::6]
    spec = _template("Scarp")._sb_spec
    auto = _two_pass(z, spec, 7, ages, angles, **masking)
    one = _two_pass(z, spec, 7, ages, angles, substreams=1, **masking)
    assert auto[0] == one[0]
    assert np.array_equal(auto[2], one[2])
    assert np.array_equal(auto[3], one[3], equal_nan=True)
    assert (auto[3][7] > 0).sum() > 300


def test_row_slabs(emu_lib):
    """Row bands of a plan equal its whole result; row slabs (spatial_search's plans: halo, shared
    curvature statistics) give neighbour planes equal to the restatement of their own sweep."""
    from scarplet_b200 import distributed as D, params as P
    ny, nx = 70, 64
    z = _dem((ny, nx), 19)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-0.4, 0.4)
    spec = _template("Scarp")._sb_spec
    whole = _two_pass(z, spec, 8, ages, angles, rows=(11, 40))
    assert np.array_equal(whole[4], whole[3][:, 11:40])
    halo = D.slab_halo(spec, 8, ages, angles, nx, ny, 1.0)
    for lo, hi in ((0, 33), (33, ny)):
        before, after, nb, out, band, _ = _two_pass(z, spec, 8, ages, angles, slab=(lo, hi, halo), curv=whole[5],
                                                    rows=(lo + 3, lo + 20))
        assert out.shape == (8, hi - lo, nx) and nb.shape == (4, hi - lo, nx)
        assert before == after
        assert np.array_equal(band, out[:, 3:20])
        want = restated_neighbours(z, spec, 8, ages, angles, out[:4], slab=(lo, hi, halo), curv=whole[5])
        assert np.array_equal(nb, want)
        check_peak(out, out[:4], nb, ages, angles)
        assert (out[7] > 0).sum() > 200


def test_recovery(emu_lib):
    """An erf scarp at an off-grid age (kt = 10^1.25, half way between two default ages) and an off-grid
    strike (0.3 rad = 17.19 deg, which the search reports as the orientation -0.3 rad), 1 mm of noise,
    Scarp templates of half-length 30 on the default ages: on the scarp's interior pixels the peak
    beats the grid on both axes.  Measured here (DESIGN.md section 17): median |log10 age error| 0.0289
    against the grid's 0.0500 (0.58x: the SNR falls off faster towards younger ages, so the parabola's
    vertex leans towards the older winner), median orientation error 0.067 deg against 0.189 deg."""
    import scarplet_b200 as sl
    ny, nx, log_kt, strike = 96, 96, 1.25, 0.3
    z, xr = _scarp_dem(ny, nx, log_kt, strike, 1e-3, seed=3)
    got = sl.fit_peak(_grid(z), _template("Scarp"), 30, ang_min=-np.radians(40.0), ang_max=np.radians(40.0))
    sl.release()
    yy, xx = np.mgrid[0:ny, 0:nx]
    inner = (np.abs(xr) <= 1.0) & (yy > 25) & (yy < ny - 25) & (xx > 25) & (xx < nx - 25) & (got[3] > 0)
    assert inner.sum() > 50 and (got[7][inner] == 3).all()
    e_age_grid = np.median(np.abs(np.log10(got[1][inner]) - log_kt))
    e_age_peak = np.median(np.abs(np.log10(got[4][inner]) - log_kt))
    e_ang_grid = np.median(np.abs(got[2][inner] + strike))
    e_ang_peak = np.median(np.abs(got[5][inner] + strike))
    assert e_age_peak <= 0.6 * e_age_grid, (e_age_peak, e_age_grid)
    assert e_ang_peak <= 0.5 * e_ang_grid, (np.degrees(e_ang_peak), np.degrees(e_ang_grid))


def test_refusals(emu_lib):
    import scarplet_b200 as sl
    import scarplet_b200.core as C
    from scarplet_b200 import params as P
    from scarplet_b200._lib import SbError, check
    from scarplet_b200.engine import Plan
    from tests.plugin_templates import ShiftedRidge
    ny, nx = 40, 48
    z = _dem((ny, nx), 1)
    grid, Scarp = _grid(z), _template("Scarp")
    kw = dict(ages=[2.0, 3.0], ang_min=-0.1, ang_max=0.1)
    sl.fit_peak(grid, Scarp, 8, **kw)                    # leaves this raster's plan in the cache

    def count():
        # a refusal must come before any device work: the cached plan launches nothing
        return [p.launches for _, p in C._cache]
    launches = count()
    assert launches
    with pytest.raises(ValueError, match="built-in"):
        sl.fit_peak(grid, ShiftedRidge, 8, **kw)
    with pytest.raises(ValueError, match="keyword"):
        sl.fit_peak(grid, Scarp, 8, shift=1, **kw)
    with pytest.raises(ValueError, match="duplicate"):
        sl.fit_peak(grid, Scarp, 8, ages=[2.0, 3.0, 2.0], ang_min=-0.1, ang_max=0.1)
    with pytest.raises(ValueError, match="at least one age"):
        sl.fit_peak(grid, Scarp, 8, ages=[], ang_min=-0.1, ang_max=0.1)
    with pytest.raises(ValueError, match="65535 ages"):
        sl.fit_peak(grid, Scarp, 8, ages=np.arange(1.0, 65537.0), ang_min=-0.1, ang_max=0.1)
    with pytest.raises(ValueError, match="65535 orientations"):
        sl.fit_peak(grid, Scarp, 8, ages=[2.0], ang_min=0.0, ang_max=1200.0)
    assert count() == launches
    # a single orientation: nothing to refine on that axis
    one = sl.fit_peak(grid, Scarp, 8, ages=[2.0, 3.0, 5.0], ang_min=0.05, ang_max=0.05)
    assert not (one[7].astype(int) & 2).any() and np.array_equal(one[5], one[2])

    spec = Scarp._sb_spec
    ages, angles = [2.0, 3.0], P.search_angles(-0.1, 0.1)
    tables = P.region_tables(ages, angles)
    n_pos, n_ranks = len(tables.pos_angle), len(ages)
    with Plan(ny, nx, 1.0, 1.0, slab=(10, 30, 20)) as plan:
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(spec, 8, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        with pytest.raises(SbError, match="no peak sweep"):
            plan.peak_planes()
        with pytest.raises(SbError, match="no peak sweep"):
            plan.peak_finalize(age_of, angle_of, tables)
        plan.peak_sweep(a, t, tables)
        assert plan.peak_finalize(age_of, angle_of, tables).shape == (8, 20, nx)
        rank = np.ascontiguousarray(tables.age_rank)
        pos = np.ascontiguousarray(tables.angle_pos)

        def sweep(rank=rank, pos=pos, n_ranks=n_ranks, n_pos=n_pos, periodic=0, recs=t):
            check(plan.lib, plan.lib.sb_peak_sweep(plan._h, a[0], a[1], recs[0], recs[1], None, rank.ctypes.data,
                                                   pos.ctypes.data, len(pos), n_ranks, n_pos, periodic))
        for bad in (0, 65536):
            with pytest.raises(SbError, match="n_ranks"):
                sweep(n_ranks=bad)
            with pytest.raises(SbError, match="n_pos"):
                sweep(n_pos=bad)
        with pytest.raises(SbError, match="periodic"):
            sweep(n_pos=2, pos=(pos % 2).astype(np.int32), periodic=1)
        with pytest.raises(SbError, match="out of range"):
            sweep(pos=np.where(pos == 0, n_pos, pos).astype(np.int32))
        with pytest.raises(SbError, match="out of range"):
            sweep(rank=np.full_like(rank, n_ranks))
        with pytest.raises(SbError, match="out of range"):
            sweep(rank=np.full_like(rank, -1))
        with pytest.raises(SbError, match="flat index"):
            sweep(pos=pos[:-1].copy(), rank=rank[:-1].copy())
        # records of another best state
        a2, t2, _, _ = plan.build_sweep(spec, 8, ages, angles, state_per_age=True)
        with pytest.raises(SbError, match="state"):
            plan.peak_sweep(a2, t2, tables)
        sweep()
        lx = np.log10(tables.rank_age)

        def fin(n_ranks=n_ranks, n_pos=n_pos, rows=(10, 30), step=0.01):
            out = np.empty((8, rows[1] - rows[0], nx))
            check(plan.lib, plan.lib.sb_peak_finalize(plan._h, rows[0], rows[1], age_of.ctypes.data,
                                                      angle_of.ctypes.data, len(age_of), lx.ctypes.data, n_ranks,
                                                      n_pos, 0, step, out.ctypes.data))
        fin()
        with pytest.raises(SbError, match="n_ranks / n_pos"):
            fin(n_ranks=n_ranks + 1)
        with pytest.raises(SbError, match="n_ranks / n_pos"):
            fin(n_pos=n_pos - 1)
        with pytest.raises(SbError, match="rows outside"):
            fin(rows=(5, 30))
        with pytest.raises(SbError, match="step"):
            fin(step=np.nan)
        # a new best-state layout voids the planes
        plan.set_states(2)
        with pytest.raises(SbError, match="no peak sweep"):
            plan.peak_planes()
    for option, value in (("precision", 64), ("fast", 0)):
        with Plan(ny, nx, 1.0, 1.0) as plan:
            plan.set_option(option, value)
            plan.set_dem(z)
            a, t, age_of, angle_of = plan.build_sweep(spec, 8, ages, angles)
            plan.reset()
            plan.sweep(a, t)
            with pytest.raises(SbError, match="precision 32 and the option fast"):
                plan.peak_sweep(a, t, tables)
    assert np.array_equal(z, _dem((ny, nx), 1))
    sl.release()


# ---------------------------------------------------------------------------
# on the B200
# ---------------------------------------------------------------------------
C3_AGES = np.logspace(0, 3.5, 30)


@pytest.mark.gpu
def test_gpu_c3_peak(cuda_lib):
    """C3 (4096^2 seed 2, Scarp 100, 30 ages x 181 orientations): planes 0..3 are match."""
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(4096, seed=2)
    grid, Scarp = _grid(z), _template("Scarp")
    got = sl.fit_peak(grid, Scarp, 100.0, ages=C3_AGES)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=C3_AGES))
    eq_match = bool(np.array_equal(got[:4], ref, equal_nan=True))
    del ref
    fit, rf = got[3] > 0, got[7].astype(int)
    save_report("c3_peak", {"planes_0_3_array_equal_match": eq_match, "valid": int(fit.sum()),
                            "age_refined": int((rf & 1 > 0).sum()), "angle_refined": int((rf & 2 > 0).sum()),
                            "snr_gain_p50": float(np.median(got[6][fit] / got[3][fit]))},
                {"config": "C3 4096^2 seed 2, Scarp 100, 30 ages x 181 orientations"})
    assert eq_match
    assert (got[6][fit] >= got[3][fit]).all()
    sl.release()


def _gpu_restated(name, z, masked):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    grid, Scarp = _grid(z), _template("Scarp")
    ages = C3_AGES[::5]
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    got = sl.fit_peak(grid, Scarp, 100.0, ages=ages, **masked)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=ages, **masked))
    sl.release()
    _, _, nb, out, _, _ = _two_pass_gpu(z, Scarp._sb_spec, 100.0, ages, angles, **masked)
    want = restated_neighbours(z, Scarp._sb_spec, 100.0, ages, angles, ref, device="cuda:0", **masked)
    eq_nb = [bool(np.array_equal(nb[j], want[j])) for j in range(4)]
    eq_out = bool(np.array_equal(out, got, equal_nan=True))
    pk = restated_peak(ref, nb, ages, angles)
    eq_5_7 = bool(np.array_equal(got[5:], pk[1:], equal_nan=True))
    ulp4 = bool(_ulp_close(got[4], pk[0], 2))
    rf = got[7].astype(int)
    save_report(name, {"planes_0_3_array_equal_match": bool(np.array_equal(got[:4], ref, equal_nan=True)),
                       "neighbour_planes_array_equal_restated": eq_nb, "plan_equals_fit_peak": eq_out,
                       "planes_5_7_array_equal_numpy": eq_5_7, "plane_4_within_2ulp": ulp4,
                       "valid": int((ref[3] > 0).sum()), "age_refined": int((rf & 1 > 0).sum()),
                       "angle_refined": int((rf & 2 > 0).sum())},
                {"config": "1024^2 seed 6, Scarp 100, 6 ages (C3's every fifth) x 181 orientations" +
                           (", ~10 %% nodata, min_coverage %g" % masked["min_coverage"] if masked else "")})
    assert np.array_equal(got[:4], ref, equal_nan=True)
    assert all(eq_nb), eq_nb
    assert eq_out and eq_5_7 and ulp4
    check_peak(got, ref, nb, ages, angles)
    return got


def _two_pass_gpu(z, spec, scale, ages, angles, **nodata):
    """``_two_pass`` on the device: the neighbour planes are copied out through torch."""
    import torch
    from scarplet_b200 import params as P
    from scarplet_b200.distributed import _as_tensor
    from scarplet_b200.engine import Plan
    ny, nx = z.shape
    tables = P.region_tables(ages, angles)
    with Plan(ny, nx, 1.0, 1.0, **nodata) as plan:
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        plan.peak_sweep(a, t, tables)
        plan.sync()
        nb = _as_tensor(plan.peak_planes(), 4 * ny * nx, "f4", "cuda:0").reshape(4, ny, nx).cpu().numpy()
        torch.cuda.synchronize()
        out = plan.peak_finalize(age_of, angle_of, tables)
        return None, None, nb, out, None, None


@pytest.mark.gpu
def test_gpu_1024_restated(cuda_lib):
    """1024^2 seed 6, 6 ages x 181 orientations: the neighbour planes equal the share restatement
    (181 one-orientation shares, folded on the device), planes 5..7 the NumPy restatement."""
    from scarplet_b200.synth import synthetic_dem
    got = _gpu_restated("restated_1024", synthetic_dem(1024, seed=6), {})
    assert ((got[7].astype(int) & 3) == 3).sum() > 1000


@pytest.mark.gpu
def test_gpu_1024_masked(cuda_lib):
    """The same with ~10 % nodata at min_coverage 0.7."""
    from scarplet_b200.synth import synthetic_dem
    z = _gpu_holes(synthetic_dem(1024, seed=6), seed=6)
    assert 0.09 < np.mean(~np.isfinite(z)) < 0.12
    got = _gpu_restated("masked_1024_peak", z, dict(nodata="mask", min_coverage=0.7))
    assert (got[:, ~np.isfinite(z)] == 0).all()


@pytest.mark.gpu
def test_gpu_neighbours_vs_fit_surface(cuda_lib):
    """An independent path: at a few hundred pixels the neighbour values agree with ``fit_surface``'s
    float64 SNR of the same templates within the parity bound (1e-4 relative above the median SNR,
    DESIGN.md section 4)."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(1024, seed=6)
    Scarp = _template("Scarp")
    ages = C3_AGES[::5]
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    _, _, nb, out, _, _ = _two_pass_gpu(z, Scarp._sb_spec, 100.0, ages, angles)
    w = Winner(out[:4], ages, angles)
    rng = np.random.default_rng(0)
    cand = np.argwhere(w.fit & (nb > 0).all(axis=0))
    px = cand[rng.choice(len(cand), size=min(300, len(cand)), replace=False)]
    surf = sl.fit_surface(_grid(z), Scarp, 100.0, px, ages=ages)
    sl.release()
    rank = np.argsort(np.argsort(ages, kind="stable"), kind="stable")
    g_of_rank = np.argsort(rank)
    A = len(angles)
    med = np.median(out[3][w.fit])
    errs = []
    for j, (tr, tp) in enumerate(w.targets()):
        r, p = tr[px[:, 0], px[:, 1]], tp[px[:, 0], px[:, 1]]
        g = g_of_rank[r]
        s64 = surf.snr[np.arange(len(px)), g, p]
        if w.periodic:                             # position 0: the larger of the +-90 degree twins
            s64 = np.where(p == 0, np.maximum(s64, surf.snr[np.arange(len(px)), g, A - 1]), s64)
        v = nb[j][px[:, 0], px[:, 1]].astype(np.float64)
        above = s64 > med
        errs.append(np.abs(v - s64)[above] / s64[above])
    e = np.concatenate(errs)
    save_report("neighbours_vs_fit_surface", {"pixels": int(len(px)), "values_above_median": int(e.size),
                                              "rel_err_max": float(e.max()), "rel_err_p50": float(np.median(e))},
                {"config": "1024^2 seed 6, Scarp 100, 6 ages x 181 orientations, 300 random pixels with four "
                           "neighbours; values above the median SNR"})
    assert e.size > 100 and e.max() <= 1e-4, (e.size, e.max())
