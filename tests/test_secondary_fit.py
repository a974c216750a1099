"""Secondary fits (``sb_secondary_sweep``, ``core.secondary_fit``, DESIGN.md section 16): the best
template at least a chosen number of orientation positions from each pixel's best, from a second sweep
of the same records into best state 1.

Planes 0..3 must equal ``match`` bit for bit.  Planes 4..7 are checked exactly against a NumPy / torch
restatement of the contract, built from every template's float32 SNR and amplitude planes:
one-orientation shares of the same search (``build_sweep(angle_slice=(i, i + 1),
state_per_age=True)``, which pass the whole search's extents to ``sb_sweep_ex``) leave in state g the
SNR and amplitude of template (age g, orientation i) wherever it is a candidate, bit for bit.  The CPU
cases run the emulator build of the kernels (tests/emu), the ``gpu`` cases the B200."""
import numpy as np
import pytest

from tests.parity import save_report, template_shares
from tests.test_nodata_mask import _gpu_holes, _holes


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
def position_distance(p, q, n_pos, periodic):
    d = np.abs(np.asarray(p) - np.asarray(q))
    return np.minimum(d, n_pos - d) if periodic else d


def positions_of(angle, angles):
    """Orientation positions (``params.region_tables``) of the decoded angles ``angle`` (each one of
    ``angles`` exactly)."""
    from scarplet_b200 import params as P
    t = P.region_tables([1.0], angles)
    ai = np.clip(np.searchsorted(angles, angle), 0, len(angles) - 1)
    assert np.array_equal(angles[ai], angle)
    return ai % len(t.pos_angle)


class Restated(object):
    """Planes 4..7 of the contract, folded one orientation at a time from the per-template float32
    SNR and amplitude planes ([ages, rows, nx] torch tensors, on the device for the gpu cases) and
    planes 0..3 of ``match``: the qualifying template with the highest SNR, then the lowest flat
    index (``g * len(angles) + i`` for age g and orientation i)."""

    def __init__(self, ref, ages, angles, min_sep_pos, device=None):
        import torch
        from scarplet_b200 import params as P
        self.torch, self.device = torch, device
        t = P.region_tables(ages, angles)
        self.n_pos, self.periodic = len(t.pos_angle), t.periodic
        self.ages, self.angles, self.m = np.asarray(ages, dtype=np.float64), np.asarray(angles), int(min_sep_pos)
        self.ref = ref
        self.fit = ref[3] > 0
        self.nan = np.isnan(ref[3])
        self.pstar = np.where(self.fit, positions_of(np.where(self.fit, ref[2], angles[0]), self.angles), -1)
        shape = ref.shape[1:]
        self.snr = torch.zeros(shape, dtype=torch.float32, device=device)
        self.amp = torch.zeros(shape, dtype=torch.float32, device=device)
        self.idx = torch.full(shape, np.iinfo(np.int64).max, dtype=torch.int64, device=device)

    def add(self, i, snr, amp):
        torch = self.torch
        d = position_distance(i % self.n_pos, self.pstar, self.n_pos, self.periodic)
        admit = torch.as_tensor(self.fit & (d >= self.m), device=self.device)
        A = len(self.angles)
        for g in range(len(self.ages)):
            s, k = snr[g], g * A + i
            q = admit & (s > 0) & ((s > self.snr) | ((s == self.snr) & (k < self.idx)))
            self.snr = torch.where(q, s, self.snr)
            self.amp = torch.where(q, amp[g], self.amp)
            self.idx = torch.where(q, torch.full_like(self.idx, k), self.idx)

    def planes(self):
        s = self.snr.cpu().numpy().astype(np.float64)
        a = self.amp.cpu().numpy().astype(np.float64)
        k = self.idx.cpu().numpy()
        hit = s > 0
        kk = np.where(hit, k, 0)
        A = len(self.angles)
        out = np.stack([np.where(hit, a, 0.0), np.where(hit, self.ages[kk // A], 0.0),
                        np.where(hit, self.angles[kk % A], 0.0), np.where(hit, s, 0.0)])
        out[0][self.nan] = np.nan
        out[3][self.nan] = np.nan
        return out


def restated_planes(z, spec, scale, ages, angles, ref, min_sep_pos, device=None, **plan_kw):
    """Planes 4..7 of ``secondary_fit`` as the contract states them, for planes 0..3 ``ref``."""
    r = Restated(ref, ages, angles, min_sep_pos, device)
    for i, snr, amp in template_shares(z, spec, scale, ages, angles, device, **plan_kw):
        r.add(i, snr, amp)
    return r.planes()


def restated_multi(z, spec, scale, ages, angles, ref, seps, **plan_kw):
    """``restated_planes`` at several separations from one pass over the shares."""
    rs = [Restated(ref, ages, angles, m) for m in seps]
    for i, snr, amp in template_shares(z, spec, scale, ages, angles, **plan_kw):
        for r in rs:
            r.add(i, snr, amp)
    return [r.planes() for r in rs]


# ---------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------
def test_separation_positions():
    """The separation is a whole number of positions: ceil(min_separation / step - 1e-9)."""
    from scarplet_b200 import params as P
    full = P.search_angles(-np.pi / 2, np.pi / 2)
    assert P.separation_positions(np.radians(10.0), full) == 10
    assert P.separation_positions(np.radians(45.0), full) == 45
    assert P.separation_positions(np.radians(10.5), full) == 11
    assert P.separation_positions(np.radians(1.0), full) == 1
    assert P.separation_positions(np.radians(90.0), full) == 90           # n_pos // 2 of a periodic search
    lin = P.search_angles(-0.4, 0.4)
    assert P.separation_positions(np.radians(5.0), lin) == 5
    assert P.separation_positions((len(lin) - 1) * (lin[1] - lin[0]), lin) == len(lin) - 1
    for bad in (0.0, -0.1, np.nan, np.inf, -np.inf, np.radians(90.5)):
        with pytest.raises(ValueError, match="min_separation"):
            P.separation_positions(bad, full)
    with pytest.raises(ValueError, match="min_separation"):
        P.separation_positions(len(lin) * (lin[1] - lin[0]), lin)
    with pytest.raises(ValueError, match="2 orientations"):
        P.separation_positions(0.1, P.search_angles(0.0, 0.0))
    assert position_distance(0, 179, 180, True) == 1 and position_distance(0, 179, 180, False) == 179


def _cases():
    nan = _dem((64, 72), 21)
    nan[30, 41] = np.nan
    return {
        # name: (template, dem, scale, ages, (ang_min, ang_max), nodata kwargs)
        "scarp_odd": ("Scarp", _dem((73, 90), 4), 9, [2.0, 6.0, 20.0], (-0.4, 0.4), {}),
        "channel_wrap": ("Channel", _dem((64, 70), 5), 5, [0.15, 0.2, 0.3], (-0.3, 0.3), {}),   # no edge mask
        "upper_break": ("RightFacingUpperBreakScarp", _dem((64, 80), 6), 9, [2.0, 6.0, 20.0], (-0.4, 0.4),
                        {}),                                                                       # get_err_mask
        "mask_holes": ("Scarp", _holes(_dem((72, 80), 2), "border+cells", seed=2), 9, [1.5, 4.0, 12.0], (-0.4, 0.4),
                       dict(nodata="mask", min_coverage=0.6)),
        "propagate_nan": ("Scarp", nan, 9, [2.0, 6.0], (-0.3, 0.3), {}),
        "periodic": ("Scarp", _dem((40, 44), 8), 6, [2.0, 8.0], (-np.pi / 2, np.pi / 2), {}),
    }


# per case: two separations in degrees; the periodic search's 80 degrees reaches across +-90
_SEPS = {"scarp_odd": (5.0, 20.0), "channel_wrap": (3.0, 12.0), "upper_break": (5.0, 20.0),
         "mask_holes": (4.0, 15.0), "propagate_nan": (3.0, 10.0), "periodic": (10.0, 80.0)}


@pytest.mark.parametrize("case", ["scarp_odd", "channel_wrap", "upper_break", "mask_holes", "propagate_nan",
                                  "periodic"])
def test_secondary_restated(emu_lib, case):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    tmpl, z, scale, ages, span, masking = _cases()[case]
    Template = _template(tmpl)
    kw = dict(ang_min=span[0], ang_max=span[1], **masking)
    angles = P.search_angles(*span)
    ref = np.stack(sl.match(_grid(z), Template, scale=scale, ages=ages, **kw))
    seps = [np.radians(d) for d in _SEPS[case]]
    ms = [P.separation_positions(s, angles) for s in seps]
    wants = restated_multi(z, Template._sb_spec, scale, ages, angles, ref, ms, **masking)
    n_pos = len(P.region_tables(ages, angles).pos_angle)
    fit = ref[3] > 0
    for sep, m, want in zip(seps, ms, wants):
        got = sl.secondary_fit(_grid(z), Template, scale, sep, ages=ages, **kw)
        assert got.shape == (8,) + z.shape and got.dtype == np.float64
        assert np.array_equal(got[:4], ref, equal_nan=True)
        assert np.array_equal(got[4:], want, equal_nan=True)
        second = got[7] > 0
        assert (got[4:][:, ~fit & ~np.isnan(ref[3])] == 0).all()
        assert not (second & ~fit).any()
        if case == "propagate_nan":
            nan = np.isnan(ref[3])
            assert nan.any() and np.isnan(got[7][nan]).all() and (got[5:7][:, nan] == 0).all()
        else:
            assert second.sum() > 100, (case, m, second.sum())
            # a secondary fit is never better than the pixel's best
            assert (got[7][second] <= got[3][second]).all()
        d = position_distance(positions_of(got[6][second], angles), positions_of(got[2][second], angles),
                              n_pos, P.region_tables(ages, angles).periodic)
        assert (d >= m).all()
    if case == "periodic":
        # the wide separation's pairs reach across +-90 degrees: position distance shorter than |index difference|
        got = sl.secondary_fit(_grid(z), Template, scale, seps[1], ages=ages, **kw)
        second = got[7] > 0
        ia = np.abs(np.searchsorted(angles, got[6][second]) - np.searchsorted(angles, got[2][second]))
        assert (ia > n_pos // 2).sum() > 0
    if case == "mask_holes":
        assert (got[:, ~np.isfinite(z)] == 0).all()
    sl.release()


def test_separation_properties(emu_lib):
    """snr2 does not grow with the separation; a secondary fit within ratio r of the best lies in
    ``fit_region``'s region at r, whose arc then spans at least the separation."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    z = _dem((72, 76), 23)
    grid, Scarp = _grid(z), _template("Scarp")
    ages, kw = [1.5, 4.0, 10.0], dict(ang_min=-np.pi / 2, ang_max=np.pi / 2)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    step = angles[1] - angles[0]
    degs = [1.0, 4.0, 10.0, 30.0, 60.0, 90.0]
    got = {d: sl.secondary_fit(grid, Scarp, 8, np.radians(d), ages=ages, **kw) for d in degs}
    for d0, d1 in zip(degs[:-1], degs[1:]):
        assert np.array_equal(got[d0][:4], got[d1][:4])
        assert (got[d1][7] <= got[d0][7]).all()
        assert (got[d1][7] < got[d0][7]).sum() > 0
    ratio = 0.5
    reg = sl.fit_region(grid, Scarp, 8, ratio, ages=ages, **kw)
    for d in degs:
        m = P.separation_positions(np.radians(d), angles)
        g = got[d]
        near = (g[7] > 0) & (g[7] >= ratio * g[3])
        if d <= 30.0:
            assert near.sum() > 20, (d, near.sum())
        assert (reg[8][near] >= 2).all()
        span = np.rint((reg[7][near] - reg[6][near]) / step).astype(int)
        assert (span >= m).all()
    sl.release()


def _two_sweeps(z, spec, scale, ages, angles, m, substreams=None, slab=None, curv=None, rows=None, **nodata):
    """On one plan with 2 states: state 0's raw planes and finalize after match's sweep, the same after
    the secondary sweep, state 1's finalize and the band ``rows`` of it."""
    from scarplet_b200 import params as P
    from scarplet_b200.distributed import _as_tensor
    from scarplet_b200.engine import Plan
    ny, nx = z.shape
    tables = P.region_tables(ages, angles)
    with Plan(ny, nx, 1.0, 1.0, states=2, slab=slab, **nodata) as plan:
        if substreams is not None:
            plan.set_option("fit_substreams", substreams)
        plan.set_dem(z)
        if curv is not None:
            plan.set_curv_stats(*curv)
        n = (plan.row_hi - plan.row_lo) * nx

        def raw0():
            plan.sync()
            ps, pa, pi = plan.best_state_pointers(0)
            return [_as_tensor(p, n, k, None).numpy().tobytes() for p, k in ((ps, "f4"), (pa, "f4"), (pi, "i4"))]
        a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        before = raw0(), plan.finalize(age_of, angle_of).copy()
        plan.secondary_sweep(a, t, tables, m)
        after = raw0(), plan.finalize(age_of, angle_of).copy()
        second = plan.finalize(age_of, angle_of, state=1).copy()
        band = None if rows is None else plan.finalize(age_of, angle_of, state=1, rows=rows).copy()
        return before, after, second, band, plan.curv_stats()


@pytest.mark.parametrize("masking", [{}, dict(nodata="mask", min_coverage=0.6)])
def test_substreams_and_state0_untouched(emu_lib, masking):
    """A raster this small deals the fit kernel's templates to sub-streams: state 1 is the same with
    one; the secondary sweep leaves state 0's three planes byte for byte as they were."""
    from scarplet_b200 import params as P
    z = _dem((64, 72), 13)
    if masking:
        z = _holes(z, "border+cells", seed=13)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-np.pi / 2, np.pi / 2)[::6]
    spec = _template("Scarp")._sb_spec
    auto = _two_sweeps(z, spec, 7, ages, angles, 3, **masking)
    one = _two_sweeps(z, spec, 7, ages, angles, 3, substreams=1, **masking)
    for before, after, second, _, _ in (auto, one):
        assert before[0] == after[0]
        assert np.array_equal(before[1], after[1])
    assert np.array_equal(auto[2], one[2])
    assert np.array_equal(auto[1][1], one[1][1])
    assert (auto[2][3] > 0).sum() > 500


def test_row_slabs(emu_lib):
    """Row bands of a plan equal its whole state 1; row slabs (spatial_search's plans: halo, shared
    curvature statistics) give planes 4..7 equal to the restatement of their own sweep."""
    from scarplet_b200 import distributed as D, params as P
    ny, nx = 70, 64
    z = _dem((ny, nx), 19)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-0.4, 0.4)
    spec = _template("Scarp")._sb_spec
    m = P.separation_positions(np.radians(8.0), angles)
    whole = _two_sweeps(z, spec, 8, ages, angles, m, rows=(11, 40))
    assert np.array_equal(whole[3], whole[2][:, 11:40])
    halo = D.slab_halo(spec, 8, ages, angles, nx, ny, 1.0)
    for lo, hi in ((0, 33), (33, ny)):
        before, after, second, band, _ = _two_sweeps(z, spec, 8, ages, angles, m, slab=(lo, hi, halo),
                                                     curv=whole[4], rows=(lo + 3, lo + 20))
        assert second.shape == (4, hi - lo, nx)
        assert before[0] == after[0]
        assert np.array_equal(band, second[:, 3:20])
        want = restated_planes(z, spec, 8, ages, angles, before[1], m, slab=(lo, hi, halo), curv=whole[4])
        assert np.array_equal(second, want)
        assert (second[3] > 0).sum() > 200


def test_refusals(emu_lib):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200._lib import SbError, check
    from scarplet_b200.engine import Plan
    from tests.plugin_templates import ShiftedRidge
    ny, nx = 40, 48
    z = _dem((ny, nx), 1)
    grid, Scarp = _grid(z), _template("Scarp")
    sep = np.radians(3.0)
    kw = dict(ages=[2.0, 3.0], ang_min=-0.1, ang_max=0.1)
    import scarplet_b200.core as C
    sl.secondary_fit(grid, Scarp, 8, sep, **kw)          # leaves this raster's plan in the cache

    def count():
        # a refusal must come before any device work: the cached plan launches nothing
        return [p.launches for _, p in C._cache]
    launches = count()
    assert launches
    with pytest.raises(ValueError, match="built-in"):
        sl.secondary_fit(grid, ShiftedRidge, 8, sep, **kw)
    with pytest.raises(ValueError, match="keyword"):
        sl.secondary_fit(grid, Scarp, 8, sep, shift=1, **kw)
    with pytest.raises(ValueError, match="duplicate"):
        sl.secondary_fit(grid, Scarp, 8, sep, ages=[2.0, 3.0, 2.0], ang_min=-0.1, ang_max=0.1)
    with pytest.raises(ValueError, match="at least one age"):
        sl.secondary_fit(grid, Scarp, 8, sep, ages=[], ang_min=-0.1, ang_max=0.1)
    with pytest.raises(ValueError, match="256 orientations"):
        sl.secondary_fit(grid, Scarp, 8, sep, ages=[2.0], ang_min=-np.pi, ang_max=np.pi / 2)
    with pytest.raises(ValueError, match="2 orientations"):
        sl.secondary_fit(grid, Scarp, 8, sep, ages=[2.0], ang_min=0.1, ang_max=0.1)
    for bad in (0.0, -0.05, np.nan, np.inf, np.radians(12.0)):        # 11 positions: at most 10 apart
        with pytest.raises(ValueError, match="min_separation"):
            sl.secondary_fit(grid, Scarp, 8, bad, **kw)
    with pytest.raises(ValueError, match="min_separation"):
        sl.secondary_fit(grid, Scarp, 8, np.radians(91.0), ages=[2.0])
    assert count() == launches
    # no limit on the number of ages
    many = np.linspace(1.0, 60.0, 70)
    got = sl.secondary_fit(grid, Scarp, 6, np.radians(2.0), ages=many, ang_min=-0.05, ang_max=0.05)
    assert np.array_equal(got[:4], np.stack(sl.match(grid, Scarp, scale=6, ages=many, ang_min=-0.05, ang_max=0.05)))
    assert (got[7] > 0).sum() > 50

    spec = Scarp._sb_spec
    ages, angles = [2.0, 3.0], P.search_angles(-0.1, 0.1)
    tables = P.region_tables(ages, angles)
    n_pos = len(tables.pos_angle)
    with Plan(ny, nx, 1.0, 1.0, states=2, slab=(10, 30, 20)) as plan:
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(spec, 8, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        plan.secondary_sweep(a, t, tables, 2)
        assert plan.finalize(age_of, angle_of, state=1).shape == (4, 20, nx)
        pos = np.ascontiguousarray(tables.angle_pos)

        def sweep(m=2, pos=pos, n_pos=n_pos, periodic=0, recs=t):
            check(plan.lib, plan.lib.sb_secondary_sweep(plan._h, a[0], a[1], recs[0], recs[1], None,
                                                        pos.ctypes.data, len(pos), n_pos, periodic, m))
        for bad in (0, -1, n_pos):
            with pytest.raises(SbError, match="min_sep_pos"):
                sweep(m=bad)
        with pytest.raises(SbError, match="min_sep_pos"):
            sweep(m=n_pos // 2 + 1, periodic=1)
        sweep(m=n_pos - 1)
        for bad in (0, 257):
            with pytest.raises(SbError, match="n_pos"):
                sweep(n_pos=bad)
        with pytest.raises(SbError, match="out of range"):
            sweep(pos=np.where(pos == 0, n_pos, pos).astype(np.int32))
        with pytest.raises(SbError, match="out of range"):
            sweep(pos=np.full_like(pos, -1))
        with pytest.raises(SbError, match="flat index"):
            sweep(pos=pos[:-1].copy())
        # records of another best state
        a2, t2, _, _ = plan.build_sweep(spec, 8, ages, angles, state_per_age=True)
        with pytest.raises(SbError, match="state"):
            plan.secondary_sweep(a2, t2, tables, 2)
    with Plan(ny, nx, 1.0, 1.0) as plan:
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(spec, 8, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        with pytest.raises(SbError, match="2 best states"):
            plan.secondary_sweep(a, t, tables, 2)
    for option, value in (("precision", 64), ("fast", 0)):
        with Plan(ny, nx, 1.0, 1.0, states=2) as plan:
            plan.set_option(option, value)
            plan.set_dem(z)
            a, t, age_of, angle_of = plan.build_sweep(spec, 8, ages, angles)
            plan.reset()
            plan.sweep(a, t)
            with pytest.raises(SbError, match="precision 32 and the option fast"):
                plan.secondary_sweep(a, t, tables, 2)
    assert np.array_equal(z, _dem((ny, nx), 1))
    sl.release()


# ---------------------------------------------------------------------------
# on the B200
# ---------------------------------------------------------------------------
C3_AGES = np.logspace(0, 3.5, 30)


@pytest.mark.gpu
def test_gpu_c3_secondary(cuda_lib):
    """C3 (4096^2 seed 2, Scarp 100, 30 ages x 181 orientations), 10 degrees: planes 0..3 are match."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(4096, seed=2)
    grid, Scarp = _grid(z), _template("Scarp")
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    got = sl.secondary_fit(grid, Scarp, 100.0, np.radians(10.0), ages=C3_AGES)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=C3_AGES))
    eq_match = bool(np.array_equal(got[:4], ref, equal_nan=True))
    del ref
    fit, second = got[3] > 0, got[7] > 0
    d = position_distance(positions_of(got[6][second], angles), positions_of(got[2][second], angles), 180, True)
    save_report("c3_secondary", {"planes_0_3_array_equal_match": eq_match, "valid": int(fit.sum()),
                                 "secondary": int(second.sum()), "min_position_distance": int(d.min()),
                                 "snr2_over_snr_p50": float(np.median(got[7][second] / got[3][second]))},
                {"config": "C3 4096^2 seed 2, Scarp 100, 30 ages x 181 orientations, min_separation 10 deg"})
    assert eq_match
    assert (d >= 10).all() and not (second & ~fit).any()
    sl.release()


@pytest.mark.gpu
@pytest.mark.parametrize("deg", [10.0, 45.0])
def test_gpu_1024_restated(cuda_lib, deg):
    """1024^2, 6 ages x 181 orientations: planes 4..7 equal the restatement, whose per-template SNR and
    amplitude planes are read and folded on the device (181 one-orientation shares)."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(1024, seed=6)
    grid, Scarp = _grid(z), _template("Scarp")
    ages = C3_AGES[::5]
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    sep = np.radians(deg)
    got = sl.secondary_fit(grid, Scarp, 100.0, sep, ages=ages)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=ages))
    sl.release()
    want = restated_planes(z, Scarp._sb_spec, 100.0, ages, angles, ref, P.separation_positions(sep, angles),
                           device="cuda:0")
    eq = [bool(np.array_equal(got[4 + k], want[k])) for k in range(4)]
    second = got[7] > 0
    save_report("restated_1024_%ddeg" % deg, {"planes_0_3_array_equal_match": bool(np.array_equal(got[:4], ref)),
                                              "planes_4_7_array_equal_restated": eq, "valid": int((ref[3] > 0).sum()),
                                              "secondary": int(second.sum())},
                {"config": "1024^2 seed 6, Scarp 100, 6 ages (C3's every fifth) x 181 orientations, "
                           "min_separation %g deg" % deg})
    assert np.array_equal(got[:4], ref)
    assert all(eq), eq
    assert second.sum() > 1000


@pytest.mark.gpu
def test_gpu_1024_masked(cuda_lib):
    """A masked 1024^2 raster with ~10 % nodata at min_coverage 0.7: planes 0..3 are masked match,
    planes 4..7 the restatement."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    z = _gpu_holes(synthetic_dem(1024, seed=6), seed=6)
    assert 0.09 < np.mean(~np.isfinite(z)) < 0.12
    grid, Scarp = _grid(z), _template("Scarp")
    masked = dict(nodata="mask", min_coverage=0.7)
    ages = C3_AGES[::5]
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    sep = np.radians(10.0)
    got = sl.secondary_fit(grid, Scarp, 100.0, sep, ages=ages, **masked)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=ages, **masked))
    sl.release()
    want = restated_planes(z, Scarp._sb_spec, 100.0, ages, angles, ref, P.separation_positions(sep, angles),
                           device="cuda:0", **masked)
    eq_match = bool(np.array_equal(got[:4], ref, equal_nan=True))
    eq = [bool(np.array_equal(got[4 + k], want[k])) for k in range(4)]
    save_report("masked_1024_secondary", {"planes_0_3_array_equal_match": eq_match,
                                          "planes_4_7_array_equal_restated": eq, "valid": int((ref[3] > 0).sum()),
                                          "secondary": int((got[7] > 0).sum()),
                                          "nodata_share": float(np.mean(~np.isfinite(z)))},
                {"config": "1024^2 seed 6, ~10 % nodata (border + cells), Scarp 100, 6 ages (C3's every fifth) x "
                           "181, min_coverage 0.7, min_separation 10 deg"})
    assert eq_match and all(eq), eq
    assert (got[:, ~np.isfinite(z)] == 0).all()
