"""Fit confidence regions (``sb_region_sweep`` / ``sb_region_finalize``, ``core.fit_region``, DESIGN.md
section 14): the (age, orientation) templates whose SNR is within ``snr_ratio`` of each pixel's best,
from a threshold pass over the same sweep.

Planes 0..3 must equal ``match`` and planes 4, 5 ``age_range`` bit for bit.  Planes 4..8 are checked
exactly against a NumPy / torch restatement of the contract, built from every template's float32 SNR
plane: one-orientation shares of the same search (``build_sweep(angle_slice=(i, i + 1),
state_per_age=True)``, which pass the whole search's extents to ``sb_sweep_ex``) leave in state g the
SNR of template (age g, orientation i) wherever it is a candidate, bit for bit.  The CPU cases run the
emulator build of the kernels (tests/emu), the ``gpu`` cases the B200."""
import numpy as np
import pytest

from tests.parity import save_report, stack_report
from tests.test_nodata_mask import _gpu_holes, _holes


def _template(name):
    from scarplet_b200 import templates as T
    return getattr(T, name)


def _grid(z):
    import scarplet_b200 as sl
    return sl.DEMGrid(z, 1.0)


# ---------------------------------------------------------------------------
# the contract, restated
# ---------------------------------------------------------------------------
def restated_arc(orient, pos_angle, periodic, chunk=1 << 16):
    """Planes 6, 7 from ``orient`` [n_pos, ...] (position p holds a qualifying orientation): the
    shortest arc holding every qualifying position; periodic: the complement of the largest circular
    gap between consecutive qualifying positions (equal gaps: the lowest p_lo), ``angle_hi + pi`` when
    the arc wraps.  0 where no position qualifies."""
    n = orient.shape[0]
    flat = orient.reshape(n, -1)
    lo = np.zeros(flat.shape[1])
    hi = np.zeros(flat.shape[1])
    pos = np.arange(n)[:, None]
    for c0 in range(0, flat.shape[1], chunk):
        q = flat[:, c0:c0 + chunk]
        cols = np.arange(q.shape[1])
        if not periodic:
            p_lo = np.argmax(q, axis=0)
            p_hi = n - 1 - np.argmax(q[::-1], axis=0)
        else:
            upto = np.maximum.accumulate(np.where(q, pos, -1), axis=0)        # last qualifying <= p
            prev = np.vstack([np.full((1, q.shape[1]), -1), upto[:-1]])      # last qualifying < p
            prev = np.where(prev < 0, upto[-1] - n, prev)                    # the first one: gap across the wrap
            p_lo = np.argmax(np.where(q, pos - prev, -1), axis=0)            # first maximum: the lowest p_lo
            p_hi = prev[p_lo, cols] % n
        a_lo = pos_angle[p_lo]
        a_hi = np.where(p_hi < p_lo, pos_angle[p_hi] + np.pi, pos_angle[p_hi])
        some = q.any(axis=0)
        lo[c0:c0 + chunk] = np.where(some, a_lo, 0.0)
        hi[c0:c0 + chunk] = np.where(some, a_hi, 0.0)
    return lo.reshape(orient.shape[1:]), hi.reshape(orient.shape[1:])


class Restated(object):
    """Planes 4..8 of the contract, accumulated one orientation at a time from the per-template
    float32 SNR planes ([ages, rows, nx] torch tensors, on the device for the gpu cases) and the
    pixel's best SNR (plane 3 of ``match``)."""

    def __init__(self, best, ages, angles, ratio, device=None):
        import torch
        from scarplet_b200 import params as P
        self.torch, self.device = torch, device
        self.tables = P.region_tables(ages, angles)
        self.ages = [float(a) for a in ages]
        best = torch.as_tensor(np.asarray(best, dtype=np.float64), device=device)
        self.fit = best > 0
        self.floor = ratio * best
        self.count = torch.zeros(best.shape, dtype=torch.int64, device=device)
        self.lo = torch.full(best.shape, np.inf, dtype=torch.float64, device=device)
        self.hi = torch.full(best.shape, -np.inf, dtype=torch.float64, device=device)
        self.orient = torch.zeros((len(self.tables.pos_angle),) + tuple(best.shape), dtype=torch.bool, device=device)

    def add(self, i, snr):
        torch = self.torch
        s = snr.double()
        q = (s > 0) & (s >= self.floor[None]) & self.fit[None]
        self.count += q.sum(0)
        for g, a in enumerate(self.ages):
            self.lo = torch.where(q[g], torch.clamp(self.lo, max=a), self.lo)
            self.hi = torch.where(q[g], torch.clamp(self.hi, min=a), self.hi)
        p = i % len(self.tables.pos_angle)
        self.orient[p] |= q.any(0)

    def planes(self):
        fit = self.fit.cpu().numpy()
        some = (self.count > 0).cpu().numpy() & fit
        lo = np.where(some, self.lo.cpu().numpy(), 0.0)
        hi = np.where(some, self.hi.cpu().numpy(), 0.0)
        a_lo, a_hi = restated_arc(self.orient.cpu().numpy() & fit[None], self.tables.pos_angle, self.tables.periodic)
        return np.stack([lo, hi, a_lo, a_hi, np.where(fit, self.count.cpu().numpy(), 0).astype(np.float64)])


def template_snr_shares(z, spec, scale, ages, angles, device=None, curv=None, **plan_kw):
    """Yields ``(i, snr)``: the float32 SNR planes [ages, rows, nx] of the templates of orientation i,
    from one-orientation shares of the search on a plan with one best state per age (read in place
    through the plan's device pointers; valid until the next yield).  ``curv``: the curvature
    statistics of a row slab's whole raster."""
    from scarplet_b200.distributed import _as_tensor
    from scarplet_b200.engine import Plan
    ny, nx = z.shape
    G = len(ages)
    cuda = device is not None
    with Plan(ny, nx, 1.0, 1.0, states=G, **plan_kw) as plan:
        plan.set_dem(z)
        if curv is not None:
            plan.set_curv_stats(*curv)
        rows = plan.row_hi - plan.row_lo
        for i in range(len(angles)):
            a, t, _, _ = plan.build_sweep(spec, scale, ages, angles, angle_slice=(i, i + 1), state_per_age=True)
            assert t[2] is not None             # the whole search's extents go with the share
            plan.reset()
            plan.sweep(a, t)
            plan.sync()
            ps, _, _ = plan.best_state_pointers(0)
            yield i, _as_tensor(ps, G * rows * nx, "f4", device).reshape(G, rows, nx)
            if cuda:
                import torch
                torch.cuda.synchronize(device)


def restated_planes(z, spec, scale, ages, angles, best, ratio, device=None, **plan_kw):
    """Planes 4..8 of ``fit_region`` as the contract states them, for the pixel's best SNR ``best``."""
    r = Restated(best, ages, angles, ratio, device)
    for i, snr in template_snr_shares(z, spec, scale, ages, angles, device, **plan_kw):
        r.add(i, snr)
    return r.planes()


# ---------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------
def test_restated_arc_examples():
    """The orientation arc of the contract at 1-degree steps over -90 .. 90 degrees (periodic: -90
    and 90 are one line, position 0), and a linear search."""
    from scarplet_b200 import params as P
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    t = P.region_tables([1.0], angles)
    assert t.periodic and len(t.pos_angle) == 180 and t.angle_pos[180] == 0
    deg = np.round(np.degrees(angles)).astype(int)

    def arc(members):
        q = np.zeros(180, dtype=bool)
        for d in members:
            q[t.angle_pos[int(np.flatnonzero(deg == d)[0])]] = True
        lo, hi = restated_arc(q[:, None], t.pos_angle, True)
        return lo[0], hi[0]

    a = dict(zip(deg.tolist(), angles.tolist()))
    assert arc([-89, 89, 90]) == (a[89], a[-89] + np.pi)              # [89, 91] degrees
    assert arc([-89, 89, -90]) == (a[89], a[-89] + np.pi)
    assert arc([88, 89, 90]) == (a[88], a[-90] + np.pi)               # [88, 90]
    assert arc([-90, -89]) == (a[-90], a[-89])
    assert arc([0, 90]) == (a[-90], a[0])                              # equal gaps: the lowest p_lo
    assert arc([17]) == (a[17], a[17])
    for (lo, hi), want in zip([arc([-89, 89, 90]), arc([88, 89, 90]), arc([-90, -89]), arc([0, 90])],
                              [(89, 91), (88, 90), (-90, -89), (-90, 0)]):
        assert np.allclose(np.degrees([lo, hi]), want, atol=1e-9)
    lin = P.search_angles(-0.5, 0.5)
    tl = P.region_tables([1.0, 2.0], lin)
    assert not tl.periodic and len(tl.pos_angle) == len(lin)
    q = np.zeros(len(lin), dtype=bool)
    q[[3, 20, 40]] = True
    assert restated_arc(q[:, None], tl.pos_angle, False) == (lin[3], lin[40])
    assert restated_arc(np.zeros((len(lin), 1), dtype=bool), tl.pos_angle, False) == (0.0, 0.0)


def _dem(shape, seed):
    from scarplet_b200.synth import synthetic_dem
    return synthetic_dem(shape[0], seed=seed, nx=shape[1])


def _cases():
    nan = _dem((64, 72), 21)
    nan[30, 41] = np.nan
    return {
        # name: (template, dem, scale, ages, (ang_min, ang_max), ratio, nodata kwargs)
        "scarp_odd": ("Scarp", _dem((73, 90), 4), 9, [2.0, 6.0, 20.0], (-0.4, 0.4), 0.8, {}),
        "channel_wrap": ("Channel", _dem((64, 70), 5), 5, [0.15, 0.2, 0.3], (-0.3, 0.3), 0.8, {}),   # no edge mask
        "upper_break": ("RightFacingUpperBreakScarp", _dem((64, 80), 6), 9, [2.0, 6.0, 20.0], (-0.4, 0.4), 0.8,
                        {}),                                                                         # get_err_mask
        "mask_holes": ("Scarp", _holes(_dem((72, 80), 2), "border+cells", seed=2), 9, [1.5, 4.0, 12.0], (-0.4, 0.4),
                       0.7, dict(nodata="mask", min_coverage=0.6)),
        "propagate_nan": ("Scarp", nan, 9, [2.0, 6.0], (-0.3, 0.3), 0.8, {}),
        "periodic": ("Scarp", _dem((40, 44), 8), 6, [2.0, 8.0], (-np.pi / 2, np.pi / 2), 0.6, {}),
    }


@pytest.mark.parametrize("case", ["scarp_odd", "channel_wrap", "upper_break", "mask_holes", "propagate_nan",
                                  "periodic"])
def test_region_restated(emu_lib, case):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    tmpl, z, scale, ages, span, ratio, masking = _cases()[case]
    Template = _template(tmpl)
    kw = dict(ang_min=span[0], ang_max=span[1], **masking)
    got = sl.fit_region(_grid(z), Template, scale, ratio, ages=ages, **kw)
    ref = np.stack(sl.match(_grid(z), Template, scale=scale, ages=ages, **kw))
    assert got.shape == (9,) + z.shape and got.dtype == np.float64
    assert np.array_equal(got[:4], ref, equal_nan=True)
    angles = P.search_angles(*span)
    want = restated_planes(z, Template._sb_spec, scale, ages, angles, ref[3], ratio, **masking)
    assert np.array_equal(got[4:], want)
    fit = ref[3] > 0
    if case == "propagate_nan":
        assert np.isnan(ref[3]).any() and (got[4:][:, ~fit] == 0).all()
    else:
        assert fit.sum() > 500 and (got[8][fit] >= 1).all() and (got[4:][:, ~fit] == 0).all()
        assert (got[4][fit] <= got[1][fit]).all() and (got[1][fit] <= got[5][fit]).all()
        assert (got[6][fit] <= got[7][fit]).all() and (got[7][fit] - got[6][fit] < np.pi).all()
        assert (got[7][fit] > got[6][fit]).sum() > 50                   # arcs, not only single orientations
    if case == "periodic":
        assert (got[7][fit] > np.pi / 2).sum() > 0                      # arcs across +-90 degrees
    if case == "mask_holes":
        assert (got[:, ~np.isfinite(z)] == 0).all()
    sl.release()


@pytest.mark.parametrize("ratio", [0.5, 0.9, 1.0])
def test_age_planes_equal_age_range(emu_lib, ratio):
    import scarplet_b200 as sl
    z = _dem((80, 96), 17)
    grid, Scarp = _grid(z), _template("Scarp")
    ages, kw = [1.0, 2.5, 6.0, 15.0, 40.0], dict(ang_min=-0.5, ang_max=0.5)
    got = sl.fit_region(grid, Scarp, 9, ratio, ages=ages, **kw)
    rng = sl.age_range(grid, Scarp, 9, ratio, ages=ages, **kw)
    assert np.array_equal(got[:4], rng[:4]) and np.array_equal(got[4:6], rng[4:6])
    fit = got[3] > 0
    assert np.array_equal(got[8] >= 1, fit)
    if ratio == 1.0:
        # only the best template and exact float32 ties qualify
        assert (got[8][fit] == 1).mean() > 0.99 and (got[6][fit] == got[2][fit]).mean() > 0.99
    sl.release()


def test_ages_beyond_64(emu_lib):
    """No limit on the number of ages (age_range stops at 64: one best state per age)."""
    import scarplet_b200 as sl
    z = _dem((40, 48), 3)
    ages = np.linspace(1.0, 60.0, 70)
    got = sl.fit_region(_grid(z), _template("Scarp"), 6, 0.9, ages=ages, ang_min=-0.1, ang_max=0.1)
    ref = np.stack(sl.match(_grid(z), _template("Scarp"), scale=6, ages=ages, ang_min=-0.1, ang_max=0.1))
    assert np.array_equal(got[:4], ref)
    fit = ref[3] > 0
    assert fit.sum() > 100 and (got[8][fit] >= 1).all() and (got[8] <= 70 * 12).all()
    assert np.isin(got[4][fit], ages).all() and np.isin(got[5][fit], ages).all()
    assert (got[5][fit] > got[4][fit]).sum() > 10
    sl.release()


def _two_pass(z, spec, scale, ages, angles, ratio, substreams=None, slab=None, curv=None, rows=None):
    """On one plan: finalize after match's sweep, the region planes, finalize after the region pass,
    and the region planes of the rows ``rows``."""
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    ny, nx = z.shape
    tables = P.region_tables(ages, angles)
    with Plan(ny, nx, 1.0, 1.0, slab=slab) as plan:
        if substreams is not None:
            plan.set_option("fit_substreams", substreams)
        plan.set_dem(z)
        if curv is not None:
            plan.set_curv_stats(*curv)
        a, t, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        before = plan.finalize(age_of, angle_of).copy()
        plan.region_sweep(a, t, ratio, tables)
        after = plan.finalize(age_of, angle_of).copy()
        got = plan.region_finalize(age_of, angle_of, tables)
        band = None if rows is None else plan.region_finalize(age_of, angle_of, tables, rows=rows)
        return before, after, got, band, plan.curv_stats(), plan.device_bytes


def test_substreams_and_best_state_untouched(emu_lib):
    """A raster this small deals the fit kernel's templates to sub-streams: the region planes are the
    same with one; the region pass leaves the best state as it was."""
    from scarplet_b200 import params as P
    z = _dem((64, 72), 13)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-np.pi / 2, np.pi / 2)[::6]
    spec = _template("Scarp")._sb_spec
    auto = _two_pass(z, spec, 7, ages, angles, 0.7)
    one = _two_pass(z, spec, 7, ages, angles, 0.7, substreams=1)
    for before, after, got, _, _, _ in (auto, one):
        assert np.array_equal(before, after)
        assert np.array_equal(got[:4], before)
    assert np.array_equal(auto[2], one[2])
    assert (auto[2][8] >= 2).sum() > 100
    # region planes: 4 * (3 + ceil(n_pos / 32)) B per pixel
    from scarplet_b200.engine import Plan
    with Plan(*z.shape, 1.0, 1.0) as plan:
        plan.set_option("fit_substreams", 1)
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(spec, 7, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        b0 = plan.device_bytes
        plan.region_sweep(a, t, 0.7, P.region_tables(ages, angles))
        n_pos = len(P.region_tables(ages, angles).pos_angle)
        assert plan.device_bytes - b0 >= 4 * (3 + -(-n_pos // 32)) * z.size


def test_row_slabs(emu_lib):
    """Row bands of a plan equal its whole region planes; row slabs (spatial_search's plans: halo,
    shared curvature statistics) give planes 0..3 equal to their own match and planes 4..8 equal to
    the restatement of their own sweep, and agree with the whole raster wherever the whole raster's
    SNR planes do (the slabs' FFT domains differ, as for match)."""
    from scarplet_b200 import distributed as D, params as P
    ny, nx = 70, 64
    z = _dem((ny, nx), 19)
    ages, angles = [2.0, 5.0, 11.0], P.search_angles(-0.4, 0.4)
    spec = _template("Scarp")._sb_spec
    ratio = 0.8
    whole = _two_pass(z, spec, 8, ages, angles, ratio, rows=(11, 40))
    assert np.array_equal(whole[3], whole[2][:, 11:40])
    halo = D.slab_halo(spec, 8, ages, angles, nx, ny, 1.0)
    parts = []
    for lo, hi in ((0, 33), (33, ny)):
        before, after, got, band, _, _ = _two_pass(z, spec, 8, ages, angles, ratio, slab=(lo, hi, halo),
                                                   curv=whole[4], rows=(lo + 3, lo + 20))
        assert got.shape == (9, hi - lo, nx)
        assert np.array_equal(before, after) and np.array_equal(got[:4], before)
        assert np.array_equal(band, got[:, 3:20])
        want = restated_planes(z, spec, 8, ages, angles, got[3], ratio, slab=(lo, hi, halo), curv=whole[4])
        assert np.array_equal(got[4:], want)
        parts.append(got)
    got = np.concatenate(parts, axis=1)
    rep = stack_report(got[:4], whole[2][:4])
    assert rep["mask_equal"] and rep["index_agreement"] >= 0.999 and rep["snr_rel_max_strong"] < 2e-5, rep
    agree = (got[4:] == whole[2][4:]).all(axis=0)
    assert agree[whole[2][3] > 0].mean() >= 0.99


def test_refusals(emu_lib):
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200._lib import SbError, check
    from scarplet_b200.engine import Plan
    from tests.plugin_templates import ShiftedRidge
    ny, nx = 40, 48
    z = _dem((ny, nx), 1)
    grid, Scarp = _grid(z), _template("Scarp")
    kw = dict(ages=[2.0, 3.0], ang_min=-0.1, ang_max=0.1)
    with pytest.raises(ValueError, match="built-in"):
        sl.fit_region(grid, ShiftedRidge, 8, 0.5, **kw)
    with pytest.raises(ValueError, match="keyword"):
        sl.fit_region(grid, Scarp, 8, 0.5, shift=1, **kw)
    with pytest.raises(ValueError, match="duplicate"):
        sl.fit_region(grid, Scarp, 8, 0.5, ages=[2.0, 3.0, 2.0], ang_min=-0.1, ang_max=0.1)
    with pytest.raises(ValueError, match="at least one age"):
        sl.fit_region(grid, Scarp, 8, 0.5, ages=[], ang_min=-0.1, ang_max=0.1)
    for ratio in (0.0, -0.5, 1.0 + 1e-12, 1.5, np.nan, np.inf):
        with pytest.raises(ValueError, match="snr_ratio"):
            sl.fit_region(grid, Scarp, 8, ratio, **kw)
    with pytest.raises(ValueError, match="256 orientations"):
        sl.fit_region(grid, Scarp, 8, 0.5, ages=[2.0], ang_min=-np.pi, ang_max=np.pi / 2)
    assert len(P.search_angles(-np.pi, np.pi / 2)) > 256

    spec = Scarp._sb_spec
    ages, angles = [2.0, 3.0], P.search_angles(-0.1, 0.1)
    tables = P.region_tables(ages, angles)
    with Plan(ny, nx, 1.0, 1.0, slab=(10, 30, 20)) as plan:
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(spec, 8, ages, angles)
        plan.reset()
        plan.sweep(a, t)
        with pytest.raises(SbError, match="no region sweep"):
            plan.region_finalize(age_of, angle_of, tables)
        plan.region_sweep(a, t, 0.5, tables)
        assert plan.region_finalize(age_of, angle_of, tables).shape == (9, 20, nx)
        rank = np.ascontiguousarray(tables.age_rank)
        pos = np.ascontiguousarray(tables.angle_pos)
        n_pos = len(tables.pos_angle)

        def sweep(ratio=0.5, rank=rank, pos=pos, n_pos=n_pos, recs=t):
            check(plan.lib, plan.lib.sb_region_sweep(plan._h, a[0], a[1], recs[0], recs[1], None, ratio,
                                                     rank.ctypes.data, pos.ctypes.data, len(rank), n_pos))
        for bad in (0.0, 1.5, float("nan")):
            with pytest.raises(SbError, match="snr_ratio"):
                sweep(ratio=bad)
        for bad in (0, 257):
            with pytest.raises(SbError, match="n_pos"):
                sweep(n_pos=bad)
        with pytest.raises(SbError, match="out of range"):
            sweep(pos=np.where(pos == 0, n_pos, pos).astype(np.int32))
        with pytest.raises(SbError, match="out of range"):
            sweep(rank=np.full_like(rank, -1))
        with pytest.raises(SbError, match="flat index"):
            sweep(rank=rank[:-1].copy(), pos=pos[:-1].copy())
        out = np.empty(9 * 20 * nx)
        pos_angle = np.ascontiguousarray(tables.pos_angle)

        def fin(lo=10, hi=30, n_pos=n_pos, n_ranks=len(ages)):
            check(plan.lib, plan.lib.sb_region_finalize(plan._h, lo, hi, age_of.ctypes.data, angle_of.ctypes.data,
                                                        len(age_of), tables.rank_age.ctypes.data, n_ranks,
                                                        pos_angle.ctypes.data, n_pos, 0, out.ctypes.data, 0))
        fin()
        for bad in (dict(lo=9), dict(hi=31), dict(lo=20, hi=20)):
            with pytest.raises(SbError, match="rows outside"):
                fin(**bad)
        with pytest.raises(SbError, match="n_pos"):
            fin(n_pos=n_pos - 1)
        with pytest.raises(SbError, match="ranks"):
            fin(n_ranks=1)
        # records of another best state
        plan.set_states(2)
        a2, t2, _, _ = plan.build_sweep(spec, 8, ages, angles, state_per_age=True)
        with pytest.raises(SbError, match="state"):
            plan.region_sweep(a2, t2, 0.5, tables)
        with pytest.raises(SbError, match="no region sweep"):
            plan.region_finalize(age_of, angle_of, tables)
    for option, value in (("precision", 64), ("fast", 0)):
        with Plan(ny, nx, 1.0, 1.0) as plan:
            plan.set_option(option, value)
            plan.set_dem(z)
            a, t, age_of, angle_of = plan.build_sweep(spec, 8, ages, angles)
            plan.reset()
            plan.sweep(a, t)
            with pytest.raises(SbError, match="precision 32 and the option fast"):
                plan.region_sweep(a, t, 0.5, tables)
    assert np.array_equal(z, _dem((ny, nx), 1))
    sl.release()


# ---------------------------------------------------------------------------
# on the B200
# ---------------------------------------------------------------------------
C3_AGES = np.logspace(0, 3.5, 30)


@pytest.mark.gpu
def test_gpu_c3_region(cuda_lib):
    """C3 (4096^2 seed 2, Scarp 100, 30 ages x 181 orientations), ratio 0.9: planes 0..3 are match,
    planes 4, 5 age_range."""
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(4096, seed=2)
    grid, Scarp = _grid(z), _template("Scarp")
    got = sl.fit_region(grid, Scarp, 100.0, 0.9, ages=C3_AGES)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=C3_AGES))
    eq_match = bool(np.array_equal(got[:4], ref, equal_nan=True))
    del ref
    rng = sl.age_range(grid, Scarp, 100.0, 0.9, ages=C3_AGES)
    eq_range = bool(np.array_equal(got[4:6], rng[4:6]))
    fit = got[3] > 0
    save_report("c3_region", {"planes_0_3_array_equal_match": eq_match, "planes_4_5_array_equal_age_range": eq_range,
                              "valid": int(fit.sum()), "n_fits_ge1_where_fit": bool((got[8][fit] >= 1).all()),
                              "n_fits_p50": float(np.median(got[8][fit])),
                              "arc_width_deg_p50": float(np.degrees(np.median(got[7][fit] - got[6][fit])))},
                {"config": "C3 4096^2 seed 2, Scarp 100, 30 ages x 181 orientations, snr_ratio 0.9"})
    assert eq_match and eq_range
    assert np.array_equal(got[8] >= 1, fit)
    sl.release()


@pytest.mark.gpu
def test_gpu_1024_restated(cuda_lib):
    """1024^2, 6 ages x 181 orientations: planes 4..8 equal the restatement, whose per-template SNR
    planes are read and reduced on the device (181 one-orientation shares)."""
    import scarplet_b200 as sl
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(1024, seed=6)
    grid, Scarp = _grid(z), _template("Scarp")
    ages = C3_AGES[::5]
    angles = P.search_angles(-np.pi / 2, np.pi / 2)
    ratio = 0.9
    got = sl.fit_region(grid, Scarp, 100.0, ratio, ages=ages)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=ages))
    sl.release()
    want = restated_planes(z, Scarp._sb_spec, 100.0, ages, angles, ref[3], ratio, device="cuda:0")
    fit = ref[3] > 0
    eq = [bool(np.array_equal(got[4 + k], want[k])) for k in range(5)]
    save_report("restated_1024", {"planes_0_3_array_equal_match": bool(np.array_equal(got[:4], ref)),
                                  "planes_4_8_array_equal_restated": eq, "valid": int(fit.sum()),
                                  "wrapping_arcs": int((got[7][fit] > np.pi / 2).sum()),
                                  "n_fits_max": float(got[8].max())},
                {"config": "1024^2 seed 6, Scarp 100, 6 ages (C3's every fifth) x 181 orientations, snr_ratio 0.9"})
    assert np.array_equal(got[:4], ref)
    assert all(eq), eq


@pytest.mark.gpu
def test_gpu_1024_masked(cuda_lib):
    """A masked 1024^2 raster with ~10 % nodata at min_coverage 0.7: planes 0..3 are masked match,
    planes 4, 5 masked age_range."""
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    z = _gpu_holes(synthetic_dem(1024, seed=6), seed=6)
    assert 0.09 < np.mean(~np.isfinite(z)) < 0.12
    grid, Scarp = _grid(z), _template("Scarp")
    masked = dict(nodata="mask", min_coverage=0.7)
    got = sl.fit_region(grid, Scarp, 100.0, 0.9, ages=C3_AGES, **masked)
    ref = np.stack(sl.match(grid, Scarp, scale=100.0, ages=C3_AGES, **masked))
    rng = sl.age_range(grid, Scarp, 100.0, 0.9, ages=C3_AGES, **masked)
    fit = ref[3] > 0
    eq_match = bool(np.array_equal(got[:4], ref, equal_nan=True))
    eq_range = bool(np.array_equal(got[4:6], rng[4:6]))
    save_report("masked_1024_region", {"planes_0_3_array_equal_match": eq_match,
                                       "planes_4_5_array_equal_age_range": eq_range, "valid": int(fit.sum()),
                                       "nodata_share": float(np.mean(~np.isfinite(z)))},
                {"config": "1024^2 seed 6, ~10 % nodata (border + cells), Scarp 100, 30 ages x 181, "
                           "min_coverage 0.7, snr_ratio 0.9"})
    assert eq_match and eq_range
    assert np.array_equal(got[8] >= 1, fit) and (got[:, ~np.isfinite(z)] == 0).all()
    sl.release()
