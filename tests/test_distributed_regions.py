"""Age ranges and fit confidence regions over several ranks (``distributed.sharded_fit_region`` /
``sharded_age_range``: orientation shares, ``spatial_fit_region`` / ``spatial_age_range``: row bands;
DESIGN.md section 15) and the region-plane fold behind the orientation shares (``sb_region_merge``).

The sharded products must equal ``core.fit_region`` / ``core.age_range`` bit for bit: shares are
bit-identical to the whole search, the replicated best merge gives every rank the same thresholds and
the fold (sum, min, max, OR) is exact.  Row bands must equal one-process slab plans bit for bit and
the whole raster as ``spatial_search`` does.  The CPU cases run two gloo ranks on the emulator build
of the kernels (tests/emu); the ``gpu`` cases two NCCL ranks and the kernel on the B200."""
import os
import sys

import numpy as np
import pytest

from tests.parity import stack_report

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SHAPE = (96, 128)
SCALE, AGES, RATIO = 8, [2.0, 9.0, 30.0], 0.8
MASKED = dict(nodata="mask", min_coverage=0.6)


def _inputs():
    from scarplet_b200 import params as P
    from scarplet_b200.synth import synthetic_dem
    from tests.test_nodata_mask import _holes
    z = synthetic_dem(SHAPE[0], seed=7, nx=SHAPE[1], relief=3.0)
    return z, _holes(z, "border+cells", seed=3), P.search_angles(-np.pi / 2, np.pi / 2)[::9]


def _scarp():
    from scarplet_b200.templates import Scarp
    return Scarp


# ---------------------------------------------------------------------------
# two gloo ranks on the emulator
# ---------------------------------------------------------------------------
def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), SB_EMU_WORKERS="2")
    import torch
    import torch.distributed as dist
    from tests.emu.build_emu import build
    from scarplet_b200 import _lib
    _lib._use_library(_lib.open_library(build()))
    from scarplet_b200 import distributed as D
    from scarplet_b200.engine import Plan
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cpu = torch.device("cpu")
    spec = _scarp()._sb_spec
    z, zm, angles = _inputs()
    ny, nx = SHAPE

    def save(name, band):
        np.save(os.path.join(out_dir, "%s%d.npy" % (name, rank)), np.concatenate([[band[0], band[1]], band[2].ravel()]))

    def both(name, dem, ages, angles, **plan_kw):
        with Plan(ny, nx, 1.0, 1.0, **plan_kw) as plan:
            plan.set_dem(dem)
            save(name + "_region", D.sharded_fit_region(plan, spec, SCALE, ages, angles, RATIO, device=cpu))
            save(name + "_range", D.sharded_age_range(plan, spec, SCALE, ages, angles, RATIO, device=cpu))

    both("periodic", z, AGES, angles)                                   # 1. cost-balanced shares
    os.environ["SB_SHARE_BALANCE"] = "count"
    both("cut", z, AGES, angles)                                        # 2. a cut inside an orientation
    del os.environ["SB_SHARE_BALANCE"]
    both("empty", z, AGES[:1], angles[:1])                              # 3. rank 1 has no template
    both("masked", zm, AGES, angles, **MASKED)                          # 4. nodata mask
    plan, (lo, hi) = D.spatial_plan(ny, nx, 1.0, 1.0, spec, SCALE, AGES, angles, states=len(AGES))
    with plan:                                                          # 5. row bands
        plan.set_dem(z)
        D.share_dem_stats(plan, device=cpu)
        save("spatial_range", D.spatial_age_range(plan, spec, SCALE, AGES, angles, RATIO))
        save("spatial_region", D.spatial_fit_region(plan, spec, SCALE, AGES, angles, RATIO))
        assert plan.states == 1
    dist.destroy_process_group()


@pytest.fixture(scope="module")
def gloo_out(tmp_path_factory):
    import torch.multiprocessing as mp
    out = tmp_path_factory.mktemp("regions")
    port = 29500 + (os.getpid() + 977) % 2000
    mp.spawn(_worker, args=(2, port, str(out)), nprocs=2, join=True)
    return out


def _bands(out, name, planes, nx=SHAPE[1]):
    """[(row_lo, row_hi, stack)] of both ranks."""
    res = []
    for r in range(2):
        v = np.load(out / ("%s%d.npy" % (name, r)))
        lo, hi = int(v[0]), int(v[1])
        res.append((lo, hi, v[2:].reshape(planes, hi - lo, nx)))
    return res


def _joined(bands, ny=SHAPE[0]):
    assert bands[0][0] == 0 and bands[0][1] == bands[1][0] and bands[1][1] == ny
    return np.concatenate([b[2] for b in bands], axis=1)


def _core(dem, ages, span, **masking):
    import scarplet_b200 as sl
    grid, Scarp = sl.DEMGrid(dem, 1.0), _scarp()
    kw = dict(ages=ages, ang_min=span[0], ang_max=span[1], **masking)
    region = sl.fit_region(grid, Scarp, SCALE, RATIO, **kw)
    rng = sl.age_range(grid, Scarp, SCALE, RATIO, **kw)
    sl.release()
    return region, rng


def _core_on(dem, ages, angles, **masking):
    """``core.fit_region`` / ``core.age_range`` over exactly ``angles`` (a strided list is not a
    ``search_angles`` range): the single-plan path they run, on one plan."""
    from scarplet_b200 import distributed as D
    from scarplet_b200.engine import Plan
    spec = _scarp()._sb_spec
    with Plan(*dem.shape, 1.0, 1.0, **masking) as plan:
        plan.set_dem(dem)
        region = D.sharded_fit_region(plan, spec, SCALE, ages, angles, RATIO)[2]
        rng = D.sharded_age_range(plan, spec, SCALE, ages, angles, RATIO)[2]
    return region, rng


@pytest.mark.parametrize("case", ["periodic", "cut", "empty", "masked"])
def test_sharded_equal_single_plan(gloo_out, emu_lib, case):
    z, zm, angles = _inputs()
    dem, ages, masking = z, AGES, {}
    if case == "empty":
        ages, angles = AGES[:1], angles[:1]
    if case == "masked":
        dem, masking = zm, MASKED
    region, rng = _core_on(dem, ages, angles, **masking)
    got_region = _joined(_bands(gloo_out, case + "_region", 9))
    got_range = _joined(_bands(gloo_out, case + "_range", 6))
    assert np.array_equal(got_region, region, equal_nan=True)
    assert np.array_equal(got_range, rng, equal_nan=True)
    fit = region[3] > 0
    assert fit.sum() > 1000
    if case == "periodic":
        assert (region[7][fit] > np.pi / 2).sum() > 0                  # arcs across +-90 degrees
        assert (region[8][fit] >= 2).sum() > 500
    if case == "masked":
        assert (region[:, ~np.isfinite(zm)] == 0).all()


def test_share_cut_inside_an_orientation(emu_lib, monkeypatch):
    """The count-balanced shares of case ``cut`` split an orientation's ages over both ranks, so that
    its bits reach the fold from two candidates."""
    from scarplet_b200.engine import Plan
    z, _, angles = _inputs()
    monkeypatch.setenv("SB_SHARE_BALANCE", "count")
    with Plan(*SHAPE, 1.0, 1.0) as plan:
        cuts = Plan._share_cuts(plan, _scarp()._sb_spec, [SCALE], np.asarray(AGES), angles, 2)
    assert len(angles) * len(AGES) == 63 and cuts[1] == 32 and cuts[1] % len(AGES) != 0


@pytest.mark.parametrize("masked", [False, True])
def test_no_process_group_is_core(emu_lib, masked):
    """Without a process group every driver returns what ``core.fit_region`` / ``core.age_range``
    return, bit for bit (a row-band plan over the whole raster is an ordinary plan)."""
    from scarplet_b200 import distributed as D
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    z, zm, _ = _inputs()
    dem, masking = (zm, MASKED) if masked else (z, {})
    angles = P.search_angles(-0.4, 0.4)
    region, rng = _core(dem, AGES, (-0.4, 0.4), **masking)
    assert (region[3] > 0).sum() > 1000
    spec = _scarp()._sb_spec
    with Plan(*SHAPE, 1.0, 1.0, **masking) as plan:
        plan.set_dem(dem)
        for fn, want in ((D.sharded_fit_region, region), (D.sharded_age_range, rng), (D.spatial_fit_region, region),
                         (D.spatial_age_range, rng)):
            lo, hi, got = fn(plan, spec, SCALE, AGES, angles, RATIO)
            assert (lo, hi) == (0, SHAPE[0]) and np.array_equal(got, want, equal_nan=True), fn.__name__


def test_spatial_bands(gloo_out, emu_lib):
    """Row bands equal one-process slab plans with the shared curvature statistics bit for bit, and
    the whole raster as ``spatial_search`` does."""
    from scarplet_b200 import distributed as D
    from scarplet_b200.engine import Plan
    z, _, angles = _inputs()
    ny, nx = SHAPE
    spec = _scarp()._sb_spec
    region_b, range_b = _bands(gloo_out, "spatial_region", 9), _bands(gloo_out, "spatial_range", 6)
    halo = D.slab_halo(spec, SCALE, AGES, angles, nx, ny, 1.0)
    plans = [Plan(ny, nx, 1.0, 1.0, slab=(lo, hi, halo), states=len(AGES)) for lo, hi, _ in region_b]
    try:
        for p in plans:
            p.set_dem(z)
        stats = np.sum([p.curv_stats() for p in plans], axis=0)
        for p, rb, gb in zip(plans, region_b, range_b):
            p.set_curv_stats(*stats)
            assert np.array_equal(D.spatial_age_range(p, spec, SCALE, AGES, angles, RATIO)[2], gb[2])
            assert np.array_equal(D.spatial_fit_region(p, spec, SCALE, AGES, angles, RATIO)[2], rb[2])
    finally:
        for p in plans:
            p.close()
    whole_region, whole_range = _core_on(z, AGES, angles)
    for got, whole, extra in ((_joined(region_b), whole_region, 5), (_joined(range_b), whole_range, 2)):
        rep = stack_report(got[:4], whole[:4])
        assert rep["mask_equal"] and rep["index_agreement"] >= 0.999 and rep["snr_rel_max_strong"] < 2e-5, rep
        fit = whole[3] > 0
        assert (got[4:] == whole[4:]).all(axis=0)[fit].mean() >= 0.99 and got.shape[0] == 4 + extra


def test_refusals_before_device_work(emu_lib):
    """Every driver refuses what ``core`` refuses, with its ``ValueError``, before any launch."""
    from scarplet_b200 import distributed as D
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    z, _, angles = _inputs()
    spec = _scarp()._sb_spec
    wide = P.search_angles(-np.pi, np.pi / 2)
    assert len(wide) > 256
    with Plan(*SHAPE, 1.0, 1.0) as plan:
        plan.set_dem(z)
        n0 = plan.launches
        for fn in (D.sharded_fit_region, D.sharded_age_range, D.spatial_fit_region, D.spatial_age_range):
            for ratio in (0.0, -0.5, 1.0 + 1e-12, 1.5, np.nan, np.inf):
                with pytest.raises(ValueError, match="snr_ratio"):
                    fn(plan, spec, SCALE, AGES, angles, ratio)
            with pytest.raises(ValueError, match="duplicate"):
                fn(plan, spec, SCALE, [2.0, 9.0, 2.0], angles, RATIO)
        for fn in (D.sharded_age_range, D.spatial_age_range):
            with pytest.raises(ValueError, match="64"):
                fn(plan, spec, SCALE, np.linspace(1.0, 60.0, 65), angles, RATIO)
        for fn in (D.sharded_fit_region, D.spatial_fit_region):
            with pytest.raises(ValueError, match="256 orientations"):
                fn(plan, spec, SCALE, AGES, wide, RATIO)
        assert plan.launches == n0 and plan.states == 1


# ---------------------------------------------------------------------------
# sb_region_merge
# ---------------------------------------------------------------------------
def _merge_direct(device=None):
    """One region sweep on a slab plan, then the fold of random candidates into a band of its rows:
    the band must equal a NumPy sum / min / max / OR fold, the other rows keep the sweep's planes."""
    import torch
    from scarplet_b200 import distributed as D
    from scarplet_b200 import params as P
    from scarplet_b200._lib import SbError, check
    from scarplet_b200.engine import Plan
    z, _, _ = _inputs()
    ny, nx = 48, 56
    z = z[:ny, :nx]
    angles = P.search_angles(-np.pi / 2, np.pi / 2)[::4]         # 46 orientations: two words
    spec = _scarp()._sb_spec
    tables = P.region_tables(AGES, angles)
    dev = None if device is None else torch.device(device)
    with Plan(ny, nx, 1.0, 1.0, slab=(10, 38, 24)) as plan:
        plan.set_dem(z)
        with pytest.raises(SbError, match="no region sweep"):
            plan.region_planes()
        a, t, _, _ = plan.build_sweep(spec, SCALE, AGES, angles)
        plan.reset()
        plan.sweep(a, t)
        plan.region_sweep(a, t, RATIO, tables)
        ptr, n_planes = plan.region_planes()
        assert n_planes == 3 + -(-len(tables.pos_angle) // 32) == 5
        rows = plan.row_hi - plan.row_lo

        def planes():
            plan.sync()
            return D._as_tensor(ptr, n_planes * rows * nx, "i4", dev).cpu().numpy().reshape(n_planes, rows, nx).copy()
        before = planes()
        assert (before[0] > 0).sum() > 100
        lo, hi, n_cands = 15, 31, 3
        rng = np.random.default_rng(5)
        cands = np.empty((n_planes, n_cands, hi - lo, nx), dtype=np.int32)
        cands[0] = rng.integers(0, 1000, cands[0].shape)
        cands[1] = rng.integers(0, 40, cands[1].shape)
        cands[2] = rng.integers(0, 40, cands[2].shape)
        cands[3:] = rng.integers(-2 ** 31, 2 ** 31, cands[3:].shape, dtype=np.int64).astype(np.int32)
        cands[:, 1, :, :7] = np.array([0, 0x7f7f7f7f, -1, 0, 0], dtype=np.int32)[:, None, None]   # a cleared candidate
        buf = torch.from_numpy(cands)
        if dev is not None:
            buf = buf.to(dev)
            torch.cuda.synchronize(dev)
        plan.region_merge((lo, hi), n_cands, buf.data_ptr())
        after = planes()
        want = np.concatenate([cands[0].sum(0, dtype=np.int32)[None], cands[1].min(0)[None], cands[2].max(0)[None],
                               np.bitwise_or.reduce(cands[3:], axis=1)])
        assert np.array_equal(after[:, lo - 10:hi - 10], want)
        assert np.array_equal(after[:, :lo - 10], before[:, :lo - 10])
        assert np.array_equal(after[:, hi - 10:], before[:, hi - 10:])

        def merge(lo=lo, hi=hi, n=n_cands, p=buf.data_ptr()):
            check(plan.lib, plan.lib.sb_region_merge(plan._h, lo, hi, n, p))
        for bad, what in ((dict(n=0), "bad arguments"), (dict(p=0), "bad arguments"), (dict(lo=9), "rows outside"),
                          (dict(hi=39), "rows outside"), (dict(lo=20, hi=20), "rows outside")):
            with pytest.raises(SbError, match=what):
                merge(**bad)
        assert np.array_equal(planes(), after)
        plan.set_states(2)                       # a new best state voids the region planes
        with pytest.raises(SbError, match="no region sweep"):
            plan.region_planes()
        with pytest.raises(SbError, match="no region sweep"):
            merge()


def test_region_merge_fold(emu_lib):
    _merge_direct()


@pytest.mark.gpu
def test_gpu_region_merge_fold(cuda_lib):
    _merge_direct("cuda:0")


# ---------------------------------------------------------------------------
# two NCCL ranks on the B200
# ---------------------------------------------------------------------------
GPU_AGES = np.logspace(0, 3.5, 30)[::5]


def _gpu_dems():
    from scarplet_b200.synth import synthetic_dem
    from tests.test_nodata_mask import _gpu_holes
    z = synthetic_dem(1024, seed=6)
    return z, _gpu_holes(z, seed=6)


def _gpu_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch
    import torch.distributed as dist
    from scarplet_b200 import distributed as D
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        spec = _scarp()._sb_spec
        angles = P.search_angles(-np.pi / 2, np.pi / 2)
        z, zm = _gpu_dems()
        for name, dem, kw in (("own", z, {}), ("torch", z, dict(stream=torch.cuda.current_stream(dev).cuda_stream)),
                              ("masked", zm, dict(nodata="mask", min_coverage=0.7))):
            with Plan(1024, 1024, 1.0, 1.0, device=rank, **kw) as plan:
                plan.set_dem(dem)
                for prod, fn in (("region", D.sharded_fit_region), ("range", D.sharded_age_range)):
                    lo, hi, band = fn(plan, spec, 100.0, GPU_AGES, angles, 0.9, device=dev)
                    np.save(os.path.join(out_dir, "%s_%s%d.npy" % (name, prod, rank)),
                            np.concatenate([[lo, hi], band.ravel()]))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_gpu_two_ranks_equal_single_gpu(cuda_lib, tmp_path):
    import torch
    import torch.multiprocessing as mp
    import scarplet_b200 as sl
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    port = 29500 + (os.getpid() + 1531) % 2000
    mp.spawn(_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    z, zm = _gpu_dems()
    Scarp = _scarp()
    for name, dem, masking in (("own", z, {}), ("torch", z, {}), ("masked", zm, dict(nodata="mask", min_coverage=0.7))):
        grid = sl.DEMGrid(dem, 1.0)
        for prod, fn, planes in (("region", sl.fit_region, 9), ("range", sl.age_range, 6)):
            want = fn(grid, Scarp, 100.0, 0.9, ages=GPU_AGES, **masking)
            got = _joined(_bands(tmp_path, "%s_%s" % (name, prod), planes, nx=1024), 1024)
            assert np.array_equal(got, want, equal_nan=True), (name, prod)
            assert (want[3] > 0).sum() > 100000
    sl.release()
