"""Index logic of the CUDA kernels, checked on CPU through the fiber emulator
(tests/emu): the SAME kernel source compiled with g++ -DSB_EMU.  These tests do not
establish GPU parity (tests/test_gpu_parity.py does, on a B200); they keep the FFT
exchanges, Hermitian packing, halo/tile bookkeeping, masks and the best-state fold from
regressing when no GPU is at hand."""
import numpy as np
import pytest

from oracle import scarplet_oracle as O
from tests.parity import stack_report


def test_emulator_is_not_the_product(emu_lib):
    assert emu_lib.sb_build_info() == b"cpu-emulator (test infrastructure)"


@pytest.mark.parametrize("n", [128, 256, 1024, 4096, 8192])
def test_fft_lengths(emu_lib, n):
    from scarplet_b200.engine import Plan
    rng = np.random.default_rng(n)
    x = (rng.standard_normal((5, n)) + 1j * rng.standard_normal((5, n))).astype(np.complex64)
    with Plan(8, 8, 1.0, 1.0) as plan:
        y = plan.debug_fft(x)
        yi = plan.debug_fft(x, inverse=True)
    ref = np.fft.fft(x.astype(np.complex128), axis=1)
    assert np.abs(y - ref).max() / np.abs(ref).max() < 5e-7
    assert np.abs(yi - np.conj(np.fft.fft(np.conj(x.astype(np.complex128)), axis=1))).max() / np.abs(ref).max() < 5e-7


def test_fft_radix64_core(emu_lib):
    """The 64 x 64 decomposition of the length-4096 transform (sb_r64.cuh: 64 elements per
    thread, one shared-memory exchange): forward and inverse against NumPy."""
    from scarplet_b200.engine import Plan
    rng = np.random.default_rng(64)
    x = (rng.standard_normal((6, 4096)) + 1j * rng.standard_normal((6, 4096))).astype(np.complex64)
    with Plan(8, 8, 1.0, 1.0) as plan:
        y = plan.debug_fft(x, radix64=True)
        yi = plan.debug_fft(x, inverse=True, radix64=True)
    ref = np.fft.fft(x.astype(np.complex128), axis=1)
    refi = np.fft.ifft(x.astype(np.complex128), axis=1) * 4096
    assert np.abs(y - ref).max() / np.abs(ref).max() < 5e-7
    assert np.abs(yi - refi).max() / np.abs(refi).max() < 5e-7


def test_laplacian_bit_exact_and_nan(emu_lib):
    import scarplet_b200 as sl
    rng = np.random.default_rng(0)
    z = (rng.standard_normal((37, 53)) * 10).astype(np.float32).astype(np.float64)
    z[5, 6] = np.nan
    for alpha in (0.0, -np.pi / 2, 0.77):
        out = sl.DEMGrid(z, 2.0, 2.0)._calculate_directional_laplacian(alpha)
        assert np.array_equal(out, O.directional_laplacian(z, 2.0, 2.0, alpha), equal_nan=True)


def test_template_render_matches_oracle(emu_lib):
    from scarplet_b200 import WindowedTemplate as WT
    for angle in (0.0, 0.4, -np.pi / 2):
        t = WT.Scarp(12, 4.0, angle, 61, 50, 1.0).template()
        ref = O.template_array(O.SCARP, 12, 4.0, angle, 61, 50, 1.0)
        assert np.array_equal(t != 0, ref != 0) and np.allclose(t, ref, rtol=1e-13, atol=0)
        t = WT.Channel(5, 0.2, angle, 64, 47, 1.0).template()
        ref = O.template_array(O.RICKER, 5, 0.2, angle, 64, 47, 1.0)
        assert np.array_equal(t != 0, ref != 0) and np.allclose(t, ref, rtol=1e-12, atol=1e-300)
        t = WT.RightFacingUpperBreakScarp(12, 4.0, angle, 61, 50, 1.0).template()
        assert np.allclose(t, O.template_array(O.RIGHT_UPPER, 12, 4.0, angle, 61, 50, 1.0), rtol=1e-13, atol=0)


@pytest.mark.parametrize("shape,cls,kind,scale,age,angle", [
    ((128, 128), "Scarp", O.SCARP, 8, 2.0, 0.3),              # periodic domain
    ((100, 150), "Scarp", O.SCARP, 8, 2.0, -1.1),             # padded, rectangular
    ((61, 75), "Scarp", O.SCARP, 6, 4.0, np.pi / 2),          # odd sizes
    ((64, 128), "Channel", O.RICKER, 5, 0.2, 0.7),            # wrap-around output is live
    ((63, 90), "Channel", O.RICKER, 5, 0.02, -0.4),           # support clipped by the raster
    ((80, 96), "LeftFacingUpperBreakScarp", O.LEFT_UPPER, 8, 3.0, 0.5),
    ((80, 96), "RightFacingUpperBreakScarp", O.RIGHT_UPPER, 8, 3.0, -0.5),
])
@pytest.mark.parametrize("precision", [32, 64])
def test_match_template_vs_oracle(emu_lib, shape, cls, kind, scale, age, angle, precision):
    import scarplet_b200 as sl
    from scarplet_b200 import WindowedTemplate as WT
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(shape[0], seed=shape[1], nx=shape[1], relief=3.0)
    try:
        sl.configure(precision=precision)
        amp, a, g, snr = sl.match_template(sl.DEMGrid(z, 1.0), getattr(WT, cls), scale, age, angle)
    finally:
        sl.configure(precision=32)
    ramp, _, _, rsnr = O.match_template(z, 1.0, 1.0, kind, scale, age, angle)
    assert a == age and g == angle
    assert np.array_equal(snr > 0, rsnr > 0) and np.array_equal(amp != 0, ramp != 0)
    v = rsnr > 0
    tol = 2e-5 if precision == 32 else 1e-9
    assert np.abs(amp - ramp)[v].max() <= tol * np.abs(ramp[v]).max()
    strong = v & (rsnr >= np.median(rsnr[v]))
    assert (np.abs(snr - rsnr)[strong] / rsnr[strong]).max() < (1e-4 if precision == 32 else 1e-8)


def test_search_golden_single_age(emu_lib, golden):
    """The reference's own golden (scarplet/tests/test_core.py:44-61) through the emulated
    kernels, at the reference's np.allclose tolerance."""
    import scarplet_b200 as sl
    from scarplet_b200.WindowedTemplate import Scarp
    res = sl.match(sl.DEMGrid(golden.synthetic_dem, 1.0), Scarp, scale=100, age=10,
                   ang_max=np.pi / 2, ang_min=-np.pi / 2)
    gold = golden.npz("reference_goldens.npz")["synthetic_match2"]
    for i in range(4):
        assert np.allclose(res[i], gold[i])


def test_tiles_equal_single_domain(emu_lib):
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from scarplet_b200.templates import Scarp
    z = synthetic_dem(150, seed=4, nx=170, relief=3.0)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)[1::30]
    outs = []
    for max_fft in (512, 128):
        with Plan(150, 170, 1.0, 1.0, max_fft=max_fft) as plan:
            plan.set_dem(z)
            a, t, age_of, angle_of = plan.build_sweep(Scarp._sb_spec, 10, [2.0, 20.0], angles)
            plan.reset()
            plan.sweep(a, t)
            outs.append(plan.finalize(age_of, angle_of))
            geo = plan.last_geometry()
    assert geo["tiles_y"] > 1 and geo["tiles_x"] > 1
    ref = O.compare((O.match_template(z, 1.0, 1.0, O.SCARP, 10, age, ang)
                     for age in (2.0, 20.0) for ang in angles), 150, 170)
    for out in outs:
        rep = stack_report(out, np.stack(ref))
        assert rep["mask_mismatch_unexplained"] == 0 and rep["index_agreement"] >= 0.999, rep
        assert rep["frac_snr_over_tol"] <= 2e-3, rep


def test_compare_exact_semantics(emu_lib, golden):
    import scarplet_b200 as sl
    r1 = (np.array([[1., 2.], [3., 4.]]), 10., 0.1, np.array([[1., 5.], [2., 0.]]))
    r2 = (np.array([[5., 6.], [7., 8.]]), 20., 0.2, np.array([[1., 4.], [3., 0.]]))
    r3 = (np.array([[9., 9.], [9., 9.]]), 30., 0.3, np.array([[.5, 4.], [3., 1.]]))
    out = np.stack(sl.compare([r1, r2, r3], 2, 2))
    assert np.array_equal(out, golden.npz("reference_runs.npz")["compare_out"])
    # planes instead of scalars for age / angle (the age-sweep path of core.match)
    st = [np.stack([r[0], np.full((2, 2), r[1]), np.full((2, 2), r[2]), r[3]]) for r in (r1, r2, r3)]
    out2 = np.stack(sl.compare(st, 2, 2))
    assert np.array_equal(out2, out)


@pytest.mark.parametrize("scale,ages", [(10, [2.0, 20.0, 60.0]), (70, [5.0])])
def test_persistent_column_kernel(emu_lib, scale, ages):
    """Column FFT length 1024 takes k_conv_cols_p (one CTA per spectrum column, 8 thread
    groups behind named barriers, curvature-spectrum columns staged in shared memory per
    run of same-angle templates): runs shorter and longer than the group count, sparse
    (scale 10) and dense (scale 70 > T = 64 rows) template columns."""
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from scarplet_b200.templates import Scarp
    ny, nx = 1024, 200
    z = synthetic_dem(ny, seed=21, nx=nx, relief=3.0)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)[[3, 50, 90, 140]]
    outs = {}
    for persist in (1, 0):
        with Plan(ny, nx, 1.0, 1.0) as plan:
            plan.set_option("conv_persist", persist)
            plan.set_dem(z)
            a, t, age_of, angle_of = plan.build_sweep(Scarp._sb_spec, scale, ages, angles)
            plan.reset()
            plan.sweep(a, t)
            outs[persist] = plan.finalize(age_of, angle_of)
            assert plan.last_geometry()["Py"] == 1024
    # same arithmetic in the same order as the per-template kernel
    assert np.array_equal(outs[1], outs[0])
    ref = O.compare((O.match_template(z, 1.0, 1.0, O.SCARP, scale, age, ang)
                     for age in ages for ang in angles), ny, nx)
    rep = stack_report(outs[1], np.stack(ref))
    assert rep["mask_mismatch_unexplained"] == 0 and rep["index_agreement"] >= 0.999, rep
    # a 200-column strip holds nothing a scale-70 scarp fits (median SNR 0.07): the bound applies
    # to the upper half of the SNR range, the rest is noise-level
    assert rep["snr_rel_p50"] < 1e-5 and rep["snr_rel_max_strong"] <= 1e-4, rep


@pytest.mark.parametrize("scale,ages", [(10, [2.0, 20.0, 60.0, 150.0, 300.0]), (200, [5.0, 9.0, 14.0, 20.0])])
def test_radix64_column_kernel(emu_lib, scale, ages):
    """Column FFT length 4096 takes k_conv_cols_r (radix-64 core: 64 threads per transform, one
    exchange; the two fields of a template side by side in a pair of groups, halves swapped
    through the idle exchange buffers for the combined store): sparse (6 non-zero rows per
    thread) and dense template columns, runs longer and shorter than the pair count --
    against the radix-16 persistent kernel and the oracle."""
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from scarplet_b200.templates import Scarp
    ny, nx = 4096, 96
    z = synthetic_dem(ny, seed=23, nx=nx)
    angles = P.search_angles(-np.pi / 2, np.pi / 2)[[3, 90, 140]]
    outs = {}
    for r64 in (1, 0):
        with Plan(ny, nx, 1.0, 1.0) as plan:
            plan.set_option("conv_r64", r64)
            plan.set_option("conv_persist", 1)
            plan.set_dem(z)
            a, t, age_of, angle_of = plan.build_sweep(Scarp._sb_spec, scale, ages, angles)
            plan.reset()
            plan.sweep(a, t)
            outs[r64] = plan.finalize(age_of, angle_of)
            assert plan.last_geometry()["Py"] == 4096
    rep = stack_report(outs[1], outs[0])
    assert rep["mask_equal"] and rep["index_agreement"] >= 0.9995 and rep["snr_rel_max_strong"] < 1e-4, rep
    ref = O.compare((O.match_template(z, 1.0, 1.0, O.SCARP, scale, age, ang)
                     for age in ages for ang in angles), ny, nx)
    rep = stack_report(outs[1], np.stack(ref))
    assert rep["mask_mismatch_unexplained"] == 0 and rep["index_agreement"] >= 0.999, rep
    assert rep["snr_rel_max_strong"] <= 1e-4 and rep["amp_rel_max_strong"] <= 1e-4, rep


@pytest.mark.parametrize("shape,angle", [((128, 128), 0.3), ((90, 140), -0.8)])
def test_plugin_template_generic_path(emu_lib, shape, angle):
    """A template class the library has no generator for (tests/plugin_templates.py) goes
    through its own template() / get_window_limits() / get_err_mask() (core.py:345-375) and
    the raster entry point; the oracle's plugin restatement is pinned to the unmodified
    reference in tests/test_oracle_vs_reference.py."""
    import scarplet_b200 as sl
    from scarplet_b200.synth import synthetic_dem
    from plugin_templates import Ridge
    z = synthetic_dem(shape[0], seed=11, nx=shape[1], relief=3.0)
    amp, a, g, snr = sl.match_template(sl.DEMGrid(z, 1.0), Ridge, 9, 1.5, angle)
    ramp, _, _, rsnr = O.match_template_plugin(z, 1.0, 1.0, Ridge, 9, 1.5, angle)
    assert a == 1.5 and g == angle
    assert np.array_equal(snr > 0, rsnr > 0) and np.array_equal(amp != 0, ramp != 0)
    v = rsnr > 0
    assert np.abs(amp - ramp)[ramp != 0].max() <= 2e-5 * np.abs(ramp).max()
    strong = v & (rsnr >= np.median(rsnr[v]))
    assert (np.abs(snr - rsnr)[strong] / rsnr[strong]).max() < 1e-4
    # orientation search with compare's exact semantics (core.py:180-193)
    res = sl.calculate_best_fit_parameters(sl.DEMGrid(z, 1.0), Ridge, 9, 1.5, ang_max=0.06, ang_min=-0.06)
    ref = O.calculate_best_fit_parameters_plugin(z, 1.0, 1.0, Ridge, 9, 1.5, ang_max=0.06, ang_min=-0.06)
    rep = stack_report(res, ref, odd_template=False)
    assert rep["mask_mismatch_unexplained"] == 0 and rep["index_agreement"] >= 0.99, rep


def test_nan_in_dem_search(emu_lib):
    """SURVEY 8a-5: one NaN in the DEM spreads through fft2; compare's arithmetic select
    (core.py:230-240) then leaves NaN in amp / snr wherever some orientation is un-masked, 0
    in age / angle, and 0 where every orientation is edge-masked.  The input is not modified
    (the reference zero-fills it in place, dem.py:85-86)."""
    import scarplet_b200 as sl
    from scarplet_b200.WindowedTemplate import Scarp
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(96, seed=3, nx=128, relief=3.0)
    z[40, 77] = np.nan
    keep = z.copy()
    res = sl.calculate_best_fit_parameters(sl.DEMGrid(z, 1.0), Scarp, 8, 2.0, ang_max=0.3, ang_min=-0.3)
    ref = O.calculate_best_fit_parameters(z, 1.0, 1.0, O.SCARP, 8, 2.0, ang_max=0.3, ang_min=-0.3)
    assert np.array_equal(z, keep, equal_nan=True)
    assert np.isnan(ref[3]).any() and (ref[3] == 0).any()
    for plane in (0, 3):
        assert np.array_equal(np.isnan(res[plane]), np.isnan(ref[plane]))
        assert np.array_equal(res[plane] == 0, ref[plane] == 0)
    assert np.array_equal(res[1], ref[1]) and np.array_equal(res[2], ref[2])


def test_match_scales_one_sweep(emu_lib):
    """The multi-scale entry runs every scale in ONE device sweep (an orientation's curvature
    spectra are shared, each scale folds into its own best state): each result equals the
    oracle's for that scale and the per-scale match() (same masks and indices; values to
    rounding, because the shared FFT domain is sized for the largest scale)."""
    import scarplet_b200 as sl
    from scarplet_b200.WindowedTemplate import Scarp
    from scarplet_b200.synth import synthetic_dem
    z = synthetic_dem(96, seed=8, nx=128)
    grid = sl.DEMGrid(z, 1.0)
    multi = sl.match_scales(grid, Scarp, [6, 10, 14], age=3.0, ang_min=-0.2, ang_max=0.2)
    assert sorted(multi) == [6, 10, 14]
    for scale in (6, 10, 14):
        single = sl.match(grid, Scarp, scale=scale, age=3.0, ang_min=-0.2, ang_max=0.2)
        assert np.array_equal(multi[scale][3] > 0, single[3] > 0)
        assert np.array_equal(multi[scale][1], single[1])
        rep = stack_report(multi[scale], single)
        assert rep["index_agreement"] >= 0.999 and rep["snr_rel_max_strong"] < 1e-5, rep
        ref = O.calculate_best_fit_parameters(z, 1.0, 1.0, O.SCARP, scale, 3.0, ang_max=0.2, ang_min=-0.2,
                                              processes=2)
        rep = stack_report(multi[scale], ref)
        assert rep["mask_mismatch_unexplained"] == 0 and rep["index_agreement"] >= 0.999, rep
        assert rep["snr_rel_max_strong"] <= 1e-4 and rep["amp_rel_max_strong"] <= 1e-4, rep
    sweep = sl.match_scales(grid, Scarp, [8], ages=[2.0, 9.0], ang_min=-0.1, ang_max=0.1)
    ref = sl.match(grid, Scarp, scale=8, ages=[2.0, 9.0], ang_min=-0.1, ang_max=0.1)
    assert isinstance(sweep[8], tuple) and all(np.array_equal(a, b) for a, b in zip(sweep[8], ref))
    sl.release()


def test_results_of_one_plan_never_alias(emu_lib):
    """A long-lived plan hands out pooled (page-locked on a GPU box) result arrays from its
    second result on; an array is only reused once the caller has dropped it and its views."""
    from scarplet_b200 import params as P
    from scarplet_b200.engine import Plan
    from scarplet_b200.synth import synthetic_dem
    from scarplet_b200.templates import Scarp
    z = synthetic_dem(64, seed=2, nx=64, relief=3.0)
    angles = P.search_angles(-0.05, 0.05)
    with Plan(64, 64, 1.0, 1.0) as plan:
        plan.set_dem(z)
        a, t, age_of, angle_of = plan.build_sweep(Scarp._sb_spec, 6, [2.0], angles)
        held = []
        for _ in range(5):
            plan.reset()
            plan.sweep(a, t)
            held.append(plan.finalize(age_of, angle_of))
        assert len({id(h) for h in held}) == 5
        for h in held[1:]:
            assert not np.shares_memory(h, held[0]) and np.array_equal(h, held[0])
        view = held[4][3]
        del held
        plan.reset()
        plan.sweep(a, t)
        again = plan.finalize(age_of, angle_of)
        assert not np.shares_memory(again, view)
