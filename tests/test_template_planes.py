"""Every template's amplitude and SNR planes from the complex64 (and complex128) sweep against float64,
for each kernel variant the sweep dispatches to (DESIGN.md section 4, "per-template planes").

The planes come from one-orientation shares of a search on a plan with one best state per age
(``tests.parity.template_shares``): state g then holds template (age g, orientation i) wherever its SNR
is > 0, and each share carries the whole search's extents, so its FFT domains, tiles and kernel variants
are those the whole search uses.  The reference is the oracle's arithmetic (core.py:339-375, and
``tests/masked_oracle.py`` for the nodata mask) in float64, per template and pixel.

The error of a float32 FFT pipeline is absolute, not relative: ``snr = ts amp^2 / err`` with
``n err = T3 - ts amp^2`` cancels at weak pixels, where a correct kernel is off by 1e-3 .. 1 relative.
So the errors are scaled by each pixel's conditioning, with ``S = T3 + n sigma^2 + n eps`` (the local
curvature energy under the template, the raster's mean curvature energy -- FFT rounding is global -- and
the float64 floor the reference adds to ``err``):

    e_x   = |amp_dev - amp_ref| ts / sqrt(ts S)        (the cross-correlation)
    e_err = n |err_dev - err_ref| / S                   (the misfit, err = ts amp^2 / snr)

bounded by ``2 * 2^-24 * log2(Py Px)`` for complex64 and ``4 * 2^-24`` for complex128 (whose best state
is float32).  ``n`` and ``ts`` are the template's, or for a masked search the pixel's ``n_valid`` and
``ts - D_t``, whose own rounding widens both scales where nodata lies under the template
(``plane_errors``).  The masks ``snr > 0`` and ``amp != 0`` equal the reference's exactly outside the
pixels the reference leaves an SNR at, and inside them wherever the reference cross-correlation is
resolved from 0.

``kernel_variants`` names the kernel instantiations a sweep reaches, restating the dispatch of
``run_sweep_t``; ``test_variant_coverage`` holds the emulator matrix to every complex64 instantiation
the dispatcher can reach.  The CPU cases run the emulator build of the kernels (tests/emu), which has no
packed-FP32 arithmetic and no derived twiddles: the ``gpu`` cases check those on the B200 and keep their
measurements under ``profiles/r11_planes/``."""
import math
import time

import numpy as np
import pytest

from oracle import scarplet_oracle as O
from tests import masked_oracle as MO
from tests.parity import save_report, template_shares

F32_ULP = 2.0 ** -24
KINDS = {"Scarp": O.SCARP, "Channel": O.RICKER, "RightFacingUpperBreakScarp": O.RIGHT_UPPER,
         "LeftFacingUpperBreakScarp": O.LEFT_UPPER}
FFT_LENGTHS = (128, 256, 512, 1024, 2048, 4096, 8192)
MAX_FFT_MASKED = 4096          # sb_lib.cu kMaxFftMasked
MAX_BATCH = 64                 # kConvPMaxBatch, kConvRMaxBatch, kFitMaxBatch (sb_fast.cuh, sb_r64.cuh)


def bound(precision, Py, Px):
    return 4.0 * F32_ULP if precision == 64 else 2.0 * F32_ULP * math.log2(Py * Px)


# ---------------------------------------------------------------------------
# the float64 reference
# ---------------------------------------------------------------------------
class Reference(object):
    """Float64 per-template planes of ``z`` (core.py:339-375; with ``min_coverage`` the nodata-masked fit
    of ``tests/masked_oracle.py``), the curvature spectra of each orientation kept for its ages.
    ``rows``: the band of raster rows a row slab computes."""

    def __init__(self, z, min_coverage=None, rows=None, workers=-1):
        import scipy.fft
        self.fft = scipy.fft
        self.workers = workers
        self.z = np.asarray(z, dtype=np.float64)
        self.shape = self.z.shape
        self.masked = min_coverage is not None
        self.min_coverage = min_coverage
        self.rows = slice(None) if rows is None else slice(*rows)
        self._angle = None
        if self.masked:
            v = MO.valid_cells(self.z)
            self.v = v
            self.fu = self._rfft((~v).astype(np.float64))

    def _rfft(self, a):
        return self.fft.rfft2(a, workers=self.workers)

    def _conv(self, fa, fb):
        out = self.fft.irfft2(fa * fb, s=self.shape, workers=self.workers)
        return np.fft.fftshift(out)[self.rows]

    def _curvature(self, angle):
        if self._angle != angle:
            if self.masked:
                curv = O.directional_laplacian(np.where(np.isfinite(self.z), self.z, 0.0), 1.0, 1.0, angle)
                curv = np.where(self.v, curv, 0.0)
            else:
                curv = O.directional_laplacian(self.z, 1.0, 1.0, angle)
            self.sigma2 = float(np.mean(curv ** 2))
            self.fc, self.fc2 = self._rfft(curv), self._rfft(curv ** 2)
            self._angle = angle
        return self.fc, self.fc2

    def template(self, tmpl, scale, age, angle):
        """dict: ``amp``, ``snr`` (the oracle's planes after its masks), ``amp_raw`` (before them), ``live``
        (the pixels the masks leave an SNR at), ``n``, ``ts`` (scalars, or per pixel for a masked fit),
        ``ts_round`` (the template's whole ``ts`` where a masked fit's ``ts - D_t`` has nodata under it,
        else 0), ``T3`` and ``sigma2``."""
        kind = KINDS[tmpl]
        ny, nx = self.shape
        fc, fc2 = self._curvature(angle)
        t = O.template_array(kind, scale, age, angle, nx, ny, 1.0)
        M = (t != 0).astype(np.float64)
        n, ts = float(M.sum()), float(np.sum(t ** 2))
        ts_round = 0.0
        ft, fm = self._rfft(t), self._rfft(M)
        xcorr = self._conv(ft, fc)
        T3 = self._conv(fm, fc2)
        cand = np.ones(xcorr.shape, dtype=bool)
        if self.masked:
            miss = np.rint(self._conv(fm, self.fu)).astype(np.int64)
            D_t = self._conv(self._rfft(t ** 2), self.fu)
            n = n - miss
            ts_round = np.where(miss == 0, 0.0, ts)
            ts = np.where(miss == 0, ts, ts - D_t)
            cand = (n >= math.ceil(self.min_coverage * M.sum())) & np.isfinite(self.z[self.rows])
        with np.errstate(divide="ignore", invalid="ignore"):
            amp = xcorr / ts                                             # core.py:360
            T1 = ts * amp ** 2                                           # core.py:362
            err = (1 / (n + O.EPS)) * (T1 - 2 * amp * xcorr + T3) + O.EPS    # core.py:366
            snr = np.abs(T1 / err)                                       # core.py:367
        c, d = O.template_constants(kind, scale, age, nx)
        cand &= ~O.window_limits(kind, nx, ny, 1.0, -angle, c, d)[self.rows]   # core.py:373-375
        live = cand.copy()
        em = O.err_mask(kind, angle, nx, ny, 1.0)                        # core.py:369-371
        if em is not None:
            snr[em[self.rows]] = 0
            live &= ~em[self.rows]
        return dict(amp=np.where(cand, amp, 0.0), snr=np.where(cand, snr, 0.0), amp_raw=amp, live=live, n=n,
                    ts=ts, ts_round=ts_round, T3=T3, sigma2=self.sigma2)


def plane_errors(dev_amp, dev_snr, ref, label=""):
    """Errors of one template's device planes (float32) against ``Reference.template``: ``e_x``, ``e_err``
    (max and median), the worst pixel, and the pixels where ``snr > 0`` or ``amp != 0`` differ.  A
    device state holds a template only where its SNR is > 0, so the reference amplitude counts only there.

    A masked fit's ``ts - D_t`` comes from an FFT correlation of the template's energy ``t^2`` with the
    nodata, whose rounding is relative to the template's whole ``ts`` (not to ``D_t``, nor to the
    difference, which can be 1e-7 of ``ts``).  An error ``dts`` of it moves ``amp ts`` by ``amp dts`` and
    ``n err`` by ``amp^2 dts``; and ``err``, derived here from the device's ``amp`` and ``snr`` with the
    reference's ``ts - D_t``, moves by ``err dts / (ts - D_t)``.  So where nodata lies under the template
    the scales gain ``|amp| ts`` and ``amp^2 ts + n err ts / (ts - D_t)`` (``ts`` = ``ts_round``);
    elsewhere ``ts_round = 0`` and they are those of the module docstring.

    A mask may differ only at a pixel the reference leaves an SNR at (its window, coverage, finite cell and
    ``get_err_mask``), and there only where the unmasked reference cross-correlation is itself within
    rounding of 0 (float32 ``ts amp^2`` then rounds to 0): ``mask_mismatch_outside`` counts the others,
    ``mask_mismatch_x_max`` is the largest scaled ``|x_ref|`` over the differing pixels."""
    amp = np.asarray(dev_amp, dtype=np.float64)
    snr = np.asarray(dev_snr, dtype=np.float64)
    n, ts = np.broadcast_to(ref["n"], amp.shape), np.broadcast_to(ref["ts"], amp.shape)
    tr = np.broadcast_to(ref["ts_round"], amp.shape)
    fit = ref["snr"] > 0
    ramp = np.where(fit, ref["amp"], 0.0)
    S = np.maximum(ref["T3"], 0.0) + n * ref["sigma2"] + n * O.EPS
    both = fit & (snr > 0)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        e_x = np.where(fit, np.abs(amp - ramp) * ts / (np.sqrt(ts * S) + np.abs(ramp) * tr), 0.0)
        err_ref = ts * ramp ** 2 / ref["snr"]
        err_dev = ts * amp ** 2 / snr
        e_err = np.where(both, n * np.abs(err_dev - err_ref) / (S + ramp ** 2 * tr + n * err_ref * tr / ts), 0.0)
    e_x = np.where(np.isfinite(e_x), e_x, np.inf)
    e_err = np.where(np.isfinite(e_err), e_err, np.inf)
    worst = np.unravel_index(np.argmax(np.maximum(e_x, e_err)), amp.shape)
    flip = ((snr > 0) != fit) | ((amp != 0) != (ramp != 0))
    live = ref["live"]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        a = np.abs(ref["amp_raw"])
        xr = np.where(live, a * ts / (np.sqrt(ts * S) + a * tr), np.inf)
    xr = np.where(np.isnan(xr), np.inf, xr)
    return {
        "label": label,
        "valid": int(fit.sum()),
        "e_x_max": float(e_x.max()), "e_err_max": float(e_err.max()),
        "e_x_p50": float(np.median(e_x[fit])) if fit.any() else 0.0,
        "e_err_p50": float(np.median(e_err[both])) if both.any() else 0.0,
        "worst_pixel": [int(worst[0]), int(worst[1])],
        "worst_ref_snr": float(ref["snr"][worst]), "worst_dev_snr": float(snr[worst]),
        "nodata_pixels": int((fit & (tr > 0)).sum()),
        "snr_mask_mismatch": int(((snr > 0) != fit).sum()),
        "amp_mask_mismatch": int(((amp != 0) != (ramp != 0)).sum()),
        "mask_mismatch_outside": int((flip & ~live).sum()),
        "mask_mismatch_x_max": float(xr[flip & live].max()) if (flip & live).any() else 0.0,
    }


def fold_errors(reps):
    """The worst of several ``plane_errors`` results (the label of the worst template goes with it)."""
    worst = max(reps, key=lambda r: max(r["e_x_max"], r["e_err_max"]))
    return {"templates": len(reps), "e_x_max": max(r["e_x_max"] for r in reps),
            "e_err_max": max(r["e_err_max"] for r in reps),
            "e_x_p50": float(np.median([r["e_x_p50"] for r in reps])),
            "e_err_p50": float(np.median([r["e_err_p50"] for r in reps])),
            "worst_template": worst["label"], "worst_pixel": worst["worst_pixel"],
            "worst_ref_snr": worst["worst_ref_snr"], "worst_dev_snr": worst["worst_dev_snr"],
            "snr_mask_mismatch": sum(r["snr_mask_mismatch"] for r in reps),
            "amp_mask_mismatch": sum(r["amp_mask_mismatch"] for r in reps),
            "mask_mismatch_outside": sum(r["mask_mismatch_outside"] for r in reps),
            "mask_mismatch_x_max": max(r["mask_mismatch_x_max"] for r in reps),
            "valid_min": min(r["valid"] for r in reps), "nodata_pixels": sum(r["nodata_pixels"] for r in reps)}


def assert_within(rep, limit):
    assert rep["mask_mismatch_outside"] == 0, rep
    assert rep["mask_mismatch_x_max"] <= limit, (limit, rep)
    assert rep["e_x_max"] <= limit and rep["e_err_max"] <= limit, (limit, rep)


# ---------------------------------------------------------------------------
# which kernel instantiations a sweep reaches
# ---------------------------------------------------------------------------
def _length_weight(P):
    # sb_lib.cu length_weight
    return {8192: 1.2, 4096: 1.0, 2048: 1.1, 1024: 1.15}.get(P, 1.3)


def axis_tiles(n, length, lo, hi, max_fft, allow_periodic, mixed=True, force_pad=False):
    """FFT lengths of the tiles of one axis: a restatement of ``plan_axis`` (sb_lib.cu:390-471) for
    ``length`` output pixels of an axis of ``n`` (a row slab: fewer, and no periodic domain)."""
    lo, hi = min(lo, 0), max(hi, 0)
    ext = hi - lo + 1
    pow2 = n > 0 and n & (n - 1) == 0
    can_periodic = allow_periodic and pow2 and 128 <= n <= max_fft and not force_pad
    if can_periodic and (not mixed or n <= 4096):
        return [n]
    Ps = [P for P in FFT_LENGTHS if P <= max_fft and not (P < ext + 1 or hi >= P // 2 or -lo > P // 2)]
    if not Ps:
        assert can_periodic, "template support does not fit max_fft"
        return [n]
    if mixed:
        best, pick = [0.0] * (length + 1), [0] * (length + 1)
        for r in range(1, length + 1):
            best[r] = -1.0
            for P in Ps:
                c = P * _length_weight(P) + 48.0 + best[max(0, r - (P - ext))]
                if best[r] < 0 or c < best[r] - 1e-9:
                    best[r], pick[r] = c, P
        if can_periodic and n * _length_weight(n) <= best[length]:
            return [n]
        chosen, r = [], length
        while r > 0:
            chosen.append(pick[r])
            r = max(0, r - (pick[r] - ext))
        return sorted(chosen, reverse=True)
    cost = [(-(-length // (P - ext)) * P, P) for P in Ps]
    best = min(c for c, _ in cost)
    P = 4096 if (best, 4096) in cost else min(P for c, P in cost if c == best)
    return [P] * (-(-length // (P - ext)))


def kernel_variants(shape, extents, n_ages, geom, precision=32, masked=False, options=None, rows=None,
                    max_fft=None, per_angle=None):
    """The kernel instantiations (names as in the CUDA source) one-orientation shares of an ``n_ages``
    search reach: the dispatch of ``run_sweep_t`` (sb_lib.cu) restated --
    k_diff_rows_f/fm and k_curv_cols per tile (:813-831), k_tmpl_rows / k_tmpl_rows_sq with ``xsparse``
    (:868-897), the column kernel (:911-947: k_conv_cols_r with ``sparse64`` when Py = 4096, conv_r64,
    persistent and <= kConvRMaxBatch records; k_conv_cols_p for Py 1024 .. 4096, persistent and
    <= kConvPMaxBatch records; else k_conv_cols_f, each with ``sparse``), the fit kernel (:1028-1045:
    k_fit_rows_gm when masked, else k_fit_rows_g) and the complex128 pipeline (:849-863, 950-958,
    1057-1065).  ``extents``: the whole search's (sy_lo, sy_hi, sx_lo, sx_hi) (``params.support_extents``);
    ``geom``: the share's ``last_geometry()``, whose template batch cuts the chunks and whose largest
    tiles and tile counts must agree with the restated tile plan.  ``per_angle``: templates per
    orientation of the whole search (default ``n_ages``), which picks the persistent column kernels."""
    options = dict(options or {})
    ny, nx = shape
    lo_y, hi_y, lo_x, hi_x = min(extents[0], 0), max(extents[1], 0), min(extents[2], 0), max(extents[3], 0)
    cap = 4096 if precision == 64 else MAX_FFT_MASKED if masked else 8192
    max_fft = min(cap, max_fft or 8192)
    mixed, force_pad = bool(options.get("mixed_tiles", 1)), bool(options.get("force_pad", 0))
    whole = rows is None
    ty = axis_tiles(ny, ny if whole else rows[1] - rows[0], lo_y, hi_y, max_fft, whole, mixed, force_pad)
    tx = axis_tiles(nx, nx, lo_x, hi_x, max_fft, True, mixed, force_pad)
    assert (max(ty), max(tx), len(ty), len(tx)) == (geom["Py"], geom["Px"], geom["tiles_y"], geom["tiles_x"]), \
        (ty, tx, geom)
    rec = 2 if masked else 1
    Bt = geom["template_batch"]
    counts = {min(Bt, n_ages - k) * rec for k in range(0, n_ages, Bt)}
    per_angle = n_ages if per_angle is None else per_angle
    persist = options.get("conv_persist", -1) > 0 or (options.get("conv_persist", -1) < 0 and per_angle >= 4)
    r64 = bool(options.get("conv_r64", 1))
    out = set()
    for N in set(tx):
        if precision == 64:
            out |= {"k_curv_rows<%d, double>" % N, "k_tmpl_rows<%d, double, %s>" % (N, _b(N >= 256 and hi_x <= N // 16 - 1 and lo_x >= -N // 16)),
                    "k_fit_rows<%d, double>" % N}
            continue
        xsparse = N >= 256 and hi_x <= N // 16 - 1 and lo_x >= -(N // 16)
        out.add("k_diff_rows_%s<%d>" % ("fm" if masked else "f", N))
        out.add("k_tmpl_rows<%d, %s>" % (N, _b(xsparse)))
        if masked:
            out.add("k_tmpl_rows_sq<%d, %s>" % (N, _b(xsparse)))
        out.add("k_fit_rows_%s<%d>" % ("gm" if masked else "g", N))
    for N in set(ty):
        if precision == 64:
            out |= {"k_curv_cols<%d, double>" % N, "k_conv_cols<%d, double>" % N}
            continue
        out.add("k_curv_cols<%d>" % N)
        sparse = hi_y <= N // 16 - 1 and lo_y >= -(N // 16)
        for cnt in counts:
            if N == 4096 and r64 and persist and cnt <= MAX_BATCH:
                out.add("k_conv_cols_r<%s>" % _b(hi_y <= 3 * 64 - 1 and lo_y >= -3 * 64))
            elif 1024 <= N <= 4096 and persist and cnt <= MAX_BATCH:
                out.add("k_conv_cols_p<%d, %s>" % (N, _b(sparse)))
            else:
                out.add("k_conv_cols_f<%d, %s>" % (N, _b(sparse)))
    return sorted(out)


def _b(v):
    return "true" if v else "false"


def reachable_complex64():
    """Every complex64 instantiation the dispatcher of ``run_sweep_t`` can launch for FFT lengths
    128 .. 8192 (masked variants up to 4096; ``xsparse`` from 256; persistent column kernels for
    1024 .. 4096, the radix-64 one at 4096)."""
    out = set()
    for N in FFT_LENGTHS:
        xs = (False, True) if N >= 256 else (False,)
        out |= {"k_diff_rows_f<%d>" % N, "k_curv_cols<%d>" % N, "k_fit_rows_g<%d>" % N}
        out |= {"k_tmpl_rows<%d, %s>" % (N, _b(x)) for x in xs}
        out |= {"k_conv_cols_f<%d, %s>" % (N, _b(s)) for s in (False, True)}
        if 1024 <= N <= 4096:
            out |= {"k_conv_cols_p<%d, %s>" % (N, _b(s)) for s in (False, True)}
        if N <= MAX_FFT_MASKED:
            out |= {"k_diff_rows_fm<%d>" % N, "k_fit_rows_gm<%d>" % N}
            out |= {"k_tmpl_rows_sq<%d, %s>" % (N, _b(x)) for x in xs}
    out |= {"k_conv_cols_r<false>", "k_conv_cols_r<true>"}
    return out


# ---------------------------------------------------------------------------
# one case: every template of a search against the reference
# ---------------------------------------------------------------------------
def run_case(z, tmpl, scale, ages, angles, precision=32, min_coverage=None, options=None, device=None,
             slab=None, run=None, max_fft=None, workspace_mb=None, angle_ids=None):
    """``(report, variants, bound)`` of the search ``tmpl`` x ``scale`` x ``ages`` x ``angles`` on ``z``:
    the per-template errors folded over every template (``fold_errors``).  ``run`` (a slice of ``ages``)
    and ``angle_ids`` pick the templates checked; the shares keep the whole search's extents."""
    from scarplet_b200 import params as P
    from scarplet_b200 import templates as T
    spec = getattr(T, tmpl)._sb_spec
    ages = np.asarray(ages, dtype=np.float64)
    angles = np.asarray(angles, dtype=np.float64)
    ny, nx = z.shape
    plan_kw = {}
    if precision != 32:
        plan_kw["precision"] = precision
    if min_coverage is not None:
        plan_kw.update(nodata="mask", min_coverage=min_coverage)
    if max_fft is not None:
        plan_kw["max_fft"] = max_fft
    if workspace_mb is not None:
        plan_kw["workspace_mb"] = workspace_mb
    curv, rows = None, None
    if slab is not None:
        from scarplet_b200 import distributed as D
        from scarplet_b200.engine import Plan
        rows = slab
        plan_kw["slab"] = (slab[0], slab[1], D.slab_halo(spec, scale, ages, angles, nx, ny, 1.0))
        with Plan(ny, nx, 1.0, 1.0) as whole:
            whole.set_dem(z)
            curv = whole.curv_stats()
    run_ages = ages if run is None else ages[run]
    ref = Reference(z, min_coverage, rows)
    geoms, reps = [], []
    for i, snr, amp in template_shares(z, spec, scale, ages, angles, device, curv=curv, options=options,
                                       geometry=geoms, run=run, angle_ids=angle_ids, **plan_kw):
        snr = snr.cpu().numpy() if device is not None else snr.numpy()
        amp = amp.cpu().numpy() if device is not None else amp.numpy()
        for g, age in enumerate(run_ages):
            r = ref.template(tmpl, scale, float(age), float(angles[i]))
            reps.append(plane_errors(amp[g], snr[g], r, "age %g angle %.4f" % (age, angles[i])))
    extents = P.support_extents(spec, scale, ages, angles, nx, ny, 1.0)
    variants = set()
    for g in geoms:
        variants |= set(kernel_variants((ny, nx), extents, len(run_ages), g, precision, min_coverage is not None,
                                        options, rows, max_fft, per_angle=len(ages)))
    rep = fold_errors(reps)
    rep["geometry"] = geoms[0]
    rep["variants"] = sorted(variants)
    return rep, sorted(variants), bound(precision, geoms[0]["Py"], geoms[0]["Px"])


# ---------------------------------------------------------------------------
# CPU: the emulator matrix
# ---------------------------------------------------------------------------
def _dem(shape, seed, relief=None):
    from scarplet_b200.synth import synthetic_dem
    kw = {} if relief is None else dict(relief=relief)
    return synthetic_dem(shape[0], seed=seed, nx=shape[1], **kw)


def _holes(z, seed):
    from tests.test_nodata_mask import _holes as holes
    return holes(z, "border+cells", seed=seed)


_PI2 = np.pi / 2
_A2 = [-0.3, 0.7]
# name: (shape, seed, template, scale, ages, angles, keyword arguments of run_case); SLOW: marked slow
CASES = {
    # periodic and padded domains, odd and rectangular rasters
    "periodic_128": ((128, 128), 1, "Scarp", 8, [2.0, 30.0], _A2, {}),
    "periodic_128_sparse": ((128, 128), 2, "Scarp", 5, [0.5, 2.0], [0.0], {}),
    "padded_96x128": ((96, 128), 3, "Scarp", 8, [2.0, 30.0], _A2, {}),
    "odd_61x75": ((61, 75), 4, "Scarp", 6, [1.0, 8.0], [_PI2], {}),
    "rect_100x300": ((100, 300), 5, "Scarp", 12, [3.0, 60.0], [-1.1], {}),
    # Channel: no edge mask, a live wrap-around; and its support clipped by the raster
    "channel_wrap_64x128": ((64, 128), 6, "Channel", 5, [0.15, 0.3], [-0.2, 0.4], {}),
    "channel_clipped_63x90": ((63, 90), 7, "Channel", 40, [0.05, 0.2], [1.2], {}),
    # get_err_mask column ranges (the fit kernel's ``cross``)
    "left_upper_break": ((80, 96), 8, "LeftFacingUpperBreakScarp", 9, [2.0, 20.0], _A2, {}),
    "right_upper_break": ((80, 96), 9, "RightFacingUpperBreakScarp", 9, [2.0, 20.0], [-1.2, 0.5], {}),
    # column lengths 1024 / 2048 at scale 10 and 70: persistent (_p) and per-template (_f) column kernels
    "col1024_s10_p": ((1024, 64), 10, "Scarp", 10, [1.0, 3.0, 9.0, 30.0], [0.1], dict(options={"conv_persist": 1})),
    "col1024_s10_f": ((1024, 64), 10, "Scarp", 10, [1.0, 3.0, 9.0, 30.0], [0.1], dict(options={"conv_persist": 0})),
    "col1024_s70_p": ((1024, 200), 11, "Scarp", 70, [4.0, 30.0, 200.0, 600.0], [0.1], dict(options={"conv_persist": 1})),
    "col1024_s70_f": ((1024, 200), 11, "Scarp", 70, [4.0, 30.0, 200.0, 600.0], [0.1], dict(options={"conv_persist": 0})),
    "col2048_s20": ((2048, 64), 12, "Scarp", 20, [2.0, 40.0], [0.05], {}),
    # column length 4096: radix-64 (_r, sparse64), radix-16 persistent
    "col4096_s10_r": ((4096, 96), 14, "Scarp", 10, [1.0, 4.0, 16.0, 64.0], [0.0], {}),
    "col4096_s10_p": ((4096, 96), 14, "Scarp", 10, [1.0, 64.0], [0.0], dict(options={"conv_persist": 1, "conv_r64": 0})),
    "col4096_s200_r": ((4096, 96), 15, "Channel", 200, [0.05, 0.2], [0.0], dict(options={"conv_persist": 1})),
    # multi-tile domains, mixed tile lengths, a row slab
    "multitile_max128": ((200, 300), 26, "Scarp", 10, [2.0, 20.0], _A2, dict(max_fft=128)),
    "mixed_tiles_600": ((600, 96), 27, "Scarp", 20, [2.0, 20.0], [0.2], {}),
    "row_slab": ((140, 128), 28, "Scarp", 8, [2.0, 20.0], _A2, dict(slab=(40, 100))),
    # more templates than one chunk holds: a small workspace, and a 70-age search in runs of 64 and 6
    # (the first a full chunk of 64 records)
    "chunks_small_workspace": ((128, 128), 29, "Scarp", 8, list(np.linspace(1.0, 40.0, 9)), [0.4],
                               dict(workspace_mb=1)),
    "ages_70_runs_64_6": ((128, 96), 30, "Scarp", 8, list(np.logspace(0, 2, 70)), [0.4], dict(run_len=64)),
    # supports exactly one row past the sparse column kernels' limits: T = N / 16 rows (hi_y = 8 at
    # N = 128: dense) and 3 R = 192 rows of the radix-64 kernel (hi_y = 192: dense)
    "sparse_edge_128": ((128, 128), 43, "Scarp", 6, [0.5, 2.0], [0.0], {}),
    "sparse64_edge_4096": ((4096, 64), 44, "Channel", 190, [0.05, 0.2], [0.0], dict(options={"conv_persist": 1})),
    # nodata mask: holes and min_coverage 0.6
    "masked_scarp": ((96, 128), 31, "Scarp", 8, [2.0, 20.0], _A2, dict(min_coverage=0.6)),
    "masked_channel": ((64, 128), 32, "Channel", 5, [0.15, 0.3], _A2, dict(min_coverage=0.6)),
    "masked_col1024_p": ((1024, 200), 33, "Scarp", 70, [4.0, 30.0, 200.0, 600.0], [0.1],
                         dict(min_coverage=0.6, options={"conv_persist": 1})),
    "masked_col4096_r": ((4096, 96), 34, "Scarp", 10, [1.0, 4.0, 16.0, 64.0], [0.0], dict(min_coverage=0.6)),
    # complex128
    "precision64_periodic": ((128, 128), 40, "Scarp", 8, [2.0, 30.0], _A2, dict(precision=64)),
    "precision64_padded": ((90, 140), 41, "RightFacingUpperBreakScarp", 9, [2.0, 20.0], [-1.0], dict(precision=64)),
    # DEM magnitude
    "scaled_2m30": ((96, 128), 42, "Scarp", 8, [2.0, 30.0], _A2, dict(dem_scale=2.0 ** -30)),
    "scaled_2p30": ((96, 128), 42, "Scarp", 8, [2.0, 30.0], _A2, dict(dem_scale=2.0 ** 30)),
}
SLOW = {"col4096_s10_p", "col4096_s200_r", "masked_col4096_r", "ages_70_runs_64_6", "sparse64_edge_4096"}


def _generated_cases():
    """Column FFT lengths 256 .. 8192 with sparse (Scarp 5) and dense (Channel N / 8: no edge mask, support
    rows beyond N / 16) template columns, through _f and, for 1024 .. 4096, _p and _r; template rows of
    every length 256 .. 8192 with and without xsparse (Channel N / 8 at +pi/2 against Scarp 5), masked
    up to 4096.  A 8192 axis takes its periodic domain (mixed_tiles 0)."""
    out = {}
    seed = 100
    for N in (256, 512, 1024, 2048, 4096, 8192):
        big = {"mixed_tiles": 0} if N == 8192 else {}
        persists = [("f", {"conv_persist": 0})]
        if 1024 <= N <= 4096:
            persists.append(("p", {"conv_persist": 1, "conv_r64": 0}))
        if N == 4096:
            persists.append(("r", {"conv_persist": 1}))
        for tag, opt in persists:
            out["gen_col%d_sparse_%s" % (N, tag)] = ((N, 64), seed, "Scarp", 5, [1.0, 3.0], [0.0],
                                                    dict(options=dict(big, **opt)))
            out["gen_col%d_dense_%s" % (N, tag)] = ((N, 64), seed + 1, "Channel", N // 8, [0.05, 0.2], [0.0],
                                                   dict(options=dict(big, **opt)))
            seed += 2
        for masked in ((False, True) if N <= 4096 else (False,)):
            kw = dict(options=big)
            if masked:
                kw["min_coverage"] = 0.6
            pre = "gen_masked_row%d" % N if masked else "gen_row%d" % N
            out[pre + "_xsparse"] = ((64, N), seed, "Scarp", 5, [1.0, 3.0], [_PI2], dict(kw))
            out[pre + "_dense"] = ((64, N), seed + 1, "Channel", N // 8, [0.05, 0.2], [_PI2], dict(kw))
            seed += 2
    return out


CASES.update(_generated_cases())
SLOW |= {n for n in CASES if n.startswith("gen_") and ("4096_" in n or "8192_" in n)}


def _run_cpu_case(name):
    shape, seed, tmpl, scale, ages, angles, kw = CASES[name]
    kw = dict(kw)
    z = _dem(shape, seed)
    if "dem_scale" in kw:
        z = z * kw.pop("dem_scale")
    if kw.get("min_coverage") is not None:
        z = _holes(z, seed)
    per = kw.pop("run_len", None)
    if per is None:
        return run_case(z, tmpl, scale, ages, angles, **kw)
    out = [run_case(z, tmpl, scale, ages, angles, run=slice(k, k + per), **kw) for k in range(0, len(ages), per)]
    rep = fold_errors([dict(r, label="run %d" % k, valid=r["valid_min"]) for k, (r, _, _) in enumerate(out)])
    rep["variants"] = sorted(set().union(*(v for _, v, _ in out)))
    return rep, rep["variants"], max(b for _, _, b in out)


def _params():
    return [pytest.param(n, marks=pytest.mark.slow) if n in SLOW else n for n in CASES]


@pytest.mark.parametrize("name", _params())
def test_template_planes(emu_lib, name):
    t0 = time.time()
    rep, variants, limit = _run_cpu_case(name)
    rep["seconds"] = time.time() - t0
    print(name, rep)
    assert rep["valid_min"] > 50, rep
    assert_within(rep, limit)


# instantiations no emulator case reaches, with the reason (none: every one is reached)
GPU_ONLY = {}


def case_variants(name):
    """The variants of a CPU case without its reference: the geometry of its first share's sweep."""
    from scarplet_b200 import params as P
    from scarplet_b200 import templates as T
    shape, seed, tmpl, scale, ages, angles, kw = CASES[name]
    spec = getattr(T, tmpl)._sb_spec
    ages = np.asarray(ages, dtype=np.float64)
    per = kw.get("run_len", len(ages))
    plan_kw = {k: kw[k] for k in ("precision", "max_fft", "workspace_mb") if kw.get(k) is not None}
    if kw.get("min_coverage") is not None:
        plan_kw.update(nodata="mask", min_coverage=kw["min_coverage"])
    rows = kw.get("slab")
    curv = None
    if rows is not None:
        from scarplet_b200 import distributed as D
        plan_kw["slab"] = (rows[0], rows[1], D.slab_halo(spec, scale, ages, angles, shape[1], shape[0], 1.0))
        curv = (1.0, 1.0)
    geoms = []
    for _ in template_shares(_dem(shape, seed), spec, scale, ages, angles, curv=curv, options=kw.get("options"),
                             geometry=geoms, run=slice(0, per), angle_ids=[0], **plan_kw):
        pass
    extents = P.support_extents(spec, scale, ages, angles, shape[1], shape[0], 1.0)
    return kernel_variants(shape, extents, per, geoms[0], kw.get("precision", 32), kw.get("min_coverage") is not None,
                           kw.get("options"), rows, kw.get("max_fft"), per_angle=len(ages))


@pytest.mark.slow
def test_variant_coverage(emu_lib):
    """The emulator matrix reaches every complex64 instantiation the dispatcher can launch (one sweep
    per case, no reference)."""
    reached = set()
    for name in CASES:
        reached |= set(case_variants(name))
    missing = reachable_complex64() - reached - set(GPU_ONLY)
    assert not missing, sorted(missing)
    assert not (set(GPU_ONLY) & reached), sorted(set(GPU_ONLY) & reached)
    assert reached - reachable_complex64() == {v for v in reached if "double" in v}, sorted(reached)


# ---------------------------------------------------------------------------
# on the B200: the packed-FP32 butterflies and derived twiddles, at the shapes users run
# ---------------------------------------------------------------------------
C3_AGES = np.logspace(0, 3.5, 30)


def _full_angles():
    from scarplet_b200 import params as P
    return P.search_angles(-np.pi / 2, np.pi / 2)


# name: (size, seed, template, scale, ages, run of the ages checked, orientations checked, keywords);
# each share carries the extents of the whole search (all ``ages`` x 181 orientations)
GPU_CASES = {
    "g1024_s100": (1024, 6, "Scarp", 100, C3_AGES, slice(0, 30, 6), [37], {}),
    "g4096_s100": (4096, 2, "Scarp", 100, C3_AGES, slice(0, 30, 6), [37], {}),
    "g4096_s10": (4096, 2, "Scarp", 10, C3_AGES, slice(2, 30, 6), [120], {}),
    "g4096_s300": (4096, 3, "Scarp", 300, C3_AGES, slice(3, 30, 6), [100], {}),
    "g4096_s100_r64off": (4096, 2, "Scarp", 100, C3_AGES, slice(0, 30, 6), [37], dict(options={"conv_r64": 0})),
    "g8192_s200": (8192, 4, "Scarp", 200, C3_AGES, slice(1, 30, 6), [70], {}),
    "g3601_channel": (3601, 5, "Channel", 30, np.array([0.05, 0.1, 0.2, 0.3]), slice(0, 4), [10], {}),
    "g1024_masked": (1024, 6, "Scarp", 100, C3_AGES, slice(0, 30, 6), [37], dict(min_coverage=0.7)),
    "g4096_masked": (4096, 2, "Scarp", 100, C3_AGES, slice(0, 30, 6), [150], dict(min_coverage=0.7)),
    "g1024_precision64": (1024, 6, "Scarp", 100, C3_AGES, slice(0, 30, 6), [37], dict(precision=64)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_gpu_template_planes(cuda_lib, name):
    from scarplet_b200.synth import synthetic_dem
    size, seed, tmpl, scale, ages, run, angle_ids, kw = GPU_CASES[name]
    z = synthetic_dem(size, seed=seed)
    if kw.get("min_coverage") is not None:
        from tests.test_nodata_mask import _gpu_holes
        z = _gpu_holes(z, seed=seed)
    t0 = time.time()
    angles = _full_angles()
    rep, variants, limit = run_case(z, tmpl, scale, ages, angles, device="cuda:0", run=run, angle_ids=angle_ids, **kw)
    rep["seconds"] = time.time() - t0
    rep["bound"] = limit
    rep["margin"] = limit / max(rep["e_x_max"], rep["e_err_max"], 1e-30)
    save_report(name, rep, {"config": "%d^2 seed %d, %s %g, ages %s at orientation %s (the shares carry the extents "
                                      "of all %d ages x 181 orientations), %s; one B200"
                                      % (size, seed, tmpl, scale, [round(float(a), 4) for a in ages[run]],
                                         [round(float(angles[i]), 4) for i in angle_ids], len(ages),
                                         kw or "default options")})
    assert rep["valid_min"] > 1000, rep
    assert_within(rep, limit)
