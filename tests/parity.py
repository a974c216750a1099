"""Shared parity metrics (north_star tolerances, SURVEY.md 8(d)).

The tolerance is enforced as a BOUND, not as a fraction:

* amplitude and SNR: ``max`` relative error <= 1e-4 over every pixel whose reference SNR is at
  or above the median of the valid pixels (the pixels a search can report as a detection),
  and at most 5e-5 of ALL valid pixels above 1e-4.  The pixels that exceed it are those whose
  best fit over the whole search has an amplitude ~1e-4 of the raster's typical one (SNR
  ~1e-5, a few rows next to the edge mask): their cross-correlation is a difference of terms
  10^4 times larger, which no float32 transform resolves to 1e-4 *relative*;
* orientation / age: identical on >= 99.9 % of the valid pixels modulo the +-90 degree
  equivalence, and EVERY disagreement explained -- either the reference zeroed the pixel at
  our (age, +-90 degree) through compare's exact-tie reset (core.py:230-240), or our SNR is
  within 1e-4 of the reference's best (top two closer than the tolerance);
* masks: ``snr > 0`` identical except for the reference's exact-tie resets.
"""
import json
import os

import numpy as np

AMP_SNR_RTOL = 1e-4        # north_star: amplitude and SNR relative error <= 1e-4
INDEX_AGREEMENT = 0.999    # north_star: best angle/age identical on >= 99.9 % of valid pixels
FRAC_OVER_TOL = 5e-5       # share of all valid pixels allowed above AMP_SNR_RTOL (measured: ~1e-5)


def stack_report(res, ref, odd_template=True, ref_age_stacks=None, ages=None):
    """Compare two [amp, age, angle, snr] stacks.

    Index agreement is counted modulo the +-90 degree degeneracy (the first and last
    orientation are the same line; for odd templates the amplitude flips sign), as the
    reference itself resolves that pair by 1e-11-level noise (SURVEY.md 8a-3).
    ``ref_age_stacks`` [G, 4, ny, nx] with ``ages`` [G]: the reference's per-age results of a
    multi-age search (core.py:288-291), used to recognise pixels the reference zeroed at
    one age through an exact tie and refilled from another."""
    res = np.asarray(res)
    ref = np.asarray(ref)
    amp, age, ang, snr = res
    ramp, rage, rang, rsnr = ref
    valid = rsnr > 0
    nvalid = int(valid.sum())
    same_age = np.isclose(age, rage, rtol=1e-12, atol=0)
    same = np.isclose(ang, rang, rtol=0, atol=1e-12) & same_age
    a_lo, a_hi = rang[valid].min() if nvalid else 0, rang[valid].max() if nvalid else 0
    full_circle = bool(nvalid and np.isclose(a_hi - a_lo, np.pi))
    degenerate = np.zeros_like(valid)
    if full_circle:
        degenerate = ((np.isclose(ang, a_lo) & np.isclose(rang, a_hi)) |
                      (np.isclose(ang, a_hi) & np.isclose(rang, a_lo))) & same_age
    agree = (same | degenerate) & valid
    sign = np.where(degenerate & odd_template, -1.0, 1.0)
    with np.errstate(divide='ignore', invalid='ignore'):
        snr_rel = np.abs(snr - rsnr) / np.abs(rsnr)
        amp_rel = np.abs(sign * amp - ramp) / np.abs(ramp)
    # Pixels the reference zeroed through compare's exact-tie reset (core.py:230-240): the
    # reference holds 0 while the first-wins device fold keeps the tied maximum.  For the
    # +-90 degree pair the tie is exact in ~7 % of the pixels whose best fit lies there
    # (SURVEY.md 8a-3), so those show up as "mask" differences that are not mask errors.
    tie_reset = (rsnr == 0) & (snr > 0)
    ends = np.isclose(ang, a_lo) | np.isclose(ang, a_hi) if full_circle else np.zeros_like(valid)
    if full_circle:
        tie_reset &= ends
    out = {
        "valid": nvalid,
        "tie_reset_pixels": int(tie_reset.sum()),
        "mask_mismatch_unexplained": int((((snr > 0) != valid) & ~tie_reset).sum()),
        "mask_equal": bool(((snr > 0) == valid).all()),
        "mask_mismatch": int(((snr > 0) != valid).sum()),
        "index_agreement": float(agree.sum() / max(nvalid, 1)),
        "snr_rel_max": float(snr_rel[agree].max()) if agree.any() else 0.0,
        "snr_rel_p50": float(np.median(snr_rel[agree])) if agree.any() else 0.0,
        "amp_rel_p999": float(np.quantile(amp_rel[agree], 0.999)) if agree.any() else 0.0,
        "amp_rel_max": float(amp_rel[agree].max()) if agree.any() else 0.0,
        "frac_snr_over_tol": float((snr_rel[agree] > AMP_SNR_RTOL).mean()) if agree.any() else 0.0,
        "frac_amp_over_tol": float((amp_rel[agree] > AMP_SNR_RTOL).mean()) if agree.any() else 0.0,
        "disagree_snr_gap_max": float(snr_rel[valid & ~agree].max()) if (valid & ~agree).any() else 0.0,
    }
    # ---- the bound: pixels at or above the median reference SNR -------------------------
    if agree.any():
        med = float(np.median(rsnr[valid]))
        strong = agree & (rsnr >= med)
        out["snr_median_ref"] = med
        out["snr_rel_max_strong"] = float(snr_rel[strong].max()) if strong.any() else 0.0
        out["amp_rel_max_strong"] = float(amp_rel[strong].max()) if strong.any() else 0.0
        worst = np.unravel_index(np.argmax(np.where(agree, snr_rel, -1.0)), snr_rel.shape)
        out["worst_pixel"] = [int(worst[0]), int(worst[1])]
        out["worst_pixel_ref_snr"] = float(rsnr[worst])
        out["worst_pixel_snr_percentile"] = float(100.0 * (rsnr[valid] < rsnr[worst]).mean())
    # ---- every disagreement explained ------------------------------------------------------
    dis = valid & ~agree
    n_dis = int(dis.sum())
    explained_tie = np.zeros_like(valid)
    if n_dis and ref_age_stacks is not None and full_circle:
        ages = np.asarray(ages, dtype=np.float64)
        stacks = np.asarray(ref_age_stacks)
        for i, j in np.argwhere(dis & ends):
            k = int(np.argmin(np.abs(np.log(ages) - np.log(max(age[i, j], 1e-300)))))
            if np.isclose(ages[k], age[i, j], rtol=1e-12) and stacks[k][3, i, j] == 0:
                explained_tie[i, j] = True       # the reference zeroed OUR winner at this age by an exact tie
    close = dis & ~explained_tie & (snr_rel <= AMP_SNR_RTOL)
    out["disagree"] = n_dis
    out["disagree_tie_reset"] = int(explained_tie.sum())
    out["disagree_top_two_within_tol"] = int(close.sum())
    out["disagree_unexplained"] = int((dis & ~explained_tie & ~close).sum())
    return out


def assert_parity(rep, frac=None, agreement=INDEX_AGREEMENT, explain=True, tie_share=3e-3):
    """The north_star tolerances as bounds (module docstring).  ``frac`` defaults to
    FRAC_OVER_TOL, but never fewer than three pixels of a small raster."""
    if frac is None:
        frac = max(FRAC_OVER_TOL, 3.0 / max(rep["valid"], 1))
    assert rep["mask_mismatch_unexplained"] == 0, rep
    assert rep["tie_reset_pixels"] <= max(3, int(tie_share * rep["valid"])), rep
    assert rep["index_agreement"] >= agreement, rep
    if explain:
        assert rep["disagree_unexplained"] == 0, rep
    assert rep.get("snr_rel_max_strong", 0.0) <= AMP_SNR_RTOL, rep
    assert rep.get("amp_rel_max_strong", 0.0) <= AMP_SNR_RTOL, rep
    assert rep["frac_snr_over_tol"] <= frac and rep["frac_amp_over_tol"] <= frac, rep


def template_shares(z, spec, scale, ages, angles, device=None, curv=None, options=None, geometry=None, run=None,
                    angle_ids=None, **plan_kw):
    """Yields ``(i, snr, amp)``: the float32 SNR and amplitude planes [ages, rows, nx] of the templates of
    orientation i, from one-orientation shares of the search on a plan with one best state per age
    (read in place through the plan's device pointers; valid until the next yield).  Each share carries
    the whole search's extents (``sb_sweep_ex``), so its planes are those the whole search computes.
    ``curv``: the curvature statistics of a row slab's whole raster.  ``options``: plan options
    (``set_option``) set before the DEM.  ``geometry``: a list that gets each share's ``last_geometry()``.
    ``run``: a slice of at most 64 of ``ages`` (a search over more ages goes in runs); the planes are then
    [len(ages[run]), rows, nx] and the shares still carry the extents of the search over all ``ages``.
    ``angle_ids``: the orientations to yield (default: all)."""
    import ctypes
    from scarplet_b200 import params as P
    from scarplet_b200.distributed import _as_tensor
    from scarplet_b200.engine import Plan
    ny, nx = z.shape
    ages = np.asarray(ages, dtype=np.float64)
    G = len(ages if run is None else ages[run])
    cuda = device is not None
    with Plan(ny, nx, 1.0, 1.0, states=G, **plan_kw) as plan:
        for key, value in (options or {}).items():
            plan.set_option(key, value)
        plan.set_dem(z)
        if curv is not None:
            plan.set_curv_stats(*curv)
        rows = plan.row_hi - plan.row_lo
        if run is not None:
            whole = (ctypes.c_int * 5)(*P.support_extents(spec, scale, ages, angles, nx, ny, 1.0), len(ages))
        for i in (range(len(angles)) if angle_ids is None else angle_ids):
            if run is None:
                a, t, _, _ = plan.build_sweep(spec, scale, ages, angles, angle_slice=(i, i + 1), state_per_age=True)
            else:
                a, t, _, _ = plan.build_sweep(spec, scale, ages[run], angles, angle_slice=(i, i + 1),
                                              state_per_age=True)
                t = (t[0], t[1], whole)
            assert t[2] is not None or len(angles) == 1     # the whole search's extents go with the share
            plan.reset()
            plan.sweep(a, t)
            plan.sync()
            if geometry is not None:
                geometry.append(plan.last_geometry())
            ps, pa, _ = plan.best_state_pointers(0)
            yield (i, _as_tensor(ps, G * rows * nx, "f4", device).reshape(G, rows, nx),
                   _as_tensor(pa, G * rows * nx, "f4", device).reshape(G, rows, nx))
            if cuda:
                import torch
                torch.cuda.synchronize(device)


def save_report(name, rep, extra=None):
    """Keep a parity report as JSON (``gpurun_out/parity/<name>.json`` by default; the kept
    copies of a round live under ``profiles/``)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out_dir = os.environ.get("SB_PARITY_DIR", os.path.join(root, "gpurun_out", "parity"))
    try:
        os.makedirs(out_dir, exist_ok=True)
        doc = dict(rep)
        if extra:
            doc.update(extra)
        with open(os.path.join(out_dir, name + ".json"), "w") as f:
            json.dump(doc, f, indent=1, sort_keys=True)
    except OSError:
        pass
