"""Python handle on an ``sb_plan`` (include/scarplet_b200.h): owns the device
workspace for one raster shape and drives sweeps.  Thin by design — tiling, batching
and every kernel launch live in the CUDA library."""
import ctypes
import os
import threading
import weakref
from ctypes import byref, c_double, c_int, c_long, c_void_p

import numpy as np

from . import _lib
from ._lib import SbAngle, SbError, SbTemplate, check  # noqa: F401
from . import params as P


# Process-wide defaults applied to every new Plan (see ``configure``).
DEFAULTS = {"precision": int(os.environ.get("SCARPLET_B200_PRECISION", "32")),
            "workspace_mb": None, "max_fft": None}


def configure(precision=None, workspace_mb=None, max_fft=None):
    """Defaults for plans created by the ``core`` functions.

    ``precision`` 32 (default) runs the FFT pipeline in complex64 — the fast path, within
    the 1e-4 SNR/amplitude tolerance on real terrain; 64 runs the same kernels in
    complex128 and reproduces the reference to ~1e-7 even on noise-free synthetic
    surfaces whose far field is below the float32 FFT noise floor."""
    if precision is not None:
        if int(precision) not in (32, 64):
            raise ValueError("precision must be 32 or 64")
        DEFAULTS["precision"] = int(precision)
    if workspace_mb is not None:
        DEFAULTS["workspace_mb"] = int(workspace_mb)
    if max_fft is not None:
        DEFAULTS["max_fft"] = int(max_fft)


def _as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Plan(object):
    """One raster geometry bound to one CUDA device."""

    def __init__(self, ny, nx, dx, dy, device=-1, stream=None, workspace_mb=None,
                 max_fft=None, force_pad=None, precision=None, slab=None, states=1,
                 nodata="propagate", min_coverage=1.0):
        """``slab=(row_lo, row_hi, halo)``: the plan keeps the geometry of the whole ``ny x nx``
        raster but computes (and holds the DEM for) that band of rows only -- one rank's share
        of a raster sharded spatially over GPUs.  ``states``: independent best states (one per
        template scale of a multi-scale search).  ``nodata``, ``min_coverage``: see
        ``set_nodata``."""
        self.lib = _lib.load()
        self.ny, self.nx = int(ny), int(nx)
        self.dx, self.dy = dx, dy
        self.row_lo, self.row_hi = 0, self.ny
        self.states = 1
        self._pool_lock = threading.Lock()
        self._h = c_void_p()
        # dx ** 2 / dy ** 2 evaluated in Python like dem.py:95,99
        check(self.lib, self.lib.sb_plan_create(byref(self._h), self.ny, self.nx, float(dx),
                                                float(dx ** 2), float(dy ** 2), int(device),
                                                c_void_p(stream or 0), 0))
        self.x, self.y = P.axis_vectors(self.nx, self.ny, dx)     # de = dx, core.py:343
        xs, ys = _as_f64(self.x), _as_f64(self.y)
        check(self.lib, self.lib.sb_set_axes_host(self._h, xs.ctypes.data, ys.ctypes.data))
        workspace_mb = DEFAULTS["workspace_mb"] if workspace_mb is None else workspace_mb
        max_fft = DEFAULTS["max_fft"] if max_fft is None else max_fft
        precision = DEFAULTS["precision"] if precision is None else precision
        if workspace_mb is not None:
            self.set_option("workspace_mb", workspace_mb)
        if max_fft is not None:
            self.set_option("max_fft", max_fft)
        if precision != 32:
            self.set_option("precision", precision)
        if force_pad is not None:
            self.set_option("force_pad", int(force_pad))
        if states != 1:
            self.set_states(states)
        if slab is not None:
            self.set_slab(*slab)
        self.nodata, self.min_coverage = "propagate", 1.0
        if nodata != "propagate" or min_coverage != 1.0:
            self.set_nodata(nodata, min_coverage)

    # -- lifecycle ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.sb_plan_destroy(self._h)
            self._h = c_void_p()
        self.__dict__.pop("_result_pool", None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_option(self, key, value):
        check(self.lib, self.lib.sb_plan_set_option(self._h, key.encode(), int(value)))

    NODATA_MODES = {"propagate": 0, "mask": 1}      # SB_NODATA_PROPAGATE, SB_NODATA_MASK

    def set_nodata(self, mode="propagate", min_coverage=1.0):
        """Nodata policy of the searches; takes effect at the next ``set_dem``.

        ``"propagate"`` (default): the reference's semantics, a NaN anywhere in the DEM makes
        every un-masked pixel NaN.  ``"mask"``: each fit uses only the template cells whose
        curvature is defined (every DEM cell of its stencil finite); a template counts at a pixel
        when those cells are at least ``min_coverage`` (in (0, 1]) of its support, and a pixel
        whose own cell is nodata gets no result.  With ``min_coverage=1`` the values equal the
        reference's on the DEM with its holes filled by anything.  Masked plans need
        precision 32; ``match_template`` keeps the reference's semantics and refuses them."""
        if mode not in Plan.NODATA_MODES:
            raise ValueError("nodata must be 'propagate' or 'mask', not %r" % (mode,))
        check(self.lib, self.lib.sb_plan_set_nodata(self._h, Plan.NODATA_MODES[mode], float(min_coverage)))
        self.nodata, self.min_coverage = mode, float(min_coverage)

    def set_states(self, n):
        """Number of independent best states (resets them)."""
        self.set_option("states", int(n))
        self.states = int(n)

    def set_slab(self, row_lo, row_hi, halo):
        """Restrict the plan to raster rows ``row_lo .. row_hi - 1`` (see ``__init__``)."""
        check(self.lib, self.lib.sb_plan_set_slab(self._h, int(row_lo), int(row_hi), int(halo)))
        self.row_lo, self.row_hi = int(row_lo), int(row_hi)
        self.__dict__.pop("_result_pool", None)

    def dem_rows(self):
        """(first raster row, number of rows) of the DEM band the plan holds (periodic in ny)."""
        r0, n = c_int(), c_int()
        check(self.lib, self.lib.sb_plan_dem_rows(self._h, byref(r0), byref(n)))
        return r0.value, n.value

    @property
    def stream_handle(self):
        """The ``cudaStream_t`` (as an integer) the plan's work is ordered on."""
        return int(self.lib.sb_plan_stream(self._h) or 0)

    @property
    def device_bytes(self):
        return int(self.lib.sb_plan_device_bytes(self._h))

    @property
    def fft_area(self):
        """Sum over the FFT tiles of the last sweep of Py * Px."""
        return float(self.lib.sb_plan_last_fft_area(self._h))

    def curv_stats(self):
        s, n = c_double(), c_double()
        check(self.lib, self.lib.sb_plan_curv_stats(self._h, byref(s), byref(n)))
        return s.value, n.value

    def set_curv_stats(self, sumsq, count):
        """Totals over all slabs of a sharded raster (see ``distributed.share_dem_stats``)."""
        check(self.lib, self.lib.sb_plan_set_curv_stats(self._h, float(sumsq), float(count)))

    @property
    def launches(self):
        return int(self.lib.sb_plan_launch_count(self._h))

    KERNELS = ("k_curv_rows", "k_curv_cols", "k_tmpl_rows", "k_tmpl_sums", "k_conv_cols",
               "k_fit_rows")

    def profile(self, reset=True):
        """Per-kernel device time accumulated while option ``profile`` is on:
        ``{kernel: (total_ms, launches)}``."""
        ms = (ctypes.c_double * 6)()
        n = (ctypes.c_long * 6)()
        check(self.lib, self.lib.sb_plan_profile(self._h, ms, n, int(reset)))
        return {k: (ms[i], n[i]) for i, k in enumerate(self.KERNELS)}

    def last_geometry(self):
        out = (c_int * 6)()
        check(self.lib, self.lib.sb_plan_last_geometry(self._h, out))
        keys = ("Py", "Px", "tiles_y", "tiles_x", "angle_batch", "template_batch")
        return dict(zip(keys, list(out)))

    def sync(self):
        check(self.lib, self.lib.sb_sync(self._h))

    # -- inputs --------------------------------------------------------------
    def set_dem(self, z):
        """Upload ``DEMGrid._griddata`` (host float64, never modified).  A slab plan takes
        either the whole raster (its band is cut out here) or just the band ``dem_rows()``
        describes."""
        r0, nrows = self.dem_rows()
        if np.shape(z) == (self.ny, self.nx) and nrows != self.ny:
            z = np.take(z, (r0 + np.arange(nrows)) % self.ny, axis=0)
        z = _as_f64(z)
        if z.shape != (nrows, self.nx):
            raise ValueError("DEM shape %r does not match the plan %r" % (z.shape, (nrows, self.nx)))
        check(self.lib, self.lib.sb_set_dem_host(self._h, z.ctypes.data))

    def set_dem_device(self, ptr):
        """Borrow a float64 device buffer (e.g. ``tensor.data_ptr()``) holding the rows
        ``dem_rows()`` describes; it must outlive the plan's use of it."""
        check(self.lib, self.lib.sb_set_dem_dev(self._h, c_void_p(int(ptr))))

    # -- single operations -----------------------------------------------------
    def directional_laplacian(self, alpha):
        out = np.empty((self.ny, self.nx), dtype=np.float64)
        a = P.angle_record(alpha)
        check(self.lib, self.lib.sb_directional_laplacian(self._h, byref(a), out.ctypes.data, 0))
        return out

    def render_template(self, spec, scale, age, angle):
        rec = P.template_record(spec, scale, age, angle, self.nx, self.ny, self.dx,
                                self.x, self.y, 0, 0)
        out = np.empty((self.ny, self.nx), dtype=np.float64)
        check(self.lib, self.lib.sb_render_template(self._h, byref(rec), out.ctypes.data, 0))
        return out

    def match_template(self, spec, scale, age, angle):
        rec = P.template_record(spec, scale, age, angle, self.nx, self.ny, self.dx,
                                self.x, self.y, 0, 0)
        a = P.angle_record(angle)
        amp = np.empty((self.ny, self.nx), dtype=np.float64)
        snr = np.empty((self.ny, self.nx), dtype=np.float64)
        check(self.lib, self.lib.sb_match_template(self._h, byref(a), byref(rec),
                                                   amp.ctypes.data, snr.ctypes.data, 0))
        return amp, snr

    def match_template_raster(self, t, angle):
        """Raw ``amp, snr`` planes (core.py:359-367, no masks) for a template raster rendered
        on the host by a plugin class (core.py:345-346); the curvature is taken along
        ``angle``.  Only the box that holds the raster's non-zeros is uploaded."""
        t = _as_f64(t)
        if t.shape != (self.ny, self.nx):
            raise ValueError("template shape %r does not match the plan %r" % (t.shape, (self.ny, self.nx)))
        rows = np.flatnonzero(np.any(t != 0, axis=1))
        cols = np.flatnonzero(np.any(t != 0, axis=0))
        if len(rows) == 0:
            raise ValueError("template is zero everywhere")
        a0, b0 = self.ny // 2, self.nx // 2
        box = np.ascontiguousarray(t[rows[0]:rows[-1] + 1, cols[0]:cols[-1] + 1])
        nz = box[box != 0]
        rms = float(np.sqrt(np.mean(nz * nz)))
        tscale = float(2.0 ** np.clip(np.round(-np.log2(rms)), -300, 300)) if np.isfinite(rms) and rms > 1e-280 else 1.0
        a = P.angle_record(angle)
        amp = np.empty((self.ny, self.nx), dtype=np.float64)
        snr = np.empty((self.ny, self.nx), dtype=np.float64)
        check(self.lib, self.lib.sb_match_template_raster(
            self._h, byref(a), box.ctypes.data, int(rows[0]) - a0, int(rows[-1]) - a0,
            int(cols[0]) - b0, int(cols[-1]) - b0, tscale, amp.ctypes.data, snr.ctypes.data, 0))
        return amp, snr

    def fit_surface(self, spec, scale, ages, angles, rows, cols):
        """Fit surfaces at pixels ``(rows[p], cols[p])`` (``sb_fit_surface``, DESIGN.md section 12):
        float64 ``(amp, snr)`` of shape ``(n_pix, len(ages), len(angles))``, the post-mask values
        ``match_template`` returns there for every (age, angle), by direct correlation.  The records
        are in the sweep's ``age_major`` order, so ``snr.reshape(n_pix, -1)`` is indexed by the flat
        index a search over the same ages and angles decodes."""
        ages = np.atleast_1d(np.asarray(ages, dtype=np.float64))
        angles = np.atleast_1d(np.asarray(angles, dtype=np.float64))
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        cols = np.ascontiguousarray(cols, dtype=np.int32)
        if rows.shape != cols.shape or rows.ndim != 1:
            raise ValueError("rows and cols must be 1-D and of equal length")
        A, G, n = len(angles), len(ages), len(rows)
        arr_a = (SbAngle * max(A, 1))()
        for k, a in enumerate(angles):
            arr_a[k] = P.angle_record(a)
        ai, gi = np.meshgrid(np.arange(A), np.arange(G), indexing="ij")
        recs = P.template_records(spec, scale, ages, angles, self.nx, self.ny, self.dx, self.x, self.y,
                                  np.arange(A), gi * A + ai)                       # [A, G]
        arr_t = P.records_to_ctypes(np.ascontiguousarray(recs.T))               # k = age * A + angle
        amp = np.empty((n, G, A), dtype=np.float64)
        snr = np.empty((n, G, A), dtype=np.float64)
        check(self.lib, self.lib.sb_fit_surface(self._h, arr_a, A, arr_t, A * G, rows.ctypes.data, cols.ctypes.data,
                                                n, amp.ctypes.data, snr.ctypes.data, 0))
        return amp, snr

    # -- sweeps ------------------------------------------------------------------
    def build_sweep(self, spec, scale, ages, angles, order="age_major", angle_slice=None, template_share=None,
                    state_per_age=False):
        """Records for the fan-out over ``angles`` x ``ages``.

        ``order`` fixes the flat result index (the tie priority of ``compare``):
        ``"age_major"`` = ``match``'s hierarchical reduce (core.py:285-292),
        ``"angle_major"`` = ``calculate_best_fit_parameters_serial`` (core.py:116-134).
        ``angle_slice`` restricts the records to a contiguous shard of the angle list
        (multi-GPU) without changing any index.  ``template_share=(rank, world)`` cuts finer:
        the orientation-major list of (orientation, scale, age) templates is split into
        ``world`` contiguous shares that differ by at most one template (181 orientations
        over 8 ranks are 23 / 22 whole orientations, 4 % apart; 5430 templates are 679 / 678),
        an orientation at a cut being shared by two ranks.
        ``scale`` may be a sequence: one best state per scale (``Plan(states=len(scale))``),
        all scales of an orientation in the same sweep so that they share its curvature
        spectra; every state uses the same flat index space.
        ``state_per_age``: the templates of ``ages[g]`` fold into best state ``g``
        (``Plan(states=len(ages))``, read with ``age_range`` or ``finalize(state=g)``); one scale,
        ``"age_major"`` order and at most 64 ages.  The flat indices stay those of ``match``.
        Returns ``(angle_records, template_records, age_of, angle_of)``.
        """
        ages = np.atleast_1d(np.asarray(ages, dtype=np.float64))
        angles = np.asarray(angles, dtype=np.float64)
        scales = [scale] if np.ndim(scale) == 0 else list(scale)
        if state_per_age and (len(scales) != 1 or order != "age_major" or not 1 <= len(ages) <= 64):
            raise ValueError("state_per_age needs one scale, age_major order and 1 .. 64 ages")
        # the records depend on the arguments and the plan's geometry only: a repeated search
        # (the same templates on the next raster of this shape) reuses them (read-only)
        key = (id(spec), tuple(float(s) for s in scales), ages.tobytes(), angles.tobytes(), order,
               None if angle_slice is None else tuple(angle_slice),
               None if template_share is None else tuple(template_share), bool(state_per_age))
        memo = getattr(self, "_sweep_memo", None)
        if memo is None:
            memo = []
            setattr(self, "_sweep_memo", memo)
        for k, sp, val in memo:
            if k == key and sp is spec:
                return val
        val = Plan._build_sweep(self, spec, scales, ages, angles, order, angle_slice, template_share, state_per_age)
        memo.append((key, spec, val))
        del memo[:-4]
        return val

    def _build_sweep(self, spec, scales, ages, angles, order, angle_slice, template_share, state_per_age=False):
        A, G = len(angles), len(ages)
        lo, hi = (0, A) if angle_slice is None else angle_slice
        t_lo = t_hi = None
        ai, gi = np.meshgrid(np.arange(A), np.arange(G), indexing="ij")
        if template_share is not None:
            rank, world = template_share
            per_angle = G * len(scales)
            cuts = Plan._share_cuts(self, spec, scales, ages, angles, world)
            t_lo, t_hi = int(cuts[rank]), int(cuts[rank + 1])
            lo, hi = t_lo // per_angle, -(-t_hi // per_angle)
            if t_hi == t_lo:
                lo = hi = 0
        idx = gi * A + ai if order == "age_major" else ai * G + gi          # [A, G]
        age_of = np.empty(A * G, dtype=np.float64)
        angle_of = np.empty(A * G, dtype=np.float64)
        age_of[idx] = ages[gi]
        angle_of[idx] = angles[ai]
        arr_a = (SbAngle * max(hi - lo, 1))()
        for k, a in enumerate(range(lo, hi)):
            arr_a[k] = P.angle_record(angles[a])
        recs = [P.template_records(spec, sc, ages, angles[lo:hi], self.nx, self.ny, self.dx,
                                   self.x, self.y, np.arange(hi - lo), idx[lo:hi], state=k)
                for k, sc in enumerate(scales)]
        if state_per_age:
            recs[0]["state"] = np.arange(G, dtype=np.int32)[None, :]
        recs = np.stack(recs, axis=1).reshape(-1) if hi > lo else np.zeros(0, dtype=P.TEMPLATE_DTYPE)   # [angle][scale][age]
        if t_lo is not None:
            recs = recs[t_lo - lo * G * len(scales): t_hi - lo * G * len(scales)]
        arr_t = P.records_to_ctypes(recs)
        whole = None
        if (lo, hi) != (0, A) or t_lo is not None:
            # a share of a larger search: the extents of the whole one, so that FFT domains, tiles and
            # kernel variants are chosen as the undivided search chooses them (sb_sweep_ex)
            ext = [P.support_extents(spec, sc, ages, angles, self.nx, self.ny, self.dx) for sc in scales]
            whole = (c_int * 5)(min(e[0] for e in ext), max(e[1] for e in ext), min(e[2] for e in ext),
                                max(e[3] for e in ext), G * len(scales))
        return (arr_a, hi - lo), (arr_t, len(recs), whole), age_of, angle_of

    # relative device time of the per-template kernels in a many-ages search (C3 on one B200:
    # column kernel 338 ms, fit kernel 276 ms, template rows 24 ms of a 643 ms step)
    SHARE_COST = (0.53, 0.43, 0.04)

    def _share_cuts(self, spec, scales, ages, angles, world):
        """Cut points [world + 1] of the orientation-major template list into contiguous shares of
        equal estimated device time.  The column kernel costs the same for every template; the
        fit kernel works on the rows of the template's un-masked window (3344 .. 4094 of 4096
        rows at scale 100, by orientation) and the template kernel on the rows of its support
        (9 .. 333): equal COUNTS leave the ranks of an 8-way C3 search 6 % apart.
        ``SB_SHARE_BALANCE=count`` restores equal counts (shares differ by at most one template)."""
        A, G, S = len(angles), len(ages), len(scales)
        n = A * G * S
        if os.environ.get("SB_SHARE_BALANCE", "cost") == "count" or n < 2 * world:
            base, extra = divmod(n, world)
            return np.array([r * base + min(r, extra) for r in range(world + 1)], dtype=np.int64)
        zero = np.zeros((A, G), dtype=np.int64)
        recs = [P.template_records(spec, sc, ages, angles, self.nx, self.ny, self.dx, self.x, self.y,
                                   np.arange(A), zero, state=k) for k, sc in enumerate(scales)]
        recs = np.stack(recs, axis=1).reshape(-1)                                        # [angle][scale][age]
        rows = np.maximum(recs["i_hi"] - recs["i_lo"] + 1, 0).astype(np.float64)
        sup = np.maximum(recs["sy_hi"] - recs["sy_lo"] + 1, 1).astype(np.float64)
        c_col, c_fit, c_tmpl = Plan.SHARE_COST
        cost = c_col + c_fit * rows / max(rows.mean(), 1.0) + c_tmpl * sup / sup.mean()
        mid = np.cumsum(cost) - 0.5 * cost                       # a template goes to the share its midpoint falls into
        share = np.minimum((mid / cost.sum() * world).astype(np.int64), world - 1)
        return np.searchsorted(share, np.arange(world + 1), side="left").astype(np.int64)

    def reset(self):
        check(self.lib, self.lib.sb_best_reset(self._h))

    def sweep(self, angle_records, template_records):
        arr_a, na = angle_records
        arr_t, nt = template_records[0], template_records[1]
        whole = template_records[2] if len(template_records) > 2 else None
        if nt == 0:
            return
        check(self.lib, self.lib.sb_sweep_ex(self._h, arr_a, na, arr_t, nt, whole))

    # -- results -----------------------------------------------------------------
    def _result_array(self, rows):
        """Host array for a (4, rows, nx) result.  The first result of a plan is an ordinary
        NumPy array.  A plan that keeps producing results (a service looping over rasters of
        one shape, or the plan cache behind ``core.match``) hands out page-locked arrays from
        a small pool instead: the 32 B/px device-to-host copy then runs at PCIe speed instead
        of through page faults and the driver's bounce buffers (5x).  Ownership is explicit:
        an entry is busy from the moment its array is handed out until that array object --
        which every view of it keeps alive through ``.base`` -- is garbage collected
        (``weakref.finalize``), so results never alias, whatever the interpreter does with
        reference counts."""
        shape = (4, rows, self.nx)
        self._n_results = getattr(self, "_n_results", 0) + 1
        if self._n_results < 2:
            return np.empty(shape, dtype=np.float64)
        with self._pool_lock:
            pool = self.__dict__.setdefault("_result_pool", [])
            entry = next((e for e in pool if not e["busy"] and e["rows"] == rows), None)
            if entry is None and len(pool) < 3:
                try:
                    import torch
                    entry = {"tensor": torch.empty(shape, dtype=torch.float64, pin_memory=True),
                             "busy": False, "rows": rows}
                    pool.append(entry)
                except Exception:                  # no torch / no page-locked memory left
                    entry = None
            if entry is None:
                return np.empty(shape, dtype=np.float64)
            entry["busy"] = True
        arr = entry["tensor"].numpy()              # a fresh ndarray object over the pinned block

        def _release(e=entry, lock=self._pool_lock):
            with lock:
                e["busy"] = False
        weakref.finalize(arr, _release)
        return arr

    def finalize(self, age_of, angle_of, state=0, rows=None, out=None):
        """(4, rows, nx) float64 stack [amp, age, angle, snr] (core.py:190-193) of best state
        ``state``; ``rows=(lo, hi)`` restricts it to a band of the plan's rows (default: all
        of them).  ``out``: a caller-owned C-contiguous float64 array of that shape (e.g.
        page-locked) to fill instead of a new one."""
        age_of, angle_of = _as_f64(age_of), _as_f64(angle_of)
        lo, hi = (self.row_lo, self.row_hi) if rows is None else (int(rows[0]), int(rows[1]))
        if out is None:
            out = self._result_array(hi - lo)
        elif (out.shape != (4, hi - lo, self.nx) or out.dtype != np.float64 or
              not out.flags["C_CONTIGUOUS"]):
            raise ValueError("out must be a C-contiguous float64 array of shape %r" % ((4, hi - lo, self.nx),))
        check(self.lib, self.lib.sb_finalize_ex(self._h, int(state), lo, hi, age_of.ctypes.data,
                                                angle_of.ctypes.data, len(age_of), out.ctypes.data, 0))
        return out

    def age_range(self, age_of, angle_of, snr_ratio, rows=None):
        """Age-resolved search (``sb_age_range``, DESIGN.md section 13) after a sweep built with
        ``state_per_age``: (6, rows, nx) float64 [amp, age, angle, snr, age_lo, age_hi].  Planes
        0..3 fold the per-age states as the single-state sweep folds its templates (bit-identical
        to ``finalize`` of that sweep); ``age_lo`` / ``age_hi`` are the smallest / largest age
        whose best SNR is at least ``snr_ratio`` (in (0, 1]) times the pixel's best, 0 where the
        pixel has no fit.  ``rows=(lo, hi)``: a band of the plan's rows (default: all of them)."""
        age_of, angle_of = _as_f64(age_of), _as_f64(angle_of)
        lo, hi = (self.row_lo, self.row_hi) if rows is None else (int(rows[0]), int(rows[1]))
        out = np.empty((6, max(hi - lo, 0), self.nx), dtype=np.float64)
        check(self.lib, self.lib.sb_age_range(self._h, self.states, lo, hi, float(snr_ratio), age_of.ctypes.data,
                                              angle_of.ctypes.data, len(age_of), out.ctypes.data, 0))
        return out

    def region_sweep(self, angle_records, template_records, snr_ratio, tables):
        """Pass 2 of a fit confidence region (``sb_region_sweep``, DESIGN.md section 14): best state 0
        must hold the result of ``sweep`` over the same records.  Sweeps them again and records, per
        pixel, the templates whose SNR is at least ``snr_ratio`` (in (0, 1]) times the pixel's best;
        ``tables``: ``params.region_tables`` of the search.  The best state is not modified."""
        arr_a, na = angle_records
        arr_t, nt = template_records[0], template_records[1]
        whole = template_records[2] if len(template_records) > 2 else None
        rank = np.ascontiguousarray(tables.age_rank, dtype=np.int32)
        pos = np.ascontiguousarray(tables.angle_pos, dtype=np.int32)
        check(self.lib, self.lib.sb_region_sweep(self._h, arr_a, na, arr_t, nt, whole, float(snr_ratio),
                                                 rank.ctypes.data, pos.ctypes.data, len(rank),
                                                 len(tables.pos_angle)))

    def secondary_sweep(self, angle_records, template_records, tables, min_sep_pos):
        """The sweep of a secondary fit (``sb_secondary_sweep``, DESIGN.md section 16): best state 0
        must hold the result of ``sweep`` over the same records, on a plan with 2 best states.  Resets
        best state 1 and sweeps the records into it, folding at each pixel only the templates at least
        ``min_sep_pos`` orientation positions (``params.separation_positions``) from the winner of
        state 0; ``tables``: ``params.region_tables`` of the search.  ``finalize(state=1)`` decodes
        the result; state 0 is not modified."""
        arr_a, na = angle_records
        arr_t, nt = template_records[0], template_records[1]
        whole = template_records[2] if len(template_records) > 2 else None
        pos = np.ascontiguousarray(tables.angle_pos, dtype=np.int32)
        check(self.lib, self.lib.sb_secondary_sweep(self._h, arr_a, na, arr_t, nt, whole, pos.ctypes.data, len(pos),
                                                    len(tables.pos_angle), int(tables.periodic), int(min_sep_pos)))

    def peak_sweep(self, angle_records, template_records, tables):
        """Pass 2 of a sub-grid fit peak (``sb_peak_sweep``, DESIGN.md section 17): best state 0 must
        hold the result of ``sweep`` over the same records.  Sweeps them again and records, per pixel,
        the largest SNR of the templates one age rank and one orientation position either side of the
        winner (``peak_planes``); ``tables``: ``params.region_tables`` of the search.  The best state
        is not modified."""
        arr_a, na = angle_records
        arr_t, nt = template_records[0], template_records[1]
        whole = template_records[2] if len(template_records) > 2 else None
        rank = np.ascontiguousarray(tables.age_rank, dtype=np.int32)
        pos = np.ascontiguousarray(tables.angle_pos, dtype=np.int32)
        check(self.lib, self.lib.sb_peak_sweep(self._h, arr_a, na, arr_t, nt, whole, rank.ctypes.data,
                                               pos.ctypes.data, len(rank), len(tables.rank_age),
                                               len(tables.pos_angle), int(tables.periodic)))

    def peak_finalize(self, age_of, angle_of, tables, rows=None):
        """(8, rows, nx) float64 [amp, age, angle, snr, age_peak, angle_peak, snr_peak, refined] after
        ``peak_sweep`` (``sb_peak_finalize``): planes 0..3 are ``finalize``'s, 4..7 the vertex of the
        parabola through the winner and its neighbours on each axis (``core.fit_peak``).
        ``rows=(lo, hi)``: a band of the plan's rows (default: all of them)."""
        age_of, angle_of = _as_f64(age_of), _as_f64(angle_of)
        lx = np.log10(_as_f64(tables.rank_age))
        pos_angle = _as_f64(tables.pos_angle)
        step = float(pos_angle[1] - pos_angle[0]) if len(pos_angle) > 1 else 0.0
        lo, hi = (self.row_lo, self.row_hi) if rows is None else (int(rows[0]), int(rows[1]))
        out = np.empty((8, max(hi - lo, 0), self.nx), dtype=np.float64)
        check(self.lib, self.lib.sb_peak_finalize(self._h, lo, hi, age_of.ctypes.data, angle_of.ctypes.data,
                                                  len(age_of), lx.ctypes.data, len(lx), len(pos_angle),
                                                  int(tables.periodic), step, out.ctypes.data))
        return out

    def peak_planes(self):
        """Device pointer (int32) of the four neighbour planes after ``peak_sweep`` (``sb_peak_planes``):
        the bits of float32 SNRs, plane ``j`` (age-, age+, orientation-, orientation+) of pixel ``i``
        of the plan's rows at ``[j * rows * nx + i]``."""
        p = c_void_p()
        check(self.lib, self.lib.sb_peak_planes(self._h, byref(p)))
        return p.value

    def region_finalize(self, age_of, angle_of, tables, rows=None):
        """(9, rows, nx) float64 [amp, age, angle, snr, age_lo, age_hi, angle_lo, angle_hi, n_fits] after
        ``region_sweep`` (``sb_region_finalize``): planes 0..3 are ``finalize``'s, 4..8 the region's
        extent in age and orientation and its template count, 0 where the pixel has no fit.
        ``rows=(lo, hi)``: a band of the plan's rows (default: all of them)."""
        age_of, angle_of = _as_f64(age_of), _as_f64(angle_of)
        rank_age, pos_angle = _as_f64(tables.rank_age), _as_f64(tables.pos_angle)
        lo, hi = (self.row_lo, self.row_hi) if rows is None else (int(rows[0]), int(rows[1]))
        out = np.empty((9, max(hi - lo, 0), self.nx), dtype=np.float64)
        check(self.lib, self.lib.sb_region_finalize(self._h, lo, hi, age_of.ctypes.data, angle_of.ctypes.data,
                                                    len(age_of), rank_age.ctypes.data, len(rank_age),
                                                    pos_angle.ctypes.data, len(pos_angle), int(tables.periodic),
                                                    out.ctypes.data, 0))
        return out

    def region_planes(self):
        """``(ptr, n_planes)`` of the region planes after ``region_sweep`` (``sb_region_planes``): int32
        device memory, plane ``p`` of pixel ``i`` of the plan's rows at ``[p * rows * nx + i]``; planes
        count, rank_lo, rank_hi and ``n_planes - 3`` orientation words."""
        p, n = c_void_p(), c_int()
        check(self.lib, self.lib.sb_region_planes(self._h, byref(p), byref(n)))
        return p.value, n.value

    def region_merge(self, rows, n_cands, cands_ptr):
        """Replace the region planes on raster rows ``rows`` by the fold of ``n_cands`` candidates
        (int32 device buffer laid out [plane][candidate][row][nx], ``sb_region_merge``): counts
        summed, rank_lo minimum, rank_hi maximum, orientation words OR-ed."""
        check(self.lib, self.lib.sb_region_merge(self._h, int(rows[0]), int(rows[1]), int(n_cands),
                                                 c_void_p(int(cands_ptr))))

    def finalize_device(self, age_of, angle_of, out_ptr, state=0, rows=None):
        """``finalize`` into device memory (4 * rows * nx float64 at ``out_ptr``)."""
        age_of, angle_of = _as_f64(age_of), _as_f64(angle_of)
        lo, hi = (self.row_lo, self.row_hi) if rows is None else (int(rows[0]), int(rows[1]))
        check(self.lib, self.lib.sb_finalize_ex(self._h, int(state), lo, hi, age_of.ctypes.data,
                                                angle_of.ctypes.data, len(age_of), c_void_p(int(out_ptr)), 1))

    def best_state_pointers(self, state=0):
        """Device pointers (snr float32, amp float32, idx int32) of best state ``state``:
        one value per pixel of the plan's rows."""
        s, a, i = c_void_p(), c_void_p(), c_void_p()
        check(self.lib, self.lib.sb_best_state_ex(self._h, int(state), byref(s), byref(a), byref(i)))
        return s.value, a.value, i.value

    def best_merge(self, state, rows, n_cands, snr_ptr, amp_ptr, idx_ptr):
        """Fold ``n_cands`` candidate states for raster rows ``rows`` (device buffers laid out
        [candidate][row][nx]) into best state ``state``."""
        check(self.lib, self.lib.sb_best_merge(self._h, int(state), int(rows[0]), int(rows[1]), int(n_cands),
                                               c_void_p(int(snr_ptr)), c_void_p(int(amp_ptr)),
                                               c_void_p(int(idx_ptr))))

    def best_pack(self, keys_ptr):
        check(self.lib, self.lib.sb_best_pack(self._h, c_void_p(int(keys_ptr))))

    def best_select(self, gkeys_ptr, amp_ptr):
        check(self.lib, self.lib.sb_best_select(self._h, c_void_p(int(gkeys_ptr)), c_void_p(int(amp_ptr))))

    def best_unpack(self, gkeys_ptr, amp_ptr):
        check(self.lib, self.lib.sb_best_unpack(self._h, c_void_p(int(gkeys_ptr)), c_void_p(int(amp_ptr))))

    def compare_fold(self, best4, amp, age, angle, snr):
        """One step of core.compare (core.py:230-240) with the reference's exact
        strict-compare semantics, on the device in float64."""
        amp, snr = _as_f64(amp), _as_f64(snr)
        age_p = angle_p = None
        age_s = angle_s = 0.0
        if np.ndim(age) == 2:
            age_p = _as_f64(age)
        else:
            age_s = float(age)
        if np.ndim(angle) == 2:
            angle_p = _as_f64(angle)
        else:
            angle_s = float(angle)
        check(self.lib, self.lib.sb_compare_host(
            self._h, best4.ctypes.data, amp.ctypes.data,
            age_p.ctypes.data if age_p is not None else None,
            angle_p.ctypes.data if angle_p is not None else None,
            snr.ctypes.data, age_s, angle_s))
        return best4

    def curvature_noise_moments(self, sigma=100.0, truncate=4.0):
        """Sums behind ``DEMGrid._estimate_curvature_noiselevel`` (dem.py:152-179), see
        ``sb_curvature_noise_moments``."""
        out = (c_double * 10)()
        check(self.lib, self.lib.sb_curvature_noise_moments(self._h, float(sigma), float(truncate), out))
        return np.array(list(out), dtype=np.float64)

    def fill_nodata_pass(self, z, max_search_distance):
        """One filling pass over a host raster (modified in place); returns the NaN count left."""
        if z.shape != (self.ny, self.nx) or z.dtype != np.float64 or not z.flags["C_CONTIGUOUS"]:
            raise ValueError("fill_nodata_pass needs the plan's C-contiguous float64 raster")
        left = c_long()
        check(self.lib, self.lib.sb_fill_nodata(self._h, z.ctypes.data, float(max_search_distance), byref(left)))
        return int(left.value)

    def debug_fft_bench(self, n, rows, reps=10, radix64=False):
        """Developer hook: ms per launch of the batched FFT kernel alone."""
        ms = ctypes.c_float()
        check(self.lib, self.lib.sb_debug_fft_bench(self._h, int(n), int(rows), int(reps), int(bool(radix64)), byref(ms)))
        return float(ms.value)

    def debug_fft(self, x, inverse=False, radix64=False):
        """Unit-test hook: batched complex64 FFT over rows (``radix64``: the 64 x 64 core)."""
        x = np.ascontiguousarray(x, dtype=np.complex64)
        rows, n = x.shape
        out = np.empty_like(x)
        check(self.lib, self.lib.sb_debug_fft(self._h, n, rows, x.ctypes.data, out.ctypes.data,
                                              int(bool(inverse)) | (2 if radix64 else 0)))
        return out
