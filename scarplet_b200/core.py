"""Host-side mirror of scarplet/core.py for the template-matching path.

Same function names, positional order, keyword arguments and return layouts as the
reference; the work is done by the CUDA library behind ``engine.Plan``:

* the Pool fan-out over orientations (core.py:180-183) and the age list
  comprehension (core.py:288-291) become one batched sweep on the device;
* ``match_template``'s six FFTs and numexpr passes (core.py:340-375) become the
  kernels in ``csrc/sb_kernels.cuh``;
* the serial ``compare`` fold (core.py:227-241) runs in registers inside the last
  kernel (first maximum wins; see DESIGN.md for the one documented difference on
  exact float64 ties).

Plans (device workspace, twiddle tables, page-locked result buffers) are cached per raster
geometry, so that a second ``match`` on a raster of the same shape pays for nothing but the
DEM upload, the search and the result download; ``release()`` frees them.
"""
import collections
import threading

import numpy as np

from . import engine
from . import params as P
from .engine import Plan
from .templates import device_spec


def _grid_fields(data):
    z = data._griddata
    return z, data._georef_info.dx, data._georef_info.dy


# ---------------------------------------------------------------------------
# plan cache
# ---------------------------------------------------------------------------
_CACHE_SLOTS = 2
_cache = []                      # [(key, plan)], most recently used last
_cache_lock = threading.Lock()


class _Lease(object):
    """A cached plan taken out for one call (context manager: goes back on exit)."""

    def __init__(self, key, plan):
        self.key, self.plan = key, plan

    def __enter__(self):
        return self.plan

    def __exit__(self, exc_type, exc, tb):
        if exc_type is not None:        # a failed call leaves no half-used plan behind
            self.plan.close()
            return False
        with _cache_lock:
            _cache.append((self.key, self.plan))
            while len(_cache) > _CACHE_SLOTS:
                _cache.pop(0)[1].close()
        return False


def _plan_for(data, states=1, nodata="propagate", min_coverage=1.0):
    """A plan for ``data``'s geometry with its DEM uploaded, out of the cache when one is
    free (a plan is used by one call at a time: concurrent callers get their own)."""
    z, dx, dy = _grid_fields(data)
    ny, nx = z.shape
    d = engine.DEFAULTS
    key = (ny, nx, float(dx), float(dy), d["precision"], d["workspace_mb"], d["max_fft"], nodata, float(min_coverage))
    plan = None
    with _cache_lock:
        for i, (k, p) in enumerate(_cache):
            if k == key:
                plan = _cache.pop(i)[1]
                break
    for attempt in (0, 1):
        try:
            if plan is None:
                plan = Plan(ny, nx, dx, dy, nodata=nodata, min_coverage=min_coverage)
            if plan.states != states:
                plan.set_states(states)
            plan.set_dem(z)
            break
        except engine.SbError:
            # most likely device memory held by cached plans of other shapes: drop them, try once more
            if plan is not None:
                plan.close()
                plan = None
            if attempt == 1:
                raise
            release()
    return _Lease(key, plan)


def release():
    """Free the cached plans (device workspace and page-locked result buffers)."""
    with _cache_lock:
        while _cache:
            _cache.pop()[1].close()


# ---------------------------------------------------------------------------
# plugin templates (classes without an on-device generator)
# ---------------------------------------------------------------------------
def _plugin_match_template(plan, data, Template, scale, age, angle, **kwargs):
    """core.py:339-375 for a template class without an on-device generator -- the plugin
    surface: the class is instantiated and asked for its raster and masks exactly as the
    reference does; correlation and fit run on the device (``sb_match_template_raster``).
    One host-rendered raster per call: slow by design, any ``WindowedTemplate`` works."""
    z, dx, _ = _grid_fields(data)
    ny, nx = z.shape
    tobj = Template(scale, age, angle, nx, ny, dx, **kwargs)        # core.py:345
    amp, snr = plan.match_template_raster(tobj.template(), angle)   # core.py:346-367
    if hasattr(tobj, 'get_err_mask'):                               # core.py:369-371
        snr[np.asarray(tobj.get_err_mask(), dtype=bool)] = 0
    mask = np.asarray(tobj.get_window_limits(), dtype=bool)         # core.py:373-375
    amp[mask] = 0
    snr[mask] = 0
    return amp, snr


def _plugin_sweep(data, Template, scale, ages, ang_max, ang_min, order, **kwargs):
    """The reference's own loops (core.py:100-134, 180-188, 288-291) around
    ``_plugin_match_template``, folded with ``compare``'s exact semantics."""
    z, _, _ = _grid_fields(data)
    ny, nx = z.shape
    angles = P.search_angles(ang_min, ang_max)
    with _plan_for(data) as plan:
        def one(age, angle):
            amp, snr = _plugin_match_template(plan, data, Template, scale, age, angle, **kwargs)
            return amp, age, angle, snr
        if order == "angle_major":                                  # core.py:100-134
            best = np.zeros((4, ny, nx), dtype=np.float64)
            for angle in angles:
                for age in ages:
                    plan.compare_fold(best, *one(age, angle))
            return best
        outer = np.zeros((4, ny, nx), dtype=np.float64)
        for age in ages:                                            # core.py:288-291
            best = np.zeros((4, ny, nx), dtype=np.float64)
            for angle in angles:                                    # core.py:180-188
                plan.compare_fold(best, *one(age, angle))
            if len(ages) == 1:
                return best
            plan.compare_fold(outer, best[0], best[1], best[2], best[3])
        return outer


# ---------------------------------------------------------------------------
# the reference API
# ---------------------------------------------------------------------------
def match_template(data, Template, scale, age, angle, **kwargs):
    """Fit one (scale, age, angle) template to the directional curvature
    (core.py:297-377).  Returns ``(amp, age, angle, snr)`` with float64 planes.  Extra
    keyword arguments go to the template's constructor like the reference's (core.py:345);
    a class that takes any is served through its own ``template()``."""
    spec = None if kwargs else device_spec(Template)
    with _plan_for(data) as plan:
        if spec is None:
            amp, snr = _plugin_match_template(plan, data, Template, scale, age, angle, **kwargs)
        else:
            amp, snr = plan.match_template(spec, scale, age, angle)
    return amp, age, angle, snr


def _sweep(data, Template, scales, ages, ang_max, ang_min, order, masking, /, **kwargs):
    """One search per entry of ``scales`` in a single device sweep (they share each
    orientation's curvature spectra); returns the list of (4, ny, nx) stacks.
    ``masking = (nodata, min_coverage)`` of ``engine.Plan.set_nodata`` (positional: every keyword
    argument belongs to the template, as in ``calculate_best_fit_parameters_serial``)."""
    nodata, min_coverage = masking
    spec = None if kwargs else device_spec(Template)
    if spec is None:
        if nodata != "propagate":
            raise ValueError("nodata=%r needs a built-in template class; plugin templates follow the "
                             "reference's NaN semantics" % (nodata,))
        return [_plugin_sweep(data, Template, s, ages, ang_max, ang_min, order, **kwargs) for s in scales]
    angles = P.search_angles(ang_min, ang_max)
    with _plan_for(data, states=len(scales), nodata=nodata, min_coverage=min_coverage) as plan:
        a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, list(scales), ages, angles, order)
        plan.reset()
        plan.sweep(a_rec, t_rec)
        return [plan.finalize(age_of, angle_of, state=k) for k in range(len(scales))]


def calculate_best_fit_parameters(dem, Template, scale, age, ang_max=np.pi / 2,
                                  ang_min=-np.pi / 2, nodata="propagate", min_coverage=1.0, **kwargs):
    """Best amplitude / orientation / SNR at one age over a 1-degree orientation
    search (core.py:139-195).  Returns ndarray (4, ny, nx): [amp, age, angle, snr].
    Like the reference (core.py:182) further keyword arguments are accepted and not
    forwarded to the template.  ``nodata="mask"`` fits only the cells with data
    (``engine.Plan.set_nodata``); the default keeps the reference's NaN semantics."""
    return _sweep(dem, Template, [scale], [age], ang_max, ang_min, "age_major", (nodata, min_coverage))[0]


def calculate_best_fit_parameters_serial(dem, Template, scale, ang_max=np.pi / 2,
                                         ang_min=-np.pi / 2, **kwargs):
    """Flat search over orientations x the 35 default ages (core.py:65-136); keyword
    arguments are forwarded to the template's constructor (core.py:116-121).
    Returns ``(best_amp, best_age, best_angle, best_snr)``."""
    out = _sweep(dem, Template, [scale], P.default_ages(), ang_max, ang_min, "angle_major", _PROPAGATE, **kwargs)[0]
    return out[0], out[1], out[2], out[3]


def _match_args(kwargs):
    ang_max = kwargs.get('ang_max', np.pi / 2)
    ang_min = kwargs.get('ang_min', -np.pi / 2)
    if 'age' in kwargs:
        return [kwargs['age']], ang_max, ang_min, True
    # extension: ``ages=`` replaces the hard-coded 35-age grid of core.py:286
    ages = kwargs.get('ages', None)
    ages = P.default_ages() if ages is None else np.asarray(ages, dtype=np.float64)
    return ages, ang_max, ang_min, False


_PROPAGATE = ("propagate", 1.0)


def _masking(kwargs):
    return kwargs.get("nodata", "propagate"), kwargs.get("min_coverage", 1.0)


def match(data, Template, **kwargs):
    """core.py:266-294.  With ``age=`` one orientation search, returned as a stacked
    ndarray (4, ny, nx); without it the 35-age search, returned like
    ``compare`` as a tuple of four planes.  ``nodata=`` / ``min_coverage=``: see
    ``calculate_best_fit_parameters``."""
    if 'age' in kwargs:
        return calculate_best_fit_parameters(data, Template, **kwargs)
    ages, ang_max, ang_min, _ = _match_args(kwargs)
    out = _sweep(data, Template, [kwargs['scale']], ages, ang_max, ang_min, "age_major", _masking(kwargs))[0]
    return out[0], out[1], out[2], out[3]


def match_scales(data, Template, scales, **kwargs):
    """One ``match`` result per template scale -- the multi-scale product the reference
    publishes as one 4-band raster per scale (CHANGELOG.md:20-24), which its users obtain by
    calling ``match`` in a loop (core.py:266-294 per scale).  Here all scales run in ONE
    device sweep: an orientation's curvature spectra are built once and every scale folds
    into its own best state.  Returns ``{scale: result}`` with ``result`` exactly what
    ``match(..., scale=scale)`` returns."""
    scales = list(scales)
    ages, ang_max, ang_min, single = _match_args(kwargs)
    res = _sweep(data, Template, scales, ages, ang_max, ang_min, "age_major", _masking(kwargs))
    return {s: (r if single else (r[0], r[1], r[2], r[3])) for s, r in zip(scales, res)}


FitSurface = collections.namedtuple("FitSurface", ["amp", "snr", "ages", "angles"])


def fit_surface(data, Template, scale, pixels, ages=None, ang_min=-np.pi / 2, ang_max=np.pi / 2,
                nodata="propagate", min_coverage=1.0, **kwargs):
    """Fit surfaces at chosen pixels: for every (age, orientation) template of the search that
    ``match`` runs with the same arguments, the amplitude and SNR ``match_template`` returns at
    each pixel (masks applied), in float64 -- how sharply the best fit is constrained in age and
    orientation.  Computed by direct correlation over each template's support, not by
    whole-raster FFTs (DESIGN.md section 12).

    ``pixels``: ``(n, 2)`` integers ``(row, col)``.  ``ages=None``: the 35 default ages of
    ``match``.  Returns ``FitSurface(amp, snr, ages, angles)`` with ``amp``, ``snr`` of shape
    ``(n, len(ages), len(angles))``; ``snr.reshape(n, -1).argmax(1)`` is the flat index the search
    picks (up to its float32 near-ties).  ``nodata`` / ``min_coverage``: see
    ``calculate_best_fit_parameters``.  Only the built-in template classes are supported (the
    direct path needs their on-device generators): a plugin class or constructor keyword
    arguments raise ``ValueError``."""
    if kwargs:
        raise ValueError("fit_surface takes no template keyword arguments (%s): the direct path needs a "
                         "built-in template class" % ", ".join(sorted(kwargs)))
    spec = device_spec(Template)
    if spec is None:
        raise ValueError("fit_surface needs a built-in template class; %r has no on-device generator" % (Template,))
    z, _, _ = _grid_fields(data)
    ny, nx = np.shape(z)
    px = np.asarray(pixels)
    if px.size == 0:
        px = np.zeros((0, 2), dtype=np.int64)
    if px.ndim != 2 or px.shape[1] != 2 or px.dtype.kind not in "iu":
        raise ValueError("pixels must be an (n, 2) integer array of (row, col)")
    if px.size and ((px[:, 0] < 0).any() or (px[:, 0] >= ny).any() or (px[:, 1] < 0).any() or (px[:, 1] >= nx).any()):
        raise ValueError("pixels outside the %d x %d raster" % (ny, nx))
    ages = P.default_ages() if ages is None else np.atleast_1d(np.asarray(ages, dtype=np.float64))
    angles = P.search_angles(ang_min, ang_max)
    if len(px) == 0:
        empty = np.zeros((0, len(ages), len(angles)), dtype=np.float64)
        return FitSurface(empty, empty.copy(), ages, angles)
    with _plan_for(data, nodata=nodata, min_coverage=min_coverage) as plan:
        amp, snr = plan.fit_surface(spec, scale, ages, angles, px[:, 0], px[:, 1])
    return FitSurface(amp, snr, ages, angles)


def _age_search(name, Template, ages, kwargs, snr_ratio=None, max_ages=64, angles=None, max_angles=256):
    """(device spec, float64 ages) of an age-resolved search; ``ValueError`` for what it does not take."""
    if kwargs:
        raise ValueError("%s takes no template keyword arguments (%s): the per-age states need a built-in "
                         "template class" % (name, ", ".join(sorted(kwargs))))
    spec = device_spec(Template)
    if spec is None:
        raise ValueError("%s needs a built-in template class; %r has no on-device generator" % (name, Template))
    return spec, search_args(name, ages, snr_ratio, max_ages, angles, max_angles)


def search_args(name, ages, snr_ratio=None, max_ages=64, angles=None, max_angles=256):
    """Float64 ages of an age-resolved search or a fit region (``None``: the 35 default ages);
    ``ValueError`` for what ``name`` does not take: no or more than ``max_ages`` ages (``None``: no
    limit), duplicate ages, ``snr_ratio`` outside (0, 1] and, when ``angles`` is given (a fit region),
    more than ``max_angles`` orientations.  Shared by ``core`` and the multi-GPU drivers of
    ``distributed``, which check before any device work or collective."""
    ages = P.default_ages() if ages is None else np.atleast_1d(np.asarray(ages, dtype=np.float64))
    if max_ages is None:
        if ages.ndim != 1 or len(ages) < 1:
            raise ValueError("%s takes at least one age" % name)
    elif ages.ndim != 1 or not 1 <= len(ages) <= max_ages:
        raise ValueError("%s takes 1 .. %d ages (one best state each), not %d" % (name, max_ages, ages.size))
    if len(np.unique(ages)) != len(ages):
        raise ValueError("%s: duplicate ages" % name)
    if snr_ratio is not None and not (np.isfinite(snr_ratio) and 0.0 < snr_ratio <= 1.0):
        raise ValueError("snr_ratio must be in (0, 1], not %r" % (snr_ratio,))
    if angles is not None and len(angles) > max_angles:
        raise ValueError("%s takes at most %d orientations, not %d" % (name, max_angles, len(angles)))
    return ages


def _age_sweep(plan, spec, scale, ages, ang_min, ang_max):
    angles = P.search_angles(ang_min, ang_max)
    a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, "age_major", state_per_age=True)
    plan.reset()
    plan.sweep(a_rec, t_rec)
    return age_of, angle_of


def match_ages(data, Template, scale, ages=None, ang_min=-np.pi / 2, ang_max=np.pi / 2, nodata="propagate",
               min_coverage=1.0, **kwargs):
    """The best fit over orientations at EVERY age, from one device sweep: ``{age: (4, ny, nx)}``,
    entry ``a`` being what ``calculate_best_fit_parameters(data, Template, scale, a, ...)`` returns
    (up to the float32 rounding of the FFT pipeline) -- the per-age results ``match`` folds
    (core.py:288-291), e.g. the SNR as a function of age at every pixel.  Each age folds into its
    own best state (DESIGN.md section 13); the values are views into one (len(ages), 4, ny, nx)
    array.  ``ages=None``: the 35 default ages.  Device memory: the best states take 12 B x ages per
    pixel (x the fit kernel's sub-stream copies on small rasters): 6 GB at 4096^2 with 30 ages.
    Built-in template classes only, at most 64 distinct ages; ``nodata`` / ``min_coverage``: see
    ``calculate_best_fit_parameters``."""
    spec, ages = _age_search("match_ages", Template, ages, kwargs)
    z, _, _ = _grid_fields(data)
    ny, nx = np.shape(z)
    with _plan_for(data, states=len(ages), nodata=nodata, min_coverage=min_coverage) as plan:
        age_of, angle_of = _age_sweep(plan, spec, scale, ages, ang_min, ang_max)
        out = np.empty((len(ages), 4, ny, nx), dtype=np.float64)
        for s in range(len(ages)):
            plan.finalize(age_of, angle_of, state=s, out=out[s])
    return {float(a): out[s] for s, a in enumerate(ages)}


def age_range(data, Template, scale, snr_ratio, ages=None, ang_min=-np.pi / 2, ang_max=np.pi / 2,
              nodata="propagate", min_coverage=1.0, **kwargs):
    """The age range each pixel's SNR supports: (6, ny, nx) float64 [amp, age, angle, snr, age_lo,
    age_hi].  Planes 0..3 are exactly ``match(data, Template, scale=scale, ages=ages, ...)``;
    ``age_lo`` / ``age_hi`` are the smallest / largest age whose best fit over the orientations has
    an SNR of at least ``snr_ratio`` (in (0, 1]) times the pixel's best (compared in float64), 0
    where the pixel has no fit.  One device sweep with one best state per age, reduced on the
    device: 48 B per pixel cross PCIe whatever the number of ages.  Arguments, limits and device
    memory as ``match_ages``."""
    spec, ages = _age_search("age_range", Template, ages, kwargs, snr_ratio)
    with _plan_for(data, states=len(ages), nodata=nodata, min_coverage=min_coverage) as plan:
        age_of, angle_of = _age_sweep(plan, spec, scale, ages, ang_min, ang_max)
        return plan.age_range(age_of, angle_of, snr_ratio)


def fit_region(data, Template, scale, snr_ratio, ages=None, ang_min=-np.pi / 2, ang_max=np.pi / 2,
               nodata="propagate", min_coverage=1.0, **kwargs):
    """Fit confidence region of every pixel: the (age, orientation) templates whose SNR is at least
    ``snr_ratio`` (in (0, 1]) times the pixel's best (compared in float64).  Returns (9, ny, nx)
    float64 [amp, age, angle, snr, age_lo, age_hi, angle_lo, angle_hi, n_fits]:

    * planes 0..3 are exactly ``match(data, Template, scale=scale, ages=ages, ...)``;
    * ``age_lo`` / ``age_hi``: the smallest / largest age among the qualifying templates (what
      ``age_range`` gives, without its 64-age limit);
    * ``angle_lo`` / ``angle_hi``: the shortest orientation arc holding every qualifying
      orientation.  A search spanning pi (the default) is periodic: -pi/2 and pi/2 are one line,
      and an arc across it has ``angle_hi = angle + pi``, so ``angle_lo <= angle_hi < angle_lo + pi``
      -- the strike uncertainty of the fit;
    * ``n_fits``: the number of qualifying templates;

    planes 4..8 are 0 where the pixel has no fit.  Two device sweeps on one plan: ``match``'s, then
    a threshold pass (DESIGN.md section 14) that records the qualifying templates in 4 * (3 +
    ceil(orientations / 32)) B per pixel of device memory, whatever the number of ages (36 B for
    181 orientations).  Built-in template classes only, at most 256 orientations, distinct ages;
    ``nodata`` / ``min_coverage``: see ``calculate_best_fit_parameters``."""
    angles = P.search_angles(ang_min, ang_max)
    spec, ages = _age_search("fit_region", Template, ages, kwargs, snr_ratio, max_ages=None, angles=angles)
    tables = P.region_tables(ages, angles)
    with _plan_for(data, nodata=nodata, min_coverage=min_coverage) as plan:
        a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, "age_major")
        plan.reset()
        plan.sweep(a_rec, t_rec)
        plan.region_sweep(a_rec, t_rec, snr_ratio, tables)
        return plan.region_finalize(age_of, angle_of, tables)


def secondary_fit(data, Template, scale, min_separation, ages=None, ang_min=-np.pi / 2, ang_max=np.pi / 2,
                  nodata="propagate", min_coverage=1.0, **kwargs):
    """The best fit at every pixel among the templates at least ``min_separation`` (radians) in
    orientation from the pixel's best -- what else fits where a scarp crosses a channel or two fault
    sets intersect, and whether a detection fits any strike.  Returns (8, ny, nx) float64
    [amp, age, angle, snr, amp2, age2, angle2, snr2]:

    * planes 0..3 are exactly ``match(data, Template, scale=scale, ages=ages, ...)``;
    * planes 4..7 are the template with the highest float32 SNR (ties: the lowest flat index, the
      search's rule) among those the masks leave a candidate at the pixel, with SNR > 0 and an
      orientation position at least ``params.separation_positions(min_separation, angles)`` from the
      best's.  A search spanning pi (the default) is periodic: -pi/2 and pi/2 are one position, and
      the distance wraps across them.  They are 0 where nothing qualifies or the pixel has no fit,
      and ``[NaN, 0, 0, NaN]`` where plane 3 is NaN.

    Two device sweeps on one plan (DESIGN.md section 16): ``match``'s into best state 0, then the
    same templates into best state 1 with the separation test in the fit kernel.  Device memory
    beyond ``match``'s: 14 B per pixel (best state 1 and a 2-byte position plane; 235 MB at 4096^2).
    Built-in template classes only, at least 2 and at most 256 orientations, distinct ages (any
    number); ``nodata`` / ``min_coverage``: see ``calculate_best_fit_parameters``."""
    angles = P.search_angles(ang_min, ang_max)
    spec, ages = _age_search("secondary_fit", Template, ages, kwargs, max_ages=None, angles=angles)
    m = P.separation_positions(min_separation, angles)
    tables = P.region_tables(ages, angles)
    z, _, _ = _grid_fields(data)
    ny, nx = np.shape(z)
    with _plan_for(data, states=2, nodata=nodata, min_coverage=min_coverage) as plan:
        a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, "age_major")
        plan.reset()
        plan.sweep(a_rec, t_rec)
        plan.secondary_sweep(a_rec, t_rec, tables, m)
        out = np.empty((8, ny, nx), dtype=np.float64)
        plan.finalize(age_of, angle_of, state=0, out=out[:4])
        plan.finalize(age_of, angle_of, state=1, out=out[4:])
        return out


def fit_peak(data, Template, scale, ages=None, ang_min=-np.pi / 2, ang_max=np.pi / 2, nodata="propagate",
             min_coverage=1.0, **kwargs):
    """Each pixel's age and orientation between the grid points: the vertex of the parabola through
    the SNR of its best template and of the templates one age and one orientation either side.
    Returns (8, ny, nx) float64 [amp, age, angle, snr, age_peak, angle_peak, snr_peak, refined]:

    * planes 0..3 are exactly ``match(data, Template, scale=scale, ages=ages, ...)``;
    * the winner has age rank r and orientation position p (``params.region_tables``); its neighbour
      values are the largest float32 SNR > 0 among the templates at (r -+ 1, p) and (r, p -+ 1) that
      the masks leave a candidate at the pixel, 0 where there is none.  A search spanning pi (the
      default) is periodic: -pi/2 and pi/2 share position 0 and positions wrap round;
    * the age axis is refined where 0 < r < len(ages) - 1, both neighbours are > 0 and
      d- + d+ > 0 (d-+ = snr - neighbour, in float64).  On x = log10(sorted ages), with
      h- = x[r] - x[r-1] and h+ = x[r+1] - x[r], ``age_peak = 10 ** (x[r] + u)`` with
      ``u = (d- h+^2 - d+ h-^2) / (2 (d- h+ + d+ h-))`` in [-h-/2, h+/2];
    * the orientation axis is refined where the winner has both orientation neighbours (always in
      a periodic search), they are > 0 and d- + d+ > 0: ``angle_peak = angle + step * (d- - d+) /
      (2 (d- + d+))``, within half a step of ``angle``;
    * ``snr_peak`` is ``snr`` plus the gain of each refined axis (the maximum of the separable
      quadratic), ``refined`` is 1 (age) + 2 (orientation); an unrefined axis keeps its grid value.

    Planes 4..7 are 0 where the pixel has no fit and ``[0, 0, NaN, 0]`` where plane 3 is NaN.  Two
    device sweeps on one plan (DESIGN.md section 17): ``match``'s, then a neighbour pass that
    records the four neighbour SNRs.  Device memory beyond ``match``'s: 20 B per pixel (336 MB at
    4096^2).  Built-in template classes only, distinct ages; at most 65535 ages and orientations
    (the 16-bit fields of the winner's code); ``nodata`` / ``min_coverage``: see
    ``calculate_best_fit_parameters``."""
    angles = P.search_angles(ang_min, ang_max)
    spec, ages = _age_search("fit_peak", Template, ages, kwargs, max_ages=None, angles=angles, max_angles=0xffff)
    if len(ages) > 0xffff:
        raise ValueError("fit_peak takes at most 65535 ages, not %d" % len(ages))
    tables = P.region_tables(ages, angles)
    with _plan_for(data, nodata=nodata, min_coverage=min_coverage) as plan:
        a_rec, t_rec, age_of, angle_of = plan.build_sweep(spec, scale, ages, angles, "age_major")
        plan.reset()
        plan.sweep(a_rec, t_rec)
        plan.peak_sweep(a_rec, t_rec, tables)
        return plan.peak_finalize(age_of, angle_of, tables)


def compare(results, ny, nx):
    """Per-pixel best-SNR select over an iterable of ``(amp, age, angle, snr)``
    (core.py:198-243), with the reference's exact semantics (strict compares, an
    exact tie zeroes the pixel), folded on the device in float64."""
    best = np.zeros((4, ny, nx), dtype=np.float64)
    with Plan(ny, nx, 1.0, 1.0) as plan:
        for this_amp, this_age, this_angle, this_snr in results:
            plan.compare_fold(best, this_amp, this_age, this_angle, this_snr)
    return best[0], best[1], best[2], best[3]
