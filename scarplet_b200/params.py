"""Host-side float64 precomputation for the device kernels.

Everything that decides a mask or an index is evaluated here with NumPy exactly as
the reference evaluates it (same expressions, same operation order), then handed to
the CUDA library as plain numbers, so that masks come out bit-exact:

* axis vectors ``x``, ``y``                     WindowedTemplate.py:50-53
* ``cos``/``sin`` of the search angle and of ``alpha = -angle``   dem.py:103, WindowedTemplate.py:57
* the edge mask of ``get_window_limits`` reduced to an index rectangle   WindowedTemplate.py:66-84
* a conservative support box of the template (the device evaluates the exact window
  ``(abs(xr) < c) & (abs(yr) < d)`` inside it)   WindowedTemplate.py:61-64
"""
import collections

import numpy as np
from scipy.special import erfinv

from ._lib import SbAngle, SbTemplate

KIND_SCARP = 0
KIND_RICKER = 1
ERRMASK_NONE = 0
ERRMASK_XR_LE0 = 1
ERRMASK_XR_GE0 = 2

# exp(-u**2) is exactly 0.0 in float64 beyond this u**2 (denormal underflow); it
# bounds the Ricker support along xr (WindowedTemplate.py:514-515)
_EXP_UNDERFLOW = 745.2


def axis_vectors(nx, ny, de):
    """Centred pixel coordinates, WindowedTemplate.py:50-53."""
    x = de * np.linspace(1, nx, num=nx)
    y = de * np.linspace(1, ny, num=ny)
    x = x - np.mean(x)
    y = y - np.mean(y)
    return x, y


def search_angles(ang_min, ang_max):
    """1-degree orientation grid, core.py:173-175."""
    ang_stepsize = 1
    num_angles = int((180 / np.pi) * (ang_max - ang_min) / ang_stepsize + 1)
    return np.linspace(ang_min, ang_max, num_angles)


RegionTables = collections.namedtuple("RegionTables", ["age_rank", "angle_pos", "rank_age", "pos_angle", "periodic"])


def region_tables(ages, angles, order="age_major"):
    """Per flat index of a sweep over ``angles`` x ``ages`` (``order`` as ``Plan.build_sweep``): the
    rank of its age among the sorted ages and its orientation position, with the inverse tables
    ``rank_age`` and ``pos_angle``.  When the angles span exactly pi (within 1e-9, e.g. the default
    -pi/2 .. pi/2) the search is periodic: the last angle is the first one's line and shares its
    position 0, and positions run 0 .. len(angles) - 2."""
    ages = np.atleast_1d(np.asarray(ages, dtype=np.float64))
    angles = np.atleast_1d(np.asarray(angles, dtype=np.float64))
    A, G = len(angles), len(ages)
    periodic = A > 1 and abs((angles[-1] - angles[0]) - np.pi) <= 1e-9
    n_pos = A - 1 if periodic else A
    rank = np.argsort(np.argsort(ages, kind="stable"), kind="stable")
    pos = np.arange(A) % n_pos
    ai, gi = np.meshgrid(np.arange(A), np.arange(G), indexing="ij")
    idx = gi * A + ai if order == "age_major" else ai * G + gi
    age_rank = np.empty(A * G, dtype=np.int32)
    angle_pos = np.empty(A * G, dtype=np.int32)
    age_rank[idx] = rank[gi]
    angle_pos[idx] = pos[ai]
    return RegionTables(age_rank, angle_pos, np.sort(ages), angles[:n_pos].copy(), bool(periodic))


def separation_positions(min_separation, angles):
    """The orientation separation ``min_separation`` (radians) of a secondary fit as a whole number of
    orientation positions of ``region_tables(ages, angles)``: ``ceil(min_separation / step - 1e-9)``
    with ``step = angles[1] - angles[0]``, so that 10 degrees on the 1-degree grid is 10 positions.
    ``ValueError`` for a single orientation, a ``min_separation`` that is not finite or gives less
    than 1 position, and more positions than the largest distance between two positions
    (``n_pos // 2`` in a periodic search, ``len(angles) - 1`` otherwise)."""
    angles = np.atleast_1d(np.asarray(angles, dtype=np.float64))
    if len(angles) < 2:
        raise ValueError("a secondary fit needs at least 2 orientations, not %d" % len(angles))
    if not np.isfinite(min_separation):
        raise ValueError("min_separation must be finite, not %r" % (min_separation,))
    m = int(np.ceil(float(min_separation) / (angles[1] - angles[0]) - 1e-9))
    t = region_tables([1.0], angles)
    n_pos = len(t.pos_angle)
    max_dist = n_pos // 2 if t.periodic else n_pos - 1
    if not 1 <= m <= max_dist:
        raise ValueError("min_separation %r is %d orientation positions; it must be 1 .. %d" % (min_separation, m,
                                                                                               max_dist))
    return m


def default_ages():
    """core.py:107, 286"""
    return 10 ** np.arange(0, 3.5, 0.1)


def angle_record(angle):
    """Curvature direction as dem.py:103-104 evaluates it."""
    return SbAngle(float(np.cos(angle)), float(np.sin(angle)),
                   float(np.cos(angle) ** 2), float(np.sin(angle) ** 2))


def scarp_halfwidth(kt):
    """WindowedTemplate.py:156-157"""
    frac = 0.9
    return abs(2 * np.sqrt(kt) * erfinv(frac))


def window_rectangle(x, y, alpha, c, d):
    """Rows/cols NOT masked by ``get_window_limits`` (WindowedTemplate.py:66-84) as an
    inclusive index rectangle ``(i_lo, i_hi, j_lo, j_hi)``; empty -> lo > hi."""
    x4 = d * np.cos(alpha - np.pi / 2)
    y4 = d * np.sin(alpha - np.pi / 2)
    x1 = d * np.cos(alpha)
    y1 = d * np.sin(alpha)
    an_y = abs((x4 - x1) + 2 * c * np.cos(alpha - np.pi / 2))
    an_x = abs((y1 - y4) + 2 * c * np.sin(alpha - np.pi / 2))
    keep_x = ~((x < (min(x) + an_x)) | (x > (max(x) - an_x)))
    keep_y = ~((y < (min(y) + an_y)) | (y > (max(y) - an_y)))
    jj = np.flatnonzero(keep_x)
    ii = np.flatnonzero(keep_y)
    if jj.size == 0 or ii.size == 0:
        return 1, 0, 1, 0
    # x and y are monotonic, so the kept set is one run
    return int(ii[0]), int(ii[-1]), int(jj[0]), int(jj[-1])


def support_box(nx, ny, de, ca, sa, c_eff, d):
    """Conservative bounding box of ``(abs(xr) < c_eff) & (abs(yr) < d)`` in pixel
    offsets from the template centre ``(ny // 2, nx // 2)``, clipped to the raster."""
    step = abs(float(de))
    ex = (c_eff * abs(ca) + d * abs(sa)) / step
    ey = (c_eff * abs(sa) + d * abs(ca)) / step
    a0, b0 = ny // 2, nx // 2
    rx = int(min(ex, 4.0 * nx)) + 2
    ry = int(min(ey, 4.0 * ny)) + 2
    sx_lo, sx_hi = max(-rx, -b0), min(rx, nx - 1 - b0)
    sy_lo, sy_hi = max(-ry, -a0), min(ry, ny - 1 - a0)
    return sy_lo, sy_hi, sx_lo, sx_hi


def packing_scale(kind, k0, k1, half_width):
    """Power of two close to 1 / rms(t) over the window.  The kernels transform the pair
    (t * scale, M) as one complex row; without the factor the 0/1 mask M would dominate
    the magnitude and its rounding noise would leak into the (much smaller) template
    spectrum.  A power of two changes no mantissa bit, so results are unaffected
    otherwise."""
    if not np.isfinite(half_width) or half_width <= 0:
        return 1.0
    xr = (np.arange(256) + 0.5) / 256.0 * half_width
    if kind == KIND_SCARP:
        w = (xr / k0) * np.exp(-xr ** 2 / k1)
    else:
        u = k0 * xr
        w = (1. - 2. * u ** 2) * np.exp(-u ** 2)
    rms = float(np.sqrt(np.mean(w ** 2)))
    if not np.isfinite(rms) or rms < 1e-280:
        return 1.0
    return float(2.0 ** np.clip(np.round(-np.log2(rms)), -300, 300))


class DeviceSpec(object):
    """What a built-in template class contributes to an ``SbTemplate`` record."""

    def __init__(self, kind, sign=1.0, errmode=ERRMASK_NONE, edge_mask=True):
        self.kind = kind
        self.sign = sign
        self.errmode = errmode
        self.edge_mask = edge_mask


def _age_scalars(spec, age, nx, de):
    """(c, k0, k1, c_eff, tscale) of one age: everything in ``template_record`` that does
    not depend on the orientation."""
    if spec.kind == KIND_SCARP:
        kt = age
        c = float(scarp_halfwidth(kt))
        k0 = float(2. * kt ** (3 / 2.) * np.sqrt(np.pi))   # WindowedTemplate.py:177
        k1 = float(4. * kt)                                # :178
        c_eff = c
    elif spec.kind == KIND_RICKER:
        f = age
        c = float(nx)                                      # WindowedTemplate.py:491
        k0 = float(np.pi * f)                              # :514
        k1 = 0.0
        c_eff = c
        if abs(k0) > 0:
            c_eff = min(c, np.sqrt(_EXP_UNDERFLOW) / abs(k0) + abs(de))
    else:
        raise ValueError("unknown template kind %r" % (spec.kind,))
    return c, k0, k1, c_eff, packing_scale(spec.kind, k0, k1, c_eff)


TEMPLATE_DTYPE = np.dtype([(name, np.float64 if ctype is SbTemplate._fields_[0][1] else np.int32)
                           for name, ctype in SbTemplate._fields_], align=True)


def template_records(spec, scale, ages, angles, nx, ny, de, x, y, angle_ids, idx, state=0):
    """All ``SbTemplate`` records of the fan-out ``angles`` x ``ages`` at once: a structured
    array of shape (len(angles), len(ages)), field for field what ``template_record``
    returns (tests/test_host_logic.py holds the two against each other).  The reference
    evaluates the trigonometry on scalars (WindowedTemplate.py:57, 68-75), so it is done per
    angle here too; the rest is IEEE arithmetic in the reference's operation order,
    vectorised.  ``angle_ids`` [A] and ``idx`` [A, G] are copied into the records."""
    ages = np.asarray(ages, dtype=np.float64)
    angles = np.asarray(angles, dtype=np.float64)
    A, G = len(angles), len(ages)
    if A == 0 or G == 0 or not (np.all(np.diff(x) > 0) and np.all(np.diff(y) > 0)):
        out = np.zeros((A, G), dtype=TEMPLATE_DTYPE)
        for a in range(A):
            for g in range(G):
                rec = template_record(spec, scale, ages[g], angles[a], nx, ny, de, x, y,
                                      angle_ids[a], idx[a][g], state)
                out[a, g] = tuple(getattr(rec, name) for name, _ in SbTemplate._fields_)
        return out
    alpha = [-float(a) for a in angles]              # WindowedTemplate.py:151, 489
    ca = np.array([float(np.cos(a)) for a in alpha])[:, None]
    sa = np.array([float(np.sin(a)) for a in alpha])[:, None]
    cq = np.array([float(np.cos(a - np.pi / 2)) for a in alpha])[:, None]
    sq = np.array([float(np.sin(a - np.pi / 2)) for a in alpha])[:, None]
    d = float(scale)
    per_age = [_age_scalars(spec, float(age), nx, de) for age in ages]
    c, k0, k1, c_eff, tscale = (np.array(v, dtype=np.float64)[None, :] for v in zip(*per_age))

    out = np.zeros((A, G), dtype=TEMPLATE_DTYPE)
    out["cos_t"], out["sin_t"] = ca, sa
    out["c"], out["d"], out["k0"], out["k1"], out["tscale"] = c, d, k0, k1, tscale
    out["sign"], out["kind"], out["errmode"] = float(spec.sign), spec.kind, spec.errmode
    # support_box
    step = abs(float(de))
    ex = (c_eff * np.abs(ca) + d * np.abs(sa)) / step
    ey = (c_eff * np.abs(sa) + d * np.abs(ca)) / step
    a0, b0 = ny // 2, nx // 2
    rx = np.minimum(ex, 4.0 * nx).astype(np.int64) + 2
    ry = np.minimum(ey, 4.0 * ny).astype(np.int64) + 2
    out["sx_lo"], out["sx_hi"] = np.maximum(-rx, -b0), np.minimum(rx, nx - 1 - b0)
    out["sy_lo"], out["sy_hi"] = np.maximum(-ry, -a0), np.minimum(ry, ny - 1 - a0)
    # window_rectangle
    if spec.edge_mask:
        x4, y4, x1, y1 = d * cq, d * sq, d * ca, d * sa
        an_y = np.abs((x4 - x1) + 2 * c * cq)
        an_x = np.abs((y1 - y4) + 2 * c * sq)
        # ~((v < lo) | (v > hi)) on a rising axis is the run [first v >= lo, last v <= hi]
        j_lo = np.searchsorted(x, np.min(x) + an_x, side="left")
        j_hi = np.searchsorted(x, np.max(x) - an_x, side="right") - 1
        i_lo = np.searchsorted(y, np.min(y) + an_y, side="left")
        i_hi = np.searchsorted(y, np.max(y) - an_y, side="right") - 1
        empty = (j_lo > j_hi) | (i_lo > i_hi)
        out["i_lo"], out["i_hi"] = np.where(empty, 1, i_lo), np.where(empty, 0, i_hi)
        out["j_lo"], out["j_hi"] = np.where(empty, 1, j_lo), np.where(empty, 0, j_hi)
    else:
        out["i_lo"], out["i_hi"], out["j_lo"], out["j_hi"] = 0, ny - 1, 0, nx - 1
    out["angle_id"] = np.asarray(angle_ids, dtype=np.int32)[:, None]
    out["idx"] = np.asarray(idx, dtype=np.int32)
    out["state"] = int(state)
    return out


def support_extents(spec, scale, ages, angles, nx, ny, de):
    """(sy_lo, sy_hi, sx_lo, sx_hi): union of the support boxes of ``template_records`` over
    ``angles`` x ``ages`` (the same arithmetic, without building the records)."""
    ages = np.atleast_1d(np.asarray(ages, dtype=np.float64))
    angles = np.asarray(angles, dtype=np.float64)
    alpha = [-float(a) for a in angles]
    ca = np.array([float(np.cos(a)) for a in alpha])[:, None]
    sa = np.array([float(np.sin(a)) for a in alpha])[:, None]
    c_eff = np.array([_age_scalars(spec, float(age), nx, de)[3] for age in ages], dtype=np.float64)[None, :]
    d = float(scale)
    step = abs(float(de))
    ex = (c_eff * np.abs(ca) + d * np.abs(sa)) / step
    ey = (c_eff * np.abs(sa) + d * np.abs(ca)) / step
    a0, b0 = ny // 2, nx // 2
    rx = np.minimum(ex, 4.0 * nx).astype(np.int64) + 2
    ry = np.minimum(ey, 4.0 * ny).astype(np.int64) + 2
    return (int(np.maximum(-ry, -a0).min()), int(np.minimum(ry, ny - 1 - a0).max()),
            int(np.maximum(-rx, -b0).min()), int(np.minimum(rx, nx - 1 - b0).max()))


def records_to_ctypes(records):
    """Flat ctypes ``SbTemplate`` array (what ``sb_sweep`` takes) from a structured array."""
    flat = np.ascontiguousarray(records).reshape(-1)
    arr = (SbTemplate * max(len(flat), 1))()
    if len(flat):
        np.frombuffer(arr, dtype=TEMPLATE_DTYPE, count=len(flat))[:] = flat
    return arr


def template_record(spec, scale, age, angle, nx, ny, de, x, y, angle_id, idx, state=0):
    """``SbTemplate`` for ``Template(scale, age, angle, nx, ny, de)`` (core.py:345)."""
    alpha = -angle                                   # WindowedTemplate.py:151, 489
    ca = float(np.cos(alpha))
    sa = float(np.sin(alpha))
    d = float(scale)
    if spec.kind == KIND_SCARP:
        kt = age
        c = float(scarp_halfwidth(kt))
        k0 = float(2. * kt ** (3 / 2.) * np.sqrt(np.pi))   # WindowedTemplate.py:177
        k1 = float(4. * kt)                                # :178
        c_eff = c
    elif spec.kind == KIND_RICKER:
        f = age
        c = float(nx)                                      # WindowedTemplate.py:491
        k0 = float(np.pi * f)                              # :514
        k1 = 0.0
        c_eff = c
        if abs(k0) > 0:
            c_eff = min(c, np.sqrt(_EXP_UNDERFLOW) / abs(k0) + abs(de))
    else:
        raise ValueError("unknown template kind %r" % (spec.kind,))
    sy_lo, sy_hi, sx_lo, sx_hi = support_box(nx, ny, de, ca, sa, c_eff, d)
    if spec.edge_mask:
        i_lo, i_hi, j_lo, j_hi = window_rectangle(x, y, alpha, c, d)
    else:
        i_lo, i_hi, j_lo, j_hi = 0, ny - 1, 0, nx - 1      # WindowedTemplate.py:494-495
    tscale = packing_scale(spec.kind, k0, k1, c_eff)
    return SbTemplate(ca, sa, c, d, k0, k1, float(spec.sign), tscale, spec.kind, spec.errmode,
                      sy_lo, sy_hi, sx_lo, sx_hi, i_lo, i_hi, j_lo, j_hi,
                      int(angle_id), int(idx), int(state), 0)
