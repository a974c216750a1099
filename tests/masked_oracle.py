"""Float64 restatement of the nodata-masked fit (``sb_plan_set_nodata(SB_NODATA_MASK)``,
DESIGN.md section 11) on the conventions of ``oracle.scarplet_oracle.match_template``
(``fft2`` / ``fftshift``, template centred at (ny // 2, nx // 2)).  Test infrastructure only.

``V(p)`` is 1 where the second differences at ``p`` (dem.py:88-99) read only finite cells,
``U = 1 - V``; ``curv_m = V * curv``.  Per template (``M = t != 0``, ``n = sum(M)``,
``ts = sum(t**2)``):

    xcorr = t (*) curv_m      T3 = M (*) curv_m**2      D_t = t**2 (*) U      D_m = M (*) U
    n_valid = n - rint(D_m)   ts_m = ts - D_t   (ts where rint(D_m) == 0)

and the fit of core.py:360-367 with ``ts_m`` and ``n_valid`` in place of ``ts`` and ``n``.  A
pixel is a candidate where the reference's masks allow it, ``n_valid >= ceil(min_coverage * n)``
and its own DEM cell is finite.
"""
import math

import numpy as np

from oracle import scarplet_oracle as O


def valid_cells(z):
    """V: the curvature at a pixel depends on finite DEM cells only (dem.py:88-99: dxx reads the
    row neighbours, dyy the column neighbours, dxy the left, upper and upper-left cells)."""
    f = np.isfinite(np.asarray(z, dtype=np.float64))
    v = f.copy()
    v[:, 1:-1] &= f[:, :-2] & f[:, 2:]                       # dxx, dem.py:95-97
    v[1:-1, :] &= f[:-2, :] & f[2:, :]                       # dyy, dem.py:99-101
    v[1:, 1:] &= f[1:, :-1] & f[:-1, 1:] & f[:-1, :-1]       # dxy, dem.py:88-93
    return v


def match_template_masked(z, dx, dy, kind, scale, age, angle, min_coverage=1.0):
    """Masked counterpart of ``O.match_template``: ``(amp, age, angle, snr)`` with 0 in amp and snr
    wherever the template is not a candidate."""
    fft2, ifft2, fftshift = np.fft.fft2, np.fft.ifft2, np.fft.fftshift
    z = np.asarray(z, dtype=np.float64)
    ny, nx = z.shape
    v = valid_cells(z)
    u = (~v).astype(np.float64)
    curv = O.directional_laplacian(np.where(np.isfinite(z), z, 0.0), dx, dy, angle)
    curv = np.where(v, curv, 0.0)
    t = O.template_array(kind, scale, age, angle, nx, ny, dx)
    M = t != 0
    n = int(M.sum())
    ts = np.sum(t ** 2)

    def conv(a, b):
        return np.real(fftshift(ifft2(fft2(a) * fft2(b))))

    xcorr = conv(t, curv)
    T3 = conv(M, curv ** 2)
    D_t = conv(t ** 2, u)
    miss = np.rint(conv(M, u)).astype(np.int64)
    n_valid = n - miss                                       # exact integers
    ts_m = np.where(miss == 0, ts, ts - D_t)
    with np.errstate(divide='ignore', invalid='ignore'):    # ts_m = 0 where U covers the whole template
        amp = xcorr / ts_m                                   # core.py:360
        T1 = ts_m * amp ** 2                                 # core.py:362
        error = (1 / (n_valid + O.EPS)) * (T1 - 2 * amp * xcorr + T3) + O.EPS   # core.py:366
        snr = np.abs(T1 / error)                             # core.py:367

    cand = (n_valid >= math.ceil(min_coverage * n)) & np.isfinite(z)
    em = O.err_mask(kind, angle, nx, ny, dx)                 # core.py:369-371
    if em is not None:
        snr[em] = 0
    c, d = O.template_constants(kind, scale, age, nx)
    cand &= ~O.window_limits(kind, nx, ny, dx, -angle, c, d)   # core.py:373-375
    amp = np.where(cand, amp, 0.0)
    snr = np.where(cand, snr, 0.0)
    return amp, age, angle, snr


def search_masked(z, dx, dy, kind, scale, ages, angles, min_coverage=1.0):
    """Age-major sweep of ``match_template_masked`` folded with ``compare`` -> (4, ny, nx)."""
    ny, nx = np.shape(z)
    return np.stack(O.compare((match_template_masked(z, dx, dy, kind, scale, age, a, min_coverage)
                               for age in ages for a in angles), ny, nx))
