"""ctypes binding of the C ABI in ``include/scarplet_b200.h``.

The product path has no CPU fallback: ``load()`` opens the CUDA library built
in-tree by ``__graft_entry__.build()`` (``scarplet_b200/libscarplet_b200.so``) and
raises if it is missing; creating a plan raises if no CUDA device is present.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, byref, c_char_p, c_double, c_float, c_int,
                    c_int32, c_long, c_uint, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libscarplet_b200.so"


class SbAngle(Structure):
    _fields_ = [("cos_a", c_double), ("sin_a", c_double),
                ("cos2_a", c_double), ("sin2_a", c_double)]


class SbTemplate(Structure):
    _fields_ = [("cos_t", c_double), ("sin_t", c_double),
                ("c", c_double), ("d", c_double),
                ("k0", c_double), ("k1", c_double), ("sign", c_double),
                ("tscale", c_double),
                ("kind", c_int32), ("errmode", c_int32),
                ("sy_lo", c_int32), ("sy_hi", c_int32),
                ("sx_lo", c_int32), ("sx_hi", c_int32),
                ("i_lo", c_int32), ("i_hi", c_int32),
                ("j_lo", c_int32), ("j_hi", c_int32),
                ("angle_id", c_int32), ("idx", c_int32),
                ("state", c_int32), ("reserved", c_int32)]


class SbError(RuntimeError):
    pass


_lib = None


def _declare(lib):
    P = c_void_p
    dp = POINTER(c_double)
    lib.sb_last_error.restype = c_char_p
    lib.sb_build_info.restype = c_char_p
    lib.sb_plan_create.argtypes = [POINTER(P), c_int, c_int, c_double, c_double, c_double,
                                   c_int, c_void_p, c_uint]
    lib.sb_plan_destroy.argtypes = [P]
    lib.sb_plan_set_option.argtypes = [P, c_char_p, c_long]
    lib.sb_plan_set_nodata.argtypes = [P, c_int, c_double]
    lib.sb_plan_launch_count.argtypes = [P]
    lib.sb_plan_launch_count.restype = c_long
    lib.sb_plan_device_bytes.argtypes = [P]
    lib.sb_plan_device_bytes.restype = c_long
    lib.sb_plan_last_fft_area.argtypes = [P]
    lib.sb_plan_last_fft_area.restype = c_double
    lib.sb_plan_stream.argtypes = [P]
    lib.sb_plan_stream.restype = c_void_p
    lib.sb_plan_set_slab.argtypes = [P, c_int, c_int, c_int]
    lib.sb_plan_dem_rows.argtypes = [P, POINTER(c_int), POINTER(c_int)]
    lib.sb_plan_curv_stats.argtypes = [P, dp, dp]
    lib.sb_plan_set_curv_stats.argtypes = [P, c_double, c_double]
    lib.sb_finalize_ex.argtypes = [P, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int]
    lib.sb_age_range.argtypes = [P, c_int, c_int, c_int, c_double, c_void_p, c_void_p, c_int, c_void_p, c_int]
    lib.sb_region_sweep.argtypes = [P, POINTER(SbAngle), c_int, POINTER(SbTemplate), c_int, POINTER(c_int32), c_double,
                                    c_void_p, c_void_p, c_int, c_int]
    lib.sb_region_finalize.argtypes = [P, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int,
                                       c_int, c_void_p, c_int]
    lib.sb_best_state_ex.argtypes = [P, c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p)]
    lib.sb_best_merge.argtypes = [P, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]
    lib.sb_region_planes.argtypes = [P, POINTER(c_void_p), POINTER(c_int)]
    lib.sb_secondary_sweep.argtypes = [P, POINTER(SbAngle), c_int, POINTER(SbTemplate), c_int, POINTER(c_int32),
                                       c_void_p, c_int, c_int, c_int, c_int]
    lib.sb_region_merge.argtypes = [P, c_int, c_int, c_int, c_void_p]
    lib.sb_peak_sweep.argtypes = [P, POINTER(SbAngle), c_int, POINTER(SbTemplate), c_int, POINTER(c_int32), c_void_p,
                                  c_void_p, c_int, c_int, c_int, c_int]
    lib.sb_peak_finalize.argtypes = [P, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                     c_double, c_void_p]
    lib.sb_peak_planes.argtypes = [P, POINTER(c_void_p)]
    lib.sb_curvature_noise_moments.argtypes = [P, c_double, c_double, dp]
    lib.sb_fill_nodata.argtypes = [P, c_void_p, c_double, POINTER(c_long)]
    lib.sb_plan_last_geometry.argtypes = [P, POINTER(c_int)]
    lib.sb_plan_profile.argtypes = [P, POINTER(c_double), POINTER(c_long), c_int]
    lib.sb_set_dem_host.argtypes = [P, c_void_p]
    lib.sb_set_dem_dev.argtypes = [P, c_void_p]
    lib.sb_set_axes_host.argtypes = [P, c_void_p, c_void_p]
    lib.sb_directional_laplacian.argtypes = [P, POINTER(SbAngle), c_void_p, c_int]
    lib.sb_render_template.argtypes = [P, POINTER(SbTemplate), c_void_p, c_int]
    lib.sb_match_template.argtypes = [P, POINTER(SbAngle), POINTER(SbTemplate), c_void_p,
                                      c_void_p, c_int]
    lib.sb_best_reset.argtypes = [P]
    lib.sb_sweep.argtypes = [P, POINTER(SbAngle), c_int, POINTER(SbTemplate), c_int]
    lib.sb_sweep_ex.argtypes = [P, POINTER(SbAngle), c_int, POINTER(SbTemplate), c_int, POINTER(c_int32)]
    lib.sb_sweep_ex.restype = c_int
    lib.sb_finalize.argtypes = [P, c_void_p, c_void_p, c_int, c_void_p, c_int]
    lib.sb_best_state.argtypes = [P, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p)]
    lib.sb_best_pack.argtypes = [P, c_void_p]
    lib.sb_match_template_raster.argtypes = [P, POINTER(SbAngle), c_void_p, c_int, c_int, c_int, c_int,
                                             c_double, c_void_p, c_void_p, c_int]
    lib.sb_best_select.argtypes = [P, c_void_p, c_void_p]
    lib.sb_best_unpack.argtypes = [P, c_void_p, c_void_p]
    lib.sb_compare_host.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_double, c_double]
    lib.sb_debug_fft.argtypes = [P, c_int, c_int, c_void_p, c_void_p, c_int]
    lib.sb_debug_fft_bench.argtypes = [P, c_int, c_int, c_int, c_int, POINTER(c_float)]
    lib.sb_debug_fft_bench.restype = c_int
    lib.sb_fit_surface.argtypes = [P, POINTER(SbAngle), c_int, POINTER(SbTemplate), c_int, c_void_p, c_void_p,
                                   c_int, c_void_p, c_void_p, c_int]
    lib.sb_sync.argtypes = [P]
    for name in ("sb_plan_create", "sb_plan_destroy", "sb_plan_set_option",
                 "sb_plan_last_geometry", "sb_plan_profile", "sb_set_dem_host", "sb_set_dem_dev",
                 "sb_set_axes_host", "sb_directional_laplacian", "sb_render_template",
                 "sb_match_template", "sb_match_template_raster", "sb_best_reset", "sb_sweep", "sb_finalize",
                 "sb_best_state", "sb_best_pack", "sb_best_select", "sb_best_unpack",
                 "sb_compare_host", "sb_debug_fft", "sb_sync", "sb_plan_set_slab", "sb_plan_dem_rows",
                 "sb_plan_curv_stats", "sb_plan_set_curv_stats", "sb_finalize_ex", "sb_best_state_ex",
                 "sb_best_merge", "sb_curvature_noise_moments", "sb_fill_nodata", "sb_plan_set_nodata",
                 "sb_fit_surface", "sb_age_range", "sb_region_sweep", "sb_region_finalize", "sb_region_planes",
                 "sb_region_merge", "sb_secondary_sweep", "sb_peak_sweep", "sb_peak_finalize", "sb_peak_planes"):
        getattr(lib, name).restype = c_int
    return lib


EXPORTED = ("sb_last_error", "sb_build_info", "sb_plan_create", "sb_plan_destroy",
            "sb_plan_set_option", "sb_plan_launch_count", "sb_plan_last_geometry", "sb_plan_profile",
            "sb_set_dem_host", "sb_set_dem_dev", "sb_set_axes_host",
            "sb_directional_laplacian", "sb_render_template", "sb_match_template",
            "sb_match_template_raster", "sb_best_reset", "sb_sweep", "sb_finalize", "sb_best_state", "sb_best_pack",
            "sb_best_select", "sb_best_unpack", "sb_compare_host",
            "sb_debug_fft", "sb_sync", "sb_plan_set_slab", "sb_plan_dem_rows", "sb_plan_curv_stats",
            "sb_plan_set_curv_stats", "sb_plan_stream", "sb_plan_device_bytes", "sb_plan_last_fft_area",
            "sb_finalize_ex", "sb_best_state_ex", "sb_best_merge", "sb_curvature_noise_moments",
            "sb_fill_nodata", "sb_debug_fft_bench", "sb_sweep_ex", "sb_plan_set_nodata", "sb_fit_surface",
            "sb_age_range", "sb_region_sweep", "sb_region_finalize", "sb_region_planes", "sb_region_merge",
            "sb_secondary_sweep", "sb_peak_sweep", "sb_peak_finalize", "sb_peak_planes")


def library_path():
    return os.path.join(_HERE, LIB_NAME)


def open_library(path):
    """dlopen a build of the C ABI and declare its prototypes."""
    return _declare(ctypes.CDLL(path))


def load():
    """The CUDA library; raises if it has not been built."""
    global _lib
    if _lib is None:
        path = library_path()
        if not os.path.exists(path):
            raise SbError(
                "%s not found: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (nvcc, sm_100a). scarplet_b200 has no CPU fallback." % path)
        _lib = open_library(path)
    return _lib


def _use_library(lib):
    """Test hook (tests/emu): route the host layer to another build of the same ABI."""
    global _lib
    prev = _lib
    _lib = lib
    return prev


def check(lib, status):
    if status != 0:
        raise SbError(lib.sb_last_error().decode("utf-8", "replace"))
