"""scarplet_b200 — B200-native implementation of scarplet's template-matching hot path.

Drop-in for the reference's ``import scarplet as sl`` on that path::

    import scarplet_b200 as sl
    from scarplet_b200.WindowedTemplate import Scarp
    res = sl.match(data, Scarp, scale=100, age=10, ang_min=-np.pi / 2, ang_max=np.pi / 2)
"""
from .core import (age_range, calculate_best_fit_parameters,  # noqa: F401
                   calculate_best_fit_parameters_serial, compare, fit_peak, fit_region, fit_surface, match,
                   match_ages, match_scales, match_template, release, secondary_fit)
from .dem import DEMGrid  # noqa: F401
from .engine import configure  # noqa: F401
from .geotiff import write_results as save_results  # noqa: F401
from . import WindowedTemplate  # noqa: F401

__version__ = "0.1.0"
