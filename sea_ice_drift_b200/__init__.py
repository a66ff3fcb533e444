"""B200-native pattern matching (MCC) for sea-ice drift: a drop-in for the hot path
of nansencenter/sea_ice_drift (``pattern_matching`` / ``rotate_and_match`` /
``SeaIceDrift.get_drift_PM``).  Importing this package does not touch CUDA."""
from .pmlib import (get_hessian, get_template, match_template, rotate_and_match, use_mcc, use_mcc_mp,
                    use_mcc_batch, prepare_first_guess, get_distance_to_nearest_keypoint,
                    get_initial_rotation, pattern_matching, coarse_tracking)
from .lib import interpolation_poly, interpolation_near
from .seaicedrift import SeaIceDrift
from . import ftlib
from . import libdefor

__version__ = "0.1.0"
__all__ = ['get_hessian', 'get_template', 'match_template', 'rotate_and_match', 'use_mcc', 'use_mcc_mp',
           'use_mcc_batch', 'prepare_first_guess', 'get_distance_to_nearest_keypoint',
           'get_initial_rotation', 'pattern_matching', 'coarse_tracking', 'interpolation_poly', 'interpolation_near',
           'SeaIceDrift']
