"""smmregrid_b200 -- B200-native weight application for smmregrid-style regridding.

Public names mirror ``smmregrid/__init__.py`` for the part of the API on the hot path.
"""
from .packing import CFPacking
from .regrid import Regridder, regrid
from .util import detect_nan_variation_dims
from .weights import (CdoWeights, WeightsMatrix, check_mask, compute_weights_matrix,
                      compute_weights_matrix3d, enable_operator_cache, mask_tensordot, mask_weights)

__version__ = "0.2.0"

__all__ = [
    "Regridder", "regrid", "CFPacking", "CdoWeights", "WeightsMatrix", "compute_weights_matrix",
    "compute_weights_matrix3d", "mask_tensordot", "mask_weights", "check_mask", "enable_operator_cache",
    "detect_nan_variation_dims",
]
