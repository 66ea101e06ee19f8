"""B200-native stereo block search — drop-in for the matching path of
6dwavenminer/Unsynchronized_Stereo_Vision_Proj325 (Match / GenerateMatchingList /
ResolveMatchList / DistanceCalculator). Host code is C++ + a C-ABI shared
library of hand-written sm_100a CUDA kernels; this Python package is the thin
ctypes mirror used by the tests and the bench. There is no CPU fallback.
"""
from . import _abi  # noqa: F401
from ._abi import (COST_CENSUS, COST_NCC, COST_SAD, COST_SSD, COST_ZNCC, DIST_NONE, DIST_PINHOLE, DIST_POWERLAW,  # noqa: F401
                   LEFT_CAM, MATCH_DTYPE, NO_DISPARITY, NO_MATCH, RIGHT_CAM, make_params)

__all__ = ["_abi", "make_params", "MATCH_DTYPE"]
