"""varsens_b200 -- B200-native drop-in for the Saltelli pipeline of LoLab-MSM/varsens.

Same public surface as ``varsens/__init__.py:1-4`` (``Varsens, Sample, Objective`` plus the star
export of ``scale``), with the numerical work done by hand-written sm_100a CUDA kernels behind the
C ABI in include/varsens_b200.h.  Extras: registered device functors and the ``vectorized`` marker.
"""
from .saltelli import Varsens, Sample, Objective
from .scale import *          # noqa: F401,F403  (the reference star-exports linear/power/percentage/magnitude)
from . import scale
from .functors import GFunction, Ishigami, RK4Chain, MassActionNetwork, AdaptiveMassActionNetwork, Param, vectorized
from .sobol import sobol_raw, joe_kuo_direction_numbers, quantlib_direction_numbers, read_sobol_initializers
from ._cabi import Context, VarsensError

__all__ = ['scale', 'Varsens', 'Sample', 'Objective']
__version__ = "0.1.0"
