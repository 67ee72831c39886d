"""espm_b200 -- B200-native (sm_100a) implementation of espm's SmoothNMF fit loop.

Drop-in for ``espm.estimators.SmoothNMF`` and for the update / bisection / loss operators of
``espm.estimators.updates``, ``espm.estimators.dicotomy`` and ``espm.measures`` that sit on that path.
All arithmetic runs in hand-written CUDA kernels (``espm_b200/csrc``) behind the C ABI declared in
``include/espm_b200.h``; there is no CPU fallback.
"""
from . import config  # noqa: F401
from .estimators import (AbundanceUncertainty, FitStatistics, PhaseUncertainty, ResidualComponents,  # noqa: F401
                         SmoothNMF)
from . import ops  # noqa: F401

__all__ = ["SmoothNMF", "FitStatistics", "AbundanceUncertainty", "PhaseUncertainty", "ResidualComponents", "ops",
           "config"]
__version__ = "0.1.0"
