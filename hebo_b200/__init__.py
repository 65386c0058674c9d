"""hebo_b200 -- B200-native exact-GP fit + batched MACE acquisition behind HEBO's plugin surface."""
from . import _lib  # noqa: F401
from .gp import GP, B200GP, MultiTaskModel, register  # noqa: F401
from .acq import MACE, FusedMACE, GeneralAcq, Mean, Sigma, LCB  # noqa: F401
from .general import GeneralBO  # noqa: F401

__all__ = ["GP", "B200GP", "MultiTaskModel", "MACE", "FusedMACE", "GeneralAcq", "GeneralBO", "Mean", "Sigma", "LCB", "register"]
