"""pycwt_b200 -- B200-native continuous wavelet transform engine with the call surface
of regeirk/pycwt (``import pycwt_b200 as pycwt``).

Public functions keep the reference signatures: cwt, icwt, significance, xwt, wct,
wct_significance, and the mother wavelets Morlet, Paul, DOG, MexicanHat.  The array math
runs in hand-written sm_100a CUDA kernels behind a C-ABI shared library
(include/cwt_b200.h, loaded with ctypes; no PyTorch).  See DESIGN.md.
"""
from . import helpers, mothers, wavelet  # noqa: F401  (reachable as attributes, like pycwt's)
from .wavelet import *  # noqa: F401,F403
from ._engine import Engine, EngineError, default_engine, device_count  # noqa: F401
from .resident import cwt_resident, ResidentTransform  # noqa: F401  (B200 extension, SURVEY 8f)
from .batch import cwt_batch, BatchProducts  # noqa: F401  (B200 extension: per-channel products of a batch)

__all__ = ['cwt', 'icwt', 'significance', 'xwt', 'wct', 'wct_significance',
           'mothers', 'Morlet', 'Paul', 'DOG', 'MexicanHat']
__version__ = '0.3.0a22+b200.1'
