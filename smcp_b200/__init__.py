"""smcp-b200: B200-native Newton-system hot path of SMCP's chordal interior-point solvers.

Drop-in surface of the reference package (``src/python/__init__.py``): ``SDP``,
``band_SDP``, ``mtxnorm_SDP``, ``rand_SDP``, ``solvers``, ``misc``.
"""
from . import misc, solvers  # noqa: F401
from .base import SDP, band_SDP, mtxnorm_SDP, rand_SDP, maxcut_SDP, mk_rand, completion, completion_sample  # noqa: F401

__version__ = "0.1.0"
