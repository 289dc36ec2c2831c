# -*- coding: utf-8 -*-
"""wlsqm_b200 -- B200-native drop-in for the hot path of wlsqm (batched local polynomial WLS fits).

``import wlsqm_b200 as wlsqm`` gives the reference's flat namespace (``wlsqm/__init__.py:22-28``):
the ``defs`` constants, the 18 ``fit_*`` functions, ``interpolate_fit`` / ``lambdify_fit``,
``number_of_dofs`` and ``ExpertSolver`` -- implemented as hand-written sm_100a CUDA kernels behind the
C ABI of ``include/wlsqm_b200.h``.  There is no CPU fallback.
"""
__version__ = "0.1.0"

from .fitter.defs import *      # noqa: F401,F403
from .fitter.simple import *    # noqa: F401,F403
from .fitter.interp import *    # noqa: F401,F403
from .fitter.expert import *    # noqa: F401,F403
from ._lib import pinned_empty, pinned_free, pool_stats, pool_trim, LIB_PATH  # noqa: F401
from .neighbors import PointGrid, knn_hoods, ball_hoods, gather  # noqa: F401  (extension: device-side neighbour search)
from . import fitter, utils     # noqa: F401  (the reference exposes its subpackages as attributes)
from .fitter import impl, infra, polyeval  # noqa: F401  (module layout of the reference; see their docstrings)
from .utils import ptrwrap      # noqa: F401
from .utils import lapackdrivers  # noqa: F401
