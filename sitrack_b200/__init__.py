"""sitrack_b200 -- B200-native drop-in for the buoy-advection hot path of
stephanieleroux/sitrack.  Same flat namespace as the reference package
(`import sitrack_b200 as sit`; reference sitrack/__init__.py:6-13) plus the
batched engine (`sit.TrackEngine`).  Importing never touches the GPU; every
compute call needs libsitrack_b200.so and a CUDA device (no CPU fallback).
"""
from .util import *          # noqa: F401,F403
from .ncio import *          # noqa: F401,F403
from .tracking import *      # noqa: F401,F403
from .locate import *        # noqa: F401,F403
from .deform import *        # noqa: F401,F403
from .deform_scales import *  # noqa: F401,F403
from .deform_grid import *    # noqa: F401,F403
from .dispersion import *     # noqa: F401,F403
from . import config                      # noqa: F401
from .engine import TrackEngine          # noqa: F401
from ._lib import SitrackCudaError       # noqa: F401

__version__ = "0.1.0"
