"""mvsim-b200: B200-native (sm_100a CUDA) per-view acquisition pipeline of multiview-simulation.

Importable as `mvsim_b200` (the directory name carries the reference's hyphen; mvsim_b200.py at the
repository root aliases it).  Everything computes through libmvsim.so; see include/mvsim.h.
"""
from . import tiff                                     # noqa: F401
from ._lib import LIB_PATH, MvsimError, ViewParams     # noqa: F401
from .api import (Context, DeviceVolume, JavaRandom, PinnedBuffer, SimulateBeads, SimulateMultiViewDataset, Tools,   # noqa: F401
                  default_context, make_view_params)
from .drivers import SimulateTileStitching, default_psf, open_psf, run_main, simulate_dataset   # noqa: F401
from .distributed import Group                         # noqa: F401
from .sharding import views_for_rank                   # noqa: F401
from .slab import SlabConvolution, SlabView            # noqa: F401
