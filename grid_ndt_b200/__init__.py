"""grid_ndt_b200 — B200-native (sm_100a) drop-in for the map-construction path of
daysun/grid_ndt.  The product is libgndt.so (C ABI, include/gndt.h); this package is the
Python host side: the TwoDmap mirror, synthetic clouds, the multi-GPU strip plumbing
(tiles.py) and the overlapped host-cloud pipeline (pipeline.py)."""
from ._abi import COLUMN_DTYPE, SLOPE_DTYPE, VOXEL_DTYPE, Params, default_ndt_params, default_params  # noqa: F401
from ._lib import GndtError, build_library, lib  # noqa: F401
from .builder import Cell, Slope, TwoDmap, morton_string, morton_strings  # noqa: F401
