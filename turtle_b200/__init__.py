"""turtle-b200: the DEM ray-stepping hot path of niess/turtle on B200 (sm_100a).

The product is the C-ABI shared library ``libturtle_b200.so`` (include/turtle.h,
include/turtle_b200.h). This package is its ctypes mirror plus the synthetic
workload generators used by tests/ and bench.py.
"""
from .api import (Map, Plan, Projection, Stack, States, Stepper, TurtleError,  # noqa: F401
                  TRACE_RESULT, HORIZON_RESULT, VOXEL_ENTRY, device_count, dfma_peak, kernel_info, ecef_from_geodetic,
                  ecef_from_geodetic_batch, ecef_from_horizontal,
                  ecef_from_horizontal_batch, ecef_to_geodetic, ecef_to_geodetic_batch,
                  trace_rule, voxel_grid, residency_from_rays)
