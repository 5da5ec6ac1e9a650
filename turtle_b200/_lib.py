"""ctypes binding of libturtle_b200.so (the C ABI of include/turtle.h + turtle_b200.h).

The library is built in-tree by ``turtle_b200.build`` (nvcc, sm_100a). There is no
Python or CPU fallback for the batched path: if the shared library is missing the
import fails loudly, and the batch calls themselves fail without a CUDA device.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# (TURTLE_B200_LIB: development hook to A/B another build of the same library)
LIB_PATH = os.environ.get("TURTLE_B200_LIB") or os.path.join(HERE, "libturtle_b200.so")

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class MapInfo(C.Structure):
    """struct turtle_map_info (ref: include/turtle.h:93-106)."""
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("x", C.c_double * 2),
                ("y", C.c_double * 2), ("z", C.c_double * 2),
                ("encoding", C.c_char_p)]


class TraceRule(C.Structure):
    """struct turtle_trace_rule (include/turtle_b200.h)."""
    _fields_ = [("altitude_min", C.c_double), ("altitude_max", C.c_double),
                ("length_max", C.c_double), ("max_steps", C.c_int32),
                ("reserved", C.c_int32)]


class Residency(C.Structure):
    """struct turtle_residency (include/turtle_b200.h)."""
    _fields_ = [("latitude_min", C.c_double), ("latitude_max", C.c_double),
                ("longitude_min", C.c_double), ("longitude_max", C.c_double),
                ("memory_limit", C.c_size_t)]


class ResidencyReport(C.Structure):
    """struct turtle_residency_report (include/turtle_b200.h)."""
    _fields_ = [("tiles_resident", C.c_uint64), ("tiles_skipped", C.c_uint64),
                ("tiles_ingested", C.c_uint64), ("bytes", C.c_uint64),
                ("read_ms", C.c_double), ("upload_ms", C.c_double)]


class TraceFields(C.Structure):
    """struct turtle_trace_fields (include/turtle_b200.h): one array per column, NULL = not
    wanted."""
    _fields_ = [("length", C.c_void_p * 4), ("total", C.c_void_p), ("altitude", C.c_void_p),
                ("position", C.c_void_p), ("n_steps", C.c_void_p), ("status", C.c_void_p),
                ("index", C.c_void_p), ("medium_hash", C.c_void_p), ("n_changes", C.c_void_p)]


class Fan(C.Structure):
    """struct turtle_fan (include/turtle_b200.h)."""
    _fields_ = [("latitude", C.c_double), ("longitude", C.c_double),
                ("position", C.c_double * 3), ("n_azimuth", C.c_size_t),
                ("n_elevation", C.c_size_t), ("azimuth", C.c_void_p),
                ("elevation", C.c_void_p), ("bundle", C.c_size_t)]


class Fans(C.Structure):
    """struct turtle_fans (include/turtle_b200.h): one angle grid, n_station stations."""
    _fields_ = [("n_station", C.c_size_t), ("latitude", C.c_void_p), ("longitude", C.c_void_p),
                ("position", C.c_void_p), ("n_azimuth", C.c_size_t),
                ("n_elevation", C.c_size_t), ("azimuth", C.c_void_p),
                ("elevation", C.c_void_p), ("bundle", C.c_size_t)]


class VoxelGrid(C.Structure):
    """struct turtle_voxel_grid (include/turtle_b200.h): cells in the East / North / Up frame
    of a point."""
    _fields_ = [("latitude", C.c_double), ("longitude", C.c_double), ("height", C.c_double),
                ("corner", C.c_double * 3), ("size", C.c_double * 3), ("n", C.c_int32 * 3),
                ("media", C.c_uint32)]


class VoxelEntry(C.Structure):
    """struct turtle_voxel_entry (include/turtle_b200.h)."""
    _fields_ = [("length", C.c_double), ("voxel", C.c_int32), ("medium", C.c_int32)]


class VoxelOpacity(C.Structure):
    """struct turtle_voxel_opacity (include/turtle_b200.h): the arrays of L @ rho and L.T @ w."""
    _fields_ = [("density", C.c_void_p), ("opacity", C.c_void_p), ("outside", C.c_void_p),
                ("weight", C.c_void_p), ("gradient", C.c_void_p)]


class PlanCounters(C.Structure):
    """struct turtle_plan_counters (include/turtle_b200.h)."""
    _fields_ = [("rays", C.c_uint64), ("steps", C.c_uint64),
                ("samples", C.c_uint64), ("launches", C.c_uint64),
                ("kernel_ms", C.c_double), ("rebuilds", C.c_uint64),
                ("window_hits", C.c_uint64)]


ERROR_HANDLER = C.CFUNCTYPE(None, C.c_int, C.c_void_p, C.c_char_p)

# name -> (restype, argtypes). Every symbol declared in include/*.h is listed: the
# CPU test-suite checks that the library exports all of them.
_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_D = C.c_double
_I = C.c_int
_N = C.c_size_t
SIGNATURES = {
    # turtle.h -- error handling
    "turtle_error_function": (C.c_char_p, [_P]),
    "turtle_error_handler_get": (_P, []),
    "turtle_error_handler_set": (None, [_P]),
    # projections
    "turtle_projection_create": (_I, [_PP, C.c_char_p]),
    "turtle_projection_destroy": (None, [_PP]),
    "turtle_projection_configure": (_I, [_P, C.c_char_p]),
    "turtle_projection_name": (C.c_char_p, [_P]),
    "turtle_projection_project": (_I, [_P, _D, _D, c_double_p, c_double_p]),
    "turtle_projection_unproject": (_I, [_P, _D, _D, c_double_p, c_double_p]),
    # maps
    "turtle_map_create": (_I, [_PP, C.POINTER(MapInfo), C.c_char_p]),
    "turtle_map_destroy": (None, [_PP]),
    "turtle_map_load": (_I, [_PP, C.c_char_p]),
    "turtle_map_dump": (_I, [_P, C.c_char_p]),
    "turtle_map_fill": (_I, [_P, _I, _I, _D]),
    "turtle_map_node": (_I, [_P, _I, _I, c_double_p, c_double_p, c_double_p]),
    "turtle_map_elevation": (_I, [_P, _D, _D, c_double_p, c_int_p]),
    "turtle_map_gradient": (_I, [_P, _D, _D, c_double_p, c_double_p, c_int_p]),
    "turtle_map_projection": (_P, [_P]),
    "turtle_map_meta": (None, [_P, C.POINTER(MapInfo), C.POINTER(C.c_char_p)]),
    # ecef
    "turtle_ecef_from_geodetic": (None, [_D, _D, _D, c_double_p]),
    "turtle_ecef_to_geodetic": (None, [c_double_p, c_double_p, c_double_p, c_double_p]),
    "turtle_ecef_from_horizontal": (None, [_D, _D, _D, _D, c_double_p]),
    "turtle_ecef_to_horizontal": (None, [_D, _D, c_double_p, c_double_p, c_double_p]),
    # stacks / clients
    "turtle_stack_create": (_I, [_PP, C.c_char_p, _I, _P, _P]),
    "turtle_stack_destroy": (None, [_PP]),
    "turtle_stack_clear": (_I, [_P]),
    "turtle_stack_load": (_I, [_P]),
    "turtle_stack_elevation": (_I, [_P, _D, _D, c_double_p, c_int_p]),
    "turtle_stack_gradient": (_I, [_P, _D, _D, c_double_p, c_double_p, c_int_p]),
    "turtle_client_create": (_I, [_PP, _P]),
    "turtle_client_destroy": (_I, [_PP]),
    "turtle_client_clear": (_I, [_P]),
    "turtle_client_elevation": (_I, [_P, _D, _D, c_double_p, c_int_p]),
    # stepper
    "turtle_stepper_create": (_I, [_PP]),
    "turtle_stepper_destroy": (_I, [_PP]),
    "turtle_stepper_geoid_set": (None, [_P, _P]),
    "turtle_stepper_geoid_get": (_P, [_P]),
    "turtle_stepper_reset": (None, [_P]),
    "turtle_stepper_range_set": (None, [_P, _D]),
    "turtle_stepper_range_get": (_D, [_P]),
    "turtle_stepper_slope_get": (_D, [_P]),
    "turtle_stepper_slope_set": (None, [_P, _D]),
    "turtle_stepper_resolution_get": (_D, [_P]),
    "turtle_stepper_resolution_set": (None, [_P, _D]),
    "turtle_stepper_add_layer": (_I, [_P]),
    "turtle_stepper_add_stack": (_I, [_P, _P, _D]),
    "turtle_stepper_add_map": (_I, [_P, _P, _D]),
    "turtle_stepper_add_flat": (_I, [_P, _D]),
    "turtle_stepper_step": (_I, [_P, c_double_p, c_double_p, c_double_p, c_double_p,
                                 c_double_p, c_double_p, c_double_p, c_int_p]),
    "turtle_stepper_position": (_I, [_P, _D, _D, _D, _I, c_double_p, c_int_p]),
    # turtle_b200.h -- plans
    "turtle_stepper_freeze": (_I, [_P, _I, _PP]),
    "turtle_plan_destroy": (None, [_PP]),
    "turtle_plan_device": (_I, [_P]),
    "turtle_plan_bytes": (_N, [_P]),
    "turtle_plan_counters_get": (None, [_P, C.POINTER(PlanCounters)]),
    "turtle_plan_counters_sync": (None, [_P]),
    "turtle_plan_launch_set": (None, [_P, _I, _I]),
    "turtle_plan_schedule_set": (None, [_P, _I]),
    "turtle_plan_specialise_set": (None, [_P, _I]),
    "turtle_plan_pipeline_set": (None, [_P, _I]),
    "turtle_plan_gather_set": (_I, [_P, _I, _D, _D]),
    "turtle_stack_tiles_loaded": (_I, [_P]),
    "turtle_map_resample": (_I, [_P, _P, _I, C.POINTER(C.c_size_t)]),
    "turtle_stepper_freeze_region": (_I, [_P, _I, C.POINTER(Residency), _PP]),
    "turtle_plan_residency_get": (None, [_P, C.POINTER(ResidencyReport)]),
    "turtle_residency_from_rays": (_I, [_N, _P, _P, C.POINTER(TraceRule), C.c_double,
                                        C.c_double, C.POINTER(Residency)]),
    # peer memory
    "turtle_b200_peer_alloc": (_I, [_N, _PP]),
    "turtle_b200_peer_free": (_I, [_P]),
    "turtle_b200_peer_export": (_I, [_P, _P]),
    "turtle_b200_peer_open": (_I, [_P, _PP]),
    "turtle_b200_peer_close": (_I, [_P]),
    # rays
    "turtle_stepper_trace_batch": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule), _P]),
    "turtle_stepper_trace_batch_device": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule), _P, _P]),
    "turtle_stepper_trace_fan": (_I, [_P, C.POINTER(Fan), C.POINTER(TraceRule), _P,
                                      C.POINTER(TraceFields)]),
    "turtle_stepper_trace_fan_device": (_I, [_P, C.POINTER(Fan), C.POINTER(TraceRule), _P,
                                             C.POINTER(TraceFields), _P]),
    "turtle_stepper_trace_fans": (_I, [_P, C.POINTER(Fans), C.POINTER(TraceRule), _P,
                                       C.POINTER(TraceFields)]),
    "turtle_stepper_trace_fans_device": (_I, [_P, C.POINTER(Fans), C.POINTER(TraceRule), _P,
                                              C.POINTER(TraceFields), _P]),
    "turtle_stepper_trace_fields": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule),
                                         C.POINTER(TraceFields)]),
    "turtle_stepper_trace_fields_device": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule),
                                                C.POINTER(TraceFields), _P]),
    "turtle_stepper_trace_crossings": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule), _P, _P, _I]),
    "turtle_stepper_trace_crossings_device": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule), _P, _P,
                                                   _I, _P]),
    "turtle_stepper_trace_voxels": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule),
                                         C.POINTER(VoxelGrid), _P, _P, _I, _P]),
    "turtle_stepper_trace_voxels_device": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule),
                                                C.POINTER(VoxelGrid), _P, _P, _I, _P, _P]),
    "turtle_stepper_trace_fans_voxels": (_I, [_P, C.POINTER(Fans), C.POINTER(TraceRule),
                                              C.POINTER(VoxelGrid), _P, _P, _I, _P]),
    "turtle_stepper_trace_fans_voxels_device": (_I, [_P, C.POINTER(Fans), C.POINTER(TraceRule),
                                                     C.POINTER(VoxelGrid), _P, _P, _I, _P, _P]),
    "turtle_stepper_trace_opacity": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule),
                                          C.POINTER(VoxelGrid), C.POINTER(VoxelOpacity), _P]),
    "turtle_stepper_trace_opacity_device": (_I, [_P, _N, _P, _P, C.POINTER(TraceRule),
                                                 C.POINTER(VoxelGrid), C.POINTER(VoxelOpacity),
                                                 _P, _P]),
    "turtle_stepper_trace_fans_opacity": (_I, [_P, C.POINTER(Fans), C.POINTER(TraceRule),
                                               C.POINTER(VoxelGrid), C.POINTER(VoxelOpacity), _P]),
    "turtle_stepper_trace_fans_opacity_device": (_I, [_P, C.POINTER(Fans), C.POINTER(TraceRule),
                                                      C.POINTER(VoxelGrid),
                                                      C.POINTER(VoxelOpacity), _P, _P]),
    "turtle_stepper_horizon": (_I, [_P, _D, _D, _P, _N, _P, _D, _D, _D, C.POINTER(TraceRule), _P]),
    "turtle_stepper_horizon_device": (_I, [_P, _D, _D, _P, _N, _P, _D, _D, _D,
                                           C.POINTER(TraceRule), _P, _P]),
    "turtle_stepper_horizons": (_I, [_P, _N, _P, _P, _P, _N, _P, _D, _D, _D,
                                     C.POINTER(TraceRule), _P]),
    "turtle_stepper_horizons_device": (_I, [_P, _N, _P, _P, _P, _N, _P, _D, _D, _D,
                                            C.POINTER(TraceRule), _P, _P]),
    # particle steps
    "turtle_states_create": (_I, [_P, _N, _PP]),
    "turtle_states_destroy": (None, [_PP]),
    "turtle_states_reset": (_I, [_P]),
    "turtle_states_bytes_per_particle": (_N, [_P]),
    "turtle_stepper_step_batch": (_I, [_P, _P, _N] + [_P] * 8),
    "turtle_stepper_step_batch_device": (_I, [_P, _P, _N] + [_P] * 8 + [_P]),
    "turtle_stepper_walk_batch": (_I, [_P, _P, _N, _I] + [_P] * 8),
    "turtle_stepper_walk_batch_device": (_I, [_P, _P, _N, _I] + [_P] * 8 + [_P]),
    "turtle_stepper_position_batch": (_I, [_P, _N, _P, _P, _P, _I, _P, _P]),
    # frames
    "turtle_ecef_to_geodetic_batch": (_I, [_N, _P, _P, _P, _P]),
    "turtle_ecef_to_geodetic_batch_device": (_I, [_N, _P, _P, _P, _P, _P]),
    "turtle_ecef_from_geodetic_batch": (_I, [_N, _P, _P, _P, _P]),
    "turtle_ecef_from_geodetic_batch_device": (_I, [_N, _P, _P, _P, _P, _P]),
    "turtle_ecef_from_horizontal_batch": (_I, [_N, _P, _P, _P, _P, _P]),
    "turtle_ecef_from_horizontal_batch_device": (_I, [_N, _P, _P, _P, _P, _P, _P]),
    # elevation
    "turtle_map_gather_set": (None, [_P, _I]),
    "turtle_map_elevation_batch": (_I, [_P, _N, _P, _P, _P, _P]),
    "turtle_map_elevation_batch_device": (_I, [_P, _N, _P, _P, _P, _P, _P]),
    "turtle_map_elevation_ecef_batch": (_I, [_P, _N, _P, _P, _P, _P, _P, _P]),
    "turtle_map_elevation_ecef_batch_device": (_I, [_P, _N, _P, _P, _P, _P, _P, _P, _P]),
    "turtle_projection_project_batch": (_I, [_P, _N, _P, _P, _P, _P]),
    "turtle_projection_project_batch_device": (_I, [_P, _N, _P, _P, _P, _P, _P]),
    "turtle_projection_unproject_batch": (_I, [_P, _N, _P, _P, _P, _P]),
    "turtle_projection_unproject_batch_device": (_I, [_P, _N, _P, _P, _P, _P, _P]),
    "turtle_map_gradient_batch": (_I, [_P, _N, _P, _P, _P, _P, _P]),
    "turtle_map_gradient_batch_device": (_I, [_P, _N, _P, _P, _P, _P, _P, _P]),
    "turtle_stack_elevation_batch": (_I, [_P, _I, _N, _P, _P, _P, _P]),
    "turtle_stack_elevation_batch_device": (_I, [_P, _I, _N, _P, _P, _P, _P, _P]),
    "turtle_stack_gradient_batch": (_I, [_P, _I, _N, _P, _P, _P, _P, _P]),
    "turtle_stack_gradient_batch_device": (_I, [_P, _I, _N, _P, _P, _P, _P, _P, _P]),
    "turtle_map_fill_batch": (_I, [_P, _P]),
    "turtle_map_fill_rows": (_I, [_P, _I, _I, _P]),
    # utilities
    "turtle_b200_device_count": (_I, []),
    "turtle_b200_dfma_peak": (_D, [_I]),
    "turtle_b200_version": (C.c_char_p, []),
    "turtle_b200_kernel_info": (_I, [C.c_char_p, c_int_p, c_int_p]),
    "turtle_b200_selftest_division": (C.c_longlong, [_N, C.c_uint64]),
}


def load(path=LIB_PATH):
    """Load the shared library and attach the signatures. Raises if it is absent."""
    if not os.path.exists(path):
        raise ImportError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). turtle_b200 has no Python/CPU fallback." % path)
    lib = C.CDLL(path, mode=getattr(os, "RTLD_LOCAL", 0) | getattr(os, "RTLD_NOW", 2))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


lib = load()
