"""
ctypes binding of the C ABI in include/lidar_snow_sim.h (liblss_b200.so, built in-tree by lidar_snow_sim_b200.build).

There is NO CPU fallback: if the shared library is missing or no CUDA device is usable, loading / engine creation
raises.  (oracle/ is test infrastructure and is never imported from here.)
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'liblss_b200.so')

LSS_OK = 0
LSS_ERR_INVALID_ARG = 1
LSS_ERR_CUDA = 2
LSS_ERR_NO_TABLE = 3
LSS_ERR_RANGE_INDEX = 4
LSS_ERR_NEGATIVE_INTENSITY = 5
LSS_ERR_OCCLUDER_OVERFLOW = 6
LSS_ERR_WORKSPACE = 7
LSS_ERR_NO_SENSOR = 8
LSS_ERR_TOO_FEW_GROUND = 9

FLAG_THRESHOLD_FILTER = 0x1
FLAG_CAMERA_FOV = 0x2
FLAG_DEVICE_PREPASS = 0x4
FLAG_ASSUME_SORTED = 0x8
FOG_HARD, FOG_SOFT, FOG_GAIN = 0x1, 0x2, 0x4

# status -> exception type the reference would have raised at the corresponding place (SURVEY.md 8b "Errors")
_EXC = {
    LSS_ERR_INVALID_ARG: ValueError,
    LSS_ERR_CUDA: RuntimeError,
    LSS_ERR_NO_TABLE: FileNotFoundError,         # np.load of a missing particle file, simulation.py:329
    LSS_ERR_RANGE_INDEX: IndexError,             # i[k] beyond the 1230-sample grid, simulation.py:149
    LSS_ERR_NEGATIVE_INTENSITY: AssertionError,  # simulation.py:184
    LSS_ERR_OCCLUDER_OVERFLOW: RuntimeError,
    LSS_ERR_WORKSPACE: RuntimeError,
    LSS_ERR_NO_SENSOR: AssertionError,           # simulation.py:35
    LSS_ERR_TOO_FEW_GROUND: TypeError,           # estimate_laser_parameters -> None, simulation.py:457-462
}

# every symbol include/lidar_snow_sim.h declares: (name, restype, argtypes)
_c = ctypes
_P = ctypes.c_void_p
SIGNATURES = [
    ('lss_create', _c.c_int, [_c.c_int, _c.POINTER(_P)]),
    ('lss_destroy', None, [_P]),
    ('lss_status_string', _c.c_char_p, [_c.c_int]),
    ('lss_last_error', _c.c_char_p, [_P]),
    ('lss_version', _c.c_int, []),
    ('lss_set_sensor', _c.c_int, [_P, _c.c_int, _P, _P, _P, _P]),
    ('lss_set_camera', _c.c_int, [_P, _P, _P, _P, _c.c_int, _c.c_int]),
    ('lss_upload_particles', _c.c_int, [_P, _c.c_int, _P, _P, _c.c_double, _c.c_int, _P, _c.POINTER(_c.c_int)]),
    ('lss_upload_particles_device', _c.c_int, [_P, _c.c_int, _P, _P, _c.c_double, _c.c_int, _P,
                                               _c.POINTER(_c.c_int)]),
    ('lss_free_particles', _c.c_int, [_P, _c.c_int]),
    ('lss_table_info', _c.c_int, [_P, _c.c_int, _c.POINTER(_c.c_int64), _c.POINTER(_c.c_int64),
                                  _c.POINTER(_c.c_int64)]),
    ('lss_snowfall_batch', _c.c_int, [_P, _c.c_int, _P, _P, _c.c_int, _P, _c.c_double, _P, _P, _P, _P, _c.c_double,
                                      _c.c_uint32, _P, _P, _P, _P, _P, _P, _P, _c.c_int64, _P]),
    ('lss_snowfall_workspace_bytes', _c.c_int64, [_c.c_int64, _c.c_int]),
    ('lss_host_pipe_trace', _c.c_int, [_P, _P, _c.c_int]),
    ('lss_snowfall_batch_host', _c.c_int, [_P, _c.c_int, _P, _P, _c.c_int, _P, _c.c_double, _P, _c.c_double, _c.c_uint32,
                                           _c.c_int, _P, _P, _P]),
    ('lss_snowfall_batch_host_submit', _c.c_int, [_P, _c.c_int, _P, _P, _c.c_int, _P, _c.c_double, _P, _c.c_double,
                                                  _c.c_uint32, _c.c_int, _P, _P, _P, _c.POINTER(_c.c_int)]),
    ('lss_snowfall_batch_host_wait', _c.c_int, [_P, _c.c_int]),
    ('lss_check_async', _c.c_int, [_P, _P]),
    ('lss_launch_count', _c.c_int64, [_P]),
    ('lss_debug_range_grid', _c.c_int, [_P]),
    ('lss_debug_azimuth', _c.c_int, [_P, _P, _P, _c.c_int64, _P, _P]),
    ('lss_noise_threshold_poly', _c.c_int, [_P, _P, _P, _c.c_int, _c.c_double, _P, _P, _P, _P, _P, _P, _P, _c.c_int64,
                                            _P]),
    ('lss_prepass_workspace_bytes', _c.c_int64, [_c.c_int64, _c.c_int]),
    ('lss_wet_ground_batch', _c.c_int, [_P, _P, _P, _P, _c.c_int, _c.c_double, _c.c_double, _c.c_double, _c.c_double,
                                        _c.c_int, _c.c_double, _c.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _c.c_int64, _P]),
    ('lss_wet_ground_workspace_bytes', _c.c_int64, [_c.c_int64, _c.c_int]),
    ('lss_fog_batch', _c.c_int, [_P, _P, _c.c_int, _P, _c.c_int, _c.c_double, _c.c_double, _c.c_double, _P, _c.c_uint32,
                                 _c.c_int, _c.c_int, _P, _P, _P, _P, _P, _P, _P, _c.c_int64, _P]),
    ('lss_fog_workspace_bytes', _c.c_int64, [_c.c_int64, _c.c_int]),
    ('lss_lisa_batch', _c.c_int, [_P, _P, _c.c_int, _c.c_int64, _c.c_double, _c.c_int, _c.c_double, _c.c_double, _c.c_double,
                                  _c.c_double, _c.c_double, _c.c_double, _c.c_int, _P, _c.c_int, _c.c_uint64, _P, _P]),
    ('lss_voxelize_batch', _c.c_int, [_P, _P, _c.c_int, _P, _P, _c.c_int, _P, _P, _c.c_int, _c.c_int, _c.c_int, _P, _P, _P,
                                      _P, _P, _c.c_int64, _P]),
    ('lss_voxelize_workspace_bytes', _c.c_int64, [_c.c_int64, _c.c_int, _c.c_int, _c.c_int]),
    ('lss_dror_batch', _c.c_int, [_P, _P, _c.c_int, _P, _P, _c.c_int, _c.c_double, _c.c_double, _c.c_int, _c.c_double,
                                  _P, _P, _P, _P, _P, _P, _c.c_int64, _P]),
    ('lss_dror_workspace_bytes', _c.c_int64, [_c.c_int64, _c.c_int]),
    ('lss_gather_push', _c.c_int, [_P, _P, _P, _P, _c.c_int, _c.c_int64, _c.c_int, _c.c_int, _P, _P, _P, _P, _c.c_int, _P]),
    ('lss_dart_throwing', _c.c_int, [_c.c_double, _c.c_double, _c.c_double, _c.c_int, _P, _P, _c.c_int64,
                                     _c.POINTER(_c.c_int64)]),
    ('lss_dart_throwing_planes', _c.c_int, [_c.c_int, _c.c_double, _c.c_double, _c.c_double, _c.c_int, _P, _P,
                                            _c.c_int64, _P, _c.c_int]),
    ('lss_sample_particles', _c.c_int, [_P, _c.c_int, _c.c_double, _c.c_double, _c.c_double, _c.c_int, _c.c_uint64,
                                        _c.c_int64, _P, _c.c_int64, _P, _P, _P, _c.c_int64, _P]),
    ('lss_sample_particles_workspace_bytes', _c.c_int64, [_c.c_int, _c.c_int64]),
    ('lss_set_profiling', _c.c_int, [_P, _c.c_int]),
    ('lss_kernel_times', _c.c_int, [_P, _c.c_int, _P, _P, _c.c_int]),
    ('lss_kernel_name', _c.c_char_p, [_c.c_int]),
]

_lib = None


def load():
    """Load liblss_b200.so and bind every declared symbol.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f'{LIB_PATH} not found: build it with `python -m lidar_snow_sim_b200.build` '
                          f'(or __graft_entry__.build()); this engine has no CPU fallback')
    lib = ctypes.CDLL(LIB_PATH)
    for name, res, args in SIGNATURES:
        fn = getattr(lib, name)           # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, engine_handle=None):
    if status == LSS_OK:
        return
    lib = load()
    msg = lib.lss_status_string(status).decode()
    if engine_handle:
        detail = lib.lss_last_error(engine_handle).decode()
        if detail:
            msg = f'{msg}: {detail}'
    raise _EXC.get(status, RuntimeError)(msg)
