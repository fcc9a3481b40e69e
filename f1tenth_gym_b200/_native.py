"""ctypes binding of libf110_b200.so (C ABI declared in include/f110_b200.h).

There is NO fallback: if the shared library is missing or fails to load, every product entry point
raises.  Build it with `python -m f1tenth_gym_b200.build` (nvcc, sm_100a) — __graft_entry__.build()
does that.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libf110_b200.so')

F110_NPARAM = 18
F110_NSTATE = 7
ABI_VERSION = 2

_dp = C.c_void_p   # device / host pointers are passed as raw addresses


class F110Map(C.Structure):
    _fields_ = [('height', C.c_int32), ('width', C.c_int32),
                ('resolution', C.c_double), ('orig_x', C.c_double), ('orig_y', C.c_double),
                ('orig_c', C.c_double), ('orig_s', C.c_double),
                ('eps', C.c_double), ('max_range', C.c_double),
                ('theta_dis', C.c_int32), ('fast_path', C.c_int32),
                ('dt_oob', C.c_double),
                ('dt', _dp), ('dt_cells', _dp), ('dt_codes', _dp), ('dt_lut', _dp),
                ('sines', _dp), ('cosines', _dp), ('sincos', _dp),
                ('dt_cells_pad', _dp), ('dt_codes_pad', _dp), ('codes_pitch', C.c_uint32), ('sincos2', _dp),
                ('dt_min_positive', C.c_double), ('num_layers', C.c_int32)]


class F110Beams(C.Structure):
    _fields_ = [('num_beams', C.c_int32),
                ('fov', C.c_double), ('angle_increment', C.c_double), ('theta_index_increment', C.c_double),
                ('scan_angles', _dp), ('cosines', _dp), ('side_distances', _dp), ('cos_side', _dp),
                ('side_max', C.c_double)]


class F110Sim(C.Structure):
    _fields_ = [('num_envs', C.c_int32), ('num_agents', C.c_int32), ('integrator', C.c_int32),
                ('ego_idx', C.c_int32), ('params_per_env', C.c_int32),
                ('timestep', C.c_double), ('lidar_dist', C.c_double), ('ttc_thresh', C.c_double),
                ('sim_length', C.c_double), ('sim_width', C.c_double),
                ('params', _dp), ('state', _dp), ('steer_buf', _dp), ('steer_cnt', _dp),
                ('scan_pose', _dp), ('agent_poses', _dp), ('scans', _dp), ('wall_flag', _dp),
                ('collisions', _dp), ('collision_idx', _dp),
                ('current_time', _dp), ('lap_times', _dp), ('lap_counts', _dp), ('toggle_list', _dp),
                ('near_starts', _dp), ('start_xs', _dp), ('start_ys', _dp), ('start_thetas', _dp),
                ('start_rot', _dp), ('done', _dp), ('checkpoint_done', _dp), ('env_arrivals', _dp), ('env_layer', _dp),
                ('lookup_counter', _dp), ('tick_counter', _dp),
                ('march_cost', _dp), ('march_order', _dp), ('march_count', _dp), ('march_ipa', C.c_int32),
                ('march_rec', _dp), ('noise_std', C.c_double), ('noise_seed', C.c_uint64)]


class F110HostObs(C.Structure):
    _fields_ = [('scans', _dp), ('state', _dp), ('collisions', _dp), ('done', _dp),
                ('lap_times', _dp), ('lap_counts', _dp), ('scans_u24', _dp)]


class F110View(C.Structure):
    _fields_ = [('width', C.c_int32), ('height', C.c_int32), ('channels', C.c_int32), ('camera', C.c_int32),
                ('center_x', C.c_double), ('center_y', C.c_double), ('metres_per_pixel', C.c_double),
                ('draw_scan', C.c_int32), ('palette', (C.c_uint8 * 3) * 8),
                ('wx', _dp), ('wy', _dp), ('num_waypoints', C.c_int32),
                ('table_start', _dp), ('num_tables', C.c_int32), ('env_table', _dp)]


# name -> (restype, argtypes); this table is also what tests use to check that every symbol declared
# in include/f110_b200.h is exported.
_P = C.POINTER
SIGNATURES = {
    'f110_abi_version': (C.c_int, []),
    'f110_status_string': (C.c_char_p, [C.c_int]),
    'f110_last_cuda_error': (C.c_char_p, []),
    'f110_step': (C.c_int, [_P(F110Sim), _P(F110Map), _P(F110Beams), _dp, _dp]),
    'f110_step_profile': (C.c_int, [_P(F110Sim), _P(F110Map), _P(F110Beams), _dp, _P(C.c_float), _dp]),
    'f110_reset': (C.c_int, [_P(F110Sim), _dp, _dp, _dp]),
    'f110_env_reset': (C.c_int, [_P(F110Sim), _dp, _dp, _dp]),
    'f110_env_post_step': (C.c_int, [_P(F110Sim), _dp]),
    'f110_autoreset': (C.c_int, [_P(F110Sim), _dp, C.c_int32, C.c_int32, C.c_uint64, C.c_uint64, _dp]),
    'f110_tick': (C.c_int, [_P(F110Sim), _P(F110Map), _P(F110Beams), _dp, C.c_int32, _dp, C.c_int32, C.c_int32,
                            C.c_uint64, _dp]),
    'f110_step_host': (C.c_int, [_P(F110Sim), _P(F110Map), _P(F110Beams), _dp, _dp, _P(F110HostObs), _dp]),
    'f110_step_host_async': (C.c_int, [_P(F110Sim), _P(F110Map), _P(F110Beams), _dp, _dp, _P(F110HostObs),
                                       _P(F110HostObs), _dp, _dp, _dp, _dp]),
    'f110_scan': (C.c_int, [_P(F110Map), _P(F110Beams), _dp, C.c_int32, _dp, _dp, _dp, _dp]),
    'f110_vehicle_dynamics_st': (C.c_int, [_dp, _dp, _dp, C.c_int32, _dp, _dp]),
    'f110_vehicle_dynamics_ks': (C.c_int, [_dp, _dp, _dp, C.c_int32, _dp, _dp]),
    'f110_pid': (C.c_int, [_dp, _dp, C.c_int32, _dp, _dp]),
    'f110_get_vertices': (C.c_int, [_dp, C.c_double, C.c_double, C.c_int32, _dp, _dp]),
    'f110_collision': (C.c_int, [_dp, _dp, C.c_int32, _dp, _dp]),
    'f110_collision_multiple': (C.c_int, [_dp, C.c_int32, C.c_int32, _dp, _dp, _dp]),
    'f110_check_ttc': (C.c_int, [_P(F110Beams), _dp, _dp, C.c_double, C.c_int32, _dp, _dp]),
    'f110_ray_cast': (C.c_int, [_P(F110Beams), _dp, _dp, C.c_int32, _dp, _dp, _dp]),
    'f110_pure_pursuit': (C.c_int, [_dp, _dp, _dp, C.c_int32, _dp, _dp, _dp, C.c_int32, C.c_double, C.c_double, C.c_double,
                                    C.c_double, _dp, _dp]),
    'f110_pure_pursuit_tables': (C.c_int, [_dp, _dp, _dp, _dp, C.c_int32, _dp, _dp, _dp, _dp, C.c_int32, C.c_double,
                                           C.c_double, C.c_double, C.c_double, _dp, _dp]),
    'f110_edt': (C.c_int, [_dp, C.c_int32, C.c_int32, C.c_double, _dp, _dp, _dp, _dp]),
    'f110_rasterize_track': (C.c_int, [_dp, C.c_int32, C.c_double, C.c_double, C.c_int32, C.c_int32, _dp, _dp, _dp]),
    'f110_scan_noise': (C.c_int, [_dp, C.c_int64, C.c_double, C.c_uint64, C.c_uint64, _dp]),
    'f110_pack_scans_u24': (C.c_int, [_dp, C.c_int64, _dp, _dp]),
    'f110_render': (C.c_int, [_P(F110Sim), _P(F110Map), _P(F110Beams), _P(F110View), _dp, C.c_int32, _dp, _dp, _dp]),
}

# measurement / test aids exported by the library but not part of the public header
DEBUG_SIGNATURES = {
    'f110_debug_set_variant': (None, [C.c_int]),
    'f110_debug_set_chunk': (None, [C.c_int]),
    'f110_debug_set_dyn': (None, [C.c_int, C.c_int]),
    'f110_debug_set_ipt': (None, [C.c_int, C.c_int, C.c_int, C.c_int]),
    'f110_debug_set_pdl': (None, [C.c_int]),
    'f110_debug_set_tail': (None, [C.c_int]),
    'f110_debug_set_tail2': (None, [C.c_int, C.c_int]),
    'f110_debug_set_tile_counter': (None, [C.c_void_p]),
}

_LIB = None


class NativeLibraryError(RuntimeError):
    pass


class F110Error(RuntimeError):
    def __init__(self, status, message):
        RuntimeError.__init__(self, message)
        self.status = status


def lib():
    """Load libf110_b200.so (once).  Raises NativeLibraryError when it is absent — no CPU fallback."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            'f1tenth_gym_b200: native CUDA library %s is missing. Build it with '
            '`python -m f1tenth_gym_b200.build` (needs nvcc); there is no CPU fallback.' % LIB_PATH)
    try:
        L = C.CDLL(LIB_PATH)
    except OSError as e:
        raise NativeLibraryError('f1tenth_gym_b200: cannot load %s: %s' % (LIB_PATH, e))
    for name, (res, args) in SIGNATURES.items():
        try:
            f = getattr(L, name)
        except AttributeError:
            raise NativeLibraryError('f1tenth_gym_b200: %s does not export %s (stale build?)' % (LIB_PATH, name))
        f.restype = res
        f.argtypes = args
    for name, (res, args) in DEBUG_SIGNATURES.items():
        f = getattr(L, name, None)
        if f is not None:
            f.restype = res
            f.argtypes = args
    if L.f110_abi_version() != ABI_VERSION:
        raise NativeLibraryError('f1tenth_gym_b200: ABI version mismatch (lib %d, python %d); rebuild'
                                 % (L.f110_abi_version(), ABI_VERSION))
    _LIB = L
    return L


# status -> Python exception type, mirroring the reference's error behaviour
# (ValueError: laser_models.py:445-446, base_classes.py:625-626; IndexError: base_classes.py:534;
#  SyntaxError: base_classes.py:397-398)
_EXC = {-2: ValueError, -5: ValueError, -6: IndexError, -4: SyntaxError}


def check(status):
    if status == 0:
        return
    L = lib()
    msg = L.f110_status_string(status).decode()
    if status == -3:
        msg += ': ' + L.f110_last_cuda_error().decode()
    exc = _EXC.get(status)
    if exc is not None:
        raise exc(msg)
    raise F110Error(status, 'f1tenth_gym_b200: %s (status %d)' % (msg, status))


def ptr(t):
    """Raw address of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()
