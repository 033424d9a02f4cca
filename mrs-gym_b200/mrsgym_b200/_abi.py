"""ctypes binding of include/mrs_b200.h (libmrs_b200.so).

This is the only place Python touches the C ABI.  There is no CPU fallback: if the shared
library is missing, ``lib()`` raises with the build command instead of degrading to torch ops.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('MRS_B200_LIB') or os.path.join(_HERE, 'libmrs_b200.so')   # override: A/B builds

ABI_VERSION = 6
STATE_PLANES = 13
CTRL_PLANES = 18
STATS_SLOTS = 8
SCRATCH_PLANES = 7
SYNC_WORDS = 8208

# MrsActionType: the reference's ACTION_TYPE strings are Quadcopter method names
# (/root/reference/mrsgym/Environment.py:92)
ACTION_TYPES = dict(set_target_vel=0, set_target_pos=1, set_target_accel=2, set_force=3,
                    set_target_ori=4, set_control=5, set_speeds=6)
NO_ACTION = 7
ACTION_DIMS = {0: 3, 1: 3, 2: 3, 3: 3, 4: 3, 5: 4, 6: 4, 7: 0}

X_NONE, X_POS_VEL, X_FULL = 0, 1, 2
STATE_DIMS = {X_NONE: 0, X_POS_VEL: 6, X_FULL: 13}

STATUS_NAN_ACTION = 1
STATUS_NONFINITE = 2
STATUS_COMM_TIMEOUT = 4
STATUS_SYNC_TIMEOUT = 8
STATUS_CONTACT_OVERFLOW = 16
STATUS_NEIGHBOR_OVERFLOW = 32
COMM_MAX_WORLD = 16
COMM_HANDLE_BYTES = 64
STAT_NAMES = ('agent_contact_rows', 'ground_contacts', 'nonfinite', 'nan_actions', 'contact_chunks', 'solver_sweeps',
              'neighbor_overflow')

f = C.c_float


class MrsQuadParams(C.Structure):
    _fields_ = [('mass', f), ('ixx', f), ('iyy', f), ('izz', f),
                ('kf', f), ('km', f), ('arm', f),
                ('gnd_eff_coeff', f), ('prop_radius', f), ('gnd_hclip', f),
                ('drag_xy', f), ('drag_z', f),
                ('dw1', f), ('dw2', f), ('dw3', f),
                ('prop_x', f * 4), ('prop_y', f * 4),
                ('pos_p', f), ('pos_i', f), ('pos_d', f),
                ('vel_p', f), ('vel_i', f), ('vel_d', f),
                ('ori_p', f * 3), ('ori_i', f * 3), ('ori_d', f * 3),
                ('min_pwm', f), ('max_pwm', f), ('pwm2rpm_a', f), ('pwm2rpm_b', f),
                ('ctrl_dt', f), ('ctrl_gravity', f),
                ('mix_ainv', f * 16), ('mix_a', f * 16), ('nnls_tab', f * 256)]


class MrsPhysicsParams(C.Structure):
    _fields_ = [('mass', f), ('inertia', f * 3),
                ('lin_damping', f), ('ang_damping', f), ('max_coord_vel', f),
                ('gyro', C.c_int), ('ang_motion_threshold', f),
                ('erp2', f), ('slop', f), ('contact_margin', f),
                ('mu_ground', f), ('ground_z', f),
                ('col_radius', f), ('col_halfheight', f), ('col_margin', f),
                ('ground_contact', C.c_int), ('agent_contact', C.c_int),
                ('agent_radius', f), ('contact_radius', f), ('mu_agent', f), ('solver_iters', C.c_int),
                ('solver_tol', f)]


class MrsConfig(C.Structure):
    _fields_ = [('E', C.c_int), ('N', C.c_int), ('K', C.c_int), ('L', C.c_int),
                ('action_type', C.c_int), ('state_layout', C.c_int),
                ('dt', f), ('gravity', f), ('comm_range', f),
                ('quad', MrsQuadParams), ('phys', MrsPhysicsParams)]


class MrsBuffers(C.Structure):
    _fields_ = [('state', C.c_void_p), ('ctrl', C.c_void_p), ('rpm', C.c_void_p),
                ('X_tape', C.c_void_p), ('A_tape', C.c_void_p), ('scratch', C.c_void_p),
                ('status', C.c_void_p), ('stats', C.c_void_p), ('sync', C.c_void_p), ('wrench', C.c_void_p)]


class MrsAutoResetArgs(C.Structure):
    _fields_ = [('seed', C.c_ulonglong), ('env_offset', C.c_ulonglong),
                ('z_lo', f), ('z_hi', f), ('xy_radius', f), ('xy_sigma', f), ('yaw_lo', f), ('yaw_hi', f),
                ('max_rounds', C.c_int), ('episode_length', C.c_int), ('max_timesteps', C.c_int)]


class Derived(C.Structure):
    """mirror of the library's internal struct Derived (mrs_device.cuh), as mrs_debug_derived fills it: the constants
    the step derives from a config (tools/gen_baked.py bakes them; the tests read thresholds from them)"""
    _fields_ = [('inv_mass', f), ('inv_I', f * 3), ('gnd_c', f), ('dw_c', f), ('rpm2rad', f), ('q_x2', f),
                ('cap_w2', f), ('cap_k', f), ('cap_c', f), ('lim2', f), ('gnd_skip_z', f), ('inv_dt', f),
                ('erp_dt', f), ('s_max', f), ('comm_inf', C.c_int), ('inv_ctrl_dt', f), ('inv_4kf', f),
                ('inv_pwm_a', f), ('inv_qmass', f)]


class MrsError(RuntimeError):
    pass


_SIGNATURES = {
    'mrs_abi_version': (C.c_int, []),
    'mrs_strerror': (C.c_char_p, [C.c_int]),
    'mrs_state_dim': (C.c_int, [C.c_int]),
    'mrs_action_dim': (C.c_int, [C.c_int]),
    'mrs_scratch_planes': (C.c_int, [C.c_int, C.c_int]),
    'mrs_sizeof_config': (C.c_size_t, []),
    'mrs_sizeof_buffers': (C.c_size_t, []),
    'mrs_default_config': (C.c_int, [C.POINTER(MrsConfig)]),
    'mrs_config_is_baked': (C.c_int, [C.POINTER(MrsConfig)]),
    'mrs_debug_derived': (C.c_int, [C.POINTER(MrsConfig), C.c_void_p, C.c_size_t]),
    'mrs_step': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    'mrs_step_many': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_int, C.c_int, C.c_int,
                                C.c_void_p]),
    'mrs_rollout': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_int, C.c_int, C.c_int,
                              C.c_void_p]),
    'mrs_observe': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_int, C.c_int, C.c_int, C.c_void_p]),
    'mrs_adjacency': (C.c_int, [C.POINTER(MrsConfig), C.c_void_p, C.c_void_p, C.c_void_p]),
    'mrs_neighbors': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    'mrs_set_state': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p]),
    'mrs_tape_fill': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_void_p]),
    'mrs_step_host': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    'mrs_pack_adjacency': (C.c_int, [C.POINTER(MrsConfig), C.c_void_p, C.c_void_p, C.c_void_p]),
    'mrs_rollout_host': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    'mrs_spawn': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_ulonglong, C.c_ulonglong, C.c_float, C.c_float,
                            C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_void_p]),
    'mrs_autoreset': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.POINTER(MrsAutoResetArgs), C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    'mrs_proximity': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p]),
    'mrs_raycast': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_int, C.POINTER(C.c_float),
                              C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    'mrs_comm_create': (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'mrs_comm_handle': (C.c_int, [C.c_void_p, C.c_char_p]),
    'mrs_comm_connect': (C.c_int, [C.c_void_p, C.c_char_p]),
    'mrs_comm_mailbox': (C.c_void_p, [C.c_void_p]),
    'mrs_comm_connect_ptrs': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]),
    'mrs_comm_destroy': (C.c_int, [C.c_void_p]),
    'mrs_comm_barrier': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    'mrs_stats_allreduce': (C.c_int, [C.POINTER(MrsConfig), C.POINTER(MrsBuffers), C.c_void_p, C.c_void_p, C.c_void_p]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def lib():
    """The loaded C ABI.  Raises (never falls back) when the extension is not built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise MrsError('libmrs_b200.so is not built (%s): run `python -c "import __graft_entry__ as g; '
                           'g.build()"` or `make -C mrs-gym_b200`.  There is no CPU fallback.' % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.mrs_abi_version() != ABI_VERSION:
            raise MrsError('ABI version mismatch: library %d, binding %d' % (handle.mrs_abi_version(), ABI_VERSION))
        if handle.mrs_sizeof_config() != C.sizeof(MrsConfig) or handle.mrs_sizeof_buffers() != C.sizeof(MrsBuffers):
            raise MrsError('struct layout mismatch between libmrs_b200.so and mrsgym_b200/_abi.py')
        _lib = handle
    return _lib


def check(rc, what=''):
    if rc != 0:
        raise MrsError('%s failed: %s (%d)' % (what or 'mrs call', lib().mrs_strerror(rc).decode(), rc))


def default_config() -> MrsConfig:
    cfg = MrsConfig()
    check(lib().mrs_default_config(C.byref(cfg)), 'mrs_default_config')
    return cfg
