"""ctypes mirror of ``include/mate_b200.h`` and the loader of ``libmate_b200.so``.

The product path has NO CPU fallback: :func:`load_library` raises if the CUDA library has
not been built (``python -c "import __graft_entry__ as g; g.build()"``).
"""

import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('MATE_B200_LIB') or os.path.join(HERE, 'csrc', 'libmate_b200.so')

c_double_p = ctypes.POINTER(ctypes.c_double)
c_float_p = ctypes.POINTER(ctypes.c_float)
c_int32_p = ctypes.POINTER(ctypes.c_int32)
c_uint8_p = ctypes.POINTER(ctypes.c_uint8)
c_int8_p = ctypes.POINTER(ctypes.c_int8)

MATE_STEP_AUTO_RESET = 1
MATE_STEP_HOST_ROWS_KEPT = 2
MATE_OBS_FORMAT_F32 = 0
MATE_OBS_FORMAT_F16 = 1
MATE_SNAPSHOT_VERSION = 1
MATE_LOAD_STATE_RESUME = 1


class MateConfig(ctypes.Structure):
    _fields_ = [
        ('num_cameras', ctypes.c_int32),
        ('num_targets', ctypes.c_int32),
        ('num_obstacles', ctypes.c_int32),
        ('max_episode_steps', ctypes.c_int32),
        ('num_cargoes_per_target', ctypes.c_int32),
        ('num_high_capacity_targets', ctypes.c_int32),
        ('targets_start_with_cargoes', ctypes.c_int32),
        ('shuffle_entities', ctypes.c_int32),
        ('reward_sparse', ctypes.c_int32),
        ('reserved0', ctypes.c_int32),
        ('bounty_factor', ctypes.c_double),
        ('camera_radius', ctypes.c_double),
        ('camera_min_viewing_angle', ctypes.c_double),
        ('camera_max_sight_range', ctypes.c_double),
        ('camera_rotation_step', ctypes.c_double),
        ('camera_zooming_step', ctypes.c_double),
        ('target_step_size', ctypes.c_double),
        ('target_sight_range', ctypes.c_double),
        ('obstacle_transmittance', ctypes.c_double),
        ('obstacle_radius_low', ctypes.c_double),
        ('obstacle_radius_high', ctypes.c_double),
        ('camera_location_ranges', c_double_p),
        ('target_location_ranges', c_double_p),
        ('obstacle_location_ranges', c_double_p),
    ]


STATE_FIELDS = [
    # name, ctype pointer, numpy dtype, shape as function of (B, Nc, Nt, No)
    ('cam_xy', c_double_p, np.float64, lambda B, nc, nt, no: (B, nc, 2)),
    ('cam_phi', c_double_p, np.float64, lambda B, nc, nt, no: (B, nc)),
    ('cam_theta', c_double_p, np.float64, lambda B, nc, nt, no: (B, nc)),
    ('tgt_xy', c_double_p, np.float64, lambda B, nc, nt, no: (B, nt, 2)),
    ('obs_xyr', c_double_p, np.float64, lambda B, nc, nt, no: (B, no, 3)),
    ('tgt_capacity', c_int32_p, np.int32, lambda B, nc, nt, no: (B, nt)),
    ('tgt_goal', c_int32_p, np.int32, lambda B, nc, nt, no: (B, nt)),
    ('tgt_weight', c_int32_p, np.int32, lambda B, nc, nt, no: (B, nt)),
    ('tgt_bounty', c_int32_p, np.int32, lambda B, nc, nt, no: (B, nt)),
    ('tgt_empty_bits', c_int32_p, np.int32, lambda B, nc, nt, no: (B, nt)),
    ('remaining', c_int32_p, np.int32, lambda B, nc, nt, no: (B, 4, 4)),
    ('awaiting', c_int32_p, np.int32, lambda B, nc, nt, no: (B, 4)),
    ('num_delivered', c_int32_p, np.int32, lambda B, nc, nt, no: (B,)),
    ('episode_step', c_int32_p, np.int32, lambda B, nc, nt, no: (B,)),
    ('episode_id', c_int32_p, np.int32, lambda B, nc, nt, no: (B,)),
    ('episode_reward', c_double_p, np.float64, lambda B, nc, nt, no: (B, 2)),
]


class MateStateView(ctypes.Structure):
    _fields_ = [(name, ctype) for name, ctype, _, _ in STATE_FIELDS]


AUX_FIELDS = [
    ('mask_ct', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nc, nt)),
    ('mask_cc', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nc, nc)),
    ('mask_co', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nc, no)),
    ('mask_tc', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nt, nc)),
    ('mask_to', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nt, no)),
    ('mask_tt', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nt, nt)),
    ('coverage', c_float_p, np.float32, lambda B, nc, nt, no: (B, 3)),
    ('num_delivered', c_int32_p, np.int32, lambda B, nc, nt, no: (B,)),
    ('target_dones', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nt)),
    ('is_colliding', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nt)),
    ('warehouse_dist', c_float_p, np.float32, lambda B, nc, nt, no: (B, nt, 4)),
    ('episode_step', c_int32_p, np.int32, lambda B, nc, nt, no: (B,)),
    ('tgt_goal', c_int32_p, np.int32, lambda B, nc, nt, no: (B, nt)),
    ('tgt_empty_bits', c_uint8_p, np.uint8, lambda B, nc, nt, no: (B, nt)),
]


class MateStepAux(ctypes.Structure):
    _fields_ = [(name, ctype) for name, ctype, _, _ in AUX_FIELDS]


class MateAgentReplay(ctypes.Structure):
    _fields_ = [('binomial', c_uint8_p), ('sample', c_double_p), ('choice', c_int8_p), ('reset_sample', c_double_p)]


class MateCameraAgentReplay(ctypes.Structure):
    _fields_ = [('binomial', c_int8_p), ('sample', c_double_p), ('delay', c_int32_p)]


AGENT_MEMORY = 6   # MATE_AGENT_MEMORY


class MateMessageFilter(ctypes.Structure):
    _fields_ = [('range_limit', ctypes.c_double * 2), ('keep_probability', ctypes.c_double * 2),
                ('delivered', ctypes.c_void_p * 2), ('total_edges', ctypes.c_void_p * 2)]


class MateMessageExchange(ctypes.Structure):
    _fields_ = [('content', ctypes.c_void_p), ('recipients', ctypes.c_void_p), ('inbox', ctypes.c_void_p),
                ('delivered', ctypes.c_void_p), ('episode', ctypes.c_void_p), ('team', ctypes.c_int32),
                ('dim', ctypes.c_int32), ('reduction', ctypes.c_int32), ('reserved', ctypes.c_int32)]


# reductions of mate_b200_exchange_messages (MATE_MESSAGES_*)
MATE_MESSAGES_NONE, MATE_MESSAGES_SUM, MATE_MESSAGES_MEAN = 0, 1, 2
MESSAGE_REDUCTIONS = {'none': MATE_MESSAGES_NONE, 'sum': MATE_MESSAGES_SUM, 'mean': MATE_MESSAGES_MEAN}


class MateReplay(ctypes.Structure):
    _fields_ = [('transmit', c_uint8_p), ('goal_choice', c_int8_p)]


SNAPSHOT_INFO_FIELDS = ('version', 'num_cameras', 'num_targets', 'num_obstacles', 'count', 'config_hash', 'seed', 'payload_bytes')


class MateSnapshotInfo(ctypes.Structure):
    _fields_ = [
        ('version', ctypes.c_int32),
        ('num_cameras', ctypes.c_int32),
        ('num_targets', ctypes.c_int32),
        ('num_obstacles', ctypes.c_int32),
        ('count', ctypes.c_int32),
        ('reserved', ctypes.c_int32),
        ('config_hash', ctypes.c_uint64),
        ('seed', ctypes.c_uint64),
        ('payload_bytes', ctypes.c_uint64),
    ]


def alloc_state_arrays(B, nc, nt, no):
    """Fresh host arrays for every MateStateView field."""
    return {name: np.zeros(shape(B, nc, nt, no), dtype=dtype) for name, _, dtype, shape in STATE_FIELDS}


def state_view_from_arrays(arrays):
    """Build a MateStateView over C-contiguous numpy arrays (missing / None => NULL)."""
    view = MateStateView()
    keep = []
    for name, ctype, dtype, _ in STATE_FIELDS:
        arr = arrays.get(name)
        if arr is None:
            setattr(view, name, ctype())
            continue
        arr = np.ascontiguousarray(arr, dtype=dtype)
        arrays[name] = arr
        keep.append(arr)
        setattr(view, name, arr.ctypes.data_as(ctype))
    view._keepalive = keep
    return view


def make_config_struct(cfg):
    """MateConfig from the flat dict produced by :func:`mate_b200.config.flatten_config`."""
    out = MateConfig()
    keep = []
    for name, ctype in MateConfig._fields_:
        if name.endswith('_location_ranges'):
            arr = np.ascontiguousarray(cfg[name], dtype=np.float64).reshape(-1, 4)
            keep.append(arr)
            setattr(out, name, arr.ctypes.data_as(c_double_p))
        elif name == 'reserved0':
            out.reserved0 = 0
        else:
            setattr(out, name, cfg[name])
    out._keepalive = keep
    return out


_LIB = None


def load_library():
    """Load ``libmate_b200.so`` (built in-tree by ``__graft_entry__.build()``).  No fallback."""
    global _LIB  # pylint: disable=global-statement
    if _LIB is not None:
        return _LIB
    path = os.environ.get('MATE_B200_LIB', LIB_PATH)   # override: A/B builds with other tuning knobs
    if not os.path.exists(path):
        raise RuntimeError(
            f'{path} is missing: the CUDA extension has not been built. '
            'Run `python -c "import __graft_entry__ as g; g.build()"` in the repo root. '
            'mate_b200 has no CPU fallback.'
        )
    lib = ctypes.CDLL(path)
    void_p = ctypes.c_void_p
    lib.mate_b200_last_error.restype = ctypes.c_char_p
    lib.mate_b200_abi_version.restype = ctypes.c_int
    lib.mate_b200_create.argtypes = [ctypes.POINTER(MateConfig), ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, ctypes.POINTER(void_p)]
    lib.mate_b200_destroy.argtypes = [void_p]
    lib.mate_b200_obs_dims.argtypes = [void_p, c_int32_p, c_int32_p]
    lib.mate_b200_set_observation_format.argtypes = [void_p, ctypes.c_int32]
    lib.mate_b200_reset.argtypes = [void_p, void_p, ctypes.c_uint64, void_p, void_p, void_p]
    lib.mate_b200_seed.argtypes = [void_p, void_p, ctypes.c_uint64, void_p]
    lib.mate_b200_step.argtypes = [void_p, void_p, void_p, void_p, void_p, void_p, void_p,
                                   ctypes.POINTER(MateStepAux), ctypes.POINTER(MateReplay), ctypes.c_uint32, void_p]
    lib.mate_b200_observe.argtypes = [void_p, void_p, void_p, ctypes.POINTER(MateStepAux), ctypes.POINTER(MateReplay), void_p]
    lib.mate_b200_step_host.argtypes = [void_p, void_p, void_p, void_p, void_p, void_p, void_p, ctypes.c_uint32]
    lib.mate_b200_get_state.argtypes = [void_p, ctypes.POINTER(MateStateView)]
    lib.mate_b200_set_state.argtypes = [void_p, ctypes.POINTER(MateStateView)]
    lib.mate_b200_episode_stats.argtypes = [void_p, void_p, ctypes.c_int32, void_p]
    lib.mate_b200_snapshot_bytes.argtypes = [void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_uint64)]
    lib.mate_b200_save_state.argtypes = [void_p, void_p, ctypes.c_int32, void_p, ctypes.POINTER(MateSnapshotInfo), void_p]
    lib.mate_b200_load_state.argtypes = [void_p, void_p, ctypes.POINTER(MateSnapshotInfo), void_p, ctypes.c_uint32, void_p]
    lib.mate_b200_launch_count.argtypes = [void_p]
    lib.mate_b200_launch_count.restype = ctypes.c_int64
    lib.mate_b200_host_leg_info.argtypes = [void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_uint64)]
    lib.mate_b200_host_leg_info.restype = ctypes.c_int
    lib.mate_b200_transform_observations.argtypes = [void_p, void_p, void_p, c_int32_p, ctypes.c_int32, void_p, void_p, void_p]
    lib.mate_b200_set_observation_ops.argtypes = [void_p, c_int32_p, ctypes.c_int32, void_p, void_p]
    lib.mate_b200_decode_actions.argtypes = [void_p, void_p, ctypes.c_int32, void_p, ctypes.c_int64, void_p]
    lib.mate_b200_fov_range.argtypes = [void_p, void_p, void_p, void_p, void_p, ctypes.c_int64, void_p]
    lib.mate_b200_render.argtypes = [void_p, void_p, ctypes.c_int32, ctypes.c_int32, void_p, void_p]
    lib.mate_b200_auxiliary_terms.argtypes = [void_p, ctypes.POINTER(MateStepAux), void_p, void_p, void_p, void_p, void_p]
    lib.mate_b200_greedy_target_actions.argtypes = [void_p, void_p, void_p, ctypes.c_double, ctypes.c_uint64, ctypes.c_uint64,
                                                    ctypes.POINTER(MateAgentReplay), void_p, void_p]
    lib.mate_b200_greedy_camera_actions.argtypes = [void_p, void_p, void_p, void_p, ctypes.c_uint64, ctypes.c_uint64,
                                                    ctypes.POINTER(MateCameraAgentReplay), void_p, void_p]
    lib.mate_b200_soft_coverage.argtypes = [void_p, void_p, void_p, void_p, void_p]
    lib.mate_b200_set_message_filter.argtypes = [void_p, ctypes.POINTER(MateMessageFilter)]
    lib.mate_b200_exchange_messages.argtypes = [void_p, ctypes.POINTER(MateMessageExchange), ctypes.c_uint64, void_p]
    for name in ('create', 'destroy', 'obs_dims', 'set_observation_format', 'reset', 'seed', 'step', 'observe', 'step_host',
                 'get_state', 'set_state', 'snapshot_bytes', 'save_state', 'load_state', 'episode_stats', 'transform_observations', 'set_observation_ops', 'decode_actions', 'auxiliary_terms', 'fov_range', 'soft_coverage', 'greedy_target_actions', 'greedy_camera_actions', 'set_message_filter',
                 'exchange_messages', 'render'):
        getattr(lib, 'mate_b200_' + name).restype = ctypes.c_int
    _LIB = lib
    return lib


EXPORTED_SYMBOLS = [
    'mate_b200_last_error', 'mate_b200_abi_version', 'mate_b200_create', 'mate_b200_destroy',
    'mate_b200_obs_dims', 'mate_b200_set_observation_format', 'mate_b200_reset', 'mate_b200_seed', 'mate_b200_step', 'mate_b200_observe',
    'mate_b200_step_host', 'mate_b200_get_state', 'mate_b200_set_state', 'mate_b200_snapshot_bytes', 'mate_b200_save_state',
    'mate_b200_load_state',
    'mate_b200_episode_stats', 'mate_b200_launch_count', 'mate_b200_host_leg_info', 'mate_b200_transform_observations', 'mate_b200_set_observation_ops',
    'mate_b200_decode_actions', 'mate_b200_auxiliary_terms', 'mate_b200_fov_range', 'mate_b200_soft_coverage', 'mate_b200_greedy_target_actions', 'mate_b200_greedy_camera_actions',
    'mate_b200_set_message_filter', 'mate_b200_exchange_messages', 'mate_b200_render',
]

# observation wrapper codes (include/mate_b200.h)
OBS_ENHANCED_CAMERA, OBS_ENHANCED_TARGET, OBS_SHARED_CAMERA, OBS_SHARED_TARGET, OBS_RELATIVE, OBS_RESCALED = range(1, 7)
MAX_OBS_OPS = 8
CAM_TERMS, TGT_TERMS = 8, 16   # MATE_CAM_TERMS / MATE_TGT_TERMS
RENDER_MIN_SIZE, RENDER_MAX_SIZE = 16, 4096   # MATE_RENDER_MIN_SIZE / MATE_RENDER_MAX_SIZE
