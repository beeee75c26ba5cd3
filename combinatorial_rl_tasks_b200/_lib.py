"""ctypes binding of include/crl_b200.h.  There is no CPU fallback: if the CUDA
library is missing or fails to load, importing the product raises."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# CRL_B200_LIB: a tuning variant built by build.py (another CUDA build of the same source), never a fallback
LIB_PATH = os.environ.get('CRL_B200_LIB') or os.path.join(HERE, 'libcrl_b200.so')

c_void_p, c_int32, c_int64, c_uint32, c_uint64, c_double = (
    ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_double)

TASK_TSP, TASK_TTSP, TASK_CM = 0, 1, 2
SEED_INCREMENT, SEED_FIXED_RANGE = 0, 1
STEP_AUTO_RESET, STEP_PHYSICS_ONLY, STEP_CHAINED, STEP_CHAIN_START, STEP_TRACK_ROWS = 1, 2, 4, 8, 16
STEP_GOALS, STEP_WAIT, STEP_ACTION_COUNTER, STEP_NO_ZONE_OBS, STEP_HOST_PLANES = 32, 64, 128, 512, 1024
STEP_ZONE_OBS_DELTA = 2048
ABI_VERSION = 9
NUM_PLANES = 23

# every symbol include/crl_b200.h declares
SYMBOLS = ['crl_abi_version', 'crl_strerror', 'crl_plane_bytes', 'crl_step_bytes', 'crl_reset',
           'crl_prefetch_layouts', 'crl_prefetch_publish', 'crl_reset_from_layout', 'crl_step', 'crl_step_host',
           'crl_host_call_create', 'crl_host_call_step', 'crl_host_call_destroy',
           'crl_set_goal', 'crl_goal_query', 'crl_set_qpos_qvel',
           'crl_get_qpos_qvel', 'crl_gae', 'crl_check_state', 'crl_counters_read',
           'crl_encoder_packed_bytes', 'crl_encoder_pack', 'crl_zone_encode', 'crl_zone_encode_state',
           'crl_encoder_head_packed_bytes', 'crl_encoder_pack_head', 'crl_encoder_head',
           'crl_encoder_workspace_bytes', 'crl_encoder_forward',
           'crl_encoder_precise_packed_bytes', 'crl_encoder_pack_precise', 'crl_zone_encode_precise',
           'crl_encoder_backward_workspace_bytes', 'crl_zone_encode_backward',
           'crl_frame_capture', 'crl_zone_encode_frames', 'crl_zone_encode_backward_frames', 'crl_frames_zone_obs',
           'crl_copy_envs']
FRAME_NO_LAYOUT = 0xffffffff


class CrlConfig(ctypes.Structure):
    _fields_ = [('task', c_int32), ('num_envs', c_int32), ('num_zones', c_int32), ('num_steps', c_int32),
                ('frameskip', c_int32), ('max_cooldown', c_int32), ('seed_mode', c_int32),
                ('env_offset', c_int32), ('min_seed', c_int64), ('max_seed', c_int64),
                ('zone_size', c_double), ('time_saved_reward', c_double), ('beta_a', c_double),
                ('beta_b', c_double), ('robot_keepout', c_double), ('zone_keepout', c_double),
                ('extent', c_double), ('initial_visited', c_uint32), ('walled', c_uint32)]


class CrlState(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ('pose', 'aux', 'zone_xy', 'zone_tmax', 'cooldown', 'seed',
                                        'episode', 'origin', 'counters', 'next_zone_xy', 'next_task',
                                        'next_origin', 'next_seed', 'next_ready', 'stamp',
                                        'prefetch_work', 'row_list', 'goal', 'bank_zone_xy', 'bank_origin',
                                        'bank_task', 'fixed_layout', 'prefetch_epoch')]


class CrlOut(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ('obs', 'zone_obs', 'result', 'shaped_reward')]


class CrlEncoderShape(ctypes.Structure):
    _fields_ = [('obs_dim', c_int32), ('zone_dim', c_int32), ('hidden', c_int32), ('num_zones', c_int32)]


class CrlLayoutIn(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ('xy0', 'rot0', 'zone_xy', 'zone_max_steps', 'colours')]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'{LIB_PATH} is missing: build it with `python -m combinatorial_rl_tasks_b200.build` '
            '(nvcc, sm_100a).  This package has no CPU fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    P = ctypes.POINTER
    lib.crl_abi_version.restype = ctypes.c_int
    lib.crl_strerror.restype = ctypes.c_char_p
    lib.crl_strerror.argtypes = [ctypes.c_int]
    lib.crl_plane_bytes.argtypes = [P(CrlConfig), P(c_int64), c_int32]
    lib.crl_step_bytes.argtypes = [P(CrlConfig), P(c_int64), P(c_int64)]
    lib.crl_reset.argtypes = [P(CrlConfig), P(CrlState), P(CrlOut), c_void_p, c_void_p]
    lib.crl_prefetch_layouts.argtypes = [P(CrlConfig), P(CrlState), c_int32, c_uint32, c_void_p]
    lib.crl_prefetch_publish.argtypes = [P(CrlState), c_uint32, c_void_p]
    lib.crl_reset_from_layout.argtypes = [P(CrlConfig), P(CrlState), P(CrlOut), P(CrlLayoutIn), c_void_p,
                                          c_int32, c_void_p]
    lib.crl_step.argtypes = [P(CrlConfig), P(CrlState), c_void_p, P(CrlOut), c_uint32, c_uint64, c_uint64,
                             c_void_p]
    lib.crl_step_host.argtypes = [P(CrlConfig), P(CrlState), c_void_p, c_void_p, P(CrlOut), P(CrlOut),
                                  c_uint32, c_void_p]
    lib.crl_host_call_create.argtypes = [P(CrlConfig), P(CrlState), P(CrlOut), P(CrlOut), c_uint32, P(c_void_p)]
    lib.crl_host_call_step.argtypes = [c_void_p, c_void_p, c_void_p]
    lib.crl_host_call_destroy.argtypes = [c_void_p]
    lib.crl_host_call_destroy.restype = None
    lib.crl_set_goal.argtypes = [P(CrlConfig), P(CrlState), c_void_p, c_void_p]
    lib.crl_goal_query.argtypes = [P(CrlConfig), P(CrlState), c_void_p, c_void_p, c_void_p, c_void_p]
    lib.crl_set_qpos_qvel.argtypes = [P(CrlConfig), P(CrlState), c_void_p, c_void_p, c_void_p, c_int32,
                                      c_void_p]
    lib.crl_get_qpos_qvel.argtypes = [P(CrlConfig), P(CrlState), c_void_p, c_void_p, c_void_p, c_int32,
                                      c_void_p]
    lib.crl_gae.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_double, c_int32, c_int32,
                            c_void_p, c_void_p, c_void_p]
    lib.crl_check_state.argtypes = [P(CrlConfig), P(CrlState), c_void_p, c_void_p]
    lib.crl_counters_read.argtypes = [P(CrlState), P(c_double), c_void_p]
    lib.crl_encoder_packed_bytes.argtypes = [P(CrlEncoderShape), P(c_int64)]
    lib.crl_encoder_pack.argtypes = [P(CrlEncoderShape)] + [c_void_p] * 6
    lib.crl_zone_encode.argtypes = [P(CrlEncoderShape), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p]
    lib.crl_zone_encode_state.argtypes = [P(CrlEncoderShape), P(CrlConfig), P(CrlState), c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p]
    lib.crl_encoder_head_packed_bytes.argtypes = [P(CrlEncoderShape), P(c_int64)]
    lib.crl_encoder_pack_head.argtypes = [P(CrlEncoderShape)] + [c_void_p] * 4
    lib.crl_encoder_head.argtypes = [P(CrlEncoderShape), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p]
    lib.crl_encoder_workspace_bytes.argtypes = [P(CrlEncoderShape), c_int32, P(c_int64)]
    lib.crl_encoder_precise_packed_bytes.argtypes = [P(CrlEncoderShape), P(c_int64)]
    lib.crl_encoder_pack_precise.argtypes = [P(CrlEncoderShape)] + [c_void_p] * 6
    lib.crl_zone_encode_precise.argtypes = [P(CrlEncoderShape), c_int32] + [c_void_p] * 6
    lib.crl_encoder_forward.argtypes = [P(CrlEncoderShape), P(CrlConfig), P(CrlState), c_int32] + [c_void_p] * 8
    lib.crl_encoder_backward_workspace_bytes.argtypes = [P(CrlEncoderShape), c_int32, P(c_int64)]
    lib.crl_zone_encode_backward.argtypes = [P(CrlEncoderShape), c_int32] + [c_void_p] * 11
    lib.crl_frame_capture.argtypes = [P(CrlConfig), P(CrlState), c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_uint32,
                                      c_void_p, c_void_p]
    lib.crl_zone_encode_frames.argtypes = [P(CrlEncoderShape), P(CrlConfig), c_int32] + [c_void_p] * 8
    lib.crl_zone_encode_backward_frames.argtypes = [P(CrlEncoderShape), P(CrlConfig), c_int32] + [c_void_p] * 13
    lib.crl_frames_zone_obs.argtypes = [P(CrlConfig), c_int32] + [c_void_p] * 5
    lib.crl_copy_envs.argtypes = [P(CrlConfig), P(CrlState), P(CrlOut), c_void_p, P(CrlConfig), P(CrlState), P(CrlOut),
                                  c_void_p, c_int32, c_void_p, c_void_p]
    for name in SYMBOLS:
        getattr(lib, name)
    if lib.crl_abi_version() != ABI_VERSION:
        raise RuntimeError('libcrl_b200.so ABI version mismatch; rebuild it')
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError('crl_b200: ' + load().crl_strerror(rc).decode())
