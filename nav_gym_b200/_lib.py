"""Loader for libnavgym_b200.so (the C ABI declared in include/navgym_b200.h).

The library is built in-tree by :func:`build` (called from ``__graft_entry__.build``) with
``nvcc -gencode arch=compute_100a,code=sm_100a``.  There is no CPU fallback: if the shared
object is missing or no CUDA device is present the product raises.
"""
import ctypes as C
import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
SRC = os.path.join(_PKG, 'csrc', 'navgym_b200.cu')
HDR = os.path.join(_ROOT, 'include', 'navgym_b200.h')
SO = os.environ.get('NAVGYM_LIB') or os.path.join(_PKG, 'libnavgym_b200.so')

NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-fmad=false',
              '-shared', '-Xcompiler', '-fPIC', '-std=c++17']

NB = 512
OBS_TAIL = 7
OBS_DIM = NB + OBS_TAIL
HIT_NONE = -32768
MAX_DISC = 64
MAX_SEG = 128
SCHED_BUCKETS = 32
OBS_F32, OBS_F16 = 0, 1   # navgym_step_args_t.obs_format
AUTORESET_NEXT_STEP = 2   # navgym_step_args_t.auto_reset: start ended episodes in the next launch
NS = 10
S_PX, S_PY, S_TH, S_GX, S_GY, S_PPX, S_PPY, S_PYAW, S_PV, S_PW = range(NS)


def _nvcc():
    for c in (shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if c and os.path.exists(c):
            return c
    return None


SO_NOFMA = os.path.join(_PKG, 'libnavgym_b200_nofma.so')  # -DNAVGYM_MARCH_NO_FMA build (tests)


def build_variants(force=False):
    """The alternative builds the parity tests exercise: the march with separately rounded
    multiply and add (see csrc/device_helpers.cuh march_pos)."""
    csrc = os.path.dirname(SRC)
    newest = max([os.path.getmtime(HDR)] + [os.path.getmtime(os.path.join(csrc, f)) for f in os.listdir(csrc)])
    if force or not os.path.exists(SO_NOFMA) or os.path.getmtime(SO_NOFMA) < newest:
        subprocess.check_call([_nvcc()] + NVCC_FLAGS + ['-DNAVGYM_MARCH_NO_FMA', '-o', SO_NOFMA, SRC])
    return SO_NOFMA


def build(force=False, verbose=False):
    """Compile the CUDA library for sm_100a (cross-compiles without a GPU)."""
    if not force and os.path.exists(SO):
        csrc = os.path.dirname(SRC)  # navgym_b200.cu includes the other files of csrc/
        newest = max([os.path.getmtime(HDR)] + [os.path.getmtime(os.path.join(csrc, f)) for f in os.listdir(csrc)])
        if os.path.getmtime(SO) >= newest:
            return SO
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError('nvcc not found: cannot build %s' % SO)
    cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-o', SO, SRC]
    subprocess.check_call(cmd)
    return SO


class MapT(C.Structure):
    _fields_ = [('W', C.c_int32), ('H', C.c_int32), ('edt_offset', C.c_int64),
                ('ox', C.c_double), ('oy', C.c_double), ('res', C.c_double),
                ('spawn_offset', C.c_int64), ('spawn_count', C.c_int32), ('_pad', C.c_int32)]


_P = C.c_void_p


class StepArgs(C.Structure):
    _fields_ = [
        ('dt', C.c_double), ('dist_thresh', C.c_double), ('min_turn_radius', C.c_double),
        ('r_scale', C.c_double), ('r_success', C.c_double), ('r_crash', C.c_double),
        ('r_progress', C.c_double), ('r_forward', C.c_double), ('r_rotation', C.c_double),
        ('r_discomfort', C.c_double),
        ('range_max', C.c_float), ('t_stop', C.c_float),
        ('cell_rule', C.c_int32), ('max_disc', C.c_int32), ('max_seg', C.c_int32),
        ('num_envs', C.c_int32), ('obs_stride', C.c_int32), ('auto_reset', C.c_int32),
        ('max_episode_steps', C.c_int32), ('num_maps', C.c_int32), ('resample_map', C.c_int32),
        ('seed', C.c_uint64), ('env_offset', C.c_int64),
        ('sched_phase', C.c_int32), ('num_scan_stack', C.c_int32),
        ('env_begin', C.c_int32), ('env_count', C.c_int32),
        ('noise_lo', C.c_float), ('noise_hi', C.c_float),
        ('maps', _P), ('edt_pool', _P), ('spawn_pool', _P), ('map_id', _P),
        ('lin', _P), ('thr', _P), ('dthr', _P),
        ('state', _P), ('steps', _P), ('episodes', _P), ('actions', _P),
        ('discs', _P), ('ndisc', _P), ('segs', _P), ('nseg', _P),
        ('noise', _P), ('noise_std', _P),
        ('obs', _P), ('tail64', _P), ('reward', _P),
        ('done', _P), ('is_success', _P), ('is_crash', _P), ('truncated', _P),
        ('distance', _P), ('hits', _P), ('sched', _P),
        ('reward_mirror', _P), ('done_mirror', _P),
        ('discs_reset', _P), ('ndisc_reset', _P), ('segs_reset', _P), ('nseg_reset', _P),
        ('obs_format', C.c_int32), ('_pad', C.c_int32),
    ]


class HerArgs(C.Structure):
    _fields_ = [('dist_thresh', C.c_double), ('r_scale', C.c_double), ('r_success', C.c_double),
                ('r_crash', C.c_double), ('r_progress', C.c_double), ('r_forward', C.c_double),
                ('r_rotation', C.c_double), ('r_discomfort', C.c_double),
                ('count', C.c_int32), ('obs_stride', C.c_int32),
                ('num_scan_stack', C.c_int32), ('_pad', C.c_int32),
                ('obs', _P), ('goals', _P), ('thr', _P), ('dthr', _P), ('reward', _P),
                ('done', _P), ('is_success', _P), ('is_crash', _P), ('distance', _P),
                ('obs_format', C.c_int32), ('_pad2', C.c_int32)]


class ScanArgs(C.Structure):
    _fields_ = [('num_envs', C.c_int32), ('agents_per_env', C.c_int32), ('num_beams', C.c_int32),
                ('max_seg', C.c_int32), ('cell_rule', C.c_int32), ('_pad', C.c_int32),
                ('range_max', C.c_float), ('t_stop', C.c_float),
                ('maps', _P), ('edt_pool', _P), ('map_id', _P), ('nagent', _P), ('pose', _P),
                ('lin', _P), ('segs', _P), ('nseg', _P), ('skip', _P), ('ranges', _P),
                ('robot_state', _P), ('env_mask', _P),
                ('robot_fp', C.c_double * 8), ('agent_fp', C.c_double * 8)]


class PlanMapT(C.Structure):
    _fields_ = [('W', C.c_int32), ('H', C.c_int32), ('num_goals', C.c_int32), ('_pad', C.c_int32),
                ('field_offset', C.c_int64), ('goal_offset', C.c_int64),
                ('free_offset', C.c_int64), ('free_count', C.c_int64),
                ('ox', C.c_double), ('oy', C.c_double), ('res', C.c_double)]


class PlanArgs(C.Structure):
    _fields_ = [('num_envs', C.c_int32), ('max_ped', C.c_int32), ('step', C.c_int32), ('_pad', C.c_int32),
                ('seed', C.c_uint64), ('env_offset', C.c_int64), ('min_goal_dist', C.c_double),
                ('maps', _P), ('fields', _P), ('goals', _P), ('map_id', _P), ('nped', _P), ('pose', _P),
                ('goal_id', _P), ('waypoint', _P), ('goal_local', _P),
                ('respawn', _P), ('free_xy', _P), ('robot_state', _P),
                ('min_robot_dist', C.c_double), ('v_pref_lo', C.c_double), ('v_pref_hi', C.c_double),
                ('has_legs_ratio', C.c_double),
                ('pose_rw', _P), ('v_pref', _P), ('has_legs', _P), ('dist_travelled', _P), ('vel', _P),
                ('prev_action', _P),
                ('cand_pose', _P), ('cand_v_pref', _P), ('cand_legs', _P), ('cand_goal', _P), ('cand_rows', _P),
                ('robot_maps', _P), ('spawn_pool', _P), ('episodes', _P), ('robot_seed', C.c_uint64),
                ('num_maps', C.c_int32), ('resample_map', C.c_int32),
                ('cand_next_spawn', C.c_int32), ('_pad2', C.c_int32),
                ('num_humans_lo', C.c_int32), ('num_humans_hi', C.c_int32),
                ('cand_nped_prev', _P), ('cand_nped', _P), ('nped_out', _P)]


class MoveArgs(C.Structure):
    _fields_ = [('num_envs', C.c_int32), ('max_ped', C.c_int32), ('dt', C.c_double),
                ('nped', _P), ('mean', _P), ('v_pref', _P), ('has_legs', _P), ('pose', _P), ('vel', _P),
                ('dist_travelled', _P), ('prev_action', _P), ('rows', _P)]


PED_F = 16


class ActionBank(C.Structure):
    _fields_ = [('actions', _P), ('rows', C.c_int32), ('num_envs', C.c_int32)]


# navgym_policy_fn (include/navgym_b200.h): user, group, env_begin, env_end, step, obs, reward,
# done, actions
POLICY_FN = C.CFUNCTYPE(None, _P, C.c_int, C.c_int, C.c_int, C.c_int64, _P, _P, _P, _P)


class PedsArgs(C.Structure):
    _fields_ = [('num_envs', C.c_int32), ('max_ped', C.c_int32), ('max_disc', C.c_int32),
                ('max_seg', C.c_int32), ('advance', C.c_int32), ('trunk_mode', C.c_int32),
                ('dt', C.c_float), ('_pad', C.c_int32),
                ('peds', _P), ('nped', _P), ('discs', _P), ('ndisc', _P), ('segs', _P), ('nseg', _P)]


class PolicyParams(C.Structure):
    _fields_ = [('max_n', C.c_int32), ('_pad', C.c_int32),
                ('cv1_w', _P), ('cv1_b', _P), ('cv2_w', _P), ('cv2_b', _P), ('fc1_w', _P), ('fc1_b', _P),
                ('fc2_w', _P), ('fc2_b', _P), ('a1_w', _P), ('a1_b', _P), ('a2_w', _P), ('a2_b', _P),
                ('workspace', _P), ('workspace_bytes', C.c_uint64)]


EXPORTS = [
    'navgym_step_batch', 'navgym_reset_obs_batch', 'navgym_reset_envs', 'navgym_host_pipe_create', 'navgym_host_pipe_destroy',
    'navgym_step_batch_host', 'navgym_step_batch_host_submit', 'navgym_step_batch_host_wait', 'navgym_edt_build', 'navgym_calc_range_many',
    'navgym_raymarching_create_host', 'navgym_raymarching_calc_range_many_host',
    'navgym_raymarching_edt_dev', 'navgym_raymarching_edt_host', 'navgym_raymarching_destroy',
    'navgym_render_in_lidar_host',
    'navgym_error_string', 'navgym_device_count', 'navgym_abi_version', 'navgym_launch_count',
    'navgym_sizeof_step_args', 'navgym_sizeof_map', 'navgym_grid_bfs',
    'navgym_sizeof_her_args', 'navgym_sizeof_peds_args', 'navgym_compute_rewards', 'navgym_peds_advance',
    'navgym_agent_scan_batch', 'navgym_sizeof_scan_args',
    'navgym_peds_plan', 'navgym_sizeof_plan_args', 'navgym_sizeof_plan_map',
    'navgym_peds_move', 'navgym_sizeof_move_args',
    'navgym_host_pipe_groups', 'navgym_host_pipe_group_bounds', 'navgym_host_rollout',
    'navgym_policy_action_bank', 'navgym_export_env', 'navgym_export_env_len', 'navgym_march_is_fused',
    'navgym_policy_workspace_bytes', 'navgym_sizeof_policy_params', 'navgym_policy_create',
    'navgym_policy_destroy', 'navgym_policy_mean', 'navgym_policy_workspace_layout',
]

_lib = None


def load():
    """dlopen the C-ABI library.  Raises if it has not been built (no fallback path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        raise RuntimeError(
            '%s is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nav_gym_b200 has no CPU fallback)' % SO)
    lib = C.CDLL(SO)
    lib.navgym_step_batch.argtypes = [C.POINTER(StepArgs), _P]
    lib.navgym_reset_obs_batch.argtypes = [C.POINTER(StepArgs), _P]
    lib.navgym_reset_envs.argtypes = [C.POINTER(StepArgs), _P, _P]
    lib.navgym_host_pipe_create.restype = _P
    lib.navgym_host_pipe_create.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.navgym_host_pipe_destroy.restype = None
    lib.navgym_host_pipe_destroy.argtypes = [_P]
    lib.navgym_step_batch_host.argtypes = [_P, C.POINTER(StepArgs), _P, _P, _P, _P, _P]
    lib.navgym_step_batch_host_submit.argtypes = [_P, C.POINTER(StepArgs), C.c_int, _P, _P, _P, _P]
    lib.navgym_step_batch_host_wait.argtypes = [_P, C.c_int]
    lib.navgym_host_pipe_groups.argtypes = [_P]
    lib.navgym_host_pipe_group_bounds.argtypes = [_P, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.navgym_host_rollout.argtypes = [_P, C.POINTER(StepArgs), C.c_int64, _P, _P, _P, _P, _P, _P]
    lib.navgym_export_env.argtypes = [C.POINTER(StepArgs), C.c_int, _P, _P]
    lib.navgym_export_env_len.argtypes = [C.c_int]
    lib.navgym_edt_build.argtypes = [_P, C.c_int, C.c_int, _P, _P, _P]
    lib.navgym_calc_range_many.argtypes = [_P, C.c_int, C.c_int, _P, _P, C.c_int, C.c_float,
                                           C.c_float, _P, _P]
    lib.navgym_raymarching_create_host.restype = _P
    lib.navgym_raymarching_create_host.argtypes = [_P, C.c_int, C.c_int, C.c_float]
    lib.navgym_raymarching_calc_range_many_host.argtypes = [_P, _P, _P, C.c_int]
    lib.navgym_raymarching_edt_dev.restype = _P
    lib.navgym_raymarching_edt_dev.argtypes = [_P]
    lib.navgym_raymarching_edt_host.argtypes = [_P, _P]
    lib.navgym_raymarching_destroy.restype = None
    lib.navgym_raymarching_destroy.argtypes = [_P]
    lib.navgym_render_in_lidar_host.argtypes = [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int,
                                                C.c_float, C.c_float]
    lib.navgym_grid_bfs.restype = None
    lib.navgym_grid_bfs.argtypes = [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P]
    lib.navgym_error_string.restype = C.c_char_p
    lib.navgym_error_string.argtypes = [C.c_int]
    lib.navgym_launch_count.restype = C.c_uint64
    lib.navgym_compute_rewards.argtypes = [C.POINTER(HerArgs), _P]
    lib.navgym_peds_advance.argtypes = [C.POINTER(PedsArgs), _P]
    lib.navgym_agent_scan_batch.argtypes = [C.POINTER(ScanArgs), _P]
    lib.navgym_peds_plan.argtypes = [C.POINTER(PlanArgs), _P]
    lib.navgym_peds_move.argtypes = [C.POINTER(MoveArgs), _P]
    lib.navgym_policy_workspace_bytes.restype = C.c_size_t
    lib.navgym_policy_workspace_bytes.argtypes = [C.c_int]
    lib.navgym_policy_create.restype = _P
    lib.navgym_policy_create.argtypes = [C.POINTER(PolicyParams), _P]
    lib.navgym_policy_destroy.restype = None
    lib.navgym_policy_destroy.argtypes = [_P]
    lib.navgym_policy_mean.argtypes = [_P, _P, _P, _P, C.c_int, _P, _P]
    lib.navgym_policy_workspace_layout.restype = None
    lib.navgym_policy_workspace_layout.argtypes = [C.c_int, C.POINTER(C.c_uint64)]
    if (lib.navgym_sizeof_step_args() != C.sizeof(StepArgs) or lib.navgym_sizeof_map() != C.sizeof(MapT)
            or lib.navgym_sizeof_her_args() != C.sizeof(HerArgs)
            or lib.navgym_sizeof_peds_args() != C.sizeof(PedsArgs)
            or lib.navgym_sizeof_scan_args() != C.sizeof(ScanArgs)
            or lib.navgym_sizeof_plan_args() != C.sizeof(PlanArgs)
            or lib.navgym_sizeof_plan_map() != C.sizeof(PlanMapT)
            or lib.navgym_sizeof_move_args() != C.sizeof(MoveArgs)
            or lib.navgym_sizeof_policy_params() != C.sizeof(PolicyParams)):
        raise RuntimeError('libnavgym_b200.so ABI mismatch with nav_gym_b200/_lib.py (rebuild)')
    _lib = lib
    return lib


def check(code, what=''):
    if code != 0:
        msg = load().navgym_error_string(int(code))
        raise RuntimeError('libnavgym_b200 %s failed: CUDA error %d (%s)'
                           % (what, code, msg.decode() if msg else '?'))


def require_device():
    lib = load()
    if lib.navgym_device_count() <= 0:
        raise RuntimeError('nav_gym_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    return lib
