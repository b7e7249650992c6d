"""ctypes binding of the C-ABI declared in include/bgw.h (libbgw.so, built from csrc/ by build.py).

This is the only place the product touches native code.  There is no CPU fallback: if the shared library
is missing or does not load, importing the engine raises.
"""
import ctypes as C
import os

BGW_ABI_VERSION = 5
BGW_MAX_ENCODING = 63
BGW_MAX_AGENTS = 4096
BGW_NONE = 0xFFFF
BGW_RW_COUNT = 8
BGW_STAT_COUNT = 4

# enums (include/bgw.h)
AG_OBSERVING, AG_MOVING, AG_ATTACKING, AG_HEALTH, AG_ORIENT, AG_LEARNER, AG_BLOCKING, AG_AMMO = (1 << i for i in range(8))
ROLE_NONE, ROLE_NAVIGATOR, ROLE_TARGET, ROLE_PACMAN, ROLE_FOOD, ROLE_BADDIE, ROLE_WALL, ROLE_RUNNER = range(8)
PROG_TEAM_BATTLE, PROG_MAZE, PROG_MULTI_MAZE, PROG_PACMAN, PROG_REACH_TARGET, PROG_TRAFFIC, PROG_PACMAN_SIMPLE, PROG_USER = range(8)
ROLE_SCRIPTED_BADDIE = 16
MOVE_NONE, MOVE_BOX, MOVE_CROSS, MOVE_DRIFT = range(4)
ATTACK_NONE, ATTACK_BINARY, ATTACK_ENCODING, ATTACK_RESTRICTED, ATTACK_SELECTIVE = range(5)
BGW_MAX_VICTIMS, BGW_MAX_SIMATT = 256, 16
OBS_POSITION_CENTERED, OBS_ABSOLUTE, OBS_STACKED = range(3)
DONE_ACTIVE, DONE_ONE_TEAM, DONE_TARGET_AGENT, DONE_TARGET_DESTROYED = (1 << i for i in range(4))
MANAGER_ALL_STEP, MANAGER_TURN_BASED, MANAGER_DYNAMIC_ORDER = range(3)
RW_ATTACK_FAIL, RW_KILL, RW_DIE, RW_MOVE_FAIL, RW_ENTROPY, RW_TARGET, RW_EAT_FOOD = range(7)
ST_ACTIVE, ST_IN_GRID, ST_DONE_REPORTED, ST_NEXT = 1, 2, 4, 8
ST_ORIENT_SHIFT = 4
OUT_DONE, OUT_VALID = 1, 2
ENV_ALL_DONE, ENV_RESET, ENV_TRUNCATED, ENV_ERROR = 1, 2, 4, 8
STAT_AGENT_STEPS, STAT_EPISODES, STAT_KILLS, STAT_ENV_STEPS = range(4)
SITE_PLACE, SITE_HEALTH, SITE_ORIENT, SITE_ACC, SITE_SUBSET, SITE_OBS, SITE_ACTION, SITE_MAZE, SITE_AMMO, SITE_SCRIPT, \
    SITE_ORDER, SITE_PLACE_ORDER, SITE_PROGRAM = range(13)

_p = C.c_void_p


class BgwSpec(C.Structure):
    _fields_ = [
        ('abi_version', C.c_int32), ('rows', C.c_int32), ('cols', C.c_int32), ('n_agents', C.c_int32),
        ('n_envs', C.c_int32), ('env_offset', C.c_int32), ('program', C.c_int32), ('move_actor', C.c_int32),
        ('attack_actor', C.c_int32), ('observer', C.c_int32), ('observe_self', C.c_int32),
        ('done_mask', C.c_int32), ('manager', C.c_int32), ('ravel_actions', C.c_int32),
        ('no_overlap_at_reset', C.c_int32), ('stacked_attacks', C.c_int32), ('horizon', C.c_int32),
        ('auto_reset', C.c_int32), ('ammo_observer', C.c_int32), ('layout_kind', C.c_int32), ('layout_target', C.c_int32),
        ('cluster_barriers', C.c_int32), ('scatter_free_agents', C.c_int32), ('randomize_placement_order', C.c_int32),
        ('randomize_action_input', C.c_int32), ('position_observer', C.c_int32), ('seed', C.c_uint64),
        ('barrier_encodings', C.c_uint64), ('free_encodings', C.c_uint64), ('reward', C.c_double * BGW_RW_COUNT),
        ('encoding', _p), ('klass', _p), ('role', _p), ('init_row', _p), ('init_col', _p),
        ('init_health', _p), ('init_orient', _p), ('view_range', _p), ('move_range', _p),
        ('attack_range', _p), ('attack_strength', _p), ('attack_accuracy', _p),
        ('simultaneous_attacks', _p), ('target', _p), ('initial_ammo', _p), ('overlap', _p), ('attack_map', _p),
    ]


class BgwState(C.Structure):
    _fields_ = [(n, _p) for n in ('cell', 'next', 'flags', 'health', 'reward_acc', 'episode', 'step',
                                  'env_flags', 'turn', 'error', 'layout', 'stats', 'ammo')]


class BgwDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('n_envs', 'n_agents', 'n_learners', 'obs_h', 'obs_w', 'obs_c',
                                         'obs_stride', 'action_stride', 'threads_per_env', 'envs_per_cta',
                                         'smem_bytes', 'ammo_offset', 'device_layouts', 'position_offset')]


LAYOUT_POSITION_STATE, LAYOUT_MAZE, LAYOUT_TARGET_BARRIERS_FREE = range(3)

EXPORTS = ('bgw_create', 'bgw_destroy', 'bgw_dims', 'bgw_bind_state', 'bgw_reset', 'bgw_observe', 'bgw_specialize', 'bgw_set_program', 'bgw_set_program_vars', 'bgw_step', 'bgw_generate_layouts',
           'bgw_maze_layout_host', 'bgw_use_device_layouts',
           'bgw_sample_actions', 'bgw_step_sampled', 'bgw_rollout_sampled', 'bgw_gather_valid', 'bgw_rng_draw', 'bgw_los_mask', 'bgw_launch_count', 'bgw_last_error',
           'bgw_abi_version')

_LIB = None


def lib_path():
    # BGW_LIB: an alternative build of the same sources (A/B measurements of kernel variants)
    return os.environ.get('BGW_LIB') or os.path.join(os.path.dirname(os.path.abspath(__file__)), 'csrc', 'libbgw.so')


def load():
    """Load libbgw.so (once).  Raises if it has not been built: there is no fallback path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: build the CUDA extension first (python -m abmarl_b200.csrc.build, or "
            f"__graft_entry__.build()).  abmarl_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    h = C.c_void_p
    lib.bgw_create.argtypes = [C.POINTER(BgwSpec), C.c_int, C.POINTER(h)]
    lib.bgw_destroy.argtypes = [h]
    lib.bgw_dims.argtypes = [h, C.POINTER(BgwDims)]
    lib.bgw_bind_state.argtypes = [h, C.POINTER(BgwState)]
    lib.bgw_reset.argtypes = [h, _p, _p, _p]
    lib.bgw_step.argtypes = [h, _p, _p, _p, _p, _p, _p, _p]
    lib.bgw_sample_actions.argtypes = [h, _p, _p]
    lib.bgw_observe.argtypes = [h, _p, _p, _p]
    lib.bgw_observe.restype = C.c_int
    lib.bgw_specialize.argtypes = [h, C.c_char_p]
    lib.bgw_specialize.restype = C.c_int
    lib.bgw_set_program.argtypes = [h, C.c_char_p, C.c_char_p]
    lib.bgw_set_program.restype = C.c_int
    lib.bgw_set_program_vars.argtypes = [h, C.c_int, C.c_int, _p, _p]
    lib.bgw_set_program_vars.restype = C.c_int
    lib.bgw_step_sampled.argtypes = [h, _p, _p, _p, _p, _p, _p, _p]
    lib.bgw_step_sampled.restype = C.c_int
    lib.bgw_rollout_sampled.argtypes = [h, C.c_int, _p, _p, _p, _p, _p, _p, _p]
    lib.bgw_rollout_sampled.restype = C.c_int
    lib.bgw_gather_valid.argtypes = [h] + [_p] * 10
    lib.bgw_gather_valid.restype = C.c_int
    lib.bgw_rng_draw.argtypes = [C.c_uint64] + [C.c_uint32] * 6 + [C.POINTER(C.c_uint32 * 4)]
    lib.bgw_generate_layouts.argtypes = [h, _p, C.c_int, _p]
    lib.bgw_generate_layouts.restype = C.c_int
    lib.bgw_use_device_layouts.argtypes = [h, C.c_int]
    lib.bgw_use_device_layouts.restype = C.c_int
    lib.bgw_maze_layout_host.argtypes = [C.POINTER(BgwSpec), C.c_uint32, C.c_uint32, _p]
    lib.bgw_maze_layout_host.restype = C.c_int
    lib.bgw_los_mask.argtypes = [C.c_int, C.c_int, C.c_int, _p]
    lib.bgw_launch_count.argtypes = [h]
    lib.bgw_launch_count.restype = C.c_uint64
    lib.bgw_last_error.restype = C.c_char_p
    lib.bgw_abi_version.restype = C.c_int
    for name in ('bgw_create', 'bgw_destroy', 'bgw_dims', 'bgw_bind_state', 'bgw_reset', 'bgw_step',
                 'bgw_sample_actions', 'bgw_rng_draw', 'bgw_los_mask'):
        getattr(lib, name).restype = C.c_int
    if lib.bgw_abi_version() != BGW_ABI_VERSION:
        raise RuntimeError("libbgw.so ABI version mismatch; rebuild the extension")
    _LIB = lib
    return lib


def check(rc, lib=None):
    if rc != 0:
        lib = lib or load()
        raise RuntimeError(f"libbgw: {lib.bgw_last_error().decode()} (code {rc})")
