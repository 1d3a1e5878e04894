"""ctypes binding of libsnk.so (the C ABI in include/snk.h).

The library is the product: if it is missing the import fails loudly -- there is no CPU or
PyTorch fallback for the step path.  Build it with `python __graft_entry__.py` (or
`make -C marl-snake_b200/csrc`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SNK_LIB_PATH') or os.path.join(_HERE, 'libsnk.so')   # override: A/B builds

SNK_ABI_VERSION = 1
SNK_RNG_PHILOX, SNK_RNG_REPLAY = 0, 1
SNK_XFER_RAW, SNK_XFER_PACKED = 0, 1
DEV_ERRORS = {1: 'action outside {0,1,2}', 2: 'replay stream exhausted',
              4: 'replayed draw out of range / replayed spawn overlaps', 8: 'spawn sampling gave up',
              16: 'internal bounds check failed (debug build)',
              32: "a record tile's bulk copy timed out; the tile was skipped",
              64: 'set_state: grid is not walls + fruits + live snakes, or too many fruit cells',
              128: 'a map id was not below the number of wall maps; map 0 was used',
              256: 'snapshot of an env id outside [0, N), or restore from a slot index out of range or a slot of '
                   'another configuration; that env was left unchanged'}
SNK_MAX_MAPS = 256
STAT_NAMES = ('episodes', 'return_sum', 'episode_steps_sum', 'fruits_sum', 'kills_sum', 'deaths',
              'env_steps', 'reserved')


class SnkConfig(C.Structure):
    _fields_ = [('abi_version', C.c_int32), ('device', C.c_int32), ('num_envs', C.c_int32),
                ('height', C.c_int32), ('width', C.c_int32), ('num_snakes', C.c_int32),
                ('snake_length', C.c_int32), ('vision_range', C.c_int32), ('frame_stack', C.c_int32),
                ('num_fruits', C.c_int32), ('auto_reset', C.c_int32), ('done_mode', C.c_int32),
                ('rng_mode', C.c_int32), ('observer', C.c_int32),
                ('seed', C.c_uint64), ('env_id_offset', C.c_uint64),
                ('max_episode_steps', C.c_double),
                ('reward_fruit', C.c_double), ('reward_kill', C.c_double), ('reward_lose', C.c_double),
                ('reward_win', C.c_double), ('reward_time', C.c_double)]


class SnkStepExtra(C.Structure):
    _fields_ = [('finished', C.c_void_p), ('rank', C.c_void_p), ('episode_scores', C.c_void_p),
                ('episode_steps', C.c_void_p), ('episode_fruits', C.c_void_p), ('episode_kills', C.c_void_p)]


class SnkStateView(C.Structure):
    _fields_ = [('grid', C.c_void_p), ('head', C.c_void_p), ('tail', C.c_void_p), ('length', C.c_void_p),
                ('dir', C.c_void_p), ('alive', C.c_void_p), ('alive_counter', C.c_void_p),
                ('episode_length', C.c_void_p), ('cells', C.c_void_p), ('max_cells', C.c_int32)]


# name -> (restype, argtypes); tests check that the library exports every one of these.
PROTOTYPES = {
    'snk_create': (C.c_int, [C.POINTER(SnkConfig), C.POINTER(C.c_void_p)]),
    'snk_create_map': (C.c_int, [C.POINTER(SnkConfig), C.c_void_p, C.POINTER(C.c_void_p)]),
    'snk_create_maps': (C.c_int, [C.POINTER(SnkConfig), C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    'snk_map_ids_dev': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    'snk_num_maps': (C.c_int, [C.c_void_p]),
    'snk_destroy': (C.c_int, [C.c_void_p]),
    'snk_last_error': (C.c_char_p, []),
    'snk_abi_version': (C.c_int, []),
    'snk_obs_shape': (C.c_int, [C.c_void_p, C.POINTER(C.c_int32 * 4)]),
    'snk_obs_bytes': (C.c_size_t, [C.c_void_p]),
    'snk_num_envs': (C.c_int, [C.c_void_p]),
    'snk_algorithmic_bytes_per_env_step': (C.c_size_t, [C.c_void_p]),
    'snk_reset': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'snk_step': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                           C.POINTER(SnkStepExtra), C.c_void_p]),
    'snk_reset_bits': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'snk_step_bits': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.POINTER(SnkStepExtra), C.c_void_p]),
    'snk_step_many': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                C.c_void_p, C.POINTER(SnkStepExtra), C.c_void_p]),
    'snk_reset_grid': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'snk_step_grid': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.POINTER(SnkStepExtra), C.c_void_p]),
    'snk_step_many_grid': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.POINTER(SnkStepExtra), C.c_void_p]),
    'snk_step_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'snk_step_host_info': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(SnkStepExtra)]),
    'snk_step_host_bits': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'snk_reset_host': (C.c_int, [C.c_void_p, C.c_void_p]),
    'snk_note_stream': (C.c_int, [C.c_void_p, C.c_void_p]),
    'snk_set_host_transport': (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    'snk_get_host_transport': (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'snk_pack_obs': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'snk_widen_bits_host': (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    'snk_alloc_obs': (C.c_int, [C.c_int, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]),
    'snk_free_obs': (C.c_int, [C.c_void_p]),
    'snk_get_state': (C.c_int, [C.c_void_p, C.POINTER(SnkStateView), C.c_void_p]),
    'snk_set_state': (C.c_int, [C.c_void_p, C.POINTER(SnkStateView), C.c_void_p, C.c_void_p]),
    'snk_checkpoint_bytes': (C.c_size_t, [C.c_void_p]),
    'snk_checkpoint_save': (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    'snk_checkpoint_load': (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    'snk_snapshot_bytes': (C.c_size_t, [C.c_void_p]),
    'snk_snapshot': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    'snk_restore': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p]),
    'snk_set_replay': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    'snk_replay_cursors': (C.c_int, [C.c_void_p, C.c_void_p]),
    'snk_device_errors': (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.c_int]),
    'snk_stats_dev': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    'snk_stats': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    'snk_spawn_count': (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    'snk_spawn_cells': (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64]),
    'snk_spawn_count_map': (C.c_int64, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    'snk_spawn_cells_map': (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} is missing: the Snake-v1 step path is a CUDA library with no CPU fallback. '
            'Build it with `python __graft_entry__.py` or `make -C marl-snake_b200/csrc`.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError here = library/header mismatch
        fn.restype, fn.argtypes = res, args
    if lib.snk_abi_version() != SNK_ABI_VERSION:
        raise ImportError('libsnk.so ABI version mismatch; rebuild it')
    return lib


lib = _load()


class SnkError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise SnkError(f'libsnk error {rc}: {lib.snk_last_error().decode()}')
