"""ctypes binding of `libbsuite_b200.so` (the C ABI in include/bsuite_b200.h).

This is the stub a reference maintainer would add to call the engine from
Python (INTEGRATION.md).  There is deliberately NO fallback: if the shared
library is missing or fails to load, importing the engine raises.
"""

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# BSB_LIBRARY points the binding at another build of the SAME library (tools/host_sanitize.sh: ASan/UBSan build)
LIB_PATH = os.environ.get('BSB_LIBRARY') or os.path.join(_HERE, 'libbsuite_b200.so')

ABI_VERSION = 8
DEVICE_HOST = -1
MAX_INFO = 4
COMM_ID_BYTES = 128

# enum bsb_family
DEEP_SEA, CATCH, CARTPOLE, CARTPOLE_SWINGUP, MOUNTAIN_CAR, MEMORY_CHAIN, BANDIT, UMBRELLA_CHAIN, \
    DISCOUNTING_CHAIN, MNIST = range(10)
FAMILY_NAMES = ('deep_sea', 'catch', 'cartpole', 'cartpole_swingup', 'mountain_car', 'memory_chain',
                'bandit', 'umbrella_chain', 'discounting_chain', 'mnist')
# enum bsb_wrapper
WRAP_NONE, WRAP_REWARD_NOISE, WRAP_REWARD_SCALE = range(3)
# enum bsb_rng_kind
RNG_PHILOX, RNG_MT19937 = range(2)
FLAG_TRACK_EPISODES, FLAG_SCORE_SUMMARY, FLAG_NO_LOG_ROWS = 1, 2, 4          # bsb_config.flags
HOST_ORDER_AFTER_STREAM, HOST_PRELAUNCH, HOST_FENCE_CALLER, HOST_NO_WAIT = 1, 2, 4, 8      # bsb_step_host flags
EPISODE_STAT_FIELDS = ('steps', 'episode', 'total_return', 'episode_len', 'episode_return')


class Config(ctypes.Structure):
  """struct bsb_config."""
  _fields_ = [
      ('family', ctypes.c_int32), ('wrapper', ctypes.c_int32), ('rng_kind', ctypes.c_int32), ('flags', ctypes.c_int32),
      ('size', ctypes.c_int32), ('deterministic', ctypes.c_int32),
      ('rows', ctypes.c_int32), ('columns', ctypes.c_int32),
      ('memory_length', ctypes.c_int32), ('num_bits', ctypes.c_int32),
      ('chain_length', ctypes.c_int32), ('n_distractor', ctypes.c_int32),
      ('num_actions', ctypes.c_int32), ('max_steps', ctypes.c_int32),
      ('num_data', ctypes.c_int32), ('image_rows', ctypes.c_int32), ('image_cols', ctypes.c_int32),
      ('score_experiment', ctypes.c_int32),
      ('unscaled_move_cost', ctypes.c_double),
      ('height_threshold', ctypes.c_double), ('x_threshold', ctypes.c_double), ('timescale', ctypes.c_double),
      ('max_time', ctypes.c_double), ('init_range', ctypes.c_double),
      ('theta_dot_threshold', ctypes.c_double), ('x_reward_threshold', ctypes.c_double), ('move_cost', ctypes.c_double),
      ('noise_scale', ctypes.c_double), ('reward_scale', ctypes.c_double),
      ('table', ctypes.c_void_p), ('table_bytes', ctypes.c_int64),
      ('table2', ctypes.c_void_p), ('table2_bytes', ctypes.c_int64),
      ('log_schedule', ctypes.c_void_p), ('log_schedule_len', ctypes.c_int64),
  ]


class Outputs(ctypes.Structure):
  """struct bsb_outputs."""
  _fields_ = [('observation', ctypes.c_void_p), ('reward', ctypes.c_void_p), ('reward_f64', ctypes.c_void_p),
              ('discount', ctypes.c_void_p), ('step_type', ctypes.c_void_p)]


class ScoreSource(ctypes.Structure):
  """struct bsb_score_source."""
  _fields_ = [('experiment', ctypes.c_int32), ('device', ctypes.c_int32), ('batch', ctypes.c_int64),
              ('n_points', ctypes.c_int32), ('n_columns', ctypes.c_int32),
              ('col_episode', ctypes.c_int32), ('col_value', ctypes.c_int32), ('col_best', ctypes.c_int32),
              ('layout', ctypes.c_int32), ('group_key', ctypes.c_double),
              ('rows', ctypes.c_void_p), ('counts', ctypes.c_void_p)]


NUM_EXPERIMENTS, NUM_TAGS = 23, 7
SCORE_ROWS, SCORE_SUMMARY = 0, 1                    # bsb_score_source.layout
# bsb_read_score_summary: the fields of a score summary, in order
SUMMARY_FIELDS = ('last_episode', 'last_value', 'prev_episode', 'prev_value', 'best', 'first_solved')


EXPORTS = {
    # name: (restype, argtypes)
    'bsb_abi_version': (ctypes.c_int32, []),
    'bsb_last_error': (ctypes.c_char_p, []),
    'bsb_create': (ctypes.c_int32, [ctypes.POINTER(Config), ctypes.c_int64, ctypes.c_int32, ctypes.c_uint64,
                                    ctypes.c_uint64, ctypes.POINTER(ctypes.c_void_p)]),
    'bsb_destroy': (ctypes.c_int32, [ctypes.c_void_p]),
    'bsb_obs_numel': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    'bsb_obs_shape': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    'bsb_num_actions': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]),
    'bsb_batch': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    'bsb_reset': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(Outputs), ctypes.c_void_p]),
    'bsb_step': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(Outputs), ctypes.c_void_p]),
    'bsb_rollout': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_uint64,
                                     ctypes.POINTER(Outputs), ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_random_actions': (ctypes.c_int32, [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int64, ctypes.c_int64,
                                            ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p]),
    'bsb_steps_done': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    'bsb_info_count': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]),
    'bsb_info_name': (ctypes.c_char_p, [ctypes.c_void_p, ctypes.c_int32]),
    'bsb_read_info': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_read_episode_stats': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_sum_episode_stats': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_sum_episode_stats_many': (ctypes.c_int32, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int32, ctypes.c_void_p,
                                                    ctypes.c_void_p]),
    'bsb_log_layout': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    'bsb_read_log_rows': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_read_score_summary': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_state_bytes': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    'bsb_get_state': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    'bsb_set_state': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    'bsb_step_host': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(Outputs), ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_uint32]),
    'bsb_host_flush': (ctypes.c_int32, [ctypes.c_void_p]),
    'bsb_host_wait': (ctypes.c_int32, [ctypes.c_void_p]),
    'bsb_host_timing': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_invalid_actions': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]),
    'bsb_comm_unique_id': (ctypes.c_int32, [ctypes.c_void_p]),
    'bsb_comm_create': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                         ctypes.POINTER(ctypes.c_void_p)]),
    'bsb_comm_destroy': (ctypes.c_int32, [ctypes.c_void_p]),
    'bsb_comm_world': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    'bsb_log_point': (ctypes.c_int32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_int32, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_comm_wait': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_experiment_name': (ctypes.c_char_p, [ctypes.c_int32]),
    'bsb_tag_name': (ctypes.c_char_p, [ctypes.c_int32]),
    'bsb_score_source_from_env': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_double,
                                                   ctypes.POINTER(ScoreSource)]),
    'bsb_score_summarize': (ctypes.c_int32, [ctypes.POINTER(ScoreSource), ctypes.c_void_p, ctypes.c_void_p]),
    'bsb_scorer_create': (ctypes.c_int32, [ctypes.POINTER(ScoreSource), ctypes.c_int32, ctypes.c_int64, ctypes.c_int32,
                                           ctypes.POINTER(ctypes.c_void_p)]),
    'bsb_scorer_run': (ctypes.c_int32, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_void_p]),
    'bsb_scorer_destroy': (ctypes.c_int32, [ctypes.c_void_p]),
    'bsb_launch_count': (ctypes.c_int64, []),
}

_lib = None
_lock = threading.Lock()


class EngineError(RuntimeError):
  """A bsb_* call returned a non-zero status."""


def load():
  """Loads the shared library once; raises if it is missing (no fallback)."""
  global _lib
  with _lock:
    if _lib is not None:
      return _lib
    if not os.path.exists(LIB_PATH):
      raise ImportError(
          f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
          '(or `python -m bsuite_b200.build`). bsuite_b200 has no pure-Python or CPU fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in EXPORTS.items():
      fn = getattr(lib, name)   # AttributeError if the symbol is not exported
      fn.restype = restype
      fn.argtypes = argtypes
    got = lib.bsb_abi_version()
    if got != ABI_VERSION:
      raise ImportError(f'{LIB_PATH} has ABI version {got}, binding expects {ABI_VERSION}; rebuild.')
    _lib = lib
    return _lib


def check(status: int):
  if status != 0:
    message = load().bsb_last_error()
    raise EngineError(f'bsuite_b200 status {status}: {message.decode() if message else "?"}')
