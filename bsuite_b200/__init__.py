"""bsuite_b200: a B200-native batched engine for bsuite's environment dynamics.

Public surface (mirrors `bsuite/__init__.py:18-24` and `bsuite/bsuite.py`):

  load_from_id(bsuite_id)                      -> B = 1 dm_env.Environment (drop-in)
  load_from_id(bsuite_id, batch=B, device=...) -> BatchedEnvironment (torch tensors)
  load(experiment_name, kwargs, ...)           -> same, from explicit kwargs
  make(environment_class, batch=..., **kwargs) -> construct a raw environment class
  sweep                                        -> SETTINGS / SWEEP / TAGS / TESTING / EPISODES
  EXPERIMENT_NAME_TO_ENVIRONMENT               -> experiment name -> loader
  SweepBatch(ids, lanes=B, record_rows=True)   -> many bsuite_ids at once; .scores() per lane
  Scorer(envs_by_id).run()                     -> per-lane scores / finished / tag averages (scoring)

The compute lives in `libbsuite_b200.so` (hand-written sm_100a CUDA behind the C
ABI of include/bsuite_b200.h); importing this package does not load it, creating
an environment does, and that raises if the library has not been built.
"""

import sys as _sys

try:  # prefer the real dm_env when it is installed
  import dm_env  # type: ignore  # noqa: F401
except ImportError:  # this image: use the bundled compatible module
  from bsuite_b200 import dm_env_compat as dm_env  # noqa: F401
_sys.modules.setdefault('bsuite_b200.dm_env', dm_env)

from bsuite_b200 import sweep  # noqa: E402,F401
from bsuite_b200.registry import (  # noqa: E402,F401
    EXPERIMENT_NAME_TO_ENVIRONMENT,
    load,
    load_and_record,
    load_and_record_to_csv,
    load_and_record_to_terminal,
    load_from_id,
    make,
    unpack_bsuite_id,
)
from bsuite_b200.environment import BatchedEnvironment, DmEnvAdapter, StepBuffers  # noqa: E402,F401
from bsuite_b200 import scoring  # noqa: E402,F401
from bsuite_b200.scoring import Scorer  # noqa: E402,F401
from bsuite_b200.suite import SweepBatch  # noqa: E402,F401

__version__ = '0.1.0'
