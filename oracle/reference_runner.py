"""Runs the UNMODIFIED reference (/root/reference) as the ground truth.

TEST INFRASTRUCTURE ONLY -- nothing under bsuite_b200/ imports this module.
It works only where /root/reference exists (this container, not the GPU box):
its outputs travel as committed fixtures under tests/golden/ (oracle/gen_golden.py).

How a reference environment is made to consume a per-lane Philox stream without
touching its source: every reference constructor forwards its `seed` argument
to `numpy.random.RandomState(seed)` (deep_sea.py:77, catch.py:58, cartpole.py:91,
mountain_car.py:55, memory_chain.py:45, umbrella_chain.py:52, mnist.py:53,
wrappers.py:267,330), and `RandomState` accepts a BitGenerator instance as the
seed.  Passing `numpy.random.Philox(key=[seed, lane], counter=[0,0,0,stream])`
therefore gives the reference numpy's own legacy distribution code over exactly
the stream lane `lane` of the engine consumes.
"""

import hashlib
import os
import struct
import sys
from typing import Any, Dict, Optional

import numpy as np

REFERENCE_ROOT = '/root/reference'
_SHIMS = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'shims')
STREAM_ENV, STREAM_WRAPPER = 0, 1


def reference_available() -> bool:
  return os.path.isdir(os.path.join(REFERENCE_ROOT, 'bsuite'))


def import_reference():
  """Imports and returns the reference's `bsuite` package (with shims for 4 absent pure-Python deps)."""
  if not reference_available():
    raise RuntimeError(f'{REFERENCE_ROOT} is not present on this machine')
  root = REFERENCE_ROOT
  repo_root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  for path in (root, _SHIMS, repo_root):
    if path not in sys.path:
      sys.path.insert(0, path)
  import bsuite  # pylint: disable=import-outside-toplevel
  return bsuite


def philox_bitgen(seed: int, lane: int, stream: int = STREAM_ENV) -> np.random.Philox:
  return np.random.Philox(key=np.array([seed, lane], dtype=np.uint64),
                          counter=np.array([0, 0, 0, stream], dtype=np.uint64))


def lane_seed(rng: str, seed: int, lane: int, stream: int = STREAM_ENV):
  """The `seed` argument to hand to a reference constructor for engine lane `lane`."""
  if rng == 'philox':
    return philox_bitgen(seed, lane, stream)
  if rng == 'mt19937':
    return (seed + lane) % (2**32)   # engine: RandomState(seed + global lane), same integer for the wrapper
  raise ValueError(rng)


# environment class name -> (module path, class name) inside the reference
_CLASSES = {
    'deep_sea': ('bsuite.environments.deep_sea', 'DeepSea'),
    'catch': ('bsuite.environments.catch', 'Catch'),
    'cartpole': ('bsuite.environments.cartpole', 'Cartpole'),
    'cartpole_swingup': ('bsuite.experiments.cartpole_swingup.cartpole_swingup', 'CartpoleSwingup'),
    'mountain_car': ('bsuite.environments.mountain_car', 'MountainCar'),
    'memory_chain': ('bsuite.environments.memory_chain', 'MemoryChain'),
    'bandit': ('bsuite.environments.bandit', 'SimpleBandit'),
    'umbrella_chain': ('bsuite.environments.umbrella_chain', 'UmbrellaChain'),
    'discounting_chain': ('bsuite.environments.discounting_chain', 'DiscountingChain'),
    'mnist': ('bsuite.environments.mnist', 'MNISTBandit'),
}
_SEEDLESS = ('bandit', 'discounting_chain')   # constructors without a `seed` kwarg


def make_reference_env(env_class: str, kwargs: Dict[str, Any], rng: str, seed: int, lane: int,
                       wrapper: Optional[str] = None, wrapper_arg: float = 0.0, mnist_dir: Optional[str] = None):
  """Builds reference environment `env_class(**kwargs)` wired to engine lane `lane`'s streams."""
  import importlib  # pylint: disable=import-outside-toplevel
  import_reference()
  module_name, class_name = _CLASSES[env_class]
  cls = getattr(importlib.import_module(module_name), class_name)
  kwargs = dict(kwargs)
  if env_class not in _SEEDLESS:
    kwargs['seed'] = lane_seed(rng, seed, lane, STREAM_ENV)
  if env_class == 'mnist':
    env = _make_mnist(cls, kwargs, mnist_dir)
  else:
    env = cls(**kwargs)
  if wrapper is None:
    return env
  from bsuite.utils import wrappers  # pylint: disable=import-outside-toplevel
  wrapper_seed = lane_seed(rng, seed, lane, STREAM_WRAPPER)
  if wrapper == 'noise':
    return wrappers.RewardNoise(env=env, noise_scale=wrapper_arg, seed=wrapper_seed)
  if wrapper == 'scale':
    return wrappers.RewardScale(env=env, reward_scale=wrapper_arg, seed=wrapper_seed)
  raise ValueError(wrapper)


def _make_mnist(cls, kwargs, mnist_dir):
  """MNISTBandit loads from a fixed directory (datasets.py:42); point it at `mnist_dir` for the call."""
  from bsuite.utils import datasets  # pylint: disable=import-outside-toplevel
  original = datasets.load_mnist
  if mnist_dir is not None:
    datasets.load_mnist = lambda directory=mnist_dir: original(directory)
  try:
    return cls(**kwargs)
  finally:
    datasets.load_mnist = original


def run_trace(env, actions: np.ndarray, explicit_reset: bool = False) -> Dict[str, np.ndarray]:
  """Calls env.step(a) for every action (after an optional explicit reset()) and records every TimeStep."""
  step_type, reward, discount, observation = [], [], [], []

  def record(ts):
    step_type.append(int(ts.step_type))
    reward.append(np.nan if ts.reward is None else float(ts.reward))
    discount.append(np.nan if ts.discount is None else float(ts.discount))
    observation.append(np.asarray(ts.observation, dtype=np.float32).copy())

  if explicit_reset:
    record(env.reset())
  for a in actions:
    record(env.step(int(a)))
  info = {k: float(v) for k, v in env.bsuite_info().items()}
  return dict(step_type=np.asarray(step_type, np.int32), reward=np.asarray(reward, np.float64),
              discount=np.asarray(discount, np.float64), observation=np.stack(observation), info=info)


def trace_digest(trace: Dict[str, np.ndarray]) -> str:
  """SHA-256 over every timestep's (<i step_type | <d reward | <d discount | obs bytes); SURVEY.md 8c."""
  h = hashlib.sha256()
  for st, r, d, obs in zip(trace['step_type'], trace['reward'], trace['discount'], trace['observation']):
    h.update(struct.pack('<i', int(st)))
    h.update(struct.pack('<d', float(r)))
    h.update(struct.pack('<d', float(d)))
    h.update(np.ascontiguousarray(obs, dtype=np.float32).tobytes())
  return h.hexdigest()[:16]
