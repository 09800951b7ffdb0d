"""Test configuration: marker registration, library build check, shared helpers."""

import functools
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, 'tests', 'golden')
REFERENCE_DIR = os.path.join(GOLDEN_DIR, 'reference')


def pytest_configure(config):
  config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')
  config.addinivalue_line('markers', 'runs_last: scheduled after every other test of the session (a CUDA fault in it '
                                     'cannot poison the context of tests that were known to pass)')


def _have_cuda() -> bool:
  import torch
  return torch.cuda.is_available()


def pytest_collection_modifyitems(config, items):
  items.sort(key=lambda item: 1 if 'runs_last' in item.keywords else 0)      # stable: everything else keeps its order
  if _have_cuda():
    return
  skip = pytest.mark.skip(reason='no CUDA device in this container')
  for item in items:
    if 'gpu' in item.keywords:
      item.add_marker(skip)


@pytest.fixture(scope='session', autouse=True)
def _library_is_built():
  """The engine has no fallback: make sure the shared library exists (build it here if not)."""
  from bsuite_b200 import _lib
  if not os.path.exists(_lib.LIB_PATH):
    from bsuite_b200 import build
    build.build_library()
  _lib.load()


@pytest.fixture(scope='session')
def mnist_dir(tmp_path_factory):
  """Synthetic idx-ubyte files identical to the ones oracle/gen_golden.py fed the reference."""
  from bsuite_b200 import datasets
  meta = dict(seed=0, num_train=256, num_test=16)
  path = str(tmp_path_factory.mktemp('mnist'))
  datasets.write_synthetic_mnist(path, meta['num_train'], meta['num_test'], meta['seed'])
  os.environ[datasets.ENV_VAR] = path
  return path


def golden_case_names():
  return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith('.npz'))


def load_golden(name):
  data = np.load(os.path.join(GOLDEN_DIR, name + '.npz'))
  meta = json.loads(bytes(data['meta']).decode())
  return meta, data


@functools.lru_cache(maxsize=None)
def load_reference(name):
  """What the unmodified reference returned for a test's inputs (tests/golden/reference/<name>.npz, recorded by
  oracle/gen_reference_checks.py): arrays by key, the payloads of `.json` keys decoded."""
  data = np.load(os.path.join(REFERENCE_DIR, name + '.npz'))
  return {k: json.loads(bytes(data[k]).decode()) if k.endswith('.json') else data[k] for k in data.files}


def none_nan(x):
  """A timestep's reward or discount as the fixtures store it: None (FIRST) as NaN."""
  return np.nan if x is None else float(x)


# float-dynamics families: north_star tolerance 1e-6 (libm vs CUDA sin/cos/log differ in the last ulp)
FLOAT_FAMILIES = ('cartpole', 'cartpole_swingup', 'mountain_car')
FLOAT_TOL = 1e-6
