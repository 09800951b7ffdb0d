"""INTEGRATION.md's reference-side binding, executed: `examples/reference_binding_stub.py` (plain ctypes, nothing
from the bsuite_b200 package) reproduces the unmodified reference's deep_sea known answers -- digest, #LAST,
bsuite_info -- and, built the way the reference's own registry builds an environment, its traces."""

import hashlib
import importlib.util
import json
import os
import struct

import numpy as np
import pytest

from tests import conftest as cf


def _stub():
  path = os.path.join(cf.ROOT, 'examples', 'reference_binding_stub.py')
  spec = importlib.util.spec_from_file_location('reference_binding_stub', path)
  module = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(module)
  return module


def _digest(rows):
  h = hashlib.sha256()
  for ts in rows:
    h.update(struct.pack('<i', int(ts.step_type)))
    h.update(struct.pack('<d', float('nan') if ts.reward is None else float(ts.reward)))
    h.update(struct.pack('<d', float('nan') if ts.discount is None else float(ts.discount)))
    h.update(np.ascontiguousarray(ts.observation, dtype=np.float32).tobytes())
  return h.hexdigest()[:16]


def _rows():
  answers = json.load(open(os.path.join(cf.GOLDEN_DIR, 'known_answers.json')))
  return [r for r in answers if r['label'] in ('deep_sea/0', 'deep_sea/11')]


@pytest.mark.parametrize('row', _rows(), ids=lambda r: r['label'])
def test_stub_reproduces_reference_known_answers(row):
  size = {'deep_sea/0': 10, 'deep_sea/11': 32}[row['label']]
  env = _stub().DeepSeaB200(size=size, mapping_seed=42)        # deep_sea/sweep.py:20
  actions = np.random.RandomState(0).randint(2, size=1000)
  rows = [env.reset()] + [env.step(int(a)) for a in actions]
  assert rows[0].first() and rows[0].reward is None and rows[0].discount is None
  assert sum(ts.last() for ts in rows) == row['num_last']
  assert _digest(rows) == row['digest']
  assert {k: float(v) for k, v in env.bsuite_info().items()} == row['info']
  env.close()


def test_stub_registers_in_the_reference():
  """The reference's registry builds an environment as EXPERIMENT_NAME_TO_ENVIRONMENT[name](**sweep.SETTINGS[id]);
  the stub class built that way for 'deep_sea/2', with the reference's own settings for that id, gives the trace the
  reference's class gave (tests/golden/reference/registry.npz)."""
  ref = cf.load_reference('registry')
  stub = _stub()
  actions = np.random.RandomState(3).randint(2, size=300)
  env = stub.DeepSeaB200(**ref['tables.json']['SETTINGS']['deep_sea/2'])
  got = [env.reset()] + [env.step(int(a)) for a in actions]
  env.close()
  assert _digest(got) == ref['deep_sea_2_digest.json']
