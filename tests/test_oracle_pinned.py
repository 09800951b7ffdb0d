"""Pins oracle/bsuite_oracle.py (the CPU restatement) to the UNMODIFIED reference.

The fixtures under tests/golden/ were recorded by oracle/gen_golden.py and
oracle/gen_reference_checks.py from the reference itself.  The oracle must
reproduce every one of them exactly -- including the float-dynamics families,
since both run numpy/libm on the CPU -- and the SURVEY.md 8c known-answer digests.
"""

import hashlib
import json
import os
import struct

import numpy as np
import pytest

from oracle import bsuite_oracle as oracle
from tests import conftest as cf


def _oracle_kwargs(meta, mnist_dir):
  kwargs = dict(meta['kwargs'])
  if meta['env_class'] == 'mnist':
    from bsuite_b200 import datasets
    images, labels = datasets.load_mnist_train(mnist_dir)
    kwargs.update(images=images, labels=labels)
  return kwargs


@pytest.mark.parametrize('name', cf.golden_case_names())
def test_oracle_reproduces_reference_trace(name, mnist_dir):
  meta, data = cf.load_golden(name)
  res = oracle.run_lanes(meta['env_class'], _oracle_kwargs(meta, mnist_dir), data['actions'], rng=meta['rng'],
                         seed=meta['seed'], wrapper=meta['wrapper'], wrapper_arg=meta['wrapper_arg'],
                         reset_at=meta['reset_at'])
  np.testing.assert_array_equal(res['step_type'], data['step_type'])
  np.testing.assert_array_equal(res['reward'], np.nan_to_num(data['reward'], nan=0.0))
  np.testing.assert_array_equal(res['discount'], np.nan_to_num(data['discount'], nan=0.0).astype(np.float32))
  np.testing.assert_array_equal(res['observation'], data['observation'])
  for k, info_name in enumerate(meta['info_names']):
    np.testing.assert_array_equal(res['info'][info_name], data['info'][:, k], err_msg=info_name)


def _digest(rows):
  h = hashlib.sha256()
  for st, r, d, obs in rows:
    h.update(struct.pack('<i', int(st)))
    h.update(struct.pack('<d', float('nan') if r is None else float(r)))
    h.update(struct.pack('<d', float('nan') if d is None else float(d)))
    h.update(np.ascontiguousarray(obs, dtype=np.float32).tobytes())
  return h.hexdigest()[:16]


_ID_TO_CLASS = {   # the kwargs the experiment `load` factories fix (SURVEY.md 8a a13)
    'deep_sea/0': ('deep_sea', dict(size=10, mapping_seed=42), None, 0., 0),
    'deep_sea/11': ('deep_sea', dict(size=32, mapping_seed=42), None, 0., 0),
    'discounting_chain/0': ('discounting_chain', dict(mapping_seed=0), None, 0., 0),
    'bandit/0': ('bandit', dict(mapping_seed=0), None, 0., 0),
    'bandit_scale/0': ('bandit', dict(mapping_seed=0), 'scale', 0.001, 0),
    'memory_len/5': ('memory_chain', dict(memory_length=6, num_bits=1), None, 0., 0),
    'memory_size/16': ('memory_chain', dict(memory_length=2, num_bits=40), None, 0., 0),
    'umbrella_distract/0': ('umbrella_chain', dict(chain_length=20, n_distractor=1), None, 0., 0),
}


def _known_answers():
  return json.load(open(os.path.join(cf.GOLDEN_DIR, 'known_answers.json')))


@pytest.mark.parametrize('row', _known_answers(), ids=lambda r: r['label'][:40])
def test_oracle_known_answer_digests(row):
  """reset() + 1000 step() calls of a single MT19937-seeded environment (SURVEY.md 8c table)."""
  if row['kind'] == 'load_from_id':
    env_class, kwargs, wrapper, arg, seed = _ID_TO_CLASS[row['bsuite_id']]
  else:
    kwargs = dict(row['kwargs'])
    seed = kwargs.pop('seed')
    env_class, wrapper, arg = row['env_class'], None, 0.
  env = oracle.OracleEnv(env_class, kwargs, rng='mt19937', seed=seed, lane=0, wrapper=wrapper, wrapper_arg=arg)
  actions = np.random.RandomState(0).randint(env.num_actions, size=1000)
  rows = [env.reset()] + [env.step(int(a)) for a in actions]
  assert _digest(rows) == row['digest']
  assert sum(1 for r in rows if r[0] == 2) == row['num_last']
  info = {k: float(v) for k, v in env.bsuite_info().items()}
  assert info == row['info']


@pytest.mark.parametrize('env_class,kwargs,wrapper,arg', [
    ('deep_sea', dict(size=14, deterministic=False, mapping_seed=7), None, 0.),
    ('catch', dict(rows=6, columns=4), 'noise', 0.3),
    ('cartpole_swingup', dict(height_threshold=0.1, x_reward_threshold=0.9), None, 0.),
    ('umbrella_chain', dict(chain_length=5, n_distractor=7), 'scale', 30.),
    ('memory_chain', dict(memory_length=3, num_bits=5), None, 0.),
])
def test_oracle_live_against_reference(env_class, kwargs, wrapper, arg):
  """Fresh configurations (not among the trace fixtures above): every call's timestep and the final bsuite_info()
  against what the reference returned for them (tests/golden/reference/fresh_configurations.npz)."""
  want = cf.load_reference('fresh_configurations')
  for rng, seed in (('philox', 99), ('mt19937', 3)):
    key = f'{env_class}/{rng}'
    env = oracle.OracleEnv(env_class, kwargs, rng=rng, seed=seed, lane=2, wrapper=wrapper, wrapper_arg=arg)
    actions = np.random.RandomState(1).randint(env.num_actions, size=400)
    for t, a in enumerate(actions):
      st, r, d, o = env.step(int(a))
      assert want[f'{key}/step_type'][t] == st
      np.testing.assert_array_equal([cf.none_nan(r), cf.none_nan(d)], [want[f'{key}/reward'][t], want[f'{key}/discount'][t]])
      np.testing.assert_array_equal(want[f'{key}/observation'][t], o)
    assert want[f'{key}/info.json'] == {k: float(v) for k, v in env.bsuite_info().items()}
