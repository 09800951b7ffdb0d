"""The experiment registry: ids, kwargs, episodes and tags equal the reference's bsuite/sweep.py."""

import numpy as np
import pytest

import bsuite_b200
from bsuite_b200 import experiments
from bsuite_b200 import sweep
from tests import conftest as cf


def test_census():
  """SURVEY.md appendix B: 23 experiments, 468 ids, 13 testing ids."""
  assert len(sweep.SWEEP) == 468 and len(set(sweep.SWEEP)) == 468
  assert len(sweep.BY_EXPERIMENT) == 23
  assert len(sweep.TESTING) == 13 and all(i.endswith('/0') for i in sweep.TESTING)
  assert not any(i.split('/')[0].endswith(('_noise', '_scale')) for i in sweep.TESTING)
  assert len(sweep.DEEP_SEA) == 21 and len(sweep.MEMORY_LEN) == 23 and len(sweep.MEMORY_SIZE) == 17
  assert sweep.SETTINGS['deep_sea/11'] == {'size': 32, 'mapping_seed': 42}
  assert sweep.SETTINGS['memory_size/16'] == {'num_bits': 40}
  assert sweep.SETTINGS['umbrella_length/10'] == {'chain_length': 12, 'n_distractor': 20}
  assert sweep.EPISODES['cartpole/3'] == 1000 and sweep.EPISODES['catch_noise/3'] == 10000
  assert set(sweep.TAGS) == {'basic', 'noise', 'scale', 'exploration', 'credit_assignment', 'generalization', 'memory'}
  assert set(experiments.EXPERIMENT_NAME_TO_SPEC) == set(sweep.BY_EXPERIMENT)
  assert set(bsuite_b200.EXPERIMENT_NAME_TO_ENVIRONMENT) == set(sweep.BY_EXPERIMENT)


def test_settings_are_read_only():
  with pytest.raises(TypeError):
    sweep.SETTINGS['catch/0']['seed'] = 1
  with pytest.raises(TypeError):
    sweep.SETTINGS['new/0'] = {}


def test_id_parsing():
  assert bsuite_b200.unpack_bsuite_id('deep_sea/11') == ('deep_sea', 11)
  for bad in ('deep_sea', 'deep_sea/', '/3', 'a/b/c'):
    with pytest.raises(ValueError):
      bsuite_b200.unpack_bsuite_id(bad)


def test_registry_equals_reference():
  """Against the reference's sweep tables and registry keys (tests/golden/reference/registry.npz)."""
  ref = cf.load_reference('registry')['tables.json']
  assert tuple(ref['SWEEP']) == sweep.SWEEP
  assert tuple(ref['TESTING']) == sweep.TESTING
  assert ref['SETTINGS'] == {k: dict(v) for k, v in sweep.SETTINGS.items()}
  assert ref['EPISODES'] == dict(sweep.EPISODES)
  assert {k: tuple(v) for k, v in ref['TAGS'].items()} == dict(sweep.TAGS)
  assert set(ref['EXPERIMENT_NAME_TO_ENVIRONMENT']) == set(bsuite_b200.EXPERIMENT_NAME_TO_ENVIRONMENT)
  for name in ('BANDIT', 'CARTPOLE_SWINGUP', 'DEEP_SEA_STOCHASTIC', 'UMBRELLA_LENGTH'):
    assert tuple(ref[name]) == tuple(getattr(sweep, name))


def test_every_setting_loads_with_reference_specs(mnist_dir):
  """One id per (experiment, distinct kwargs set) -- bsuite/tests/environments_test.py:25-49 -- on the host path;
  specs and bsuite_num_episodes must equal the reference environment's (tests/golden/reference/registry.npz)."""
  want = cf.load_reference('registry')['specs.json']
  checked = set()
  for ids in sweep.BY_EXPERIMENT.values():
    for bsuite_id in (ids[0], ids[-1]):
      env = bsuite_b200.load_from_id(bsuite_id, device='cpu')
      ref = want[bsuite_id]
      assert env.bsuite_num_episodes == ref['bsuite_num_episodes'], bsuite_id
      a = env.action_spec()
      assert [int(a.num_values), str(np.dtype(a.dtype)), a.name] == ref['action'], bsuite_id
      a = env.observation_spec()
      assert [list(a.shape), str(np.dtype(a.dtype)), a.name, type(a).__name__] == ref['observation'], bsuite_id
      assert sorted(env.bsuite_info()) == ref['info'], bsuite_id
      env.close()
      checked.add(bsuite_id)
  assert checked == set(want)
