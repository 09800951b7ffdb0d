"""Randomised differential test: engine vs oracle over randomly drawn configurations.

The fixtures under tests/golden/ pin hand-picked cases against the reference itself; this test sweeps the
configuration space (sizes, lengths, bit widths, wrappers, seeds, batch sizes, lane offsets, mid-episode resets,
fused vs single-step calls) against the pinned oracle.  Host path here; the CUDA path runs the same draws on the
GPU box with a smaller count."""

import numpy as np
import pytest
import torch

import bsuite_b200
from oracle import bsuite_oracle as oracle
from tests import conftest as cf


def _draw_case(rng):
  family = rng.choice(['deep_sea', 'catch', 'cartpole', 'cartpole_swingup', 'mountain_car', 'memory_chain', 'bandit',
                       'umbrella_chain', 'discounting_chain'])
  if family == 'deep_sea':
    kwargs = dict(size=int(rng.randint(1, 24)), deterministic=bool(rng.randint(2)), mapping_seed=int(rng.randint(100)),
                  unscaled_move_cost=float(rng.choice([0.01, 0.0, 0.5])))
    if rng.rand() < 0.15:
      kwargs['randomize_actions'] = False
  elif family == 'catch':
    kwargs = dict(rows=int(rng.randint(2, 14)), columns=int(rng.randint(1, 9)))
  elif family == 'cartpole':
    kwargs = dict(height_threshold=float(rng.uniform(0.3, 0.95)), x_threshold=float(rng.uniform(0.5, 4)),
                  max_time=float(rng.choice([0.05, 0.3, 10.])), init_range=float(rng.uniform(0.0, 0.3)))
  elif family == 'cartpole_swingup':
    kwargs = dict(height_threshold=float(rng.uniform(0, 1)), x_reward_threshold=float(rng.uniform(0.05, 1)),
                  move_cost=float(rng.choice([0.1, 0.0, 1.0])), max_time=float(rng.choice([0.2, 10.])))
  elif family == 'mountain_car':
    kwargs = dict(max_steps=int(rng.choice([1, 2, 7, 60, 1000])))
  elif family == 'memory_chain':
    kwargs = dict(memory_length=int(rng.randint(1, 12)), num_bits=int(rng.choice([1, 2, 3, 7, 31, 32, 33, 64])))
  elif family == 'bandit':
    kwargs = dict(mapping_seed=int(rng.randint(1000)), num_actions=int(rng.randint(1, 16)))
  elif family == 'umbrella_chain':
    kwargs = dict(chain_length=int(rng.randint(1, 15)), n_distractor=int(rng.choice([0, 1, 5, 29, 64])))
  else:
    kwargs = dict(mapping_seed=int(rng.randint(50)))
  wrapper, arg = None, 0.0
  roll = rng.rand()
  if roll < 0.2:
    wrapper, arg = 'noise', float(rng.choice([0.1, 1.0, 10.]))
  elif roll < 0.4:
    wrapper, arg = 'scale', float(rng.choice([0.001, 30., 1000.]))
  return dict(family=str(family), kwargs=kwargs, wrapper=wrapper, arg=arg, batch=int(rng.choice([1, 2, 31, 33, 70])),
              steps=int(rng.randint(5, 60)), seed=int(rng.randint(2**31)), offset=int(rng.choice([0, 5, 10**6])),
              rng=str(rng.choice(['philox', 'philox', 'mt19937'])), fused=bool(rng.randint(2)),
              reset_at=sorted(set(int(x) for x in rng.randint(0, 60, size=rng.randint(0, 3)))))


def _check(case, device):
  wrap = {}
  if case['wrapper'] == 'noise':
    wrap['noise_scale'] = case['arg']
  elif case['wrapper'] == 'scale':
    wrap['reward_scale'] = case['arg']
  seed = case['seed'] % (2**32 - 10**6 - 100) if case['rng'] == 'mt19937' else case['seed']
  env = bsuite_b200.make(case['family'], batch=case['batch'], device=device, seed=seed, rng=case['rng'],
                         engine_kwargs=dict(reward_dtype='float64', lane_offset=case['offset']), **wrap, **case['kwargs'])
  T, B = case['steps'], case['batch']
  actions = np.random.RandomState(case['seed'] % 1000).randint(env.num_actions, size=(T, B)).astype(np.int32)
  reset_at = [t for t in case['reset_at'] if t < T]
  got = {k: [] for k in ('step_type', 'reward', 'discount', 'observation')}
  if case['fused'] and not reset_at:
    ts = env.rollout(T, actions=torch.as_tensor(actions))
    got = {k: getattr(ts, k).cpu().numpy() for k in got}
  else:
    for t in range(T):
      ts = env.reset() if t in reset_at else env.step(torch.as_tensor(actions[t]))
      for k in got:
        got[k].append(getattr(ts, k).cpu().numpy().copy())
    got = {k: np.stack(v) for k, v in got.items()}
  want = oracle.run_lanes(case['family'], case['kwargs'], actions, rng=case['rng'], seed=seed, lane_offset=case['offset'],
                          wrapper=case['wrapper'], wrapper_arg=case['arg'], reset_at=reset_at)
  exact = device == 'cpu' or (case['family'] not in cf.FLOAT_FAMILIES and case['wrapper'] != 'noise'
                              and not (case['family'] == 'deep_sea' and not case['kwargs']['deterministic']))
  np.testing.assert_array_equal(got['step_type'], want['step_type'], err_msg=str(case))
  np.testing.assert_array_equal(got['discount'], want['discount'], err_msg=str(case))
  if exact:
    np.testing.assert_array_equal(got['reward'], want['reward'], err_msg=str(case))
    np.testing.assert_array_equal(got['observation'], want['observation'], err_msg=str(case))
  else:
    scale = max(1.0, abs(case['arg'])) if case['wrapper'] else 1.0
    np.testing.assert_allclose(got['reward'], want['reward'], rtol=0, atol=1e-6 * scale, err_msg=str(case))
    np.testing.assert_allclose(got['observation'], want['observation'], rtol=0, atol=1e-6, err_msg=str(case))
  for k, v in env.bsuite_info().items():
    if exact:
      np.testing.assert_array_equal(v.cpu().numpy(), want['info'][k], err_msg=f'{k} {case}')
    else:
      np.testing.assert_allclose(v.cpu().numpy(), want['info'][k], rtol=1e-9, atol=1e-6, err_msg=f'{k} {case}')
  env.close()


@pytest.mark.parametrize('chunk', range(8))
def test_host_path_matches_oracle_on_random_configurations(chunk):
  rng = np.random.RandomState(1000 + chunk)
  for _ in range(30):
    _check(_draw_case(rng), 'cpu')


@pytest.mark.gpu
@pytest.mark.parametrize('chunk', range(4))
def test_cuda_matches_oracle_on_random_configurations(chunk):
  rng = np.random.RandomState(5000 + chunk)
  for _ in range(25):
    _check(_draw_case(rng), 'cuda')


@pytest.mark.parametrize('chunk', range(4))
def test_oracle_matches_live_reference_on_random_configurations(chunk):
  """Widens the oracle's pin beyond the trace fixtures: the same random configuration generator, oracle vs what the
  UNMODIFIED reference returned for each drawn case, lane by lane (tests/golden/reference/random_configurations.npz,
  observations by digest; exact, float families included: both are numpy/libm on the CPU)."""
  from oracle.gen_reference_checks import observation_digest
  recorded = cf.load_reference('random_configurations')[f'chunk_{chunk}.json']
  rng = np.random.RandomState(9000 + chunk)
  for want in recorded:
    case = _draw_case(rng)
    assert case == want['case']
    seed = case['seed'] % (2**32 - 10**6 - 100) if case['rng'] == 'mt19937' else case['seed']
    T = case['steps']
    lanes = min(case['batch'], 3)
    assert len(want['lanes']) == lanes
    for lane, ref in enumerate(want['lanes']):
      env = oracle.OracleEnv(case['family'], case['kwargs'], rng=case['rng'], seed=seed, lane=case['offset'] + lane,
                             wrapper=case['wrapper'], wrapper_arg=case['arg'])
      actions = np.random.RandomState(lane).randint(env.num_actions, size=T)
      observations = []
      for t, a in enumerate(actions):
        st, r, d, o = env.reset() if t in case['reset_at'] else env.step(int(a))
        assert ref['step_type'][t] == st, case
        np.testing.assert_array_equal([cf.none_nan(r), cf.none_nan(d)], [ref['reward'][t], ref['discount'][t]],
                                      err_msg=str(case))
        observations.append(np.asarray(o, np.float32))
      assert observation_digest(np.stack(observations)) == ref['observation_sha256'], case
      assert ref['info'] == {k: float(v) for k, v in env.bsuite_info().items()}
