"""Engine features beyond single steps: fused rollouts with on-device actions, Logging accumulators,
state snapshots, edge cases (ragged batches, B = 1, unaligned tiles).  Each test runs on the explicit host path
here and on the CUDA path on the GPU box (-m gpu), always checked against the oracle."""

import numpy as np
import pytest
import torch

import bsuite_b200
from oracle import bsuite_oracle as oracle
from tests import conftest as cf

DEVICES = [pytest.param('cpu', id='host'), pytest.param('cuda', id='cuda', marks=pytest.mark.gpu)]


def _np(t):
  return t.cpu().numpy()


@pytest.mark.parametrize('device', DEVICES)
@pytest.mark.parametrize('env_class,kwargs,batch', [
    ('deep_sea', dict(size=10, mapping_seed=42), 77),          # ragged: 2 full warps + 13 lanes
    ('deep_sea', dict(size=7, deterministic=False, mapping_seed=1), 33),   # odd N: unaligned tiles
    ('catch', dict(), 45),
    ('catch', dict(rows=3, columns=3), 1),
    ('umbrella_chain', dict(chain_length=4, n_distractor=5), 40),
    ('memory_chain', dict(memory_length=3, num_bits=64), 9),    # maximum context width
    ('discounting_chain', dict(mapping_seed=1), 65),
    ('bandit', dict(mapping_seed=5), 31),
    ('umbrella_chain', dict(chain_length=3, n_distractor=300), 70),   # 303-float rows: 77 KB stage per warp
    ('catch', dict(rows=20, columns=20), 50),                        # 400-float boards: 102 KB stage per warp
    ('deep_sea', dict(size=100, mapping_seed=2), 40),                # 40 KB tiles: beyond the staged bulk path
])
def test_rollout_with_device_sampled_actions_matches_oracle(device, env_class, kwargs, batch):
  """Actions sampled ON DEVICE by the Philox action stream; `random_actions` is the host mirror; the whole
  trajectory must equal the oracle fed the same actions, for every lane (integer families: bit-exact)."""
  T, seed, action_seed, offset = 37, 123, 9, 1000
  env = bsuite_b200.make(env_class, batch=batch, device=device, seed=seed,
                         engine_kwargs=dict(reward_dtype='float64', lane_offset=offset), **kwargs)
  mirror = env.random_actions(T, action_seed=action_seed)
  out = env.make_buffers(T, with_actions=True)
  ts = env.rollout(T, action_seed=action_seed, out=out)
  np.testing.assert_array_equal(_np(out.actions), mirror)
  assert mirror.min() >= 0 and mirror.max() < env.num_actions
  want = oracle.run_lanes(env_class, kwargs, mirror, rng='philox', seed=seed, lane_offset=offset)
  np.testing.assert_array_equal(_np(ts.step_type), want['step_type'])
  np.testing.assert_array_equal(_np(ts.observation), want['observation'])
  np.testing.assert_array_equal(_np(ts.discount), want['discount'])
  if env_class == 'deep_sea' and not kwargs.get('deterministic', True) and device != 'cpu':
    np.testing.assert_allclose(_np(ts.reward), want['reward'], rtol=1e-12, atol=1e-12)   # log() in randn
  else:
    np.testing.assert_array_equal(_np(ts.reward), want['reward'])
  for k, v in env.bsuite_info().items():
    np.testing.assert_array_equal(_np(v), want['info'][k], err_msg=k)
  # a second rollout continues both the environment and the action stream
  assert env.steps_done == T
  ts2 = env.rollout(5, action_seed=action_seed)
  mirror2 = env.random_actions(5, action_seed=action_seed, first_step=T)
  want2 = oracle.run_lanes(env_class, kwargs, np.concatenate([mirror, mirror2]), rng='philox', seed=seed, lane_offset=offset)
  np.testing.assert_array_equal(_np(ts2.step_type), want2['step_type'][T:])
  np.testing.assert_array_equal(_np(ts2.observation), want2['observation'][T:])
  env.close()


@pytest.mark.parametrize('device', DEVICES)
def test_action_sampler_is_uniform_and_shard_invariant(device):
  env = bsuite_b200.load_from_id('catch/0', batch=4096, device=device, seed=0)
  acts = env.random_actions(64, action_seed=3)
  counts = np.bincount(acts.ravel(), minlength=3) / acts.size
  assert np.all(np.abs(counts - 1 / 3) < 0.01)
  shard = bsuite_b200.load_from_id('catch/0', batch=100, device=device, seed=0, lane_offset=1000)
  np.testing.assert_array_equal(shard.random_actions(64, action_seed=3), acts[:, 1000:1100])


@pytest.mark.parametrize('device', DEVICES)
def test_state_snapshot_restores_trajectory(device):
  """get/set_state (checkpoint-resume; SURVEY.md 8f row 4): restoring a snapshot replays the same future."""
  env = bsuite_b200.load_from_id('catch_noise/3', batch=50, device=device, seed=4, track_episodes=True,
                                 reward_dtype='float64')
  actions = torch.as_tensor(np.random.RandomState(0).randint(3, size=(40, 50)).astype(np.int32))
  env.rollout(13, actions=actions[:13])
  snapshot = env.state_dict()
  a = env.rollout(27, actions=actions[13:])
  a = {k: _np(getattr(a, k)).copy() for k in ('step_type', 'reward', 'observation')}
  info_a = {k: _np(v).copy() for k, v in env.bsuite_info().items()}
  env.load_state_dict(snapshot)
  assert env.steps_done == 13
  b = env.rollout(27, actions=actions[13:])
  for k in a:
    np.testing.assert_array_equal(a[k], _np(getattr(b, k)))
  for k, v in env.bsuite_info().items():
    np.testing.assert_array_equal(info_a[k], _np(v))
  other = bsuite_b200.load_from_id('catch_noise/3', batch=50, device=device, seed=5)
  with pytest.raises(ValueError):
    other.load_state_dict(snapshot)


@pytest.mark.parametrize('device', DEVICES)
def test_episode_stats_match_reference_logging_wrapper(device):
  """The per-lane Logging accumulators (utils/wrappers.py:85-110) against the same bookkeeping applied to the oracle
  trace, and against the rows the reference's own wrapper wrote (tests/golden/reference/final_logging_rows.npz)."""
  kwargs, seed, T, B = dict(rows=5, columns=3), 21, 90, 6
  env = bsuite_b200.make('catch', batch=B, device=device, seed=seed, reward_scale=30.0,
                         engine_kwargs=dict(reward_dtype='float64', track_episodes=True), **kwargs)
  actions = np.random.RandomState(2).randint(3, size=(T, B)).astype(np.int32)
  env.rollout(T, actions=torch.as_tensor(actions))
  stats = {k: _np(v) for k, v in env.episode_stats().items()}
  want = oracle.run_lanes('catch', kwargs, actions, rng='philox', seed=seed, wrapper='scale', wrapper_arg=30.0)
  for lane in range(B):
    steps = episode = ep_len = 0
    total = ep_ret = 0.0
    for t in range(T):
      st, r = want['step_type'][t, lane], want['reward'][t, lane]
      if st == 0:
        ep_len, ep_ret = 0, 0.0            # zeroed when the next episode starts
        continue
      steps += 1; ep_len += 1
      ep_ret += r; total += r
      if st == 2:
        episode += 1
    got = [stats[k][lane] for k in ('steps', 'episode', 'total_return', 'episode_len', 'episode_return')]
    assert got == [steps, episode, total, ep_len, ep_ret]
  # The reference's own Logging wrapper writes its row at LAST timesteps; compare the engine's columns at exactly
  # such a moment (T2 chosen so that every lane's final call is a LAST: catch episodes are 5 calls).
  T2 = 85
  env2 = bsuite_b200.make('catch', batch=B, device=device, seed=seed, reward_scale=30.0,
                          engine_kwargs=dict(reward_dtype='float64', track_episodes=True), **kwargs)
  ts = env2.rollout(T2, actions=torch.as_tensor(actions[:T2]))
  assert np.all(_np(ts.step_type)[-1] == 2)
  stats2 = {k: _np(v) for k, v in env2.episode_stats().items()}
  finals = cf.load_reference('final_logging_rows')['rows.json']
  assert len(finals) == B
  for lane, final in enumerate(finals):
    for key in ('steps', 'episode', 'total_return', 'episode_len', 'episode_return'):
      assert final[key] == stats2[key][lane], key
    assert final['total_regret'] == _np(env2.bsuite_info()['total_regret'])[lane]


@pytest.mark.parametrize('device', DEVICES)
def test_unsupported_configurations_are_rejected(device):
  from bsuite_b200 import _lib
  with pytest.raises(_lib.EngineError, match='num_bits'):
    bsuite_b200.make('memory_chain', batch=4, device=device, memory_length=2, num_bits=65)
  with pytest.raises(_lib.EngineError, match='size'):
    bsuite_b200.make('deep_sea', batch=4, device=device, size=300)
  env = bsuite_b200.load_from_id('catch/0', batch=4, device=device)
  with pytest.raises(ValueError, match='shape'):
    env.step(torch.zeros(5, dtype=torch.int32))


@pytest.mark.parametrize('device', DEVICES)
@pytest.mark.parametrize('with_obs', [False, True])
def test_step_host_matches_step(device, with_obs):
  """`bsb_step_host` (host actions in, host scalars out, observation left on the device) == `bsb_step`."""
  a = bsuite_b200.load_from_id('deep_sea_stochastic/3', batch=96, device=device, seed=2)
  b = bsuite_b200.load_from_id('deep_sea_stochastic/3', batch=96, device=device, seed=2)
  host = b.make_host_buffers(with_observation=with_obs)
  actions = torch.as_tensor(np.random.RandomState(3).randint(2, size=(40, 96)).astype(np.int32))
  if device != 'cpu':
    actions = actions.pin_memory()
  for t in range(40):
    want = a.step(actions[t])
    got, dev_obs = b.step_host(actions[t], host)
    np.testing.assert_array_equal(_np(got.step_type), _np(want.step_type))
    np.testing.assert_array_equal(_np(got.reward), _np(want.reward))
    np.testing.assert_array_equal(_np(got.discount), _np(want.discount))
    np.testing.assert_array_equal(_np(dev_obs), _np(want.observation))
    if with_obs:
      np.testing.assert_array_equal(_np(got.observation), _np(want.observation))


@pytest.mark.gpu
def test_step_reads_pinned_host_actions_and_writes_pinned_host_scalars_in_place():
  """Zero-copy through the ordinary step(): pinned host action tensor in, scalars into pinned host memory, the
  observation on the device; identical to the all-device path."""
  a = bsuite_b200.load_from_id('catch_noise/2', batch=4096, device='cuda', seed=6)
  b = bsuite_b200.load_from_id('catch_noise/2', batch=4096, device='cuda', seed=6)
  mixed = [b.make_mixed_buffers() for _ in range(2)]
  assert mixed[0].reward.is_pinned() and mixed[0].observation.is_cuda
  actions = torch.as_tensor(np.random.RandomState(0).randint(3, size=(30, 4096)).astype(np.int32)).pin_memory()
  for t in range(30):
    want = a.step(actions[t].cuda())
    got = b.step(actions[t], out=mixed[t % 2])
    torch.cuda.synchronize()
    np.testing.assert_array_equal(got.reward.numpy(), want.reward.cpu().numpy())
    np.testing.assert_array_equal(got.step_type.numpy(), want.step_type.cpu().numpy())
    np.testing.assert_array_equal(got.discount.numpy(), want.discount.cpu().numpy())
    assert torch.equal(got.observation, want.observation)


@pytest.mark.parametrize('device', DEVICES)
@pytest.mark.parametrize('batch', [1, 33, 1000])
def test_episode_stat_sums_equal_the_per_lane_columns(device, batch):
  """`bsb_sum_episode_stats` (one reduction kernel) against the per-lane columns of `bsb_read_episode_stats`:
  the five sums are integers or sums of +-1 rewards here, so the comparison is exact."""
  env = bsuite_b200.make('catch', batch=batch, device=device, seed=4,
                         engine_kwargs=dict(track_episodes=True), rows=6, columns=4)
  for T in (1, 40, 23):
    env.rollout(T)
    stats = env.episode_stats()
    want = [float(stats[k].sum()) for k in ('steps', 'episode', 'total_return', 'episode_len', 'episode_return')]
    assert _np(env.episode_stat_sums()).tolist() == want


def test_episode_stat_sums_need_tracking():
  env = bsuite_b200.make('catch', batch=4, device='cpu')
  with pytest.raises(RuntimeError):
    env.episode_stat_sums()


@pytest.mark.gpu
def test_async_log_point_equals_the_synchronous_reduction_on_cuda():
  """distributed.LogPoint: reduction in stream order, result through the ticket; steps issued AFTER the log point
  must not leak into it (the block is a snapshot), and slots are reused safely."""
  import torch
  from bsuite_b200 import distributed as bd
  envs = [bsuite_b200.load_from_id(i, batch=4096, device='cuda', seed=5, track_episodes=True) for i in ('catch/0', 'deep_sea/0')]
  lp = bd.LogPoint(envs, slots=2)
  for round_ in range(6):
    for env in envs:
      env.rollout(9, action_seed=round_)
    want = torch.stack([env.episode_stat_sums() for env in envs])
    ticket = lp.issue()
    for env in envs:                      # work queued behind the log point
      env.rollout(3, action_seed=100 + round_)
    got = lp.result(ticket, host_sync=(round_ % 2 == 0))
    torch.cuda.synchronize()
    assert got.shape == (1, 2, 5) and torch.equal(got[0], want)
  for env in envs:
    env.close()
