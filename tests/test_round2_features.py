"""Round-2 additions: action validation, Logging bookkeeping across mid-episode resets, snapshot fingerprints,
seed precedence, host-driven steps through the mailbox (spin / pre-launch), staged-emitter fallbacks."""

import time

import numpy as np
import pytest
import torch

import bsuite_b200
from bsuite_b200 import _lib

from tests import conftest as cf

DEVICES = ['cpu', pytest.param('cuda', marks=pytest.mark.gpu)]


def _np(t):
  return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------- invalid actions (ADVICE r01)
@pytest.mark.parametrize('bsuite_id,bad', [('bandit/0', 11), ('bandit/0', -1), ('discounting_chain/0', 5),
                                           ('discounting_chain/0', 10**6), ('catch/0', 3), ('deep_sea/0', 2)])
def test_host_path_rejects_out_of_range_actions_without_stepping(bsuite_id, bad):
  env = bsuite_b200.load_from_id(bsuite_id, batch=4, device='cpu', seed=1, track_episodes=True)
  env.reset()
  before = env.state_dict()['blob'].copy()
  actions = torch.zeros(4, dtype=torch.int32)
  actions[2] = bad
  with pytest.raises(_lib.EngineError, match='outside'):
    env.step(actions)
  with pytest.raises(_lib.EngineError, match='outside'):
    env.rollout(3, actions=actions.repeat(3, 1))
  np.testing.assert_array_equal(env.state_dict()['blob'], before)      # nothing moved
  env.step(torch.zeros(4, dtype=torch.int32))                          # and the handle is still usable


def test_single_environment_adapter_rejects_out_of_range_actions():
  env = bsuite_b200.load_from_id('bandit/0', device='cpu', seed=0)
  env.reset()
  for bad in (11, 1000, 10**6, -1):
    with pytest.raises(ValueError, match='action_spec'):
      env.step(bad)
  assert env.step(10).last()


@pytest.mark.gpu
@pytest.mark.parametrize('bsuite_id', ['bandit/0', 'discounting_chain/0', 'catch/0', 'mnist/0'])
def test_device_actions_out_of_range_are_clamped_and_flagged(bsuite_id, mnist_dir):
  env = bsuite_b200.load_from_id(bsuite_id, batch=256, device='cuda', seed=1)
  twin = bsuite_b200.load_from_id(bsuite_id, batch=256, device='cuda', seed=1)
  env.reset(); twin.reset()
  assert not env.invalid_actions_seen()
  good = torch.randint(0, env.num_actions, (256,), dtype=torch.int32, device='cuda')
  bad = good.clone()
  bad[7], bad[100] = 10**6, -5
  clamped = good.clone()
  clamped[7], clamped[100] = env.num_actions - 1, 0
  got, want = env.step(bad), twin.step(clamped)
  assert env.invalid_actions_seen() and not env.invalid_actions_seen()      # reported once, then cleared
  for field in ('step_type', 'reward', 'discount', 'observation'):
    assert torch.equal(getattr(got, field), getattr(want, field)), field
  np.testing.assert_array_equal(env.state_dict()['blob'], twin.state_dict()['blob'])
  # host-driven steps validate up front (pageable) or report after the step (pinned, zero-copy)
  host = env.make_host_buffers()
  with pytest.raises(_lib.EngineError, match='outside'):
    env.step_host(bad.cpu(), host)
  with pytest.raises(_lib.EngineError, match='outside'):
    env.step_host(bad.cpu().pin_memory(), host)
  env.step_host(good.cpu().pin_memory(), host)


# ---------------------------------------------------------------------------- Logging bookkeeping vs the reference
@pytest.mark.parametrize('device', DEVICES)
def test_episode_stats_follow_the_reference_wrapper_across_mid_episode_resets(device):
  """utils/wrappers.py:85-110 zeroes episode_len / episode_return after a LAST only: an explicit reset() in the
  middle of an episode leaves them running.  Columns are compared at every LAST (when the reference writes) with the
  rows the reference's wrapper (log_every) wrote for the same seed and script (tests/golden/reference/
  mid_episode_resets.npz)."""
  ref = cf.load_reference('mid_episode_resets')
  kwargs, seed, B = dict(rows=6, columns=3), 5, 4
  env = bsuite_b200.make('catch', batch=B, device=device, seed=seed,
                         engine_kwargs=dict(reward_dtype='float64', track_episodes=True), **kwargs)
  rng = np.random.RandomState(0)
  script = ['reset'] + ['step'] * 3 + ['reset'] + ['step'] * 7 + ['reset', 'reset'] + ['step'] * 11 + ['reset'] + ['step'] * 9
  assert script == ref['script.json']
  for i, op in enumerate(script):
    if op == 'reset':
      ts = env.reset()
    else:
      actions = rng.randint(3, size=B).astype(np.int32)
      ts = env.step(torch.as_tensor(actions))
    stats = {k: _np(v) for k, v in env.episode_stats().items()}
    for lane in range(B):
      wrote = ref['counts'][i, lane] > (ref['counts'][i - 1, lane] if i else 0)
      assert wrote == (int(_np(ts.step_type)[lane]) == 2), (op, lane)
      if wrote:                                          # the reference has just written a row for this lane
        row = ref['last_row'][i, lane]
        for k, key in enumerate(('steps', 'episode', 'total_return', 'episode_len', 'episode_return')):
          assert row[k] == stats[key][lane], (op, lane, key)
  assert ref['counts'][-1].sum() >= 8


# ---------------------------------------------------------------------------- snapshots and seeds
def test_state_dict_refuses_a_differently_configured_environment():
  a = bsuite_b200.make('umbrella_chain', batch=8, device='cpu', seed=0, chain_length=10, n_distractor=3)
  b = bsuite_b200.make('umbrella_chain', batch=8, device='cpu', seed=0, chain_length=20, n_distractor=3)
  c = bsuite_b200.make('umbrella_chain', batch=8, device='cpu', seed=0, rng='mt19937', chain_length=10, n_distractor=3)
  state = a.state_dict()
  with pytest.raises(ValueError, match='differently configured'):
    b.load_state_dict(state)
  with pytest.raises(ValueError):
    c.load_state_dict(state)
  a.load_state_dict(state)


def test_an_explicit_engine_seed_overrides_the_experiment_default():
  """memory_len fixes seed=0 in its factory (experiments/memory_len/memory_len.py:31-37); without an explicit seed
  that default applies (the reference's behaviour), with one the caller's seed does."""
  def contexts(**kw):
    env = bsuite_b200.load_from_id('memory_size/16', batch=16, device='cpu', **kw)
    return _np(env.reset().observation).copy()
  np.testing.assert_array_equal(contexts(), contexts(seed=0))
  assert not np.array_equal(contexts(seed=0), contexts(seed=1))


# ---------------------------------------------------------------------------- host-driven steps (mailbox)
@pytest.mark.gpu
@pytest.mark.parametrize('bsuite_id', ['deep_sea/11', 'catch_noise/2', 'cartpole/0', 'mnist/0', 'umbrella_length/10'])
@pytest.mark.parametrize('prelaunch', [False, True])
def test_host_driven_steps_through_the_mailbox_equal_ordinary_steps(bsuite_id, prelaunch, mnist_dir):
  """bsb_step_host on pinned buffers: completion through the pinned mailbox (no stream synchronise) and, with
  prelaunch, kernels queued ahead that wait for the doorbell.  Interleaved with ordinary calls (which stand a
  queued launch down) and with a pause longer than the doorbell timeout (the queued launch stands down by itself)."""
  B, T = 4096, 36
  a = bsuite_b200.load_from_id(bsuite_id, batch=B, device='cuda', seed=3, track_episodes=True)
  b = bsuite_b200.load_from_id(bsuite_id, batch=B, device='cuda', seed=3, track_episodes=True)
  host = b.make_host_buffers()
  outs = [b.make_buffers() for _ in range(2)]
  actions = torch.as_tensor(np.random.RandomState(3).randint(a.num_actions, size=(T, B)).astype(np.int32)).pin_memory()
  a.reset(); b.reset()                       # b: no synchronise -- step_host must order itself behind this
  for t in range(T):
    want = a.step(actions[t].cuda())
    if t == 12:                              # an ordinary call in the middle: the queued launch must stand down
      got = b.step(actions[t].cuda())
      got_obs = got.observation
    else:
      if t == 20 and prelaunch:
        time.sleep(0.35)                     # > BSB_DOORBELL_TIMEOUT_MS: the queued launch gives up, the step still happens
      got, got_obs = b.step_host(actions[t], host, out=outs[t % 2], prelaunch=prelaunch)
    tol = cf.FLOAT_TOL if bsuite_id.startswith('cartpole') else 0
    for field in ('step_type', 'reward', 'discount'):
      np.testing.assert_allclose(_np(getattr(got, field)), _np(getattr(want, field)), rtol=0, atol=tol, err_msg=f'{field} t={t}')
    assert torch.equal(got_obs, want.observation), t
  assert a.steps_done == b.steps_done == T + 1
  assert torch.equal(a.episode_stat_sums(), b.episode_stat_sums())
  np.testing.assert_array_equal(a.state_dict()['blob'], b.state_dict()['blob'])
  b.close(); a.close()


@pytest.mark.gpu
def test_closing_an_environment_with_a_queued_launch_does_not_hang():
  env = bsuite_b200.load_from_id('catch/0', batch=1024, device='cuda', seed=0)
  host = env.make_host_buffers()
  actions = torch.zeros(1024, dtype=torch.int32).pin_memory()
  for _ in range(3):
    env.step_host(actions, host, prelaunch=True)
  env.host_flush()
  env.step_host(actions, host, prelaunch=True)
  env.close()
  torch.cuda.synchronize()


# ---------------------------------------------------------------------------- emitters
@pytest.mark.gpu
def test_mnist_pixel_conversion_is_exact_for_every_int8_value(tmp_path):
  """image.astype(float32) / 255 (mnist.py:64) with the int8 reinterpretation (utils/datasets.py:55-56): the TMA
  path's FMA-refined quotient and the vector path's table against numpy, for all 256 byte values."""
  import gzip, struct
  from bsuite_b200 import datasets
  d = str(tmp_path)
  pixels = np.zeros((8, 28, 28), dtype=np.uint8)
  pixels.reshape(8, -1)[:, :256] = np.arange(256, dtype=np.uint8)
  pixels.reshape(8, -1)[:, 256:512] = np.arange(255, -1, -1, dtype=np.uint8)
  for images_name, labels_name in ((datasets.TRAIN_IMAGES, datasets.TRAIN_LABELS), (datasets.TEST_IMAGES, datasets.TEST_LABELS)):
    with gzip.open(f'{d}/{images_name}', 'wb') as fh:
      fh.write(struct.pack('>IIII', 2051, 8, 28, 28)); fh.write(pixels.tobytes())
    with gzip.open(f'{d}/{labels_name}', 'wb') as fh:
      fh.write(struct.pack('>II', 2049, 8)); fh.write(np.arange(8, dtype=np.uint8).tobytes())
  want = pixels.view(np.int8).astype(np.float32) / 255
  import os
  old = os.environ.get(datasets.ENV_VAR)
  os.environ[datasets.ENV_VAR] = d
  try:
    for batch in (64, 20000):                 # small: 8-lane chunks; large: persistent grid
      env = bsuite_b200.load_from_id('mnist/0', batch=batch, device='cuda', seed=0)
      obs = _np(env.reset().observation)
      assert all(any(np.array_equal(o, w) for w in want) for o in obs[:: max(1, batch // 64)])
      zero = _np(env.step(torch.zeros(batch, dtype=torch.int32)).observation)
      assert not zero.any()
      env.close()
  finally:
    if old is None:
      os.environ.pop(datasets.ENV_VAR, None)
    else:
      os.environ[datasets.ENV_VAR] = old


@pytest.mark.gpu
@pytest.mark.parametrize('env_class,kwargs', [('catch', dict(rows=30, columns=31)),
                                              ('umbrella_chain', dict(chain_length=5, n_distractor=900))])
def test_observations_too_long_for_the_shared_memory_stage_fall_back(env_class, kwargs):
  """ADVICE r01: validate() accepts these, so the device must too (host path == device path)."""
  B, T = 70, 14
  dev = bsuite_b200.make(env_class, batch=B, device='cuda', seed=2, **kwargs)
  host = bsuite_b200.make(env_class, batch=B, device='cpu', seed=2, **kwargs)
  actions = torch.as_tensor(np.random.RandomState(1).randint(dev.num_actions, size=(T, B)).astype(np.int32))
  got, want = dev.rollout(T, actions=actions), host.rollout(T, actions=actions)
  for field in ('step_type', 'reward', 'discount', 'observation'):
    np.testing.assert_array_equal(_np(getattr(got, field)), _np(getattr(want, field)), err_msg=field)
  one = dev.step(actions[0].cuda())
  np.testing.assert_array_equal(_np(one.observation), _np(host.step(actions[0]).observation))


@pytest.mark.gpu
@pytest.mark.parametrize('bsuite_id,batch', [('catch/0', 1003), ('deep_sea/3', 77), ('deep_sea/11', 30001)])
def test_two_phase_host_steps_with_ragged_batches_and_float64_rewards(bsuite_id, batch):
  """Two-phase host steps (scalars staged on the device, shipped by copier blocks): batch sizes that leave the
  staging arrays unaligned, a ragged last chunk, the persistent grid (30 001 lanes), float64 rewards."""
  a = bsuite_b200.load_from_id(bsuite_id, batch=batch, device='cuda', seed=9, track_episodes=True, reward_dtype='float64')
  b = bsuite_b200.load_from_id(bsuite_id, batch=batch, device='cuda', seed=9, track_episodes=True, reward_dtype='float64')
  host = b.make_host_buffers()
  T = 25
  actions = torch.as_tensor(np.random.RandomState(1).randint(a.num_actions, size=(T, batch)).astype(np.int32)).pin_memory()
  for t in range(T):
    want = a.step(actions[t].cuda())
    got, obs = b.step_host(actions[t], host)
    for field in ('step_type', 'reward', 'discount'):
      np.testing.assert_array_equal(_np(getattr(got, field)), _np(getattr(want, field)), err_msg=f'{field} t={t}')
    assert torch.equal(obs, want.observation), t
  np.testing.assert_array_equal(a.state_dict()['blob'], b.state_dict()['blob'])


# ---------------------------------------------------------------------------- split host steps (BSB_HOST_NO_WAIT)
@pytest.mark.gpu
@pytest.mark.parametrize('bsuite_id,batch', [('deep_sea/11', 8192 + 37), ('deep_sea_stochastic/3', 300), ('catch/0', 1000),
                                             ('cartpole/0', 777), ('bandit_noise/0', 2)])
def test_two_halves_driven_alternately_are_one_batch(bsuite_id, batch):
  """rollouts.HostHalves: two handles, one step in flight on each, collected alternately -- every lane's trajectory is
  the one it has in a single `batch`-lane environment (lane keys continue across the split)."""
  from bsuite_b200 import rollouts
  T = 30
  halves = rollouts.HostHalves(bsuite_id, batch, device='cuda', seed=5, track_episodes=True)
  whole = bsuite_b200.load_from_id(bsuite_id, batch=batch, device='cuda', seed=5, track_episodes=True)
  assert sum(halves.sizes) == batch and halves.envs[1].lane_offset == halves.sizes[0]
  split = halves.sizes[0]
  actions = torch.as_tensor(np.random.RandomState(2).randint(whole.num_actions, size=(T, batch)).astype(np.int32))
  pinned = [actions[:, :split].contiguous().pin_memory(), actions[:, split:].contiguous().pin_memory()]
  halves.reset(); whole.reset()
  want = [whole.step(actions[t].cuda(), out=whole.make_buffers()) for t in range(T)]
  torch.cuda.synchronize()
  tol = cf.FLOAT_TOL if bsuite_id.startswith('cartpole') else 0

  def check(half, t, ts, obs):
    lanes = slice(0, split) if half == 0 else slice(split, batch)
    for field in ('step_type', 'reward', 'discount'):
      np.testing.assert_allclose(_np(getattr(ts, field)), _np(getattr(want[t], field))[lanes], rtol=0, atol=tol,
                                 err_msg=f'{field} half={half} t={t}')
    torch.cuda.synchronize()
    assert torch.equal(obs, want[t].observation[lanes]), (half, t)

  for half in (0, 1):
    halves.submit(half, pinned[half][0])
  with pytest.raises(RuntimeError):
    halves.submit(0, pinned[0][1])             # one step in flight per half
  assert halves.envs[0].steps_done == 2        # reset + the step in flight
  for t in range(1, T):
    for half in (0, 1):
      check(half, t - 1, *halves.collect(half))
      halves.submit(half, pinned[half][t])
  for half in (0, 1):
    check(half, T - 1, *halves.collect(half))
  sums = halves.envs[0].episode_stat_sums() + halves.envs[1].episode_stat_sums()
  np.testing.assert_allclose(_np(sums), _np(whole.episode_stat_sums()), rtol=1e-12)
  # the same through run(): the policy sees each half's latest timestep
  seen = []
  last = halves.run(lambda half, step, ts: (seen.append((half, step, ts is not None)), pinned[half][step % T])[1], 5)
  assert seen[:2] == [(0, 0, False), (1, 0, False)] and seen[2:4] == [(0, 1, True), (1, 1, True)] and len(seen) == 10
  assert all(e.steps_done == T + 1 + 5 for e in halves.envs) and last[0].reward.shape[0] == split
  halves.close(); whole.close()


@pytest.mark.gpu
def test_a_step_in_flight_is_collected_by_whatever_runs_next_and_reports_bad_actions():
  env = bsuite_b200.load_from_id('deep_sea/11', batch=4096, device='cuda', seed=1, track_episodes=True)
  twin = bsuite_b200.load_from_id('deep_sea/11', batch=4096, device='cuda', seed=1, track_episodes=True)
  host = env.make_host_buffers()
  actions = torch.as_tensor(np.random.RandomState(0).randint(2, size=(4, 4096)).astype(np.int32)).pin_memory()
  env.host_wait()                                               # nothing outstanding: no-op
  for t in range(3):
    env.step_host(actions[t], host, wait=False)                 # never waited for: the next call collects it
    twin.step(actions[t].cuda())
  got = env.step(actions[3].cuda()); want = twin.step(actions[3].cuda())
  assert torch.equal(got.observation, want.observation) and env.steps_done == twin.steps_done == 4
  bad = actions[0].clone().pin_memory(); bad[7] = 5
  env.step_host(bad, host, wait=False)
  with pytest.raises(_lib.EngineError, match='outside'):
    env.host_wait()
  env.host_wait()                                               # reported once
  status = env._lib.bsb_step_host(env._handle.ptr, actions[0].data_ptr(), host.as_outputs(), env.make_buffers().observation.data_ptr(),
                                  None, _lib.HOST_NO_WAIT | _lib.HOST_PRELAUNCH)
  assert status != 0
  env.close(); twin.close()


def test_host_halves_refuses_host_environments():
  from bsuite_b200 import rollouts
  with pytest.raises(ValueError):
    rollouts.HostHalves('catch/0', 64, device='cpu')
  with pytest.raises(ValueError):
    rollouts.HostParts('catch/0', 64, device='cpu', parts=3)
  with pytest.raises(ValueError):
    rollouts.HostParts('catch/0', 64, device='cpu', parts=1)
  with pytest.raises(ValueError):
    rollouts.HostParts('catch/0', 2, device='cpu', parts=3)


@pytest.mark.parametrize('batch,parts', [(65536, 2), (65536, 3), (65536, 4), (8229, 3), (300, 3), (2, 2), (5, 4), (127, 2), (100, 3)])
def test_parts_cover_the_batch_in_whole_warps(batch, parts):
  from bsuite_b200 import rollouts
  sizes = rollouts.split_sizes(batch, parts)
  assert len(sizes) == parts and sum(sizes) == batch and min(sizes) > 0
  if batch >= 64 * parts:
    assert all(size % 32 == 0 for size in sizes[:-1]) and max(sizes) - min(sizes) <= 63
  else:
    assert max(sizes) - min(sizes) <= 1


@pytest.mark.gpu
@pytest.mark.parametrize('bsuite_id,batch,parts', [('deep_sea/11', 8192 + 37, 3), ('deep_sea/11', 4096, 4), ('catch/0', 1000, 3)])
def test_more_than_two_parts_driven_round_robin_are_one_batch(bsuite_id, batch, parts):
  """rollouts.HostParts with 3 / 4 handles: one step in flight on each, collected round-robin; every lane's trajectory
  is the one it has in a single `batch`-lane environment."""
  from bsuite_b200 import rollouts
  T = 20
  group = rollouts.HostParts(bsuite_id, batch, device='cuda', seed=5, track_episodes=True, parts=parts)
  whole = bsuite_b200.load_from_id(bsuite_id, batch=batch, device='cuda', seed=5, track_episodes=True)
  assert sum(group.sizes) == batch and len(group.envs) == parts
  bounds = np.concatenate([[0], np.cumsum(group.sizes)])
  assert [e.lane_offset for e in group.envs] == list(bounds[:-1])
  actions = torch.as_tensor(np.random.RandomState(3).randint(whole.num_actions, size=(T, batch)).astype(np.int32))
  pinned = [actions[:, bounds[p]:bounds[p + 1]].contiguous().pin_memory() for p in range(parts)]
  group.reset(); whole.reset()
  want = [whole.step(actions[t].cuda(), out=whole.make_buffers()) for t in range(T)]
  torch.cuda.synchronize()

  def check(part, t, ts, obs):
    lanes = slice(int(bounds[part]), int(bounds[part + 1]))
    for field in ('step_type', 'reward', 'discount'):
      np.testing.assert_array_equal(_np(getattr(ts, field)), _np(getattr(want[t], field))[lanes], err_msg=f'{field} part={part} t={t}')
    torch.cuda.synchronize()
    assert torch.equal(obs, want[t].observation[lanes]), (part, t)

  for part in range(parts):
    group.submit(part, pinned[part][0])
  for t in range(1, T):
    for part in range(parts):
      check(part, t - 1, *group.collect(part))
      group.submit(part, pinned[part][t])
  for part in range(parts):
    check(part, T - 1, *group.collect(part))
  sums = sum(e.episode_stat_sums() for e in group.envs)
  np.testing.assert_allclose(_np(sums), _np(whole.episode_stat_sums()), rtol=1e-12)
  group.close(); whole.close()
