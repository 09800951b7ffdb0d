"""Batched agent loop, random agent and trajectory collection (SURVEY.md 8f row 2)."""

import numpy as np
import pytest
import torch

import bsuite_b200
from bsuite_b200 import rollouts
from oracle import bsuite_oracle as oracle
from tests import conftest as cf

DEVICES = [pytest.param('cpu', id='host'), pytest.param('cuda', id='cuda', marks=pytest.mark.gpu)]


@pytest.mark.parametrize('device', DEVICES)
def test_collect_returns_the_reference_trajectory_layout(device):
  env = bsuite_b200.load_from_id('catch/0', batch=48, device=device, seed=5, reward_dtype='float64')
  a = rollouts.collect(env, 25, action_seed=3)
  b = rollouts.collect(env, 10, action_seed=3, last_observation=a.observations[-1])
  assert tuple(a.observations.shape) == (26, 48, 10, 5) and tuple(a.actions.shape) == (25, 48)
  assert torch.equal(b.observations[0], a.observations[-1])
  actions = torch.cat([a.actions, b.actions]).cpu().numpy()
  want = oracle.run_lanes('catch', {}, actions, seed=5)
  np.testing.assert_array_equal(torch.cat([a.observations[1:], b.observations[1:]]).cpu().numpy(), want['observation'])
  np.testing.assert_array_equal(torch.cat([a.rewards, b.rewards]).cpu().numpy(), want['reward'])
  np.testing.assert_array_equal(torch.cat([a.step_types, b.step_types]).cpu().numpy(), want['step_type'])


@pytest.mark.parametrize('device', DEVICES)
def test_batched_run_loop_with_random_agent(device):
  env = bsuite_b200.load_from_id('bandit/0', batch=200, device=device, seed=1, track_episodes=True)
  agent = rollouts.RandomAgent(env.action_spec(), batch=200, device=device, seed=7)
  rollouts.run(agent, env, 400)
  stats = env.episode_stats()
  # bandit: the explicit reset() returns FIRST, then LAST / FIRST alternate for 400 step() calls
  assert float(stats['episode'].min()) == float(stats['episode'].max()) == 200.0
  mean_return = float((stats['total_return'] / stats['episode']).mean())
  assert abs(mean_return - 0.5) < 0.02          # uniform policy over rewards linspace(0, 1, 11)


def test_reference_experiment_loop_runs_unmodified_on_the_adapter():
  """bsuite/baselines/experiment.run + baselines/random/agent.Random(seed=2) on the reference's catch(seed=9): the
  actions that loop took, episode by episode, drive our B = 1 environment through the same reset() / step() calls to
  the same episode ends and the same returns (tests/golden/reference/experiment_loop.npz)."""
  ref = cf.load_reference('experiment_loop')
  ours = bsuite_b200.make('catch', device='cpu', seed=9)
  assert len(ref['episodes.json']) == 40
  for actions in ref['episodes.json']:
    ts = ours.reset()
    for t, action in enumerate(actions):
      assert not ts.last()
      ts = ours.step(action)
      assert ts.last() == (t == len(actions) - 1)
  assert {k: float(v) for k, v in ours.bsuite_info().items()} == ref['info.json']


def test_replay_ring_matches_the_reference_semantics():
  """rollouts.Replay against bsuite/baselines/utils/replay.py: ring overwrite, size, fraction_filled, sample shapes;
  and Trajectory -> (o_tm1, a_tm1, r_t, d_t, o_t) tuples without the restart calls."""
  import numpy as np
  import torch
  import bsuite_b200
  from bsuite_b200 import rollouts
  replay = rollouts.Replay(capacity=5, device='cpu', seed=0)
  for i in range(7):
    replay.add([np.full((2, 2), i, np.float32), i, float(i) / 2])
  assert replay.size == 5 and replay.fraction_filled == 1.0
  obs, ints, floats = replay.sample(64)
  assert obs.shape == (64, 2, 2) and set(ints.tolist()) <= {2, 3, 4, 5, 6} and torch.equal(obs[:, 0, 0].long(), ints)
  assert torch.allclose(floats.double(), ints.double() / 2)
  replay.reset()
  assert replay.size == 0
  env = bsuite_b200.load_from_id('catch/0', batch=6, device='cpu', seed=1)
  traj = rollouts.collect(env, 25)
  big = rollouts.Replay(capacity=1000, device='cpu')
  added = big.add_transitions(traj)
  assert added == int((traj.step_types != 0).sum()) == big.size
  o_tm1, a, r, d, o_t = big.sample(200)
  assert o_tm1.shape == o_t.shape == (200, 10, 5) and a.shape == r.shape == d.shape == (200,)
  assert float(o_tm1.sum(dim=(1, 2)).min()) >= 1.0          # a transition starts from a real board, never from a LAST frame's successor
  # the tuples are the trajectory's own: every sampled (o_tm1, o_t) pair is adjacent in some lane
  pairs = {(traj.observations[t, b].numpy().tobytes(), traj.observations[t + 1, b].numpy().tobytes())
           for t in range(25) for b in range(6) if int(traj.step_types[t, b]) != 0}
  assert all((x.numpy().tobytes(), y.numpy().tobytes()) in pairs for x, y in zip(o_tm1[:50], o_t[:50]))
