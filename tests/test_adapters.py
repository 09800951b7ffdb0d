"""Gym call convention and ImageObservation (SURVEY.md 8f row 3)."""

import numpy as np
import pytest
import torch

import bsuite_b200
from bsuite_b200 import adapters
from tests import conftest as cf

DEVICES = [pytest.param('cpu', id='host'), pytest.param('cuda', id='cuda', marks=pytest.mark.gpu)]


def test_gym_adapter_follows_gym_wrapper_semantics():
  """gym_wrapper_test.py:31-53 style: episode runs, done on LAST, reward 0 on FIRST, spaces from the specs."""
  env = adapters.GymAdapter(bsuite_b200.load_from_id('catch/0', device='cpu', seed=2))
  assert env.action_space.n == 3
  space = env.observation_space
  assert space.shape == (10, 5) and space.dtype == np.float32 and float(space.low.min()) == 0. and float(space.high.max()) == 1.
  assert env.reward_range == (-float('inf'), float('inf'))
  with pytest.raises(ValueError):
    env.render()
  obs = env.reset()
  assert space.contains(obs) and not env.game_over and env.bsuite_num_episodes == 10000
  done, steps = False, 0
  while not done:
    obs, reward, done, info = env.step(env.action_space.sample())
    steps += 1
    assert space.contains(obs) and info == {} and (reward == 0. or done)
  assert steps == 9 and env.game_over and reward in (-1., 1.)
  np.testing.assert_array_equal(env.render('rgb_array'), obs)
  unbounded = adapters.GymAdapter(bsuite_b200.load_from_id('cartpole/0', device='cpu', seed=2)).observation_space
  assert np.all(np.isinf(unbounded.low)) and unbounded.shape == (1, 6)


@pytest.mark.parametrize('size', [1, 2, 3, 4])
@pytest.mark.parametrize('shape', [(8, 6), (84, 84, 4), (5, 7, 3)])
def test_small_state_tiling_matches_reference(size, shape):
  values = np.arange(1, size + 1, dtype=np.float32) * 1.5
  got = adapters.to_image(shape, values.reshape(1, size))
  assert got.shape == shape and got.dtype == np.float32
  batched = adapters.to_image(shape, torch.as_tensor(np.stack([values, values * 2])).reshape(2, 1, size), batch_dims=1)
  np.testing.assert_array_equal(batched[0].numpy(), got)
  np.testing.assert_array_equal(batched[1].numpy(), got * 2)
  want = cf.load_reference('to_image')[f'{size}/{"x".join(map(str, shape))}']     # the reference's wrappers.to_image
  np.testing.assert_array_equal(got, want)


def test_large_observations_need_skimage():
  with pytest.raises(NotImplementedError, match='scikit-image|skimage'):
    adapters.to_image((84, 84), np.zeros((10, 5), np.float32))
  with pytest.raises(ValueError):
    adapters.to_image((84, 84), np.zeros((2, 3, 4), np.float32))


@pytest.mark.parametrize('device', DEVICES)
def test_image_observation_on_both_faces(device):
  single = adapters.ImageObservation(bsuite_b200.load_from_id('mountain_car/0', device=device, seed=3), (16, 16, 2))
  assert single.observation_spec().shape == (16, 16, 2) and single.bsuite_num_episodes == 1000
  ts = single.reset()
  assert ts.first() and ts.observation.shape == (16, 16, 2)
  assert ts.observation[0, 0, 0] == ts.observation[7, 7, 1] and ts.observation[0, 0, 0] != ts.observation[8, 0, 0]
  batch = adapters.ImageObservation(bsuite_b200.load_from_id('discounting_chain/0', batch=64, device=device), (8, 8))
  raw = bsuite_b200.load_from_id('discounting_chain/0', batch=64, device=device)
  actions = torch.arange(64, dtype=torch.int32) % 5
  for _ in range(3):
    a, b = batch.step(actions), raw.step(actions)
  assert tuple(a.observation.shape) == (64, 8, 8) and a.observation.device.type == device
  np.testing.assert_array_equal(a.observation[:, 0, 0].cpu().numpy(), b.observation[:, 0, 0].cpu().numpy())
  np.testing.assert_array_equal(a.observation[:, 3, 7].cpu().numpy(), b.observation[:, 0, 1].cpu().numpy())
