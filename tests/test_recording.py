"""Recorder / CsvLogger: the Logging bookkeeping pinned by the reference's utils/wrappers_test.py:84-121, the log
schedule of wrappers.py:140-147, and CSV files the reference's own csv_load can read."""

import os

import numpy as np
import pytest

import bsuite_b200
from bsuite_b200 import dm_env
from bsuite_b200 import recording
from tests import conftest as cf


class _Cycle(dm_env.Environment):
  """Replays canned timesteps (the FakeEnvironment of utils/wrappers_test.py:32-79)."""
  bsuite_num_episodes = 1000

  def __init__(self, timesteps):
    self._timesteps, self._i = timesteps, 0

  def _next(self):
    ts = self._timesteps[self._i % len(self._timesteps)]
    self._i += 1
    return ts

  def reset(self):
    self._i = 0
    return self._next()

  def step(self, action):
    return self._next()

  def observation_spec(self):
    return dm_env.specs.Array((), np.float32)

  def action_spec(self):
    return dm_env.specs.DiscreteArray(1)

  def bsuite_info(self):
    return {}


class _Rows:
  def __init__(self):
    self.rows = []

  def write(self, data):
    self.rows.append(dict(data))


def test_bookkeeping_matches_reference_wrapper_test():
  """The one numeric pin in the reference repo: 5 episodes of rewards (1, 2, 3) with log_every=True."""
  timesteps = [dm_env.restart([]), dm_env.transition(1, []), dm_env.transition(2, []), dm_env.termination(3, [])]
  rows = _Rows()
  env = recording.Recorder(_Cycle(timesteps), rows, log_every=True)
  for _ in range(5):
    ts = env.reset()
    while not ts.last():
      ts = env.step(0)
  assert rows.rows == [dict(steps=3 * i, episode=i, total_return=6 * i, episode_len=3, episode_return=6)
                       for i in range(1, 6)]


def test_log_schedule():
  points = [n for n in range(1, 10001) if recording.is_log_point(n)]
  assert points[:14] == [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 14, 17, 20]
  assert len(points) == 49 and points[-1] == 10000          # SURVEY.md section 5: 49 writes in 10 000 episodes


def test_csv_recorder_round_trip(tmp_path):
  env = bsuite_b200.load_and_record_to_csv('catch/3', str(tmp_path), device='cpu', seed=1)
  assert env.bsuite_num_episodes == 10000 and env.raw_env is not env
  rng = np.random.RandomState(0)
  for _ in range(25):
    ts = env.reset()
    while not ts.last():
      ts = env.step(int(rng.randint(3)))
  path = tmp_path / 'bsuite_id_-_catch-3.csv'
  lines = path.read_text().strip().splitlines()
  assert lines[0] == 'steps,episode,total_return,episode_len,episode_return,total_regret'
  episodes = [int(line.split(',')[1]) for line in lines[1:]]
  assert episodes == [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 14, 17, 20, 25]
  assert all(line.split(',')[3] == '9' for line in lines[1:])        # catch episodes are 9 transitions
  with pytest.raises(ValueError, match='already exists'):
    bsuite_b200.load_and_record_to_csv('catch/3', str(tmp_path), device='cpu')
  with pytest.raises(ValueError, match='logging_mode'):
    bsuite_b200.load_and_record('catch/3', str(tmp_path), logging_mode='sqlite', device='cpu')


def test_reference_csv_load_reads_our_files(tmp_path):
  """Same seed, same actions -> ours writes the file the reference's Logging + csv_logging wrote (same name, same
  bytes; tests/golden/reference/recording.npz), so the reference's csv_load.load_bsuite parses ours as its own."""
  want = cf.load_reference('recording')['csv/catch_seed_5.json']
  ours_dir = str(tmp_path / 'ours')
  ours = recording.Recorder(bsuite_b200.make('catch', device='cpu', seed=5),
                            recording.CsvLogger('catch/0', ours_dir))
  rng, rewards = np.random.RandomState(1), []
  for _ in range(30):
    a = ours.reset()
    while not a.last():
      a = ours.step(int(rng.randint(3)))
      rewards.append(a.reward)
  assert rewards == want['rewards']
  assert os.listdir(ours_dir) == [want['file_name']]
  with open(os.path.join(ours_dir, want['file_name'])) as fh:
    assert fh.read() == want['text']


def test_terminal_logger_formats_like_the_reference():
  """`k1 = v1 | k2 = v2`, keys sorted, integers plain, other numbers with 4 decimals (terminal_logging.py:57-74);
  compared with the line the reference's own formatter made of the same dict."""
  data = {'steps': 12, 'total_return': -3.0, 'episode': np.int64(4), 'episode_return': np.float64(0.123456),
          'name': 'catch/0', 'flag': True}
  lines = []
  recording.TerminalLogger(print_fn=lines.append).write(data)
  assert lines == ['episode = 4 | episode_return = 0.1235 | flag = True | name = catch/0 | steps = 12 | total_return = -3.0000']
  raw = []
  recording.TerminalLogger(pretty_print=False, print_fn=raw.append).write(data)
  assert raw == [data]
  assert cf.load_reference('recording')['terminal/pretty_dict.json'] == lines[0]


def test_load_and_record_modes(tmp_path, capsys):
  """bsuite.load_and_record (bsuite.py:111-123): 'csv' and 'terminal' modes, ValueError otherwise."""
  env = bsuite_b200.load_and_record('bandit/0', str(tmp_path), logging_mode='csv', device='cpu')
  assert isinstance(env, recording.Recorder) and env.bsuite_num_episodes > 0
  env.reset()
  env.step(0)
  env.flush()
  assert [f.name for f in tmp_path.iterdir()] == ['bsuite_id_-_bandit-0.csv']
  with pytest.raises(ValueError):        # the reference refuses to overwrite existing results (csv_logging.py:77-80)
    bsuite_b200.load_and_record_to_csv('bandit/0', str(tmp_path), device='cpu')
  bsuite_b200.load_and_record_to_csv('bandit/0', str(tmp_path), overwrite=True, device='cpu')
  terminal = bsuite_b200.load_and_record('bandit/0', str(tmp_path), logging_mode='terminal', device='cpu')
  terminal.reset()
  terminal.step(1)                        # episode 1 is a log point (wrappers.py:140-147)
  printed = capsys.readouterr().out
  assert 'episode = 1 |' in printed and 'total_regret = ' in printed
  with pytest.raises(ValueError, match='Unrecognised logging_mode'):
    bsuite_b200.load_and_record('bandit/0', str(tmp_path), logging_mode='sqlite', device='cpu')


# ---------------------------------------------------------------------------- batched, device-side log rows
_BATCHED_DEVICES = [pytest.param('cpu', id='host'),
                    pytest.param('cuda', id='cuda', marks=[pytest.mark.gpu, pytest.mark.runs_last])]


def _reference_rows(bsuite_id, lane):
  """Rows the reference's own Logging wrapper wrote for one lane (utils/wrappers.py:85-125), recorded with the
  same seed and actions as the tests below (tests/golden/reference/recording.npz)."""
  ref = cf.load_reference('recording')
  columns = ref[f'{bsuite_id}/columns.json']
  return [dict(zip(columns, row)) for row in ref[f'{bsuite_id}/rows'][lane, :ref[f'{bsuite_id}/counts'][lane]].tolist()]


@pytest.mark.parametrize('device', _BATCHED_DEVICES)
def test_batched_log_rows_equal_the_reference_logging_wrapper_row_for_row(device, tmp_path):
  """VERDICT r01 item 8: 64 lanes x 1 000 episodes of catch.  Every lane's rows, recorded on the device at the
  log-spaced episode counts, equal the rows the reference wrapper writes for the same lane -- and the CSV file
  written from a lane's rows is the one the reference's csv_logging writes for it, byte for byte."""
  import torch
  B, episodes = 64, 1000
  T = episodes * 10                                 # catch: 9 transitions + the auto-reset call per episode
  env = bsuite_b200.load_from_id('catch/0', batch=B, device=device, seed=11, record_rows=True)
  actions = np.random.RandomState(5).randint(3, size=(T, B)).astype(np.int32)
  for t0 in range(0, T, 2000):                      # fused rollouts and single steps mixed
    env.rollout(1999, actions=torch.as_tensor(actions[t0:t0 + 1999]))
    env.step(torch.as_tensor(actions[t0 + 1999]))
  logged = env.logged_rows()
  rows, counts = logged['rows'].cpu().numpy(), logged['counts'].cpu().numpy()
  assert list(logged['columns']) == ['steps', 'episode', 'total_return', 'episode_len', 'episode_return', 'total_regret']
  assert (counts == 36).all()                       # 1, 2, ..., 10, 12, ..., 1000: 10 + 13 + 13 rows
  for lane in range(B):
    want = _reference_rows('catch/0', lane)
    assert len(want) == counts[lane]
    for k, row in enumerate(want):
      got = dict(zip(logged['columns'], rows[k, :, lane]))
      assert {c: float(v) for c, v in row.items()} == got, (lane, k)
  dirs = recording.write_lane_csvs(env, 'catch/0', str(tmp_path), lanes=range(4))
  want = cf.load_reference('recording')['catch/0/lane_2_csv.json']
  assert os.listdir(dirs[2]) == [want['file_name']]
  with open(os.path.join(dirs[2], want['file_name'])) as fh:
    assert fh.read() == want['text']
  with pytest.raises(ValueError, match='already exists'):
    recording.write_lane_csvs(env, 'catch/0', str(tmp_path), lanes=range(2))


@pytest.mark.parametrize('device', _BATCHED_DEVICES)
@pytest.mark.parametrize('bsuite_id,env_class,kwargs,n_act,wrapper,arg', [
    ('cartpole/0', 'cartpole', {}, 3, None, None),                      # info kept in registers between steps
    ('deep_sea_stochastic/0', 'deep_sea', dict(size=10, deterministic=False, mapping_seed=42), 2, None, None),
    ('bandit_scale/3', 'bandit', dict(mapping_seed=3), 11, 'scale', 1.0),
])
def test_batched_log_rows_for_other_families(device, bsuite_id, env_class, kwargs, n_act, wrapper, arg):
  """The reference rows were recorded from `env_class(**kwargs)` with `wrapper` (reward_scale from the sweep
  settings), seed 2, on the same actions."""
  import torch
  B, T = 6, 3000
  env = bsuite_b200.load_from_id(bsuite_id, batch=B, device=device, seed=2, record_rows=True)
  actions = np.random.RandomState(9).randint(n_act, size=(T, B)).astype(np.int32)
  env.rollout(T, actions=torch.as_tensor(actions))
  logged = env.logged_rows()
  rows, counts = logged['rows'].cpu().numpy(), logged['counts'].cpu().numpy()
  for lane in range(B):
    want = _reference_rows(bsuite_id, lane)
    assert len(want) == counts[lane] > 0
    for k, row in enumerate(want):
      for c, v in row.items():
        got = rows[k, list(logged['columns']).index(c), lane]
        assert got == pytest.approx(float(v), abs=1e-6 if env_class == 'cartpole' and device == 'cuda' else 0), (lane, k, c)


# ---------------------------------------------------------------------------- CUDA rows against the host path's rows
# The tests above compare the device-side recorder with the rows the reference's own Logging wrapper wrote; these
# compare the same `__host__ __device__` recorder on CUDA with the engine's host path over more configurations and
# call patterns (two-phase host steps, mid-episode resets).


@pytest.mark.gpu
@pytest.mark.runs_last
@pytest.mark.parametrize('bsuite_id,batch,steps', [('catch/0', 64, 10000), ('cartpole/0', 6, 3000),
                                                   ('deep_sea_stochastic/0', 6, 3000), ('bandit_scale/3', 6, 3000),
                                                   ('deep_sea/11', 70, 4000)])
def test_device_log_rows_equal_the_host_path_rows(bsuite_id, batch, steps):
  import torch
  cuda = bsuite_b200.load_from_id(bsuite_id, batch=batch, device='cuda', seed=11, record_rows=True)
  host = bsuite_b200.load_from_id(bsuite_id, batch=batch, device='cpu', seed=11, record_rows=True)
  actions = np.random.RandomState(5).randint(cuda.num_actions, size=(steps, batch)).astype(np.int32)
  chunk = 997                                         # fused rollouts and single steps mixed
  for t0 in range(0, steps, chunk + 1):
    block = torch.as_tensor(actions[t0:t0 + chunk])
    if len(block):
      cuda.rollout(len(block), actions=block.cuda()); host.rollout(len(block), actions=block)
    if t0 + chunk < steps:
      last = torch.as_tensor(actions[t0 + chunk])
      cuda.step(last.cuda()); host.step(last)
  got, want = cuda.logged_rows(), host.logged_rows()
  assert list(got['columns']) == list(want['columns'])
  counts = want['counts'].numpy()
  np.testing.assert_array_equal(got['counts'].cpu().numpy(), counts)
  assert counts.min() > 0
  got_rows, want_rows = got['rows'].cpu().numpy(), want['rows'].numpy()
  tol = 1e-6 if bsuite_id.startswith('cartpole') else 0
  for lane in range(batch):                           # rows beyond a lane's count are unwritten memory
    np.testing.assert_allclose(got_rows[:counts[lane], :, lane], want_rows[:counts[lane], :, lane], rtol=0, atol=tol,
                               err_msg=f'lane {lane}')
  cuda.close(); host.close()


@pytest.mark.gpu
@pytest.mark.runs_last
def test_device_log_rows_through_host_driven_steps_equal_the_host_path_rows():
  """The two-phase host step (deep_sea N = 32: transitions first, rows written from its phase 1) records the same rows."""
  import torch
  batch, steps = 96, 1500
  cuda = bsuite_b200.load_from_id('deep_sea/11', batch=batch, device='cuda', seed=3, record_rows=True)
  host = bsuite_b200.load_from_id('deep_sea/11', batch=batch, device='cpu', seed=3, record_rows=True)
  pinned = torch.as_tensor(np.random.RandomState(7).randint(2, size=(steps, batch)).astype(np.int32)).pin_memory()
  buffers = cuda.make_host_buffers()
  for t in range(steps):
    cuda.step_host(pinned[t], buffers)
    host.step(pinned[t])
  got, want = cuda.logged_rows(), host.logged_rows()
  counts = want['counts'].numpy()
  np.testing.assert_array_equal(got['counts'].cpu().numpy(), counts)
  assert counts.min() > 0
  for lane in range(batch):
    np.testing.assert_array_equal(got['rows'].cpu().numpy()[:counts[lane], :, lane], want['rows'].numpy()[:counts[lane], :, lane])
  cuda.close(); host.close()


@pytest.mark.gpu
@pytest.mark.runs_last
def test_device_episode_stats_across_mid_episode_resets_equal_the_host_path():
  """tests/test_round2_features.py pins the Logging columns across explicit mid-episode reset() calls to the reference's
  wrapper on the host path (its CUDA variant needs the reference tree); here CUDA against that host path, after
  every call of the same script."""
  import torch
  kwargs, seed, B = dict(rows=6, columns=3), 5, 4
  make = lambda device: bsuite_b200.make('catch', batch=B, device=device, seed=seed,
                                         engine_kwargs=dict(reward_dtype='float64', track_episodes=True), **kwargs)
  cuda, host = make('cuda'), make('cpu')
  rng = np.random.RandomState(0)
  script = ['reset'] + ['step'] * 3 + ['reset'] + ['step'] * 7 + ['reset', 'reset'] + ['step'] * 11 + ['reset'] + ['step'] * 9
  for op in script:
    if op == 'reset':
      got, want = cuda.reset(), host.reset()
    else:
      actions = torch.as_tensor(rng.randint(3, size=B).astype(np.int32))
      got, want = cuda.step(actions.cuda()), host.step(actions)
    np.testing.assert_array_equal(got.step_type.cpu().numpy(), want.step_type.numpy())
    stats_cuda, stats_host = cuda.episode_stats(), host.episode_stats()
    for key in ('steps', 'episode', 'total_return', 'episode_len', 'episode_return'):
      np.testing.assert_array_equal(stats_cuda[key].cpu().numpy(), stats_host[key].numpy(), err_msg=f'{op} {key}')
  cuda.close(); host.close()
