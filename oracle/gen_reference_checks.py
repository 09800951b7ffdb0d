"""Generates tests/golden/reference/*: what the reference-comparison tests compare against, recorded from the
UNMODIFIED reference so that those tests run without it.

TEST INFRASTRUCTURE ONLY.  Needs the reference's source tree (oracle/reference_runner.py):

    python oracle/gen_reference_checks.py            # regenerates every fixture
    python oracle/gen_reference_checks.py --check    # regenerates in memory and diffs against the committed files

Every fixture is an .npz: arrays under their own keys, and JSON payloads (bsuite_info() dicts, logged rows, spec
tables) as uint8 arrays under keys ending in `.json` (tests/conftest.py: load_reference).  A reward or discount of
None (FIRST timesteps) is stored as NaN.
"""

import argparse
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
sys.path.insert(0, _ROOT)

from oracle import reference_runner as rr  # noqa: E402

OUT_DIR = os.path.join(_ROOT, 'tests', 'golden', 'reference')
LOG_COLUMNS = ('steps', 'episode', 'total_return', 'episode_len', 'episode_return')


def _none_nan(x):
  return np.nan if x is None else float(x)


def _json(obj):
  return np.frombuffer(json.dumps(obj, sort_keys=True).encode(), dtype=np.uint8)


def _info(env):
  return {k: float(v) for k, v in env.bsuite_info().items()}


def _trace(env, actions, reset_at=()):
  """(step_type, reward, discount, observation) of every call, reset() at the indices in `reset_at`."""
  st, rew, disc, obs = [], [], [], []
  for t, a in enumerate(actions):
    ts = env.reset() if t in reset_at else env.step(int(a))
    st.append(int(ts.step_type)); rew.append(_none_nan(ts.reward)); disc.append(_none_nan(ts.discount))
    obs.append(np.asarray(ts.observation))
  return dict(step_type=np.asarray(st, np.int32), reward=np.asarray(rew, np.float64),
              discount=np.asarray(disc, np.float64), observation=np.stack(obs))


class _Rows:
  def __init__(self):
    self.rows = []

  def write(self, data):
    self.rows.append({k: float(v) for k, v in data.items()})


# ---------------------------------------------------------------------------- tests/test_oracle_pinned.py
LIVE_CONFIGS = [
    ('deep_sea', dict(size=14, deterministic=False, mapping_seed=7), None, 0.),
    ('catch', dict(rows=6, columns=4), 'noise', 0.3),
    ('cartpole_swingup', dict(height_threshold=0.1, x_reward_threshold=0.9), None, 0.),
    ('umbrella_chain', dict(chain_length=5, n_distractor=7), 'scale', 30.),
    ('memory_chain', dict(memory_length=3, num_bits=5), None, 0.),
]


def fresh_configurations():
  out = {}
  for env_class, kwargs, wrapper, arg in LIVE_CONFIGS:
    for rng, seed in (('philox', 99), ('mt19937', 3)):
      ref = rr.make_reference_env(env_class, kwargs, rng, seed, lane=2, wrapper=wrapper, wrapper_arg=arg)
      actions = np.random.RandomState(1).randint(int(ref.action_spec().num_values), size=400)
      key = f'{env_class}/{rng}'
      for k, v in _trace(ref, actions).items():
        out[f'{key}/{k}'] = v
      out[f'{key}/info.json'] = _json(_info(ref))
  return out


# ---------------------------------------------------------------------------- tests/test_randomized_differential.py
def observation_digest(observations) -> str:
  """SHA-256 of a lane's observations as float32 bytes: the observations of 100 random configurations would not fit
  a small fixture, their digests do."""
  return hashlib.sha256(np.ascontiguousarray(observations, dtype=np.float32).tobytes()).hexdigest()


def random_configurations():
  from tests import test_randomized_differential as trd  # the test's own case generator
  out = {}
  for chunk in range(4):
    rng = np.random.RandomState(9000 + chunk)
    cases = []
    for _ in range(25):
      case = trd._draw_case(rng)  # pylint: disable=protected-access
      seed = case['seed'] % (2**32 - 10**6 - 100) if case['rng'] == 'mt19937' else case['seed']
      lanes = []
      for lane in range(min(case['batch'], 3)):
        ref = rr.make_reference_env(case['family'], case['kwargs'], case['rng'], seed, case['offset'] + lane,
                                    case['wrapper'], case['arg'])
        actions = np.random.RandomState(lane).randint(int(ref.action_spec().num_values), size=case['steps'])
        trace = _trace(ref, actions, set(case['reset_at']))
        lanes.append(dict({k: trace[k].tolist() for k in ('step_type', 'reward', 'discount')},
                          observation_sha256=observation_digest(trace['observation']), info=_info(ref)))
      cases.append(dict(case=case, lanes=lanes))
    out[f'chunk_{chunk}.json'] = _json(cases)       # one entry per chunk: thousands of small arrays bloat an .npz
  return out


# ---------------------------------------------------------------------------- tests/test_recording.py
def _logged_rows(env_class, kwargs, seed, lane, actions, wrapper=None, arg=None):
  from bsuite.utils import wrappers  # pylint: disable=import-outside-toplevel
  raw = rr.make_reference_env(env_class, kwargs, 'philox', seed, lane, wrapper, arg)
  raw.bsuite_num_episodes = 10000
  sink = _Rows()
  logged = wrappers.Logging(raw, sink)
  for a in actions:
    logged.step(int(a))
  return sink.rows


def _padded(rows_per_lane):
  columns = list(rows_per_lane[0][0])
  counts = np.asarray([len(r) for r in rows_per_lane], np.int32)
  table = np.full((len(rows_per_lane), counts.max(), len(columns)), np.nan)
  for lane, rows in enumerate(rows_per_lane):
    for k, row in enumerate(rows):
      table[lane, k] = [row[c] for c in columns]
  return columns, counts, table


def recording():
  from bsuite.environments import catch as ref_catch  # pylint: disable=import-outside-toplevel
  from bsuite.logging import csv_logging, terminal_logging  # pylint: disable=import-outside-toplevel
  out = {}
  # test_reference_csv_load_reads_our_files: catch(seed=5), 30 episodes of RandomState(1) actions
  with tempfile.TemporaryDirectory() as tmp:
    ref = csv_logging.wrap_environment(ref_catch.Catch(seed=5), 'catch/0', tmp)
    rng, rewards = np.random.RandomState(1), []
    for _ in range(30):
      ts = ref.reset()
      while not ts.last():
        ts = ref.step(int(rng.randint(3)))
        rewards.append(float(ts.reward))
    (name,) = os.listdir(tmp)
    with open(os.path.join(tmp, name)) as fh:
      out['csv/catch_seed_5.json'] = _json(dict(file_name=name, text=fh.read(), rewards=rewards))
  # test_terminal_logger_formats_like_the_reference
  data = {'steps': 12, 'total_return': -3.0, 'episode': np.int64(4), 'episode_return': np.float64(0.123456),
          'name': 'catch/0', 'flag': True}
  out['terminal/pretty_dict.json'] = _json(terminal_logging.pretty_dict(data))
  # test_batched_log_rows_equal_the_reference_logging_wrapper_row_for_row: catch/0, 64 lanes x 10 000 calls
  B, T = 64, 10000
  actions = np.random.RandomState(5).randint(3, size=(T, B)).astype(np.int32)
  columns, counts, table = _padded([_logged_rows('catch', {}, 11, lane, actions[:, lane]) for lane in range(B)])
  out['catch/0/columns.json'], out['catch/0/counts'], out['catch/0/rows'] = _json(columns), counts, table
  with tempfile.TemporaryDirectory() as tmp:       # the reference's own CSV of lane 2
    from bsuite.utils import wrappers  # pylint: disable=import-outside-toplevel
    raw = rr.make_reference_env('catch', {}, 'philox', 11, 2)
    raw.bsuite_num_episodes = 10000
    logged = csv_logging.wrap_environment(raw, 'catch/0', tmp)
    assert isinstance(logged, wrappers.Logging)
    for a in actions[:, 2]:
      logged.step(int(a))
    del logged
    (name,) = os.listdir(tmp)
    with open(os.path.join(tmp, name)) as fh:
      out['catch/0/lane_2_csv.json'] = _json(dict(file_name=name, text=fh.read()))
  # test_batched_log_rows_for_other_families
  from bsuite_b200 import sweep  # pylint: disable=import-outside-toplevel
  for bsuite_id, env_class, kwargs, n_act, wrapper, arg in (
      ('cartpole/0', 'cartpole', {}, 3, None, None),
      ('deep_sea_stochastic/0', 'deep_sea', dict(size=10, deterministic=False, mapping_seed=42), 2, None, None),
      ('bandit_scale/3', 'bandit', dict(mapping_seed=3), 11, 'scale', 1.0)):
    arg = dict(sweep.SETTINGS[bsuite_id]).get('reward_scale', arg)
    actions = np.random.RandomState(9).randint(n_act, size=(3000, 6)).astype(np.int32)
    columns, counts, table = _padded([_logged_rows(env_class, kwargs, 2, lane, actions[:, lane], wrapper, arg)
                                      for lane in range(6)])
    out[f'{bsuite_id}/columns.json'], out[f'{bsuite_id}/counts'], out[f'{bsuite_id}/rows'] = _json(columns), counts, table
  return out


# ---------------------------------------------------------------------------- tests/test_round2_features.py
def mid_episode_resets():
  """catch(6x3), 4 lanes: after every call of the script, how many rows each lane's Logging wrapper (log_every) has
  written and the last of them."""
  from bsuite.utils import wrappers  # pylint: disable=import-outside-toplevel
  kwargs, seed, B = dict(rows=6, columns=3), 5, 4
  refs, sinks = [], []
  for lane in range(B):
    raw = rr.make_reference_env('catch', kwargs, 'philox', seed, lane)
    raw.bsuite_num_episodes = 10**9
    sinks.append(_Rows())
    refs.append(wrappers.Logging(raw, sinks[-1], log_every=True))
  rng = np.random.RandomState(0)
  script = ['reset'] + ['step'] * 3 + ['reset'] + ['step'] * 7 + ['reset', 'reset'] + ['step'] * 11 + ['reset'] + ['step'] * 9
  counts = np.zeros((len(script), B), np.int32)
  last = np.full((len(script), B, len(LOG_COLUMNS)), np.nan)
  for i, op in enumerate(script):
    if op == 'reset':
      for ref in refs:
        ref.reset()
    else:
      actions = rng.randint(3, size=B).astype(np.int32)
      for lane, ref in enumerate(refs):
        ref.step(int(actions[lane]))
    for lane in range(B):
      counts[i, lane] = len(sinks[lane].rows)
      if sinks[lane].rows:
        last[i, lane] = [sinks[lane].rows[-1][c] for c in LOG_COLUMNS]
  return {'script.json': _json(script), 'counts': counts, 'last_row': last}


# ---------------------------------------------------------------------------- tests/test_engine_features.py
def final_logging_rows():
  """catch(5x3) with reward_scale 30, 6 lanes, 85 calls of RandomState(2) actions: the last row of each lane's Logging
  wrapper (log_every) and its total_regret."""
  from bsuite.utils import wrappers  # pylint: disable=import-outside-toplevel
  kwargs, seed, T, T2, B = dict(rows=5, columns=3), 21, 90, 85, 6
  actions = np.random.RandomState(2).randint(3, size=(T, B)).astype(np.int32)
  rows = []
  for lane in range(B):
    raw = rr.make_reference_env('catch', kwargs, 'philox', seed, lane, 'scale', 30.0)
    raw.bsuite_num_episodes = 10**9
    sink = _Rows()
    logged = wrappers.Logging(raw, sink, log_every=True)
    for t in range(T2):
      logged.step(int(actions[t, lane]))
    rows.append(sink.rows[-1])
  return {'rows.json': _json(rows)}


# ---------------------------------------------------------------------------- tests/test_adapters.py
def to_image():
  from bsuite.utils import wrappers  # pylint: disable=import-outside-toplevel
  out = {}
  for size in (1, 2, 3, 4):
    for shape in ((8, 6), (84, 84, 4), (5, 7, 3)):
      values = np.arange(1, size + 1, dtype=np.float32) * 1.5
      out[f'{size}/{"x".join(map(str, shape))}'] = wrappers.to_image(shape, values.reshape(1, size))
  return out


# ---------------------------------------------------------------------------- tests/test_sweep_registry.py
def registry(mnist_dir):
  bsuite = rr.import_reference()
  from bsuite import sweep as ref  # pylint: disable=import-outside-toplevel
  from bsuite.utils import datasets as ref_datasets  # pylint: disable=import-outside-toplevel
  from bsuite_b200 import sweep  # pylint: disable=import-outside-toplevel
  tables = dict(SWEEP=list(ref.SWEEP), TESTING=list(ref.TESTING),
                SETTINGS={k: dict(v) for k, v in ref.SETTINGS.items()}, EPISODES=dict(ref.EPISODES),
                TAGS={k: list(v) for k, v in ref.TAGS.items()},
                EXPERIMENT_NAME_TO_ENVIRONMENT=sorted(bsuite.bsuite.EXPERIMENT_NAME_TO_ENVIRONMENT),
                **{name: list(getattr(ref, name)) for name in ('BANDIT', 'CARTPOLE_SWINGUP', 'DEEP_SEA_STOCHASTIC',
                                                               'UMBRELLA_LENGTH')})
  specs = {}
  original = ref_datasets.load_mnist
  ref_datasets.load_mnist = lambda directory=mnist_dir: original(directory)
  try:
    for ids in sweep.BY_EXPERIMENT.values():
      for bsuite_id in (ids[0], ids[-1]):
        env = bsuite.load_from_id(bsuite_id)
        a, o = env.action_spec(), env.observation_spec()
        specs[bsuite_id] = dict(bsuite_num_episodes=env.bsuite_num_episodes,
                                action=[int(a.num_values), str(np.dtype(a.dtype)), a.name],
                                observation=[list(o.shape), str(np.dtype(o.dtype)), o.name, type(o).__name__],
                                info=sorted(env.bsuite_info()))
  finally:
    ref_datasets.load_mnist = original
  # tests/test_integration_stub.py: deep_sea/2 through the reference's registry, reset() + 300 RandomState(3) steps
  env = bsuite.load_from_id('deep_sea/2')
  actions = np.random.RandomState(3).randint(2, size=300)
  deep_sea_2 = rr.trace_digest(rr.run_trace(env, actions, explicit_reset=True))
  return {'tables.json': _json(tables), 'specs.json': _json(specs), 'deep_sea_2_digest.json': _json(deep_sea_2)}


# ---------------------------------------------------------------------------- tests/test_rollouts.py
def experiment_loop():
  """baselines/experiment.run with baselines/random/agent.Random(seed=2) on catch(seed=9), 40 episodes: the actions
  the agent chose, episode by episode, and the final bsuite_info()."""
  rr.import_reference()
  from bsuite.baselines import experiment  # pylint: disable=import-outside-toplevel
  from bsuite.baselines.random import agent as random_agent  # pylint: disable=import-outside-toplevel
  from bsuite.environments import catch as ref_catch  # pylint: disable=import-outside-toplevel
  env = ref_catch.Catch(seed=9)
  episodes = []
  reset, step = env.reset, env.step

  def logged_reset():
    episodes.append([])
    return reset()

  def logged_step(action):
    episodes[-1].append(int(action))
    return step(action)

  env.reset, env.step = logged_reset, logged_step
  experiment.run(random_agent.Random(env.action_spec(), seed=2), env, num_episodes=40)
  return {'episodes.json': _json(episodes), 'info.json': _json(_info(env))}


def build_all():
  from bsuite_b200 import datasets  # writer of the synthetic idx files (format only; no dynamics)
  rr.import_reference()
  mnist_dir = tempfile.mkdtemp(prefix='bsb_mnist_')
  datasets.write_synthetic_mnist(mnist_dir, 256, 16, 0)   # the files tests/conftest.py:mnist_dir writes
  return {'fresh_configurations': fresh_configurations(), 'random_configurations': random_configurations(),
          'recording': recording(), 'mid_episode_resets': mid_episode_resets(),
          'final_logging_rows': final_logging_rows(), 'to_image': to_image(), 'registry': registry(mnist_dir),
          'experiment_loop': experiment_loop()}


def main():
  parser = argparse.ArgumentParser()
  parser.add_argument('--check', action='store_true')
  args = parser.parse_args()
  os.makedirs(OUT_DIR, exist_ok=True)
  failures = 0
  for name, data in build_all().items():
    path = os.path.join(OUT_DIR, name + '.npz')
    if args.check:
      old = np.load(path)
      same = set(old.files) == set(data) and all(np.array_equal(old[k], data[k], equal_nan=True) for k in data)
      print(('ok   ' if same else 'DIFF ') + name)
      failures += not same
    else:
      np.savez_compressed(path, **data)
      print(f'wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)')
  return failures


if __name__ == '__main__':
  sys.exit(main())
