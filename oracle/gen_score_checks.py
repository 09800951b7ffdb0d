"""Generates tests/golden/reference/scores.npz: the reference's bsuite scores for recorded row tables, so that
tests/test_scoring.py checks the scorer against the UNMODIFIED reference analysis without it.

TEST INFRASTRUCTURE ONLY.  Needs the reference's source tree (oracle/reference_runner.py) and pandas:

    python oracle/gen_score_checks.py            # regenerates the fixture
    python oracle/gen_score_checks.py --check    # regenerates in memory and diffs against the committed file

Two parts:
  syn/*  synthetic row tables for every id of every experiment, 16 lanes: cumulative per-episode outcomes sampled
         at the log schedule; finished, truncated (per id), missing ids and an empty lane; deep_sea crossings early,
         late, never and exactly at the threshold; scores clipped at 0 and 1; mnist with and without rows past
         episode 9000.  Stored: the value columns (the episode column is the schedule), the counts, and what
         summary_analysis.bsuite_score / ave_score_by_tag return for each lane's frame.
  e2e/*  the unmodified reference environments, wrapped in the reference's Logging, driven by the engine's own
         action stream (bsb_random_actions, Philox lane seeds as reference_runner wires them) to NUM_EPISODES;
         the reference's scores of those runs.

A lane's frame is built as csv_load.load_one_result_set builds it (one id after the other, each id's rows
ascending, the CSV dtypes: int64 for the integer columns), then logging_utils.join_metadata.  The reference's
deep_sea.find_solution calls pd.Series.append, which pandas 2 removed: it is pointed at pd.concat here, for the
run of this script only.  plotnine and matplotlib are inert stand-ins (oracle/shims): the scores use neither.
"""

import argparse
import json
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
sys.path.insert(0, _ROOT)

from oracle import reference_runner as rr  # noqa: E402

OUT_PATH = os.path.join(_ROOT, 'tests', 'golden', 'reference', 'scores.npz')
SYN_LANES = 16
SYN_SEED = 20261017
E2E_IDS = ('bandit/0', 'bandit/1', 'bandit/2', 'bandit/3', 'bandit_noise/0', 'bandit_noise/4', 'bandit_noise/8',
           'discounting_chain/0', 'discounting_chain/1', 'discounting_chain/2', 'discounting_chain/3',
           'discounting_chain/4', 'catch/0', 'catch/1')
E2E_LANES, E2E_SEED, E2E_ACTION_SEED = 2, 3, 11
_INT_COLUMNS = ('episode', 'total_bad_episodes', 'total_perfect')      # written as integers (recording.py)


def _json(obj):
  return np.frombuffer(json.dumps(obj, sort_keys=True).encode(), dtype=np.uint8)


def _reference():
  rr.import_reference()
  import pandas as pd  # pylint: disable=import-outside-toplevel
  if not hasattr(pd.Series, 'append'):
    pd.Series.append = lambda self, other: pd.concat([self, other])
  from bsuite.experiments import summary_analysis  # pylint: disable=import-outside-toplevel
  from bsuite.logging import logging_utils  # pylint: disable=import-outside-toplevel
  return pd, summary_analysis, logging_utils


def columns_of(experiment):
  from bsuite_b200 import scoring  # pylint: disable=import-outside-toplevel
  cols = [scoring.VALUE_COLUMNS[experiment]]
  if experiment in scoring.NEEDS_BEST:
    cols.append('best_episode')
  return cols


# ---------------------------------------------------------------------------- synthetic tables
def _per_episode(experiment, good, rng):
  """Per-episode outcomes [lanes, episodes] for each value column, from `good` flags; dyadic values, so every
  cumulative sum is exact."""
  shape = good.shape
  pick = lambda values: np.asarray(values)[rng.randint(len(values), size=shape)]
  if experiment.startswith('bandit'):
    return [np.where(good, 0.0, pick([0.5, 0.75, 1.0]))]
  if experiment.startswith(('catch', 'mnist', 'umbrella')):
    return [np.where(good, 0.0, 2.0)]
  if experiment.startswith('cartpole_swingup'):
    ret = np.where(good, pick([101.5, 250.0, 700.0]), pick([0.0, 12.5, 100.0]))
    return [ret, ret]                                   # total_return, best_episode (running max below)
  if experiment.startswith('cartpole'):
    ret = np.where(good, pick([600.0, 1000.0]), pick([10.0, 200.0, 500.0]))
    return [ret, ret]                                   # raw_return, best_episode
  if experiment.startswith('mountain_car'):
    return [np.where(good, pick([-100.0, -150.0]), pick([-500.0, -1000.0]))]
  if experiment == 'discounting_chain':
    return [np.where(good, pick([1.0625, 1.125]), pick([0.0, 1.0]))]
  if experiment.startswith('memory'):
    return [good.astype(np.float64)]                    # total_perfect
  raise ValueError(experiment)


def _deep_sea_bad(thresh, size, lanes, num, rng):
  """total_bad_episodes increments: bad for the first X episodes, X chosen per lane to cross thresh early, late,
  never, or to sit exactly on it at episode 1000 (X = thresh * 1000: not below, so the crossing is one log point
  later)."""
  out = np.zeros((lanes, num))
  for lane in range(lanes):
    kind = (lane + size) % 4
    x = {0: rng.randint(0, 2 ** min(size, 12) // 2), 1: rng.randint(3000, 9000), 2: num,
         3: int(round(thresh * 1000))}[kind]
    out[lane, :x] = 1.0
  return out


def synthetic_tables():
  from bsuite_b200 import recording, sweep  # pylint: disable=import-outside-toplevel
  rng = np.random.RandomState(SYN_SEED)
  B = SYN_LANES
  tables = {}
  quality = np.clip(np.array([1.0, 0.0, 0.6, 0.85] + list(rng.uniform(0, 1, B - 4))), 0, 1)
  for experiment, ids in sweep.BY_EXPERIMENT.items():
    num = sweep.EPISODES[ids[0]]
    schedule = np.asarray(recording.log_schedule(num))
    n_points = len(schedule)
    for bsuite_id in ids:
      if experiment.startswith('deep_sea'):
        size = int(sweep.SETTINGS[bsuite_id]['size'])
        per = [_deep_sea_bad(0.8 if experiment.endswith('stochastic') else 0.9, size, B, num, rng)]
      else:
        q = np.clip(quality[:, None] + rng.uniform(-0.1, 0.1, (B, 1)) * (quality[:, None] % 1 != 0), 0, 1)
        per = _per_episode(experiment, rng.uniform(size=(B, num)) < q, rng)
      values = []
      for c, inc in enumerate(per):
        acc = np.maximum.accumulate(inc, axis=1) if c == 1 else np.cumsum(inc, axis=1)
        values.append(acc[:, schedule - 1])             # [B, n_points]
      rows = np.stack(values, axis=0).transpose(2, 0, 1).copy()     # [n_points, n_value_cols, B]
      counts = np.full(B, n_points, np.int32)
      for lane in range(4, 8):                          # truncated at a different log point per id
        counts[lane] = rng.randint(1, n_points + 1)
      for lane in range(8, 12):                         # some ids missing, the rest finished or truncated
        counts[lane] = 0 if rng.uniform() < 0.3 else (n_points if lane % 2 else rng.randint(1, n_points + 1))
      if experiment.startswith('mnist'):                # lanes that stop just before / just after episode 9000
        counts[12] = int(np.searchsorted(schedule, 9000, side='right'))
        counts[13] = int(np.searchsorted(schedule, 9000, side='right')) + 1
      counts[B - 1] = 0                                 # a lane with no rows at all
      for lane in range(B):
        rows[counts[lane]:, :, lane] = np.nan           # never read
      tables[bsuite_id] = dict(rows=rows, counts=counts, schedule=schedule)
  return tables


def lane_frame(pd, logging_utils, tables, lane, columns_for):
  """The DataFrame csv_load.load_one_result_set reads back from lane `lane`'s CSV files (None: no rows)."""
  parts = []
  for bsuite_id, table in tables.items():
    c = int(table['counts'][lane])
    if c == 0:
      continue
    data = {'episode': table['schedule'][:c].astype(np.int64)}
    for j, name in enumerate(columns_for(bsuite_id)):
      col = table['rows'][:c, j, lane]
      data[name] = col.astype(np.int64) if name in _INT_COLUMNS else col.astype(np.float64)
    df = pd.DataFrame(data)
    df['bsuite_id'] = bsuite_id
    parts.append(df)
  if not parts:
    return None
  return logging_utils.join_metadata(pd.concat(parts, sort=False))


def reference_scores(tables, lanes, columns_for):
  """What bsuite_score / ave_score_by_tag give for each lane's frame: scores, finished [23, lanes], tags [7, lanes]."""
  from bsuite_b200 import scoring  # pylint: disable=import-outside-toplevel
  pd, summary_analysis, logging_utils = _reference()
  scores = np.full((len(scoring.EXPERIMENTS), lanes), np.nan)
  finished = np.zeros((len(scoring.EXPERIMENTS), lanes), np.int32)
  tags = np.full((len(scoring.TAGS), lanes), np.nan)
  for lane in range(lanes):
    df = lane_frame(pd, logging_utils, tables, lane, columns_for)
    if df is None:
      continue
    score_df = summary_analysis.bsuite_score(df)
    for _, row in score_df.iterrows():
      e = scoring.EXPERIMENTS.index(row['bsuite_env'])
      scores[e, lane] = float(row['score'])
      finished[e, lane] = int(bool(row['finished']))
    tag_df = summary_analysis.ave_score_by_tag(score_df, None)
    for _, row in tag_df.iterrows():
      tags[scoring.TAGS.index(row['tag']), lane] = float(row['score'])
  return scores, finished, tags


def synthetic():
  tables = synthetic_tables()
  scores, finished, tags = reference_scores(tables, SYN_LANES, lambda i: columns_of(i.split('/')[0]))
  out = {'syn/scores': scores, 'syn/finished': finished, 'syn/tags': tags}
  for bsuite_id, table in tables.items():
    out[f'syn/{bsuite_id}/rows'] = table['rows']
    out[f'syn/{bsuite_id}/counts'] = table['counts']
  return out


# ---------------------------------------------------------------------------- end-to-end runs
class _Rows:
  def __init__(self):
    self.rows = []

  def write(self, data):
    self.rows.append({k: float(v) for k, v in data.items()})


def reference_spec(bsuite_id):
  """(environment class, kwargs, wrapper, wrapper argument, number of actions, calls per episode)."""
  from bsuite_b200 import sweep  # pylint: disable=import-outside-toplevel
  settings = dict(sweep.SETTINGS[bsuite_id])
  experiment = bsuite_id.split('/')[0]
  if experiment == 'bandit':
    return 'bandit', dict(mapping_seed=settings['mapping_seed']), None, None, 11, 2
  if experiment == 'bandit_noise':
    return 'bandit', dict(mapping_seed=settings['mapping_seed']), 'noise', settings['noise_scale'], 11, 2
  if experiment == 'discounting_chain':
    return 'discounting_chain', dict(mapping_seed=settings['mapping_seed']), None, None, 5, 101
  if experiment == 'catch':
    return 'catch', {}, None, None, 3, 10
  raise ValueError(bsuite_id)


def e2e_steps(bsuite_id) -> int:
  """Engine step() calls that complete exactly NUM_EPISODES episodes (each episode starts with a FIRST call)."""
  from bsuite_b200 import sweep  # pylint: disable=import-outside-toplevel
  return sweep.EPISODES[bsuite_id] * reference_spec(bsuite_id)[5]


def end_to_end():
  import ctypes  # pylint: disable=import-outside-toplevel
  from bsuite.utils import wrappers  # pylint: disable=import-outside-toplevel
  from bsuite_b200 import _lib, recording, sweep  # pylint: disable=import-outside-toplevel
  lib = _lib.load()
  tables, columns = {}, {}
  for bsuite_id in E2E_IDS:
    env_class, kwargs, wrapper, arg, n_act, _ = reference_spec(bsuite_id)
    T = e2e_steps(bsuite_id)
    schedule = np.asarray(recording.log_schedule(sweep.EPISODES[bsuite_id]))
    per_lane = []
    for lane in range(E2E_LANES):
      actions = np.zeros(T, np.int32)
      _lib.check(lib.bsb_random_actions(E2E_ACTION_SEED, lane, 1, 0, T, n_act, ctypes.c_void_p(actions.ctypes.data)))
      raw = rr.make_reference_env(env_class, kwargs, 'philox', E2E_SEED, lane, wrapper, arg)
      raw.bsuite_num_episodes = sweep.EPISODES[bsuite_id]
      sink = _Rows()
      logged = wrappers.Logging(raw, sink)
      for a in actions:
        logged.step(int(a))
      assert [r['episode'] for r in sink.rows] == list(schedule), bsuite_id
      per_lane.append(sink.rows)
    names = [c for c in per_lane[0][0] if c != 'episode']
    columns[bsuite_id] = names
    rows = np.asarray([[[r[c] for c in names] for r in lane_rows] for lane_rows in per_lane])   # [lanes, P, C]
    tables[bsuite_id] = dict(rows=rows.transpose(1, 2, 0).copy(), counts=np.full(E2E_LANES, len(schedule), np.int32),
                             schedule=schedule)
  scores, finished, tags = reference_scores(tables, E2E_LANES, lambda i: columns[i])
  return {'e2e/scores': scores, 'e2e/finished': finished, 'e2e/tags': tags,
          'e2e/config.json': _json(dict(ids=list(E2E_IDS), lanes=E2E_LANES, seed=E2E_SEED,
                                        action_seed=E2E_ACTION_SEED,
                                        steps={i: e2e_steps(i) for i in E2E_IDS}))}


def build():
  return dict(synthetic(), **end_to_end())


def main():
  parser = argparse.ArgumentParser()
  parser.add_argument('--check', action='store_true')
  args = parser.parse_args()
  data = build()
  if args.check:
    old = np.load(OUT_PATH)
    same = set(old.files) == set(data) and all(np.array_equal(old[k], data[k], equal_nan=True) for k in data)
    print(('ok   ' if same else 'DIFF ') + os.path.basename(OUT_PATH))
    return 0 if same else 1
  os.makedirs(os.path.dirname(OUT_PATH), exist_ok=True)
  np.savez_compressed(OUT_PATH, **data)
  print(f'wrote {OUT_PATH} ({os.path.getsize(OUT_PATH) / 1024:.0f} KiB)')
  return 0


if __name__ == '__main__':
  sys.exit(main())
