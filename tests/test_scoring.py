"""Per-lane bsuite scores (bsuite_b200.scoring, bsb_scorer_*) against the reference's analysis.

tests/golden/reference/scores.npz (oracle/gen_score_checks.py) holds what the unmodified
summary_analysis.bsuite_score / ave_score_by_tag return for each lane of synthetic row tables covering every id of
every experiment, and for reference runs of bandit, bandit_noise, discounting_chain and catch driven by the
engine's own action stream.
"""

import ctypes

import numpy as np
import pytest

import bsuite_b200
from bsuite_b200 import _lib, recording, scoring, sweep
from bsuite_b200.suite import SweepBatch, one_per_experiment
from tests import conftest as cf

TOL = 1e-12
# Experiments whose score is a ratio of threshold decisions (deep_sea solved / beat-dither, memory and umbrella
# regret < threshold): these must agree exactly.
THRESHOLD_EXPERIMENTS = ('deep_sea', 'deep_sea_stochastic', 'memory_len', 'memory_size', 'umbrella_distract',
                         'umbrella_length')


def _fixture():
  return cf.load_reference('scores')


def synthetic_tables():
  """bsuite_id -> dict(rows [n_points, 1 + value columns, B], counts, columns): the fixture's value columns with
  the episode column (the log schedule) in front."""
  ref = _fixture()
  tables = {}
  for bsuite_id in sweep.SWEEP:
    name = bsuite_id.split('/')[0]
    values = ref[f'syn/{bsuite_id}/rows']
    schedule = np.asarray(recording.log_schedule(sweep.EPISODES[bsuite_id]), np.float64)
    episode = np.broadcast_to(schedule[:, None, None], (values.shape[0], 1, values.shape[2]))
    columns = ['episode', scoring.VALUE_COLUMNS[name]] + (['best_episode'] if name in scoring.NEEDS_BEST else [])
    tables[bsuite_id] = dict(rows=np.concatenate([episode, values], axis=1), counts=ref[f'syn/{bsuite_id}/counts'],
                             columns=columns)
  return tables


def _assert_matches_reference(got, scores, finished, tags):
  np.testing.assert_array_equal(got['finished'], finished)
  np.testing.assert_array_equal(np.isnan(got['scores']), np.isnan(scores))
  np.testing.assert_allclose(got['scores'], scores, rtol=0, atol=TOL, equal_nan=True)
  np.testing.assert_array_equal(np.isnan(got['tags']), np.isnan(tags))
  np.testing.assert_allclose(got['tags'], tags, rtol=0, atol=TOL, equal_nan=True)


def _score_tables(tables, device):
  scorer = scoring.Scorer.from_rows(tables, device=device)
  try:
    return scoring.as_numpy(scorer.run())
  finally:
    scorer.close()


def test_experiment_and_tag_orders_are_the_librarys():
  lib = _lib.load()
  assert scoring.EXPERIMENTS == tuple(lib.bsb_experiment_name(i).decode() for i in range(_lib.NUM_EXPERIMENTS))
  assert scoring.TAGS == tuple(lib.bsb_tag_name(i).decode() for i in range(_lib.NUM_TAGS))
  assert lib.bsb_experiment_name(_lib.NUM_EXPERIMENTS) is None and lib.bsb_tag_name(-1) is None
  assert set(scoring.TAGS) == set(sweep.TAGS)


def test_tag_membership_follows_the_sweep():
  """A lane whose only experiment is e scores exactly the tags e carries (sweep.TAGS), NaN for the others."""
  tables = synthetic_tables()
  for name, ids in sweep.BY_EXPERIMENT.items():
    got = _score_tables({i: tables[i] for i in ids}, 'cpu')
    carried = {t for t in scoring.TAGS if ids[0] in sweep.TAGS[t]}
    lane = 0                                           # finished, perfect lane: every score is a number
    for t, tag in enumerate(scoring.TAGS):
      assert np.isnan(got['tags'][t, lane]) == (tag not in carried), (name, tag)


def test_host_scorer_matches_the_reference_on_synthetic_tables():
  ref = _fixture()
  got = _score_tables(synthetic_tables(), 'cpu')
  _assert_matches_reference(got, ref['syn/scores'], ref['syn/finished'], ref['syn/tags'])
  for name in THRESHOLD_EXPERIMENTS:
    e = scoring.EXPERIMENTS.index(name)
    np.testing.assert_array_equal(got['scores'][e], ref['syn/scores'][e], err_msg=name)


def test_fixture_covers_the_cases_it_is_meant_to():
  ref = _fixture()
  scores = ref['syn/scores']
  assert np.all(np.isnan(scores[:, -1]))                        # the lane without rows
  assert np.any(scores == 0.0) and np.any(scores == 1.0)        # clipped at both ends
  for name in ('mnist', 'mnist_noise', 'mnist_scale'):          # no row past episode 9000: NaN
    assert np.isnan(scores[scoring.EXPERIMENTS.index(name), 12])
    assert not np.isnan(scores[scoring.EXPERIMENTS.index(name), 13])
  assert np.any(ref['syn/finished'] == 1) and np.any((ref['syn/finished'] == 0) & ~np.isnan(scores))


def _run_e2e(device):
  config = _fixture()['e2e/config.json']
  batch = SweepBatch(config['ids'], lanes=config['lanes'], device=device, seed=config['seed'], record_rows=True)
  try:
    total, chunk = max(config['steps'].values()), 10100
    assert total % chunk == 0
    for _ in range(total // chunk):
      batch.rollout(chunk, action_seed=config['action_seed'])
    return scoring.as_numpy(batch.scores())
  finally:
    batch.close()


def test_end_to_end_host_runs_score_as_the_reference():
  ref = _fixture()
  got = _run_e2e('cpu')
  _assert_matches_reference(got, ref['e2e/scores'], ref['e2e/finished'], ref['e2e/tags'])
  assert np.all(got['finished'][[scoring.EXPERIMENTS.index(n) for n in ('bandit', 'bandit_noise', 'catch',
                                                                         'discounting_chain')]] == 1)


def test_two_shards_concatenate_to_the_unsharded_scores(mnist_dir):
  ids = one_per_experiment()
  results = []
  for rank, world in ((0, 1), (0, 2), (1, 2)):
    batch = SweepBatch(ids, lanes=6, device='cpu', seed=5, rank=rank, world=world, record_rows=True)
    batch.rollout(3000, action_seed=2)
    results.append(scoring.as_numpy(batch.scores()))
    batch.close()
  whole, first, second = results
  for k in ('scores', 'finished', 'tags'):
    np.testing.assert_array_equal(np.concatenate([first[k], second[k]], axis=1), whole[k], err_msg=k)
  assert not np.all(np.isnan(whole['scores']))


def test_subset_of_ids_scores_only_those_ids():
  """Scoring a subset is scoring the frame that holds only those ids."""
  tables = synthetic_tables()
  subset = {i: tables[i] for i in ('catch/3', 'deep_sea/5', 'memory_len/0', 'memory_len/9')}
  got = _score_tables(subset, 'cpu')
  scored = ~np.all(np.isnan(got['scores']), axis=1)
  assert [scoring.EXPERIMENTS[e] for e in np.flatnonzero(scored)] == ['catch', 'deep_sea', 'memory_len']
  alone = _score_tables({'catch/3': tables['catch/3']}, 'cpu')
  np.testing.assert_array_equal(alone['scores'][scoring.EXPERIMENTS.index('catch')],
                                got['scores'][scoring.EXPERIMENTS.index('catch')])


def _source(rows, counts, experiment, batch, n_columns=3, col_value=1, col_best=-1):
  return _lib.ScoreSource(experiment=experiment, device=_lib.DEVICE_HOST, batch=batch, n_points=rows.shape[0],
                          n_columns=n_columns, col_episode=0, col_value=col_value, col_best=col_best,
                          group_key=0.0, rows=rows.ctypes.data, counts=counts.ctypes.data)


def _create(sources, batch=4):
  lib = _lib.load()
  array = (_lib.ScoreSource * len(sources))(*sources)
  handle = ctypes.c_void_p()
  status = lib.bsb_scorer_create(array, len(sources), batch, _lib.DEVICE_HOST, ctypes.byref(handle))
  if status == 0:
    lib.bsb_scorer_destroy(handle)
  return status, lib.bsb_last_error().decode()


def test_malformed_sources_are_rejected_with_a_message():
  rows = np.zeros((3, 3, 4))
  rows4, rows5 = rows, np.zeros((3, 3, 5))
  counts4, counts5 = np.zeros(4, np.int32), np.zeros(5, np.int32)
  catch = scoring.EXPERIMENTS.index('catch')
  cartpole = scoring.EXPERIMENTS.index('cartpole')
  assert _create([_source(rows4, counts4, catch, 4)])[0] == 0
  status, message = _create([_source(rows4, counts4, catch, 4), _source(rows5, counts5, catch, 5)])
  assert status == 1 and 'batch' in message
  status, message = _create([_source(rows4, counts4, 23, 4)])
  assert status == 1 and 'unknown experiment' in message
  status, message = _create([_source(rows4, counts4, catch, 4, col_value=-1)])
  assert status == 1 and 'missing column' in message and 'total_regret' in message
  status, message = _create([_source(rows4, counts4, cartpole, 4, col_value=1, col_best=7)])
  assert status == 1 and 'best_episode' in message
  status, message = _create([_source(rows4, counts4, catch, 4, n_columns=3, col_value=3)])
  assert status == 1 and 'missing column' in message
  wrong = _source(rows4, counts4, catch, 4)
  wrong.device = 0
  status, message = _create([wrong])
  assert status == 1 and 'device' in message
  status, message = _create([_source(rows4, counts4, catch, 4)] * 129)
  assert status == 1 and '128' in message
  # an environment without record_rows has no rows to point a source at
  env = bsuite_b200.load_from_id('catch/0', batch=4, device='cpu', track_episodes=True)
  source = _lib.ScoreSource()
  lib = _lib.load()
  assert lib.bsb_score_source_from_env(env._handle.ptr, catch, 0.0, ctypes.byref(source)) == 1
  assert b'log schedule' in lib.bsb_last_error()
  with pytest.raises(ValueError, match='record_rows=True'):
    scoring.Scorer({'catch/0': env})
  recorded = bsuite_b200.load_from_id('catch/0', batch=4, device='cpu', record_rows=True)
  assert lib.bsb_score_source_from_env(recorded._handle.ptr, cartpole, 0.0, ctypes.byref(source)) == 1
  assert b'family' in lib.bsb_last_error()
  env.close()
  recorded.close()


def test_sweep_batch_without_record_rows_is_unchanged_and_cannot_score():
  ids = ['catch/0', 'bandit/1']
  plain = SweepBatch(ids, lanes=3, device='cpu', seed=1)
  recorded = SweepBatch(ids, lanes=3, device='cpu', seed=1, record_rows=True)
  assert not plain.record_rows and all(env._log_schedule is None for env in plain.envs.values())
  a, b = plain.rollout(40, action_seed=4), recorded.rollout(40, action_seed=4)
  for k in ids:
    for field in ('observation', 'reward', 'discount', 'step_type'):
      np.testing.assert_array_equal(getattr(a[k], field).numpy(), getattr(b[k], field).numpy())
  with pytest.raises(RuntimeError, match='record_rows=True'):
    plain.scores()
  plain.close()
  recorded.close()


def test_run_writes_into_given_outputs():
  tables = synthetic_tables()
  subset = {i: tables[i] for i in sweep.BY_EXPERIMENT['bandit']}
  scorer = scoring.Scorer.from_rows(subset)
  out = scorer.empty_outputs()
  assert scorer.run(out) is out
  with pytest.raises(ValueError, match='contiguous'):
    scorer.run(dict(out, tags=out['tags'][:, :2]))
  scorer.close()


# ---------------------------------------------------------------------------- CUDA
@pytest.mark.gpu
def test_cuda_scorer_equals_the_host_scorer_bit_for_bit():
  tables = synthetic_tables()
  host, cuda = _score_tables(tables, 'cpu'), _score_tables(tables, 'cuda')
  for k in ('scores', 'finished', 'tags'):
    np.testing.assert_array_equal(cuda[k], host[k], err_msg=k)
  ref = _fixture()
  _assert_matches_reference(cuda, ref['syn/scores'], ref['syn/finished'], ref['syn/tags'])


@pytest.mark.gpu
def test_cuda_end_to_end_runs_score_as_the_host_and_the_reference():
  ref = _fixture()
  cuda, host = _run_e2e('cuda'), _run_e2e('cpu')
  for k in ('scores', 'finished', 'tags'):
    np.testing.assert_array_equal(cuda[k], host[k], err_msg=k)
  _assert_matches_reference(cuda, ref['e2e/scores'], ref['e2e/finished'], ref['e2e/tags'])


@pytest.mark.gpu
def test_a_sweep_is_scored_in_one_launch_and_replays_from_a_graph(mnist_dir):
  import torch
  batch = SweepBatch(one_per_experiment(), lanes=100, device='cuda', seed=9, record_rows=True)
  batch.rollout(2000, action_seed=1)
  eager = batch.scores()
  torch.cuda.synchronize()
  lib = _lib.load()
  before = lib.bsb_launch_count()
  eager = batch.scores()
  assert lib.bsb_launch_count() - before == 1
  scorer = batch._scorer
  out = scorer.empty_outputs()
  stream = torch.cuda.Stream()
  stream.wait_stream(torch.cuda.current_stream())
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph, stream=stream):
    scorer.run(out)
  graph.replay()
  torch.cuda.synchronize()
  for k in ('scores', 'finished', 'tags'):
    np.testing.assert_array_equal(out[k].cpu().numpy(), eager[k].cpu().numpy(), err_msg=k)
  # the graph reads the rows at replay time: more steps, then replay == eager again
  batch.rollout(3000, action_seed=1)
  graph.replay()
  again = batch.scores()
  torch.cuda.synchronize()
  for k in ('scores', 'finished', 'tags'):
    np.testing.assert_array_equal(out[k].cpu().numpy(), again[k].cpu().numpy(), err_msg=k)
  assert not np.array_equal(again['scores'].cpu().numpy(), eager['scores'].cpu().numpy(), equal_nan=True)
  batch.close()
