"""Score summaries (`track_scores=True`, bsb_read_score_summary, bsb_score_summarize): scores without the row store.

A summary is six float64 values per id and lane, folded in as each log row falls due.  Scores from summaries must
be the same bits as scores from the rows they were folded from, and so match the reference's analysis on the
fixture tests/golden/reference/scores.npz (see tests/test_scoring.py).
"""

import ctypes

import numpy as np
import pytest

import bsuite_b200
from bsuite_b200 import _lib, environment, experiments, recording, scoring
from bsuite_b200.suite import SweepBatch, one_per_experiment
from tests import conftest as cf
from tests.test_scoring import synthetic_tables

KEYS = ('scores', 'finished', 'tags')


def _fixture():
  return cf.load_reference('scores')


def _assert_same(got, want, what=''):
  for k in KEYS:
    np.testing.assert_array_equal(got[k], want[k], err_msg=f'{what} {k}')


def _run(scorer):
  try:
    return scoring.as_numpy(scorer.run())
  finally:
    scorer.close()


def _summary_numpy(summary):
  return {k: (v.cpu().numpy() if hasattr(v, 'cpu') else v) for k, v in summary.items()}


def _assert_summaries_equal(got, want, what, atol=0.0):
  got, want = _summary_numpy(got), _summary_numpy(want)
  np.testing.assert_array_equal(got['counts'], want['counts'], err_msg=f'{what} counts')
  for field in _lib.SUMMARY_FIELDS:
    np.testing.assert_allclose(got[field], want[field], rtol=0, atol=atol, equal_nan=True, err_msg=f'{what} {field}')


def _summaries_match_rows(batch, what):
  """Every environment of `batch` (both keywords on): its summary equals the host fold of its rows, field by field,
  and the scores from the summaries equal the scores from the rows, bit for bit."""
  summaries = {}
  for bsuite_id, env in batch.envs.items():
    summary = env.score_summary()
    _assert_summaries_equal(summary, scoring.summarize(bsuite_id, env.logged_rows()), f'{what} {bsuite_id}')
    summaries[bsuite_id] = summary
  from_rows = _run(scoring.Scorer(batch.envs))
  from_summaries = _run(scoring.Scorer.from_summaries(summaries, device=batch._device))
  _assert_same(from_summaries, from_rows, what)
  return from_rows


# ---------------------------------------------------------------------------- host
def test_folded_synthetic_tables_score_as_the_reference_and_the_rows_bit_for_bit():
  ref = _fixture()
  tables = synthetic_tables()
  folded = _run(scoring.Scorer.from_rows(tables, device='cpu', summarize=True))
  rows = _run(scoring.Scorer.from_rows(tables, device='cpu'))
  _assert_same(folded, rows, 'rows')
  _assert_same(folded, dict(scores=ref['syn/scores'], finished=ref['syn/finished'], tags=ref['syn/tags']), 'reference')


def test_the_synthetic_tables_hold_the_edge_cases():
  """Truncated and missing ids, the empty lane, deep_sea crossings and mnist lanes 12 / 13 around episode 9 000 (the
  cases tests/test_scoring.py names) are all in what the summaries score above."""
  ref = _fixture()
  counts = np.stack([ref[f'syn/{i}/counts'] for i in synthetic_tables()])
  assert np.any(counts == 0) and np.all(counts[:, -1] == 0)               # missing ids, the empty lane
  schedule = recording.log_schedule(10000)
  assert np.any((counts > 0) & (counts < len(schedule)))                   # truncated ids
  mnist = ref['syn/mnist/0/counts']
  assert schedule[mnist[12] - 1] <= 9000 < schedule[mnist[13] - 1]


def test_summary_fields_of_a_hand_made_table():
  """deep_sea_stochastic: rows below episode 100 never solve; the first row at or past it with
  total_bad_episodes / episode < 0.8 does.  cartpole: best is the running max of best_episode."""
  schedule = np.asarray(recording.log_schedule(10000), np.float64)
  n = 30
  episodes = schedule[:n]
  bad = episodes * 0.9
  bad[episodes >= 170] = episodes[episodes >= 170] * 0.5                       # solved from 170 on
  bad[3] = 0.0                                                                 # episode 4: below 100, ignored
  rows = np.stack([schedule[:n], bad], axis=1)[:, :, None]
  summary = scoring.summarize('deep_sea_stochastic/0', dict(rows=rows, counts=np.array([n], np.int32),
                                                            columns=['episode', 'total_bad_episodes']))
  assert summary['first_solved'].item() == 170.0
  assert summary['last_episode'].item() == schedule[n - 1] and summary['prev_episode'].item() == schedule[n - 2]
  assert summary['last_value'].item() == bad[n - 1] and summary['prev_value'].item() == bad[n - 2]
  assert np.isnan(summary['best'].item()) and summary['counts'].item() == n

  best = np.array([3., 7., 7., 2., 9., 1.])
  rows = np.stack([schedule[:6], np.zeros(6), best], axis=1)[:, :, None]
  table = dict(rows=rows, counts=np.array([6], np.int32), columns=['episode', 'raw_return', 'best_episode'])
  summary = scoring.summarize('cartpole/0', table)
  assert summary['best'].item() == 9.0 and np.isnan(summary['first_solved'].item())
  one = scoring.summarize('cartpole/0', dict(table, counts=np.array([1], np.int32)))
  assert np.isnan(one['prev_episode'].item()) and one['best'].item() == 3.0
  empty = scoring.summarize('cartpole/0', dict(table, counts=np.array([0], np.int32)))
  assert all(np.isnan(empty[f].item()) for f in _lib.SUMMARY_FIELDS) and empty['counts'].item() == 0


def _run_e2e(device, **kw):
  config = _fixture()['e2e/config.json']
  batch = SweepBatch(config['ids'], lanes=config['lanes'], device=device, seed=config['seed'], **kw)
  try:
    total, chunk = max(config['steps'].values()), 10100
    for _ in range(total // chunk):
      batch.rollout(chunk, action_seed=config['action_seed'])
    for env in batch.envs.values():
      with pytest.raises(RuntimeError, match='record_rows=True'):
        env.logged_rows()
    return scoring.as_numpy(batch.scores())
  finally:
    batch.close()


def test_end_to_end_host_summaries_score_as_the_reference():
  ref = _fixture()
  got = _run_e2e('cpu', track_scores=True)
  _assert_same(got, dict(scores=ref['e2e/scores'], finished=ref['e2e/finished'], tags=ref['e2e/tags']), 'e2e')


def test_host_summaries_follow_the_rows_through_every_call_pattern(mnist_dir):
  batch = SweepBatch(one_per_experiment(), lanes=5, device='cpu', seed=21, record_rows=True, track_scores=True)
  rng = np.random.RandomState(3)
  import torch
  try:
    batch.rollout(1200, action_seed=4)
    _summaries_match_rows(batch, 'rollout')
    for env in batch.envs.values():                     # single steps
      for _ in range(150):
        env.step(torch.as_tensor(rng.randint(env.num_actions, size=env.batch).astype(np.int32)))
    _summaries_match_rows(batch, 'step')
    for env in batch.envs.values():                     # host-driven steps, with a mid-episode reset in between
      host = env.make_host_buffers()
      for t in range(120):
        if t == 60:
          env.reset()
        env.step_host(torch.as_tensor(rng.randint(env.num_actions, size=env.batch).astype(np.int32)), host)
    _summaries_match_rows(batch, 'step_host')
    batch.rollout(2500, action_seed=5)
    scores = _summaries_match_rows(batch, 'rollout again')
    scored = [n for e, n in enumerate(scoring.EXPERIMENTS) if not np.isnan(scores['scores'][e, 0])]
    assert scored == [n for n in scoring.EXPERIMENTS if not n.startswith('mnist')]   # mnist: no row past 9 000 yet
  finally:
    batch.close()


def _load(bsuite_id, **kw):
  return bsuite_b200.load_from_id(bsuite_id, batch=6, device='cpu', seed=13, **kw)


@pytest.mark.parametrize('bsuite_id', ['deep_sea_stochastic/0', 'cartpole_swingup/3', 'catch_noise/2'])
def test_a_summary_only_environment_steps_as_a_plain_one_and_keeps_no_rows(bsuite_id):
  plain, summary_only = _load(bsuite_id, track_episodes=True), _load(bsuite_id, track_scores=True)
  both = _load(bsuite_id, record_rows=True, track_scores=True)
  a, b = plain.rollout(3000, action_seed=2), summary_only.rollout(3000, action_seed=2)
  for field in ('observation', 'reward', 'discount', 'step_type'):
    np.testing.assert_array_equal(getattr(a, field).numpy(), getattr(b, field).numpy(), err_msg=field)
  with pytest.raises(RuntimeError, match='record_rows=True'):
    summary_only.logged_rows()
  lib = _lib.load()
  rows, counts = np.empty(1 << 16), np.empty(6, np.int32)
  assert lib.bsb_read_log_rows(summary_only._handle.ptr, rows.ctypes.data, counts.ctypes.data, None) == 1
  assert b'no log rows' in lib.bsb_last_error()
  n_points = len(recording.log_schedule(both.bsuite_num_episodes))
  sizes = {}
  for name, env in (('both', both), ('summary_only', summary_only)):
    n = ctypes.c_int64()
    _lib.check(lib.bsb_state_bytes(env._handle.ptr, ctypes.byref(n)))
    sizes[name] = n.value
  assert sizes['both'] - sizes['summary_only'] == n_points * (5 + len(both.info_names)) * both.batch * 8
  plain.close(); summary_only.close(); both.close()


def test_state_dict_round_trip_carries_the_summary():
  bsuite_id = 'deep_sea_stochastic/1'
  uninterrupted, restored = _load(bsuite_id, track_scores=True), _load(bsuite_id, track_scores=True)
  uninterrupted.rollout(2500, action_seed=7)
  state = uninterrupted.state_dict()
  restored.load_state_dict(state)
  _assert_summaries_equal(restored.score_summary(), uninterrupted.score_summary(), 'restored')
  uninterrupted.rollout(3000, action_seed=7)
  restored.rollout(3000, action_seed=7)
  want = _run(scoring.Scorer({bsuite_id: uninterrupted}))
  _assert_same(_run(scoring.Scorer({bsuite_id: restored})), want, 'restored')
  assert not np.all(np.isnan(want['scores'][scoring.EXPERIMENTS.index('deep_sea_stochastic')]))
  # the summary mode is part of the snapshot's configuration; other configurations keep their fingerprints
  rows_only = _load(bsuite_id, record_rows=True)
  assert rows_only._config_fingerprint() == _load(bsuite_id, track_episodes=True)._config_fingerprint()
  assert rows_only._config_fingerprint() != uninterrupted._config_fingerprint()
  with pytest.raises(ValueError, match='differently configured'):
    rows_only.load_state_dict(state)
  uninterrupted.close(); restored.close(); rows_only.close()


def test_two_shards_of_summaries_concatenate_to_the_unsharded_scores(mnist_dir):
  ids = one_per_experiment()
  results = []
  for rank, world in ((0, 1), (0, 2), (1, 2)):
    batch = SweepBatch(ids, lanes=6, device='cpu', seed=5, rank=rank, world=world, track_scores=True)
    batch.rollout(3000, action_seed=2)
    results.append(scoring.as_numpy(batch.scores()))
    batch.close()
  whole, first, second = results
  for k in KEYS:
    np.testing.assert_array_equal(np.concatenate([first[k], second[k]], axis=1), whole[k], err_msg=k)
  rows = SweepBatch(ids, lanes=6, device='cpu', seed=5, record_rows=True)
  rows.rollout(3000, action_seed=2)
  _assert_same(whole, scoring.as_numpy(rows.scores()), 'rows')
  rows.close()


def test_malformed_input_is_refused_with_a_message():
  # rows that are not a prefix of the experiment's log schedule
  schedule = np.asarray(recording.log_schedule(10000), np.float64)
  rows = np.stack([schedule[:5], np.zeros(5)], axis=1)[:, :, None].copy()
  rows[2, 0, 0] = 1.3
  with pytest.raises(_lib.EngineError, match='prefix'):
    scoring.summarize('catch/0', dict(rows=rows, counts=np.array([5], np.int32), columns=['episode', 'total_regret']))
  with pytest.raises(_lib.EngineError, match='prefix'):
    scoring.Scorer.from_rows({'catch/0': dict(rows=rows, counts=np.array([5], np.int32),
                                              columns=['episode', 'total_regret'])}, summarize=True)
  # a score_experiment of another family; a summary without the experiment's log schedule
  with pytest.raises(_lib.EngineError, match='family'):
    bsuite_b200.load('catch', {}, batch=2, device='cpu', track_scores=True, score_experiment='bandit')
  with pytest.raises(ValueError, match='score_experiment'):
    environment.BatchedEnvironment(experiments.catch(), batch=2, device='cpu', track_scores=True)
  spec = experiments.catch()
  spec.bsuite_num_episodes = 20000
  with pytest.raises(_lib.EngineError, match='prefix'):
    environment.BatchedEnvironment(spec, batch=2, device='cpu', track_scores=True, score_experiment='catch')
  # a summary source of the wrong shape, and one for another experiment
  lib = _lib.load()
  block, counts = np.zeros((6, 4)), np.zeros(4, np.int32)
  source = _lib.ScoreSource(experiment=scoring.EXPERIMENTS.index('catch'), device=_lib.DEVICE_HOST, batch=4,
                            n_points=10, n_columns=5, layout=_lib.SCORE_SUMMARY, rows=block.ctypes.data,
                            counts=counts.ctypes.data)
  handle = ctypes.c_void_p()
  assert lib.bsb_scorer_create(ctypes.byref(source), 1, 4, _lib.DEVICE_HOST, ctypes.byref(handle)) == 1
  assert b'n_columns' in lib.bsb_last_error()
  source.n_columns, source.layout = 6, 7
  assert lib.bsb_scorer_create(ctypes.byref(source), 1, 4, _lib.DEVICE_HOST, ctypes.byref(handle)) == 1
  assert b'layout' in lib.bsb_last_error()
  env = bsuite_b200.load_from_id('catch/0', batch=4, device='cpu', track_scores=True)
  got = _lib.ScoreSource()
  assert lib.bsb_score_source_from_env(env._handle.ptr, scoring.EXPERIMENTS.index('catch_noise'), 0.1,
                                       ctypes.byref(got)) == 1
  assert b'score summary of catch' in lib.bsb_last_error()
  assert lib.bsb_score_source_from_env(env._handle.ptr, scoring.EXPERIMENTS.index('catch'), 0.0, ctypes.byref(got)) == 0
  assert got.layout == _lib.SCORE_SUMMARY and got.n_columns == 6
  env.close()
  # scoring a SweepBatch that keeps neither
  plain = SweepBatch(['catch/0'], lanes=2, device='cpu', seed=1)
  with pytest.raises(RuntimeError, match=r'record_rows=True.*track_scores=True'):
    plain.scores()
  plain.close()


def test_mixed_layouts_score_as_either():
  """Rows for some ids and summaries for the others, within one experiment and across experiments."""
  tables = synthetic_tables()
  ids = [i for i in tables if i.split('/')[0] in ('deep_sea', 'cartpole_swingup', 'mnist', 'catch_noise')]
  folded = {i: scoring.summarize(i, tables[i]) for i in ids}
  want = _run(scoring.Scorer.from_rows({i: tables[i] for i in ids}))
  sources, keep = [], []
  for n, i in enumerate(ids):
    if n % 2:
      source, rows, counts = scoring._rows_source(i, tables[i], __import__('torch').device('cpu'))
      keep += [rows, counts]
    else:
      import torch
      block = torch.stack([folded[i][f] for f in _lib.SUMMARY_FIELDS]).contiguous()
      keep += [block, folded[i]['counts']]
      source = _lib.ScoreSource(experiment=scoring.EXPERIMENTS.index(scoring.experiment_of(i)),
                                device=_lib.DEVICE_HOST, batch=block.shape[1], n_points=folded[i]['n_points'],
                                n_columns=6, col_episode=-1, col_value=-1, col_best=-1, layout=_lib.SCORE_SUMMARY,
                                group_key=scoring.group_key(i), rows=block.data_ptr(),
                                counts=folded[i]['counts'].data_ptr())
    sources.append(source)
  scorer = scoring.Scorer.__new__(scoring.Scorer)
  scorer._init(sources, want['scores'].shape[1], 'cpu', keep=keep)
  _assert_same(_run(scorer), want, 'mixed')


# ---------------------------------------------------------------------------- CUDA
# cartpole(_swingup)'s rows differ between CUDA and the host path in the last bits (tests/test_recording.py): so do
# their summaries.  Everything else is bit for bit.
def _tolerance(bsuite_id):
  return 1e-6 if bsuite_id.startswith('cartpole') else 0.0


def _assert_cuda_matches_host(cuda, host, what):
  for bsuite_id in cuda.envs:
    _assert_summaries_equal(cuda.envs[bsuite_id].score_summary(), host.envs[bsuite_id].score_summary(),
                            f'{what} {bsuite_id}', atol=_tolerance(bsuite_id))


@pytest.mark.gpu
@pytest.mark.runs_last
def test_cuda_summaries_equal_the_host_path_through_steps_rollouts_and_graph_replays(mnist_dir):
  import torch
  kw = dict(lanes=8, seed=17, record_rows=True, track_scores=True)
  cuda, host = SweepBatch(one_per_experiment(), device='cuda', **kw), SweepBatch(one_per_experiment(), device='cpu', **kw)
  try:
    cuda.rollout(1500, action_seed=3); host.rollout(1500, action_seed=3)
    torch.cuda.synchronize()
    _assert_cuda_matches_host(cuda, host, 'rollout')
    _summaries_match_rows(cuda, 'cuda rollout')
    rng = np.random.RandomState(1)
    for bsuite_id, env in cuda.envs.items():
      for _ in range(100):
        actions = torch.as_tensor(rng.randint(env.num_actions, size=env.batch).astype(np.int32))
        env.step(actions.cuda()); host.envs[bsuite_id].step(actions)
    torch.cuda.synchronize()
    _assert_cuda_matches_host(cuda, host, 'step')
    graphed = cuda.capture(num_steps=400, action_seed=6)
    for _ in range(3):
      graphed.replay(); host.rollout(400, action_seed=6)
    torch.cuda.synchronize()
    _assert_cuda_matches_host(cuda, host, 'graph replay')
    _summaries_match_rows(cuda, 'cuda graph replay')
  finally:
    cuda.close(); host.close()


@pytest.mark.gpu
@pytest.mark.runs_last
def test_cuda_summaries_through_host_driven_steps_equal_the_host_path():
  """deep_sea N = 32 runs host steps in two phases (rows fall due in phase 1), and as two launches with wait=False."""
  import torch
  batch, steps = 96, 1500
  make = lambda device: bsuite_b200.load_from_id('deep_sea/11', batch=batch, device=device, seed=3, track_scores=True)
  two_phase, parts, host = make('cuda'), make('cuda'), make('cpu')
  pinned = torch.as_tensor(np.random.RandomState(7).randint(2, size=(steps, batch)).astype(np.int32)).pin_memory()
  buffers, parts_buffers = two_phase.make_host_buffers(), parts.make_host_buffers()
  for t in range(steps):
    two_phase.step_host(pinned[t], buffers)
    parts.step_host(pinned[t], parts_buffers, wait=False)
    parts.host_wait()
    host.step(pinned[t])
  want = host.score_summary()
  assert want['counts'].min().item() > 0
  _assert_summaries_equal(two_phase.score_summary(), want, 'two-phase')
  _assert_summaries_equal(parts.score_summary(), want, 'parts')
  two_phase.close(); parts.close(); host.close()


@pytest.mark.gpu
def test_cuda_summary_scorer_equals_the_host_and_the_reference_on_the_folded_fixture():
  tables = synthetic_tables()
  host = _run(scoring.Scorer.from_rows(tables, device='cpu', summarize=True))
  cuda = _run(scoring.Scorer.from_rows(tables, device='cuda', summarize=True))
  _assert_same(cuda, host, 'cuda')
  ref = _fixture()
  _assert_same(cuda, dict(scores=ref['syn/scores'], finished=ref['syn/finished'], tags=ref['syn/tags']), 'reference')


@pytest.mark.gpu
def test_a_summary_sweep_is_scored_in_one_launch_and_replays_from_a_graph(mnist_dir):
  import torch
  batch = SweepBatch(one_per_experiment(), lanes=100, device='cuda', seed=9, track_scores=True)
  batch.rollout(2000, action_seed=1)
  batch.scores()
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
  for k in KEYS:
    np.testing.assert_array_equal(out[k].cpu().numpy(), eager[k].cpu().numpy(), err_msg=k)
  batch.rollout(3000, action_seed=1)
  graph.replay()
  again = batch.scores()
  torch.cuda.synchronize()
  for k in KEYS:
    np.testing.assert_array_equal(out[k].cpu().numpy(), again[k].cpu().numpy(), err_msg=k)
  assert not np.array_equal(again['scores'].cpu().numpy(), eager['scores'].cpu().numpy(), equal_nan=True)
  batch.close()


@pytest.mark.gpu
def test_cuda_end_to_end_summaries_score_as_the_reference():
  ref = _fixture()
  got = _run_e2e('cuda', track_scores=True)
  _assert_same(got, dict(scores=ref['e2e/scores'], finished=ref['e2e/finished'], tags=ref['e2e/tags']), 'e2e')
