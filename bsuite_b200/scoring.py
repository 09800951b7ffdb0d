"""bsuite scores from the log rows recorded on the device (`record_rows=True`), one score per lane.

The reference scores a run with `experiments/<name>/analysis.py::score`, collected by
`experiments/summary_analysis.py::bsuite_score` and averaged per tag by `ave_score_by_tag`, on the CSV rows of
its `Logging` wrapper.  Here every lane of a batch is one such run: `Scorer.run()` returns, for every lane, what
those functions return for the DataFrame that lane's CSV files would load into -- computed where the rows live,
in one kernel launch for a whole sweep (`bsb_scorer_run`), without writing or reading a file.

    envs = {bsuite_id: bsuite_b200.load_from_id(bsuite_id, batch=B, record_rows=True) for bsuite_id in ids}
    ... step them ...
    result = scoring.Scorer(envs).run()     # scores [23, B], finished [23, B], tags [7, B]

Row i of `scores` / `finished` is experiment `EXPERIMENTS[i]`, row t of `tags` is tag `TAGS[t]`.  An experiment
without a row in a lane is not scored there (NaN, finished 0); a tag average skips NaN, as pandas' mean does.

Scores need far less than the rows: `track_scores=True` instead of `record_rows=True` keeps, per id and lane, a
score summary of six float64 values (`_lib.SUMMARY_FIELDS`), folded in on the device as each row falls due.  A
lane's rows are always a prefix of the log schedule, so the summary holds everything the scoring rules read of
them, and the scores from summaries are the same bits as the scores from the rows.
"""

import ctypes
from typing import Any, Dict, Mapping, Optional, Sequence

import numpy as np

from bsuite_b200 import _lib
from bsuite_b200 import sweep

# bsb_experiment: the reference's registration order (bsuite/sweep.py)
EXPERIMENTS = tuple(sweep.BY_EXPERIMENT)
# bsb_tag: the tag names, sorted
TAGS = ('basic', 'credit_assignment', 'exploration', 'generalization', 'memory', 'noise', 'scale')

# The sweep setting each experiment's rule groups by (score_by_scaling, per-size / per-length loops).
GROUP_KEYS = {
    'bandit_noise': 'noise_scale', 'bandit_scale': 'reward_scale',
    'cartpole_noise': 'noise_scale', 'cartpole_scale': 'reward_scale', 'cartpole_swingup': 'height_threshold',
    'catch_noise': 'noise_scale', 'catch_scale': 'reward_scale',
    'deep_sea': 'size', 'deep_sea_stochastic': 'size',
    'memory_len': 'memory_length', 'memory_size': 'num_bits',
    'mnist_noise': 'noise_scale', 'mnist_scale': 'reward_scale',
    'mountain_car_noise': 'noise_scale', 'mountain_car_scale': 'reward_scale',
    'umbrella_distract': 'n_distractor', 'umbrella_length': 'chain_length',
}

# The column each rule reads besides `episode` (bsb_score_source.col_value), and best_episode where it needs it.
VALUE_COLUMNS = {name: 'total_regret' for name in EXPERIMENTS}
VALUE_COLUMNS.update({name: 'raw_return' for name in EXPERIMENTS if name.startswith(('cartpole', 'mountain_car'))})
VALUE_COLUMNS.update(cartpole_swingup='total_return', discounting_chain='total_return', deep_sea='total_bad_episodes',
                     deep_sea_stochastic='total_bad_episodes', memory_len='total_perfect', memory_size='total_perfect')
NEEDS_BEST = frozenset(name for name in EXPERIMENTS if name.startswith('cartpole'))


def experiment_of(bsuite_id: str) -> str:
  return bsuite_id.split(sweep.SEPARATOR)[0]


def group_key(bsuite_id: str) -> float:
  """The value of the id's grouping setting in sweep.SETTINGS (0 for experiments that do not group)."""
  key = GROUP_KEYS.get(experiment_of(bsuite_id))
  return float(sweep.SETTINGS[bsuite_id][key]) if key else 0.0


def _check_orders(lib):
  got = tuple(lib.bsb_experiment_name(i).decode() for i in range(_lib.NUM_EXPERIMENTS))
  tags = tuple(lib.bsb_tag_name(i).decode() for i in range(_lib.NUM_TAGS))
  if got != EXPERIMENTS or tags != TAGS:
    raise ImportError(f'{_lib.LIB_PATH} orders experiments / tags differently from bsuite_b200.scoring; rebuild')


class Scorer:
  """Scores every lane of a set of record-rows environments (one per bsuite_id, same batch and device).

  Built once, run as often as wanted: `run()` reads the rows as they are at that point of the stream, so it can
  follow the steps at any log point, and on CUDA it is one kernel launch that a CUDA graph can capture.
  """

  def __init__(self, envs_by_id: Mapping[str, Any]):
    """Reads an environment's rows when it records them (`record_rows=True`), its score summary otherwise
    (`track_scores=True`); both give the same scores."""
    sources = []
    lib = _lib.load()
    for bsuite_id, env in envs_by_id.items():
      if not (getattr(env, '_record_rows', False) or getattr(env, '_track_scores', False)):
        raise ValueError(f'{bsuite_id}: create the environment with record_rows=True or track_scores=True to score it')
      experiment = EXPERIMENTS.index(experiment_of(bsuite_id))
      source = _lib.ScoreSource()
      _lib.check(lib.bsb_score_source_from_env(env._handle.ptr, experiment, group_key(bsuite_id),  # pylint: disable=protected-access
                                               ctypes.byref(source)))
      sources.append(source)
    if not sources:
      raise ValueError('no environments to score')
    first = next(iter(envs_by_id.values()))
    self._init(sources, first.batch, first.device, keep=dict(envs_by_id))

  @classmethod
  def from_rows(cls, tables: Mapping[str, Mapping[str, Any]], device='cpu', summarize: bool = False) -> 'Scorer':
    """A scorer over caller-owned rows: bsuite_id -> dict(rows=[n_points, n_columns, B] float64,
    counts=[B] int32, columns=names of the n_columns columns), numpy arrays or tensors (copied to `device` when
    they are not already there as contiguous tensors of those dtypes).  summarize=True folds the rows into score
    summaries on the host first (`summarize`) and scores those on `device`."""
    import torch
    device = torch.device(device)
    if summarize:
      return cls.from_summaries({bsuite_id: _summarize(bsuite_id, table)
                                 for bsuite_id, table in tables.items()}, device=device)
    sources, keep, batch = [], [], None
    for bsuite_id, table in tables.items():
      source, rows, counts = _rows_source(bsuite_id, table, device)
      sources.append(source)
      keep += [rows, counts]
      batch = rows.shape[2] if batch is None else batch
    if not sources:
      raise ValueError('no rows to score')
    scorer = cls.__new__(cls)
    scorer._init(sources, batch, device, keep=keep)  # pylint: disable=protected-access
    return scorer

  @classmethod
  def from_summaries(cls, summaries: Mapping[str, Mapping[str, Any]], device='cpu') -> 'Scorer':
    """A scorer over caller-owned score summaries: bsuite_id -> dict as `summarize` or
    `BatchedEnvironment.score_summary` return it (a float64 [B] per field of `_lib.SUMMARY_FIELDS`, counts [B],
    n_points), copied to `device`."""
    import torch
    device = torch.device(device)
    sources, keep, batch = [], [], None
    for bsuite_id, summary in summaries.items():
      block = torch.stack([torch.as_tensor(summary[f]).to(device=device, dtype=torch.float64)
                           for f in _lib.SUMMARY_FIELDS]).contiguous()
      counts = torch.as_tensor(summary['counts']).to(device=device, dtype=torch.int32).contiguous()
      if block.dim() != 2 or counts.shape != (block.shape[1],):
        raise ValueError(f'{bsuite_id}: every summary field and counts must be [B]')
      sources.append(_lib.ScoreSource(
          experiment=EXPERIMENTS.index(experiment_of(bsuite_id)), device=_ordinal(device), batch=block.shape[1],
          n_points=int(summary['n_points']), n_columns=block.shape[0], col_episode=-1, col_value=-1, col_best=-1,
          layout=_lib.SCORE_SUMMARY, group_key=group_key(bsuite_id), rows=block.data_ptr(),
          counts=counts.data_ptr()))
      keep += [block, counts]
      batch = block.shape[1] if batch is None else batch
    if not sources:
      raise ValueError('no summaries to score')
    scorer = cls.__new__(cls)
    scorer._init(sources, batch, device, keep=keep)  # pylint: disable=protected-access
    return scorer

  def _init(self, sources: Sequence[Any], batch: int, device, keep):
    import torch
    self._torch = torch
    self._lib = _lib.load()
    _check_orders(self._lib)
    self._keep = keep                     # the row stores the scorer reads must outlive it
    self.batch = int(batch)
    self.device = torch.device(device)
    self._ordinal = _lib.DEVICE_HOST if self.device.type == 'cpu' else (self.device.index or 0)
    array = (_lib.ScoreSource * len(sources))(*sources)
    handle = ctypes.c_void_p()
    _lib.check(self._lib.bsb_scorer_create(array, len(sources), self.batch, self._ordinal, ctypes.byref(handle)))
    self._ptr = handle

  def empty_outputs(self) -> Dict[str, Any]:
    torch = self._torch
    kw = dict(device=self.device)
    return dict(scores=torch.empty((_lib.NUM_EXPERIMENTS, self.batch), dtype=torch.float64, **kw),
                finished=torch.empty((_lib.NUM_EXPERIMENTS, self.batch), dtype=torch.int32, **kw),
                tags=torch.empty((_lib.NUM_TAGS, self.batch), dtype=torch.float64, **kw))

  def run(self, out: Optional[Dict[str, Any]] = None) -> Dict[str, Any]:
    """scores float64 [23, B], finished int32 [23, B] and tags float64 [7, B] on the environments' device, written
    on the current stream (into `out`, a dict like `empty_outputs()`, when given)."""
    if self._ptr is None:
      raise RuntimeError('the scorer is closed')
    if out is None:
      out = self.empty_outputs()
    else:
      torch = self._torch
      for k, dtype, rows in (('scores', torch.float64, _lib.NUM_EXPERIMENTS),
                             ('finished', torch.int32, _lib.NUM_EXPERIMENTS), ('tags', torch.float64, _lib.NUM_TAGS)):
        t = out[k]
        if tuple(t.shape) != (rows, self.batch) or t.dtype != dtype or t.device != self.device or not t.is_contiguous():
          raise ValueError(f'out[{k!r}] must be a contiguous {dtype} tensor {(rows, self.batch)} on {self.device}')
    stream = None
    if self._ordinal >= 0:
      stream = self._torch.cuda.current_stream(self.device).cuda_stream
    _lib.check(self._lib.bsb_scorer_run(self._ptr, out['scores'].data_ptr(), out['finished'].data_ptr(),
                                        out['tags'].data_ptr(), stream))
    return out

  def close(self):
    if getattr(self, '_ptr', None) is not None:
      self._lib.bsb_scorer_destroy(self._ptr)
      self._ptr = None

  def __del__(self):
    try:
      self.close()
    except Exception:  # pylint: disable=broad-except
      pass


def _ordinal(device) -> int:
  return _lib.DEVICE_HOST if device.type == 'cpu' else (device.index or 0)


def _rows_source(bsuite_id: str, table: Mapping[str, Any], device):
  """A BSB_SCORE_ROWS source over `table` (see Scorer.from_rows), and the tensors it points at."""
  import torch
  name = experiment_of(bsuite_id)
  rows = torch.as_tensor(table['rows']).to(device=device, dtype=torch.float64).contiguous()
  counts = torch.as_tensor(table['counts']).to(device=device, dtype=torch.int32).contiguous()
  columns = list(table['columns'])
  if rows.dim() != 3 or rows.shape[1] != len(columns) or counts.shape != (rows.shape[2],):
    raise ValueError(f'{bsuite_id}: rows must be [n_points, len(columns), B] and counts [B]')
  index = lambda c: columns.index(c) if c in columns else -1
  source = _lib.ScoreSource(
      experiment=EXPERIMENTS.index(name), device=_ordinal(device),
      batch=rows.shape[2], n_points=rows.shape[0], n_columns=rows.shape[1], col_episode=index('episode'),
      col_value=index(VALUE_COLUMNS[name]), col_best=index('best_episode') if name in NEEDS_BEST else -1,
      group_key=group_key(bsuite_id), rows=rows.data_ptr(), counts=counts.data_ptr())
  return source, rows, counts


def summarize(bsuite_id: str, table: Mapping[str, Any]) -> Dict[str, Any]:
  """Folds one id's rows (a table as `Scorer.from_rows` takes it, or `BatchedEnvironment.logged_rows()`) into its
  score summary on the host (`bsb_score_summarize`), in the form `BatchedEnvironment.score_summary` returns:
  a CPU float64 [B] tensor per field of `_lib.SUMMARY_FIELDS`, counts, n_points and experiment.  Raises when a
  lane's episode column is not a prefix of the experiment's log schedule."""
  import torch
  lib = _lib.load()
  source, rows, counts = _rows_source(bsuite_id, table, torch.device('cpu'))
  batch = rows.shape[2]
  block = torch.empty((len(_lib.SUMMARY_FIELDS), batch), dtype=torch.float64)
  folded = torch.empty(batch, dtype=torch.int32)
  _lib.check(lib.bsb_score_summarize(ctypes.byref(source), block.data_ptr(), folded.data_ptr()))
  del rows, counts
  result = {name: block[f] for f, name in enumerate(_lib.SUMMARY_FIELDS)}
  result.update(counts=folded, n_points=int(source.n_points), experiment=experiment_of(bsuite_id))
  return result


_summarize = summarize        # Scorer.from_rows's `summarize` keyword hides the function's name there


def as_numpy(result: Mapping[str, Any]) -> Dict[str, np.ndarray]:
  """`Scorer.run()`'s tensors as host arrays."""
  return {k: v.cpu().numpy() for k, v in result.items()}
