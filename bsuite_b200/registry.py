"""`load` / `load_from_id`: the drop-in boundary (SURVEY.md 8b).

Same names, ids and keyword arguments as `bsuite/bsuite.py:57-108`.  With
`batch=None` the result is a single `dm_env.Environment` (the reference's
contract); with `batch=B` it is a `BatchedEnvironment` of B lanes.
"""

import functools
from typing import Any, Mapping, Optional, Tuple

from bsuite_b200 import experiments
from bsuite_b200 import sweep
from bsuite_b200.environment import BatchedEnvironment, DmEnvAdapter


def unpack_bsuite_id(bsuite_id: str) -> Tuple[str, int]:
  """'deep_sea/11' -> ('deep_sea', 11)   (bsuite.py:84-90)."""
  name, _, index = bsuite_id.partition(sweep.SEPARATOR)
  if not name or not index or sweep.SEPARATOR in index:
    raise ValueError(f'malformed bsuite_id {bsuite_id!r}')
  return name, int(index)


def _instantiate(spec, batch, device, seed, rng, **engine_kwargs):
  if batch is None:
    if engine_kwargs:
      raise TypeError(f'{sorted(engine_kwargs)} only apply to batched environments (pass batch=...)')
    return DmEnvAdapter(spec, device=device, seed=seed, rng=rng)
  return BatchedEnvironment(spec, batch=batch, device=device, seed=seed, rng=rng or 'philox', **engine_kwargs)


def load(experiment_name: str, kwargs: Mapping[str, Any], batch: Optional[int] = None, device='cuda',
         seed: Optional[int] = None, rng: Optional[str] = None, **engine_kwargs):
  """Returns a bsuite environment given an experiment name and settings (bsuite.py:93-98)."""
  spec = experiments.EXPERIMENT_NAME_TO_SPEC[experiment_name](**kwargs)
  if engine_kwargs.get('track_scores'):      # the score summary is the experiment's
    engine_kwargs.setdefault('score_experiment', experiment_name)
  return _instantiate(spec, batch, device, seed, rng, **engine_kwargs)


def load_from_id(bsuite_id: str, batch: Optional[int] = None, device='cuda', seed: Optional[int] = None,
                 rng: Optional[str] = None, **engine_kwargs):
  """Returns a bsuite environment given a bsuite_id (bsuite.py:101-108)."""
  kwargs = sweep.SETTINGS[bsuite_id]
  experiment_name, _ = unpack_bsuite_id(bsuite_id)
  return load(experiment_name, kwargs, batch=batch, device=device, seed=seed, rng=rng, **engine_kwargs)


def make(environment_class: str, batch: Optional[int] = None, device='cuda', seed: Optional[int] = None,
         rng: Optional[str] = None, noise_scale: Optional[float] = None, reward_scale: Optional[float] = None,
         engine_kwargs: Optional[Mapping[str, Any]] = None, **kwargs):
  """Constructs a raw environment class, e.g. make('deep_sea', size=10, deterministic=False, seed=0).

  `noise_scale` / `reward_scale` wrap it in the fused RewardNoise / RewardScale
  epilogue (utils/wrappers.py:250-373), as the `*_noise` / `*_scale` factories do.
  """
  spec = experiments.ENVIRONMENT_CLASSES[environment_class](**kwargs)
  if noise_scale is not None and reward_scale is not None:
    raise ValueError('at most one reward wrapper')
  if noise_scale is not None:
    spec = experiments._with_noise(spec, noise_scale, spec.bsuite_num_episodes)  # pylint: disable=protected-access
  if reward_scale is not None:
    spec = experiments._with_scale(spec, reward_scale, spec.bsuite_num_episodes)  # pylint: disable=protected-access
  return _instantiate(spec, batch, device, seed, rng, **(engine_kwargs or {}))


def load_and_record_to_csv(bsuite_id: str, results_dir: str, overwrite: bool = False, **kwargs):
  """A bsuite environment that saves results to CSV, loadable by the reference's csv_load (bsuite.py:126-157)."""
  from bsuite_b200 import recording  # pylint: disable=import-outside-toplevel
  return recording.Recorder(load_from_id(bsuite_id, **kwargs), recording.CsvLogger(bsuite_id, results_dir, overwrite))


def load_and_record_to_terminal(bsuite_id: str, **kwargs):
  """A bsuite environment that logs to the terminal (bsuite.py:160-167)."""
  from bsuite_b200 import recording  # pylint: disable=import-outside-toplevel
  return recording.Recorder(load_from_id(bsuite_id, **kwargs), recording.TerminalLogger())


def load_and_record(bsuite_id: str, save_path: str, logging_mode: str = 'csv', overwrite: bool = False, **kwargs):
  """CSV or terminal logging by `logging_mode` (bsuite.py:111-123)."""
  if logging_mode == 'csv':
    return load_and_record_to_csv(bsuite_id, save_path, overwrite, **kwargs)
  if logging_mode == 'terminal':
    return load_and_record_to_terminal(bsuite_id, **kwargs)
  raise ValueError(f'Unrecognised logging_mode "{logging_mode}". Must be "csv" or "terminal".')


# experiment name -> loader accepting that experiment's kwargs (bsuite.py:57-81)
EXPERIMENT_NAME_TO_ENVIRONMENT = {
    name: functools.partial(lambda _name, **kw: load(_name, kw), name)
    for name in experiments.EXPERIMENT_NAME_TO_SPEC
}
