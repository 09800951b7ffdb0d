"""Heterogeneous batches: many bsuite_ids at once (BASELINE config #5, SURVEY.md 8d/8e).

`SweepBatch` holds one `BatchedEnvironment` per bsuite_id, each with `lanes` lanes, and advances all of them
"in lock-step" from the caller's point of view: every environment's fused rollout is enqueued on its own CUDA
stream, so the 23 small kernels of a full-sweep step overlap on the GPU instead of queueing behind each other.
Across GPUs every id's lanes are sharded evenly (rank r owns lanes [r*lanes/W, (r+1)*lanes/W) of EVERY id), so the
observation-heavy families (deep_sea, mnist) do not imbalance the ranks; the only collective is the all-gather of
per-rank return statistics at log points.
"""

from typing import Dict, List, Optional, Sequence

from bsuite_b200 import distributed
from bsuite_b200 import registry
from bsuite_b200 import sweep


def one_per_experiment(setting: int = 0) -> List[str]:
  """`<experiment>/<setting>` for each of the 23 experiments (the sweep.TESTING idea, including noise/scale)."""
  return [ids[min(setting, len(ids) - 1)] for ids in sweep.BY_EXPERIMENT.values()]


# Compact lane state read + written per lane-step by family id (SURVEY.md 8d: deep_sea / catch one packed word,
# cartpole / swingup 5 x f64, mountain_car 2 x f64 + the step word, the rest a word + an 8-byte RNG position).
_STATE_BYTES = {0: 8, 1: 8, 2: 80, 3: 80, 4: 48}


def algorithmic_bytes_per_lane_step(env) -> int:
  numel = 1
  for d in env.obs_shape:
    numel *= d
  return 4 * numel + 16 + _STATE_BYTES.get(env.family, 16)


class GraphedSweep:
  """Captured lock-step(s) of a `SweepBatch` (`SweepBatch.capture`): `replay()` returns id -> TimeStep (a list of
  them, one per captured lock-step, when several were captured) -- the same tensors every time, leading axis =
  the captured number of steps."""

  def __init__(self, graph, timesteps):
    self.graph, self.timesteps = graph, timesteps

  def replay(self):
    self.graph.replay()
    return self.timesteps


class SweepBatch:

  def __init__(self, bsuite_ids: Optional[Sequence[str]] = None, lanes: int = 4096, device='cuda', seed: int = 0,
               rank: int = 0, world: int = 1, track_episodes: bool = True, ring: int = 1, record_rows: bool = False,
               track_scores: bool = False):
    import torch
    self._torch = torch
    self.bsuite_ids = list(bsuite_ids) if bsuite_ids is not None else one_per_experiment()
    first, count = distributed.shard_range(lanes, rank, world)
    self.lanes, self.local_lanes, self.lane_offset = lanes, count, first
    self.envs = {
        bsuite_id: registry.load_from_id(bsuite_id, batch=count, device=device, seed=seed, lane_offset=first,
                                         track_episodes=track_episodes, record_rows=record_rows,
                                         track_scores=track_scores)
        for bsuite_id in self.bsuite_ids
    }
    self._device = next(iter(self.envs.values())).device
    self._cuda = self._device.type == 'cuda'
    self._streams = {k: torch.cuda.Stream(device=self._device) for k in self.envs} if self._cuda else {}
    self._ring = max(1, int(ring))      # output buffer sets cycled through by successive rollouts (> L2 when timing)
    self._turn = 0
    self._buffers: Dict[str, object] = {}
    self._buffer_steps = None
    self._lp = None
    self._cols = None
    self.record_rows = bool(record_rows)
    self.track_scores = bool(track_scores)
    self._scorer = None

  def _ensure_buffers(self, num_steps: int):
    if self._buffer_steps != num_steps:
      self._buffers = {}
      self._buffers = {k: [env.make_buffers(num_steps, with_actions=True) for _ in range(self._ring)]
                       for k, env in self.envs.items()}
      self._buffer_steps = num_steps

  def rollout(self, num_steps: int, action_seed: int = 0):
    """`num_steps` fused steps of every environment (on-device uniform random actions); returns id -> TimeStep.

    The returned tensors are reused `ring` calls later.  On CUDA each environment runs on its own stream; the
    caller's current stream waits for all of them before this function returns control of the outputs.
    """
    torch = self._torch
    self._ensure_buffers(num_steps)
    slot = self._turn % self._ring
    self._turn += 1
    result = {}
    if not self._cuda or len(self.envs) == 1:      # nothing to overlap: stay on the caller's stream
      for k, env in self.envs.items():
        result[k] = env.rollout(num_steps, action_seed=action_seed, out=self._buffers[k][slot])
      return result
    current = torch.cuda.current_stream(self._device)
    for k, env in self.envs.items():
      stream = self._streams[k]
      stream.wait_stream(current)
      with torch.cuda.stream(stream):
        result[k] = env.rollout(num_steps, action_seed=action_seed, out=self._buffers[k][slot])
    for stream in self._streams.values():
      current.wait_stream(stream)
    return result

  def capture(self, num_steps: int = 1, action_seed: int = 0, lock_steps: int = 1) -> 'GraphedSweep':
    """Records `lock_steps` successive lock-steps of every id (a `num_steps`-step rollout each, on-device actions)
    into a single CUDA graph: the per-id launches fork from the capturing stream onto the ids' streams and join
    again, so a replay costs one `cudaGraphLaunch` instead of one launch per id and lock-step -- 23 launches per
    lock-step are launch-bound when each id holds a few hundred lanes (BASELINE config #5 sharded over 8 GPUs).
    Each captured lock-step writes its own output buffer set.  The environments keep their step counters on the
    device from here on (graph-safe mode), so replays and eager rollouts can be mixed."""
    torch = self._torch
    if not self._cuda:
      raise RuntimeError('CUDA graphs need CUDA environments')
    lock_steps = max(1, int(lock_steps))
    self.set_ring(lock_steps)
    self._turn = 0
    states = {k: env.state_dict() for k, env in self.envs.items()}
    self.rollout(num_steps, action_seed=action_seed)      # eager pass: module loading and function attributes
    torch.cuda.synchronize(self._device)
    for k, env in self.envs.items():
      env.load_state_dict(states[k])
    self._turn = 0
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, capture_error_mode='thread_local'):   # other threads (NCCL watchdog) may touch CUDA
      results = [self.rollout(num_steps, action_seed=action_seed) for _ in range(lock_steps)]
    return GraphedSweep(graph, results[0] if lock_steps == 1 else results)

  def set_ring(self, ring: int):
    """Number of output buffer sets successive rollouts cycle through (drops the current buffers)."""
    self._ring = max(1, int(ring))
    self._buffers, self._buffer_steps = {}, None

  def last_buffers(self, bsuite_id: str):
    """The `StepBuffers` (outputs + the actions sampled on the device) the latest rollout of `bsuite_id` wrote."""
    return self._buffers[bsuite_id][(self._turn - 1) % self._ring]

  def _log_point(self):
    if self._lp is None:
      self._lp = distributed.LogPoint(list(self.envs.values()))
      self._cols = self._torch.tensor([2, 1, 0], device=self._device)     # (total_return, episode, steps)
    return self._lp

  def issue_log_point(self) -> int:
    """Asynchronous log point (`distributed.LogPoint`): one reduction kernel per id on the current stream, writing
    into a preallocated block; the all-gather runs on a side stream, so further rollouts are not held up."""
    return self._log_point().issue()

  def log_point_result(self, ticket: int, host_sync: bool = False):
    """float64 [world, n_ids, 3]: per-rank, per-id sums of (total_return, episode, steps) of `ticket`."""
    return self._log_point().result(ticket, host_sync=host_sync).index_select(-1, self._cols)

  def join_log_points(self):
    """Makes the caller's stream wait (on the device) for every log point still in flight."""
    if self._lp is not None:
      self._lp.join()

  def local_returns(self):
    """float64 [n_ids, 3] on the device: per-id sums of (total_return, episode, steps) over this rank's lanes."""
    torch = self._torch
    block = torch.empty((len(self.envs), 5), dtype=torch.float64, device=self._device)
    for i, env in enumerate(self.envs.values()):
      env.episode_stat_sums(out=block[i])                     # one reduction kernel per id, written in place
    return block.index_select(-1, self._log_point() and self._cols)

  def gather_returns(self):
    """The one collective of the path, synchronous form: returns [world, n_ids, 3] (see `issue_log_point`)."""
    return self.log_point_result(self.issue_log_point())

  def scores(self, out=None):
    """Per-lane bsuite scores of this rank's lanes (`record_rows=True` or `track_scores=True`):
    dict(scores=[23, local_lanes], finished=[23, local_lanes], tags=[7, local_lanes]) on the batch's device,
    computed by one kernel launch on the current stream from the rows recorded so far, or from the score summaries
    kept in their place (`scoring.Scorer`; both give the same bits).  Lanes are independent runs, so a rank needs
    no collective to score; a caller that wants the whole population gathers these blocks itself."""
    if not (self.record_rows or self.track_scores):
      raise RuntimeError('SweepBatch.scores() needs the rows or score summaries of every lane: create the SweepBatch '
                         'with record_rows=True or track_scores=True')
    if self._scorer is None:
      from bsuite_b200 import scoring  # pylint: disable=import-outside-toplevel
      self._scorer = scoring.Scorer(self.envs)
    return self._scorer.run(out)

  def bytes_per_step(self) -> int:
    """Algorithmic bytes of one lock-step of the whole local batch (SURVEY.md 8d: dense observation + action +
    reward + discount + step_type + compact lane state read and written)."""
    return sum(env.batch * algorithmic_bytes_per_lane_step(env) for env in self.envs.values())

  def close(self):
    if self._scorer is not None:
      self._scorer.close()
      self._scorer = None
    for env in self.envs.values():
      env.close()
