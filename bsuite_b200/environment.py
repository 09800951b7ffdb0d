"""Python faces of the engine.

`BatchedEnvironment`  -- B lanes of one bsuite environment stepping in lock-step;
    `reset()/step(actions)` return a `dm_env.TimeStep` whose fields are torch
    tensors living on the environment's device (agents consume observations on
    the GPU directly).  FIRST lanes carry reward = 0 / discount = 0 and are
    identified by `step_type == 0` (the reference returns `None` there).
`DmEnvAdapter`        -- a B = 1 `dm_env.Environment` with numpy observations,
    Python-float rewards and `None` on FIRST: the object contract of
    `bsuite/environments/base.py:34-77`, for unmodified agents.

Both call the C ABI (include/bsuite_b200.h) through ctypes; torch is used only
to allocate device memory and to pick the CUDA stream.
"""

import ctypes
from typing import Any, Dict, Optional

import numpy as np

from bsuite_b200 import _lib
from bsuite_b200 import dm_env
from bsuite_b200.experiments import EnvSpec

specs = dm_env.specs

_INT_INFO = frozenset(['total_bad_episodes', 'total_perfect'])
_MASK64 = (1 << 64) - 1


def _fresh_seed() -> int:
  """seed=None in the reference means OS entropy (numpy RandomState(None))."""
  return int(np.random.SeedSequence().generate_state(1, dtype=np.uint32)[0])


def _resolve_device(device) -> int:
  """Returns a CUDA ordinal or DEVICE_HOST; never silently falls back."""
  import torch
  if device is None:
    device = 'cuda'
  dev = torch.device(device)
  if dev.type == 'cpu':
    return _lib.DEVICE_HOST
  if dev.type != 'cuda':
    raise ValueError(f'unsupported device {device!r}: expected "cuda[:i]" or "cpu"')
  if not torch.cuda.is_available():
    raise RuntimeError(
        'bsuite_b200: a CUDA device was requested but none is available. There is no implicit CPU '
        'fallback; pass device="cpu" explicitly to use the host path of the C ABI.')
  return dev.index if dev.index is not None else torch.cuda.current_device()


def _make_config(spec: EnvSpec, rng_kind: int, flags: int, log_schedule=None, score_experiment: int = 0):
  cfg = _lib.Config()
  cfg.family = spec.family
  cfg.wrapper = spec.wrapper
  cfg.rng_kind = rng_kind
  cfg.flags = flags
  cfg.score_experiment = score_experiment
  cfg.deterministic = 1
  cfg.reward_scale = 1.0
  for key, value in spec.fields.items():
    setattr(cfg, key, value)
  keep = []
  if spec.table is not None:
    table = np.ascontiguousarray(spec.table)
    cfg.table = table.ctypes.data
    cfg.table_bytes = table.nbytes
    keep.append(table)
  if spec.table2 is not None:
    table2 = np.ascontiguousarray(spec.table2)
    cfg.table2 = table2.ctypes.data
    cfg.table2_bytes = table2.nbytes
    keep.append(table2)
  if log_schedule is not None and len(log_schedule):
    schedule = np.ascontiguousarray(log_schedule, dtype=np.int64)
    cfg.log_schedule = schedule.ctypes.data
    cfg.log_schedule_len = schedule.size
    keep.append(schedule)
  return cfg, keep


class _Handle:
  """Owns one bsb_env*."""

  def __init__(self, spec: EnvSpec, batch: int, device_ordinal: int, seed: int, lane_offset: int,
               rng_kind: int, flags: int, log_schedule=None, score_experiment: int = 0):
    self.lib = _lib.load()
    cfg, keep = _make_config(spec, rng_kind, flags, log_schedule, score_experiment)
    ptr = ctypes.c_void_p()
    _lib.check(self.lib.bsb_create(ctypes.byref(cfg), batch, device_ordinal, seed & _MASK64,
                                   lane_offset & _MASK64, ctypes.byref(ptr)))
    del keep
    self.ptr = ptr

  def close(self):
    if self.ptr is not None and self.ptr.value:
      self.lib.bsb_destroy(self.ptr)
      self.ptr = None

  def __del__(self):
    try:
      self.close()
    except Exception:  # interpreter shutdown
      pass


class StepBuffers:
  """Caller-owned output tensors for one step (or T fused steps)."""

  def __init__(self, observation, reward, discount, step_type, actions=None):
    self.observation = observation
    self.reward = reward
    self.discount = discount
    self.step_type = step_type
    self.actions = actions
    self._outputs = None      # struct bsb_outputs over these tensors, built once (the tensors are never swapped)
    self._timestep = None

  def as_outputs(self) -> _lib.Outputs:
    if self._outputs is None:
      self._outputs = self._build_outputs()
    return self._outputs

  def _build_outputs(self) -> _lib.Outputs:
    import torch
    out = _lib.Outputs()
    if self.observation is not None:
      out.observation = self.observation.data_ptr()
    if self.reward is not None:
      if self.reward.dtype == torch.float64:
        out.reward_f64 = self.reward.data_ptr()
      else:
        out.reward = self.reward.data_ptr()
    if self.discount is not None:
      out.discount = self.discount.data_ptr()
    if self.step_type is not None:
      out.step_type = self.step_type.data_ptr()
    return out

  def timestep(self) -> 'dm_env.TimeStep':
    if self._timestep is None:
      self._timestep = dm_env.TimeStep(step_type=self.step_type, reward=self.reward, discount=self.discount,
                                       observation=self.observation)
    return self._timestep


class GraphedSteps:
  """`num_steps` step() calls of one environment recorded in a CUDA graph (`BatchedEnvironment.capture`).

  Write the next actions into `actions` ([T, B] int32, absent when the actions are sampled on the device), call
  `replay()`, read `timestep` (fields with a leading T axis, the same tensors every time).  The environment keeps
  its step count on the device from the first capture on, so eager calls and replays can be mixed freely."""

  def __init__(self, env, graph, actions, buffers):
    self.env = env
    self.graph = graph
    self.actions = actions
    self.buffers = buffers
    self.timestep = buffers.timestep()

  def replay(self):
    self.graph.replay()
    return self.timestep


class BatchedEnvironment:
  """`batch` independent lanes of one environment on one device."""

  def __init__(self, spec: EnvSpec, batch: int, device='cuda', seed: Optional[int] = None,
               rng: str = 'philox', lane_offset: int = 0, track_episodes: bool = False,
               reward_dtype='float32', record_rows: bool = False, track_scores: bool = False,
               score_experiment: Optional[str] = None):
    import torch
    self._torch = torch
    self._spec = spec
    self._batch = int(batch)
    self._ordinal = _resolve_device(device)
    self._device = torch.device('cpu') if self._ordinal < 0 else torch.device('cuda', self._ordinal)
    if rng not in ('philox', 'mt19937'):
      raise ValueError(f'rng must be "philox" or "mt19937", got {rng!r}')
    self._rng_kind = _lib.RNG_PHILOX if rng == 'philox' else _lib.RNG_MT19937
    # An explicit engine `seed` wins; otherwise the experiment's own default (memory_len, memory_size and
    # umbrella_distract fix seed=0: experiments/memory_len/memory_len.py:31-37), otherwise OS entropy.
    seed = seed if seed is not None else spec.seed
    self._seed = _fresh_seed() if seed is None else int(seed)
    if self._rng_kind == _lib.RNG_MT19937 and not 0 <= self._seed < 2**32:
      raise ValueError('Seed must be between 0 and 2**32 - 1')   # numpy's own message
    self._lane_offset = int(lane_offset)
    self._async_work = False        # something was enqueued on a torch stream since the last host-driven step
    # record_rows: every lane keeps the rows the reference's Logging wrapper would have written for it, at the
    # log-spaced episode counts of utils/wrappers.py:140-147 (recording.write_lane_csvs turns them into files)
    # track_scores: every lane keeps only what experiment `score_experiment`'s scoring rule reads of those rows (a
    # score summary, 48 bytes per lane), folded in as the rows fall due; scoring.Scorer scores from it
    track_episodes = bool(track_episodes or record_rows or track_scores)
    flags = _lib.FLAG_TRACK_EPISODES if track_episodes else 0
    self._track = bool(track_episodes)
    self._record_rows, self._track_scores = bool(record_rows), bool(track_scores)
    self._log_schedule = None
    self._score_experiment = None
    experiment_index = 0
    if record_rows or track_scores:
      from bsuite_b200 import recording  # pylint: disable=import-outside-toplevel
      self._log_schedule = recording.log_schedule(spec.bsuite_num_episodes)
    if track_scores:
      from bsuite_b200 import scoring  # pylint: disable=import-outside-toplevel
      if score_experiment not in scoring.EXPERIMENTS:
        raise ValueError(f'track_scores=True needs score_experiment, one of the 23 experiment names (got '
                         f'{score_experiment!r}); load / load_from_id set it')
      self._score_experiment = score_experiment
      experiment_index = scoring.EXPERIMENTS.index(score_experiment)
      flags |= _lib.FLAG_SCORE_SUMMARY | (0 if record_rows else _lib.FLAG_NO_LOG_ROWS)
    self._reward_dtype = torch.float64 if str(reward_dtype).endswith('64') else torch.float32
    self._handle = _Handle(spec, self._batch, self._ordinal, self._seed, self._lane_offset, self._rng_kind, flags,
                           self._log_schedule, experiment_index)
    self._lib = self._handle.lib
    n = ctypes.c_int32()
    _lib.check(self._lib.bsb_info_count(self._handle.ptr, ctypes.byref(n)))
    self._info_names = tuple(self._lib.bsb_info_name(self._handle.ptr, k).decode() for k in range(n.value))
    self.bsuite_num_episodes = spec.bsuite_num_episodes

  # ---- metadata ------------------------------------------------------------
  batch = property(lambda self: self._batch)
  device = property(lambda self: self._device)
  seed = property(lambda self: self._seed)
  lane_offset = property(lambda self: self._lane_offset)
  obs_shape = property(lambda self: self._spec.obs_shape)
  family = property(lambda self: self._spec.family)
  num_actions = property(lambda self: self._spec.num_actions)
  info_names = property(lambda self: self._info_names)

  def observation_spec(self):
    """Per-lane spec, identical to the reference environment's."""
    if self._spec.obs_bounds is not None:
      lo, hi = self._spec.obs_bounds
      return specs.BoundedArray(shape=self._spec.obs_shape, dtype=np.float32, name=self._spec.obs_spec_name,
                                minimum=lo, maximum=hi)
    return specs.Array(shape=self._spec.obs_shape, dtype=np.float32, name=self._spec.obs_spec_name)

  def action_spec(self):
    return specs.DiscreteArray(self._spec.num_actions, dtype=self._spec.action_dtype, name='action')

  # ---- buffers -------------------------------------------------------------
  def make_buffers(self, num_steps: Optional[int] = None, with_actions: bool = False) -> StepBuffers:
    torch = self._torch
    lead = (self._batch,) if num_steps is None else (int(num_steps), self._batch)
    kw = dict(device=self._device)
    return StepBuffers(
        observation=torch.empty(lead + tuple(self._spec.obs_shape), dtype=torch.float32, **kw),
        reward=torch.empty(lead, dtype=self._reward_dtype, **kw),
        discount=torch.empty(lead, dtype=torch.float32, **kw),
        step_type=torch.empty(lead, dtype=torch.int32, **kw),
        actions=torch.empty(lead, dtype=torch.int32, **kw) if with_actions else None)

  def _stream(self):
    if self._ordinal < 0:
      return None
    raw = getattr(self._torch._C, '_cuda_getCurrentRawStream', None)   # the cudaStream_t as an int, no wrapper object
    if raw is not None:
      return raw(self._ordinal)
    return self._torch.cuda.current_stream(self._device).cuda_stream

  def _device_actions(self, actions, shape):
    torch = self._torch
    if not isinstance(actions, torch.Tensor):
      actions = torch.as_tensor(np.asarray(actions))
    if tuple(actions.shape) != tuple(shape):
      raise ValueError(f'actions must have shape {tuple(shape)}, got {tuple(actions.shape)}')
    if actions.dtype != torch.int32 or actions.device != self._device or not actions.is_contiguous():
      actions = actions.to(device=self._device, dtype=torch.int32, non_blocking=True).contiguous()
    return actions

  # ---- dynamics ------------------------------------------------------------
  def reset(self, out: Optional[StepBuffers] = None):
    """base.Environment.reset for every lane (base.py:54-57)."""
    out = out or self.make_buffers()
    outputs = out.as_outputs()
    self._async_work = True
    _lib.check(self._lib.bsb_reset(self._handle.ptr, ctypes.byref(outputs), self._stream()))
    return out.timestep()

  def step(self, actions, out: Optional[StepBuffers] = None):
    """base.Environment.step for every lane (base.py:59-65); actions int [B]."""
    torch = self._torch
    if not (type(actions) is torch.Tensor and actions.dtype is torch.int32 and actions.dim() == 1
            and actions.shape[0] == self._batch and actions.is_contiguous()
            and (actions.device == self._device
                 # zero-copy: a PINNED host tensor is device-addressable at the same address (unified addressing),
                 # the kernel reads it in place over PCIe; nothing is copied and nothing synchronises
                 or (self._ordinal >= 0 and actions.device.type == 'cpu' and actions.is_pinned()))):
      actions = self._device_actions(actions, (self._batch,))
    if out is None:
      out = self.make_buffers()
    self._async_work = True
    status = self._lib.bsb_step(self._handle.ptr, actions.data_ptr(), ctypes.byref(out.as_outputs()), self._stream())
    if status:
      _lib.check(status)
    return out.timestep()

  def make_mixed_buffers(self) -> StepBuffers:
    """Observation on the device, reward / discount / step_type in PINNED host memory: passed as `out=` to `step()`
    the kernel writes the scalars straight into host memory (zero-copy), asynchronously -- synchronise the stream
    (or an event) before reading them on the host."""
    torch = self._torch
    if self._ordinal < 0:
      return self.make_buffers()
    host = self.make_host_buffers()
    return StepBuffers(observation=torch.empty((self._batch,) + tuple(self._spec.obs_shape), dtype=torch.float32,
                                               device=self._device),
                       reward=host.reward, discount=host.discount, step_type=host.step_type)

  def make_host_buffers(self, with_observation: bool = False) -> StepBuffers:
    """Pinned host tensors for `step_host` (reward / discount / step_type, optionally the observation).

    The three scalar arrays are views of ONE pinned block, back to back, so `bsb_step_host` returns them with a
    single device-to-host copy."""
    torch = self._torch
    pin = self._ordinal >= 0
    B = self._batch
    if self._reward_dtype == torch.float32:
      block = torch.empty(3 * B, dtype=torch.float32, pin_memory=pin)
      reward, discount, step_type = block[:B], block[B:2 * B], block[2 * B:].view(torch.int32)
    else:
      reward = torch.empty(B, dtype=torch.float64, pin_memory=pin)
      discount = torch.empty(B, dtype=torch.float32, pin_memory=pin)
      step_type = torch.empty(B, dtype=torch.int32, pin_memory=pin)
    observation = (torch.empty((B,) + tuple(self._spec.obs_shape), dtype=torch.float32, pin_memory=pin)
                   if with_observation else None)
    return StepBuffers(observation=observation, reward=reward, discount=discount, step_type=step_type)

  def step_host(self, actions, host: StepBuffers, out: Optional[StepBuffers] = None, prelaunch: bool = False,
                wait: bool = True):
    """One step driven from HOST memory through `bsb_step_host`: the reference's call pattern, one
    `env.step(action)` per decision (baselines/experiment.py:45-57), for agents whose policy runs on the host.

    `actions`: CPU int32 tensor [batch] (ideally pinned: the kernel then reads it in place over PCIe); reward /
    discount / step_type (and the observation if `host.observation` is set) are delivered into `host`; the call
    returns after everything has landed.  Observations are also left on the device in `out.observation` for the
    agent.  Returns (host TimeStep, device observation).  Actions outside [0, num_actions) raise `EngineError`.

    Stream order: the step runs on a stream the handle owns.  Work enqueued earlier on this environment through
    `reset()` / `step()` / `rollout()` on the current torch stream is waited for on the device (the handle's
    stream is fenced behind the current stream the first time a host-driven step follows such work).

    `prelaunch=True` (pinned buffers, CUDA): the next step's kernel is queued immediately and waits for this
    method's next call on a doorbell in pinned memory, so a call costs neither a kernel launch nor a stream
    synchronise.  The waiting kernel occupies the GPU: use it for host-side policies in a tight loop; any other
    method of this environment (or 200 ms without a call) stands it down.

    `wait=False` (pinned buffers, CUDA): returns once the step is enqueued; `host` holds the results after
    `host_wait()`.  `rollouts.HostHalves` uses it to drive two half-batches alternately (`BSB_HOST_NO_WAIT`).
    """
    torch = self._torch
    if not (type(actions) is torch.Tensor and actions.dtype is torch.int32 and actions.device.type == 'cpu'
            and actions.dim() == 1 and actions.shape[0] == self._batch and actions.is_contiguous()):
      if not isinstance(actions, torch.Tensor):
        actions = torch.as_tensor(np.asarray(actions))
      if actions.device.type != 'cpu' or actions.dtype != torch.int32 or tuple(actions.shape) != (self._batch,):
        raise ValueError('step_host takes a CPU int32 tensor of shape [batch]')
      actions = actions.contiguous()
    if out is None:
      out = self.make_buffers()
    houts = host.as_outputs()          # struct bsb_outputs over the host tensors, built once per StepBuffers
    dev_obs = None if self._ordinal < 0 else out.observation.data_ptr()
    if self._ordinal < 0:        # host environment: one memory space; `out.observation` is the observation
      houts = _lib.Outputs.from_buffer_copy(houts)
      houts.observation = out.observation.data_ptr()
    flags = (_lib.HOST_PRELAUNCH if prelaunch else 0) | (0 if wait else _lib.HOST_NO_WAIT)
    stream = None
    if self._ordinal >= 0:
      # fence torch's current stream behind the step: deep_sea / catch return as soon as the scalars have landed
      # (two-phase host step), the observation is complete for whatever is enqueued on this stream afterwards
      flags |= _lib.HOST_FENCE_CALLER
      stream = self._stream()
      if self._async_work:
        flags |= _lib.HOST_ORDER_AFTER_STREAM
        self._async_work = False
    status = self._lib.bsb_step_host(self._handle.ptr, actions.data_ptr(), ctypes.byref(houts), dev_obs, stream, flags)
    if status:
      _lib.check(status)
    if self._ordinal < 0 and host.observation is not None:
      host.observation.copy_(out.observation)
    return host.timestep(), out.observation

  def host_wait(self):
    """Completes a `step_host(..., wait=False)`: returns when its host outputs have landed (no-op otherwise)."""
    status = self._lib.bsb_host_wait(self._handle.ptr)
    if status:
      _lib.check(status)

  def host_flush(self):
    """Stands down a kernel queued by `step_host(..., prelaunch=True)` (every other method does so implicitly)."""
    _lib.check(self._lib.bsb_host_flush(self._handle.ptr))

  def invalid_actions_seen(self) -> bool:
    """True if a DEVICE-resident action tensor passed to `step()` / `rollout()` since the last call held a value
    outside [0, num_actions): the kernels clamp such actions before any table lookup and raise a flag (host
    actions are rejected up front instead).  Synchronises the current stream."""
    if self._ordinal >= 0:
      self._torch.cuda.current_stream(self._device).synchronize()
    seen = ctypes.c_int32()
    _lib.check(self._lib.bsb_invalid_actions(self._handle.ptr, ctypes.byref(seen)))
    return bool(seen.value)

  def rollout(self, num_steps: int, actions=None, action_seed: int = 0, out: Optional[StepBuffers] = None):
    """`num_steps` fused step() calls; actions [T,B] or None for on-device uniform random actions.

    Returns a TimeStep with a leading T axis; when `out.actions` is set it receives the actions used.
    """
    num_steps = int(num_steps)
    out = out or self.make_buffers(num_steps, with_actions=actions is None)
    act_ptr = None
    if actions is not None:
      actions = self._device_actions(actions, (num_steps, self._batch))
      act_ptr = ctypes.c_void_p(actions.data_ptr())
    outputs = out.as_outputs()
    act_out = ctypes.c_void_p(out.actions.data_ptr()) if out.actions is not None else None
    self._async_work = True
    _lib.check(self._lib.bsb_rollout(self._handle.ptr, num_steps, act_ptr, int(action_seed) & _MASK64,
                                     ctypes.byref(outputs), act_out, self._stream()))
    return out.timestep()

  def capture(self, num_steps: int = 1, sample_actions: bool = False, fused: bool = False,
              action_seed: int = 0) -> GraphedSteps:
    """Records `num_steps` steps into a CUDA graph: one launch per step (`fused=False`, the reference's call
    pattern, baselines/experiment.py:45-57) or one fused rollout launch.  Launch arguments are frozen in a graph,
    so the library moves this handle's step counter and chunk scheduler to device memory when it sees the capture
    (include/bsuite_b200.h, "CUDA graphs").  One eager pass is made first on a snapshot of the lane state (module
    loading and function attributes must not happen inside a capture); the state is restored before recording."""
    torch = self._torch
    if self._ordinal < 0:
      raise RuntimeError('CUDA graphs need a CUDA environment')
    T = int(num_steps)
    buffers = self.make_buffers(T, with_actions=sample_actions)
    actions = None if sample_actions else torch.zeros((T, self._batch), dtype=torch.int32, device=self._device)
    slices = [StepBuffers(buffers.observation[t:t + 1], buffers.reward[t:t + 1], buffers.discount[t:t + 1],
                          buffers.step_type[t:t + 1], None if buffers.actions is None else buffers.actions[t:t + 1])
              for t in range(T)]

    def record():
      if fused:
        self.rollout(T, actions=actions, action_seed=action_seed, out=buffers)
      else:
        for t in range(T):
          self.rollout(1, actions=None if actions is None else actions[t:t + 1], action_seed=action_seed, out=slices[t])

    state = self.state_dict()
    record()
    torch.cuda.synchronize(self._device)
    self.load_state_dict(state)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, capture_error_mode='thread_local'):   # other threads (NCCL watchdog) may touch CUDA
      record()
    return GraphedSteps(self, graph, actions, buffers)

  def random_actions(self, num_steps: int, action_seed: int = 0, first_step: Optional[int] = None) -> np.ndarray:
    """Host mirror of the on-device action sampler for this environment's lanes."""
    if first_step is None:
      first_step = self.steps_done
    out = np.empty((int(num_steps), self._batch), dtype=np.int32)
    _lib.check(self._lib.bsb_random_actions(int(action_seed) & _MASK64, self._lane_offset, self._batch,
                                            int(first_step), int(num_steps), self._spec.num_actions,
                                            ctypes.c_void_p(out.ctypes.data)))
    return out

  @property
  def steps_done(self) -> int:
    n = ctypes.c_int64()
    _lib.check(self._lib.bsb_steps_done(self._handle.ptr, ctypes.byref(n)))
    return n.value

  # ---- accumulators ----------------------------------------------------------
  def bsuite_info(self) -> Dict[str, Any]:
    """Per-lane `bsuite_info()` accumulators as float64 tensors [B]."""
    torch = self._torch
    result = {}
    for k, name in enumerate(self._info_names):
      dst = torch.empty(self._batch, dtype=torch.float64, device=self._device)
      _lib.check(self._lib.bsb_read_info(self._handle.ptr, k, ctypes.c_void_p(dst.data_ptr()), self._stream()))
      result[name] = dst
    return result

  def episode_stats(self) -> Dict[str, Any]:
    """Logging-wrapper columns (utils/wrappers.py:85-110) per lane, float64 [B]."""
    if not self._track:
      raise RuntimeError('create the environment with track_episodes=True')
    torch = self._torch
    result = {}
    for k, name in enumerate(_lib.EPISODE_STAT_FIELDS):
      dst = torch.empty(self._batch, dtype=torch.float64, device=self._device)
      _lib.check(self._lib.bsb_read_episode_stats(self._handle.ptr, k, ctypes.c_void_p(dst.data_ptr()), self._stream()))
      result[name] = dst
    return result

  def logged_rows(self) -> Dict[str, Any]:
    """The per-lane log rows recorded on the device (`record_rows=True`): `columns` (the reference wrapper's five
    columns + the bsuite_info() keys), `rows` float64 [n_points, n_columns, B], `counts` int32 [B] (rows recorded
    so far per lane) and `schedule` (episode count of every row index)."""
    if not self._record_rows:
      raise RuntimeError('create the environment with record_rows=True')
    torch = self._torch
    n_points, n_cols = ctypes.c_int32(), ctypes.c_int32()
    _lib.check(self._lib.bsb_log_layout(self._handle.ptr, ctypes.byref(n_points), ctypes.byref(n_cols)))
    rows = torch.empty((n_points.value, n_cols.value, self._batch), dtype=torch.float64, device=self._device)
    counts = torch.empty(self._batch, dtype=torch.int32, device=self._device)
    _lib.check(self._lib.bsb_read_log_rows(self._handle.ptr, rows.data_ptr(), counts.data_ptr(), self._stream()))
    return dict(columns=_lib.EPISODE_STAT_FIELDS + self._info_names, rows=rows, counts=counts,
                schedule=np.asarray(self._log_schedule))

  def score_summary(self) -> Dict[str, Any]:
    """The per-lane score summary kept on the device (`track_scores=True`): float64 [B] per field of
    `_lib.SUMMARY_FIELDS` (bsb_read_score_summary explains them), `counts` int32 [B] (rows folded in so far per
    lane), `n_points` (length of the log schedule) and `experiment` (the experiment it is kept for)."""
    if not self._track_scores:
      raise RuntimeError('create the environment with track_scores=True')
    torch = self._torch
    block = torch.empty((len(_lib.SUMMARY_FIELDS), self._batch), dtype=torch.float64, device=self._device)
    counts = torch.empty(self._batch, dtype=torch.int32, device=self._device)
    _lib.check(self._lib.bsb_read_score_summary(self._handle.ptr, block.data_ptr(), counts.data_ptr(), self._stream()))
    result = {name: block[f] for f, name in enumerate(_lib.SUMMARY_FIELDS)}
    result.update(counts=counts, n_points=len(self._log_schedule), experiment=self._score_experiment)
    return result

  def episode_stat_sums(self, out=None):
    """Sums over this environment's lanes of (steps, episode, total_return, episode_len, episode_return): a float64
    tensor [5] on the environment's device, produced by ONE reduction kernel (`bsb_sum_episode_stats`).  `out`
    (contiguous float64 [5] on the same device, e.g. a row of a preallocated log-point block) receives the sums
    in place, so a log point allocates nothing."""
    if not self._track:
      raise RuntimeError('create the environment with track_episodes=True')
    torch = self._torch
    if out is None:
      out = torch.empty(5, dtype=torch.float64, device=self._device)
    elif not (out.dtype is torch.float64 and out.numel() == 5 and out.is_contiguous() and out.device == self._device):
      raise ValueError('out must be a contiguous float64 tensor of 5 elements on the environment\'s device')
    _lib.check(self._lib.bsb_sum_episode_stats(self._handle.ptr, out.data_ptr(), self._stream()))
    return out

  # ---- checkpoint ------------------------------------------------------------
  def state_dict(self) -> Dict[str, Any]:
    n = ctypes.c_int64()
    _lib.check(self._lib.bsb_state_bytes(self._handle.ptr, ctypes.byref(n)))
    blob = np.empty(n.value, dtype=np.uint8)
    _lib.check(self._lib.bsb_get_state(self._handle.ptr, ctypes.c_void_p(blob.ctypes.data), n.value, self._stream()))
    return dict(blob=blob, batch=self._batch, seed=self._seed, lane_offset=self._lane_offset,
                family=self._spec.family, config=self._config_fingerprint())

  def load_state_dict(self, state: Dict[str, Any]):
    if (state['batch'], state['family']) != (self._batch, self._spec.family):
      raise ValueError('state_dict belongs to a different environment')
    if (state['seed'], state['lane_offset']) != (self._seed, self._lane_offset):
      raise ValueError('state_dict was taken with different (seed, lane_offset); RNG keys would not match')
    if state.get('config', self._config_fingerprint()) != self._config_fingerprint():
      raise ValueError('state_dict was taken from a differently configured environment (fields, wrapper, rng or tracking differ)')
    blob = np.ascontiguousarray(state['blob'], dtype=np.uint8)
    _lib.check(self._lib.bsb_set_state(self._handle.ptr, ctypes.c_void_p(blob.ctypes.data), blob.nbytes, self._stream()))

  def _config_fingerprint(self) -> str:
    """Everything that shapes the meaning of the snapshot bytes besides (batch, family, seed, lane_offset)."""
    import hashlib
    h = hashlib.sha256()
    key = (sorted(self._spec.fields.items()), self._spec.wrapper, self._rng_kind, self._track,
           tuple(self._spec.obs_shape), self._spec.num_actions)
    if self._track_scores:                # only when on: the fingerprints of other configurations stay as they were
      key += (('track_scores', self._score_experiment, self._record_rows),)
    h.update(repr(key).encode())
    for table in (self._spec.table, self._spec.table2):
      if table is not None:
        h.update(np.ascontiguousarray(table).tobytes())
    return h.hexdigest()[:16]

  def close(self):
    self._handle.close()


class DmEnvAdapter(dm_env.Environment):
  """A single environment instance with the reference's object contract.

  Replaces `bsuite.load_from_id(bsuite_id)` / `bsuite.load(name, kwargs)`
  (bsuite/bsuite.py:93-108) for unmodified agents: numpy float32 observation,
  Python float reward / discount, `None` reward and discount on FIRST,
  `bsuite_info()` dict, `bsuite_num_episodes` attribute.
  """

  def __init__(self, spec: EnvSpec, device='cuda', seed: Optional[int] = None, rng: Optional[str] = None):
    self._spec = spec
    self._ordinal = _resolve_device(device)
    seed = seed if seed is not None else spec.seed
    if rng is None:
      rng = 'mt19937'   # numpy.random.RandomState(seed): the unpatched reference's stream
    self._seed = _fresh_seed() if seed is None else int(seed)
    rng_kind = _lib.RNG_PHILOX if rng == 'philox' else _lib.RNG_MT19937
    if rng_kind == _lib.RNG_MT19937 and not 0 <= self._seed < 2**32:
      raise ValueError('Seed must be between 0 and 2**32 - 1')
    self._handle = _Handle(spec, 1, self._ordinal, self._seed, 0, rng_kind, 0)
    self._lib = self._handle.lib
    n = ctypes.c_int32()
    _lib.check(self._lib.bsb_info_count(self._handle.ptr, ctypes.byref(n)))
    self._info_names = tuple(self._lib.bsb_info_name(self._handle.ptr, k).decode() for k in range(n.value))
    self.bsuite_num_episodes = spec.bsuite_num_episodes
    numel = int(np.prod(spec.obs_shape))
    self._obs = np.zeros(numel, dtype=np.float32)
    self._reward = np.zeros(1, dtype=np.float64)
    self._discount = np.zeros(1, dtype=np.float32)
    self._step_type = np.zeros(1, dtype=np.int32)
    self._action = np.zeros(1, dtype=np.int32)
    self._outputs = _lib.Outputs()
    self._outputs.observation = self._obs.ctypes.data
    self._outputs.reward_f64 = self._reward.ctypes.data
    self._outputs.discount = self._discount.ctypes.data
    self._outputs.step_type = self._step_type.ctypes.data
    # the per-step call passes the same three pointers every time: build their ctypes objects once
    self._action_ptr = ctypes.c_void_p(self._action.ctypes.data)
    self._outputs_ref = ctypes.byref(self._outputs)
    self._step_types = tuple(dm_env.StepType(k) for k in range(3))
    # ... and read / write the four scalars through ctypes views of the same memory (a numpy scalar index costs more
    # than the whole bandit transition)
    self._action_c = ctypes.c_int32.from_address(self._action.ctypes.data)
    self._reward_c = ctypes.c_double.from_address(self._reward.ctypes.data)
    self._discount_c = ctypes.c_float.from_address(self._discount.ctypes.data)
    self._step_type_c = ctypes.c_int32.from_address(self._step_type.ctypes.data)
    self._obs_view = self._obs.reshape(spec.obs_shape)
    self._dev = None
    self._reset_stream, self._host_flags = None, 0   # the next host step is fenced behind the stream reset() used
    if self._ordinal >= 0:   # device-side scratch for reset(); step() uses bsb_step_host
      import torch
      device_t = torch.device('cuda', self._ordinal)
      self._dev = StepBuffers(
          observation=torch.empty(numel, dtype=torch.float32, device=device_t),
          reward=torch.empty(1, dtype=torch.float64, device=device_t),
          discount=torch.empty(1, dtype=torch.float32, device=device_t),
          step_type=torch.empty(1, dtype=torch.int32, device=device_t))

  def _timestep(self):
    code = self._step_type_c.value
    observation = self._obs_view.copy()                            # caller owns a fresh array
    if code == 0:                                                  # FIRST: reward and discount are None (dm_env.restart)
      return dm_env.TimeStep(self._step_types[0], None, None, observation)
    return dm_env.TimeStep(self._step_types[code], self._reward_c.value, self._discount_c.value, observation)

  def reset(self):
    if self._ordinal < 0:
      _lib.check(self._lib.bsb_reset(self._handle.ptr, ctypes.byref(self._outputs), None))
    else:
      import torch
      outputs = self._dev.as_outputs()
      stream = ctypes.c_void_p(torch.cuda.current_stream(self._dev.observation.device).cuda_stream)
      self._reset_stream, self._host_flags = stream, _lib.HOST_ORDER_AFTER_STREAM
      _lib.check(self._lib.bsb_reset(self._handle.ptr, ctypes.byref(outputs), stream))
      self._obs[:] = self._dev.observation.cpu().numpy()
      self._reward[:] = self._dev.reward.cpu().numpy()
      self._discount[:] = self._dev.discount.cpu().numpy()
      self._step_type[:] = self._dev.step_type.cpu().numpy()
    return self._timestep()

  def step(self, action):
    action = int(action)
    if not 0 <= action < self._spec.num_actions:
      # the reference indexes a table with the action and fails with IndexError (bandit.py:61, catch.py:84) or
      # silently takes "the other" branch (deep_sea.py:118); an action_spec violation is an error here
      raise ValueError(f'action {action} is outside the action_spec: DiscreteArray(num_values={self._spec.num_actions})')
    self._action_c.value = action
    if self._ordinal < 0:
      status = self._lib.bsb_step(self._handle.ptr, self._action_ptr, self._outputs_ref, None)
    else:
      status = self._lib.bsb_step_host(self._handle.ptr, self._action_ptr, self._outputs_ref, None, self._reset_stream,
                                       self._host_flags)
      self._host_flags = 0
    if status:
      _lib.check(status)
    return self._timestep()

  def observation_spec(self):
    if self._spec.obs_bounds is not None:
      lo, hi = self._spec.obs_bounds
      return specs.BoundedArray(shape=self._spec.obs_shape, dtype=np.float32, name=self._spec.obs_spec_name,
                                minimum=lo, maximum=hi)
    return specs.Array(shape=self._spec.obs_shape, dtype=np.float32, name=self._spec.obs_spec_name)

  def action_spec(self):
    return specs.DiscreteArray(self._spec.num_actions, dtype=self._spec.action_dtype, name='action')

  def bsuite_info(self) -> Dict[str, Any]:
    result = {}
    for k, name in enumerate(self._info_names):
      if self._ordinal < 0:
        value = np.zeros(1, dtype=np.float64)
        _lib.check(self._lib.bsb_read_info(self._handle.ptr, k, ctypes.c_void_p(value.ctypes.data), None))
        value = float(value[0])
      else:
        import torch
        dst = torch.empty(1, dtype=torch.float64, device=self._dev.observation.device)
        _lib.check(self._lib.bsb_read_info(self._handle.ptr, k, ctypes.c_void_p(dst.data_ptr()), None))
        value = float(dst.cpu()[0])
      result[name] = int(value) if name in _INT_INFO else value
    return result

  @property
  def raw_env(self):
    return self

  def close(self):
    self._handle.close()
