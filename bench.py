#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched bsuite engine on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA engine
    python bench.py ... --dump-outputs DIR                          # + the last timed step's outputs as DIR/*.npy
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's own step() loop on host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...           # one rank per GPU (weak scaling)

Workload (BASELINE.json configs[1]): deep_sea size=32 (bsuite_id deep_sea/11), 65 536 lanes per GPU, uniform
random actions.  One "step" = one lock-step `step()` call over the whole batch = ONE kernel launch that writes a
fresh dense [B, 32, 32] float32 observation tensor (268 MB) plus reward / discount / step_type.

  value   : env-steps/s with actions already resident in HBM; outputs go to a ring of 4 buffer sets (1.07 GB of
            observations > 126 MB L2, so every step's stores reach HBM).  WINDOWS (5) timed windows of EXACTLY K
            steps, each bracketed by barrier + synchronize; CUDA-event timed, max over ranks per window, the MEDIAN
            window is reported.  Every window contains one log point after step K/2: the device-side reduction
            of the Logging columns on the compute stream and, for N > 1, the all-gather of the per-rank block on a
            side stream (bsuite_b200.distributed.LogPoint); the window closes only after that gather has joined.
  e2e     : the same metric through the public host-buffer call (BatchedEnvironment.step_host): actions in pinned
            HOST memory, reward / discount / step_type delivered to pinned HOST memory every step, the host waits
            for each step's result before the next call (observations stay on the device for the agent, which is
            the engine's contract); median of 5 windows.
  roofline: algorithmic bytes per launch (SURVEY.md 8d: 4 120 B per lane-step) / mean launch duration, against
            MEASURED_PEAKS.json hbm_gbs; `frac` uses the launches only, `frac_from_ms_per_step` the whole window.
  configs : driver-visible legs for BASELINE configs #3 (catch B = 131 072), #4 (cartpole + mountain_car,
            B = 262 144) and #5 (23 experiments x 4 096 lanes, sharded over the ranks, with the return gather).
  cpu_baseline / --impl reference: the reference's own DeepSea.step loop, one process per usable host core
            (oracle/cpu_arm.py; kind "reference" when oracle/_ref holds the installed reference, else "port").
"""

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)
# the tree may be read-only where the benchmark runs: no bytecode caches in it, from here or from the processes it starts
sys.dont_write_bytecode = True
os.environ['PYTHONDONTWRITEBYTECODE'] = '1'

BSUITE_ID = 'deep_sea/11'          # size = 32, mapping_seed = 42
SIZE = 32
BATCH_PER_GPU = 65536
ALGO_BYTES_PER_LANE_STEP = 4 * SIZE * SIZE + 4 + 4 + 4 + 4 + 4 + 4   # obs + action + reward + discount + step_type + state rd/wr
RING = 4
WINDOWS = 5
METRIC = 'env-steps/sec'
FALLBACK_HBM_GBS = 6650.0
KERNEL_NAME = 'transition_kernel<DeepSea, Philox, no-noise, track>: persistent grid, TMA bulk stores of 8 tiles (32 KB)'


def _median(values):
  ordered = sorted(values)
  return ordered[len(ordered) // 2]


# ----------------------------------------------------------------------------- reference arm / cpu baseline
def run_cpu_arm(min_passes: int, seconds: float):
  from oracle import cpu_arm            # measurement infrastructure; never on the product path
  return cpu_arm.run(rounds=3, seconds=seconds, min_passes=max(8, int(min_passes)))


def reference_main(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return 0
  # >= 2 s per timed round whatever --steps says (override only for the CPU test-suite)
  seconds = float(os.environ.get('BSB_BENCH_BUDGET_S', '2.5'))
  r = run_cpu_arm(args.steps, seconds)
  what = ("the reference's own bsuite.environments.deep_sea.DeepSea.step loop (oracle/_ref, unmodified)"
          if r['kind'] == 'reference' else 'numpy restatement of bsuite DeepSea.step (oracle/bsuite_oracle.py)')
  sample = (f"{r['lanes']} lanes ({r['lanes_per_worker']} environment objects x {r['cores']} processes, one per usable "
            f"core) of the {BATCH_PER_GPU}-lane batch; one step = one pass over those lanes; 3 rounds of "
            f">= {seconds:g} s entered through a barrier, median round; {what}")
  ms_per_step = 1e3 * r['lanes'] / r['value']
  line = {
      'metric': METRIC, 'value': r['value'], 'unit': 'env-steps/s', 'n_gpus': args.gpus, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'impl': 'reference',
      'config': {'workload': f'deep_sea size={SIZE} ({BSUITE_ID}) uniform random actions, CPU sample of the '
                             f'{BATCH_PER_GPU}-lane batch', 'sample_lanes': r['lanes'], 'passes_timed': r['passes'],
                 'seconds_timed': r['seconds'], 'rounds': r['rounds'], 'host': r['host']},
      'cpu_baseline': {'value': r['value'], 'unit': 'env-steps/s', 'cores': r['cores'], 'kind': r['kind'],
                       'sample': sample, 'single_core': r['per_core'], 'rounds': r['rounds']},
      'e2e': {'value': r['value'], 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
  }
  print(json.dumps(line))
  return 0


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
  """Samples nvidia-smi clocks / throttle reasons; `stop(t0, t1)` keeps the samples taken under load."""
  QUERY = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
           'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
           'clocks_event_reasons.sw_power_cap')

  def __init__(self, index: int):
    self.index, self.proc, self.lines = index, None, []

  def start(self):
    try:
      self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits',
                                    '-lms', '50', '-i', str(self.index)], stdout=subprocess.PIPE,
                                   stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._pump, daemon=True)
      self.thread.start()
    except OSError:
      self.proc = None

  def _pump(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def wait_first_sample(self, timeout=5.0):
    end = time.time() + timeout
    while self.proc is not None and not self.lines and time.time() < end:
      time.sleep(0.02)

  def stop(self, t0=None, t1=None):
    import datetime
    if self.proc is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except subprocess.TimeoutExpired:
      self.proc.kill()
    sm, mx, reasons, power = [], [], set(), []
    names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
    for line in self.lines:
      parts = [p.strip() for p in line.split(',')]
      if len(parts) < 8:
        continue
      try:
        stamp = datetime.datetime.strptime(parts[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
        if t0 is not None and not (t0 <= stamp <= t1):
          continue
        sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
      except ValueError:
        continue
      for name, flag in zip(names, parts[4:8]):
        if flag.lower().startswith('active'):
          reasons.add(name)
    if not sm:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples'], 'raw_lines': len(self.lines)}
    sm.sort()
    return {'sm_mhz': sm[len(sm) // 2], 'sm_mhz_min': sm[0], 'sm_max_mhz': max(mx), 'reasons': sorted(reasons),
            'samples_under_load': len(sm), 'power_w_max': max(power)}


# ----------------------------------------------------------------------------- DRAM traffic of the headline kernel
def committed_traffic_bytes():
  """dram read + write bytes per launch from the newest committed `ncu --set full` extract under profiles/."""
  import csv
  import glob
  paths = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*_deep_sea_bulk_ncu_metrics.csv')))
  if not paths:
    return None, None
  scale = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
  total = 0.0
  with open(paths[-1]) as fh:
    for row in csv.reader(fh):
      if row and row[0] in ('dram__bytes_read.sum', 'dram__bytes_write.sum') and len(row) > 2:
        total += float(row[2].replace(',', '')) * scale.get(row[1], 1.0)
  return (total or None), os.path.relpath(paths[-1], ROOT)


def probe_traffic_main():
  """Child of `measure_traffic_live` (runs under ncu): a handful of single-step launches of the headline kernel."""
  import torch
  import bsuite_b200
  env = bsuite_b200.load_from_id(BSUITE_ID, batch=BATCH_PER_GPU, device='cuda', seed=0, track_episodes=True)
  ring = [env.make_buffers() for _ in range(RING)]
  actions = torch.randint(0, 2, (8, BATCH_PER_GPU), device='cuda', dtype=torch.int32)
  for t in range(8):
    env.step(actions[t], out=ring[t % RING])
  torch.cuda.synchronize()
  return 0


def measure_traffic_live(timeout_s: float = 150.0):
  """dram__bytes_read.sum + dram__bytes_write.sum per launch of the headline kernel, measured NOW with ncu (two
  metrics, one replay pass) on a short child run of the same kernel.  Returns (bytes or None, how)."""
  import csv
  ncu = shutil.which('ncu') or ('/usr/local/cuda/bin/ncu' if os.path.exists('/usr/local/cuda/bin/ncu') else None)
  if ncu is None:
    return None, 'ncu not on PATH'
  with tempfile.TemporaryDirectory(prefix='bsb_ncu_') as tmp:
    log = os.path.join(tmp, 'traffic.csv')
    cmd = [ncu, '--metrics', 'dram__bytes_read.sum,dram__bytes_write.sum', '--clock-control', 'none',
           '-k', 'regex:transition_kernel', '--launch-skip', '4', '--launch-count', '3', '--csv', '--log-file', log,
           sys.executable, os.path.abspath(__file__), '--probe-traffic']
    try:
      proc = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s)
    except (subprocess.TimeoutExpired, OSError) as exc:
      return None, f'ncu failed: {exc!r}'[:200]
    if proc.returncode != 0 or not os.path.exists(log):
      return None, ('ncu rc=%d: %s' % (proc.returncode, (proc.stderr or proc.stdout)[-160:])).replace('\n', ' ')
    scale = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
    per_launch = {}
    with open(log) as fh:
      rows = [r for r in csv.reader(fh) if r]
    header = next((r for r in rows if 'Metric Name' in r), None)
    if header is None:
      return None, 'ncu csv without header'
    i_id, i_name, i_unit, i_val = (header.index(k) for k in ('ID', 'Metric Name', 'Metric Unit', 'Metric Value'))
    for r in rows[rows.index(header) + 1:]:
      if len(r) > i_val and r[i_name].startswith('dram__bytes_'):
        per_launch[r[i_id]] = per_launch.get(r[i_id], 0.0) + float(r[i_val].replace(',', '')) * scale.get(r[i_unit], 1.0)
    if not per_launch:
      return None, 'ncu csv without dram metrics'
    return sum(per_launch.values()) / len(per_launch), f'ncu live, mean of {len(per_launch)} launches (this run)'


# ----------------------------------------------------------------------------- legs for BASELINE configs #3 / #4 / #5
def _parity_sampled(batch, torch, steps: int = 12, lanes_checked: int = 16):
  """GPU lanes vs the engine's explicit host path (the same transition functions compiled for the CPU, which the
  CPU test-suite pins bit-for-bit to reference-recorded traces): `steps` fused steps with on-device actions, the
  first / middle / last `lanes_checked` local lanes of every id.  Integer families must agree exactly, the float
  dynamics (cartpole*, mountain_car*) within 1e-6 (north_star's tolerance)."""
  import numpy as np
  import bsuite_b200
  got = batch.rollout(steps)
  torch.cuda.synchronize()
  for bsuite_id, env in batch.envs.items():
    ts = got[bsuite_id]
    actions = batch.last_buffers(bsuite_id).actions
    n = min(lanes_checked, env.batch)
    for first in sorted({0, max(0, env.batch // 2 - n // 2), env.batch - n}):
      host = bsuite_b200.load_from_id(bsuite_id, batch=n, device='cpu', seed=env.seed, lane_offset=env.lane_offset + first)
      want = host.rollout(steps, actions=actions[:, first:first + n].cpu())
      tol = 1e-6 if bsuite_id.startswith(('cartpole', 'mountain_car')) else 0.0
      for field in ('step_type', 'reward', 'discount', 'observation'):
        a = getattr(ts, field)[:, first:first + n].cpu().numpy().astype(np.float64)
        b = getattr(want, field).numpy().astype(np.float64)
        if not (np.abs(a - b) <= tol).all():
          host.close()
          return False
      host.close()
  return True


def family_leg(name, ids, lanes, rank, world, device, torch, dist, peak_gbs, rollout_T, iters, gather):
  """One driver-visible leg: `ids` x `lanes` lanes (sharded over the ranks), timed as single-step lock-steps (one
  launch per id and step, ids on concurrent streams) and as T-fused rollouts; optionally with the return gather
  (asynchronous log point) every iteration.  Returns a dict for rank 0."""
  from bsuite_b200 import suite
  obs_bytes = 0
  probe = suite.SweepBatch(ids, lanes=lanes, device=device, seed=0, rank=rank, world=world, ring=1)
  bytes_per_lockstep = probe.bytes_per_step()
  for env in probe.envs.values():
    numel = 1
    for d in env.obs_shape:
      numel *= d
    obs_bytes += env.batch * numel * 4
  parity = _parity_sampled(probe, torch)
  probe.close()
  del probe
  ring = max(2, min(16, int(300e6 // max(obs_bytes, 1)) + 1))      # single steps: outputs cycle through > L2
  batch = suite.SweepBatch(ids, lanes=lanes, device=device, seed=0, rank=rank, world=world, ring=ring)

  def timed(T, n, windows=3):
    times = []
    for _ in range(2):
      batch.rollout(T)
    if gather:
      batch.log_point_result(batch.issue_log_point())
    torch.cuda.synchronize()
    for _ in range(windows):
      if world > 1:
        dist.barrier()
      torch.cuda.synchronize()
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(n):
        batch.rollout(T)
        if gather:
          batch.issue_log_point()          # reduction kernels in order; the all-gather rides a side stream
      if gather:
        batch.join_log_points()
      e1.record()
      torch.cuda.synchronize()
      times.append(e0.elapsed_time(e1))
    t = torch.tensor(times, dtype=torch.float64, device=device)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return _median([float(x) for x in t]) * 1e-3 / (n * T)

  step_s = timed(1, iters)                 # eager: one launch per id and step through the Python face

  T = rollout_T
  while T > 1 and T * obs_bytes * 1 > 8e9:
    T //= 2
  batch.set_ring(1 if T * obs_bytes > 300e6 else ring)
  roll_s = timed(T, max(3, iters // T))
  # the same lock-step captured ONCE into a CUDA graph (every id's launch on its own branch) and replayed
  try:
    graphed = batch.capture(1, lock_steps=ring)
  except Exception as exc:  # pylint: disable=broad-except  (deterministic per configuration: every rank takes this branch)
    graphed, graph_error = None, repr(exc)[:200]
  def timed_graph(n, per_replay, windows=3):
    times = []
    for _ in range(3):
      graphed.replay()
    torch.cuda.synchronize()
    for _ in range(windows):
      if world > 1:
        dist.barrier()
      torch.cuda.synchronize()
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(n):
        graphed.replay()
        if gather:
          batch.issue_log_point()
      if gather:
        batch.join_log_points()
      e1.record()
      torch.cuda.synchronize()
      times.append(e0.elapsed_time(e1))
    t = torch.tensor(times, dtype=torch.float64, device=device)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return _median([float(x) for x in t]) * 1e-3 / (n * per_replay)
  graph_s = timed_graph(max(3, iters // ring), ring) if graphed is not None else float('nan')
  del graphed
  # the T-fused rollout of every id captured in ONE graph: at a few hundred lanes per id and GPU the eager rollout
  # is bound by the 23 launches the Python face makes per iteration, not by the GPU
  graph_roll_s = float('nan')
  try:
    graphed = batch.capture(T, lock_steps=1)
    graph_roll_s = timed_graph(max(3, iters // T), T)
    del graphed
  except Exception:  # pylint: disable=broad-except
    pass
  total_lanes = len(ids) * lanes
  result = {
      'ids': len(ids), 'lanes_per_id': lanes, 'global_lanes': total_lanes, 'lanes_per_gpu': total_lanes // world,
      'step_us': step_s * 1e6, 'step_value': total_lanes / step_s,
      'step_frac': bytes_per_lockstep / step_s / 1e9 / peak_gbs,
      'graph_step_us': graph_s * 1e6, 'graph_step_value': total_lanes / graph_s,
      'graph_step_frac': bytes_per_lockstep / graph_s / 1e9 / peak_gbs,
      'rollout_T': T, 'rollout_us': roll_s * 1e6, 'rollout_value': total_lanes / roll_s,
      'graph_rollout_us': graph_roll_s * 1e6, 'graph_rollout_value': total_lanes / graph_roll_s,
      'graph_rollout_frac': bytes_per_lockstep / graph_roll_s / 1e9 / peak_gbs,
      'frac': bytes_per_lockstep / roll_s / 1e9 / peak_gbs,
      'algorithmic_bytes_per_lockstep_per_gpu': bytes_per_lockstep, 'parity_sampled': bool(parity),
      'gather': bool(gather), 'ring': ring, 'unit': 'env-steps/s',
      'note': 'step: eager single-step launches (one per id, ids on concurrent streams); graph_step: the same lock-step '
              'replayed from one CUDA graph; rollout: T fused steps per launch with on-device actions (graph_rollout: '
              'all ids\' T-step launches in one graph); *_frac against '
              'hbm_gbs with SURVEY 8d algorithmic bytes; single-step outputs cycle through `ring` buffer sets (> L2), '
              'eagerly and under graph replay (`ring` lock-steps per graph)',
  }
  batch.close()
  del batch
  torch.cuda.empty_cache()
  return result


def config_legs(args, rank, world, device, torch, dist, peak_gbs):
  from bsuite_b200 import datasets
  from bsuite_b200 import suite
  mnist_dir = os.path.join(tempfile.gettempdir(), f'bsb_bench_mnist_{os.getpid()}')
  datasets.write_synthetic_mnist(mnist_dir, 4096, 16, 0)
  os.environ[datasets.ENV_VAR] = mnist_dir
  wanted = [w for w in args.legs.split(',') if w]
  legs = {}
  specs = {
      'catch_131072': (['catch/0'], 131072, 16, 200, False),
      'cartpole_mc_262144': (['cartpole/0', 'mountain_car/0'], 131072, 16, 200, False),
      'sweep_23x4096': (suite.one_per_experiment(), 4096, 64, 128, True),
  }
  for name, (ids, lanes, T, iters, gather) in specs.items():
    if name not in wanted:
      continue
    try:
      legs[name] = family_leg(name, ids, lanes, rank, world, device, torch, dist, peak_gbs, T, iters, gather)
    except Exception as exc:  # pylint: disable=broad-except
      if world > 1:
        raise                      # a collective is in flight on the other ranks: do not strand them
      legs[name] = {'error': repr(exc)[:300]}
  shutil.rmtree(mnist_dir, ignore_errors=True)
  return legs


# ----------------------------------------------------------------------------- outputs of the timed path
DUMP_OBSERVATION_LANES = 4096       # 4096 lanes x 32 x 32 float32 = 16.8 MB of the 268 MB observation tensor


def dump_outputs(directory, last, summary, torch):
  """Writes what the last timed step returned to its caller, as float32 / float64 .npy files: reward, discount and
  step_type of every lane, the observations of a fixed seeded sample of lanes (sorted lane ids drawn by
  RandomState(0)), and the log point's reduction of the Logging columns from the last window."""
  import numpy as np
  lanes = np.sort(np.random.RandomState(0).choice(BATCH_PER_GPU, DUMP_OBSERVATION_LANES, replace=False))
  index = torch.as_tensor(lanes, device=last.observation.device)
  arrays = {
      'observation_sample': last.observation.index_select(0, index).cpu().numpy(),
      'reward': last.reward.cpu().numpy(),
      'discount': last.discount.cpu().numpy(),
      'step_type': last.step_type.cpu().numpy().astype(np.float32),
  }
  if summary is not None:
    arrays['log_point'] = summary.cpu().numpy().astype(np.float64)
  os.makedirs(directory, exist_ok=True)
  for name, array in arrays.items():
    np.save(os.path.join(directory, name + '.npy'), array)


# ----------------------------------------------------------------------------- engine arm
def engine_main(args):
  import torch
  import torch.distributed as dist
  import bsuite_b200
  from bsuite_b200 import _lib
  from bsuite_b200 import distributed as bdist

  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  if not torch.cuda.is_available():
    raise RuntimeError('bench.py measures the CUDA engine; no CUDA device is visible (use --impl reference for the CPU arm)')
  torch.cuda.set_device(local_rank)
  device = torch.device('cuda', local_rank)
  if world > 1:
    dist.init_process_group('nccl', device_id=device)
  if args.gpus != world:
    raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}')

  # cpu_baseline first (rank 0, N = 1 only), in a clean subprocess so worker processes never inherit CUDA state
  cpu_baseline = None
  if rank == 0 and world == 1 and not args.skip_cpu_baseline:
    try:
      proc = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '8',
                             '--warmup', '3'], capture_output=True, text=True, timeout=240,
                            env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))
      cpu_baseline = json.loads(proc.stdout.strip().splitlines()[-1])['cpu_baseline']
    except Exception as exc:  # pylint: disable=broad-except
      cpu_baseline = {'value': None, 'unit': 'env-steps/s', 'cores': os.cpu_count(), 'kind': 'port',
                      'sample': 'failed: ' + repr(exc)[-300:]}

  B, K, W = BATCH_PER_GPU, args.steps, args.warmup
  lib = _lib.load()
  env = bsuite_b200.load_from_id(BSUITE_ID, batch=B, device=device, seed=0, lane_offset=rank * B,
                                 track_episodes=not args.no_track)
  ring = [env.make_buffers() for _ in range(RING)]
  gen = torch.Generator(device=device)
  gen.manual_seed(1234 + rank)
  actions = torch.randint(0, 2, (W + K, B), generator=gen, device=device, dtype=torch.int32)
  log_points = None if args.no_track else bdist.LogPoint(env, slots=2)

  # ---- value: device-resident actions -------------------------------------
  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
    sampler.wait_first_sample()

  def keep_busy(seconds):
    """Untimed steps of the same workload, so the clock samples bracket the timed region under load."""
    end = time.time() + seconds
    t = 0
    while time.time() < end:
      for _ in range(50):
        env.step(actions[t % (W + K)], out=ring[t % RING])
        t += 1
      torch.cuda.synchronize()

  load_t0 = time.time()
  for t in range(W):
    env.step(actions[t], out=ring[t % RING])
  if log_points is not None:
    for _ in range(2):                      # communicator set-up and first-use costs belong to the warm-up
      log_points.result(log_points.issue())
  # keep_busy runs a wall-clock-dependent number of steps: the timed windows start from the state the warm-up left,
  # so that the same arguments give the same inputs (and outputs) in every run
  warm_state = env.state_dict()
  keep_busy(0.5)
  torch.cuda.synchronize()
  env.load_state_dict(warm_state)
  torch.cuda.synchronize()

  mid = max(1, K // 2)
  windows, summary, launches = [], None, 0
  for _ in range(WINDOWS):
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()
    launches0 = lib.bsb_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    ticket = None
    ev[0].record()
    for t in range(K):
      env.step(actions[W + t], out=ring[t % RING])
      if t + 1 == mid and log_points is not None:
        ev[1].record()
        ticket = log_points.issue()         # reduction kernel in stream order; the all-gather rides the side stream
        ev[2].record()
    ev[3].record()
    if log_points is not None:
      summary = log_points.result(ticket)   # the window closes only after the gather has joined this stream
    ev[4].record()
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()
    launches = lib.bsb_launch_count() - launches0
    total_ms = ev[0].elapsed_time(ev[4])
    step_ms = total_ms if log_points is None else ev[0].elapsed_time(ev[1]) + ev[2].elapsed_time(ev[3])
    windows.append((total_ms, step_ms))
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, ring[(K - 1) % RING], summary, torch)
  keep_busy(0.4)
  clocks = sampler.stop(load_t0 + 0.15, time.time()) if rank == 0 else None
  times = torch.tensor(windows, dtype=torch.float64, device=device)
  if world > 1:
    dist.all_reduce(times, op=dist.ReduceOp.MAX)       # per window: the slowest rank
  windows = [(float(a), float(b)) for a, b in times]
  total_ms, step_ms = sorted(windows)[len(windows) // 2]
  value = world * B * K / (total_ms * 1e-3)

  # ---- e2e: host actions in, scalars out, every step ---------------------------
  Ke = max(100, min(K, 200))     # steps per e2e window: short windows time the cold first calls, not the loop
  host_actions = torch.randint(0, 2, (Ke, B), dtype=torch.int32).pin_memory()
  host_small = env.make_host_buffers(with_observation=False)

  host_rows = [host_actions[i] for i in range(Ke)]

  def e2e_loop(n, host, prelaunch):
    for t in range(n):
      env.step_host(host_rows[t % Ke], host, out=ring[t % RING], prelaunch=prelaunch)
    env.host_flush()

  def timed_e2e(n, host, reps, prelaunch=False):
    e2e_loop(min(n, 10), host, prelaunch)
    secs = []
    for _ in range(reps):
      if world > 1:
        dist.barrier()
      torch.cuda.synchronize()
      t0 = time.perf_counter()
      e2e_loop(n, host, prelaunch)
      torch.cuda.synchronize()
      secs.append(time.perf_counter() - t0)
    dt = torch.tensor(secs, dtype=torch.float64, device=device)
    if world > 1:
      dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    return world * B * n / _median([float(x) for x in dt]), [world * B * n / float(x) for x in dt]

  # headline: one step_host call per step (two-phase host step: the call returns when the scalars have landed and
  # launches the next kernel while this one still streams observations); `prelaunch_value` is the same loop with
  # the next step's kernel queued ahead and rung through the doorbell
  e2e_value, e2e_windows = timed_e2e(Ke, host_small, WINDOWS, prelaunch=False)
  e2e_prelaunch, _ = timed_e2e(Ke, host_small, 3, prelaunch=True)

  # The strict loop over TWO (or three, four) part-batches driven round-robin (rollouts.HostHalves / HostParts): each
  # part's next actions are submitted only after ITS previous results have landed, while the other parts' kernels
  # have the GPU.
  halves_value, halves_windows = None, None
  parts_values, parts_errors = {}, {}
  best_parts, best_parts_value, best_parts_windows = None, None, None
  if not args.skip_halves:
    from bsuite_b200 import rollouts
    for n_parts in args.e2e_parts:
      group = None
      if world > 1:
        dist.barrier()          # the ranks run the leg side by side (it holds no collective of its own)
      try:      # an optional leg must not take the line down; no collective runs while a part may have failed
        group = rollouts.HostParts(BSUITE_ID, B, device=device, seed=0, lane_offset=rank * B, parts=n_parts,
                                   track_episodes=not args.no_track)
        bounds = [0]
        for size in group.sizes:
          bounds.append(bounds[-1] + size)
        part_rows = [[r for r in host_actions[:, bounds[i]:bounds[i + 1]].contiguous().pin_memory()]
                     for i in range(n_parts)]
        group.reset()

        def parts_loop(n):
          for i in range(n_parts):
            group.submit(i, part_rows[i][0])
          for t in range(1, n):
            row = t % Ke
            for i in range(n_parts):
              group.collect(i); group.submit(i, part_rows[i][row])
          for i in range(n_parts):
            group.collect(i)

        parts_loop(30)
        secs = []
        for _ in range(WINDOWS):
          torch.cuda.synchronize()
          t0 = time.perf_counter()
          parts_loop(Ke)
          torch.cuda.synchronize()
          secs.append(time.perf_counter() - t0)
        local = secs
      except Exception as err:      # pylint: disable=broad-except
        parts_errors[str(n_parts)] = repr(err)[:200]
        local = None
      finally:
        if group is not None:
          try:
            group.close()
          except Exception:      # pylint: disable=broad-except
            pass
        group = None
        part_rows = None
        torch.cuda.empty_cache()
      # every rank joins the reduction, failed or not (a rank that failed reports no time: the leg is dropped)
      dt = torch.tensor(local if local is not None else [float('inf')] * WINDOWS, dtype=torch.float64, device=device)
      if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
      times = [float(x) for x in dt]
      if all(x != float('inf') for x in times):
        value_n = world * B * Ke / _median(times)
        windows_n = [world * B * Ke / x for x in times]
        parts_values[str(n_parts)] = value_n
        if n_parts == 2:
          halves_value, halves_windows = value_n, windows_n
        if best_parts_value is None or value_n > best_parts_value:
          best_parts, best_parts_value, best_parts_windows = n_parts, value_n, windows_n
  strict_value, strict_windows = e2e_value, e2e_windows
  e2e_mode = 'one batch: step_host per step'
  if best_parts_value is not None and best_parts_value > e2e_value:
    e2e_value, e2e_windows = best_parts_value, best_parts_windows
    e2e_mode = (f'{best_parts} part-batches driven round-robin (rollouts.HostParts'
                f'{" = HostHalves" if best_parts == 2 else ""}), each part a strict loop')

  # The same host-memory traffic WITHOUT a host synchronise per step (actions that do not depend on the previous
  # result, as in this random-action workload): env.step() given a pinned host action tensor and outputs whose
  # scalars live in pinned host memory -- the kernel reads / writes them in place; one synchronise at the end.
  mixed = [env.make_mixed_buffers() for _ in range(RING)]
  action_rows = host_rows
  for t in range(5):
    env.step(action_rows[t % Ke], out=mixed[t % RING])
  torch.cuda.synchronize()
  if world > 1:
    dist.barrier()
  p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  p0.record()
  for t in range(K):
    env.step(action_rows[t % Ke], out=mixed[t % RING])
  p1.record()
  torch.cuda.synchronize()
  pms = torch.tensor([p0.elapsed_time(p1)], dtype=torch.float64, device=device)
  if world > 1:
    dist.all_reduce(pms, op=dist.ReduceOp.MAX)
  e2e_pipelined = world * B * K / (float(pms[0]) * 1e-3)
  host_obs_value = None
  if not args.skip_host_obs:
    host_obs_value, _ = timed_e2e(5, env.make_host_buffers(with_observation=True), 1)
  del mixed

  # ---- the T-fused variant (SURVEY.md 8d asks for both): 16 steps per launch, on-device Philox actions -------
  fused = None
  if not args.skip_fused:
    Tf, reps = 16, 8
    fbuf = [env.make_buffers(Tf) for _ in range(2)]          # 2 x 4.3 GB of observations
    for i in range(2):
      env.rollout(Tf, out=fbuf[i % 2])
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(reps):
      env.rollout(Tf, out=fbuf[i % 2])
    f1.record()
    torch.cuda.synchronize()
    fms = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=device)
    if world > 1:
      dist.all_reduce(fms, op=dist.ReduceOp.MAX)
    per_step_s = float(fms[0]) * 1e-3 / (reps * Tf)
    fused = {'T': Tf, 'value': world * B / per_step_s, 'unit': 'env-steps/s', 'us_per_step': per_step_s * 1e6,
             'achieved_gbs': ALGO_BYTES_PER_LANE_STEP * B / per_step_s / 1e9,
             'note': 'bsb_rollout: 16 steps per launch, lane state in registers, actions sampled on device'}
    del fbuf

  # ---- the same single-step launches replayed from a CUDA graph (SURVEY.md 8d: "graph-captured") ------------
  graph_replay = None
  if not args.skip_graph and world == 1:      # a per-GPU figure; the multi-rank runs measure scaling, not this
    reps, g_ms, g_err = max(1, K // RING), 0.0, None
    try:     # an optional leg must not take the line down (and holds no collective, so no rank can strand another)
      genv = bsuite_b200.load_from_id(BSUITE_ID, batch=B, device=device, seed=0, lane_offset=rank * B,
                                      track_episodes=not args.no_track)
      graphed = genv.capture(RING)          # RING launches per graph, each writing its own buffer set (> L2 in total)
      graphed.actions.copy_(actions[:RING])
      for _ in range(3):
        graphed.replay()
      torch.cuda.synchronize()
      g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      g0.record()
      for _ in range(reps):
        graphed.replay()
      g1.record()
      torch.cuda.synchronize()
      g_ms = g0.elapsed_time(g1)
      del graphed
      genv.close()
    except Exception as exc:  # pylint: disable=broad-except
      g_err = repr(exc)[:300]
    if g_err is not None:
      graph_replay = {'value': None, 'error': g_err}
    else:
      per_step_s = g_ms * 1e-3 / (reps * RING)
      graph_replay = {'value': world * B / per_step_s, 'unit': 'env-steps/s', 'us_per_step': per_step_s * 1e6,
                      'steps_per_graph': RING, 'replays': reps,
                      'note': 'cudaGraphLaunch of RING captured single-step launches; step counter and chunk scheduler '
                              'live in device memory (graph-safe mode); programmatic edges between the captured launches'}

  env.close()
  del ring, env
  torch.cuda.empty_cache()

  peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(peaks_path):
    peak, peak_src = float(json.load(open(peaks_path))['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs (measured copy)'
  else:
    peak, peak_src = FALLBACK_HBM_GBS, 'fallback 6.65 TB/s (B200_PROFILING.md)'

  # ---- BASELINE configs #3 / #4 / #5 (every rank takes part: the sweep leg shards its lanes over the ranks) ----
  configs = None if args.skip_configs else config_legs(args, rank, world, device, torch, dist, peak)

  if rank == 0:
    launch_s = (step_ms * 1e-3) / K
    achieved = ALGO_BYTES_PER_LANE_STEP * B / launch_s / 1e9
    achieved_window = ALGO_BYTES_PER_LANE_STEP * B / (total_ms * 1e-3 / K) / 1e9
    traffic, traffic_src, traffic_stale = None, None, None
    if world == 1 and not args.skip_traffic:
      traffic, traffic_src = measure_traffic_live()
      traffic_stale = False
    if traffic is None:
      why = traffic_src
      traffic, traffic_src = committed_traffic_bytes()
      traffic_stale = True
      if why:
        traffic_src = f'{traffic_src} (committed capture; live probe: {why})'
    line = {
        'metric': METRIC, 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': total_ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'u32 lane state, f64 reward, f32 observation', 'data': 'synthetic',
        'config': {'workload': f'deep_sea size={SIZE} batch={B} per GPU ({BSUITE_ID}), uniform random actions',
                   'bsuite_id': BSUITE_ID, 'batch_per_gpu': B, 'global_batch': world * B,
                   'parallelism': f'lanes sharded over {world} GPU(s), no data-path collective; one log point per '
                                  'window: reduction kernel on the compute stream + all-gather of the per-rank '
                                  'block on a side stream, joined before the window closes',
                   'l2_policy': f'outputs cycle through {RING} buffer sets ({RING * B * SIZE * SIZE * 4 / 1e9:.2f} GB '
                                'of observations > 126 MB L2)',
                   'launch': 'value / roofline: one transition_kernel launch per step (T = 1, programmatic dependent launch); the T-fused variant is reported under fused_rollout',
                   'windows': f'median of {WINDOWS} windows of {K} steps, each bracketed by barrier + synchronize, max over ranks per window',
                   'track_episodes': not args.no_track},
        'windows_ms': [w[0] for w in windows],
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'frac_from_ms_per_step': achieved_window / peak,
                     'traffic': traffic, 'traffic_source': traffic_src, 'traffic_stale': traffic_stale,
                     'peak_source': peak_src, 'algorithmic_bytes_per_launch': ALGO_BYTES_PER_LANE_STEP * B,
                     'launch_us': launch_s * 1e6, 'kernel': KERNEL_NAME},
        'cpu_baseline': cpu_baseline,
        'e2e': {'value': e2e_value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 4 * B, 'd2h_bytes_per_step': 12 * B,
                'steps': Ke, 'windows': e2e_windows, 'mode': e2e_mode,
                'one_batch_value': strict_value, 'one_batch_windows': strict_windows,
                'two_halves_value': halves_value, 'two_halves_windows': halves_windows,
                'parts_values': parts_values, 'parts_errors': parts_errors or None,
                'prelaunch_value': e2e_prelaunch,
                'host_obs_value': host_obs_value, 'pipelined_value': e2e_pipelined,
                'host_obs_d2h_bytes_per_step': 4 * B * SIZE * SIZE + 12 * B,
                'note': 'value = the fastest of one_batch_value and parts_values (mode says which; parts_values[\"2\"] = two_halves_value); all are the strict '
                        'host loop -- the next actions of a lane are submitted only after that lane\'s previous reward / '
                        'discount / step_type have landed in host memory -- with the same bytes over PCIe per step. '
                        'two_halves_value: the lanes split over two handles (lane keys continue across the split) that '
                        'the host drives alternately with BSB_HOST_NO_WAIT / bsb_host_wait, so one half\'s PCIe round '
                        'trip and decision hide behind the other half\'s kernel. one_batch_value: '
                        'BatchedEnvironment.step_host -> bsb_step_host every step, the call pattern of a host-side policy: '
                        'actions come from pinned host memory (brought over by the DMA engine on a side stream while the '
                        'previous kernel still streams observations) and reward / discount / step_type land in pinned '
                        'host memory; deep_sea runs the step in two phases -- transitions of all lanes into a device '
                        'staging block, which copier blocks ship to the host while the others stream the observations -- '
                        'and the call returns when the scalars have landed (completion word in pinned memory, no stream '
                        'synchronise); observations stay on the device (the API contract; the caller\'s stream is fenced '
                        'behind them). prelaunch_value: the same loop with the next step\'s kernel queued ahead and '
                        'waiting on a doorbell in pinned memory. host_obs_value also copies the observations to pinned '
                        'host memory every step. pipelined_value: the same per-step host traffic through env.step() with '
                        'pinned actions and pinned scalar outputs, launches queued, one synchronise at the end.'},
        'gpu_launches': int(launches),
        'fused_rollout': fused,
        'graph_replay': graph_replay,
        'configs': configs,
        'clocks': clocks,
        'log_point': None if summary is None else [float(x) for x in summary.reshape(-1).cpu()[:5]],
    }
    print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()
  return 0


def main():
  parser = argparse.ArgumentParser()
  parser.add_argument('--gpus', type=int, default=1)
  parser.add_argument('--skip-halves', action='store_true', help='skip the part-batches e2e legs')
  parser.add_argument('--e2e-parts', type=int, nargs='*', default=[2, 3, 4],
                      help='part counts of the part-batches e2e legs (rollouts.HostParts)')
  parser.add_argument('--steps', type=int, default=400, help='timed steps in each of the 5 windows of the headline value')
  parser.add_argument('--warmup', type=int, default=20)
  parser.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  parser.add_argument('--skip-cpu-baseline', action='store_true')
  parser.add_argument('--skip-host-obs', action='store_true')
  parser.add_argument('--no-track', action='store_true', help='disable the per-lane Logging accumulators')
  parser.add_argument('--skip-fused', action='store_true', help='skip the T-fused rollout variant')
  parser.add_argument('--skip-graph', action='store_true', help='skip the CUDA-graph replay variant')
  parser.add_argument('--skip-configs', action='store_true', help='skip the legs for BASELINE configs #3 / #4 / #5')
  parser.add_argument('--skip-traffic', action='store_true', help='do not re-measure DRAM traffic with ncu')
  parser.add_argument('--legs', default='catch_131072,cartpole_mc_262144,sweep_23x4096')
  parser.add_argument('--dump-outputs', metavar='DIR', default=None,
                      help='write the outputs of the last timed step to DIR/<name>.npy (rank 0)')
  parser.add_argument('--probe-traffic', action='store_true', help=argparse.SUPPRESS)
  args = parser.parse_args()
  if args.steps < 1:
    parser.error('--steps must be at least 1')
  if args.warmup < 3:
    args.warmup = 3
  if args.probe_traffic:
    return probe_traffic_main()
  if args.impl == 'reference':
    return reference_main(args)
  return engine_main(args)


if __name__ == '__main__':
  sys.exit(main())
