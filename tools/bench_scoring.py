"""Times `scoring.Scorer.run` over the rows of a whole sweep (all 468 bsuite_ids) on one GPU.

    python tools/bench_scoring.py [--lanes 4096 16384] [--calls 200] [--out FILE]

For each lane count: every id gets a row store in the engine's layout ([n_points][5 + info columns][B] float64,
counts int32 [B]), written once beforehand with full, ascending synthetic rows (every lane has reached
NUM_EPISODES, the case that reads the most); then CUDA events time `calls` back-to-back `run()` calls.  Reported:
microseconds per call, launches per call (bsb_launch_count delta), the bytes the rules must read (from the layout:
counts, the last row's episode and value column; all rows of best_episode for cartpole / cartpole_swingup and of
episode + total_bad_episodes for deep_sea; the last two rows for mnist) and that over 7.7 TB/s.  For contrast,
in the same run: the device-to-host copy of all rows, and one lane's CSV files written from them
(`recording.write_lane_csvs`) -- what scoring through the reference's pandas analysis starts with.
The card's name and power limit are read in the same call.  Prints one JSON line per lane count.
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bsuite_b200 import _lib, recording, scoring, sweep  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
INFO_COLUMNS = {                     # bsuite_info() keys per experiment family (the engine's column order)
    'bandit': ('total_regret',), 'catch': ('total_regret',), 'mnist': ('total_regret',),
    'umbrella': ('total_regret',), 'cartpole_swingup': ('raw_return', 'total_upright', 'best_episode'),
    'cartpole': ('raw_return', 'best_episode'), 'mountain_car': ('raw_return',),
    'deep_sea': ('total_bad_episodes', 'denoised_return'), 'memory': ('total_perfect', 'total_regret'),
    'discounting_chain': (),
}


def info_columns(experiment):
  for prefix in ('cartpole_swingup', 'cartpole', 'mountain_car', 'deep_sea', 'memory', 'umbrella', 'bandit', 'catch',
                 'mnist', 'discounting_chain'):
    if experiment.startswith(prefix):
      return INFO_COLUMNS[prefix]
  raise KeyError(experiment)


def card():
  props = torch.cuda.get_device_properties(0)
  try:
    power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
  except (OSError, subprocess.TimeoutExpired):
    power = 'unknown'
  return dict(name=props.name, power_limit=power, sms=props.multi_processor_count)


def make_tables(lanes, device):
  """bsuite_id -> dict(rows, counts, columns) on `device`: full rows, cumulative values ascending."""
  gen = torch.Generator(device=device).manual_seed(0)
  tables = {}
  for bsuite_id in sweep.SWEEP:
    name = bsuite_id.split('/')[0]
    columns = list(_lib.EPISODE_STAT_FIELDS) + list(info_columns(name))
    schedule = torch.tensor(recording.log_schedule(sweep.EPISODES[bsuite_id]), dtype=torch.float64, device=device)
    P, C = len(schedule), len(columns)
    inc = torch.rand((P, C, lanes), generator=gen, device=device, dtype=torch.float64)
    rows = torch.cumsum(inc, dim=0) * schedule[:, None, None]
    rows[:, 1, :] = schedule[:, None]
    tables[bsuite_id] = dict(rows=rows.contiguous(), counts=torch.full((lanes,), P, dtype=torch.int32, device=device),
                             columns=columns)
  return tables


def model_bytes(tables, lanes):
  total = 0
  for bsuite_id, t in tables.items():
    name = bsuite_id.split('/')[0]
    P = t['rows'].shape[0]
    per_lane = 4 + 2 * 8                                   # counts + last row's episode and value
    if name in scoring.NEEDS_BEST:
      per_lane += P * 8                                    # best_episode of every row
    if name.startswith('deep_sea'):
      per_lane = 4 + P * 2 * 8                             # episode + total_bad_episodes of every row (upper bound)
    if name.startswith('mnist'):
      per_lane = 4 + 2 * 2 * 8                             # the last two rows
    total += per_lane * lanes
  return total


def bench(lanes, calls):
  device = torch.device('cuda', 0)
  tables = make_tables(lanes, device)
  scorer = scoring.Scorer.from_rows(tables, device=device)
  out = scorer.empty_outputs()
  for _ in range(5):
    scorer.run(out)
  torch.cuda.synchronize()
  lib = _lib.load()
  launches0 = lib.bsb_launch_count()
  start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  start.record()
  for _ in range(calls):
    scorer.run(out)
  stop.record()
  torch.cuda.synchronize()
  launches = (lib.bsb_launch_count() - launches0) / calls
  us = start.elapsed_time(stop) * 1e3 / calls
  nbytes = model_bytes(tables, lanes)
  row_bytes = sum(t['rows'].numel() * 8 + t['counts'].numel() * 4 for t in tables.values())

  # contrast: every row to the host, then one lane's CSV files
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  host = {k: dict(rows=t['rows'].cpu(), counts=t['counts'].cpu(), columns=t['columns']) for k, t in tables.items()}
  d2h_s = time.perf_counter() - t0

  class _Recorded:                                         # what write_lane_csvs reads from an environment
    def __init__(self, table):
      self.table, self.batch, self.lane_offset = table, lanes, 0

    def logged_rows(self):
      return dict(columns=tuple(self.table['columns']), rows=self.table['rows'], counts=self.table['counts'])

  with tempfile.TemporaryDirectory() as tmp:
    t0 = time.perf_counter()
    for bsuite_id, table in host.items():
      recording.write_lane_csvs(_Recorded(table), bsuite_id, tmp, lanes=[0])
    csv_s = time.perf_counter() - t0
  scorer.close()
  return dict(lanes=lanes, ids=len(tables), calls=calls, us_per_call=round(us, 2), launches_per_call=launches,
              model_bytes_read=nbytes, model_bandwidth_tb_s=round(nbytes / (us * 1e-6) / 1e12, 3),
              share_of_7p7_tb_s=round(nbytes / (us * 1e-6) / HBM_BYTES_PER_S, 4),
              row_store_bytes=row_bytes, d2h_all_rows_s=round(d2h_s, 4), one_lane_csvs_s=round(csv_s, 4),
              finished_lanes_scored=int(out['finished'].sum().item()))


def main():
  parser = argparse.ArgumentParser()
  parser.add_argument('--lanes', type=int, nargs='+', default=[4096, 16384])
  parser.add_argument('--calls', type=int, default=200)
  parser.add_argument('--out', default=None)
  args = parser.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('bench_scoring.py measures the CUDA scorer: no CUDA device')
  info = card()
  lines = []
  for lanes in args.lanes:
    result = dict(bench(lanes, args.calls), card=info['name'], power_limit=info['power_limit'])
    lines.append(json.dumps(result))
    print(lines[-1], flush=True)
    torch.cuda.empty_cache()
  if args.out:
    with open(args.out, 'w') as fh:
      fh.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
  main()
