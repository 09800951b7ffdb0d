"""What score summaries (`track_scores=True`) cost and save against the row store (`record_rows=True`), on one GPU.

    python tools/bench_score_summary.py [--out FILE] [--rollout-lanes 4096] [--scorer-lanes 4096 16384]
                                        [--summary-only-lanes 65536] [--calls 200]

Prints one JSON line per measurement:
  * kind=state_bytes: device bytes per lane (bsb_state_bytes, batch 2 minus batch 1) summed over the 468 ids, for
    plain (track_episodes), record_rows, track_scores and both -- the row store and the summary are snapshot state.
  * kind=rollout: a full-sweep `SweepBatch.rollout` (468 ids, `--rollout-lanes` lanes each, `--steps` fused steps
    per call, on-device actions) for the three keywords none / record_rows / track_scores, built side by side and
    timed alternately in rounds with CUDA events from the first step on (rows fall due most often early in a run);
    ms per call, median and spread over the rounds.
  * kind=scorer: `Scorer.run` over all 468 ids with every lane finished (the synthetic rows of
    tools/bench_scoring.py: full, ascending, in the engine's layout), from the rows and from their summaries
    folded on the host (`scoring.summarize`), microseconds per call over `--calls` back-to-back calls; summaries
    alone at `--summary-only-lanes`, where the row store would not be worth building.
The card's name and power limit are read in the same call.
"""

import argparse
import json
import os
import statistics
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import torch  # noqa: E402

import bsuite_b200  # noqa: E402
from bsuite_b200 import _lib, datasets, recording, scoring, sweep  # noqa: E402
from bsuite_b200.suite import SweepBatch  # noqa: E402
from bench_scoring import card, info_columns  # noqa: E402

MODES = {'none': {}, 'record_rows': dict(record_rows=True), 'track_scores': dict(track_scores=True),
         'both': dict(record_rows=True, track_scores=True)}


def state_bytes_per_lane():
  import ctypes
  lib = _lib.load()
  totals = {}
  for mode, kw in MODES.items():
    total = 0
    for bsuite_id in sweep.SWEEP:
      sizes = []
      for batch in (1, 2):
        env = bsuite_b200.load_from_id(bsuite_id, batch=batch, device='cpu', seed=0, track_episodes=True, **kw)
        n = ctypes.c_int64()
        _lib.check(lib.bsb_state_bytes(env._handle.ptr, ctypes.byref(n)))
        sizes.append(n.value)
        env.close()
      total += sizes[1] - sizes[0]
    totals[mode] = total
  return dict(kind='state_bytes', ids=len(sweep.SWEEP), bytes_per_lane=totals,
              row_store_over_summary=round((totals['record_rows'] - totals['none']) /
                                           (totals['track_scores'] - totals['none']), 2))


def rollouts(lanes, steps, calls, rounds):
  batches = {mode: SweepBatch(sweep.SWEEP, lanes=lanes, device='cuda', seed=0, **MODES[mode])
             for mode in ('none', 'record_rows', 'track_scores')}
  times = {mode: [] for mode in batches}
  for _ in range(rounds):
    for mode, batch in batches.items():
      start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      start.record()
      for _ in range(calls):
        batch.rollout(steps, action_seed=1)
      stop.record()
      torch.cuda.synchronize()
      times[mode].append(start.elapsed_time(stop) / calls)
  out = dict(kind='rollout', ids=len(sweep.SWEEP), lanes=lanes, steps_per_call=steps, calls_per_round=calls,
             rounds=rounds, steps_done=rounds * calls * steps,
             ms_per_call={m: round(statistics.median(t), 3) for m, t in times.items()},
             ms_per_call_min_max={m: [round(min(t), 3), round(max(t), 3)] for m, t in times.items()})
  for batch in batches.values():
    batch.close()
  return out


def table_for(bsuite_id, lanes, device, seed):
  """One id's rows as tools/bench_scoring.py builds them: full, cumulative values ascending, engine layout."""
  gen = torch.Generator(device=device).manual_seed(seed)
  name = bsuite_id.split('/')[0]
  columns = list(_lib.EPISODE_STAT_FIELDS) + list(info_columns(name))
  schedule = torch.tensor(recording.log_schedule(sweep.EPISODES[bsuite_id]), dtype=torch.float64, device=device)
  inc = torch.rand((len(schedule), len(columns), lanes), generator=gen, device=device, dtype=torch.float64)
  rows = torch.cumsum(inc, dim=0) * schedule[:, None, None]
  rows[:, 1, :] = schedule[:, None]
  return dict(rows=rows.contiguous(), counts=torch.full((lanes,), len(schedule), dtype=torch.int32, device=device),
              columns=columns)


def time_scorer(scorer, calls):
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
  return (start.elapsed_time(stop) * 1e3 / calls, (lib.bsb_launch_count() - launches0) / calls,
          int(out['finished'].sum().item()), out)


def scorers(lanes, calls, with_rows):
  device = torch.device('cuda', 0)
  summaries, tables = {}, {}
  for k, bsuite_id in enumerate(sweep.SWEEP):
    table = table_for(bsuite_id, lanes, device if with_rows else torch.device('cpu'), k)
    host = {key: (v.cpu() if torch.is_tensor(v) else v) for key, v in table.items()}
    summaries[bsuite_id] = {key: (v.to(device) if torch.is_tensor(v) else v)
                            for key, v in scoring.summarize(bsuite_id, host).items()}
    if with_rows:
      tables[bsuite_id] = table
  result = dict(kind='scorer', ids=len(sweep.SWEEP), lanes=lanes, calls=calls)
  scorer = scoring.Scorer.from_summaries(summaries, device=device)
  us, launches, finished, out = time_scorer(scorer, calls)
  result.update(summary_us_per_call=round(us, 2), launches_per_call=launches, finished_lanes_scored=finished,
                summary_bytes=sum(6 * 8 * lanes + 4 * lanes for _ in summaries))
  if with_rows:
    rows_scorer = scoring.Scorer.from_rows(tables, device=device)
    rows_us, _, _, rows_out = time_scorer(rows_scorer, calls)
    result.update(rows_us_per_call=round(rows_us, 2),
                  row_store_bytes=sum(t['rows'].numel() * 8 + t['counts'].numel() * 4 for t in tables.values()),
                  same_bits=all(torch.equal(out[k].double().nan_to_num(nan=-7.0), rows_out[k].double().nan_to_num(nan=-7.0))
                                for k in out))
    rows_scorer.close()
  scorer.close()
  return result


def main():
  parser = argparse.ArgumentParser()
  parser.add_argument('--rollout-lanes', type=int, default=4096)
  parser.add_argument('--steps', type=int, default=10)
  parser.add_argument('--calls', type=int, default=200)
  parser.add_argument('--rollout-calls', type=int, default=10)
  parser.add_argument('--rounds', type=int, default=6)
  parser.add_argument('--scorer-lanes', type=int, nargs='+', default=[4096, 16384])
  parser.add_argument('--summary-only-lanes', type=int, nargs='*', default=[65536])
  parser.add_argument('--out', default=None)
  args = parser.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('bench_score_summary.py measures on a CUDA device: none found')
  info = card()
  lines = []

  def emit(result):
    lines.append(json.dumps(dict(result, card=info['name'], power_limit=info['power_limit'])))
    print(lines[-1], flush=True)

  with tempfile.TemporaryDirectory() as mnist_dir:
    datasets.write_synthetic_mnist(mnist_dir, 4096, 16, 0)
    os.environ[datasets.ENV_VAR] = mnist_dir
    emit(state_bytes_per_lane())
    emit(rollouts(args.rollout_lanes, args.steps, args.rollout_calls, args.rounds))
    torch.cuda.empty_cache()
  for lanes in args.scorer_lanes:
    emit(scorers(lanes, args.calls, with_rows=True))
    torch.cuda.empty_cache()
  for lanes in args.summary_only_lanes:
    emit(scorers(lanes, args.calls, with_rows=False))
    torch.cuda.empty_cache()
  if args.out:
    with open(args.out, 'w') as fh:
      fh.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
  main()
