"""
Exact value iteration by incremental pruning (`IncrementalPruning_Solver`) on the small golden models, against `GapSolver` at equal wall time.

Per model: one solve from the default start (the evaluated blind controller) with a TIME_LIMIT-second limit, stopping early at shift <=
1e-6.  Recorded: epochs; per epoch |V'|, the largest cross sum of a fold, the shift and the elapsed time; over the solve, rows dropped
pointwise / by LP / left undecided, LP counts and the phase seconds (device-synchronised wall clock); the fold and union sizes of the last
epoch; the shift reached and why the solve stopped; the
wall time to shift <= 1e-3 and <= 1e-6 where reached; V(b0) and V(b0) + shift, and the certified (lower, upper) at b0 of a `GapSolver`
run (K = 8 trials, max depth 200, target gap 1e-6) given the same wall time.
    python tools/incremental_pruning.py [--out PATH] [model ...]     (default PATH: profiles/incremental_pruning_b200.json)
Writes one JSON document with the GPU name and power limit read in the same run, and prints one summary line per model.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from pomdp_pbvi_exploration_b200 import GapSolver, IncrementalPruning_Solver  # noqa: E402
from bound_gap import golden_model  # noqa: E402

MODELS = ['tiger', 'hanks', 'network', 'grid4x4', 'grid4x4_noloop', 'cheese', 'grid4x3']
TIME_LIMIT = 20.0


def run(tag, model, gamma) -> dict:
    IncrementalPruning_Solver(gamma).solve(model, horizon=2)                      # warm-up: module loads, allocations
    torch.cuda.synchronize()
    V, hist = IncrementalPruning_Solver(gamma).solve(model, horizon=100000, target=1e-6, time_limit=TIME_LIMIT)
    b0 = model.start_belief_device[None, :]
    v0 = float(model.device.max_values(b0, V.alpha_vector_array)[0][0])
    eps = hist.epochs

    def total(key):
        return sum(ep[key] for ep in eps)

    # per epoch only what shows the trend (4 numbers); the rest as totals over the solve, so the document stays small
    per_epoch = dict(rows=[ep['rows'] for ep in eps], largest_fold=[max(ep['fold_candidates']) for ep in eps],
                     shift=[None if ep['shift'] is None else float(f"{ep['shift']:.3g}") for ep in eps],
                     elapsed=[float(f"{ep['elapsed']:.3g}") for ep in eps])
    totals = dict(dropped_pointwise=total('dropped_pointwise'), dropped_lp=total('dropped_lp'), undecided=total('undecided'),
                  lp_rows=sum(ep['prune_lp_stats'].get('lp_rows', 0) for ep in eps), lps=sum(ep['prune_lp_stats'].get('lps', 0) for ep in eps),
                  residual_lps=sum(ep['residual_stats']['lps'] for ep in eps),
                  residual_budget_rows=sum(ep['residual_stats']['budget_rows'] for ep in eps),
                  phase_seconds={k: sum(ep['seconds'][k] for ep in eps) for k in ('project', 'cross_sum', 'pointwise', 'lp', 'residual')})

    def first_time(level):
        hit = [ep['elapsed'] for ep in hist.epochs if ep['shift'] is not None and ep['shift'] <= level]
        return hit[0] if hit else None

    t0 = time.perf_counter()
    _, _, gh = GapSolver(gamma, 1e-6, trials=8, max_depth=200, seed=0).solve(model, max_rounds=10 ** 6, time_limit=hist.seconds)
    gap_wall = time.perf_counter() - t0
    return dict(model=tag, S=model.state_count, A=model.action_count, O=model.observation_count, R=model.reachable_state_count, gamma=gamma,
                time_limit=TIME_LIMIT, stopped=hist.stopped, epochs_run=len(hist.epochs), rows=len(V), shift=hist.shift, e=hist.e,
                seconds=hist.seconds, time_to_shift_1e_3=first_time(1e-3), time_to_shift_1e_6=first_time(1e-6), v_b0=v0,
                v_b0_plus_shift=None if hist.shift is None else v0 + hist.shift,
                gap_solver=dict(lower_b0=gh.lower, upper_b0=gh.upper, gap=gh.upper - gh.lower, wall_s=gap_wall, rounds=len(gh.rounds)),
                last_epoch=None if not eps else dict(fold_candidates=eps[-1]['fold_candidates'], union_candidates=eps[-1]['union_candidates'],
                                                     max_u=eps[-1]['max_u']),
                totals=totals, per_epoch=per_epoch)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'incremental_pruning_b200.json'))
    ap.add_argument('models', nargs='*', default=MODELS)
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), time_limit=TIME_LIMIT, models=[])
    t_start = time.perf_counter()
    for tag in args.models:
        model, gamma = golden_model(tag)
        res['models'].append(run(tag, model, gamma))
        m = res['models'][-1]
        print(json.dumps({k: v for k, v in m.items() if k != 'per_epoch'}), flush=True)
    res['total_seconds'] = time.perf_counter() - t_start
    text = json.dumps(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text + '\n')


if __name__ == '__main__':
    main()
