"""
Gap-driven solves with and without pruning of dominated nodes and pairs (`GapSolver(prune_growth=...)`):
  per model, the settings of tools/gap_solve.py (K = 16 trials, max depth 100, LONG_S seconds, from the blind controller and the FIB
  bound), once with prune_growth = None and once with GROWTH.  Recorded per run: the certified (lower, upper) at b0, the rounds (bounds,
  nodes and pairs after the prune, pruned counts, phase seconds including the prune), every prune as (nodes, pairs) before and after,
  then on the bounds the run ended with:
    the cost of one `gap_trial_step` level at K = 1 and K = 16 (trial beliefs of a random walk, as tools/gap_solve.py takes them);
    the cost of `pbvi_dominating_row` on the final controller rows and of `pbvi_sawtooth_witness` on the final store.
  CUDA events, median of SAMPLES samples after one warm-up call.
Models: hallway and tiger-grid (golden fixtures, gamma 0.95), the olfactory wrap model (22021 states, gamma 0.99).
    python tools/gap_prune.py [--out PATH] [model ...]        (default PATH: profiles/gap_prune_b200.json)
Writes one JSON document, with the GPU name and power limit read in the same run, and prints it.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pomdp_pbvi_exploration_b200 import GapSolver  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402
from bound_gap import golden_model, synced  # noqa: E402
from gap_solve import LONG_S, SETTINGS  # noqa: E402

SAMPLES = 11
GROWTH = 1.1


def timed(fn) -> dict:
    fn()
    samples = []
    for _ in range(SAMPLES):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        samples.append(e0.elapsed_time(e1))
    return dict(median_ms=float(np.median(samples)), samples_ms=samples)


def final_costs(model, ub, X, K, theta) -> dict:
    dev = model.device
    rng = np.random.default_rng(0)
    b0 = torch.as_tensor(model.start_probabilities, device='cuda', dtype=torch.float64)
    walk = dev.perseus_walk(b0, rng.integers(0, model.action_count, 4 * K).astype(np.int32), rng.random(4 * K))
    lists = ub._lists()
    out = dict(lower_rows=int(X.shape[0]), stored_pairs=len(ub), level={})
    for k in (1, K):
        b = walk[-k:].contiguous()
        out['level'][f'K={k}'] = timed(lambda: dev.gap_trial_step(b, X, ub._F, ub.gamma, ub.corner_values, *lists, theta))
    out['dominating_row'] = timed(lambda: dev.dominating_row(X))
    out['sawtooth_witness'] = timed(lambda: dev.sawtooth_witness(ub.corner_values, *lists)) if len(ub) else None
    return out


def run(name, model, gamma):
    target, K, depth, rounds = SETTINGS[name]
    out = dict(model=name, S=model.state_count, A=model.action_count, O=model.observation_count, gamma=gamma, target_gap=target, trials=K,
               max_depth=depth, max_rounds=rounds, time_limit_s=LONG_S, runs={})
    GapSolver(gamma, target, trials=2, max_depth=3, seed=0, prune_growth=GROWTH).solve(model, max_rounds=2)     # warm-up
    for growth in (None, GROWTH):
        t0 = synced()
        pg, ub, hist = GapSolver(gamma, target, trials=K, max_depth=depth, seed=0, prune_growth=growth).solve(
            model, max_rounds=rounds, time_limit=LONG_S)
        wall = synced() - t0
        prunes = [dict(round=r['round'], nodes_before=r['nodes'] + r['pruned_nodes'], nodes_after=r['nodes'],
                       pairs_before=r['stored_pairs'] + r['pruned_pairs'], pairs_after=r['stored_pairs'], seconds=r['phase_seconds']['prune'])
                  for r in hist.rounds if r.get('pruned_nodes') or r.get('pruned_pairs')]
        phase = {k: float(sum(r['phase_seconds'].get(k, 0.0) for r in hist.rounds)) for k in hist.rounds[0]['phase_seconds']}
        out['runs']['none' if growth is None else str(growth)] = dict(
            prune_growth=growth, wall_s=wall, reached=hist.reached, certified_lower_b0=hist.lower, certified_upper_b0=hist.upper,
            gap=hist.gap, shift=hist.shift, certified_nodes=len(pg), nodes=len(hist.uncertified), stored_pairs=len(ub),
            n_rounds=len(hist.rounds), phase_seconds_total=phase, prunes=prunes, rounds=hist.rounds,
            final=final_costs(model, ub, hist.uncertified.rows, K, target))
        print(json.dumps(dict(progress=name, growth=growth, wall_s=wall, lower=hist.lower, upper=hist.upper, rounds=len(hist.rounds))),
              file=sys.stderr, flush=True)
        del pg, ub, hist
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'gap_prune_b200.json'))
    ap.add_argument('models', nargs='*', default=['hallway', 'tigergrid', 'olfactory_wrap'])
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), growth=GROWTH, models=[])
    for tag in args.models:
        if tag == 'olfactory_wrap':
            model, gamma = olfactory_wrap_model(), 0.99
        else:
            model, gamma = golden_model(tag)
        res['models'].append(run(tag, model, gamma))
    text = json.dumps(res)
    with open(args.out, 'w') as f:
        f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
