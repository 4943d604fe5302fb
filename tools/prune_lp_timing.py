"""
Cost and effect of ValueFunction.prune(3) (LP-domination pruning, pbvi_prune_lp) on the olfactory model (22021 states):
  1. the engine's FSVI solve, 300 expansions x 100 beliefs, gamma 0.99, eps 1e-6, prune_level=1 (no pruning);
  2. prune(3) on its final value function, timed per stage (level 2, LP stage; the LP stage split into the corner screen and the
     cutting-plane kernel by torch.profiler), after a warm-up on a copy;
  3. the same solve with prune_level=3, prune_interval=10: wall time, final |V| and the change of max_v alpha . b over the final
     belief set against the unpruned solve.
    python tools/prune_lp_timing.py [expansions] [growth]
Prints the GPU name and power limit of the run.
"""
import os
import random
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pomdp_pbvi_exploration_b200 import FSVI_Solver, ValueFunction  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402


def solve(model, expansions, growth, **kw):
    np.random.seed(0)
    random.seed(0)
    solver = FSVI_Solver(gamma=0.99, eps=1e-6)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vf, hist = solver.solve(model, expansions=expansions, max_belief_growth=growth, print_progress=False, history_tracking_level=2, **kw)
    torch.cuda.synchronize()
    return vf, hist, time.perf_counter() - t0


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def main():
    expansions = int(sys.argv[1]) if len(sys.argv) > 1 else 300
    growth = int(sys.argv[2]) if len(sys.argv) > 2 else 100
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    print(f'GPU: {gpu}   (torch: {torch.cuda.get_device_name(0)})')
    model = olfactory_wrap_model()
    dev = model.device
    vf1, hist1, wall1 = solve(model, expansions, growth, prune_level=1)
    rows, actions = vf1.numpy()
    print(f'FSVI {expansions}x{growth} prune_level=1: {wall1:.1f} s, |V| = {len(vf1)}, |B| = {hist1.beliefs_counts[-1]}')

    warm = ValueFunction(model, rows, actions)
    warm.prune(3)
    vf = ValueFunction(model, rows, actions)
    keep2, t2 = timed(lambda: dev.prune_dominated(vf.alpha_vector_array))
    P = vf.alpha_vector_array[keep2.bool()].contiguous()
    (keep3, bound, counts), t3 = timed(lambda: dev.prune_lp(P))
    stats = dev.prune_lp_stats()
    print(f'prune(3) on the final V: |V| {len(rows)} -> level 2: {P.shape[0]} -> level 3: {int(keep3.sum())}')
    print(f'  counts {{kept at a corner, kept by an LP witness, pruned, kept undecided}} = {counts.tolist()}')
    print(f'  largest |J| = {stats["max_competitors"]} (cap 64), rows in the LP stage = {stats["lp_rows"]}, restricted LPs = {stats["lps"]}, '
          f'pivots = {stats["pivots"]}')
    print(f'  time: level 2 {t2:.2f} ms, LP stage (pbvi_prune_lp) {t3:.2f} ms')
    _, t_whole = timed(lambda: ValueFunction(model, rows, actions).prune(3))
    print(f'  ValueFunction.prune(3) end to end: {t_whole:.2f} ms')
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dev.prune_lp(P)
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type.name == 'CUDA' and 'prune_lp' in e.name:
            name = e.name.split('(')[0].replace('void ', '').replace('pbvi::', '')
            per[name] = per.get(name, 0.0) + e.device_time / 1e3
    for name, ms in per.items():
        print(f'    kernel {name}: {ms:.3f} ms')

    vf3, hist3, wall3 = solve(model, expansions, growth, prune_level=3, prune_interval=10)
    B = hist1.belief_sets[-1].belief_array
    v1 = dev.max_values(B, vf1.alpha_vector_array)[0]
    v3 = dev.max_values(B, vf3.alpha_vector_array)[0]
    d = (v3 - v1).abs()
    print(f'FSVI {expansions}x{growth} prune_level=3 prune_interval=10: {wall3:.1f} s (prune_level=1: {wall1:.1f} s), |V| = {len(vf3)}, '
          f'|B| = {hist3.beliefs_counts[-1]}, prune steps {len(hist3.prune_counts)} removing {-sum(hist3.prune_counts)} rows in '
          f'{sum(hist3.pruning_times):.2f} s')
    print(f'  |max_v alpha.b (pruned solve) - max_v alpha.b (unpruned solve)| over the {B.shape[0]} final beliefs of the unpruned solve: '
          f'max {float(d.max()):.3e}, mean {float(d.mean()):.3e}')


if __name__ == '__main__':
    main()
