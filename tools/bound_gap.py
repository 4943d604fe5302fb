"""
Optimality gap of FSVI solves, measured with the certified upper bounds of `bounds.py` (FIB_Solver + UpperBound):
  per model: FIB sweeps and wall time; an FSVI solve (gamma as below, 30 expansions x 100 beliefs, eps 1e-6, seed 0, tracking level 2);
  lower(b0) = max_v alpha_v . b0 of the solve, FIB upper(b0) (FIB_Solver eps 1e-3, the default, and 1e-6, whose rows
  the bound uses), then for each `improve` pass over the solve's explored beliefs its wall
  time, the stored-pair count, the pbvi_upper_backup chunk size and the improved upper(b0).
Models: the olfactory wrap model (22021 states, gamma 0.99), hallway and tiger-grid (golden fixtures, gamma 0.95).
    python tools/bound_gap.py [passes]
Prints one JSON line, with the GPU name and power limit read in the same run.
"""
import json
import os
import random
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pomdp_pbvi_exploration_b200 import FIB_Solver, FSVI_Solver, Model, UpperBound  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402


def golden_model(tag):
    m = dict(np.load(os.path.join(ROOT, 'tests', 'golden', f'model_{tag}.npz')))
    S, A, O = m['rto'].shape[0], m['rto'].shape[1], m['rto'].shape[2]
    return Model(states=S, actions=A, observations=O, transitions=m['transition_table'], rewards=m['reward_table'],
                 observation_table=m['obs_table'], start_probabilities=m['start']), float(m['gamma'])


def synced():
    torch.cuda.synchronize()
    return time.perf_counter()


def run(name, model, gamma, passes):
    out = dict(model=name, S=model.state_count, A=model.action_count, O=model.observation_count, R=model.reachable_state_count, gamma=gamma)
    FIB_Solver(gamma=gamma).solve(model, print_progress=False)                       # warm-up: module loads, allocations
    for eps in (1e-3, 1e-6):                                                          # the default, and the rows the bound uses
        t0 = synced()
        fib, fh = FIB_Solver(gamma=gamma, eps=eps).solve(model, print_progress=False)
        out[f'fib_eps{eps:g}'] = dict(sweeps=len(fh.iteration_times), wall_s=synced() - t0, residual=fh.fib_residual, shift=fh.fib_shift,
                                      upper_b0=float(model.device.max_values(model.start_belief_device[None, :], fib.alpha_vector_array)[0][0]))
    np.random.seed(0)
    random.seed(0)
    t0 = synced()
    vf, hist = FSVI_Solver(gamma=gamma, eps=1e-6).solve(model, expansions=30, max_belief_growth=100, history_tracking_level=2,
                                                       print_progress=False)
    out['fsvi'] = dict(expansions=len(hist.expansion_times), wall_s=synced() - t0, alphas=len(vf))
    B = hist.belief_sets[-1].belief_array
    warm = UpperBound(model, fib, gamma)
    warm.improve(B[:2])
    ub = UpperBound(model, fib, gamma)
    lower, upper = ub.gap(vf)
    out.update(beliefs=int(B.shape[0]), lower_b0=lower, fib_upper_b0=upper, passes=[])
    for _ in range(passes):
        chunk = ub._chunk(B.shape[0])
        t0 = synced()
        n_dec, largest = ub.improve(B)
        wall = synced() - t0
        out['passes'].append(dict(wall_s=wall, first_chunk=chunk, last_chunk=ub._chunk(B.shape[0]), decreased=n_dec, largest_decrease=largest,
                                  stored=len(ub), upper_b0=ub.gap(vf)[1]))
    return out


def main():
    passes = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), passes=passes, models=[])
    res['models'].append(run('olfactory_wrap', olfactory_wrap_model(), 0.99, passes))
    for tag in ('hallway', 'tigergrid'):
        model, gamma = golden_model(tag)
        res['models'].append(run(tag, model, gamma, passes))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
