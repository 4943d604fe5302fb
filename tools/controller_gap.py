"""
Certified lower bounds from finite-state controllers (`PolicyGraph`), beside the certified upper bounds of `bounds.py`:
  per model: an FSVI solve (as tools/bound_gap.py: 30 expansions x 100 beliefs, eps 1e-6, seed 0, tracking level 2); the controller
  extracted from it (witnesses b0 + the explored beliefs: wall time, nodes, closure rounds); its evaluation (eps 1e-6: sweeps, wall time,
  residual, shift); the time of one `pbvi_controller_sweep` launch (with the fused residual) and of `pbvi_backup_assemble` on the same rows
  and tuples, alternated, CUDA events over `REPS` launches per sample, median of `SAMPLES` samples; the bytes a sweep must move
  (N*S*8 read + N*S*8 written + the model tensors reach / RTO / Rbar, from shapes) and the rate that makes against 7.7 TB/s; at b0 the
  solve's own max_v alpha_v . b0, the certified controller value and the FIB / improved upper bound (`passes` improve passes over the
  explored beliefs); the discounted return of 1000 simulated agents (mean and standard error, horizon with gamma^H max|Rbar| / (1 - gamma)
  < 1e-6).
Models: the olfactory wrap model (22021 states, gamma 0.99), hallway and tiger-grid (golden fixtures, gamma 0.95).
    python tools/controller_gap.py [passes]
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
from pomdp_pbvi_exploration_b200 import FIB_Solver, FSVI_Solver, PolicyGraph, UpperBound  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402
from bound_gap import golden_model, synced  # noqa: E402

HBM_BYTES_PER_S = 7.7e12       # HGX B200 data sheet, one GPU
REPS, SAMPLES = 50, 7


def launch_ms(fn):
    """Mean time of one launch over REPS back-to-back launches, CUDA events."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / REPS


def run(name, model, gamma, passes):
    dev = model.device
    out = dict(model=name, S=model.state_count, A=model.action_count, O=model.observation_count, R=model.reachable_state_count, gamma=gamma)
    fib, _ = FIB_Solver(gamma=gamma, eps=1e-6).solve(model, print_progress=False)
    np.random.seed(0)
    random.seed(0)
    vf, hist = FSVI_Solver(gamma=gamma, eps=1e-6).solve(model, expansions=30, max_belief_growth=100, history_tracking_level=2,
                                                       print_progress=False)
    B = hist.belief_sets[-1].belief_array
    out.update(alphas=len(vf), beliefs=int(B.shape[0]))
    PolicyGraph.from_value_function(model, vf, B[:4])[0].evaluate(gamma, max_sweeps=2)     # warm-up: module loads, allocations
    t0 = synced()
    pg, st = PolicyGraph.from_value_function(model, vf, B)
    out['extraction'] = dict(wall_s=synced() - t0, nodes=st['nodes'], closure_rounds=st['closure_rounds'])
    t0 = synced()
    rows, h = pg.evaluate(gamma)
    out['evaluation'] = dict(wall_s=synced() - t0, sweeps=h.sweeps, final_change=h.final_change, residual=h.residual, shift=h.shift)

    act = torch.as_tensor(pg.actions, dtype=torch.int32, device=rows.device)
    succ = torch.as_tensor(pg.successors, dtype=torch.int32, device=rows.device).contiguous()
    sweep = lambda: dev.controller_sweep(rows, gamma, act, succ, want_stats=True)         # noqa: E731
    assemble = lambda: dev.backup_assemble(rows, gamma, act, succ)                         # noqa: E731
    assert sweep()[0].cpu().numpy().tobytes() == assemble().cpu().numpy().tobytes()
    t_sw, t_as = [], []
    for _ in range(SAMPLES):
        t_sw.append(launch_ms(sweep))
        t_as.append(launch_ms(assemble))
    N, S, A, O, R = len(pg), model.state_count, model.action_count, model.observation_count, model.reachable_state_count
    moved = 2 * N * S * 8 + S * A * R * 4 + S * A * O * R * 8 + S * A * 8
    ms = float(np.median(t_sw))
    out['sweep'] = dict(ms=ms, ms_samples=t_sw, bytes=moved, fits_l2=moved < 126e6, rate_TBps=moved / ms * 1e-9,
                        share_of_7_7TBps=moved / ms * 1e3 / HBM_BYTES_PER_S, backup_assemble_ms=float(np.median(t_as)), backup_assemble_ms_samples=t_as)

    ub = UpperBound(model, fib, gamma)
    lower, fib_upper = ub.gap(vf)
    for _ in range(passes):
        ub.improve(B)
    b0 = model.start_probabilities
    out['b0'] = dict(solve_lower=lower, controller_lower=float(pg.value(b0)[0][0]), fib_upper=fib_upper, improved_upper=ub.gap(vf)[1],
                     improve_passes=passes)
    rbar_max = float(np.max(np.abs(model.expected_rewards_table)))
    H = int(np.ceil(np.log(1e-6 * (1 - gamma) / rbar_max) / np.log(gamma))) + 1
    try:
        t0 = time.perf_counter()
        ret = pg.simulate(1000, H, seed=0)
        out['simulation'] = dict(agents=1000, horizon=H, mean=float(ret.mean()), se=float(ret.std(ddof=1) / np.sqrt(len(ret))),
                                 wall_s=time.perf_counter() - t0)
    except ValueError as e:
        out['simulation'] = dict(skipped=str(e))
    return out


def main():
    passes = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), models=[])
    res['models'].append(run('olfactory_wrap', olfactory_wrap_model(), 0.99, passes))
    for tag in ('hallway', 'tigergrid'):
        model, gamma = golden_model(tag)
        res['models'].append(run(tag, model, gamma, passes))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
