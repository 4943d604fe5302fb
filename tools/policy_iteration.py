"""
Point-based policy iteration on extracted controllers (`PolicyGraph.improve`), beside the certified upper bound:
  per model: the FSVI solve of tools/controller_gap.py (30 expansions x 100 beliefs, eps 1e-6, seed 0); the controller extracted from it
  (witnesses b0 + the explored beliefs) and evaluated (eps 1e-6); then up to ITERATIONS `improve` iterations over the explored beliefs,
  one call per iteration, recording per iteration the certified value at b0, nodes, appended / overwritten / pruned counts, evaluation
  sweeps, certificate shift and the seconds of each phase; at b0 the FIB upper bound and the upper bound after `passes` improve passes.
  Per-sweep cost of the evaluation, on the extracted graph and on the last improved one: K sweeps as one `pbvi_controller_evaluate`
  launch (tol 0) against K `pbvi_controller_sweep` launches each followed by its scalar read-back (the loop `evaluate` ran before),
  alternated, CUDA events around each, median of SAMPLES samples.
Models: the olfactory wrap model (22021 states, gamma 0.99), hallway and tiger-grid (golden fixtures, gamma 0.95).
    python tools/policy_iteration.py [passes]
Prints one JSON line, with the GPU name and power limit read in the same run.
"""
import json
import os
import random
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pomdp_pbvi_exploration_b200 import FIB_Solver, FSVI_Solver, PolicyGraph, UpperBound  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402
from bound_gap import golden_model, synced  # noqa: E402

ITERATIONS, K, SAMPLES = 10, 200, 7


def sweep_costs(model, pg, gamma):
    """Median ms per sweep of K sweeps: one persistent launch against K single launches with a read-back each."""
    dev = model.device
    rows = pg.rows
    act = torch.as_tensor(pg.actions, dtype=torch.int32, device=rows.device)
    succ = torch.as_tensor(pg.successors, dtype=torch.int32, device=rows.device).contiguous()

    def device_loop():
        return dev.controller_evaluate(rows, gamma, act, succ, 0.0, K)[0]

    def host_loop():
        W = rows
        for _ in range(K):
            W, st = dev.controller_sweep(W, gamma, act, succ, want_stats=True)
            float(st[2])
        return W

    assert device_loop().cpu().numpy().tobytes() == host_loop().cpu().numpy().tobytes()
    t_dev, t_host = [], []
    for _ in range(SAMPLES):
        for fn, acc in ((device_loop, t_dev), (host_loop, t_host)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            acc.append(e0.elapsed_time(e1) / K)
    single = []
    for _ in range(SAMPLES):                                   # the kernel alone: K launches, no read-back
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            dev.controller_sweep(rows, gamma, act, succ, want_stats=True)
        e1.record()
        e1.synchronize()
        single.append(e0.elapsed_time(e1) / K)
    return dict(nodes=len(pg), sweeps=K, device_loop_ms_per_sweep=float(np.median(t_dev)), host_loop_ms_per_sweep=float(np.median(t_host)),
                back_to_back_launch_ms=float(np.median(single)), device_loop_samples=t_dev, host_loop_samples=t_host,
                speedup=float(np.median(t_host) / np.median(t_dev)))


def run(name, model, gamma, passes):
    out = dict(model=name, S=model.state_count, A=model.action_count, O=model.observation_count, R=model.reachable_state_count, gamma=gamma)
    fib, _ = FIB_Solver(gamma=gamma, eps=1e-6).solve(model, print_progress=False)
    np.random.seed(0)
    random.seed(0)
    vf, hist = FSVI_Solver(gamma=gamma, eps=1e-6).solve(model, expansions=30, max_belief_growth=100, history_tracking_level=2,
                                                       print_progress=False)
    B = hist.belief_sets[-1].belief_array
    out.update(alphas=len(vf), beliefs=int(B.shape[0]))
    warm, _ = PolicyGraph.from_value_function(model, vf, B[:4])                # warm-up: module loads, allocations
    warm.evaluate(gamma, max_sweeps=2)
    warm.improve(B[:4], 1)
    t0 = synced()
    pg, st = PolicyGraph.from_value_function(model, vf, B)
    _, h = pg.evaluate(gamma)
    out['extracted'] = dict(wall_s=synced() - t0, nodes=len(pg), sweeps=h.sweeps, shift=h.shift,
                            value_b0=float(pg.value(model.start_probabilities)[0][0]))
    out['sweep_cost_extracted'] = sweep_costs(model, pg, gamma)
    its = []
    for _ in range(ITERATIONS):
        t0 = synced()
        pg, stats = pg.improve(B, 1)
        stats[0]['wall_s'] = synced() - t0
        its.append(stats[0])
        if stats[0]['appended'] == 0 and stats[0]['overwritten'] == 0:
            break
    out['iterations'] = its
    out['sweep_cost_improved'] = sweep_costs(model, pg, gamma)
    ub = UpperBound(model, fib, gamma)
    lower, fib_upper = ub.gap(pg.value_function)
    for _ in range(passes):
        ub.improve(B)
    out['b0'] = dict(extracted_lower=out['extracted']['value_b0'], improved_lower=lower, fib_upper=fib_upper,
                     improved_upper=ub.gap(pg.value_function)[1], upper_improve_passes=passes)
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
