"""
LP dominance of controller nodes (`PolicyGraph.prune_lp`) on the controllers the engine produces:
  gap       the certified controller of a LONG_S-second `GapSolver` run (K = 16, max depth 100, prune_growth = 1.1: tools/gap_prune.py)
  improved  the controller after ITERATIONS `improve` iterations over the explored beliefs of an FSVI solve (tools/policy_iteration.py)
Recorded per controller: nodes before, after `prune_dominated` and after `prune_lp`, mixtures and their members, the LP counts and
`prune_lp_stats`, the prune seconds; the certified lower(b0) before, right after the prune (bitwise the same by construction) and after a
re-`evaluate` from the pruned rows; ms per `evaluate` sweep and per `outcomes` sweep before and after (CUDA events, median of SAMPLES
after one warm-up); and for the olfactory model the outcomes at b0 with H = HORIZON, before and after.
Models: hallway and tiger-grid (golden fixtures, gamma 0.95), the olfactory wrap model (22021 states, gamma 0.99).
    python tools/controller_lp_prune.py [--out PATH] [model ...]        (default PATH: profiles/controller_lp_prune_b200.json)
Writes one JSON document, with the GPU name and power limit read in the same run, and prints it.
"""
import argparse
import json
import os
import random
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from pomdp_pbvi_exploration_b200 import FSVI_Solver, GapSolver, PolicyGraph  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402
from bound_gap import golden_model, synced  # noqa: E402
from gap_solve import LONG_S, SETTINGS  # noqa: E402

SAMPLES = 5
GROWTH = 1.1
ITERATIONS = 10
SWEEPS = 20                    # sweeps per timed evaluate / outcomes call
HORIZON = 1000


def median_ms(fn, per=1) -> float:
    fn()
    samples = []
    for _ in range(SAMPLES):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        samples.append(e0.elapsed_time(e1) / per)
    return float(np.median(samples))


def sweep_costs(model, pg, gamma) -> dict:
    dev = model.device
    act = torch.as_tensor(pg.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(pg.successors, dtype=torch.int32, device='cuda')
    if pg.mixtures is None:
        ev = lambda: dev.controller_evaluate(pg.rows, gamma, act, succ, 0.0, SWEEPS)                  # noqa: E731
    else:
        ev = lambda: dev.controller_evaluate_mixed(pg.rows, gamma, act, succ, pg.mixtures, 0.0, SWEEPS)  # noqa: E731
    return dict(evaluate_ms_per_sweep=median_ms(ev, SWEEPS), outcomes_ms_per_sweep=median_ms(lambda: pg.outcomes(SWEEPS, gamma=gamma), SWEEPS))


def b0_value(pg) -> float:
    return float(pg.value(pg.model.start_probabilities)[0][0])


def measure(model, gamma, pg, with_horizon) -> dict:
    before = b0_value(pg)
    out = dict(nodes=len(pg), lower_b0_before=before, cost_before=sweep_costs(model, pg, gamma))
    if with_horizon:
        t0 = synced()
        o = pg.outcomes(HORIZON, gamma=gamma)
        out['outcomes_H_before'] = dict(H=HORIZON, success=float(o.success[0]), steps=float(o.steps[0]),
                                        discounted_return=float(o.discounted_return[0]), seconds=synced() - t0)
    t0 = synced()
    pr = pg.prune_lp()
    out['prune_seconds'] = synced() - t0
    st = pr.prune_stats
    out.update(nodes_after_dominated=st['after_dominated'], nodes_after_lp=len(pr), mixtures=st['mixtures'], nnz=st['nnz'],
               lp_counts=dict(zip(('kept_corner', 'kept_lp_witness', 'pruned', 'kept_undecided'), st['lp_counts'])),
               lp_stats=st['lp_stats'], failed_verification=st['failed'], prune_seconds_inner=st['seconds'])
    after = b0_value(pr)
    out.update(lower_b0_after_prune=after, lower_b0_bitwise_equal=after == before, cost_after=sweep_costs(model, pr, gamma))
    if with_horizon:
        t0 = synced()
        o = pr.outcomes(HORIZON, gamma=gamma)
        out['outcomes_H_after'] = dict(H=HORIZON, success=float(o.success[0]), steps=float(o.steps[0]),
                                       discounted_return=float(o.discounted_return[0]), seconds=synced() - t0)
    re = PolicyGraph(model, pr.actions, pr.successors, mixtures=pr.mixtures)
    re._initial = pr.rows
    _, h = re.evaluate(gamma)
    out.update(lower_b0_after_reevaluate=b0_value(re), reevaluate_sweeps=h.sweeps, reevaluate_shift=h.shift)
    return out


def run(name, model, gamma):
    target, K, depth, rounds = SETTINGS[name]
    out = dict(model=name, S=model.state_count, A=model.action_count, O=model.observation_count, gamma=gamma)
    GapSolver(gamma, target, trials=2, max_depth=3, seed=0, prune_growth=GROWTH).solve(model, max_rounds=2)     # warm-up
    pg, _, hist = GapSolver(gamma, target, trials=K, max_depth=depth, seed=0, prune_growth=GROWTH).solve(
        model, max_rounds=rounds, time_limit=LONG_S)
    out['gap'] = dict(source=f'GapSolver K={K}, prune_growth={GROWTH}, {LONG_S:.0f} s', certified_upper_b0=hist.upper,
                      **measure(model, gamma, pg, name == 'olfactory_wrap'))
    np.random.seed(0)
    random.seed(0)
    vf, fh = FSVI_Solver(gamma=gamma, eps=1e-6).solve(model, expansions=30, max_belief_growth=100, history_tracking_level=2,
                                                     print_progress=False)
    B = fh.belief_sets[-1].belief_array
    pg, _ = PolicyGraph.from_value_function(model, vf, B)
    pg.evaluate(gamma)
    for _ in range(ITERATIONS):
        pg, st = pg.improve(B, 1)
        if st[0]['appended'] == 0 and st[0]['overwritten'] == 0:
            break
    out['improved'] = dict(source=f'FSVI 30 x 100, {ITERATIONS} improve iterations', **measure(model, gamma, pg, name == 'olfactory_wrap'))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'controller_lp_prune_b200.json'))
    ap.add_argument('models', nargs='*', default=['hallway', 'tigergrid', 'olfactory_wrap'])
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), samples=SAMPLES, sweeps_per_call=SWEEPS, models=[])
    for tag in args.models:
        if tag == 'olfactory_wrap':
            model, gamma = olfactory_wrap_model(), 0.99
        else:
            model, gamma = golden_model(tag)
        res['models'].append(run(tag, model, gamma))
        print(json.dumps(res['models'][-1]), flush=True)
    text = json.dumps(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
