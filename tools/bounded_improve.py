"""
Bounded policy iteration (`PolicyGraph.bounded_improve`) on the controllers the engine produces:
  extracted  the controller extracted from an FSVI 30 x 100 solve (tools/policy_iteration.py)
  gap        the certified controller of a LONG_S-second `GapSolver` run (K = 16, prune_growth = 1.1), after `prune_lp`
Recorded per controller and iteration: certified value at b0, nodes, improved / not improvable / budget / failed nodes, LP rounds, largest
column count, pivots, pool rows and the phase seconds (device-synchronised wall clock: `pbvi_bpi_lp` synchronises, and the pricing reads
its tuples back).  Iterations stop at a fixed point, after ITERATIONS, or once they have taken BUDGET_S seconds.  For comparison
`improve` runs over the explored beliefs of the FSVI solve (extracted) from the same controller for at least the same wall time.  The
ms per `pbvi_bpi_lp` launch and per pricing `backup_select` round are CUDA-event times, medians over the rounds of one LP pass.
Models: hallway and tiger-grid (golden fixtures, gamma 0.95), the olfactory wrap model (22021 states, gamma 0.99).
    python tools/bounded_improve.py [--out PATH] [--append] [model ...]     (default PATH: profiles/bounded_improve_b200.json)
Writes one JSON document and prints it; each model entry carries the GPU name and power limit read in its run.  With --append the models
are added to the document at PATH (one run per model keeps each run short).
"""
import argparse
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
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from pomdp_pbvi_exploration_b200 import FSVI_Solver, GapSolver, PolicyGraph  # noqa: E402
from pomdp_pbvi_exploration_b200 import policy_graph as pgm  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402
from bound_gap import golden_model, synced  # noqa: E402
from gap_solve import LONG_S, SETTINGS  # noqa: E402

GROWTH = 1.1
ITERATIONS = 10
BUDGET_S = 45.0


def b0_value(pg) -> float:
    return float(pg.value(pg.model.start_probabilities)[0][0])


def lp_round_costs(pg) -> dict:
    """Median ms of one `pbvi_bpi_lp` launch and of one pricing round (backup_select at the tangent beliefs) over the LP rounds."""
    dev = pg.model.device
    lp, sel = [], []
    real_lp, real_tuples = dev.bpi_lp, pgm.backup_tuples

    def timed(fn, into):
        def call(*a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a)
            e1.record()
            e1.synchronize()
            into.append(e0.elapsed_time(e1))
            return r
        return call
    timed_lp, timed_tuples = timed(real_lp, lp), timed(real_tuples, sel)
    dev.bpi_lp, pgm.backup_tuples = timed_lp, timed_tuples
    try:
        act = torch.as_tensor(pg.actions, dtype=torch.int32, device='cuda')
        succ = torch.as_tensor(pg.successors, dtype=torch.int32, device='cuda')
        own = dev.controller_evaluate_mixed(pg.rows, pg.gamma, act, succ, pg.mixtures or pgm.NO_MIXTURES, float('inf'), 1)[0]
        tau = 1e-9 * max(1.0, float(torch.max(torch.abs(pg.rows))), float(torch.max(torch.abs(own))))
        pgm.bpi_lps(dev, pg.rows, own, pg.gamma, tau)
    finally:
        del dev.bpi_lp
        pgm.backup_tuples = real_tuples
    return dict(bpi_lp_launches=len(lp), bpi_lp_ms_median=float(np.median(lp)), select_rounds=len(sel),
                select_ms_median=float(np.median(sel)) if sel else None)


def run_bpi(pg, beliefs) -> tuple:
    rows, t_all = [], 0.0
    cur = pg
    for _ in range(ITERATIONS):
        t0 = synced()
        cur, st = cur.bounded_improve(beliefs, 1)
        dt = synced() - t0
        t_all += dt
        rows.append(dict(st[0], wall_seconds=dt))
        if st[0]['improved'] == 0 or t_all >= BUDGET_S:
            break
    return cur, rows, t_all


def run_improve(pg, B, wall) -> list:
    rows, t_all, cur = [], 0.0, pg
    while t_all < wall:
        t0 = synced()
        cur, st = cur.improve(B, 1)
        dt = synced() - t0
        t_all += dt
        rows.append(dict(value_b0=st[0]['value_b0'], nodes=st[0]['nodes_after'], wall_seconds=dt, cumulative_seconds=t_all))
        if st[0]['appended'] == 0 and st[0]['overwritten'] == 0:
            break
    return rows


def run(name, model, gamma):
    target, K, depth, rounds = SETTINGS[name]
    out = dict(model=name, S=model.state_count, A=model.action_count, O=model.observation_count, gamma=gamma)
    np.random.seed(0)
    random.seed(0)
    vf, fh = FSVI_Solver(gamma=gamma, eps=1e-6).solve(model, expansions=30, max_belief_growth=100, history_tracking_level=2,
                                                     print_progress=False)
    B = fh.belief_sets[-1].belief_array
    pg, _ = PolicyGraph.from_value_function(model, vf, B)
    pg.evaluate(gamma)
    pg.bounded_improve(None, 1)                                                                         # warm-up
    ext = dict(source='FSVI 30 x 100, extracted', nodes=len(pg), value_b0=b0_value(pg), costs=lp_round_costs(pg))
    _, ext['bpi'], wall = run_bpi(pg, None)
    ext['improve_at_equal_wall_time'] = run_improve(pg, B, wall)
    out['extracted'] = ext
    GapSolver(gamma, target, trials=2, max_depth=3, seed=0, prune_growth=GROWTH).solve(model, max_rounds=2)     # warm-up
    gp, _, hist = GapSolver(gamma, target, trials=K, max_depth=depth, seed=0, prune_growth=GROWTH).solve(
        model, max_rounds=rounds, time_limit=LONG_S)
    gp = gp.prune_lp()
    gap = dict(source=f'GapSolver K={K}, prune_growth={GROWTH}, {LONG_S:.0f} s, then prune_lp', certified_upper_b0=hist.upper,
               nodes=len(gp), value_b0=b0_value(gp), mixtures=0 if gp.mixtures is None else len(gp.mixtures[0]) - 1,
               costs=lp_round_costs(gp))
    _, gap['bpi'], _ = run_bpi(gp, None)
    out['gap'] = gap
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'bounded_improve_b200.json'))
    ap.add_argument('--append', action='store_true')
    ap.add_argument('models', nargs='*', default=['hallway', 'tigergrid', 'olfactory_wrap'])
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), iterations=ITERATIONS, budget_seconds=BUDGET_S, models=[],
               total_seconds=0.0)
    if args.append and os.path.isfile(args.out):
        with open(args.out) as f:
            res = json.load(f)
    t_start = time.perf_counter()
    for tag in args.models:
        if tag == 'olfactory_wrap':
            model, gamma = olfactory_wrap_model(), 0.99
        else:
            model, gamma = golden_model(tag)
        res['models'].append(dict(run(tag, model, gamma), gpu=gpu))
        print(json.dumps(res['models'][-1]), flush=True)
    res['total_seconds'] += time.perf_counter() - t_start
    text = json.dumps(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
