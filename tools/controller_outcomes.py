"""
Exact outcomes of olfactory controllers (`PolicyGraph.outcomes`, one persistent `pbvi_controller_outcomes` launch) beside a Monte Carlo
estimate of the same quantities:
  controllers: the one extracted from the FSVI 30 x 100 solve (eps 1e-6, seed 0, as tools/controller_gap.py) and the one a 30 s
  GapSolver run certifies (the settings of tools/gap_solve.py: K = 16, max depth 100, from the blind controller and the FIB bound).
  Per controller at H = MAX_STEPS, from b0 and its best node, with the model's end state (the odour source):
    ms per sweep: CUDA events around the launch (the binding's call, which synchronises once) divided by H, median of SAMPLES calls
    after one warm-up call; wall time of the whole `outcomes` call; the 6 N S doubles of rows and scratch;
    P(T <= H), E[min(T, H)] and the discounted return G at b0 (the reference prints gamma * G as its average discounted reward);
    a host NumPy Monte Carlo of MC_AGENTS roll-outs under the same termination rule: its wall time, means and standard errors.
    python tools/controller_outcomes.py [--out PATH]        (default PATH: profiles/controller_outcomes_b200.json)
Writes one JSON document, with the GPU name and power limit read in the same run, and prints it.
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
from pomdp_pbvi_exploration_b200 import FSVI_Solver, GapSolver, PolicyGraph  # noqa: E402
from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model  # noqa: E402

MAX_STEPS = 1000
SAMPLES = 5
MC_AGENTS = 10000
GAP_SECONDS = 30.0


def synced():
    torch.cuda.synchronize()
    return time.perf_counter()


def monte_carlo(model, pg, gamma, H, n, seed):
    """n roll-outs from b0 and its best node; a run stops after a step that lands in an end state or plays an end action."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, O, R = rto.shape
    end = np.zeros(S, dtype=bool)
    end[np.asarray(model.end_states, dtype=np.int64)] = True
    end_a = np.zeros(A, dtype=bool)
    end_a[np.asarray(model.end_actions, dtype=np.int64)] = True
    t0 = time.perf_counter()
    rng = np.random.default_rng(seed)
    p = np.asarray(model.start_probabilities, dtype=np.float64)
    s = rng.choice(S, size=n, p=p / p.sum())
    node = np.full(n, int(pg.value(p)[1][0]), dtype=np.int64)
    cdf = np.cumsum(rto.reshape(S, A, O * R), axis=2)
    alive = np.ones(n, dtype=bool)
    done, steps, ret = np.zeros(n, dtype=bool), np.zeros(n), np.zeros(n)
    disc = 1.0
    for _ in range(H):
        if not alive.any():
            break
        a = pg.actions[node]
        ret += np.where(alive, disc * rbar[s, a], 0.0)
        steps += alive
        k = np.minimum((cdf[s, a] <= rng.random(n)[:, None]).sum(axis=1), O * R - 1)
        s = reach[s, a, k % R]
        node = pg.successors[node, k // R]
        stop = alive & (end[s] | end_a[a])
        done |= stop
        alive &= ~stop
        disc *= gamma

    def stat(x):
        return dict(mean=float(x.mean()), standard_error=float(x.std(ddof=1) / np.sqrt(n)))
    return dict(agents=n, seed=seed, wall_s=time.perf_counter() - t0, success=stat(done.astype(np.float64)), steps=stat(steps),
                discounted_return=stat(ret))


def measure(name, model, gamma, pg):
    dev = model.device
    N, S = len(pg), model.state_count
    b0 = torch.as_tensor(model.start_probabilities, dtype=torch.float64, device='cuda')[None, :]
    n0 = pg.value(b0)[1]
    end = np.zeros(S, dtype=np.uint8)
    end[np.asarray(model.end_states, dtype=np.int64)] = 1
    end_a = np.zeros(model.action_count, dtype=np.uint8)
    end_a[np.asarray(model.end_actions, dtype=np.int64)] = 1

    def launch():
        return dev.controller_outcomes(pg.actions, pg.successors, end, end_a, gamma, MAX_STEPS, b0, n0)
    launch()                                                                        # warm-up: module load, arena growth
    per_sweep = []
    for _ in range(SAMPLES):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        e1.synchronize()
        per_sweep.append(e0.elapsed_time(e1) / MAX_STEPS)
    t0 = synced()
    out = pg.outcomes(MAX_STEPS, gamma=gamma)
    wall = synced() - t0
    mc = monte_carlo(model, pg, gamma, MAX_STEPS, MC_AGENTS, seed=0)
    g = float(out.discounted_return[0])
    res = dict(controller=name, nodes=N, S=S, gamma=gamma, max_steps=MAX_STEPS, start_node=int(out.start_nodes[0]),
               ms_per_sweep=float(np.median(per_sweep)), ms_per_sweep_samples=per_sweep, outcomes_wall_s=wall,
               row_bytes=6 * N * S * 8, success_b0=float(out.success[0]), steps_b0=float(out.steps[0]), discounted_return_b0=g,
               reference_adr_b0=gamma * g, certified_value_b0=float(pg.value(b0)[0][0]) if pg.rows is not None else None,
               success_at=[float(out.success_curve[0, k - 1]) for k in (10, 50, 100, 200, 500, 1000)], monte_carlo=mc)
    print(json.dumps(dict(progress=name, nodes=N, ms_per_sweep=res['ms_per_sweep'], success=res['success_b0'], steps=res['steps_b0'],
                          ret=g, mc=mc['success']['mean'])), file=sys.stderr, flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'controller_outcomes_b200.json'))
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    model, gamma = olfactory_wrap_model(), 0.99
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), model='olfactory_wrap', end_states=list(map(int, model.end_states)),
               controllers=[])
    np.random.seed(0)
    random.seed(0)
    vf, hist = FSVI_Solver(gamma=gamma, eps=1e-6).solve(model, expansions=30, max_belief_growth=100, history_tracking_level=2,
                                                       print_progress=False)
    pg, _ = PolicyGraph.from_value_function(model, vf, hist.belief_sets[-1].belief_array)
    pg.evaluate(gamma)
    res['controllers'].append(measure('fsvi_30x100_extracted', model, gamma, pg))
    del pg, vf, hist
    t0 = synced()
    pg, _, hist = GapSolver(gamma, 0.1, trials=16, max_depth=100, seed=0).solve(model, max_rounds=30, time_limit=GAP_SECONDS)
    gap = dict(wall_s=synced() - t0, certified_lower_b0=hist.lower, upper_b0=hist.upper)
    res['controllers'].append(dict(measure('gap_solver_30s', model, gamma, pg), gap_solve=gap))
    text = json.dumps(res)
    with open(args.out, 'w') as f:
        f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
