"""
Gap-driven solves (`GapSolver`) beside the fixed-belief-set improvers they replace:
  per model: a GapSolver solve from the blind controller and the FIB bound, with a time limit equal to the wall time the committed
  measurements spent to reach their bounds (profiles/policy_iteration_b200.json: FSVI solve + extraction + ten `improve` iterations;
  profiles/bound_gap_b200.json: FSVI solve + ten `UpperBound.improve` passes; the larger of the two), and one of LONG_S seconds.
  Recorded round by round: certified
  lower and upper at b0 where a round certified, the uncertified lower, upper(b0), nodes, stored pairs, trial depths and phase times.
  Then the per-level cost of `gap_trial_step` against the same level composed from existing calls (upper_backup with its actions,
  read-back of a*, belief_update of the O successors of a*, max_values and UpperBound.evaluate on them, read-back, the choice on the
  host, belief_update of the chosen successors), on K trial beliefs of a random walk, the lower rows and upper bound the long solve ended
  with:
  CUDA events around each, alternated, median of SAMPLES samples; whether both give the same a*, o* and next beliefs is recorded.
Models: hallway and tiger-grid (golden fixtures, gamma 0.95), the olfactory wrap model (22021 states, gamma 0.99).
    python tools/gap_solve.py
Prints one JSON line, with the GPU name and power limit read in the same run.
"""
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

SAMPLES = 11
LONG_S = 30.0                  # the second solve of every model: what half a minute of wall time reaches
# (target gap, trials K, max depth, max rounds); the graph grows by at most K nodes per level, so by K * max_depth per round: on the
# olfactory model (22021 * 8 bytes a row) 30 rounds of 16 trials x 100 levels make at most 48 000 nodes, 8.5 GB of rows
SETTINGS = {'hallway': (0.01, 16, 100, 400), 'tigergrid': (0.01, 16, 100, 400), 'olfactory_wrap': (0.1, 16, 100, 30)}


def reference(name):
    """(lower, upper, wall seconds) at b0 of the committed fixed-belief-set measurements of this model."""
    prof = os.path.join(ROOT, 'profiles')

    def models(fname):                               # a JSON document, or log lines followed by one JSON line
        with open(os.path.join(prof, fname)) as f:
            text = f.read()
        try:
            return json.loads(text)['models']
        except json.JSONDecodeError:
            return json.loads([ln for ln in text.splitlines() if ln.startswith('{"')][-1])['models']
    pi = next(m for m in models('policy_iteration_b200.json') if m['model'] == name)
    bg = next(m for m in models('bound_gap_b200.json') if m['model'] == name)
    lower_wall = bg['fsvi']['wall_s'] + pi['extracted']['wall_s'] + sum(it['wall_s'] for it in pi['iterations'])
    upper_wall = bg['fsvi']['wall_s'] + sum(p['wall_s'] for p in bg['passes'])
    return dict(certified_lower_b0=pi['b0']['improved_lower'], upper_b0=pi['b0']['improved_upper'], lower_wall_s=lower_wall,
                upper_wall_s=upper_wall, improve_iterations=len(pi['iterations']), upper_passes=pi['b0']['upper_improve_passes'])


def composed_level(dev, ub, X, b, theta):
    """One argmax-rule level from existing calls: returns (a*, o*, next beliefs [live rows])."""
    K, O = b.shape[0], dev.O
    idx, val, count, dot, vals, n_ub = ub._lists()
    _, _, act = dev.upper_backup(b, ub._F, ub.gamma, ub.corner_values, idx, val, count, dot, vals, n_ub, want_action=True)
    a = act.cpu().numpy()
    rep = b.repeat_interleave(O, dim=0)
    succ, mass = dev.belief_update(rep, np.repeat(a, O).astype(np.int32), np.tile(np.arange(O), K).astype(np.int32), normalise=True)
    ok = mass > 0
    succ = torch.where(ok[:, None], succ, torch.zeros_like(succ))
    L = dev.max_values(succ, X)[0]
    U = ub.evaluate(succ)
    e = (mass * ((U - L) - theta)).cpu().numpy().reshape(K, O)
    ok = ok.cpu().numpy().reshape(K, O)
    e = np.where(ok & (e > 0), e, 0.0)
    o = np.where(e.max(axis=1) > 0, np.argmax(e, axis=1), -1)
    live = np.flatnonzero(o >= 0)
    nxt = dev.belief_update(b[live], a[live].astype(np.int32), o[live].astype(np.int32), normalise=True)[0] if len(live) else None
    return a, o, nxt


def level_cost(model, ub, X, K, theta):
    dev = model.device
    rng = np.random.default_rng(0)
    b0 = torch.as_tensor(model.start_probabilities, device='cuda', dtype=torch.float64)
    walk = dev.perseus_walk(b0, rng.integers(0, model.action_count, 4 * K).astype(np.int32), rng.random(4 * K))
    b = walk[-K:].contiguous()
    idx, val, count, dot, vals, n_ub = ub._lists()

    def fused():
        out, nxt = dev.gap_trial_step(b, X, ub._F, ub.gamma, ub.corner_values, idx, val, count, dot, vals, n_ub, theta)
        res = out.cpu().numpy()
        return res[:, 0].astype(np.int64), res[:, 1].astype(np.int64), nxt

    fa, fo, fn = fused()
    ca, co, cn = composed_level(dev, ub, X, b, theta)
    live = np.flatnonzero(fo >= 0)
    same = bool(np.array_equal(fa, ca) and np.array_equal(fo, co) and
                (len(live) == 0 or fn[live].cpu().numpy().tobytes() == cn.cpu().numpy().tobytes()))
    t_f, t_c = [], []
    for _ in range(SAMPLES):
        for fn_, acc in ((fused, t_f), (lambda: composed_level(dev, ub, X, b, theta), t_c)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn_()
            e1.record()
            e1.synchronize()
            acc.append(e0.elapsed_time(e1))
    return dict(K=K, lower_rows=int(X.shape[0]), stored_pairs=len(ub), theta=theta, same_choices=same, live=int(len(live)),
                gap_trial_step_ms=float(np.median(t_f)), composed_ms=float(np.median(t_c)), gap_trial_step_samples=t_f, composed_samples=t_c,
                speedup=float(np.median(t_c) / np.median(t_f)))


def run(name, model, gamma):
    target, K, depth, rounds = SETTINGS[name]
    ref = reference(name)
    limit = max(ref['lower_wall_s'], ref['upper_wall_s'])
    out = dict(model=name, S=model.state_count, A=model.action_count, O=model.observation_count, gamma=gamma, target_gap=target, trials=K,
               max_depth=depth, max_rounds=rounds, reference=ref)
    GapSolver(gamma, target, trials=2, max_depth=3, seed=0).solve(model, max_rounds=1)        # warm-up: module loads, allocations
    for key, lim in (('solve', limit), ('solve_long', LONG_S)):
        t0 = synced()
        pg, ub, hist = GapSolver(gamma, target, trials=K, max_depth=depth, seed=0).solve(model, max_rounds=rounds, time_limit=lim)
        wall = synced() - t0
        out[key] = dict(time_limit_s=lim, wall_s=wall, reached=hist.reached, certified_lower_b0=hist.lower, certified_upper_b0=hist.upper,
                        gap=hist.gap, shift=hist.shift, certified_nodes=len(pg), nodes=len(hist.uncertified), stored_pairs=len(ub),
                        rounds=hist.rounds)
    out['level_cost'] = [level_cost(model, ub, hist.uncertified.rows, k, target) for k in (1, K)]
    return out


def main():
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, torch_device=torch.cuda.get_device_name(0), models=[])
    names = sys.argv[1:] or ['hallway', 'tigergrid', 'olfactory_wrap']
    for tag in names:
        if tag == 'olfactory_wrap':
            model, gamma = olfactory_wrap_model(), 0.99
        else:
            model, gamma = golden_model(tag)
        res['models'].append(run(tag, model, gamma))
        print(json.dumps(dict(progress=tag, **{k: res['models'][-1]['solve'][k] for k in ('wall_s', 'certified_lower_b0', 'certified_upper_b0')})),
              file=sys.stderr, flush=True)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
