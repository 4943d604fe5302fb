"""
ValueFunction.prune(3): LP-domination pruning on the device (pbvi_prune_lp).

The reference's level 3 cannot run (`pruned_alpha_set` undefined, src/mdp.py:872), so it cannot serve as the oracle.  The contract
(include/pbvi_b200.h, ValueFunction.prune) is checked against:
  * HiGHS (scipy.optimize.linprog) witness margins delta_i on value functions of real solves;
  * sets whose answer is known by construction at olfactory-like sizes (tangent planes of |b|^2 are all useful, convex combinations
    of them lowered by eps >> tau are all useless), plus tiny hand-made cases;
  * the value function itself: max over the kept rows == max over all rows at corners, random beliefs and the solve's beliefs;
  * solves with prune_level=3, single-process and sharded over two ranks.
"""
import ctypes
import os
import random
import socket

import numpy as np
import pytest

from conftest import load_golden

MODELS = ['tiger', 'grid4x4', 'grid4x4_noloop', 'tigergrid', 'hallway', 'cheese', 'grid4x3', 'cit']


def tol_of(rows):
    return 1e-9 * max(1.0, float(np.max(np.abs(rows[np.isfinite(rows).all(axis=1)])))) if len(rows) else 1e-9


def lp_witness_margins(alphas):
    """delta_i = max_{b in simplex} min_{j != i} b . (alpha_i - alpha_j) per row, by HiGHS.  This is the LP the reference's level 3
    intended (src/mdp.py:834-906); its own branch is broken, so this restatement is the oracle."""
    from scipy.optimize import linprog
    n, S = alphas.shape
    out = np.full(n, np.inf)
    for i in range(n):
        others = np.delete(alphas, i, axis=0)
        if len(others) == 0:
            continue
        # variables (b_0..b_{S-1}, delta): minimise -delta s.t. delta - b . (alpha_i - alpha_j) <= 0, sum b = 1, b >= 0
        A_ub = np.hstack([-(alphas[i] - others), np.ones((len(others), 1))])
        res = linprog(np.r_[np.zeros(S), -1.0], A_ub=A_ub, b_ub=np.zeros(len(others)), A_eq=np.r_[np.ones(S), 0.0][None, :], b_eq=[1.0],
                      bounds=[(0, None)] * S + [(None, None)], method='highs',
                      options=dict(primal_feasibility_tolerance=1e-10, dual_feasibility_tolerance=1e-10))
        assert res.status == 0, res.message
        out[i] = -res.fun
    return out


# ---- CPU: argument checks of the C ABI ------------------------------------------------------------------------------------------
def test_prune_lp_rejects_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    counts = (ctypes.c_int32 * 4)()
    assert lib.pbvi_prune_lp(None, None, 3, None, None, counts, None) == _native.PBVI_ERR_BAD_ARG
    assert b'NULL' in lib.pbvi_last_error()
    assert lib.pbvi_prune_lp(None, None, -1, None, None, None, None) == _native.PBVI_ERR_BAD_ARG
    assert b'non-negative' in lib.pbvi_last_error()
    assert lib.pbvi_prune_lp_stats(None, None) == _native.PBVI_ERR_BAD_ARG


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
def seed_all(seed):
    np.random.seed(seed)
    random.seed(seed)


_models = {}


def fixture_model(tag):
    """A package `Model` carrying exactly the reference's tensors of the fixture (bypasses the constructor's own derivations)."""
    from pomdp_pbvi_exploration_b200 import Model
    if tag in _models:
        return _models[tag]
    m = load_golden('model_' + tag)
    reach = m['reach'].astype(np.int64)
    S, A, R = reach.shape
    O = m['rto'].shape[2]
    model = Model.__new__(Model)
    model._device_handle = None
    model.is_on_gpu = True
    model.state_labels = [f's_{i}' for i in range(S)]
    model.state_count, model.states = S, np.arange(S)
    model.action_labels = [f'a_{i}' for i in range(A)]
    model.action_count, model.actions = A, np.arange(A)
    model.observation_labels = [f'o_{i}' for i in range(O)]
    model.observation_count, model.observations = O, np.arange(O)
    model.reachable_states, model.reachable_state_count = reach, R
    model.reachable_probabilities = m['probs'] if 'probs' in m else np.ones(reach.shape)
    model.observation_table = m['obs_table'] if 'obs_table' in m else None
    model.reachable_transitional_observation_table = m['rto']
    model.expected_rewards_table = m['rbar']
    model.start_probabilities = m['start']
    model.end_states = m['end_states'].tolist()
    model.end_actions = []
    model._min_reward = float(m['min_reward']) if 'min_reward' in m else 0.0
    model._max_reward = float(m['max_reward']) if 'max_reward' in m else 1.0
    model.transition_table = m.get('transition_table')
    model.immediate_reward_table = m.get('reward_table')
    model.immediate_reward_function = None
    model.rewards_are_probabilistic = False
    model.state_grid = np.arange(S).reshape(1, S)
    _models[tag] = (model, float(m['gamma']))
    return _models[tag]


_devices = {}


def bare_device(S):
    """A one-action, one-observation device model with S states: pbvi_prune_lp only needs the state count."""
    from pomdp_pbvi_exploration_b200._native import DeviceModel
    if S not in _devices:
        _devices[S] = DeviceModel(np.zeros((S, 1, 1), np.int64), np.ones((S, 1, 1)), np.ones((S, 1, 1, 1)), np.zeros((S, 1)), device=0)
    return _devices[S]


_solves = {}


def seeded_solve(tag, prune_level=1, prune_interval=10):
    from pomdp_pbvi_exploration_b200 import PBVI_Solver
    key = (tag, prune_level, prune_interval)
    if key not in _solves:
        model, gamma = fixture_model(tag)
        seed_all(5)
        solver = PBVI_Solver(gamma=gamma, eps=1e-6, expand_function='perseus')
        vf, hist = solver.solve(model, expansions=8, max_belief_growth=25, prune_level=prune_level, prune_interval=prune_interval,
                                history_tracking_level=2, print_progress=False)
        _solves[key] = (model, vf, hist)
    return _solves[key]


def check_value_unchanged(rows, keep, beliefs=None, seed=0):
    """max over the kept rows == max over all rows (corners, Dirichlet and sparse beliefs, `beliefs`), and the argmax is the same
    original row wherever the best row leads the runner-up by more than 1e-9 * scale."""
    import torch
    n, S = rows.shape
    scale = max(1.0, float(np.max(np.abs(rows[np.isfinite(rows).all(axis=1)]))))
    R = torch.as_tensor(rows, device='cuda')
    kept = np.flatnonzero(keep)
    RK = R[torch.as_tensor(kept, device='cuda')]
    g = torch.Generator(device='cuda').manual_seed(seed)
    sets = []
    for b0 in range(0, S, 4096):                                            # corners
        idx = torch.arange(b0, min(S, b0 + 4096), device='cuda')
        sets.append(torch.zeros((len(idx), S), dtype=torch.float64, device='cuda').scatter_(1, idx[:, None], 1.0))
    for _ in range(5):                                                       # 5 x 1000 Dirichlet(1)
        e = -torch.log(torch.rand((1000, S), dtype=torch.float64, device='cuda', generator=g))
        sets.append(e / e.sum(dim=1, keepdim=True))
    for k, reps in ((2, 2), (5, 3)):                                         # 5 x 1000 sparse (k non-zeros)
        for _ in range(reps):
            sup = torch.randint(0, S, (1000, k), device='cuda', generator=g)
            w = -torch.log(torch.rand((1000, k), dtype=torch.float64, device='cuda', generator=g))
            b = torch.zeros((1000, S), dtype=torch.float64, device='cuda')
            b.scatter_add_(1, sup, w)
            sets.append(b / b.sum(dim=1, keepdim=True))
    if beliefs is not None:
        sets.append(torch.as_tensor(np.asarray(beliefs), dtype=torch.float64, device='cuda'))
    finite = torch.isfinite(R).all(dim=1)
    RF = R[finite]
    fidx = torch.nonzero(finite).flatten()
    kept_t = torch.as_tensor(kept, device='cuda')
    n_checked = 0
    for B in sets:
        allv = B @ RF.T
        top = torch.topk(allv, min(2, RF.shape[0]), dim=1)
        kv = B @ RK[torch.isfinite(RK).all(dim=1)].T
        kmax, karg = kv.max(dim=1)
        torch.testing.assert_close(kmax, top.values[:, 0], rtol=1e-12, atol=1e-12 * scale)
        if RF.shape[0] > 1:
            clear = (top.values[:, 0] - top.values[:, 1]) > 1e-9 * scale
            kept_f = kept_t[torch.isfinite(RK).all(dim=1)]
            assert torch.equal(kept_f[karg[clear]], fidx[top.indices[clear, 0]])
        n_checked += B.shape[0]
    return n_checked


def prune_both_levels(dev, rows):
    """Indices (into `rows`) kept by level 2 then the LP stage, and the LP's (keep, bound, counts) on the level-2 rows."""
    k2 = np.flatnonzero(dev.prune_dominated(rows).cpu().numpy())
    keep, bound, counts = dev.prune_lp(rows[k2])
    return k2, keep.cpu().numpy(), bound.cpu().numpy(), counts


@pytest.mark.gpu
@pytest.mark.parametrize('tag', MODELS)
def test_prune_lp_matches_highs_on_solved_value_functions(tag):
    model, vf, hist = seeded_solve(tag)
    rows = vf.alpha_vector_array.cpu().numpy()
    k2, keep, bound, counts = prune_both_levels(model.device, vf.alpha_vector_array)
    P = rows[k2]
    tau = tol_of(P)
    scale = tau * 1e9
    delta = lp_witness_margins(P)
    assert counts[3] == 0, counts
    assert counts.sum() == len(P) and counts[2] == int(np.sum(keep == 0))
    must_prune = delta < -tau - 1e-10 * scale
    must_keep = delta > -tau + 1e-10 * scale
    assert np.all(keep[must_prune] == 0), (tag, np.flatnonzero(must_prune & (keep != 0)))
    assert np.all(keep[must_keep] == 1), (tag, np.flatnonzero(must_keep & (keep != 1)))
    kept, pruned = keep == 1, keep == 0
    assert np.all(delta[kept] >= bound[kept] - 1e-12 * scale)
    assert np.all(delta[pruned] <= bound[pruned] + 1e-12 * scale)
    assert np.all(bound[pruned] < -tau)
    full_keep = np.zeros(len(rows), dtype=bool)
    full_keep[k2[keep == 1]] = True
    check_value_unchanged(rows, full_keep, hist.belief_sets[-1].belief_array.cpu().numpy())


def tangent_planes(S, n, k, rng):
    """alpha_k = 2 b_k - |b_k|^2 1 for k-sparse random beliefs b_k: alpha_k . b = |b|^2 - |b - b_k|^2, each one best exactly at b_k."""
    B = np.zeros((n, S))
    states = rng.permutation(S)                                   # disjoint supports
    for r in range(n):
        B[r, states[r * k:(r + 1) * k]] = rng.dirichlet(np.ones(k))
    return 2 * B - np.sum(B * B, axis=1, keepdims=True), B


@pytest.mark.gpu
@pytest.mark.parametrize('S,n_planes,n_comb', [(2000, 200, 150), (8000, 600, 400), (22021, 1200, 800)])
def test_prune_lp_ground_truth_by_construction(S, n_planes, n_comb):
    import torch
    rng = np.random.default_rng(S)
    planes, _ = tangent_planes(S, n_planes, 6, rng)
    eps = 1e-4
    comb = np.zeros((n_comb, S))
    for r in range(n_comb):
        parts = rng.choice(n_planes, size=int(rng.integers(2, 4)), replace=False)
        lam = rng.dirichlet(4 * np.ones(len(parts)))
        comb[r] = lam @ planes[parts] - eps
    rows = np.concatenate([planes, comb])[rng.permutation(n_planes + n_comb)]
    useful = np.zeros(len(rows), dtype=bool)
    order = {r.tobytes(): i for i, r in enumerate(rows)}
    for p in planes:
        useful[order[p.tobytes()]] = True
    dev = bare_device(S)
    R = torch.as_tensor(rows, device='cuda')
    assert int(dev.prune_dominated(R).sum()) == len(rows), 'level 2 must keep every row: the LP stage decides'
    keep, bound, counts = dev.prune_lp(R)
    keep, bound = keep.cpu().numpy(), bound.cpu().numpy()
    assert np.array_equal(keep == 1, useful), (np.flatnonzero((keep == 1) != useful)[:10], counts)
    assert counts[3] == 0 and counts[2] == n_comb, counts
    tau = tol_of(rows)
    assert np.all(bound[useful] > -tau) and np.all(bound[~useful] < -tau)
    # the certificate really holds in FP64 for every pruned row: checked through the bound, and pruning again removes nothing
    keep2, _, counts2 = dev.prune_lp(R[torch.as_tensor(np.flatnonzero(keep), device='cuda')])
    assert int(keep2.sum()) == int(keep.sum()) and counts2[2] == 0
    assert check_value_unchanged(rows, keep == 1, seed=S) >= 10000


def run_tiny(rows):
    import torch
    rows = np.asarray(rows, dtype=np.float64)
    keep, bound, counts = bare_device(rows.shape[1]).prune_lp(torch.as_tensor(rows, device='cuda'))
    return keep.cpu().numpy(), bound.cpu().numpy(), counts


@pytest.mark.gpu
def test_prune_lp_tiny_cases():
    keep, bound, counts = run_tiny([[1.0], [2.0], [3.0]])                  # S = 1: only the largest survives
    assert keep.tolist() == [0, 0, 1] and counts.tolist() == [1, 0, 2, 0]
    assert bound.tolist()[:2] == [-2.0, -1.0]
    keep, bound, counts = run_tiny([[0.3, -7.0]])                          # n = 1: no competitor
    assert keep.tolist() == [1] and counts.tolist() == [1, 0, 0, 0] and bound[0] == np.inf
    keep, _, counts = run_tiny([[1.0, 0.0], [0.0, 1.0], [0.5, 0.5]])       # exact three-way tie at (1/2, 1/2): the middle row is kept
    assert keep.tolist() == [1, 1, 1] and counts.tolist() == [2, 1, 0, 0]
    keep, bound, counts = run_tiny([[1.0, 0.0], [0.0, 1.0], [0.4, 0.4]])   # beaten by (1/2, 1/2) of the others by 0.1 everywhere
    assert keep.tolist() == [1, 1, 0] and counts.tolist() == [2, 0, 1, 0]
    assert abs(bound[2] - (-0.1)) < 1e-15
    keep, bound, counts = run_tiny([[1.0, 0.0], [np.nan, 0.0], [0.0, 1.0], [0.2, 0.2], [5.0, np.inf]])   # non-finite rows: kept, no competitor
    assert keep.tolist() == [1, 1, 1, 0, 1] and counts.tolist() == [4, 0, 1, 0]
    assert np.isnan(bound[1]) and np.isnan(bound[4])
    keep, _, counts = run_tiny([[1.0, 0.0], [0.0, 1.0], [0.5 - 1e-12, 0.5 - 1e-12]])    # within tau of the tie: kept
    assert keep.tolist() == [1, 1, 1]
    keep, _, counts = run_tiny(np.zeros((0, 3)))
    assert keep.shape == (0,) and counts.tolist() == [0, 0, 0, 0]


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4', 'hallway', 'cit'])
def test_prune3_on_value_function_keeps_rows_order_actions_hashes(tag):
    from pomdp_pbvi_exploration_b200 import ValueFunction
    model, vf, hist = seeded_solve(tag)
    rows, actions = vf.numpy()
    hashes = vf.row_hashes.copy()
    k2, keep, _, _ = prune_both_levels(model.device, vf.alpha_vector_array)
    sel = k2[keep == 1]
    v3 = ValueFunction(model, rows, actions)
    v3.prune(3)
    got_rows, got_actions = v3.numpy()
    assert np.array_equal(got_rows, rows[sel]) and np.array_equal(got_actions, actions[sel])
    assert np.array_equal(v3.row_hashes, hashes[sel])
    n3 = len(v3)
    again = ValueFunction(model, got_rows, got_actions)
    again.prune(3)
    assert len(again) == n3
    check_value_unchanged(rows, np.isin(np.arange(len(rows)), sel), hist.belief_sets[-1].belief_array.cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4', 'cheese'])
def test_solve_with_final_prune3_equals_prune_lp_of_level1_solve(tag):
    model, vf1, _ = seeded_solve(tag, prune_level=1)
    _, vf3, hist3 = seeded_solve(tag, prune_level=3, prune_interval=10 ** 6)
    rows1, actions1 = vf1.numpy()
    k2, keep, _, _ = prune_both_levels(model.device, vf1.alpha_vector_array)
    sel = k2[keep == 1]
    rows3, actions3 = vf3.numpy()
    assert np.array_equal(rows3, rows1[sel]) and np.array_equal(actions3, actions1[sel])
    assert hist3.prune_counts == [len(sel) - len(rows1)]


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4'])
@pytest.mark.parametrize('flavour', ['fsvi', 'perseus_full'])
def test_solves_prune3_every_second_iteration(tag, flavour):
    from pomdp_pbvi_exploration_b200 import FSVI_Solver, PBVI_Solver, ValueFunction
    model, gamma = fixture_model(tag)
    seed_all(7)
    if flavour == 'fsvi':
        solver, kw = FSVI_Solver(gamma=gamma, eps=1e-6), {}
    else:
        solver, kw = PBVI_Solver(gamma=gamma, eps=1e-6, expand_function='perseus'), dict(full_backup=True)
    vf, hist = solver.solve(model, expansions=8, max_belief_growth=10, prune_level=3, prune_interval=2, print_progress=False, **kw)
    n_iter = len(hist.backup_times)
    assert len(hist.pruning_times) == (n_iter - 1) // 2 + 1 and all(c <= 0 for c in hist.prune_counts)
    rows, actions = vf.numpy()
    again = ValueFunction(model, rows, actions)
    again.prune(3)
    assert len(again) == len(vf)


# ---- two ranks on one GPU (gloo): the sharded solve prunes its replicated value function identically on every rank ------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _sharded_solve(group):
    import torch
    from pomdp_pbvi_exploration_b200 import PBVI_Solver
    from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model
    model = olfactory_wrap_model(points_per_unit=6)
    seed_all(11)
    solver = PBVI_Solver(gamma=0.99, eps=1e-6, expand_function='perseus')
    extra = dict(group=group, replicate_below=64) if group is not None else {}
    vf, hist = solver.solve(model, expansions=6, max_belief_growth=40, full_backup=True, prune_level=3, prune_interval=2,
                            print_progress=False, **extra)
    torch.cuda.synchronize()
    return (vf.alpha_vector_array.cpu().numpy(), vf.actions.copy(), list(hist.alpha_vector_counts), list(hist.beliefs_counts),
            list(hist.prune_counts))


def _sharded_worker(rank, world, port, queue):
    import torch
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    if rank != 0:
        seed_all(999 + rank)
    queue.put((rank,) + _sharded_solve(True))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_perseus_solve_with_prune3_equals_single_process():
    import torch.multiprocessing as mp
    want = _sharded_solve(None)
    world = 2
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_sharded_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, rows, actions, n_alpha, n_belief, pruned in results:
        assert np.array_equal(rows, want[0]), rank
        assert np.array_equal(actions, want[1]), rank
        assert n_alpha == want[2] and n_belief == want[3] and pruned == want[4], rank
