"""
Bounded policy iteration (PolicyGraph.bounded_improve, pbvi_bpi_lp).  Checked:
  * the LP optimum eps* of every node against HiGHS on the full tuple set (tiger controllers small enough to enumerate A * N^O tuples);
  * certificates (sum lambda Y_J - W_n > tau) and tangent beliefs ((HW)(b*) - W_n . b* = -m*, with the oracle's backup) in NumPy FP64;
  * batching (bitwise the same for every batch split) and determinism of a whole iteration;
  * after an iteration: X <= T' X of the start rows, W <= T_pi W of the result, no fall of the certified value beyond the shift, the
    value below the certified upper bound, roll-outs that agree with it; strict improvement on tiger from the blind controller and a
    fixed point confirmed by the LP;
  * on the CPU: the graph surgery on hand-built solutions and the C ABI's argument checks.
"""
import ctypes

import numpy as np
import pytest

from test_controller_lp_prune import cpu_model, mixture_np, source_graph
from test_policy_graph import controller_sweep_np


# ---- CPU: graph surgery ------------------------------------------------------------------------------------------------------------
def test_split_groups_columns_by_action_and_flattens_mixtures():
    from pomdp_pbvi_exploration_b200.policy_graph import bpi_split
    N = 4
    mix = (np.array([0, 2]), np.array([1, 3]), np.array([0.25, 0.75]))          # entry 4 = mixture 0 = {1: 0.25, 3: 0.75}
    cols = [(0, np.array([4, 2])), (1, np.array([0, 0])), (0, np.array([1, 2])), (1, np.array([2, 0])), (2, np.array([3, 3]))]
    lam = np.array([0.2, 0.3, 0.2, 0.3, 1e-14])
    sp = bpi_split(cols, lam, N, mix)
    assert [a for a, _, _ in sp] == [0, 1]                                         # the weight below 1e-13 is dropped
    assert abs(sp[0][1] - 0.4) < 1e-15 and abs(sp[1][1] - 0.6) < 1e-15
    nodes, w = sp[0][2][0]                                                         # o = 0: 0.5 * {1: .25, 3: .75} + 0.5 * {1}
    np.testing.assert_array_equal(nodes, [1, 3])
    np.testing.assert_allclose(w, [0.625, 0.375], rtol=0, atol=1e-15)
    nodes, w = sp[0][2][1]                                                         # o = 1: both columns go to 2: merged
    np.testing.assert_array_equal(nodes, [2])
    nodes, w = sp[1][2][0]
    np.testing.assert_array_equal(nodes, [0, 2])
    np.testing.assert_allclose(w, [0.5, 0.5], rtol=0, atol=1e-15)


def test_assemble_redirects_edges_and_members_and_bounds_growth():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    from pomdp_pbvi_exploration_b200.policy_graph import bpi_assemble, bpi_split
    model, _ = cpu_model('tiger')
    A, O = model.action_count, model.observation_count
    act = np.array([0, 1, 2, 0])
    succ = np.array([[1, 4], [2, 2], [0, 3], [1, 1]])                             # entry 4 = mixture {1: 0.5, 2: 0.5}
    mix = (np.array([0, 2]), np.array([1, 2]), np.array([0.5, 0.5]))
    N = 4
    # node 1 splits into actions 0 and 2; node 3 improves with one action (in place); node 2 is left alone
    splits = {1: bpi_split([(0, np.array([0, 0])), (2, np.array([3, 3]))], [0.4, 0.6], N, mix),
              3: bpi_split([(1, np.array([0, 4]))], [1.0], N, mix)}
    a2, s2, m2, pos = bpi_assemble(act, succ, mix, splits, redirect=True)
    assert len(a2) - N == sum(len(sp) - 1 for sp in splits.values()) == 1         # growth: distinct actions - 1 per improved node
    assert pos[(1, 0)] == 1 and pos[(3, 0)] == 3 and pos[(1, 1)] == 4
    assert a2[1] == 0 and a2[4] == 2 and a2[3] == 1 and a2[0] == 0 and a2[2] == 2
    pg = PolicyGraph(model, a2, s2, mixtures=m2)                                  # a constructor-valid mixture table
    off, nodes, w = pg.mixtures
    N2 = len(a2)

    def dist(e):
        if e < N2:
            return {int(e): 1.0}
        k = e - N2
        return {int(n): float(x) for n, x in zip(nodes[off[k]:off[k + 1]], w[off[k]:off[k + 1]])}
    # edges into node 1 go to {1: 0.4, 4: 0.6}; node 0's mixture member 1 is flattened into it
    assert dist(s2[0, 0]) == pytest.approx({1: 0.4, 4: 0.6})
    assert dist(s2[2, 0]) == {0: 1.0} and dist(s2[2, 1]) == {3: 1.0}               # node 3 improved in place: no mixture
    assert dist(s2[0, 1]) == pytest.approx({1: 0.2, 4: 0.3, 2: 0.5})
    assert dist(s2[3, 1]) == pytest.approx({1: 0.2, 4: 0.3, 2: 0.5})
    assert all(v == 0 for v in (nodes >= N2))
    # without redirection every split node is appended and the old edges stay
    a3, s3, m3, pos3 = bpi_assemble(act, succ, mix, splits, redirect=False)
    assert len(a3) == N + 3 and np.array_equal(s3[:N], np.where(succ < N, succ, len(a3) + succ - N))
    assert np.array_equal(a3[:N], act)
    assert A == 3 and O == 2


def test_nodes_left_out_of_the_verified_splits_are_unchanged():
    from pomdp_pbvi_exploration_b200.policy_graph import bpi_assemble, bpi_split
    act = np.array([0, 1, 2, 0])
    succ = np.array([[1, 4], [2, 2], [0, 3], [1, 1]])
    mix = (np.array([0, 2]), np.array([1, 2]), np.array([0.5, 0.5]))
    splits = {1: bpi_split([(0, np.array([0, 0])), (2, np.array([3, 3]))], [0.4, 0.6], 4, mix),
              3: bpi_split([(1, np.array([0, 4])), (2, np.array([1, 1]))], [0.5, 0.5], 4, mix)}
    # node 1's improvement failed its verification: only node 3 is passed on
    a2, s2, m2, pos = bpi_assemble(act, succ, mix, {3: splits[3]}, redirect=True)
    N2 = len(a2)
    assert N2 == 5 and a2[1] == act[1] and np.array_equal(s2[1], succ[1]) and a2[0] == act[0] and s2[0, 0] == 1
    assert m2[1][m2[0][s2[0, 1] - N2]:m2[0][s2[0, 1] - N2 + 1]].tolist() == [1, 2]          # the mixture naming 1 and 2 is untouched
    assert s2[2, 1] >= N2 and sorted(m2[1][m2[0][s2[2, 1] - N2]:m2[0][s2[2, 1] - N2 + 1]].tolist()) == [3, 4]   # edges into 3: {3, 4}


def test_assemble_with_no_split_leaves_the_graph_unchanged():
    from pomdp_pbvi_exploration_b200.policy_graph import bpi_assemble
    act, succ = np.array([0, 1]), np.array([[1, 0], [0, 1]])
    a2, s2, m2, pos = bpi_assemble(act, succ, None, {}, redirect=True)
    assert np.array_equal(a2, act) and np.array_equal(s2, succ) and m2 is None and pos == {}


def test_reachable_nodes_follow_mixture_members():
    from pomdp_pbvi_exploration_b200.policy_graph import reachable_nodes, reachable_subgraph
    succ = np.array([[4, 0], [1, 1], [3, 3], [3, 3]])
    mix = (np.array([0, 2]), np.array([1, 2]), np.array([0.5, 0.5]))
    assert reachable_nodes(succ, [0], mix).tolist() == [True, True, True, True]
    assert reachable_nodes(succ, [2], mix).tolist() == [False, False, True, True]
    keep, _, _ = reachable_subgraph([0, 1, 0, 1], [[1, 1], [1, 1], [0, 0], [2, 2]], [3])
    assert keep.tolist() == [0, 1, 2, 3]


def test_bpi_lp_rejects_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    assert 'pbvi_bpi_lp' in _native.SIGNATURES and hasattr(lib, 'pbvi_bpi_lp')
    stats = (ctypes.c_int64 * 4)()
    assert len(_native.SIGNATURES['pbvi_bpi_lp']) == 17
    assert lib.pbvi_bpi_lp(None, None, 0, 0, 1e-9, *([None] * 10), stats, None) == _native.PBVI_ERR_BAD_ARG
    assert b'handle is NULL' in lib.pbvi_last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
def tuple_rows_np(model, W, gamma, tuples):
    """Y_t = backup_assemble(W, t) in NumPy: the controller sweep of nodes that play t."""
    ext = np.asarray(tuples, dtype=np.int64)
    T, N = len(ext), len(W)
    pad = np.concatenate([W, np.zeros((max(0, T - N), W.shape[1]))])          # the sweep writes one row per node of `pad`
    return controller_sweep_np(model, ext[:, 0], ext[:, 1:], pad, gamma)[:T]


def own_rows_np(model, pg, W, gamma):
    ext = W if pg.mixtures is None else np.concatenate([W, mixture_np(W, pg.mixtures)])
    return controller_sweep_np(model, pg.actions, pg.successors, ext, gamma)[:len(pg)]


def highs_eps(Y, w):
    """max eps s.t. sum_t lambda_t Y_t >= w + eps, sum lambda = 1, lambda >= 0 (HiGHS)."""
    from scipy.optimize import linprog
    T, S = Y.shape
    c = np.zeros(T + 1)
    c[-1] = -1.0
    A_ub = np.concatenate([-Y.T, np.ones((S, 1))], axis=1)
    A_eq = np.concatenate([np.ones((1, T)), np.zeros((1, 1))], axis=1)
    res = linprog(c, A_ub=A_ub, b_ub=-w, A_eq=A_eq, b_eq=[1.0], bounds=[(0, None)] * T + [(None, None)], method='highs',
                  options=dict(primal_feasibility_tolerance=1e-10, dual_feasibility_tolerance=1e-10))
    assert res.status == 0
    return -res.fun


def solve_lps(pg, batch=None):
    import torch
    from pomdp_pbvi_exploration_b200.policy_graph import NO_MIXTURES, bpi_lps
    dev = pg.model.device
    act = torch.as_tensor(pg.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(pg.successors, dtype=torch.int32, device='cuda')
    own = dev.controller_evaluate_mixed(pg.rows, pg.gamma, act, succ, pg.mixtures or NO_MIXTURES, float('inf'), 1)[0]
    tau = 1e-9 * max(1.0, float(torch.max(torch.abs(pg.rows))), float(torch.max(torch.abs(own))))
    return bpi_lps(dev, pg.rows, own, pg.gamma, tau, batch=batch), tau


def blind_tiger():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    from test_upper_bound import fixture_model
    model, gamma = fixture_model('tiger')
    pg = PolicyGraph.blind(model)
    pg.evaluate(gamma, eps=1e-9)
    return model, gamma, pg


@pytest.mark.gpu
@pytest.mark.parametrize('source', ['blind', 'extracted'])
def test_lp_optimum_equals_highs_on_all_tuples(source):
    import itertools
    if source == 'blind':
        model, gamma, pg = blind_tiger()
    else:
        model, gamma, _, pg = source_graph('tiger', 'extracted')
    N, A, O = len(pg), model.action_count, model.observation_count
    assert A * N ** O <= 20000
    W = pg.rows.cpu().numpy()
    tuples = [(a, *s) for a in range(A) for s in itertools.product(range(N), repeat=O)]
    Y = tuple_rows_np(model, W, gamma, tuples)
    sol, tau = solve_lps(pg)
    scale = max(1.0, float(np.abs(W).max()), float(np.abs(Y).max()))
    for n in range(N):
        eps = highs_eps(Y, W[n])
        st = sol['status'][n]
        assert st in (1, 2), (n, st)
        if st == 2:
            assert abs(-sol['delta'][n] - eps) <= 1e-9 * scale, (source, n, -sol['delta'][n], eps)
        else:
            assert eps <= 2 * tau, (source, n, eps)


def check_solution(model, pg, sol, tau):
    """Certificates and tangent beliefs of every node in NumPy FP64 (backup of the oracle)."""
    from oracle import pbvi_oracle as orc
    W = pg.rows.cpu().numpy()
    gamma = pg.gamma
    own = own_rows_np(model, pg, W, gamma)
    bstar = sol['bstar'].cpu().numpy()
    assert np.all(bstar >= 0.0) and np.all(np.abs(bstar.sum(axis=1) - 1.0) <= 1e-12)
    ref = orc.backup(np.asarray(model.reachable_states), model.reachable_transitional_observation_table, model.expected_rewards_table,
                     gamma, bstar, W)
    HW = ref['values'].max(axis=1)
    tang = HW - np.einsum('ns,ns->n', W, bstar)
    scale = max(1.0, float(np.abs(W).max()))
    checked = 0
    for n in range(len(pg)):
        st = sol['status'][n]
        if st in (1, 2):
            assert abs(tang[n] + sol['mstar'][n]) <= 1e-9 * scale, (n, tang[n], sol['mstar'][n])
        if st in (2, 3) and sol['u'][n] < -tau:
            cols = sol['columns'][n]
            cols = cols[cols > -2]
            rows = np.stack([own[n] if c == -1 else tuple_rows_np(model, W, gamma, sol['tuples'][c][None, :])[0] for c in cols])
            lam = sol['lam'][n][:len(cols)]
            assert np.all(lam >= 0.0) and abs(lam.sum() - 1.0) <= 1e-12
            assert np.all(lam @ rows - W[n] > tau), n
            checked += 1
    return checked


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x3', 'hallway', 'tigergrid'])
def test_certificates_and_tangent_beliefs(tag):
    model, gamma, B, pg = source_graph(tag, 'extracted')
    sol, tau = solve_lps(pg)
    checked = check_solution(model, pg, sol, tau)
    assert sol['stats']['max_columns'] <= 64
    assert checked > 0 or tag == 'tiger', tag


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'hallway'])
def test_batch_splits_give_bitwise_the_same_results(tag):
    model, gamma, B, pg = source_graph(tag, 'extracted')
    ref, _ = solve_lps(pg)

    def tuples_of(sol):
        return [tuple(-1 if c == -1 else tuple(sol['tuples'][c].tolist()) for c in row[row > -2]) for row in sol['columns']]
    for batch in (1, 3, max(1, len(pg) // 2)):
        got, _ = solve_lps(pg, batch=batch)
        for key in ('status', 'delta', 'u', 'mstar', 'lam'):
            assert got[key].tobytes() == ref[key].tobytes(), (tag, batch, key)
        assert got['bstar'].cpu().numpy().tobytes() == ref['bstar'].cpu().numpy().tobytes()
        assert tuples_of(got) == tuples_of(ref)


def check_iteration(model, gamma, B, pg, new, ub=None):
    import torch
    W = new.rows.cpu().numpy()
    ext = W if new.mixtures is None else np.concatenate([W, mixture_np(W, new.mixtures)])
    TW = controller_sweep_np(model, new.actions, new.successors, ext, gamma)[:len(new)]
    assert np.all(W <= TW + 1e-12 * np.maximum(1.0, np.abs(W))), float(np.max(W - TW))
    act = torch.as_tensor(new.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(new.successors, dtype=torch.int32, device='cuda')
    assert new._residual(new.rows, gamma, act, succ) <= 0.0


@pytest.mark.gpu
@pytest.mark.parametrize('source', ['extracted', 'improved', 'gap', 'lp'])
@pytest.mark.parametrize('tag', ['tiger', 'grid4x3', 'hallway', 'tigergrid'])
def test_one_iteration_is_sound(tag, source):
    from pomdp_pbvi_exploration_b200 import UpperBound
    from test_policy_graph import check_below_upper
    from test_upper_bound import fib_of
    model, gamma, B, pg = source_graph(tag, 'extracted' if source == 'lp' else source)
    if source == 'lp':
        pg = pg.prune_lp()
    R = np.concatenate([model.start_probabilities[None, :], B])
    before = pg.value(R)[0].cpu().numpy()
    new, stats = pg.bounded_improve(B, 1)
    st = stats[0]
    assert st['nodes_before'] == len(pg) and st['nodes_after'] == len(new)
    after = new.value(R)[0].cpu().numpy()
    assert np.all(after >= before - st['shift'] - 1e-12 * np.maximum(1.0, np.abs(before))), (tag, source, float(np.min(after - before)))
    if st['improved'] == 0:
        return
    check_iteration(model, gamma, B, pg, new)
    ub = UpperBound(model, fib_of(tag)[0], gamma)
    check_below_upper(model, new, ub, B)
    if not model.end_states:
        # roll-outs from b0 and its best node, long enough that the discounted tail is below 1e-6: within 4 standard errors of the
        # certified value, which lies below the controller's value by at most the evaluation tolerance
        rbar = np.abs(np.asarray(model.expected_rewards_table)).max()
        H = int(np.ceil(np.log(1e-6 * (1 - gamma) / max(rbar, 1e-300)) / np.log(gamma)))
        n = 10000
        ret = new.simulate(n, H, seed=3)
        V = float(after[0])
        se = ret.std(ddof=1) / np.sqrt(n)
        assert abs(ret.mean() - V) <= 4 * se + 1e-6 + 1e-4 * max(1.0, abs(V)), (tag, source, ret.mean(), V, se)


@pytest.mark.gpu
def test_strict_improvement_and_fixed_point_on_tiger():
    model, gamma, pg = blind_tiger()
    v0 = float(pg.value(model.start_probabilities)[0][0])
    new, stats = pg.bounded_improve(None, 1)
    assert stats[0]['improved'] >= 1 and stats[0]['value_b0'] > v0
    cur = new
    for _ in range(30):
        cur, st = cur.bounded_improve(None, 1)
        if st[-1]['improved'] == 0:
            break
    assert st[-1]['improved'] == 0 and len(cur) == st[-1]['nodes_before']
    check_iteration(model, gamma, None, cur, cur)
    # the LP over every tuple and every node's own row (HiGHS) finds no node that can be improved by more than tau, except those whose
    # improvement failed its verification
    import itertools
    N, A, O = len(cur), model.action_count, model.observation_count
    W = cur.rows.cpu().numpy()
    sol, tau = solve_lps(cur)
    if A * N ** O <= 20000:
        tuples = [(a, *s) for a in range(A) for s in itertools.product(range(N), repeat=O)]
        Y = np.concatenate([tuple_rows_np(model, W, gamma, tuples), own_rows_np(model, cur, W, gamma)])
        eps = np.asarray([highs_eps(Y, W[n]) for n in range(N)])
        assert int(np.sum(eps > 2 * tau)) <= st[-1]['failed'], (eps.max(), tau)


@pytest.mark.gpu
def test_bounded_improve_is_deterministic():
    model, gamma, B, pg = source_graph('hallway', 'extracted')
    a, sa = pg.bounded_improve(B, 2)
    b, sb = pg.bounded_improve(B, 2)
    assert np.array_equal(a.actions, b.actions) and np.array_equal(a.successors, b.successors)
    assert a.rows.cpu().numpy().tobytes() == b.rows.cpu().numpy().tobytes()
    assert (a.mixtures is None) == (b.mixtures is None)
    if a.mixtures is not None:
        assert all(x.tobytes() == y.tobytes() for x, y in zip(a.mixtures, b.mixtures))
    # a second iteration ran on a graph with mixtures when the first made any
    assert len(sa) == len(sb)


@pytest.mark.gpu
def test_bpi_lp_rejects_bad_arguments():
    import torch
    model, gamma, B, pg = source_graph('tiger', 'extracted')
    dev = model.device
    S = model.state_count
    z = lambda *shape, dt=torch.float64: torch.zeros(shape, dtype=dt, device='cuda')    # noqa: E731
    i = torch.int32
    args = [z(4, S), 2, 1e-9, z(2, dt=i), z(2, dt=i), z(2, 64, dt=i), z(2, dt=i), z(2, S), z(2), z(2), z(2, 64), z(2), z(2, dt=i)]
    with pytest.raises(ValueError, match='bpi_lp'):
        dev.bpi_lp(*args[:5], z(2, 63, dt=i), *args[6:])
    with pytest.raises(ValueError, match='2n rows'):
        dev.bpi_lp(z(3, S), *args[1:])
    with pytest.raises(ValueError, match='tau'):
        dev.bpi_lp(args[0], 2, 0.0, *args[3:])
    with pytest.raises(ValueError, match='tau'):
        dev.bpi_lp(args[0], 2, float('nan'), *args[3:])
    active = torch.full((2,), -1, dtype=torch.int32, device='cuda')
    with pytest.raises(ValueError, match='active entries'):
        dev.bpi_lp(*args[:12], active)                                              # active entries with no column
    cols = torch.full((2, 64), 4, dtype=torch.int32, device='cuda')
    with pytest.raises(ValueError, match='active entries'):
        dev.bpi_lp(*args[:5], cols, torch.ones(2, dtype=torch.int32, device='cuda'), *args[7:12], active)   # column row 4 >= 4


# ---- GPU: the start rows of the surgery -------------------------------------------------------------------------------------------
def lp_source(tag, source):
    model, gamma, B, pg = source_graph(tag, 'extracted' if source == 'lp' else source)
    return model, gamma, B, (pg.prune_lp() if source == 'lp' else pg)


@pytest.mark.gpu
@pytest.mark.parametrize('source', ['extracted', 'improved', 'gap', 'lp'])
@pytest.mark.parametrize('tag', ['tiger', 'grid4x3', 'hallway', 'tigergrid'])
def test_start_rows_lie_below_one_sweep_of_the_new_graph(tag, source):
    """X (W on the old nodes, one mixed sweep over W on the new ones) satisfies X <= T'X up to rounding, in NumPy and on the device:
    the invariant the soundness of the surgery rests on, checked before `evaluate` shifts anything."""
    import torch
    from pomdp_pbvi_exploration_b200.policy_graph import NO_MIXTURES
    model, gamma, B, pg = lp_source(tag, source)
    sol, tau = solve_lps(pg)
    nxt, splits, ok, unchanged = pg._bpi_start_graph(sol, tau)
    if nxt is None:
        assert tag == 'tiger' and not ok, (tag, source, len(splits))
        return
    X = nxt._initial.cpu().numpy()
    N = len(pg)
    assert X[:N][np.setdiff1d(np.arange(N), ok)].tobytes() == pg.rows.cpu().numpy()[np.setdiff1d(np.arange(N), ok)].tobytes()
    ext = X if nxt.mixtures is None else np.concatenate([X, mixture_np(X, nxt.mixtures)])
    TX = controller_sweep_np(model, nxt.actions, nxt.successors, ext, gamma)[:len(nxt)]
    allow = 1e-12 * max(1.0, float(np.abs(X).max()))
    assert float(np.max(X - TX)) <= allow, (tag, source, float(np.max(X - TX)))
    act = torch.as_tensor(nxt.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(nxt.successors, dtype=torch.int32, device='cuda')
    out = model.device.controller_evaluate_mixed(nxt._initial, gamma, act, succ, nxt.mixtures or NO_MIXTURES, float('inf'), 1)[0]
    assert float((nxt._initial - out).max()) <= allow
    assert len(nxt) - N <= sum(len(splits[n]) - 1 for n in ok)                      # the growth bound


# ---- GPU: the LP against HiGHS ----------------------------------------------------------------------------------------------------
def highs_lp(Y, w):
    """(eps, b*) of max eps s.t. sum_t lambda_t Y_t >= w + eps, sum lambda = 1, lambda >= 0; b* from the duals of the state rows."""
    from scipy.optimize import linprog
    T, S = Y.shape
    c = np.zeros(T + 1)
    c[-1] = -1.0
    res = linprog(c, A_ub=np.concatenate([-Y.T, np.ones((S, 1))], axis=1), b_ub=-w,
                  A_eq=np.concatenate([np.ones((1, T)), np.zeros((1, 1))], axis=1), b_eq=[1.0], bounds=[(0, None)] * T + [(None, None)],
                  method='highs', options=dict(primal_feasibility_tolerance=1e-10, dual_feasibility_tolerance=1e-10))
    assert res.status == 0
    b = np.maximum(-res.ineqlin.marginals, 0.0)
    return -res.fun, b / b.sum()


def colgen_np(model, pg, W, tau, nodes):
    """NumPy + HiGHS restatement of `bpi_lps` for `nodes`: J = [own row]; each round solves the restricted LP with HiGHS, prices with the
    oracle's backup at the LP's dual belief b* (the backup row there is the best column over every tuple), and stops on the same rules
    (m* > -tau not improvable, m* >= delta_J - tau optimal, 64 columns budget).  Returns {n: (status, eps of the last LP)}."""
    from oracle import pbvi_oracle as orc
    own = own_rows_np(model, pg, W, pg.gamma)
    reach, rto, rbar = np.asarray(model.reachable_states), model.reachable_transitional_observation_table, model.expected_rewards_table
    out = {}
    for n in nodes:
        cols = [own[n]]
        while True:
            eps, b = highs_lp(np.stack(cols), W[n])
            Y = orc.backup(reach, rto, rbar, pg.gamma, b[None, :], W)['alpha'][0]
            mstar = float(b @ (W[n] - Y))
            if mstar > -tau:
                out[n] = (1, eps)
            elif mstar >= -eps - tau:
                out[n] = (2, eps)
            elif len(cols) == 64:
                out[n] = (3, eps)
            else:
                cols.append(Y)
                continue
            break
    return out


def check_against_highs(model, pg, restate_nodes):
    W = pg.rows.cpu().numpy()
    gamma = pg.gamma
    sol, tau = solve_lps(pg)
    own = own_rows_np(model, pg, W, gamma)
    scale = max(1.0, float(np.abs(W).max()), float(np.abs(own).max()))
    tol = 1e-9 * scale
    eps_k = -sol['delta']
    for n in range(len(pg)):
        st, cols = sol['status'][n], sol['columns'][n]
        cols = cols[cols > -2]
        if st == 3 and len(cols) < 64:
            cols = cols[:-1]                                       # the pivot budget: the outputs are those of the LP before the last column
        rows = np.stack([own[n] if c == -1 else tuple_rows_np(model, W, gamma, sol['tuples'][c][None, :])[0] for c in cols])
        eps_J, _ = highs_lp(rows, W[n])
        assert abs(eps_k[n] - eps_J) <= tol, (n, st, eps_k[n], eps_J)           # delta_J is the LP optimum on the kernel's own columns
        m = sol['mstar'][n]
        assert (st == 1 and m > -tau) or (st == 2 and m >= sol['delta'][n] - tau) or st == 3, (n, st, m, sol['delta'][n])
    ref = colgen_np(model, pg, W, tau, restate_nodes)
    both = 0
    for n, (st_r, eps_r) in ref.items():
        st = sol['status'][n]
        if st == 1:
            assert eps_r <= 2 * tau + tol, (n, eps_r)                               # no column set improves it by more than tau
        if st == 2:
            assert eps_r <= eps_k[n] + tol, (n, eps_r, eps_k[n])                    # eps_k is the optimum over every tuple
        if st_r == 2:
            assert eps_k[n] <= eps_r + tol, (n, st, eps_k[n], eps_r)
            if st == 2:
                assert abs(eps_k[n] - eps_r) <= tol, (n, eps_k[n], eps_r)
                both += 1
        if st_r == 1:
            assert eps_k[n] <= 2 * tau + tol and st in (1, 2), (n, st, eps_k[n])
    return sol, both


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['grid4x3', 'hallway', 'tigergrid'])
def test_lp_equals_a_highs_column_generation_restatement(tag):
    model, gamma, B, pg = source_graph(tag, 'extracted')
    sol, _ = check_against_highs(model, pg, list(range(min(len(pg), 12))))
    assert sol['stats']['lps'] > len(pg)


def synthetic_model(seed=11, S=5, A=3, O=2, R=2):
    """A small random model (random reach, RTO rows summing to 1 over (o, r), rewards of both signs) in the layout of `fixture_model`."""
    from pomdp_pbvi_exploration_b200 import Model
    rng = np.random.default_rng(seed)
    model = Model.__new__(Model)
    model._device_handle = None
    model.is_on_gpu = True
    model.state_labels = [f's_{i}' for i in range(S)]
    model.state_count, model.states = S, np.arange(S)
    model.action_labels = [f'a_{i}' for i in range(A)]
    model.action_count, model.actions = A, np.arange(A)
    model.observation_labels = [f'o_{i}' for i in range(O)]
    model.observation_count, model.observations = O, np.arange(O)
    model.reachable_states, model.reachable_state_count = rng.integers(0, S, size=(S, A, R)).astype(np.int64), R
    model.reachable_probabilities = np.full((S, A, R), 1.0 / R)
    model.observation_table = None
    rto = rng.random((S, A, O, R)) ** 2
    model.reachable_transitional_observation_table = rto / rto.sum(axis=(2, 3), keepdims=True)
    model.expected_rewards_table = rng.normal(size=(S, A))
    model.start_probabilities = np.full(S, 1.0 / S)
    model.end_states, model.end_actions = [], []
    model._min_reward, model._max_reward = -3.0, 3.0
    model.transition_table = model.immediate_reward_table = model.immediate_reward_function = None
    model.rewards_are_probabilistic = False
    model.state_grid = np.arange(S).reshape(1, S)
    return model, 0.9


@pytest.mark.gpu
def test_lp_optimum_equals_highs_on_all_tuples_of_a_synthetic_model():
    import itertools
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = synthetic_model()
    rng = np.random.default_rng(2)
    N, A, O = 6, model.action_count, model.observation_count
    pg = PolicyGraph(model, rng.integers(0, A, N), rng.integers(0, N, (N, O)))
    pg.evaluate(gamma, eps=1e-9)
    W = pg.rows.cpu().numpy()
    tuples = [(a, *t) for a in range(A) for t in itertools.product(range(N), repeat=O)]
    Y = tuple_rows_np(model, W, gamma, tuples)
    sol, tau = solve_lps(pg)
    scale = max(1.0, float(np.abs(W).max()), float(np.abs(Y).max()))
    improvable = 0
    for n in range(N):
        eps = highs_eps(Y, W[n])
        st = sol['status'][n]
        assert st in (1, 2), (n, st)
        if st == 2:
            assert abs(-sol['delta'][n] - eps) <= 1e-9 * scale, (n, -sol['delta'][n], eps)
            improvable += eps > tau
        else:
            assert eps <= 2 * tau, (n, eps)
    assert improvable > 0
    check_solution(model, pg, sol, tau)
    check_against_highs(model, pg, list(range(N)))
    new, st = pg.bounded_improve(None, 1)
    assert st[0]['improved'] > 0 and st[0]['value_b0'] >= float(pg.value(model.start_probabilities)[0][0]) - st[0]['shift']
    check_iteration(model, gamma, None, pg, new)
