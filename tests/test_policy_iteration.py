"""
Policy iteration on finite-state controllers: the persistent evaluation loop (pbvi_controller_evaluate), the dominance of new node rows
over old ones (pbvi_first_dominating_row) and PolicyGraph.improve.  Checked against
  * k single pbvi_controller_sweep calls (bitwise rows and per-sweep changes, same k);
  * NumPy's all(Y_j >= X_i) with planted dominations, ties and a last-state violation;
  * the certificate W <= T_pi W in NumPy, monotone certified values at the improvement beliefs, the certified upper bound, the exact V*
    of tiger.95 and Monte Carlo roll-outs.
"""
import ctypes

import numpy as np
import pytest

from test_policy_graph import GOLDEN9, check_certificate, extracted
from test_upper_bound import MODELS, fib_of, fixture_model, tiger_exact_value


# ---- CPU ------------------------------------------------------------------------------------------------------------------------
def test_new_entry_points_reject_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    buf = (ctypes.c_double * 8)()
    p = ctypes.addressof(buf)
    sweeps = ctypes.c_int(0)
    BAD = _native.PBVI_ERR_BAD_ARG
    args = dict(d_in=p, n=2, actions=p, succ=p, tol=1e-6, max_sweeps=10, out=p + 8, sweeps=ctypes.byref(sweeps))

    def evaluate(**kw):
        a = dict(args, **kw)
        return lib.pbvi_controller_evaluate(kw.get('m'), a['d_in'], a['n'], 0.9, a['actions'], a['succ'], a['tol'], a['max_sweeps'],
                                            a['out'], None, a['sweeps'], None)
    assert evaluate() == BAD and b'handle is NULL' in lib.pbvi_last_error()
    for name in ('d_in', 'actions', 'succ', 'out', 'sweeps'):
        assert evaluate(**{name: None}) == BAD and b'NULL pointer' in lib.pbvi_last_error(), name
    for n in (0, -3):
        assert evaluate(n=n) == BAD and b'n >= 1' in lib.pbvi_last_error(), n
    for k in (0, -1):
        assert evaluate(max_sweeps=k) == BAD and b'max_sweeps >= 1' in lib.pbvi_last_error(), k
    assert evaluate(tol=float('nan')) == BAD and b'NaN' in lib.pbvi_last_error()

    def dominating(m=None, d_new=p, n_new=3, d_old=p, n_old=2, first=p):
        return lib.pbvi_first_dominating_row(m, d_new, n_new, d_old, n_old, first, None)
    assert dominating() == BAD and b'handle is NULL' in lib.pbvi_last_error()
    for kw in (dict(n_new=-1), dict(n_old=-1)):
        assert dominating(**kw) == BAD and b'non-negative' in lib.pbvi_last_error(), kw
    for name in ('d_new', 'd_old', 'first'):
        assert dominating(**{name: None}) == BAD and b'NULL pointer' in lib.pbvi_last_error(), name
    assert dominating(n_new=65535 * 32 + 1) == BAD and b'grid.y' in lib.pbvi_last_error()


def test_reachable_subgraph_drops_unreachable_nodes_and_renumbers():
    from pomdp_pbvi_exploration_b200.policy_graph import reachable_subgraph
    # 0 -> {0, 3}, 1 -> {1, 1} (unreachable), 2 -> {3, 4}, 3 -> {3, 0}, 4 -> {4, 4} (only through 2), 5 -> {2, 2} (unreachable)
    act = np.array([0, 1, 2, 0, 1, 2])
    succ = np.array([[0, 3], [1, 1], [3, 4], [3, 0], [4, 4], [2, 2]])
    keep, a, s = reachable_subgraph(act, succ, np.array([3, 3]))
    assert keep.tolist() == [0, 3] and a.tolist() == [0, 0] and s.tolist() == [[0, 1], [1, 0]]
    keep, a, s = reachable_subgraph(act, succ, np.array([2]))
    assert keep.tolist() == [0, 2, 3, 4] and a.tolist() == [0, 2, 0, 1]
    assert s.tolist() == [[0, 2], [2, 3], [2, 0], [3, 3]]
    keep, _, s = reachable_subgraph(act, succ, np.array([5, 1]))
    assert keep.tolist() == [0, 1, 2, 3, 4, 5] and np.array_equal(s, succ)
    # an impossible observation leads to node 0 in extracted and improved graphs: node 0 is kept through that entry alone
    keep, a, s = reachable_subgraph([1, 0, 2], [[0, 0], [2, 0], [2, 2]], [1])
    assert keep.tolist() == [0, 1, 2] and s.tolist() == [[0, 0], [2, 0], [2, 2]]
    keep, a, s = reachable_subgraph([1, 0, 2], [[0, 0], [2, 2], [2, 2]], [1])
    assert keep.tolist() == [1, 2] and a.tolist() == [0, 2] and s.tolist() == [[1, 1], [1, 1]]


# ---- GPU: the persistent evaluation loop -----------------------------------------------------------------------------------------
def host_loop(dev, W, gamma, act, succ, tol, max_sweeps):
    """PolicyGraph.evaluate's former iteration: one pbvi_controller_sweep and one read-back per sweep."""
    changes = []
    for _ in range(max_sweeps):
        W, st = dev.controller_sweep(W, gamma, act, succ, want_stats=True)
        changes.append(float(st[2]))
        if not changes[-1] >= tol:
            break
    return W, changes


def same_changes(a, b):
    return len(a) == len(b) and all((x == y) or (x != x and y != y) for x, y in zip(a, b))


def check_loop(dev, W, gamma, act, succ, tol, max_sweeps, label):
    want, want_ch = host_loop(dev, W, gamma, act, succ, tol, max_sweeps)
    got, got_ch, k = dev.controller_evaluate(W, gamma, act, succ, tol, max_sweeps)
    got_ch = got_ch.cpu().numpy().tolist()
    assert k == len(want_ch) and same_changes(got_ch, want_ch), (label, k, got_ch[-3:], want_ch[-3:])
    assert got.cpu().numpy().tobytes() == want.cpu().numpy().tobytes(), label
    return k, got_ch


@pytest.mark.gpu
@pytest.mark.parametrize('tag', MODELS)
def test_evaluate_loop_is_the_host_loop(tag):
    import torch
    model, gamma = fixture_model(tag)
    dev = model.device
    A, O, S = model.action_count, model.observation_count, model.state_count
    rbar = np.asarray(model.expected_rewards_table, dtype=np.float64)
    rng = np.random.default_rng(5)
    for N in (1, 9, 200):
        act = rng.integers(0, A, N).astype(np.int32)
        succ = rng.integers(0, N, (N, O)).astype(np.int32)
        W = torch.as_tensor(rbar.T[act], device='cuda').contiguous()
        assert check_loop(dev, W, gamma, act, succ, 1e300, 50, (tag, N, 'first'))[0] == 1
        for k in (6, 7):                                                 # the last iterate in the output buffer and in the arena
            assert check_loop(dev, W, gamma, act, succ, 0.0, k, (tag, N, k))[0] == k
        tol = 1e-3 * max(1.0, float(np.abs(rbar).max()))
        k, ch = check_loop(dev, W, gamma, act, succ, tol, 20000, (tag, N, 'tol'))
        assert ch[-1] < tol or k == 20000
    # a NaN entry: the first sweep reports NaN and the loop stops there
    W = torch.as_tensor(rbar.T[[0, A - 1]], device='cuda').contiguous()
    W[1, S - 1] = float('nan')
    k, ch = check_loop(dev, W, gamma, np.array([0, A - 1], dtype=np.int32), np.zeros((2, O), dtype=np.int32), 1e-6, 100, (tag, 'nan'))
    assert k == 1 and ch[0] != ch[0]


@pytest.mark.gpu
def test_evaluate_loop_with_thousands_of_nodes_on_olfactory():
    import torch
    model, gamma = fixture_model('olfactory_wrap')
    dev = model.device
    A, O = model.action_count, model.observation_count
    rng = np.random.default_rng(9)
    N = 3000                                                             # 3000 x 87 items: many per resident block
    act = rng.integers(0, A, N).astype(np.int32)
    succ = rng.integers(0, N, (N, O)).astype(np.int32)
    W = torch.as_tensor(np.asarray(model.expected_rewards_table, dtype=np.float64).T[act], device='cuda').contiguous()
    assert check_loop(dev, W, gamma, act, succ, 0.0, 5, 'olfactory 3000')[0] == 5


@pytest.mark.gpu
def test_evaluate_loop_rejects_oversized_grids():
    from pomdp_pbvi_exploration_b200 import _native
    model, _ = fixture_model('olfactory_wrap')                          # S = 22021: 87 items per node
    dev = model.device
    lib = _native.load_library()
    buf = (ctypes.c_double * 8)()
    p = ctypes.addressof(buf)
    k = ctypes.c_int(0)
    n = 0x7fffffff // 87 + 1
    assert lib.pbvi_controller_evaluate(dev._h, p, n, 0.9, p, p, 1e-6, 10, p + 8, None, ctypes.byref(k), None) == _native.PBVI_ERR_BAD_ARG
    assert b'too many controller nodes' in lib.pbvi_last_error()
    assert lib.pbvi_controller_evaluate(dev._h, p, 2, 0.9, p, p, 1e-6, 10, p, None, ctypes.byref(k), None) == _native.PBVI_ERR_BAD_ARG


# ---- GPU: dominance ----------------------------------------------------------------------------------------------------------------
def first_dominating_np(Y, X):
    out = np.full(len(X), -1, dtype=np.int64)
    for i in range(len(X)):
        hit = np.flatnonzero((Y >= X[i]).all(axis=1))
        if len(hit):
            out[i] = hit[0]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('tag,n_old,n_new', [('tiger', 40, 33), ('hallway', 3000, 2500), ('synth300', 200, 97), ('olfactory_wrap', 70, 45)])
def test_first_dominating_row_matches_numpy(tag, n_old, n_new):
    import torch
    model, _ = fixture_model(tag)
    dev = model.device
    S = model.state_count
    rng = np.random.default_rng(3)
    X = rng.normal(size=(n_old, S))
    Y = rng.normal(size=(n_new, S))
    planted = rng.choice(n_old, n_old // 3, replace=False)
    for q, i in enumerate(planted):
        j = int(rng.integers(0, n_new))
        kind = q % 4
        if kind == 0:
            Y[j] = X[i] + np.abs(rng.normal(size=S)) * (rng.random(S) < 0.5)      # ties on about half the states
        elif kind == 1:
            Y[j] = X[i]                                                           # equal rows dominate
        elif kind == 2:
            Y[j] = X[i] + 1.0
            Y[j, S - 1] = np.nextafter(X[i, S - 1], -np.inf)                      # one violation, at the last state
        else:
            Y[j] = X[i] + 0.5
            if S > 1:
                Y[j, S // 2] = np.nan                                             # NaN never dominates
    X[0] = -1e300                                                                 # dominated by every row without a NaN
    got = dev.first_dominating_row(torch.as_tensor(Y, device='cuda'), torch.as_tensor(X, device='cuda')).cpu().numpy()
    assert np.array_equal(got, first_dominating_np(Y, X)), (tag, np.flatnonzero(got != first_dominating_np(Y, X))[:5])
    assert got[0] >= 0 and (got >= 0).sum() >= 2
    empty = dev.first_dominating_row(torch.zeros((0, S), device='cuda', dtype=torch.float64), torch.as_tensor(X, device='cuda'))
    assert empty.cpu().numpy().tolist() == [-1] * n_old


# ---- GPU: improve ----------------------------------------------------------------------------------------------------------------
def check_graph(model, pg, B):
    from pomdp_pbvi_exploration_b200.policy_graph import reachable_subgraph
    N = len(pg)
    assert pg.successors.min() >= 0 and pg.successors.max() < N and pg.rows.shape == (N, model.state_count)
    roots = pg.value(np.concatenate([model.start_probabilities[None, :], B]))[1].cpu().numpy()
    assert len(reachable_subgraph(pg.actions, pg.successors, roots)[0]) == N


def belief_values(pg, model, B):
    return pg.value(np.concatenate([model.start_probabilities[None, :], B]))[0].cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize('tag', GOLDEN9)
def test_improve_raises_a_certified_bound(tag):
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma, _, B, pg, _ = extracted(tag)
    ub = UpperBound(model, fib_of(tag)[0], gamma)
    upper = ub.evaluate(np.concatenate([model.start_probabilities[None, :], B])).cpu().numpy()
    prev = belief_values(pg, model, B)
    cur = pg
    for it in range(3):
        nxt, stats = cur.improve(B, 1)
        assert len(stats) == 1
        st = stats[0]
        assert st['nodes_before'] == len(cur) and st['nodes_after'] == len(nxt)
        assert st['nodes_after'] == st['nodes_before'] + st['appended'] - st['pruned']
        val = belief_values(nxt, model, B)
        slack = st['shift'] + 1e-9 * float(np.abs(cur.rows.cpu().numpy()).max())
        assert np.all(val >= prev - slack), (tag, it, float(np.min(val - prev)), slack)
        assert np.all(val <= upper + 1e-9 * np.maximum(1.0, np.abs(upper))), (tag, it, float(np.max(val - upper)))
        assert st['value_b0'] == val[0]
        check_certificate(model, gamma, nxt)
        check_graph(model, nxt, B)
        if st['appended'] == 0 and st['overwritten'] == 0:
            assert nxt is cur
            break
        prev, cur = val, nxt


def tiger_setup():
    import torch
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model('tiger')
    grid = np.linspace(0.0, 1.0, 101)
    B = torch.as_tensor(np.stack([1 - grid, grid], axis=1), device='cuda')
    pg = PolicyGraph.blind(model)
    pg.evaluate(gamma)
    return model, gamma, B, pg


@pytest.mark.gpu
def test_improve_reaches_tiger_optimum_and_a_fixed_point():
    model, gamma, B, pg = tiger_setup()
    vstar = float(tiger_exact_value(model, gamma, np.array([model.start_probabilities[1]]))[0])
    pg, stats = pg.improve(B, iterations=100, eps=1e-9)
    got = float(pg.value(model.start_probabilities)[0][0])
    assert got <= vstar + 1e-9, (got, vstar)
    assert abs(got - vstar) <= 1e-3 * abs(vstar), (got, vstar, len(pg), len(stats))
    assert all(b['value_b0'] >= a['value_b0'] - b['shift'] - 1e-9 for a, b in zip(stats, stats[1:]))
    last = stats[-1]
    assert last['appended'] == 0 and last['overwritten'] == 0, last                    # the fixed point at B was reached
    again, st = pg.improve(B, iterations=1, eps=1e-9)
    assert again is pg and len(st) == 1 and st[0]['appended'] == 0 and st[0]['overwritten'] == 0


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['hallway', 'olfactory_fsvi'])
def test_improve_is_deterministic(tag):
    model, gamma, _, B, pg, _ = extracted(tag)
    g1, s1 = pg.improve(B, 2)
    g2, s2 = pg.improve(B, 2)
    assert np.array_equal(g1.actions, g2.actions) and np.array_equal(g1.successors, g2.successors)
    assert g1.rows.cpu().numpy().tobytes() == g2.rows.cpu().numpy().tobytes()
    assert [s['value_b0'] for s in s1] == [s['value_b0'] for s in s2]


@pytest.mark.gpu
def test_improved_controller_agrees_with_monte_carlo():
    model, gamma, _, B, pg, _ = extracted('tiger')
    pg, stats = pg.improve(B, 3)
    rbar_max = float(np.max(np.abs(model.expected_rewards_table)))
    H = int(np.ceil(np.log(1e-6 * (1 - gamma) / rbar_max) / np.log(gamma))) + 1
    ret = pg.simulate(4000, H, seed=3)
    mean, se = float(ret.mean()), float(ret.std(ddof=1) / np.sqrt(len(ret)))
    v0 = float(pg.value(model.start_probabilities)[0][0])
    shift = max([s['shift'] for s in stats] + [0.0])
    assert abs(mean - v0) <= 5 * se + shift, (mean, se, v0, shift)
