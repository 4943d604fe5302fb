"""
IncrementalPruning_Solver: exact value iteration by incremental pruning, and the three entry points under it (pbvi_ip_project,
pbvi_ip_cross_sum, pbvi_ip_residual_lp).

CPU: the symbols and their binding, argument checks without a device, the tuple bookkeeping and the rounding allowance, the refusal of
non-finite start rows.  GPU: the fold of projections and cross sums is bitwise backup_assemble; one exact backup equals brute force over
every tuple; H V agrees with the point-based backup; the residual LP against FP64 and HiGHS; tiger.95 against its exact value; soundness
of the certificate against the package's other bounds; finite horizons against a NumPy expectimax; determinism.
"""
import ctypes
import itertools

import numpy as np
import pytest

from conftest import load_golden
from test_upper_bound import fib_of, fixture_model, tiger_exact_value

GOLDEN = ['tiger', 'hanks', 'network', 'grid4x4', 'grid4x4_noloop', 'cheese', 'grid4x3', 'hallway']
O2 = ['tiger', 'hanks', 'network', 'grid4x4', 'grid4x4_noloop']
SMALL = ['tiger', 'hanks', 'network', 'grid4x4', 'grid4x4_noloop', 'cheese', 'grid4x3']


# ---- CPU -----------------------------------------------------------------------------------------------------------------------------
def test_entry_points_are_declared_and_bound():
    from test_cabi_and_host import declared_symbols
    from pomdp_pbvi_exploration_b200 import _native
    for name in ('pbvi_ip_project', 'pbvi_ip_cross_sum', 'pbvi_ip_residual_lp'):
        assert name in declared_symbols() and name in _native.SIGNATURES
    assert len(declared_symbols()) == 65


def test_entry_points_reject_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    lib = _native.load_library()
    bad = _native.PBVI_ERR_BAD_ARG
    assert lib.pbvi_ip_project(None, None, 1, 0.95, 0, None, None) == bad
    assert b'NULL' in lib.pbvi_last_error()
    assert lib.pbvi_ip_cross_sum(None, None, 1, None, 1, 0, None, None) == bad
    assert lib.pbvi_ip_residual_lp(None, None, 1, None, 1, 1e-9, None, None, None, None, None, None, None) == bad
    st = (ctypes.c_int64 * 4)(7, 7, 7, 7)
    assert lib.pbvi_ip_residual_lp(None, None, 1, None, 1, 1e-9, None, None, None, None, None, st, None) == bad


def test_tuple_product_is_i_major():
    from pomdp_pbvi_exploration_b200.incremental_pruning import tuple_product
    x = np.array([[4, 7], [5, 8], [6, 9]])
    g = np.array([2, 0])
    t = tuple_product(x, g)
    want = [[4, 7, 2], [4, 7, 0], [5, 8, 2], [5, 8, 0], [6, 9, 2], [6, 9, 0]]
    assert t.tolist() == want
    t1 = tuple_product(np.array([[3], [1]]), np.array([5]))
    assert t1.tolist() == [[3, 5], [1, 5]]


def test_rounding_allowance_formula():
    from pomdp_pbvi_exploration_b200.incremental_pruning import rounding_allowance
    rho_rows, rho_u = rounding_allowance(O=2, R=3, rbar_max=10.0, gamma=0.5, rto_mass=1.0, alpha_max=4.0, new_max=6.0)
    assert rho_rows == (2 * 3 + 2) * 2.0 ** -52 * (10.0 + 0.5 * 1.0 * 4.0)
    assert rho_u == 66 * 2.0 ** -52 * (6.0 + 4.0)
    # larger inputs never give a smaller allowance
    assert rounding_allowance(3, 3, 10.0, 0.5, 1.0, 4.0, 6.0)[0] > rho_rows


def test_solver_refuses_non_finite_rows():
    import torch
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver, ValueFunction
    model, gamma = fixture_model('tiger')
    vf = ValueFunction.__new__(ValueFunction)
    vf._array = torch.tensor([[0.0, float('nan')]], dtype=torch.float64)
    vf._actions = np.zeros(1, dtype=np.int64)
    with pytest.raises(ValueError, match='finite'):
        IncrementalPruning_Solver(gamma).solve(model, horizon=1, initial_value_function=vf)
    vf._array = torch.tensor([[0.0, float('inf')]], dtype=torch.float64)
    with pytest.raises(ValueError, match='finite'):
        IncrementalPruning_Solver(gamma).solve(model, horizon=1, initial_value_function=vf)
    with pytest.raises(ValueError):
        IncrementalPruning_Solver(1.0)


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------------------
def golden_device(tag):
    from pomdp_pbvi_exploration_b200._native import DeviceModel
    m = load_golden('model_' + tag)
    return DeviceModel(m['reach'].astype(np.int64), m.get('probs'), m['rto'], m['rbar']), float(m['gamma']), m


def synthetic_device(O=1, seed=0):
    """A random model with O observations, R = 2, and -0.0 / +0.0 entries of Rbar next to zero RTO terms."""
    from pomdp_pbvi_exploration_b200._native import DeviceModel
    rng = np.random.default_rng(seed)
    S, A, R = 9, 3, 2
    reach = rng.integers(0, S, (S, A, R)).astype(np.int64)
    rto = rng.random((S, A, O, R))
    rto[rng.random(rto.shape) < 0.4] = 0.0
    rto /= np.maximum(rto.sum(axis=(2, 3), keepdims=True), 1e-300)
    rbar = rng.normal(size=(S, A))
    rbar[::2, 0] = -0.0
    rbar[1::3, 1] = 0.0
    return DeviceModel(reach, None, rto, rbar), 0.9


def fold_rows(dev, V, gamma, acts, vsel):
    """Rbar + ((G_0 + G_1) + ...) of every tuple from ip_project and ip_cross_sum, one tuple at a time."""
    import torch
    out = []
    for a, v in zip(acts, vsel):
        G = dev.ip_project(V, gamma, int(a))
        O = G.shape[0]
        if O == 1:
            out.append(dev.ip_cross_sum(None, G[0, v[0]][None], int(a)))
            continue
        x = G[0, v[0]][None]
        for o in range(1, O):
            x = dev.ip_cross_sum(x, G[o, v[o]][None], int(a) if o == O - 1 else -1)
        out.append(x)
    return torch.cat(out)


def check_fold_equals_assemble(dev, gamma, V, n, seed):
    import torch
    rng = np.random.default_rng(seed)
    acts = rng.integers(0, dev.A, n).astype(np.int32)
    vsel = rng.integers(0, V.shape[0], (n, dev.O)).astype(np.int32)
    want = dev.backup_assemble(V, gamma, acts, vsel)
    got = fold_rows(dev, V, gamma, acts, vsel)
    assert torch.equal(got.view(torch.int64), want.view(torch.int64))
    # a batched cross sum is every pair of the two sets, i-major, each one IEEE addition
    if dev.O >= 2:
        G = dev.ip_project(V, gamma, 0)
        i, j = np.divmod(np.arange(V.shape[0] ** 2), V.shape[0])
        ref = G[0][torch.as_tensor(i, device=V.device)] + G[1][torch.as_tensor(j, device=V.device)]
        assert torch.equal(dev.ip_cross_sum(G[0], G[1], -1).view(torch.int64), ref.view(torch.int64))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', GOLDEN + ['olfactory_wrap'])
def test_projection_and_cross_sum_are_bitwise_assemble(tag):
    import torch
    dev, gamma, m = golden_device(tag)
    rng = np.random.default_rng(1)
    nV = 3 if tag == 'olfactory_wrap' else 6
    V = torch.as_tensor(rng.normal(size=(nV, dev.S)) * 10.0, device=dev.device)
    check_fold_equals_assemble(dev, gamma, V, 40 if tag != 'olfactory_wrap' else 6, seed=2)


@pytest.mark.gpu
@pytest.mark.parametrize('O', [1, 3])
def test_projection_and_cross_sum_on_signed_zero_rewards(O):
    import torch
    dev, gamma = synthetic_device(O=O)
    rng = np.random.default_rng(3)
    V = torch.as_tensor(rng.normal(size=(5, dev.S)), device=dev.device)
    V[0] = 0.0
    V[1] = -0.0
    check_fold_equals_assemble(dev, gamma, V, 64, seed=4)


@pytest.mark.gpu
def test_projection_rejects_bad_arguments():
    import torch
    dev, gamma, _ = golden_device('tiger')
    V = torch.zeros((2, 2), dtype=torch.float64, device=dev.device)
    with pytest.raises(ValueError):
        dev.ip_project(V, gamma, dev.A)
    with pytest.raises(ValueError, match='finite'):
        dev.ip_project(torch.full((1, 2), float('nan'), dtype=torch.float64, device=dev.device), gamma, 0)
    with pytest.raises(ValueError):
        dev.ip_cross_sum(V, V, dev.A)
    with pytest.raises(ValueError):
        dev.ip_residual_lp(V, V[:0], 1e-9)
    with pytest.raises(ValueError):
        dev.ip_residual_lp(V, V, -1.0)
    lib = dev._lib
    bad = -1
    assert lib.pbvi_ip_project(dev._h, V.data_ptr(), -1, gamma, 0, V.data_ptr(), None) == bad
    assert lib.pbvi_ip_project(dev._h, None, 2, gamma, 0, V.data_ptr(), None) == bad
    assert lib.pbvi_ip_project(dev._h, V.data_ptr(), 2, float('inf'), 0, V.data_ptr(), None) == bad
    assert lib.pbvi_ip_cross_sum(dev._h, V.data_ptr(), -1, V.data_ptr(), 2, -1, V.data_ptr(), None) == bad
    assert lib.pbvi_ip_cross_sum(dev._h, V.data_ptr(), 2, V.data_ptr(), -2, -1, V.data_ptr(), None) == bad
    assert lib.pbvi_ip_cross_sum(dev._h, V.data_ptr(), 2, None, 2, -1, V.data_ptr(), None) == bad
    p = V.data_ptr()
    assert lib.pbvi_ip_residual_lp(dev._h, p, -1, p, 2, 1e-9, p, p, p, p, p, None, None) == bad
    assert lib.pbvi_ip_residual_lp(dev._h, p, 2, p, 0, 1e-9, p, p, p, p, p, None, None) == bad
    assert lib.pbvi_ip_residual_lp(dev._h, p, 2, p, 2, 1e-9, None, p, p, p, p, None, None) == bad
    assert lib.pbvi_ip_residual_lp(dev._h, p, 2, p, 2, float('nan'), p, p, p, p, p, None, None) == bad


def random_beliefs(S, n, seed):
    rng = np.random.default_rng(seed)
    B = rng.random((n, S)) ** 3
    B /= B.sum(axis=1, keepdims=True)
    return np.concatenate([np.eye(S), B])


def highs_margin(y, others):
    """max_b min_j b . (y - x_j) over the simplex (HiGHS)."""
    from scipy.optimize import linprog
    S = y.shape[0]
    D = y[None, :] - others                                         # [k, S]
    c = np.zeros(S + 1)
    c[-1] = -1.0                                                    # maximise delta
    A_ub = np.concatenate([-D, np.ones((D.shape[0], 1))], axis=1)   # delta - b . d_j <= 0
    A_eq = np.concatenate([np.ones((1, S)), np.zeros((1, 1))], axis=1)
    r = linprog(c, A_ub=A_ub, b_ub=np.zeros(D.shape[0]), A_eq=A_eq, b_eq=[1.0], bounds=[(0, None)] * S + [(None, None)], method='highs')
    assert r.status == 0
    return -r.fun


def one_epoch(tag, nV, seed):
    import torch
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver
    model, gamma = fixture_model(tag)
    rng = np.random.default_rng(seed)
    X = torch.as_tensor(rng.normal(size=(nV, model.state_count)) * 5.0, device=model.device.device)
    solver = IncrementalPruning_Solver(gamma)
    Y, tuples, acc = solver._epoch(model, X)
    return model, gamma, solver, X, Y, tuples, acc


@pytest.mark.gpu
@pytest.mark.parametrize('tag', O2)
def test_one_exact_backup_equals_brute_force(tag):
    import torch
    model, gamma, solver, X, Y, tuples, acc = one_epoch(tag, 4, seed=5)
    dev = model.device
    A, O, S = model.action_count, model.observation_count, model.state_count
    # every row is bitwise the assemble row of its recorded tuple
    again = dev.backup_assemble(X, gamma, tuples[:, 0].astype(np.int32), tuples[:, 1:].astype(np.int32))
    assert torch.equal(again.view(torch.int64), Y.view(torch.int64))
    # all A * |V|^O tuples
    allt = np.array([(a, *v) for a in range(A) for v in itertools.product(range(X.shape[0]), repeat=O)], dtype=np.int32)
    full = dev.backup_assemble(X, gamma, allt[:, 0], allt[:, 1:])
    B = random_beliefs(S, 10000, seed=6)
    got = dev.max_values(B, Y)[0].cpu().numpy()
    want = dev.max_values(B, full)[0].cpu().numpy()
    # a pointwise-dominated row has a dot product no larger (rounding is monotone, the order is the same) and an LP-pruned row lies more
    # than 1e-9 * scale below a kept one: the maxima agree bitwise
    assert np.array_equal(got, want), float(np.max(np.abs(got - want)))
    # every kept row has an LP witness (margin > -2 tau against the other kept rows), except the rows the last prune left undecided
    Yn = Y.cpu().numpy()
    tau = 1e-9 * max(1.0, float(np.max(np.abs(Yn))))
    low = [i for i in range(Yn.shape[0]) if Yn.shape[0] > 1 and highs_margin(Yn[i], np.delete(Yn, i, axis=0)) <= -2 * tau]
    assert len(low) <= acc['undecided'], (low, acc['undecided'])


@pytest.mark.gpu
@pytest.mark.parametrize('tag', SMALL)
def test_exact_backup_agrees_with_the_point_based_backup(tag):
    model, gamma, solver, X, Y, tuples, acc = one_epoch(tag, 3, seed=7)
    dev = model.device
    B = random_beliefs(model.state_count, 1000, seed=8)
    pb_rows = dev.backup(B, X, gamma)[0]
    exact = dev.max_values(B, Y)[0].cpu().numpy()
    point = dev.max_values(B, pb_rows)[0].cpu().numpy()
    scale = max(1.0, float(Y.abs().max()))
    # the point-based backup picks, at each belief, the best tuple: H V there, up to the rounding of the dot products
    assert np.max(np.abs(exact - point)) <= 1e-12 * scale
    assert np.all(exact >= point - 1e-12 * scale)


def residual_np_checks(Y, X, res, tau):
    u, m = res['u'].cpu().numpy(), res['mstar'].cpu().numpy()
    bstar, idx, w = res['bstar'].cpu().numpy(), res['cert_idx'].cpu().numpy(), res['cert_w'].cpu().numpy()
    scale = max(1.0, np.max(np.abs(Y)), np.max(np.abs(X)))
    over = 0
    for i in range(Y.shape[0]):
        k = int(np.sum(idx[i] >= 0))
        assert k >= 1 and np.all(idx[i, :k] >= 0) and np.all(idx[i, :k] < X.shape[0]) and np.all(idx[i, k:] == -1)
        assert np.all(w[i] >= 0.0) and abs(w[i].sum() - 1.0) < 1e-12 and np.all(w[i, k:] == 0.0)
        comb = w[i, :k] @ X[idx[i, :k]]
        assert np.all(comb >= Y[i] - u[i] - 1e-13 * scale)                     # the certificate holds in FP64
        assert m[i] <= u[i] + 1e-13 * scale
        assert np.all(bstar[i] >= 0.0) and abs(bstar[i].sum() - 1.0) < 1e-12
        assert abs(m[i] - (bstar[i] @ Y[i] - np.max(X @ bstar[i]))) <= 1e-12 * scale
        over += int(u[i] - m[i] > tau)
    assert over <= res['stats']['budget_rows']
    return u, m


@pytest.mark.gpu
@pytest.mark.parametrize('tag', O2 + ['cheese'])
def test_residual_lp_bounds(tag):
    model, gamma, solver, X, Y, tuples, acc = one_epoch(tag, 4, seed=9)
    dev = model.device
    tau = 1e-10 * max(1.0, float(Y.abs().max()))
    res = dev.ip_residual_lp(Y, X, tau)
    Yn, Xn = Y.cpu().numpy(), X.cpu().numpy()
    u, m = residual_np_checks(Yn, Xn, res, tau)
    if model.observation_count == 2:
        scale = max(1.0, np.max(np.abs(Yn)))
        for i in range(Yn.shape[0]):
            d = highs_margin(Yn[i], Xn)
            assert m[i] - 1e-9 * scale <= d <= u[i] + 1e-9 * scale, (i, m[i], d, u[i])


@pytest.mark.gpu
def test_residual_lp_of_a_set_against_itself_is_zero():
    model, gamma, solver, X, Y, tuples, acc = one_epoch('hanks', 4, seed=10)
    res = model.device.ip_residual_lp(Y, Y, 0.0)
    u = res['u'].cpu().numpy()
    assert np.all(u == 0.0)                       # lambda = e_i: y_i - y_i is exactly 0


@pytest.mark.gpu
def test_tiger_exact_value_lies_inside_the_certificate():
    """tiger.95 from the default start: V <= V* <= V + shift on a 1001-point grid.  Its near-tied rows (margins within the LP prune's
    tau) multiply from epoch to epoch, so the solve ends at the candidate limit or the time limit, not at a small shift."""
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver
    model, gamma = fixture_model('tiger')
    V, hist = IncrementalPruning_Solver(gamma, max_candidates=500_000).solve(model, horizon=2000, target=1e-6, time_limit=30)
    assert hist.shift is not None and len(hist.epochs) >= 5
    grid = np.linspace(0.0, 1.0, 1001)
    vstar = tiger_exact_value(model, gamma, grid)
    B = np.stack([1 - grid, grid], axis=1)
    v = model.device.max_values(B, V.alpha_vector_array)[0].cpu().numpy()
    assert np.all(v <= vstar + 1e-9), float(np.max(v - vstar))
    assert np.all(vstar <= v + hist.shift + 1e-9), float(np.max(vstar - v - hist.shift))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['hanks', 'network', 'grid4x4_noloop', 'cheese'])
def test_solve_reaches_a_small_shift(tag):
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver
    model, gamma = fixture_model(tag)
    V, hist = IncrementalPruning_Solver(gamma).solve(model, horizon=5000, target=1e-6, time_limit=60)
    assert hist.stopped == 'target' and hist.shift <= 1e-6
    shifts = [ep['shift'] for ep in hist.epochs]
    assert shifts[-1] == hist.shift and len(V) == hist.epochs[-1]['rows']


_solves = {}


def short_solve(tag):
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver
    if tag not in _solves:
        model, gamma = fixture_model(tag)
        solver = IncrementalPruning_Solver(gamma)
        V, hist = solver.solve(model, horizon=200, time_limit=4.0)
        _solves[tag] = (model, gamma, V, hist)
    return _solves[tag]


@pytest.mark.gpu
@pytest.mark.parametrize('tag', SMALL)
def test_certificate_is_sound_against_the_other_bounds(tag):
    from pomdp_pbvi_exploration_b200 import GapSolver, PolicyGraph, UpperBound
    model, gamma, V, hist = short_solve(tag)
    assert hist.shift is not None and len(hist.epochs) >= 1
    S = model.state_count
    B = np.concatenate([model.start_probabilities[None, :], random_beliefs(S, 1000, seed=11)])
    dev = model.device
    rows = V.alpha_vector_array
    v = dev.max_values(B, rows)[0].cpu().numpy()
    scale = max(1.0, float(rows.abs().max()))
    slack = 1e-9 * scale
    pg, _ = PolicyGraph.from_value_function(model, V)
    pg.evaluate(gamma, eps=1e-9)
    low = pg.value(B)[0].cpu().numpy()
    assert np.all(v + hist.shift >= low - slack), float(np.min(v + hist.shift - low))
    gpg, _, _ = GapSolver(gamma, 0.01, trials=4, max_depth=10, seed=0).solve(model, max_rounds=2)
    glow = gpg.value(B)[0].cpu().numpy()
    assert np.all(v + hist.shift >= glow - slack), float(np.min(v + hist.shift - glow))
    fib, _ = fib_of(tag)
    assert np.all(v <= dev.max_values(B, fib.alpha_vector_array)[0].cpu().numpy() + slack)
    ub = UpperBound(model, fib, gamma)
    ub.improve(B[:64])
    assert np.all(v <= ub.evaluate(B).cpu().numpy() + slack)


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'hanks', 'network'])
def test_value_grows_epoch_by_epoch_from_the_default_start(tag):
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver
    model, gamma = fixture_model(tag)
    B = np.concatenate([model.start_probabilities[None, :], random_beliefs(model.state_count, 1000, seed=12)])
    solver = IncrementalPruning_Solver(gamma)
    V, hist = solver.solve(model, horizon=1)
    prev = model.device.max_values(B, hist.previous)[0].cpu().numpy()
    for _ in range(6):
        cur = model.device.max_values(B, V.alpha_vector_array)[0].cpu().numpy()
        scale = max(1.0, float(np.max(np.abs(cur))))
        assert np.all(cur >= prev - 1e-12 * scale), float(np.min(cur - prev))
        prev = cur
        V, hist = solver.solve(model, horizon=1, initial_value_function=V)


def expectimax_np(rto, reach, rbar, gamma, B, H):
    """max_a [b . Rbar_a + gamma * sum_o V_{H-1}(tau(b, a, o))] with unnormalised successors (V_k is positively homogeneous)."""
    if H == 0:
        return np.zeros(B.shape[0])
    S, A, O, R = rto.shape
    best = np.full(B.shape[0], -np.inf)
    for a in range(A):
        val = B @ rbar[:, a]
        for o in range(O):
            nxt = np.zeros_like(B)
            for r in range(R):
                np.add.at(nxt.T, reach[:, a, r], (B * rto[:, a, o, r][None, :]).T)
            val = val + gamma * expectimax_np(rto, reach, rbar, gamma, nxt, H - 1)
        best = np.maximum(best, val)
    return best


@pytest.mark.gpu
@pytest.mark.parametrize('tag,H', [('tiger', 1), ('tiger', 3), ('tiger', 5), ('hanks', 2), ('hanks', 3)])
def test_finite_horizon_equals_expectimax(tag, H):
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver, ValueFunction
    model, gamma = fixture_model(tag)
    zero = ValueFunction(model, np.zeros((1, model.state_count)), [0])
    V, hist = IncrementalPruning_Solver(gamma).solve(model, horizon=H, initial_value_function=zero)
    assert hist.stopped == 'horizon' and len(hist.epochs) == H
    B = random_beliefs(model.state_count, 60, seed=13)
    got = model.device.max_values(B, V.alpha_vector_array)[0].cpu().numpy()
    m = load_golden('model_' + tag)
    want = expectimax_np(m['rto'], m['reach'].astype(np.int64), m['rbar'], gamma, B, H)
    assert np.max(np.abs(got - want)) <= 1e-12 * max(1.0, np.max(np.abs(want)))


@pytest.mark.gpu
def test_solves_are_bitwise_repeatable():
    import torch
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver
    model, gamma = fixture_model('hanks')
    runs = [IncrementalPruning_Solver(gamma).solve(model, horizon=6) for _ in range(2)]
    (V1, h1), (V2, h2) = runs
    assert torch.equal(V1.alpha_vector_array.view(torch.int64), V2.alpha_vector_array.view(torch.int64))
    assert np.array_equal(V1.actions, V2.actions) and np.array_equal(h1.tuples, h2.tuples)
    assert h1.comparable() == h2.comparable() and h1.stopped == h2.stopped == 'horizon'


@pytest.mark.gpu
def test_candidate_limit_returns_the_last_completed_epoch():
    from pomdp_pbvi_exploration_b200 import IncrementalPruning_Solver
    model, gamma = fixture_model('hanks')
    V1, h1 = IncrementalPruning_Solver(gamma).solve(model, horizon=2)
    limit = max(h1.epochs[0]['fold_candidates'])
    assert max(h1.epochs[1]['fold_candidates']) > limit
    V, h = IncrementalPruning_Solver(gamma, max_candidates=limit).solve(model, horizon=50)
    assert h.stopped == 'candidates' and len(h.epochs) == 1
    assert h.shift == h.epochs[-1]['shift'] and len(V) == h.epochs[-1]['rows']
