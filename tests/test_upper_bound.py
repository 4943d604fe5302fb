"""
Certified upper bounds: the FIB sweep (pbvi_fib_sweep, FIB_Solver) and the point-based upper-bound backup (pbvi_upper_backup,
UpperBound).  Checked against
  * NumPy restatements of one FIB sweep (bit-identical on R = 1 models) and of one chunk of upper-bound backups;
  * the FIB certificate H U <= U on every fixture model;
  * the exact V* of tiger.95 (alpha-vector value iteration with 1-D envelope pruning: S = 2);
  * lower bounds of real solves: max_v alpha_v . b <= upper(b) at b0 and at every explored belief, before and after `improve`.
"""
import ctypes
import random

import numpy as np
import pytest

from conftest import load_golden

MODELS = ['tiger', 'grid4x4', 'grid4x4_noloop', 'tigergrid', 'hallway', 'cheese', 'grid4x3', 'cit', 'synth300', 'olfactory_wrap']


# ---- CPU: argument checks of the C ABI ------------------------------------------------------------------------------------------
def test_bound_entry_points_reject_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    buf = (ctypes.c_double * 8)()
    p = ctypes.addressof(buf)
    BAD = _native.PBVI_ERR_BAD_ARG
    assert lib.pbvi_fib_sweep(None, p, 2, 0.9, p, None, None) == BAD
    assert b'handle is NULL' in lib.pbvi_last_error()
    assert lib.pbvi_fib_sweep(None, None, 2, 0.9, p, None, None) == BAD
    assert b'NULL pointer' in lib.pbvi_last_error()
    assert lib.pbvi_fib_sweep(None, p, 2, 0.9, None, None, None) == BAD
    assert b'NULL pointer' in lib.pbvi_last_error()
    assert lib.pbvi_fib_sweep(None, p, -1, 0.9, p, None, None) == BAD
    assert b'positive' in lib.pbvi_last_error()
    args = dict(b=p, n=3, fib=p, k=2, corner=p, lists=[p] * 5, n_ub=0, u=p)

    def call(**kw):
        a = dict(args, **kw)
        return lib.pbvi_upper_backup(kw.get('m'), a['b'], a['n'], a['fib'], a['k'], 0.9, a['corner'], *a['lists'], a['n_ub'], a['u'], None,
                                     None, None)
    assert call() == BAD and b'handle is NULL' in lib.pbvi_last_error()
    for name in ('b', 'fib', 'corner', 'u'):
        assert call(**{name: None}) == BAD and b'NULL pointer' in lib.pbvi_last_error(), name
    assert call(n_ub=4, lists=[None] * 5) == BAD and b'NULL pointer' in lib.pbvi_last_error()
    for kw in (dict(n=-1), dict(n_ub=-1)):
        assert call(**kw) == BAD and b'non-negative' in lib.pbvi_last_error(), kw
    assert call(k=0) == BAD and b'positive' in lib.pbvi_last_error()


# ---- fixtures -------------------------------------------------------------------------------------------------------------------
def seed_all(seed):
    np.random.seed(seed)
    random.seed(seed)


_models = {}


def fixture_model(tag, rto_scale=1.0):
    """A package `Model` carrying exactly the reference's tensors of the fixture (bypasses the constructor's own derivations)."""
    from pomdp_pbvi_exploration_b200 import Model
    key = (tag, rto_scale)
    if key in _models:
        return _models[key]
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
    model.reachable_transitional_observation_table = m['rto'] * rto_scale
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
    _models[key] = (model, float(m['gamma']))
    return _models[key]


def test_fib_solver_rejects_a_non_contracting_model():
    from pomdp_pbvi_exploration_b200 import FIB_Solver
    model, gamma = fixture_model('tiger', rto_scale=1.1)            # gamma * m = 0.95 * 1.1 >= 1
    with pytest.raises(ValueError, match='contraction'):
        FIB_Solver(gamma=gamma).solve(model, print_progress=False)


def fib_np(model, U, gamma):
    """One FIB sweep in NumPy, in the kernel's order: r ascending inside, then o ascending, one rounding per product and sum."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, R = reach.shape
    O = rto.shape[2]
    out = np.empty((A, S))
    for a in range(A):
        acc = np.zeros(S)
        for o in range(O):
            inner = None
            for r in range(R):
                prod = rto[:, a, o, r][:, None] * U[:, reach[:, a, r]].T            # [S, k]
                inner = prod if r == 0 else inner + prod
            acc = acc + inner.max(axis=1)
        out[a] = rbar[:, a] + gamma * acc
    return out


_fibs = {}


def fib_of(tag):
    from pomdp_pbvi_exploration_b200 import FIB_Solver
    if tag not in _fibs:
        model, gamma = fixture_model(tag)
        _fibs[tag] = FIB_Solver(gamma=gamma, eps=1e-6).solve(model, print_progress=False)
    return _fibs[tag]


# ---- GPU: the FIB sweep and solver -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('tag', MODELS)
def test_fib_sweep_matches_numpy(tag):
    import torch
    model, gamma = fixture_model(tag)
    dev = model.device
    A, S, R = model.action_count, model.state_count, model.reachable_state_count
    rng = np.random.default_rng(3)
    rbar = model.expected_rewards_table
    inputs = [np.full((A, S), float(rbar.max()) / (1 - gamma)),                  # k = A: the solver's start
              rng.normal(size=(A, S)) * 10,                                       # k = A
              np.full((1, S), float(rbar.min()) / (1 - gamma)),                  # k = 1
              rng.normal(size=(A + 2, S))]                                       # k = A + 2
    for U in inputs:
        want = fib_np(model, U, gamma)
        if U.shape[0] == A:
            got, stats = dev.fib_sweep(torch.as_tensor(U, device='cuda'), gamma, want_stats=True)
            st = stats.cpu().numpy()
            assert st[0] == np.max(got.cpu().numpy() - U) and st[1] == np.max(np.abs(got.cpu().numpy() - U))
        else:
            got = dev.fib_sweep(torch.as_tensor(U, device='cuda'), gamma)
        got = got.cpu().numpy()
        if R == 1:
            assert np.array_equal(got, want), (tag, U.shape)
        else:
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12 * max(1.0, float(np.max(np.abs(want)))))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', MODELS)
def test_fib_solver_certificate(tag):
    model, gamma = fixture_model(tag)
    vf, hist = fib_of(tag)
    rows, actions = vf.numpy()
    A = model.action_count
    assert len(vf) <= A and np.isfinite(rows).all()
    assert hasattr(hist, 'fib_residual') and hist.fib_shift >= 0.0
    HU = fib_np(model, rows, gamma)                        # the max over a' of the kept rows = the max over all A rows (dedup drops copies)
    own = {int(a): rows[i] for i, a in enumerate(actions)}
    for a in range(A):
        # a row merged by the byte-dedup equals one of the kept rows, all of which lie below their elementwise maximum
        U_a = own.get(a, rows.max(axis=0))
        assert np.all(HU[a] <= U_a + 1e-12 * np.maximum(1.0, np.abs(U_a))), (tag, a, float(np.max(HU[a] - U_a)))


# ---- exact V* of tiger.95 ------------------------------------------------------------------------------------------------------
def upper_envelope(alphas):
    """Rows of [n,2] alphas that are maximal somewhere on b = (1 - p, p), p in [0, 1] (lines c + m p, convex-hull trick)."""
    c, m = alphas[:, 0], alphas[:, 1] - alphas[:, 0]
    order = np.lexsort((c, m))
    hull = []
    for i in order:
        if hull and m[hull[-1]] == m[i]:
            hull.pop()                                       # same slope: the later one has the larger intercept
        while len(hull) >= 2:
            i1, i2 = hull[-2], hull[-1]
            # i2 is never strictly on top if the new line meets i1 left of where i2 does
            if (c[i] - c[i1]) * (m[i2] - m[i1]) >= (c[i2] - c[i1]) * (m[i] - m[i1]):
                hull.pop()
            else:
                break
        hull.append(i)
    keep = []
    for j, i in enumerate(hull):                             # restrict to [0, 1]: interval of line j on the hull
        lo = -np.inf if j == 0 else (c[hull[j - 1]] - c[i]) / (m[i] - m[hull[j - 1]])
        hi = np.inf if j == len(hull) - 1 else (c[i] - c[hull[j + 1]]) / (m[hull[j + 1]] - m[i])
        if hi >= 0.0 and lo <= 1.0:
            keep.append(i)
    return alphas[keep]


def tiger_exact_value(model, gamma, grid):
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, R = reach.shape
    O = rto.shape[2]
    V = np.full((1, S), float(rbar.min()) / (1 - gamma))
    B = np.stack([1 - grid, grid], axis=1)
    prev = None
    for _ in range(5000):
        new = []
        for a in range(A):
            # g[o][v] = sum_r RTO[s,a,o,r] V_v[reach[s,a,r]]
            g = [np.stack([sum(rto[:, a, o, r] * V[v, reach[:, a, r]] for r in range(R)) for v in range(len(V))]) for o in range(O)]
            acc = g[0]
            for o in range(1, O):
                acc = upper_envelope((acc[:, None, :] + g[o][None, :, :]).reshape(-1, S))
            new.append(rbar[:, a][None, :] + gamma * acc)
        V = upper_envelope(np.concatenate(new))
        val = np.max(B @ V.T, axis=1)
        if prev is not None and np.max(np.abs(val - prev)) < 1e-13:
            break
        prev = val
    return val


@pytest.mark.gpu
def test_tiger_upper_bound_against_exact_value():
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma = fixture_model('tiger')
    fine = np.linspace(0.0, 1.0, 1001)
    vstar = tiger_exact_value(model, gamma, fine)
    fib, _ = fib_of('tiger')
    ub = UpperBound(model, fib, gamma)
    B_fine = np.stack([1 - fine, fine], axis=1)
    f0 = ub.evaluate(B_fine).cpu().numpy()
    assert np.all(f0 >= vstar - 1e-9), float(np.min(f0 - vstar))
    coarse = np.linspace(0.0, 1.0, 101)
    B = np.stack([1 - coarse, coarse], axis=1)
    b0 = model.start_probabilities
    fib_b0 = ub.gap(fib, b0)[1]
    prev_vals = None
    for it in range(5000):
        n_dec, largest = ub.improve(B)
        vals = ub.value_array.cpu().numpy()
        if prev_vals is not None:
            assert np.all(vals[:len(prev_vals)] <= prev_vals), it
        prev_vals = vals.copy()
        if largest <= 1e-12:
            break
    assert largest <= 1e-12
    up = ub.evaluate(B_fine).cpu().numpy()
    assert np.all(up >= vstar - 1e-9), float(np.min(up - vstar))
    assert np.all(up <= f0)
    upper_b0 = ub.evaluate(b0[None, :]).cpu().numpy()[0]
    assert upper_b0 < fib_b0, (upper_b0, fib_b0)


# ---- one chunk of upper-bound backups against NumPy ----------------------------------------------------------------------------
_solves = {}


def seeded_solve(tag, lower_start=False):
    from pomdp_pbvi_exploration_b200 import PBVI_Solver, ValueFunction
    key = (tag, lower_start)
    if key not in _solves:
        model, gamma = fixture_model(tag)
        seed_all(5)
        kw = {}
        if lower_start:
            S = model.state_count
            lo = float(model.expected_rewards_table.min()) / (1 - gamma)
            kw['initial_value_function'] = ValueFunction(model, np.full((1, S), lo), [0])
        solver = PBVI_Solver(gamma=gamma, eps=1e-6, expand_function='perseus')
        vf, hist = solver.solve(model, expansions=8, max_belief_growth=25, history_tracking_level=2, print_progress=False, **kw)
        _solves[key] = (model, vf, hist)
    return _solves[key]


def successors_np(model, b):
    reach, rto = model.reachable_states, model.reachable_transitional_observation_table
    S, A, R = reach.shape
    O = rto.shape[2]
    succ = np.zeros((A, O, S))
    for a in range(A):
        for o in range(O):
            for r in range(R):
                np.add.at(succ[a, o], reach[:, a, r], b * rto[:, a, o, r])
    mass = succ.sum(axis=2)
    with np.errstate(invalid='ignore', divide='ignore'):
        return succ / mass[:, :, None], mass


def sawtooth_np(q, corner, store_rows, store_vals):
    v0 = q @ corner
    best = v0
    for bi, vi in zip(store_rows, store_vals):
        sup = bi > 0
        ratio = np.min(q[sup] / bi[sup])
        best = min(best, v0 + (vi - bi @ corner) * ratio)
    return best


def upper_backup_np(model, gamma, F, store_rows, store_vals, b):
    corner = F.max(axis=0)
    rbar = model.expected_rewards_table
    succ, mass = successors_np(model, b)
    A, O = mass.shape
    qs = []
    for a in range(A):
        acc = 0.0
        for o in range(O):
            if mass[a, o] > 0:
                q = succ[a, o]
                acc += mass[a, o] * min(np.max(F @ q), sawtooth_np(q, corner, store_rows, store_vals))
        qs.append(b @ rbar[:, a] + gamma * acc)
    cur = min(np.max(F @ b), sawtooth_np(b, corner, store_rows, store_vals))
    return max(qs), cur


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4', 'hallway', 'cheese'])
def test_one_chunk_matches_numpy(tag):
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, vf, hist = seeded_solve(tag)
    gamma = fixture_model(tag)[1]
    fib, _ = fib_of(tag)
    F = fib.alpha_vector_array.cpu().numpy()
    B = hist.belief_sets[-1].belief_array.cpu().numpy()
    ub = UpperBound(model, fib, gamma)
    ub.improve(B[: len(B) // 2])                                # a non-empty store to start from
    store_rows, store_vals = ub.belief_array.cpu().numpy().copy(), ub.value_array.cpu().numpy().copy()
    assert len(store_rows) > 0
    assert ub._chunk(len(B)) == len(B)                          # the pass below is one pbvi_upper_backup call
    rev = B[::-1]
    want = np.array([upper_backup_np(model, gamma, F, store_rows, store_vals, b) for b in rev])
    dev = model.device
    idx, val, count, dot, vals, n_ub = ub._lists()
    u, cur = dev.upper_backup(rev.copy(), fib.alpha_vector_array, gamma, ub.corner_values, idx, val, count, dot, vals, n_ub)
    got = np.stack([u.cpu().numpy(), cur.cpu().numpy()], axis=1)
    scale = np.maximum(1.0, np.abs(want))
    assert np.all(np.abs(got - want) <= 1e-9 * scale), (tag, float(np.max(np.abs(got - want) / scale)))
    # the same pass through `improve`: the same beliefs get stored / lowered, with u
    n_before = len(ub)
    ub.improve(B)
    rows_after, vals_after = ub.belief_array.cpu().numpy(), ub.value_array.cpu().numpy()
    clear = np.abs(want[:, 0] - want[:, 1]) > 1e-9 * scale[:, 0]
    keys = {r.tobytes(): i for i, r in enumerate(rows_after)}
    for j, b in enumerate(rev):
        if not clear[j]:
            continue
        pos = keys.get(b.tobytes())
        old = next((store_vals[i] for i, r in enumerate(store_rows) if np.array_equal(r, b)), None)
        if want[j, 0] < want[j, 1]:
            assert pos is not None, (tag, j)
            assert abs(vals_after[pos] - min(want[j, 0], old if old is not None else np.inf)) <= 1e-9 * scale[j, 0]
        else:
            assert (pos is None) == (old is None) and (pos is None or pos < n_before and vals_after[pos] == old), (tag, j)


# ---- lower <= upper at scale, determinism ---------------------------------------------------------------------------------------
def check_lower_below_upper(model, vf, ub, rows):
    import torch
    R = torch.as_tensor(np.concatenate([model.start_probabilities[None, :], rows]), device='cuda')
    lower = model.device.max_values(R, vf.alpha_vector_array)[0].cpu().numpy()
    upper = ub.evaluate(R).cpu().numpy()
    assert np.all(lower <= upper + 1e-9 * np.maximum(1.0, np.abs(upper))), float(np.max(lower - upper))
    return lower, upper


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4', 'grid4x4_noloop', 'tigergrid', 'hallway', 'cheese', 'grid4x3', 'cit', 'synth300'])
def test_lower_below_upper_on_golden_models(tag):
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, vf, hist = seeded_solve(tag, lower_start=True)
    gamma = fixture_model(tag)[1]
    fib, _ = fib_of(tag)
    B = hist.belief_sets[-1].belief_array.cpu().numpy()
    ub = UpperBound(model, fib, gamma)
    check_lower_below_upper(model, vf, ub, B)
    ub.improve(B, passes=2)
    assert len(ub) > 0
    check_lower_below_upper(model, vf, ub, B)


_olfactory = {}


def olfactory_solve(expansions, growth, seed):
    """The olfactory recipe model (its observation table drives FSVI's trajectories), its FIB rows and a seeded FSVI solve."""
    from pomdp_pbvi_exploration_b200 import FIB_Solver, FSVI_Solver
    from pomdp_pbvi_exploration_b200.recipes import olfactory_wrap_model
    if 'model' not in _olfactory:
        model = olfactory_wrap_model()
        _olfactory['model'] = model
        _olfactory['fib'] = FIB_Solver(gamma=0.99, eps=1e-6).solve(model, print_progress=False)[0]
    model = _olfactory['model']
    seed_all(seed)
    vf, hist = FSVI_Solver(gamma=0.99, eps=1e-6).solve(model, expansions=expansions, max_belief_growth=growth, history_tracking_level=2,
                                                      print_progress=False)
    return model, 0.99, _olfactory['fib'], vf, hist


@pytest.mark.gpu
def test_lower_below_upper_on_olfactory_fsvi_multi_chunk():
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma, fib, vf, hist = olfactory_solve(10, 100, 0)
    assert float(model.expected_rewards_table.min()) >= 0.0         # the R-bar start of the solve is a lower bound
    B = hist.belief_sets[-1].belief_array.cpu().numpy()
    ub = UpperBound(model, fib, gamma)
    _, up0 = check_lower_below_upper(model, vf, ub, B)
    ub._chunk_bytes = 64 << 20                                       # about 20 beliefs per call: many chunks
    assert ub._chunk(len(B)) < len(B) // 4
    n_dec, largest = ub.improve(B)
    assert n_dec > 0 and largest > 0.0
    _, up1 = check_lower_below_upper(model, vf, ub, B)
    assert np.all(up1 <= up0)


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['hallway', 'olfactory_wrap'])
def test_improve_is_deterministic(tag):
    from pomdp_pbvi_exploration_b200 import UpperBound
    if tag == 'olfactory_wrap':
        model, gamma, fib, _, hist = olfactory_solve(4, 50, 1)
    else:
        model, gamma = fixture_model(tag)
        fib, _ = fib_of(tag)
        _, _, hist = seeded_solve(tag)
    B = hist.belief_sets[-1].belief_array
    out = []
    for _ in range(2):
        ub = UpperBound(model, fib, gamma)
        ub._chunk_bytes = 16 << 20
        ub.improve(B, passes=2)
        out.append((ub.belief_array.cpu().numpy(), ub.value_array.cpu().numpy()))
    assert np.array_equal(out[0][0], out[1][0]) and out[0][1].tobytes() == out[1][1].tobytes()


@pytest.mark.gpu
def test_upper_bound_rejects_non_finite_beliefs():
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma = fixture_model('tiger')
    fib, _ = fib_of('tiger')
    ub = UpperBound(model, fib, gamma)
    with pytest.raises(ValueError):
        ub.improve(np.array([[0.5, np.nan]]))
    with pytest.raises(ValueError):
        ub.evaluate(np.array([[np.inf, 0.0]]))
