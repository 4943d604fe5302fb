"""
Gap-driven trials (pbvi_gap_trial_step, GapSolver).  Checked against
  * pbvi_upper_backup (bitwise a* and Q*), pbvi_belief_update (bitwise next beliefs) and NumPy restatements of U, L, the excess and
    both observation rules (the argmax and NumPy's sampling rule);
  * the invariant X <= T_pi X of the append-only controller, monotone bounds at b0 round by round, the exact V* of tiger.95, the blind
    controller and the FIB bound on nine fixture models, and the determinism of a seeded solve.
"""
import ctypes

import numpy as np
import pytest

from test_policy_graph import GOLDEN9, check_certificate, controller_sweep_np
from test_upper_bound import fib_of, fixture_model, sawtooth_np, successors_np


# ---- CPU --------------------------------------------------------------------------------------------------------------------------
def test_gap_trial_step_rejects_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    buf = (ctypes.c_double * 8)()
    p = ctypes.addressof(buf)
    BAD = _native.PBVI_ERR_BAD_ARG
    args = dict(b=p, K=3, lower=p, N=2, fib=p, k=2, corner=p, lists=[p] * 5, n_ub=0, theta=0.0, uniform=None, out=p, nxt=p, U=None, L=None)

    def call(**kw):
        a = dict(args, **kw)
        return lib.pbvi_gap_trial_step(kw.get('m'), a['b'], a['K'], a['lower'], a['N'], a['fib'], a['k'], 0.95, a['corner'], *a['lists'],
                                       a['n_ub'], a['theta'], a['uniform'], a['out'], a['nxt'], a['U'], a['L'], None)
    assert call() == BAD and b'handle is NULL' in lib.pbvi_last_error()
    for name in ('b', 'lower', 'fib', 'corner', 'out', 'nxt'):
        assert call(**{name: None}) == BAD and b'NULL pointer' in lib.pbvi_last_error(), name
    assert call(n_ub=4, lists=[None] * 5) == BAD and b'NULL pointer' in lib.pbvi_last_error()
    for kw in (dict(K=-1), dict(n_ub=-1)):
        assert call(**kw) == BAD and b'non-negative' in lib.pbvi_last_error(), kw
    for kw in (dict(N=0), dict(N=-2), dict(k=0)):
        assert call(**kw) == BAD and b'N >= 1' in lib.pbvi_last_error(), kw
    assert call(theta=float('nan')) == BAD and b'NaN' in lib.pbvi_last_error()
    assert call(U=p) == BAD and b'together' in lib.pbvi_last_error()
    assert call(K=0, b=None, out=None) == BAD and b'handle is NULL' in lib.pbvi_last_error()     # nothing to do, but still a handle


def test_node_bookkeeping_matches_numpy():
    from pomdp_pbvi_exploration_b200.policy_graph import match_tuples, node_index
    rng = np.random.default_rng(2)
    for O, N, n in ((1, 5, 10), (3, 40, 200), (6, 200, 64)):
        actions = rng.integers(0, 3, N)
        succ = rng.integers(0, 4, (N, O))                     # few distinct values: many repeated (action, successors) tuples
        node_of = node_index(actions, succ)
        table = np.concatenate([actions[:, None], succ], axis=1)
        for t, node in node_of.items():
            hits = np.flatnonzero(np.all(table == np.asarray(t)[None, :], axis=1))
            assert node == hits[0]
        assert len(node_of) == len(np.unique(table, axis=0))
        tuples = np.concatenate([table[rng.integers(0, N, n // 2)], np.concatenate([rng.integers(0, 3, (n // 2, 1)),
                                                                                      rng.integers(0, 6, (n // 2, O))], axis=1)])
        tuples = tuples[rng.permutation(n)]
        in_use, new_t = match_tuples(node_of, tuples)
        known = np.array([any(np.array_equal(r, t) for r in table) for t in tuples])
        first_rows = [hits[0] for hits in (np.flatnonzero(np.all(table == t[None, :], axis=1)) for t in tuples[known])]
        assert in_use == set(int(i) for i in first_rows)
        _, first = np.unique(tuples[~known], axis=0, return_index=True)
        assert np.array_equal(new_t, tuples[~known][np.sort(first)])


def choose_np(e, u):
    """The observation rules of pbvi_gap_trial_step on the excesses e [O] (NaN: impossible): the first argmax of e over {e > 0}
    without a uniform (u None or < 0), else NumPy's draw with weights max(e, 0); -1 when no excess is positive."""
    pos = np.where(e > 0, e, 0.0)                           # NaN > 0 is False
    if not np.any(pos > 0):
        return -1
    if u is None or u < 0:
        return int(np.argmax(pos))
    cdf = np.cumsum(pos)
    cdf /= cdf[-1]
    return int(min(np.searchsorted(cdf, u, side='right'), np.flatnonzero(pos > 0)[-1]))


def test_sampling_rule_is_numpys():
    rng = np.random.default_rng(4)
    for trial in range(2000):
        O = int(rng.integers(1, 9))
        e = rng.normal(size=O)
        e[rng.random(O) < 0.2] = np.nan
        seed = int(rng.integers(1 << 30))
        u = np.random.RandomState(seed).random_sample()
        got = choose_np(e, u)
        pos = np.where(e > 0, e, 0.0)
        if not np.any(pos > 0):
            assert got == -1
            continue
        assert pos[got] > 0                                  # never an impossible or non-positive observation
        cdf = np.cumsum(pos) / np.cumsum(pos)[-1]
        if np.min(np.abs(cdf - u)) < 1e-12:
            continue
        # np.random.choice draws one uniform and searches the normalised cdf of p
        want = np.random.RandomState(seed).choice(O, p=pos / pos.sum())
        assert got == want, (trial, e, u)
    assert choose_np(np.array([0.5, 2.0, 2.0, np.nan]), None) == 1
    assert choose_np(np.array([-1.0, 0.0, np.nan]), 0.3) == -1


# ---- GPU: one step against NumPy ------------------------------------------------------------------------------------------------
STEP_MODELS = ['tiger', 'grid4x4', 'hallway', 'tigergrid', 'cheese', 'grid4x3', 'olfactory_wrap']


def walk_beliefs(model, n, seed):
    """n + 1 beliefs: b0 and a seeded random walk from it (device draws of the observations)."""
    import torch
    dev = model.device
    rng = np.random.default_rng(seed)
    b0 = torch.as_tensor(model.start_probabilities, device='cuda', dtype=torch.float64)
    walk = dev.perseus_walk(b0, rng.integers(0, model.action_count, n).astype(np.int32), rng.random(n))
    return torch.cat([b0[None, :], walk]).contiguous()


def step_np(model, gamma, F, X, store_rows, store_vals, b, a):
    """U_o, L_o [O] at the successors of b under a (NaN for impossible observations) and the masses P(o|b,a)."""
    succ, mass = successors_np(model, b)
    corner = F.max(axis=0)
    O = mass.shape[1]
    U, L = np.full(O, np.nan), np.full(O, np.nan)
    for o in range(O):
        if mass[a, o] > 0:
            q = succ[a, o]
            U[o] = min(np.max(F @ q), sawtooth_np(q, corner, store_rows, store_vals))
            L[o] = np.max(X @ q)
    return U, L, mass[a]


_steps = {}


def step_inputs(tag):
    """(model, gamma, fib, lower rows X, beliefs, UpperBound with stored pairs): X = the blind controller's rows and perturbed copies."""
    import torch
    from pomdp_pbvi_exploration_b200 import PolicyGraph, UpperBound
    if tag not in _steps:
        model, gamma = fixture_model(tag)
        fib, _ = fib_of(tag)
        blind = PolicyGraph.blind(model)
        blind.evaluate(gamma)
        W = blind.rows
        X = torch.cat([W, W + torch.as_tensor(np.random.default_rng(1).normal(size=tuple(W.shape)) * 0.05 * (1 + W.abs().max().item()),
                                              device='cuda')]).contiguous()
        B = walk_beliefs(model, 200, 3)
        ub = UpperBound(model, fib, gamma)
        ub.improve(B[130:])
        _steps[tag] = (model, gamma, fib, X, B, ub)
    return _steps[tag]


@pytest.mark.gpu
@pytest.mark.parametrize('tag', STEP_MODELS)
@pytest.mark.parametrize('K', [1, 2, 129])
@pytest.mark.parametrize('stored', [False, True])
def test_step_matches_numpy(tag, K, stored):
    import torch
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma, fib, X, B, ub_stored = step_inputs(tag)
    ub = ub_stored if stored else UpperBound(model, fib, gamma)
    assert (len(ub) > 0) == stored
    dev = model.device
    O = model.observation_count
    b = B[:K].contiguous()
    idx, val, count, dot, vals, n_ub = ub._lists()
    F = fib.alpha_vector_array
    u_ref, _, a_ref = dev.upper_backup(b, F, gamma, ub.corner_values, idx, val, count, dot, vals, n_ub, want_action=True)
    a_ref, u_ref = a_ref.cpu().numpy(), u_ref.cpu().numpy()
    _, mass_all = dev.belief_successors(b)
    mass_all = mass_all.cpu().numpy()
    Fh, Xh = F.cpu().numpy(), X.cpu().numpy()
    store_rows, store_vals = ub.belief_array.cpu().numpy(), ub.value_array.cpu().numpy()
    bh = b.cpu().numpy()
    rng = np.random.default_rng(K)
    uniforms = rng.random(K)
    uniforms[::3] = -1.0                                                   # every third trial takes the argmax rule
    ref = [step_np(model, gamma, Fh, Xh, store_rows, store_vals, bh[k], int(a_ref[k])) for k in range(K)]
    gaps = np.concatenate([r[0] - r[1] for r in ref])
    gaps = gaps[np.isfinite(gaps)]
    for theta in (0.0, float(np.median(gaps)), 1e30):
        for rule in ('argmax', 'sample'):
            u = None if rule == 'argmax' else uniforms
            out, nxt, U, L = dev.gap_trial_step(b, X, F, gamma, ub.corner_values, idx, val, count, dot, vals, n_ub, theta, u, want_bounds=True)
            out, U, L = out.cpu().numpy(), U.cpu().numpy(), L.cpu().numpy()
            a, o = out[:, 0].astype(np.int64), out[:, 1].astype(np.int64)
            assert np.array_equal(a, a_ref) and out[:, 2].tobytes() == u_ref.tobytes(), (tag, K)
            for k in range(K):
                U_np, L_np, p_np = ref[k]
                p = mass_all[k, a[k]]
                possible = p > 0
                assert np.array_equal(possible, p_np > 0)
                assert np.all(np.isnan(U[k][~possible])) and np.all(np.isnan(L[k][~possible]))
                sc = np.maximum(1.0, np.abs(U_np[possible]))
                assert np.all(np.abs(U[k][possible] - U_np[possible]) <= 1e-9 * sc), (tag, k)
                sc = np.maximum(1.0, np.abs(L_np[possible]))
                assert np.all(np.abs(L[k][possible] - L_np[possible]) <= 1e-9 * sc), (tag, k)
                e_dev = np.where(possible, p * ((U[k] - L[k]) - theta), np.nan)       # the device's own U, L: bitwise the same rule
                uk = None if u is None else u[k]
                assert o[k] == choose_np(e_dev, uk), (tag, K, k, theta, rule)
                e_np = np.where(possible, p_np * ((U_np - L_np) - theta), np.nan)
                tol = 2e-9 * p_np * (np.maximum(1.0, np.abs(U_np)) + np.maximum(1.0, np.abs(L_np)) + abs(theta))
                assert np.all(np.abs(e_dev - e_np)[possible] <= tol[possible]), (tag, k)
                if np.all(np.abs(e_np[possible]) > 1e-6) and (uk is None or uk < 0):
                    top = np.sort(e_np[possible & (e_np > 0)])
                    if len(top) < 2 or top[-1] - top[-2] > 1e-6:
                        assert o[k] == choose_np(e_np, None), (tag, k)
                if o[k] >= 0:
                    assert possible[o[k]]                                      # an impossible observation is never chosen
                    assert out[k, 3] == e_dev[o[k]]
                else:
                    assert not np.any(e_dev > 0)
                    assert out[k, 3] == (np.nanmax(e_dev) if possible.any() else -np.inf)
            if theta == 1e30:
                assert np.all(o == -1)
            live = np.flatnonzero(o >= 0)
            if len(live):
                want, _ = dev.belief_update(b[live], a[live].astype(np.int32), o[live].astype(np.int32), normalise=True)
                assert nxt[live].cpu().numpy().tobytes() == want.cpu().numpy().tobytes(), (tag, K)
            dead = np.flatnonzero(o < 0)
            if len(dead):
                assert nxt[dead].cpu().numpy().tobytes() == bh[dead].tobytes()


# ---- GPU: the solver --------------------------------------------------------------------------------------------------------------
def check_rounds(history):
    ups = [r['upper_b0'] for r in history.rounds]
    los = [r['lower_b0'] for r in history.rounds]
    assert all(u1 <= u0 for u0, u1 in zip(ups, ups[1:])), ups
    assert all(l1 >= l0 for l0, l1 in zip(los, los[1:])), los
    if history.reached:
        assert history.upper - history.lower <= history.target_gap
    assert history.lower <= history.upper


def check_uncertified(model, gamma, history):
    """X <= T_pi X on the append-only rows, within the rounding allowance of `evaluate`."""
    pg = history.uncertified
    W = pg.rows.cpu().numpy()
    TW = controller_sweep_np(model, pg.actions, pg.successors, W, gamma)
    ulps = (model.observation_count * model.reachable_state_count + 2) * 2.0 ** -52
    assert np.all(W <= TW + ulps * np.max(np.abs(W)) + 1e-12 * np.maximum(1.0, np.abs(W))), float(np.max(W - TW))


TIGER_TARGET, TIGER_ROUNDS = 0.1, 40            # measured on a B200: the target is certified after 18 rounds


@pytest.mark.gpu
def test_tiger_reaches_its_target_around_the_exact_value():
    from test_upper_bound import tiger_exact_value
    from pomdp_pbvi_exploration_b200 import GapSolver
    model, gamma = fixture_model('tiger')
    grid = np.linspace(0.0, 1.0, 201)
    vstar = tiger_exact_value(model, gamma, grid)
    pg, ub, hist = GapSolver(gamma, TIGER_TARGET, trials=4, max_depth=60, seed=0).solve(model, max_rounds=TIGER_ROUNDS)
    assert hist.reached and hist.gap <= TIGER_TARGET, (hist.lower, hist.upper, len(hist.rounds))
    check_rounds(hist)
    check_uncertified(model, gamma, hist)
    check_certificate(model, gamma, pg)
    v0 = tiger_exact_value(model, gamma, np.array([float(model.start_probabilities[1])]))[0]
    assert hist.lower <= v0 + 1e-9 <= hist.upper + 2e-9, (hist.lower, v0, hist.upper)
    B = np.stack([1 - grid, grid], axis=1)
    lo = pg.value(B)[0].cpu().numpy()
    up = ub.evaluate(B).cpu().numpy()
    assert np.all(lo <= vstar + 1e-9) and np.all(vstar <= up + 1e-9), (float(np.max(lo - vstar)), float(np.max(vstar - up)))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', GOLDEN9)
def test_bounds_stay_sound_on_golden_models(tag):
    from pomdp_pbvi_exploration_b200 import GapSolver, PolicyGraph, UpperBound
    model, gamma = fixture_model(tag)
    fib, _ = fib_of(tag)
    b0 = model.start_probabilities[None, :]
    fib_b0 = float(UpperBound(model, fib, gamma).evaluate(b0)[0])
    blind = PolicyGraph.blind(model)
    blind.evaluate(gamma)
    blind_b0 = float(blind.value(b0)[0][0])
    pg, ub, hist = GapSolver(gamma, 1e-3, trials=4, max_depth=25, seed=1).solve(model, max_rounds=3,
                                                                                 upper=UpperBound(model, fib, gamma))
    check_rounds(hist)
    check_uncertified(model, gamma, hist)
    check_certificate(model, gamma, pg)
    assert hist.lower >= blind_b0 - hist.shift - 1e-12 * max(1.0, abs(blind_b0)), (tag, hist.lower, blind_b0, hist.shift)
    assert hist.upper <= fib_b0, (tag, hist.upper, fib_b0)
    assert len(hist.rounds) == 3 or hist.reached
    assert all(max(r['depths']) < 25 for r in hist.rounds)


@pytest.mark.gpu
def test_olfactory_solve_keeps_its_bounds():
    from pomdp_pbvi_exploration_b200 import GapSolver
    model, gamma = fixture_model('olfactory_wrap')
    pg, ub, hist = GapSolver(gamma, 0.1, trials=8, max_depth=40, seed=0).solve(model, max_rounds=2)
    check_rounds(hist)
    assert hist.rounds[-1]['nodes'] > model.action_count and hist.rounds[-1]['stored_pairs'] > 0
    assert hist.lower <= hist.upper


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['hallway', 'tigergrid'])
def test_solve_is_deterministic(tag):
    from pomdp_pbvi_exploration_b200 import GapSolver
    model, gamma = fixture_model(tag)

    def run(trials, seed):
        pg, ub, hist = GapSolver(gamma, 1e-3, trials=trials, max_depth=20, seed=seed).solve(model, max_rounds=3)
        rounds = [{k: v for k, v in r.items() if k not in ('phase_seconds', 'seconds')} for r in hist.rounds]
        return (pg.actions.tolist(), pg.successors.tolist(), pg.rows.cpu().numpy().tobytes(), ub.value_array.cpu().numpy().tobytes(),
                rounds, hist.lower, hist.upper)
    a = run(6, 3)
    assert a == run(6, 3)
    assert a != run(6, 4)                                  # the sampled trials do see the seed
    assert run(1, 3) == run(1, 99)


@pytest.mark.gpu
def test_solver_rejects_bad_settings():
    from pomdp_pbvi_exploration_b200 import GapSolver, PolicyGraph
    model, gamma = fixture_model('tiger')
    with pytest.raises(ValueError):
        GapSolver(1.0, 0.1).solve(model)
    scaled, _ = fixture_model('tiger', rto_scale=1.1)
    with pytest.raises(ValueError, match='contraction'):
        GapSolver(gamma, 0.1).solve(scaled)
    with pytest.raises(ValueError):
        GapSolver(gamma, 0.1).solve(model, lower=PolicyGraph.blind(model))                 # not evaluated
    with pytest.raises(ValueError):
        GapSolver(gamma, 0.0)
