"""
Exact outcomes of finite-state controllers that stop at end states (pbvi_controller_outcomes, PolicyGraph.outcomes).  Checked against
  * a NumPy restatement of the three recursions in the kernel's order (bitwise), and k pbvi_controller_sweep calls when nothing ends;
  * a NumPy forward propagation of the run distribution over (node, state) (the series: CDF, truncated steps and return);
  * the certified controller value (no ends, gamma < 1), the closed form of a tiger controller, and Monte Carlo roll-outs under the
    reference's termination rule;
  * edge cases: zero steps, a start in an end state, every action an end action, determinism, a long horizon on a large controller.
"""
import copy
import ctypes

import numpy as np
import pytest

from test_policy_graph import extracted
from test_upper_bound import fixture_model


# ---- CPU ------------------------------------------------------------------------------------------------------------------------
def test_controller_outcomes_rejects_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    buf = (ctypes.c_double * 8)()
    p = ctypes.addressof(buf)
    BAD = _native.PBVI_ERR_BAD_ARG
    args = dict(m=p, n=2, actions=p, succ=p, end_state=p, end_action=p, steps=3, queries=p, qnodes=p, q=1, P=p, M=p, G=p, series=p)

    def call(**kw):
        a = dict(args, **kw)
        return lib.pbvi_controller_outcomes(a['m'], a['n'], a['actions'], a['succ'], a['end_state'], a['end_action'], 0.9, a['steps'],
                                            a['queries'], a['qnodes'], a['q'], a['P'], a['M'], a['G'], a['series'], None)
    assert call(m=None) == BAD and b'handle is NULL' in lib.pbvi_last_error()
    for name in ('actions', 'succ', 'end_state', 'end_action', 'P', 'M', 'G', 'queries', 'qnodes', 'series'):
        assert call(**{name: None}) == BAD and b'NULL pointer' in lib.pbvi_last_error(), name
    for n in (0, -3):
        assert call(n=n) == BAD and b'n >= 1' in lib.pbvi_last_error(), n
    assert call(steps=-1) == BAD and b'steps >= 0' in lib.pbvi_last_error()
    assert call(q=-1) == BAD and b'q >= 0' in lib.pbvi_last_error()


@pytest.mark.parametrize('tag', ['hanks', 'network'])
def test_outcomes_rejects_leaking_rto_rows(tag):
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model(tag)
    assert np.max(np.abs(model.reachable_transitional_observation_table.sum(axis=(2, 3)) - 1.0)) > 0.5
    with pytest.raises(ValueError, match='sum to 1'):
        PolicyGraph.blind(model).outcomes(10, start_nodes=[0], gamma=gamma)


def test_outcomes_rejects_bad_settings():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model('tiger')
    pg = PolicyGraph.blind(model)
    with pytest.raises(ValueError, match='gamma'):
        pg.outcomes(5)                                                  # no evaluate, no gamma
    for g in (0.0, -0.5, 1.0 + 1e-12, float('nan'), float('inf')):
        with pytest.raises(ValueError, match='gamma'):
            pg.outcomes(5, start_nodes=[0], gamma=g)
    for h in (-1, 2.5):
        with pytest.raises(ValueError, match='max_steps'):
            pg.outcomes(h, start_nodes=[0], gamma=gamma)
    with pytest.raises(ValueError, match='no rows'):
        pg.outcomes(5, gamma=1.0)                                      # gamma = 1 is allowed; start nodes need rows


# ---- NumPy references ------------------------------------------------------------------------------------------------------------
def end_flags(model):
    es = np.zeros(model.state_count, dtype=bool)
    es[np.asarray(model.end_states, dtype=np.int64)] = True
    ea = np.zeros(model.action_count, dtype=bool)
    ea[np.asarray(model.end_actions, dtype=np.int64)] = True
    return es, ea


def outcomes_np(model, actions, succ, gamma, k):
    """k steps of the three recursions from zero rows, in the kernel's order: r ascending inside, then o ascending, one rounding per
    operation, a zero RTO weight taking +0.0 for all three terms unless Rbar is -0.0 (alpha_a_entry's skip)."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, R = reach.shape
    O = rto.shape[2]
    es, ea = end_flags(model)
    N = len(actions)
    P, M, G = np.zeros((N, S)), np.zeros((N, S)), np.zeros((N, S))
    for _ in range(k):
        nP, nM, nG = np.empty_like(P), np.empty_like(M), np.empty_like(G)
        for a in np.unique(actions):
            nodes = np.flatnonzero(actions == a)
            skip = ~((rbar[:, a] == 0.0) & np.signbit(rbar[:, a]))
            tP = tM = tG = None
            for o in range(O):
                sP, sM, sG = P[succ[nodes, o]], M[succ[nodes, o]], G[succ[nodes, o]]
                iP = iM = iG = None
                for r in range(R):
                    w = rto[:, a, o, r][None, :]
                    sp = reach[:, a, r]
                    cont = (~es[sp] & ~ea[a])[None, :]
                    zero = (skip & (rto[:, a, o, r] == 0.0))[None, :]
                    pp = np.where(zero, 0.0, w * np.where(cont, sP[:, sp], 1.0))
                    pm = np.where(zero, 0.0, w * np.where(cont, sM[:, sp], 0.0))
                    pg = np.where(zero, 0.0, w * np.where(cont, sG[:, sp], 0.0))
                    iP, iM, iG = (pp, pm, pg) if r == 0 else (iP + pp, iM + pm, iG + pg)
                termG = gamma * iG
                tP, tM, tG = (iP, iM, termG) if o == 0 else (tP + iP, tM + iM, tG + termG)
            nP[nodes], nM[nodes], nG[nodes] = tP, 1.0 + tM, rbar[:, a][None, :] + tG
        P, M, G = nP, nM, nG
    return P, M, G


def forward_np(model, actions, succ, gamma, b, n0, H):
    """The run distribution pushed forward from (b, n0): per step the mass absorbed by an end and the expected reward.  Returns the
    curves P(T <= k), E[min(T, k)] and E[sum_{t < min(T, k)} gamma^t r_t] for k = 1..H."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, R = reach.shape
    O = rto.shape[2]
    es, ea = end_flags(model)
    N = len(actions)
    mu = np.zeros((N, S))
    mu[n0] = b
    cdf, steps, ret = np.zeros(H), np.zeros(H), np.zeros(H)
    absorbed = alive = total = 0.0
    disc = 1.0
    s = np.arange(S)
    for t in range(H):
        alive += mu.sum()
        reward = sum(float(mu[n] @ rbar[:, actions[n]]) for n in np.flatnonzero(mu.any(axis=1)))
        total += disc * reward
        nxt = np.zeros(N * S)
        for n in np.flatnonzero(mu.any(axis=1)):
            a = int(actions[n])
            for o in range(O):
                for r in range(R):
                    flow = mu[n] * rto[:, a, o, r]
                    stop = es[reach[:, a, r]] | ea[a]
                    absorbed += flow[stop].sum()
                    nxt += np.bincount(int(succ[n, o]) * S + reach[s[~stop], a, r], weights=flow[~stop], minlength=N * S)
        mu = nxt.reshape(N, S)
        cdf[t], steps[t], ret[t] = absorbed, alive, total
        disc *= gamma
    return cdf, steps, ret


def dot_fixed(b, x):
    """b . x in the kernel's fixed shape: thread t sums states t, t + 256, ... (b = 0 skipped), then the warp shuffle tree and the eight
    warp partials in order."""
    S = len(b)
    pad = (-S) % 256
    bb = np.concatenate([b, np.zeros(pad)]).reshape(-1, 256)
    xx = np.concatenate([x, np.zeros(pad)]).reshape(-1, 256)
    acc = np.zeros(256)
    for i in range(bb.shape[0]):
        acc = np.where(bb[i] != 0.0, acc + bb[i] * xx[i], acc)
    v = acc.reshape(8, 32).copy()
    for off in (16, 8, 4, 2, 1):
        v[:, :off] = v[:, :off] + v[:, off:2 * off]
    tot = 0.0
    for w in range(8):
        tot = tot + float(v[w, 0])
    return tot


# ---- models and controllers --------------------------------------------------------------------------------------------------------
def with_ends(model, end_states=None, end_actions=None):
    """A shallow copy of a fixture model (same tables and device handle) with other end states / actions."""
    m = copy.copy(model)
    if end_states is not None:
        m.end_states = list(end_states)
    if end_actions is not None:
        m.end_actions = list(end_actions)
    return m


def on(model, pg):
    """The controller `pg` over `model` (a copy: the cached graphs keep their own model)."""
    pg = copy.copy(pg)
    pg.model = model
    return pg


def planted(model):
    """End states at the argmax-Rbar states."""
    best = model.expected_rewards_table.max(axis=1)
    return with_ends(model, end_states=np.flatnonzero(best == best.max()).tolist())


_gap = {}


def gap_graph(tag):
    """The certified and the uncertified controller of a short seeded GapSolver run."""
    from pomdp_pbvi_exploration_b200 import GapSolver
    if tag not in _gap:
        model, gamma = fixture_model(tag)
        if tag == 'olfactory_wrap':
            pg, _, hist = GapSolver(gamma, 0.1, trials=16, max_depth=100, seed=0).solve(model, max_rounds=2)
        else:
            pg, _, hist = GapSolver(gamma, 0.01, trials=4, max_depth=10, seed=0).solve(model, max_rounds=2)
        _gap[tag] = (model, gamma, pg, hist.uncertified)
    return _gap[tag]


def cases():
    """(name, model with its end states / actions, gamma, PolicyGraph) of the bitwise checks."""
    out = []
    model, gamma, _, _, pg, _ = extracted('tiger')
    m = with_ends(model, end_actions=[1, 2])
    out.append(('tiger-end-actions', m, gamma, on(m, pg)))
    model, gamma, _, _, pg, _ = extracted('synth300')
    out.append(('synth300', model, gamma, pg))
    model, gamma, _, _, pg, _ = extracted('olfactory_fsvi')
    out.append(('olfactory-fsvi', model, gamma, pg))
    for tag in ('grid4x4', 'hallway', 'tigergrid'):
        model, gamma, _, _, pg, _ = extracted(tag)
        m = planted(model)
        out.append((tag + '-planted', m, gamma, on(m, pg)))
    model, gamma, pg, _ = gap_graph('hallway')
    m = planted(model)
    out.append(('hallway-gap-planted', m, gamma, on(m, pg)))
    return out


CASES = ['tiger-end-actions', 'synth300', 'olfactory-fsvi', 'grid4x4-planted', 'hallway-planted', 'tigergrid-planted', 'hallway-gap-planted']


def case(name):
    return next(c for c in cases() if c[0] == name)[1:]


def check_series(out, rows_np, B):
    """The last series entry is the fixed-shape b_j . row_H(n_j) of the returned rows, bitwise."""
    for j, n in enumerate(out.start_nodes):
        for stat, (curve, rows) in enumerate(zip((out.success_curve, out.steps_curve, out.return_curve), rows_np)):
            assert curve[j, -1] == dot_fixed(B[j], rows[n]), (j, stat)
    assert np.array_equal(out.success, out.success_curve[:, -1]) and np.array_equal(out.discounted_return, out.return_curve[:, -1])


# ---- GPU: the recursions against NumPy -----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('name', CASES)
def test_rows_match_numpy_in_the_kernel_order(name):
    model, gamma, pg = case(name)
    assert len(model.end_states) or len(model.end_actions)
    for k in (0, 1, 2, 7, 50):
        out = pg.outcomes(k)
        want = outcomes_np(model, pg.actions, pg.successors, gamma, k)
        for got, ref, stat in zip((out.success_rows, out.steps_rows, out.return_rows), want, 'PMG'):
            assert got.cpu().numpy().tobytes() == ref.tobytes(), (name, k, stat)
        assert out.success_curve.shape == (1, k) and out.start_nodes.tolist() == [int(pg.value(model.start_probabilities)[1][0])]
        if k:
            check_series(out, want, np.asarray(model.start_probabilities, dtype=np.float64)[None, :])


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'hallway', 'olfactory_fsvi'])
def test_without_ends_return_is_the_controller_sweep(tag):
    import torch
    model, gamma, _, _, pg, _ = extracted(tag)
    pg = on(with_ends(model, end_states=[], end_actions=[]), pg)
    dev = model.device
    W = torch.zeros((len(pg), model.state_count), dtype=torch.float64, device='cuda')
    for k in range(1, 8):
        W = dev.controller_sweep(W, gamma, pg.actions, pg.successors)
        out = pg.outcomes(k)
        assert out.return_rows.cpu().numpy().tobytes() == W.cpu().numpy().tobytes(), (tag, k)
        assert not bool(out.success_rows.any()) and not np.any(out.success_curve)
        # M_k = k up to rounding: RTO rows sum to 1 only within a few ulps on most models
        assert bool((torch.abs(out.steps_rows - k) <= 1e-10 * k).all())
        assert np.all(np.abs(out.steps_curve[0] - np.arange(1, k + 1)) <= 1e-10 * k)


# ---- GPU: the series against the run distribution, and against the certificate --------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('name', ['tiger-end-actions', 'synth300', 'hallway-planted', 'tigergrid-planted', 'olfactory-fsvi'])
def test_series_matches_forward_propagation(name):
    model, gamma, pg = case(name)
    H = 12 if name == 'olfactory-fsvi' else 40
    rng = np.random.default_rng(3)
    S = model.state_count
    B = np.stack([np.asarray(model.start_probabilities, dtype=np.float64), rng.dirichlet(np.ones(S)), np.eye(S)[rng.integers(S)]])
    nodes = np.array([int(pg.value(B[:1])[1][0]), rng.integers(len(pg)), rng.integers(len(pg))])
    out = pg.outcomes(H, beliefs=B, start_nodes=nodes)
    assert out.start_nodes.tolist() == nodes.tolist() and out.success_curve.shape == (3, H)
    k = np.arange(1, H + 1)
    for j in range(3):
        for got, want in zip((out.success_curve[j], out.steps_curve[j], out.return_curve[j]),
                             forward_np(model, pg.actions, pg.successors, gamma, B[j], nodes[j], H)):
            assert np.all(np.abs(got - want) <= 1e-12 * np.maximum(1.0, np.abs(want)) * k), (name, j, np.max(np.abs(got - want)))
    check_series(out, [r.cpu().numpy() for r in (out.success_rows, out.steps_rows, out.return_rows)], B)


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4', 'hallway', 'tigergrid', 'synth300'])
def test_return_without_ends_brackets_the_certified_value(tag):
    model, gamma, _, _, pg, hist = extracted(tag)
    pg = on(with_ends(model, end_states=[], end_actions=[]), pg)
    H = 400
    out = pg.outcomes(H)
    value = float(pg.value(model.start_probabilities)[0][0])
    g = float(out.discounted_return[0])
    tail = gamma ** H * float(np.max(np.abs(model.expected_rewards_table))) / (1 - gamma)
    assert value <= g + tail + 1e-12 * max(1.0, abs(g)), (tag, value, g, tail)
    tol = hist.final_change * gamma / (1 - gamma)
    assert g <= value + hist.shift + tol + tail + 1e-12 * max(1.0, abs(g)), (tag, value, g, hist.shift, tol)


# ---- GPU: a closed form and Monte Carlo -----------------------------------------------------------------------------------------
def test_tiger_table_layout():
    """What the closed form below reads from the tiger fixture: action 0 listens (reward -1, state kept, the matching observation with
    probability 0.85), and action 2 opens the door that pays 10 in state 0 and -100 in state 1."""
    model, _ = fixture_model('tiger')
    rbar, rto, reach = model.expected_rewards_table, model.reachable_transitional_observation_table, model.reachable_states
    assert rbar.tolist() == [[-1.0, -100.0, 10.0], [-1.0, 10.0, -100.0]]
    assert reach[:, 0, 0].tolist() == [0, 1] and rto[:, 0, :, 0].tolist() == [[0.85, 0.15], [0.15, 0.85]]
    assert np.all(rto[:, 0, :, 1] == 0.0)


@pytest.mark.gpu
def test_tiger_listen_until_left_closed_form():
    """Listen until the tiger is heard on the left, then open the right door (an end action).  From state s, with p_s = P(hear left | s),
    the number L of listens is geometric: P(T <= k) = 1 - (1 - p_s)^(k - 1) for k >= 1 and, as H grows,
    E[return] -> -(1 - E[gamma^L]) / (1 - gamma) + R_s E[gamma^L] with E[gamma^L] = p_s gamma / (1 - (1 - p_s) gamma)."""
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model('tiger')
    m = with_ends(model, end_actions=[1, 2])
    pg = PolicyGraph(m, [0, 2], [[1, 0], [0, 0]])
    H = 400
    out = pg.outcomes(H, start_nodes=[0], gamma=gamma)
    p = np.array([0.85, 0.15])
    R = np.array([10.0, -100.0])
    k = np.arange(1, H + 1)
    cdf = 0.5 * ((1 - (1 - p[0]) ** (k - 1)) + (1 - (1 - p[1]) ** (k - 1)))
    assert np.all(np.abs(out.success_curve[0] - cdf) <= 1e-12 * k)
    eg = p * gamma / (1 - (1 - p) * gamma)
    want = float(np.mean(-(1 - eg) / (1 - gamma) + R * eg))
    assert abs(out.discounted_return[0] - want) <= 1e-10 * abs(want), (out.discounted_return[0], want)
    assert abs(out.steps[0] - float(np.mean(1 / p + 1))) <= 1e-10
    check_curves(out)


def check_curves(out):
    P, M = out.success_curve, out.steps_curve
    assert np.all(np.diff(P, axis=1) >= 0.0) and np.all(P <= 1.0 + 1e-12) and np.all(P >= 0.0)
    inc = np.diff(M, axis=1)
    assert np.all(np.abs(inc - (1.0 - P[:, :-1])) <= 1e-12 * np.maximum(1.0, M[:, 1:])), float(np.max(np.abs(inc - (1.0 - P[:, :-1]))))
    assert np.all(np.abs(M[:, 0] - 1.0) <= 1e-12)                     # b . 1: the belief sums to 1 within rounding


def rollouts_np(model, pg, gamma, H, n, seed):
    """n roll-outs from b0 and its best node under the reference's termination rule: (reached an end, steps taken, discounted return)."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, O, R = rto.shape
    es, ea = end_flags(model)
    rng = np.random.default_rng(seed)
    p = np.asarray(model.start_probabilities, dtype=np.float64)
    s = rng.choice(S, size=n, p=p / p.sum())
    node = np.full(n, int(pg.value(p)[1][0]), dtype=np.int64)
    cdf = np.cumsum(rto.reshape(S, A, O * R), axis=2)
    alive = np.ones(n, dtype=bool)
    done, steps, ret = np.zeros(n, dtype=bool), np.zeros(n), np.zeros(n)
    disc = 1.0
    for _ in range(H):
        a = pg.actions[node]
        ret += np.where(alive, disc * rbar[s, a], 0.0)
        steps += alive
        u = rng.random(n)
        k = np.minimum((cdf[s, a] <= u[:, None]).sum(axis=1), O * R - 1)
        o, r = k // R, k % R
        s = reach[s, a, r]
        node = pg.successors[node, o]
        stop = alive & (es[s] | ea[a])
        done |= stop
        alive &= ~stop
        disc *= gamma
    return done, steps, ret


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['tiger-end-actions', 'olfactory-fsvi'])
def test_monte_carlo_agrees_with_the_exact_outcomes(name):
    model, gamma, pg = case(name)
    H, n = 300, 10000
    out = pg.outcomes(H)
    done, steps, ret = rollouts_np(model, pg, gamma, H, n, seed=11)
    p = float(out.success[0])
    se_p = max(np.sqrt(p * (1 - p) / n), 1e-12)
    assert abs(done.mean() - p) <= 4 * se_p, (name, done.mean(), p, se_p)
    for mc, exact in ((steps, out.steps[0]), (ret, out.discounted_return[0])):
        se = max(mc.std(ddof=1) / np.sqrt(n), 1e-12 * max(1.0, abs(exact)))
        assert abs(mc.mean() - exact) <= 4 * se, (name, mc.mean(), exact, se)
    check_curves(out)


# ---- GPU: edge cases -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_zero_steps_gives_zero_rows():
    model, gamma, pg = case('hallway-planted')
    out = pg.outcomes(0)
    for rows in (out.success_rows, out.steps_rows, out.return_rows):
        assert tuple(rows.shape) == (len(pg), model.state_count) and not bool(rows.any())
    assert out.success_curve.shape == (1, 0) and out.success.tolist() == [0.0] and out.steps.tolist() == [0.0]


@pytest.mark.gpu
def test_a_run_that_starts_in_an_end_state_takes_its_first_step():
    model, gamma, pg = case('grid4x4-planted')
    rbar, rto, reach = model.expected_rewards_table, model.reachable_transitional_observation_table, model.reachable_states
    es, _ = end_flags(model)
    e = int(model.end_states[0])
    out = pg.outcomes(5, beliefs=np.eye(model.state_count)[e], start_nodes=[0])
    a = int(pg.actions[0])
    assert out.steps_curve[0, 0] == 1.0 and out.return_curve[0, 0] == rbar[e, a]
    to_end = float(rto[e, a][:, es[reach[e, a]]].sum())
    assert abs(out.success_curve[0, 0] - to_end) <= 1e-14
    check_curves(out)


@pytest.mark.gpu
def test_every_action_an_end_action_stops_after_one_step():
    model, gamma, _, _, pg, _ = extracted('hallway')
    pg = on(with_ends(model, end_actions=range(model.action_count)), pg)
    out = pg.outcomes(6)
    P, M, G = (r.cpu().numpy() for r in (out.success_rows, out.steps_rows, out.return_rows))
    assert np.all(M == 1.0) and np.all(np.abs(P - 1.0) <= 1e-12)
    assert np.array_equal(G, model.expected_rewards_table[:, pg.actions].T)
    assert np.all(out.steps_curve == out.steps_curve[:, :1]) and np.all(out.success_curve == out.success_curve[:, :1])


@pytest.mark.gpu
def test_large_olfactory_controller_is_deterministic_and_runs_long_horizons():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma, pg, _ = gap_graph('olfactory_wrap')
    rng = np.random.default_rng(5)
    N = 3000                                                           # a seeded controller: many nodes, many live successors
    big = PolicyGraph(model, rng.integers(0, model.action_count, N), rng.integers(0, N, (N, model.observation_count)))
    a = big.outcomes(50, start_nodes=[0], gamma=gamma)
    b = big.outcomes(50, start_nodes=[0], gamma=gamma)
    for x, y in zip((a.success_rows, a.steps_rows, a.return_rows), (b.success_rows, b.steps_rows, b.return_rows)):
        assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes()
    assert a.success_curve.tobytes() == b.success_curve.tobytes() and a.return_curve.tobytes() == b.return_curve.tobytes()
    long = pg.outcomes(2000)
    check_curves(long)
    assert np.all(np.isfinite(long.return_curve)) and long.success[0] > 0.0
    B = np.asarray(model.start_probabilities, dtype=np.float64)[None, :]
    check_series(long, [r.cpu().numpy() for r in (long.success_rows, long.steps_rows, long.return_rows)], B)
