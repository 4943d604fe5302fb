"""
Pruning of dominated controller nodes (pbvi_dominating_row, PolicyGraph.prune_dominated, the GapSolver's append-only graph) and of
dominated upper-bound pairs (pbvi_sawtooth_witness, UpperBound.prune).  Checked against
  * brute-force NumPy restatements of both witness rules (exact equality; the sawtooth terms with one rounding of v0 + scale * m, as
    the kernels compute them) and pbvi_sawtooth_lists on the store without the pair;
  * the values at b0, at stored and random beliefs and at successors before and after a prune (bitwise where the docstrings promise it),
    the certificate W <= T_pi W of the pruned controller, and GapSolver(prune_growth) against the solve without pruning.
"""
import ctypes
import types
from fractions import Fraction

import numpy as np
import pytest

from test_gap_solver import check_rounds, check_uncertified
from test_policy_graph import GOLDEN9, check_certificate, extracted
from test_upper_bound import fib_of, fixture_model, sawtooth_np, successors_np


def fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


# ---- CPU --------------------------------------------------------------------------------------------------------------------------
def test_prune_entry_points_reject_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    buf = (ctypes.c_double * 8)()
    p = ctypes.addressof(buf)
    BAD = _native.PBVI_ERR_BAD_ARG
    assert lib.pbvi_dominating_row(None, p, 3, p, None) == BAD and b'handle is NULL' in lib.pbvi_last_error()
    assert lib.pbvi_dominating_row(None, p, -1, p, None) == BAD and b'non-negative' in lib.pbvi_last_error()
    for rows, wit in ((None, p), (p, None)):
        assert lib.pbvi_dominating_row(None, rows, 3, wit, None) == BAD and b'NULL pointer' in lib.pbvi_last_error()
    assert lib.pbvi_dominating_row(None, None, 0, None, None) == BAD and b'handle is NULL' in lib.pbvi_last_error()

    def saw(m=None, n_ub=3, **kw):
        a = [kw.get(k, p) for k in ('corner', 'idx', 'val', 'count', 'dot', 'vals')]
        return lib.pbvi_sawtooth_witness(m, *a, n_ub, kw.get('mn', p), kw.get('arg', p), kw.get('own', p), None)
    assert saw() == BAD and b'handle is NULL' in lib.pbvi_last_error()
    assert saw(n_ub=-1) == BAD and b'non-negative' in lib.pbvi_last_error()
    for name in ('corner', 'idx', 'val', 'count', 'dot', 'vals', 'mn', 'arg', 'own'):
        assert saw(**{name: None}) == BAD and b'NULL pointer' in lib.pbvi_last_error(), name
    assert saw(n_ub=0, idx=None, mn=None) == BAD and b'handle is NULL' in lib.pbvi_last_error()


def resolve_np(w):
    """The chain rule restated: follow each chain until a kept entry (w = -1) or a repeat; a cycle keeps its lowest index, and the
    first entry (in index order) that reaches a cycle decides which cycle member that is."""
    n = len(w)
    target = [-1] * n
    for i in range(n):
        seen, j = [], i
        while target[j] < 0 and w[j] >= 0 and j not in seen:
            seen.append(j)
            j = w[j]
        end = target[j] if target[j] >= 0 else (j if w[j] < 0 else min(seen[seen.index(j):]))
        target[end] = end
        for k in seen:
            target[k] = end
    return np.asarray(target)


def test_witness_chains_resolve_to_kept_entries():
    from pomdp_pbvi_exploration_b200.bounds import resolve_witnesses
    # 0 kept; 1 -> 0; 2 -> 1 -> 0 (a chain of three); 3 -> 5 -> 4 (4 kept); 6 <-> 7 (a cycle: 6 stays); 8 -> 9 -> 10 -> 9 (cycle {9, 10})
    w = np.array([-1, 0, 1, 5, -1, 4, 7, 6, 9, 10, 9])
    got = resolve_witnesses(w)
    assert got.tolist() == [0, 0, 0, 4, 4, 4, 6, 6, 9, 9, 9]
    w2 = w.copy()
    w2[1] = -1                                                     # a protected entry is kept and ends the chains through it
    assert resolve_witnesses(w2).tolist() == [0, 1, 1, 4, 4, 4, 6, 6, 9, 9, 9]
    rng = np.random.default_rng(5)
    for n in (1, 2, 7, 60, 400):
        for _ in range(20):
            w = np.where(rng.random(n) < 0.3, -1, rng.integers(0, n, n))
            w[np.arange(n) == w] = -1
            got = resolve_witnesses(w)
            assert np.array_equal(got, resolve_np(w.tolist()))
            kept = got == np.arange(n)
            assert np.all(kept[got]) and np.all(kept[w < 0])


def redirect_np(actions, succ, target):
    keep = [i for i in range(len(actions)) if target[i] == i]
    pos = {k: p for p, k in enumerate(keep)}
    return (np.asarray(keep), np.asarray([actions[k] for k in keep]),
            np.asarray([[pos[target[s]] for s in succ[k]] for k in keep]).reshape(len(keep), succ.shape[1]))


def test_successors_are_redirected_and_node_of_rebuilt():
    import torch
    from pomdp_pbvi_exploration_b200.bounds import resolve_witnesses
    from pomdp_pbvi_exploration_b200.gap_solver import _AppendOnlyGraph
    from pomdp_pbvi_exploration_b200.policy_graph import node_index, redirect_dominated
    rng = np.random.default_rng(11)
    for N, O in ((6, 2), (50, 3), (300, 1)):
        actions = rng.integers(0, 2, N)
        succ = rng.integers(0, N, (N, O))
        succ[:, 0] = 0                                             # node-0 edges (impossible observations) are redirected as well
        w = np.full(N, -1)
        pick = rng.random(N) < 0.5
        w[pick] = rng.integers(0, N, int(pick.sum()))
        w[w == np.arange(N)] = -1
        w[(w > np.arange(N)) & (rng.random(N) < 0.5)] = -1       # mostly downward chains, some upward, no self
        keep, act, s2 = redirect_dominated(actions, succ, w)
        k_np, a_np, s_np = redirect_np(actions, succ, resolve_witnesses(w))
        assert np.array_equal(keep, k_np) and np.array_equal(act, a_np) and np.array_equal(s2, s_np)
        # the append-only graph on a stand-in device that returns the same witnesses
        S = 4
        rows = torch.arange(N * S, dtype=torch.float64).reshape(N, S)
        fake = types.SimpleNamespace(state_count=S,
                                     device=types.SimpleNamespace(dominating_row=lambda X, w=w: torch.as_tensor(w, dtype=torch.int32)))
        g = _AppendOnlyGraph(fake, 0.9, actions, succ, rows)
        removed = g.prune()
        assert removed == N - len(keep) and g.n == len(keep)
        assert np.array_equal(np.asarray(g.actions), a_np) and np.array_equal(np.stack(g.successors), s_np)
        assert torch.equal(g.rows, rows[torch.as_tensor(keep)])
        assert g.node_of == node_index(a_np, list(s_np))
        table = np.concatenate([a_np[:, None], s_np], axis=1)
        for t, node in g.node_of.items():                          # a tuple two nodes now share maps to the lower one; both stay
            assert node == np.flatnonzero(np.all(table == np.asarray(t)[None, :], axis=1))[0]


def test_gap_solver_rejects_a_bad_growth_factor():
    from pomdp_pbvi_exploration_b200 import GapSolver
    for f in (1.0, 0.5, -2.0, float('nan')):
        with pytest.raises(ValueError, match='prune_growth'):
            GapSolver(0.95, 0.1, prune_growth=f)
    assert GapSolver(0.95, 0.1).prune_growth is None


# ---- GPU: pbvi_dominating_row ------------------------------------------------------------------------------------------------------
def dominating_np(X):
    n = len(X)
    ge = np.all(X[:, None, :] >= X[None, :, :], axis=2)           # [j, i]: X_j >= X_i everywhere (NaN fails)
    gt = np.any(X[:, None, :] > X[None, :, :], axis=2)
    j = np.arange(n)[:, None]
    i = np.arange(n)[None, :]
    ok = ge & (j != i) & ((j < i) | gt)
    return np.where(ok.any(axis=0), np.argmax(ok, axis=0), -1)


def planted_rows(rng, n, S):
    X = rng.integers(0, 3, (n, S)).astype(np.float64) + 0.25 * rng.integers(0, 2, (n, S))
    if n >= 12:
        X[3] = X[7]                                                # exact duplicates (both directions)
        X[9] = X[2]
        X[10] = X[4]
        X[10, S // 2] -= 0.5                                       # equal except at one state
        X[11] = X[5] + 1.0                                         # a chain of three: 5 < 11 < 1
        X[1] = X[11] + 0.5
        X[6, 0] = np.nan                                           # a NaN row and a row equal to it elsewhere
        X[8] = X[6]
        X[8, 0] = -1.0
        X[0] = 0.0                                                 # +-0.0: equal rows
        X[n - 1] = -0.0
    return X


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['cheese', 'hallway'])                    # S = 11 and S = 60: both sides of the 32-state chunk
@pytest.mark.parametrize('n', [1, 31, 32, 33, 1100])
def test_dominating_row_matches_numpy(tag, n):
    import torch
    model, _ = fixture_model(tag)
    dev = model.device
    rng = np.random.default_rng(n)
    X = planted_rows(rng, n, model.state_count)
    got = dev.dominating_row(torch.as_tensor(X, device='cuda')).cpu().numpy()
    want = dominating_np(X)
    assert np.array_equal(got, want), (tag, n, np.flatnonzero(got != want)[:5])
    if n >= 12:
        assert got[6] == -1 and not np.any(got == 6)            # a NaN row has no witness and is none
        assert 0 <= got[7] <= 3 and got[3] != 7                 # of two equal rows the first stays
        assert got[n - 1] == 0 and got[0] != n - 1              # +0.0 and -0.0 rows are equal
    assert dev.dominating_row(torch.zeros((0, model.state_count), dtype=torch.float64, device='cuda')).shape == (0,)


# ---- GPU: pbvi_sawtooth_witness ----------------------------------------------------------------------------------------------------
def witness_np(rows, vals, dot):
    """(min_{j != i} s_j(b_i), its first j or -1 when not below v0(b_i), s_i(b_i)) with v0(b_i) = dot_i and one rounding per term
    (v0 + scale * m as one fma, computed exactly with fractions for the terms near the minimum; s_i(b_i) has m = 1 exactly)."""
    n = len(rows)
    scale = vals - dot
    own = dot + scale
    mn, arg = np.full(n, np.inf), np.full(n, -1)
    pos = rows > 0
    den = np.where(pos, rows, 1.0)
    for i in range(n):
        m = np.where(pos, rows[i][None, :] / den, np.inf).min(axis=1)
        approx = dot[i] + scale * m
        approx[i] = np.inf
        if n == 1:
            continue
        top = float(np.min(approx))
        for j in np.flatnonzero(approx <= top + 1e-9 * max(1.0, abs(top))):
            t = dot[i] + scale[j] * 0.0 if m[j] == 0.0 else fma(scale[j], m[j], dot[i])
            if t < mn[i]:
                mn[i], arg[i] = t, j
        if not mn[i] < dot[i]:
            arg[i] = -1
    return mn, arg, own


def improved_store(tag):
    """An UpperBound after two improve passes over (the first 300 of) a seeded solve's beliefs."""
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma, _, B, _, _ = extracted(tag)
    ub = UpperBound(model, fib_of(tag)[0], gamma)
    ub.improve(B[:300], passes=2)
    return model, gamma, ub


def trial_store(tag):
    """The UpperBound three GapSolver rounds leave (trial beliefs: nested supports along a trial are common)."""
    from pomdp_pbvi_exploration_b200 import GapSolver
    model, gamma = fixture_model(tag)
    _, ub, _ = GapSolver(gamma, 1e-3, trials=8, max_depth=30, seed=0).solve(model, max_rounds=3)
    return model, gamma, ub


def check_witness(dev, ub, rows, vals):
    import torch
    idx, val, count, dot, v, n = ub._lists()
    mn, arg, own = dev.sawtooth_witness(ub.corner_values, idx, val, count, dot, v, n)
    mn, arg, own = mn.cpu().numpy(), arg.cpu().numpy(), own.cpu().numpy()
    dot_h = dot[:n].cpu().numpy()
    v0 = dev.sawtooth_lists(ub.corner_values, idx, val, count, dot, v, 0, torch.as_tensor(rows, device='cuda')).cpu().numpy()
    assert v0.tobytes() == dot_h.tobytes()                        # v0(b_i) of a dense query is the list's dot, bitwise
    w_mn, w_arg, w_own = witness_np(rows, vals, dot_h)
    assert mn.tobytes() == w_mn.tobytes() and own.tobytes() == w_own.tobytes()
    assert np.array_equal(arg, w_arg), np.flatnonzero(arg != w_arg)[:5]
    return mn, arg, own


@pytest.mark.gpu
@pytest.mark.parametrize('store', [improved_store, trial_store])
@pytest.mark.parametrize('tag', ['hallway', 'tigergrid'])
def test_sawtooth_witness_matches_numpy_on_improved_stores(tag, store):
    import torch
    model, gamma, ub = store(tag)
    dev = model.device
    n = len(ub)
    assert n > 10
    rows, vals = ub.belief_array.cpu().numpy(), ub.value_array.cpu().numpy()
    mn, arg, own = check_witness(dev, ub, rows, vals)
    for i in range(0, n, max(1, n // 16)):                         # the sawtooth of the whole store at b_i, from the same terms
        want = min(float(ub._dot[i]), float(mn[i]), float(own[i]))
        assert float(dev.sawtooth_lists(ub.corner_values, *ub._lists(), torch.as_tensor(rows[i:i + 1], device='cuda'))[0]) == want
        assert abs(want - sawtooth_np(rows[i], ub.corner_values.cpu().numpy(), rows, vals)) <= 1e-12 * max(1.0, abs(want))
    # d_min[i] is the minimum over j != i of the terms pbvi_sawtooth_lists forms for the query b_i (with v0 the corner term)
    idx, val, count, dot, v, _ = ub._lists()
    for i in sorted({0, n // 3, n - 1, *np.flatnonzero(arg >= 0)[:3].tolist()}):
        others = torch.as_tensor([j for j in range(n) if j != i], device='cuda')
        got = dev.sawtooth_lists(ub.corner_values, idx[others].contiguous(), val[others].contiguous(), count[others].contiguous(),
                                 dot[others].contiguous(), v[others].contiguous(), n - 1, torch.as_tensor(rows[i:i + 1], device='cuda'))
        assert float(got[0]) == min(float(dot[i]), float(mn[i])), (tag, i)
        assert abs(float(own[i]) - float(v[i])) <= 1e-12 * max(1.0, abs(float(v[i])))


@pytest.mark.gpu
def test_sawtooth_witness_matches_numpy_on_synthetic_stores():
    import torch
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma = fixture_model('hallway')
    S = model.state_count
    ub = UpperBound(model, fib_of('hallway')[0], gamma)
    rng = np.random.default_rng(3)
    rows = []
    for k in range(40):                                            # nested supports: prefixes of one permutation
        perm = rng.permutation(S)
        for size in (S, 20, 5, 1):
            r = np.zeros(S)
            r[perm[:size]] = rng.random(size) + 0.1
            rows.append(r / r.sum())
    for s in range(0, S, 7):                                       # single-state supports (corners)
        r = np.zeros(S)
        r[s] = 1.0
        rows.append(r)
    rows.append(rows[5].copy())                                    # equal beliefs
    rows.append(rows[5].copy())
    rows = np.asarray(rows)
    corner = ub.corner_values.cpu().numpy()
    vals = rows @ corner - rng.random(len(rows)) * 0.5
    vals[-1] = vals[-2]                                            # equal pairs
    n = len(rows)
    ub._reserve(n)
    R = torch.as_tensor(rows, device='cuda')
    ub._rows[:n] = R
    ub._vals[:n] = torch.as_tensor(vals, device='cuda')
    dev = model.device
    dev.support_lists(ub._rows[:n], ub.corner_values, ub._idx[:n], ub._val[:n], ub._count[:n], ub._dot[:n])
    ub._n = n
    mn, arg, own = check_witness(dev, ub, rows, ub.value_array.cpu().numpy())
    assert arg[n - 1] >= 0 and arg[n - 2] >= 0                    # equal pairs: each has the other (or the third copy) below it
    assert (arg >= 0).sum() > n // 4


# ---- GPU: PolicyGraph.prune_dominated ----------------------------------------------------------------------------------------------
def probe_beliefs(model, B, seed):
    rng = np.random.default_rng(seed)
    Rn = rng.random((64, model.state_count)) ** 4
    Rn /= Rn.sum(axis=1, keepdims=True)
    succ, mass = successors_np(model, B[0])
    succ = succ.reshape(-1, model.state_count)[mass.reshape(-1) > 0]
    return np.concatenate([model.start_probabilities[None, :], B, Rn, succ])


@pytest.mark.gpu
@pytest.mark.parametrize('source', ['extracted', 'improved'])
@pytest.mark.parametrize('tag', ['hallway', 'tigergrid'])
def test_prune_dominated_keeps_values_and_certificate(tag, source):
    import torch
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma, _, B, pg, _ = extracted(tag)
    if source == 'improved':
        pg, _ = pg.improve(B, 2)
    dev = model.device
    rows_before = pg.rows.clone()
    P = probe_beliefs(model, B, 1)
    before = pg.value(P)[0].cpu().numpy()
    old_b0 = float(before[0])
    pr = pg.prune_dominated()
    assert torch.equal(pg.rows, rows_before) and pr is not pg               # the original graph is not changed
    assert len(pr) <= len(pg) and pr.gamma == pg.gamma
    assert pr.value(P)[0].cpu().numpy().tobytes() == before.tobytes()
    act = torch.as_tensor(pr.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(pr.successors, dtype=torch.int32, device='cuda').contiguous()
    assert float(dev.controller_sweep(pr.rows, gamma, act, succ, want_stats=True)[1][1]) <= 0.0
    check_certificate(model, gamma, pr)
    assert np.all(dev.dominating_row(pr.rows).cpu().numpy() == -1)
    assert len(pr.prune_dominated()) == len(pr)
    fresh = PolicyGraph(model, pr.actions, pr.successors)
    _, h = fresh.evaluate(gamma, eps=1e-9)
    slack = h.shift + 1e-9 / (1.0 - gamma) ** 2
    assert float(fresh.value(model.start_probabilities)[0][0]) >= old_b0 - slack


# ---- GPU: UpperBound.prune ---------------------------------------------------------------------------------------------------------
def check_index(ub):
    keys = ub.model.device.row_hash(ub.belief_array).cpu().numpy()
    assert len(ub._index) == len(ub)
    for p, k in enumerate(keys.tolist()):
        assert ub._index[(int(k[0]), int(k[1]))] == p


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['hallway', 'tigergrid'])
def test_upper_bound_prune_keeps_the_bound(tag):
    import torch
    model, gamma, ub = trial_store(tag)
    n0 = len(ub)
    stored = ub.belief_array.cpu().numpy()
    P = probe_beliefs(model, stored, 2)
    before = ub.evaluate(P).cpu().numpy()
    b0 = model.start_probabilities[None, :]
    up_b0 = ub.evaluate(b0).cpu().numpy().tobytes()
    removed = ub.prune()
    assert removed > 0 and len(ub) == n0 - removed, (tag, removed, n0)
    after = ub.evaluate(P).cpu().numpy()
    assert np.all(after >= before), float(np.min(after - before))
    assert np.all(after <= before + 1e-12 * np.maximum(1.0, np.abs(before))), float(np.max(after - before))
    assert ub.evaluate(b0).cpu().numpy().tobytes() == up_b0
    check_index(ub)
    # later backups: as if the dropped pairs had never been stored
    kept = {r.tobytes() for r in ub.belief_array.cpu().numpy()}
    gone = np.asarray([r for r in stored if r.tobytes() not in kept])
    n1 = len(ub)
    cur = ub.evaluate(gone).cpu().numpy()
    u = model.device.upper_backup(torch.as_tensor(gone, device='cuda'), ub._F, gamma, ub.corner_values, *ub._lists())[0].cpu().numpy()
    ub.improve(gone)
    added = int(np.sum(u < cur))
    assert len(ub) == n1 + added, (tag, n1, added, len(ub))
    check_index(ub)
    if added:
        tail = ub.belief_array[n1:].cpu().numpy()
        assert {r.tobytes() for r in tail} <= {r.tobytes() for r in gone}
    n2 = len(ub)
    vals = ub.value_array.cpu().numpy().copy()
    ub.improve(ub.belief_array[:n1].clone())                       # kept beliefs are lowered in place
    assert len(ub) == n2 and np.all(ub.value_array.cpu().numpy() <= vals)


@pytest.mark.gpu
def test_upper_bound_prune_protects_the_keep_beliefs():
    model, gamma, ub = trial_store('hallway')
    keep = ub.belief_array[::7].clone()
    want = ub.evaluate(keep).cpu().numpy().tobytes()
    ub.prune(keep_beliefs=keep)
    assert ub.evaluate(keep).cpu().numpy().tobytes() == want


# ---- GPU: GapSolver(prune_growth) --------------------------------------------------------------------------------------------------
def history_of(hist):
    rounds = [{k: v for k, v in r.items() if k not in ('phase_seconds', 'seconds')} for r in hist.rounds]
    return rounds, hist.lower, hist.upper


@pytest.mark.gpu
def test_pruned_tiger_solve_reaches_its_target_around_the_exact_value():
    from test_upper_bound import tiger_exact_value
    from pomdp_pbvi_exploration_b200 import GapSolver
    model, gamma = fixture_model('tiger')
    pg, ub, hist = GapSolver(gamma, 0.1, trials=4, max_depth=60, seed=0, prune_growth=1.1).solve(model, max_rounds=40)
    assert hist.reached and hist.gap <= 0.1, (hist.lower, hist.upper, len(hist.rounds))
    check_rounds(hist)
    check_uncertified(model, gamma, hist)
    check_certificate(model, gamma, pg)
    v0 = tiger_exact_value(model, gamma, np.array([float(model.start_probabilities[1])]))[0]
    assert hist.lower <= v0 + 1e-9 <= hist.upper + 2e-9


@pytest.mark.gpu
@pytest.mark.parametrize('tag', GOLDEN9)
def test_pruned_solve_stays_sound_on_golden_models(tag):
    from pomdp_pbvi_exploration_b200 import GapSolver, UpperBound
    model, gamma = fixture_model(tag)
    fib, _ = fib_of(tag)
    pg, ub, hist = GapSolver(gamma, 1e-3, trials=4, max_depth=25, seed=1, prune_growth=1.1).solve(model, max_rounds=4,
                                                                                                   upper=UpperBound(model, fib, gamma))
    check_rounds(hist)
    check_uncertified(model, gamma, hist)
    check_certificate(model, gamma, pg)
    assert all('prune' in r['phase_seconds'] and r['pruned_nodes'] >= 0 and r['pruned_pairs'] >= 0 for r in hist.rounds)


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['hallway', 'tigergrid'])
def test_pruned_solve_is_deterministic_and_none_is_the_plain_solve(tag):
    from pomdp_pbvi_exploration_b200 import GapSolver
    model, gamma = fixture_model(tag)

    def run(**kw):
        pg, ub, hist = GapSolver(gamma, 1e-3, trials=6, max_depth=20, seed=3, **kw).solve(model, max_rounds=4)
        return (pg.actions.tolist(), pg.successors.tolist(), pg.rows.cpu().numpy().tobytes(), ub.value_array.cpu().numpy().tobytes(),
                history_of(hist)), hist
    a, h = run(prune_growth=1.1)
    b, _ = run(prune_growth=1.1)
    assert a == b
    check_rounds(h)
    assert sum(r['pruned_nodes'] + r['pruned_pairs'] for r in h.rounds) > 0
    plain, hp = run()
    assert plain == run(prune_growth=None)[0]
    assert all('pruned_nodes' not in r and 'prune' not in r['phase_seconds'] for r in hp.rounds)
