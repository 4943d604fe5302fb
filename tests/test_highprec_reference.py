"""
The extended-precision reference (oracle/highprec.py) on the CPU: its bounds are sound (the float64 oracle, a different evaluation
order, satisfies the contract everywhere) and tight enough to mean something (a value moved by three times its bound, or a decided
v* swapped, is rejected; the bounds sit orders of magnitude below the 1e-9 slack of the float64 comparisons).
"""
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_golden
from oracle import highprec as hp
from oracle import pbvi_oracle as orc

GOLDEN = ['tiger', 'grid4x4', 'grid4x4_noloop', 'tigergrid', 'hallway', 'cheese', 'grid4x3', 'cit', 'synth300', 'olfactory_wrap']


def golden_case(tag):
    m, g = load_golden('model_' + tag), load_golden('backup_' + tag)
    return m['reach'].astype(np.int64), m['rto'], m['rbar'], float(m['gamma']), g['beliefs'], g['alphas']


def synthetic_case(S, A, O, R, nB, nV, seed, negative=False):
    """The configs[4] recipe of the GPU tests: random landing states, non-uniform transition probabilities, impossible observations."""
    rng = np.random.default_rng(seed)
    reach = rng.integers(0, S, (S, A, R))
    probs = rng.random((S, A, R)) + 0.05
    probs /= probs.sum(2, keepdims=True)
    obs = rng.random((S, A, O))
    obs /= obs.sum(2, keepdims=True)
    obs[rng.random((S, A, O)) < 0.3] = 0.0
    rto = orc.build_rto(reach, probs, obs)
    rbar = orc.expected_rewards(rto, orc.end_state_reachable_rewards(reach, O, [S // 2]))
    if negative:
        rbar = rbar - 0.3 * rng.random((S, A))
    B = np.zeros((nB, S))
    for i in range(nB):
        k = min(S, [S, 40, 5, 1][i % 4])
        idx = rng.choice(S, k, replace=False)
        B[i, idx] = rng.dirichlet(np.ones(k))
    V = rng.random((nV, S)) * (2.0 if negative else 1.0) - (1.0 if negative else 0.0)
    return reach, rto, rbar, 0.95, B, V


SYNTHETIC = {'s1': (60, 3, 2, 1, 30, 40, 1, False), 's2': (90, 2, 3, 3, 20, 25, 2, True), 's3': (300, 4, 5, 1, 17, 70, 3, True)}


def case(name):
    return golden_case(name) if name in GOLDEN else synthetic_case(*SYNTHETIC[name])


def test_reference_imports_nothing_from_the_product():
    text = open(os.path.join(ROOT, 'oracle', 'highprec.py')).read()
    assert not re.search(r'^\s*(from|import)\s+(pomdp_pbvi_exploration_b200|oracle)\b', text, flags=re.M)
    assert np.finfo(np.longdouble).eps <= 1e-18


@pytest.mark.parametrize('name', GOLDEN + list(SYNTHETIC))
def test_float64_oracle_satisfies_the_contract(name):
    reach, rto, rbar, gamma, B, V = case(name)
    ref = orc.backup(reach, rto, rbar, gamma, B, V)
    rows = ref['alpha'] if reach.shape[2] == 1 else None        # NumPy's einsum sums over r in its own order
    hp.check_backup(reach, rto, rbar, gamma, B, V, ref['v_star'], ref['values'], ref['a_star'], rows)
    sel = ref['v_star'][np.arange(len(B)), ref['a_star']]
    ent, eb = hp.alpha_entries(reach, rto, rbar, gamma, V, ref['a_star'], sel)
    hp.check_close(ref['alpha'], ent, eb, what='alpha_a entries')
    mx, arg = orc.max_values(B, V)
    ex, bd, zero = hp.plain_scores(B, V)
    hp.check_argmax(ex, bd, arg, zero, what='max_values')
    hp.check_close(mx, np.take_along_axis(ex, arg[:, None], 1)[:, 0], np.take_along_axis(bd, arg[:, None], 1)[:, 0])


@pytest.mark.parametrize('name', ['hallway', 'cit', 's2', 's3'])
def test_contract_rejects_a_moved_value_and_a_swapped_decided_vstar(name):
    reach, rto, rbar, gamma, B, V = case(name)
    ref = orc.backup(reach, rto, rbar, gamma, B, V)
    ev, evb = hp.values(reach, rto, rbar, gamma, B, V, ref['v_star'])
    moved = ref['values'].copy()
    i = np.unravel_index(np.argmax(np.abs(ev)), ev.shape)
    moved[i] = float(ev[i] + 3 * evb[i])
    with pytest.raises(AssertionError, match='value'):
        hp.check_backup(reach, rto, rbar, gamma, B, V, ref['v_star'], moved)
    sc = hp.scores(reach, rto, B, V)
    srt = np.sort(sc[0], axis=3)
    decided = (srt[..., -1] - srt[..., -2]) > 2 * np.max(sc[1], axis=3)
    assert decided.any()
    j = tuple(np.argwhere(decided)[-1])
    swapped = ref['v_star'].copy()
    swapped[j] = int(np.argsort(sc[0][j])[-2])
    with pytest.raises(AssertionError, match='v\\*'):
        hp.check_backup(reach, rto, rbar, gamma, B, V, swapped, sc=sc)


def test_bounds_are_far_below_the_float64_slack():
    """On the golden backups the certified bound of a value is below 1e-11 of its magnitude: a term dropped by a kernel that is worth
    1e-9 of the value -- invisible to a 1e-9 comparison -- is a hundred bounds away."""
    for name in GOLDEN:
        reach, rto, rbar, gamma, B, V = golden_case(name)
        ref = orc.backup(reach, rto, rbar, gamma, B, V)
        ev, evb = hp.values(reach, rto, rbar, gamma, B, V, ref['v_star'])
        assert np.max(evb / np.maximum(np.abs(ev.astype(np.float64)), 1e-300)) < 1e-11, name


def test_subnormal_and_tiny_terms_are_within_the_bound():
    """A belief made of 1e-310 entries (subnormal products) and one whose only mass on a chunk is 1e-13: the bound keeps its absolute
    part far below either term, so dropping it is visible."""
    reach, rto, rbar, gamma, B, V = synthetic_case(40, 2, 2, 1, 4, 6, 5)
    B[0] = 0.0
    B[0, [3, 17]] = 1e-310
    B[1] = 0.0
    B[1, 0] = 1.0 - 1e-13
    B[1, 21] = 1e-13
    ref = orc.backup(reach, rto, rbar, gamma, B, V)
    ev, evb = hp.values(reach, rto, rbar, gamma, B, V, ref['v_star'])
    assert np.all(evb[0] < 1e-318)
    hp.check_close(ref['values'], ev, evb)
    dropped = ref['values'].copy()
    dropped[1] -= float(1e-13 * hp.alpha_entries(reach, rto, rbar, gamma, V, np.arange(2), ref['v_star'][1])[0][:, 21].max())
    with pytest.raises(AssertionError):
        hp.check_close(dropped, ev, evb)


# ---- upper bounds -----------------------------------------------------------------------------------------------------------------
def model_ns(reach, rto, rbar):
    """The attributes test_upper_bound's NumPy restatements read."""
    from types import SimpleNamespace
    return SimpleNamespace(reachable_states=reach, reachable_transitional_observation_table=rto, expected_rewards_table=rbar)


def upper_case(name, seed=0):
    """(model, gamma, beliefs, F, store rows, store values): F = the case's alphas lifted above zero (its elementwise maximum is the
    corner), the store every other belief with values below its corner value so that the stored terms bind."""
    reach, rto, rbar, gamma, B, V = case(name)
    rng = np.random.default_rng(seed)
    F = V + 1.0 + rng.random(V.shape)
    corner = F.max(axis=0)
    Q = B[1::2] if len(B) > 1 else B
    S = B.shape[1]
    # stored beliefs on the support of a query (its entries reweighted): their ratios are positive and a stored term binds
    near = Q[:4] * (0.5 + rng.random((min(4, len(Q)), S)))
    rows = np.concatenate([B[::2], near / near.sum(axis=1, keepdims=True)])
    vals = rows @ corner - (0.05 + 0.5 * rng.random(len(rows))) * np.abs(rows @ corner)
    return model_ns(reach, rto, rbar), gamma, Q, F, rows, vals


UPPER_CASES = ['tiger', 'grid4x4', 'tigergrid', 'hallway', 'cheese', 'grid4x3', 'cit', 'synth300', 'olfactory_wrap', 's1', 's2', 's3']


@pytest.mark.parametrize('name', UPPER_CASES)
def test_float64_upper_restatements_satisfy_the_contract(name):
    """sawtooth_np, upper_backup_np and step_np (NumPy's order: BLAS dots, sequential sums) fall inside the intervals everywhere."""
    from test_gap_solver import choose_np, step_np
    from test_upper_bound import sawtooth_np, successors_np, upper_backup_np
    model, gamma, B, F, rows, vals = upper_case(name)
    corner = F.max(axis=0)
    lo, hi = hp.sawtooth(corner, rows, vals, B)
    hp.check_interval([sawtooth_np(b, corner, rows, vals) for b in B], (lo, hi), what='sawtooth')
    assert np.all(lo <= hi)
    X = F - 1.5
    rng = np.random.default_rng(1)
    for b in B[:6]:
        succ, mass = successors_np(model, b)
        ref = hp.upper_q(b[None], model.expected_rewards_table, gamma, succ[None], mass[None], F, corner, rows, vals)
        u, cur = upper_backup_np(model, gamma, F, rows, vals, b)
        hp.check_interval([u], ref['u'], what='u')
        hp.check_interval([cur], ref['cur'], what='cur')
        a = int(np.argmax(ref['Q'][0][0] + ref['Q'][1][0]))
        st = hp.gap_step(succ[a][None], mass[a][None], F, corner, rows, vals, X, 0.0)
        U, L, p = step_np(model, gamma, F, X, rows, vals, b, a)
        hp.check_interval(U[None], st['U'], what='U')
        hp.check_interval(L[None], st['L'], what='L')
        e = np.where(p > 0, p * ((U - L) - 0.0), np.nan)
        hp.check_interval(e[None], st['e'], what='e')
        hp.check_gap_choice(st['e'], [choose_np(e, None)])
        for uk in (0.0, float(rng.random()), 1.0 - 2.0 ** -53, 1.0, 2.0):
            hp.check_sampled_choice(st['e'], [uk], [choose_np(e, uk)])


@pytest.mark.parametrize('name', ['hallway', 'cit', 's2', 's3'])
def test_upper_contract_rejects_moved_values_swaps_and_dropped_terms(name):
    from test_upper_bound import sawtooth_np, successors_np
    model, gamma, B, F, rows, vals = upper_case(name)
    corner = F.max(axis=0)
    lo, hi = hp.sawtooth(corner, rows, vals, B)
    got = np.array([sawtooth_np(b, corner, rows, vals) for b in B])
    # a value moved by three times its bound
    moved = got.copy()
    moved[0] = float((lo[0] + hi[0]) / 2 + 3 * (hi[0] - lo[0]))
    with pytest.raises(AssertionError, match='sawtooth'):
        hp.check_interval(moved, (lo, hi), what='sawtooth')
    # one dropped support entry: the entry that decides m_i of the binding stored term
    dropped_any = False
    for j, b in enumerate(B):
        terms = [(b @ corner + (v - r @ corner) * np.min(b[r > 0] / r[r > 0]), i) for i, (r, v) in enumerate(zip(rows, vals))]
        t, i = min(terms)
        if not t < b @ corner:
            continue
        sup = np.flatnonzero(rows[i] > 0)
        ratios = b[sup] / rows[i][sup]
        if sup.size < 2 or np.sort(ratios)[1] == ratios.min():
            continue
        keep = np.delete(sup, np.argmin(ratios))
        m = np.min(b[keep] / rows[i][keep])
        alt = min([b @ corner] + [tt for tt, ii in terms if ii != i] + [b @ corner + (vals[i] - rows[i] @ corner) * m])
        if alt == got[j]:
            continue
        bad = got.copy()
        bad[j] = alt
        with pytest.raises(AssertionError, match='sawtooth'):
            hp.check_interval(bad, (lo, hi), what='sawtooth')
        dropped_any = True
    assert dropped_any
    # a* swapped where it is decided; an observation term worth 1e-12 of the value dropped from u
    decided_any = False
    for b in B[:6]:
        succ, mass = successors_np(model, b)
        ref = hp.upper_q(b[None], model.expected_rewards_table, gamma, succ[None], mass[None], F, corner, rows, vals)
        ex, bd = hp.as_center(ref['Q'])
        want = np.argmax(ex, axis=1)
        dec = hp.check_argmax(ex, bd, want, what='a*')
        if dec[0] and ex.shape[1] > 1:
            decided_any = True
            with pytest.raises(AssertionError, match='a\\*'):
                hp.check_argmax(ex, bd, [int(np.argsort(ex[0])[-2])], what='a*')
        c = float((ref['u'][0][0] + ref['u'][1][0]) / 2)
        with pytest.raises(AssertionError, match='u'):
            hp.check_interval([c - 1e-12 * abs(c)], ref['u'], what='u')
    assert decided_any


def test_gap_choice_rejects_a_swapped_decided_observation():
    e = (np.array([[0.1, 0.5, np.nan, -0.2]], dtype=hp.LD), np.array([[0.1, 0.5, np.nan, -0.2]], dtype=hp.LD))
    assert hp.check_gap_choice(e, [1]).all()
    for bad in (0, 2, 3, -1):
        with pytest.raises(AssertionError, match='o\\*'):
            hp.check_gap_choice(e, [bad])
    # the sampled rule: cdf = (1/6, 1, 1, 1); u = 0.1 -> 0, u = 0.5 -> 1, u >= 1 -> capped at the last positive weight (1)
    for uk, want in ((0.0, 0), (0.1, 0), (0.5, 1), (1.0, 1), (3.0, 1)):
        assert hp.check_sampled_choice(e, [uk], [want]).all()
        with pytest.raises(AssertionError, match='o\\*'):
            hp.check_sampled_choice(e, [uk], [1 - want])
    none = (np.array([[-0.1, np.nan]], dtype=hp.LD), np.array([[-0.1, np.nan]], dtype=hp.LD))
    assert hp.check_gap_choice(none, [-1]).all() and hp.check_sampled_choice(none, [0.5], [-1]).all()
    with pytest.raises(AssertionError):
        hp.check_gap_choice(none, [0])


def test_upper_bounds_are_far_below_the_float64_slack():
    """On the golden stores the sawtooth and u intervals are narrower than 1e-10 of the value (below 2e-11 even on the 7936-state
    supports of olfactory): a kernel that drops a term worth 1e-10 of it -- invisible to the 1e-9 comparisons -- is rejected."""
    from test_upper_bound import successors_np
    for name in GOLDEN:
        model, gamma, B, F, rows, vals = upper_case(name)
        corner = F.max(axis=0)
        lo, hi = hp.sawtooth(corner, rows, vals, B)
        assert np.max((hi - lo).astype(np.float64) / np.maximum(np.abs(hi.astype(np.float64)), 1e-300)) < 1e-10, name
        succ, mass = successors_np(model, B[0])
        ref = hp.upper_q(B[:1], model.expected_rewards_table, gamma, succ[None], mass[None], F, corner, rows, vals)
        lo, hi = ref['u']
        assert float((hi - lo)[0]) < 1e-10 * abs(float(hi[0])), name


def test_sawtooth_subnormal_store_and_overflowing_ratios():
    """A stored belief whose entries are subnormal: its ratios overflow to inf where the query is O(1), and an inf quotient never wins
    the minimum; query entries of 1e-13 move v0 by far more than its bound."""
    from test_upper_bound import sawtooth_np
    S = 12
    corner = np.linspace(1.0, 3.0, S)
    rows = np.zeros((3, S))
    rows[0, :4] = [1e-310, 2e-310, 0.0, 1.0 - 1e-300]
    rows[1, 4:] = 1.0 / 8
    rows[2, [0, 5]] = [5e-324, 1.0]
    vals = rows @ corner - np.array([0.5, 0.25, 0.1])
    Q = np.zeros((4, S))
    Q[0, :4] = 0.25
    Q[1, [1, 3, 4]] = [0.5, 0.25, 0.25]
    Q[2] = 1.0 / S
    Q[3, :6] = 1e-13
    Q[3, 6] = 1.0 - 6e-13
    lo, hi = hp.sawtooth(corner, rows, vals, Q)
    assert np.all(np.isfinite(lo)) and np.all(np.isfinite(hi))
    with np.errstate(over='ignore'):
        got = [sawtooth_np(q, corner, rows, vals) for q in Q]
    hp.check_interval(got, (lo, hi), what='sawtooth')
    skipped = Q[3].copy()
    skipped[skipped < 1e-12] = 0.0
    with pytest.raises(AssertionError):
        hp.check_interval([float(skipped @ corner)], (lo[3:], hi[3:]))
