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
