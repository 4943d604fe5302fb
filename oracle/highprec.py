"""
TEST INFRASTRUCTURE ONLY -- extended-precision reference of the point-based backup, with a-priori error bounds.

`pbvi_oracle.backup` is float64 in NumPy's order, so comparing the engine with it needs a slack (1e-9) far larger than the rounding
error of either side; a kernel that drops terms worth less than that slack passes.  Here every quantity of the backup is computed
in `np.longdouble` (x87 80-bit on x86-64: 64-bit significand) together with a bound on how far ANY float64 evaluation of the same
sum -- any order, with or without FMA, any pre-rounded partial product -- can be from the exact value.  `check_backup` applies the
engine's contract with those bounds instead of a fixed tolerance.

Error model.  With u = 2^-53 and eta = 2^-1074 (the smallest subnormal), one float64 operation gives fl(x op y) = (x op y)(1 + d) + e,
|d| <= u, |e| <= eta / 2.  A term that passes through k roundings carries a relative error of at most gamma_k = k u / (1 - k u) <=
(k + 1) u (k < 9e7).  A sum of n non-zero terms, in any order, passes each term through at most n - 1 additions, and a product folded
into an FMA is not rounded on its own.  Adding an exact zero (a pad state, a belief entry that is 0) is exact and is not counted.  So
with n the number of terms of the exact sum and sum|t| the sum of their magnitudes, every bound below has the form

    (n + c) (u + u_ld) sum|t|  +  (2 n + 2 c) eta M

where the first part covers the float64 evaluation and the reference's own longdouble rounding (u_ld = eps_ld / 2, same count), and
the second part covers roundings in the subnormal range (at most 2n + 2c roundings, each scaled by at most M, the largest factor that
multiplies it later).  The constants c:

  score, gather form (R = 1: score kernel A operand = fl(b[s] RTO[s,a,o]), DMMA over s):  a term is rounded once in b RTO, then
      at most once in the product (FMA: never) and n - 1 times in the sum: n + 1 roundings -> gamma_{n+1} <= (n + 2) u.
  score, Gamma form (R > 1: G[s,v] = fl(sum_r RTO alpha) first, then DMMA of b with G):  R roundings inside G (R products, R - 1
      additions), then n_s in the s-sum (n_s = support size): R + n_s <= n_s R + 1 = n + 1 roundings -> (n + 2) u.
  pbvi_oracle.backup additionally scales G by gamma before the s-sum (one more rounding): n + 2 roundings -> (n + 3) u.  The score is
      compared without gamma (an argmax-invariant positive scale), so C_SCORE = 3 covers all three.
  value, reference order (alpha_a[s] = rb + sum_o gamma sum_r RTO alpha, then sum_s b[s] alpha_a[s]):  a term passes R (RTO alpha and
      the r-sum) + 1 (gamma) + O - 1 (o-sum) + 1 (+ rb) + n_s (b times entry, s-sum) = n_s + R + O + 1 roundings, and with
      n = n_s (1 + O R) >= n_s + O R >= n_s + R + O - 1 that is <= n + 2 -> (n + 3) u.
  value, screened form (b . Rbar + gamma sum_o max score, in the score kernel's order):  an RTO term passes the score's n_s + R
      roundings (either form above), O - 1 in the o-sum, 1 for gamma and 1 for the final addition: n_s + R + O + 1 again.  C_VALUE = 3.
  GER eps (sum_s ((d >= 0 ? rMax : rMin) - alpha[s]) d, d = fl(succ[s] - b[s])):  1 (d) + 1 (rMax - alpha) + 1 (product, or FMA)
      + n - 1 (sum) = n + 2 roundings -> C_GER = 3.  The sign test sees fl(d), whose sign is the sign of the exact difference.

sum|t| is evaluated in float64 with non-negative terms (relative error below n u < 1e-6) and inflated by 1 + 1e-6.

Every computation runs on the support of each belief only, so a belief with 50 non-zero states over S = 20 000 costs 50 R A O V
multiply-adds.  This module imports nothing from the product package.
"""
from __future__ import annotations

import numpy as np

LD = np.longdouble
EPS_LD = float(np.finfo(LD).eps)
if not EPS_LD <= 1e-18:
    raise ImportError(f'oracle.highprec needs an extended-precision np.longdouble (eps <= 1e-18); this platform has eps = {EPS_LD:.3g}')
U = 2.0 ** -53                    # float64 unit roundoff
U_LD = EPS_LD / 2                 # longdouble unit roundoff
ETA = 2.0 ** -1074                # smallest float64 subnormal
ABS_SLACK = 1.0 + 1e-6            # sum|t| is itself evaluated in float64

C_SCORE = 3
C_VALUE = 3
C_GER = 3


def _bound(n, abs_sum, c, scale):
    n = np.asarray(n, dtype=np.float64)
    assert np.all(n < 9e7), 'the (k + 1) u form of gamma_k needs k < 9e7'
    return (n + c) * (U + U_LD) * abs_sum * ABS_SLACK + (2 * n + 2 * c) * ETA * scale


def _batches(beliefs: np.ndarray, rows_per_batch: int = 2048):
    """(row indices, support columns) of the beliefs: whole batches over the union of their supports when the model is narrow, one
    belief at a time over its own support otherwise."""
    nB, S = beliefs.shape
    if S <= 64:
        for i in range(0, nB, rows_per_batch):
            rows = np.arange(i, min(nB, i + rows_per_batch))
            cols = np.flatnonzero(np.any(beliefs[rows] != 0, axis=0))
            yield rows, cols
    else:
        for i in range(nB):
            yield np.array([i]), np.flatnonzero(beliefs[i])


# --------------------------------------------------------------------------------------------------------------------------------
# Scores
# --------------------------------------------------------------------------------------------------------------------------------
def scores(reach: np.ndarray, rto: np.ndarray, beliefs: np.ndarray, alphas: np.ndarray):
    """
    score[b,a,o,v] = sum_s sum_r b[s] RTO[s,a,o,r] alpha_v[reach[s,a,r]] (no gamma) in longdouble, its bound, and `no_terms` [B,A,O,V]:
    True where every term of the sum is zero (every float64 evaluation then gives +-0 for that entry).
    """
    S, A, R = reach.shape
    O = rto.shape[2]
    nB, V = beliefs.shape[0], alphas.shape[0]
    exact = np.zeros((nB, A, O, V), dtype=LD)
    absum = np.zeros((nB, A, O, V))
    nterm = (np.count_nonzero(beliefs, axis=1) * R).astype(np.float64)
    for rows, cols in _batches(beliefs):
        if cols.size == 0:
            continue
        k = cols.size
        bs = beliefs[np.ix_(rows, cols)]                                            # [nb, k]
        w = rto[cols]                                                               # [k, A, O, R]
        land = reach[cols]                                                          # [k, A, R]
        bw = bs.astype(LD)[:, :, None, None, None] * w.astype(LD)[None]             # [nb, k, A, O, R]
        abw = np.abs(bs)[:, :, None, None, None] * np.abs(w)[None]
        for a in range(A):
            ag = alphas[:, land[:, a, :].reshape(-1)]                               # [V, k R]
            lhs = bw[:, :, a].transpose(0, 2, 1, 3).reshape(len(rows), O, k * R)    # [nb, O, k R]
            exact[rows, a] = np.matmul(lhs, ag.astype(LD).T)
            absum[rows, a] = np.matmul(abw[:, :, a].transpose(0, 2, 1, 3).reshape(len(rows), O, k * R), np.abs(ag).T)
    scale = max(1.0, float(np.max(np.abs(alphas))))
    bound = _bound(nterm[:, None, None, None], absum, C_SCORE, scale)
    return exact, bound, absum == 0.0


def plain_scores(beliefs: np.ndarray, alphas: np.ndarray):
    """prod[b,v] = b . alpha_v (pbvi_max_values) in longdouble, its bound and `no_terms` [B,V]."""
    nB, V = beliefs.shape[0], alphas.shape[0]
    exact = np.zeros((nB, V), dtype=LD)
    absum = np.zeros((nB, V))
    for rows, cols in _batches(beliefs):
        if cols.size:
            bs = beliefs[np.ix_(rows, cols)]
            ag = alphas[:, cols]
            exact[rows] = np.matmul(bs.astype(LD), ag.astype(LD).T)
            absum[rows] = np.abs(bs) @ np.abs(ag).T
    nterm = np.count_nonzero(beliefs, axis=1).astype(np.float64)
    scale = max(1.0, float(np.max(np.abs(alphas))))
    return exact, _bound(nterm[:, None], absum, C_SCORE, scale), absum == 0.0


# --------------------------------------------------------------------------------------------------------------------------------
# alpha_a entries and values
# --------------------------------------------------------------------------------------------------------------------------------
def _entries(reach, rto, rbar, gamma, alphas, vsel, cols):
    """alpha_a[s] for every action a and s in cols, v_o = vsel[i, a, o]: longdouble [n, A, k] and sum of |terms| [n, A, k]."""
    A, R = reach.shape[1], reach.shape[2]
    land = reach[cols].transpose(1, 0, 2)                                           # [A, k, R]
    w = rto[cols].transpose(1, 2, 0, 3)                                             # [A, O, k, R]
    av = alphas[vsel[:, :, :, None, None], land[None, :, None, :, :]]               # [n, A, O, k, R]
    g = LD(gamma)
    inner = np.sum(w.astype(LD)[None] * av.astype(LD), axis=4)                      # [n, A, O, k]
    ent = rbar[cols].T.astype(LD)[None] + g * np.sum(inner, axis=2)                 # [n, A, k]
    absum = np.abs(rbar[cols].T)[None] + abs(gamma) * np.sum(np.abs(w)[None] * np.abs(av), axis=(2, 4))
    return ent, absum


def values(reach, rto, rbar, gamma: float, beliefs: np.ndarray, alphas: np.ndarray, vstar: np.ndarray):
    """value[b,a] = b . alpha_a with alpha_a built from the given v*[b,a,:] (longdouble [B,A]) and its bound [B,A]."""
    S, A, R = reach.shape
    O = rto.shape[2]
    nB = beliefs.shape[0]
    vstar = np.asarray(vstar, dtype=np.int64)
    exact = np.zeros((nB, A), dtype=LD)
    absum = np.zeros((nB, A))
    for rows, cols in _batches(beliefs):
        if cols.size == 0:
            continue
        ent, eabs = _entries(reach, rto, rbar, gamma, alphas, vstar[rows], cols)
        bs = beliefs[np.ix_(rows, cols)]
        exact[rows] = np.sum(bs.astype(LD)[:, None, :] * ent, axis=2)
        absum[rows] = np.sum(np.abs(bs)[:, None, :] * eabs, axis=2)
    nterm = (np.count_nonzero(beliefs, axis=1) * (1 + O * R)).astype(np.float64)
    scale = max(1.0, float(np.max(np.abs(beliefs)))) * max(1.0, abs(gamma)) * max(1.0, float(np.max(np.abs(alphas))), float(np.max(np.abs(rbar))))
    return exact, _bound(nterm[:, None], absum, C_VALUE, scale)


def alpha_entries(reach, rto, rbar, gamma: float, alphas: np.ndarray, actions: np.ndarray, vsel: np.ndarray):
    """alpha_a[s] of the tuples (actions[i], vsel[i, :]) on every state: longdouble [n, S] and its bound [n, S] (the value bound's
    derivation without the s-sum: R + O + 1 roundings, n = 1 + O R terms)."""
    S, A, R = reach.shape
    O = rto.shape[2]
    actions = np.asarray(actions, dtype=np.int64)
    vsel = np.asarray(vsel, dtype=np.int64)
    full = np.zeros((len(actions), A, O), dtype=np.int64)
    full[np.arange(len(actions)), actions] = vsel
    ent, eabs = _entries(reach, rto, rbar, gamma, alphas, full, np.arange(S))
    pick = np.arange(len(actions))
    scale = max(1.0, abs(gamma)) * max(1.0, float(np.max(np.abs(alphas))), float(np.max(np.abs(rbar))))
    return ent[pick, actions], _bound(1 + O * R, eabs[pick, actions], C_VALUE, scale)


def alpha_rows_f64(reach, rto, rbar, gamma: float, alphas: np.ndarray, actions: np.ndarray, vsel: np.ndarray) -> np.ndarray:
    """
    The engine's alpha_a_entry restated in float64 NumPy (one rounding per elementwise operation, no FMA):
        rb + ((g_0 + g_1) + ...),   g_o = gamma * ((w_0 alpha_0 + w_1 alpha_1) + ...)   (r ascending, then o ascending).
    The kernels skip terms whose RTO factor is 0 when the alphas are finite; for finite alphas that gives the same bits (see the
    comment on alpha_a_entry), so the rows of pbvi_backup / pbvi_backup_assemble must equal these bitwise.
    """
    S, A, R = reach.shape
    O = rto.shape[2]
    actions = np.asarray(actions, dtype=np.int64)
    vsel = np.asarray(vsel, dtype=np.int64)
    out = np.empty((len(actions), S))
    for a in np.unique(actions):
        idx = np.flatnonzero(actions == a)
        acc = None
        for o in range(O):
            nxt = alphas[vsel[idx, o]]
            inner = None
            for r in range(R):
                prod = rto[:, a, o, r][None, :] * nxt[:, reach[:, a, r]]
                inner = prod if r == 0 else inner + prod
            term = gamma * inner
            acc = term if o == 0 else acc + term
        out[idx] = rbar[:, a][None, :] + acc
    return out


# --------------------------------------------------------------------------------------------------------------------------------
# GER
# --------------------------------------------------------------------------------------------------------------------------------
def ger_eps(beliefs: np.ndarray, successors: np.ndarray, alpha_b: np.ndarray, r_min: float, r_max: float):
    """eps[n,a,o] = sum_s ((d >= 0 ? r_max : r_min) - alpha_b[n,s]) d, d = succ[n,a,o,s] - b[n,s], in longdouble, and its bound.
    NaN where the successor is NaN (an impossible observation)."""
    d = successors.astype(LD) - beliefs.astype(LD)[:, None, None, :]
    p = np.where(d >= 0, LD(r_max), LD(r_min))
    t = (p - alpha_b.astype(LD)[:, None, None, :]) * d
    exact = np.sum(t, axis=3)
    with np.errstate(invalid='ignore'):
        absum = np.sum(np.abs(t.astype(np.float64)), axis=3)
    n = successors.shape[3]
    scale = max(1.0, abs(r_min), abs(r_max), float(np.max(np.abs(alpha_b))))
    return exact, _bound(n, absum, C_GER, scale)


# --------------------------------------------------------------------------------------------------------------------------------
# The contract
# --------------------------------------------------------------------------------------------------------------------------------
def check_argmax(exact, bound, picked, no_terms=None, what='argmax'):
    """
    The first-index argmax contract with certified bounds, over the last axis:
      * where the exact top-two gap exceeds twice the largest bound of the row, `picked` is the exact argmax;
      * everywhere, the exact value of the picked column is within twice that bound of the exact maximum;
      * rows whose every term is zero (`no_terms` all True) pick column 0.
    """
    picked = np.asarray(picked, dtype=np.int64)
    K = exact.shape[-1]
    assert picked.shape == exact.shape[:-1], (what, picked.shape, exact.shape)
    assert np.all((picked >= 0) & (picked < K)), f'{what}: index out of range'
    bmax = np.max(bound, axis=-1).astype(LD)
    srt = np.sort(exact, axis=-1)
    best = srt[..., -1]
    if K > 1:
        decided = (best - srt[..., -2]) > 2 * bmax
        want = np.argmax(exact, axis=-1)
        bad = decided & (picked != want)
        if bad.any():
            i = tuple(np.argwhere(bad)[0])
            raise AssertionError(f'{what}: decided entry {i} picked {picked[i]}, exact argmax {want[i]} '
                                 f'(gap {float(best[i] - srt[i + (-2,)]):.3e}, bound {float(bmax[i]):.3e})')
    got = np.take_along_axis(exact, picked[..., None], axis=-1)[..., 0]
    short = got < best - 2 * bmax
    if short.any():
        i = tuple(np.argwhere(short)[0])
        raise AssertionError(f'{what}: entry {i} picked {picked[i]} whose exact value is {float(best[i] - got[i]):.3e} below the maximum '
                             f'(bound {float(bmax[i]):.3e})')
    if no_terms is not None:
        flat = np.all(no_terms, axis=-1)
        if np.any(picked[flat] != 0):
            raise AssertionError(f'{what}: a row whose every term is zero did not pick column 0')
    return decided if K > 1 else np.ones(picked.shape, bool)


def check_close(got, exact, bound, what='value'):
    """|got - exact| <= bound, entrywise."""
    err = np.abs(np.asarray(got, dtype=np.float64).astype(LD) - exact)
    bad = ~(err <= bound.astype(LD))
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f'{what}: entry {i} is {float(err[i]):.3e} from the exact value {float(exact[i]):.17g} '
                             f'(bound {float(bound[i]):.3e}, worst ratio {float(np.nanmax(err / np.maximum(bound, 1e-320))):.3g})')


def check_backup(reach, rto, rbar, gamma: float, beliefs, alphas, vstar, value=None, astar=None, rows=None, sc=None):
    """
    The backup contract (pbvi_backup / pbvi_backup_select outputs, any of value / astar / rows may be None):
      v*     check_argmax on the exact scores;
      value  within the bound of the exact value at the engine's own v*;
      a*     check_argmax on those exact values, and the first maximiser of the engine's own values;
      rows   bitwise alpha_rows_f64 at the engine's own (a*, v*[a*]).
    `sc` = scores(...) when the caller has it already.  Returns the exact scores' tuple.
    """
    vstar = np.asarray(vstar, dtype=np.int64)
    if sc is None:
        sc = scores(reach, rto, beliefs, alphas)
    check_argmax(sc[0], sc[1], vstar, sc[2], what='v*')
    if value is not None or astar is not None:
        ev, evb = values(reach, rto, rbar, gamma, beliefs, alphas, vstar)
        if value is not None:
            check_close(value, ev, evb, what='value')
        if astar is not None:
            astar = np.asarray(astar, dtype=np.int64)
            check_argmax(ev, evb, astar, what='a*')
            if value is not None:
                assert np.array_equal(astar, np.argmax(np.asarray(value), axis=1)), 'a*: not the first maximiser of the values'
    if rows is not None:
        assert astar is not None
        sel = vstar[np.arange(len(astar)), astar]
        want = alpha_rows_f64(reach, rto, rbar, gamma, alphas, astar, sel)
        got = np.asarray(rows)
        if got.tobytes() != want.tobytes():
            bad = np.argwhere(got.view(np.uint64) != want.view(np.uint64))[0]
            raise AssertionError(f'rows: entry {tuple(bad)} is {got[tuple(bad)]!r}, the restatement gives {want[tuple(bad)]!r}')
    return sc
