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

Upper bounds (pbvi_sawtooth / pbvi_sawtooth_lists, pbvi_upper_backup, pbvi_gap_trial_step, pbvi_hsvi_level).  Each stage is exact given
its float64 inputs: the successor rows q and masses P(o|b,a) are the device's own (pinned elsewhere: rows bitwise the reference's update,
masses bitwise NumPy's pairwise sum), and so is every value a later stage reads.  The results are intervals [lo, hi] that hold every
float64 evaluation; a minimum or maximum of values known to lie in intervals lies in the interval of the endpoints' minima / maxima, so
the intervals do not depend on which term a device reduction picks.

  sawtooth term (x_i = v0 + (v_i - d_i) m_i, v0 = q . corner, d_i = b_i . corner, m_i = min_{s: b_i[s] > 0} q[s] / b_i[s]):  m_i is a
      minimum of correctly rounded quotients, and rounding is monotone, so the device's m_i is the float64 minimum of the float64
      quotients -- NumPy's, bit for bit, overflow to inf included -- and enters as an input.  A q . corner term passes the v0 dot (n_0
      roundings) and the final addition: n_0 + 1; v_i m_i passes the subtraction, the product and the addition: 3; a b_i . corner
      term the d_i dot (n_i), then the same 3: n_i + 3.  With n = n_0 + n_i + 1 that is <= n + 2 -> (n + 3) u, C_SAW = 3.  An absolute
      (subnormal) error of the d_i dot is multiplied by m_i later: M = max(1, m_i).  The v0 term alone is the n = n_0 case.
  Q (rb + gamma sum_{o: P > 0} P y_o, rb = b . Rbar_a, y_o = min(max_v F_v . q, saw(q)) known in [y_lo, y_hi]):  Q is increasing in
      every y_o (P >= 0, gamma > 0), so the exact Q at the device's y lies in [Q(y_lo), Q(y_hi)].  Its float64 evaluation: an rb term
      passes the n_r dot roundings and the final addition; a P y term the product, O_p - 1 additions, gamma, the final addition: with
      n = n_r + O_p terms both are <= n + 2 -> C_Q = 3 (sum|t| with |y| <= max(|y_lo|, |y_hi|)).
  excess e = P ((U - L) - theta):  three roundings per term, n = 3 terms (P U, P L, P theta) -> (n + 1) u, C_EXCESS = 1; e is increasing
      in U and decreasing in L, so its exact value at the device's U, L lies in [P (U_lo - L_hi - theta), P (U_hi - L_lo - theta)].
  sampled o* (cdf_j = (sum_{o <= j} w_o) / W, w = max(e, 0), sequential sums, one division):  with w in [w_lo, w_hi] the running sums
      lie within (O + 1) (u + u_ld) of [cumsum w_lo, cumsum w_hi], and the quotient within one more rounding.
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
C_SAW = 3
C_Q = 3
C_EXCESS = 1


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
# Upper bounds
# --------------------------------------------------------------------------------------------------------------------------------
def _dots(rows: np.ndarray, vec: np.ndarray):
    """rows . vec in longdouble, sum |row[s] vec[s]| and the number of non-zero products, per row."""
    prod_abs = np.abs(rows) * np.abs(vec)[None, :]
    exact = rows.astype(LD) @ vec.astype(LD)
    return exact, prod_abs.sum(axis=1), np.count_nonzero(prod_abs, axis=1).astype(np.float64)


def sawtooth(corner: np.ndarray, stored_rows: np.ndarray, stored_vals: np.ndarray, queries: np.ndarray):
    """
    The sawtooth upper bound of each query (finite, non-negative rows) over the stored pairs: (lo, hi) longdouble [n_q] that hold
    min(v0, min_i x_i) for every float64 evaluation (module docstring, C_SAW).  A term whose m_i overflows to inf in float64 is +inf or
    -inf by the sign of its scale (and either, or skipped as NaN, when that sign is not certain).
    """
    queries = np.atleast_2d(queries)
    v0, v0abs, n0 = _dots(queries, corner)
    lo = v0 - _bound(n0, v0abs, C_SAW, 1.0).astype(LD)
    hi = v0 + _bound(n0, v0abs, C_SAW, 1.0).astype(LD)
    for bi, vi in zip(np.atleast_2d(stored_rows), np.atleast_2d(stored_vals).reshape(-1)):
        sup = np.flatnonzero(bi > 0)
        if sup.size == 0:
            m = np.full(len(queries), np.inf)
        else:
            with np.errstate(over='ignore', under='ignore'):
                m = np.min(queries[:, sup] / bi[sup], axis=1)                     # the device's minimum, bit for bit
        d, dabs, ni = _dots(bi[None, :], corner)
        sc = LD(vi) - d[0]
        sc_bound = _bound(ni[0], dabs[0], C_SAW, 1.0)
        fin = np.isfinite(m)
        mf = np.where(fin, m, 0.0)
        x = v0 + sc * mf.astype(LD)
        tabs = v0abs + (abs(vi) + dabs[0]) * mf
        e = _bound(n0 + ni[0] + 1, tabs, C_SAW, np.maximum(1.0, mf)).astype(LD)
        t_lo, t_hi = x - e, x + e
        if not fin.all():
            pos = sc > LD(sc_bound)
            neg = sc < -LD(sc_bound)
            t_lo = np.where(fin, t_lo, LD(np.inf) if pos else LD(-np.inf))
            t_hi = np.where(fin, t_hi, LD(-np.inf) if neg else LD(np.inf))
        lo = np.minimum(lo, t_lo)
        hi = np.minimum(hi, t_hi)
    return lo, hi


def max_scores(rows: np.ndarray, alphas: np.ndarray):
    """(lo, hi) longdouble [n] holding max_v rows . alpha_v for every float64 evaluation (pbvi's few-rows and plain score kernels)."""
    ex, bd, _ = plain_scores(np.atleast_2d(rows), alphas)
    bd = bd.astype(LD)
    return np.max(ex - bd, axis=1), np.max(ex + bd, axis=1)


def upper_values(rows: np.ndarray, fib_rows, corner, stored_rows, stored_vals):
    """(lo, hi) of min(max_v F_v . q, sawtooth(q)) per row (no FIB part when fib_rows is None)."""
    lo, hi = sawtooth(corner, stored_rows, stored_vals, rows)
    if fib_rows is not None:
        flo, fhi = max_scores(rows, fib_rows)
        lo, hi = np.minimum(lo, flo), np.minimum(hi, fhi)
    return lo, hi


def q_values(beliefs: np.ndarray, rbar: np.ndarray, gamma: float, mass: np.ndarray, y_lo: np.ndarray, y_hi: np.ndarray):
    """
    (lo, hi) longdouble [n, A] holding Q[b,a] = b . Rbar_a + gamma sum_{o: P > 0} P(o|b,a) y[b,a,o] for every float64 evaluation at
    every y in [y_lo, y_hi] (C_Q).  mass [n, A, O] are the device's masses; y is read only where they are positive.
    """
    n, A, O = mass.shape
    live = mass > 0
    rb = beliefs.astype(LD) @ rbar.astype(LD)                                           # [n, A]
    rb_abs = np.abs(beliefs) @ np.abs(rbar)
    n_r = np.stack([np.count_nonzero(beliefs * rbar[:, a][None, :], axis=1) for a in range(A)], axis=1).astype(np.float64)
    g = LD(gamma)
    p = np.where(live, mass, 0.0)
    ylo = np.where(live, y_lo, LD(0))
    yhi = np.where(live, y_hi, LD(0))
    q_lo = rb + g * np.sum(p.astype(LD) * ylo, axis=2)
    q_hi = rb + g * np.sum(p.astype(LD) * yhi, axis=2)
    ymag = np.maximum(np.abs(ylo), np.abs(yhi)).astype(np.float64)
    tabs = rb_abs + abs(gamma) * np.sum(p * ymag, axis=2)
    e = _bound(n_r + np.count_nonzero(live, axis=2), tabs, C_Q, max(1.0, abs(gamma))).astype(LD)
    return q_lo - e, q_hi + e


def upper_q(beliefs, rbar, gamma: float, successors, mass, fib_rows, corner, stored_rows, stored_vals, want_cur: bool = True):
    """
    The upper-bound backup (pbvi_upper_backup) from the device's successor rows [n, A, O, S] and masses [n, A, O]: a dict of longdouble
    intervals  Q [n, A],  u = max_a Q [n],  cur = min(max_v F_v . b, sawtooth(b)) [n],  and y [n, A, O] (NaN where P = 0).
    """
    n, A, O = mass.shape
    live = mass > 0
    y_lo = np.full((n, A, O), LD(np.nan))
    y_hi = np.full((n, A, O), LD(np.nan))
    if live.any():
        y_lo[live], y_hi[live] = upper_values(successors[live], fib_rows, corner, stored_rows, stored_vals)
    q_lo, q_hi = q_values(beliefs, rbar, gamma, mass, y_lo, y_hi)
    out = dict(Q=(q_lo, q_hi), u=(np.max(q_lo, axis=1), np.max(q_hi, axis=1)), y=(y_lo, y_hi))
    if want_cur:
        out['cur'] = upper_values(beliefs, fib_rows, corner, stored_rows, stored_vals)
    return out


def excess(mass, U, L, theta: float):
    """(lo, hi) of e = P ((U - L) - theta) for every float64 evaluation at every U in U = (lo, hi) and L in L = (lo, hi) (C_EXCESS);
    NaN where P = 0."""
    live = mass > 0
    p = np.where(live, mass, 0.0)
    u_lo, u_hi = (np.where(live, x, LD(0)) for x in U)
    l_lo, l_hi = (np.where(live, x, LD(0)) for x in L)
    pl, th = p.astype(LD), LD(theta)
    tabs = p * (np.maximum(np.abs(u_lo), np.abs(u_hi)) + np.maximum(np.abs(l_lo), np.abs(l_hi)) + abs(theta)).astype(np.float64)
    e = _bound(3, tabs, C_EXCESS, 1.0).astype(LD)
    lo = np.where(live, pl * (u_lo - l_hi - th) - e, LD(np.nan))
    hi = np.where(live, pl * (u_hi - l_lo - th) + e, LD(np.nan))
    return lo, hi


def gap_step(successors, mass, fib_rows, corner, stored_rows, stored_vals, lower_rows, theta: float):
    """
    One gap-trial level at the chosen actions (pbvi_gap_trial_step): successors [K, O, S] and masses [K, O] of b_k under a*_k.  Returns
    a dict of longdouble intervals U [K, O] (upper value of the successor), L [K, O] (max_n X_n . q) and e [K, O] (the excess); all three
    NaN where P = 0.
    """
    K, O = mass.shape
    live = mass > 0
    U = [np.full((K, O), LD(np.nan)) for _ in range(2)]
    L = [np.full((K, O), LD(np.nan)) for _ in range(2)]
    if live.any():
        U[0][live], U[1][live] = upper_values(successors[live], fib_rows, corner, stored_rows, stored_vals)
        L[0][live], L[1][live] = max_scores(successors[live], lower_rows)
    return dict(U=tuple(U), L=tuple(L), e=excess(mass, U, L, theta))


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


def check_interval(got, interval, what='value'):
    """lo <= got <= hi entrywise; NaN intervals (an impossible observation) take NaN only."""
    lo, hi = interval
    got = np.asarray(got, dtype=np.float64)
    gl = got.astype(LD)
    nan = np.isnan(lo)
    bad = np.where(nan, ~np.isnan(got), ~((lo <= gl) & (gl <= hi)))
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f'{what}: entry {i} is {got[i]!r}, outside [{float(lo[i])!r}, {float(hi[i])!r}] '
                             f'(width {float(hi[i] - lo[i]):.3e})')


def as_center(interval):
    """(center, half width) of an interval: the (exact, bound) pair `check_argmax` takes."""
    lo, hi = interval
    return (lo + hi) / 2, ((hi - lo) / 2).astype(np.float64) * ABS_SLACK


def check_interval_argmax(interval, picked, valid=None, what='argmax'):
    """
    A first-argmax over the valid entries of the last axis, each known to lie in its interval: `picked` is valid and not certainly below
    another entry; where one entry lies certainly above every other valid entry, `picked` is that entry.  Returns the decided rows.
    """
    lo, hi = interval
    picked = np.asarray(picked, dtype=np.int64)
    valid = np.ones(lo.shape, bool) if valid is None else valid
    lo = np.where(valid, lo, LD(-np.inf))
    hi = np.where(valid, hi, LD(-np.inf))
    rows = np.argwhere(valid.any(axis=-1))
    decided = np.zeros(picked.shape, bool)
    for i in map(tuple, rows):
        p = picked[i]
        assert 0 <= p < lo.shape[-1] and valid[i][p], f'{what}: row {i} picked {p}, not a valid entry'
        assert hi[i][p] >= np.max(lo[i]), f'{what}: row {i} picked {p}, certainly below entry {int(np.argmax(lo[i]))}'
        j = int(np.argmax(lo[i]))
        others = np.delete(hi[i], j)
        if others.size == 0 or lo[i][j] > np.max(others):
            decided[i] = True
            assert p == j, f'{what}: row {i} picked {p}, entry {j} is certainly the largest'
    return decided


def check_gap_choice(e, picked, what='o*'):
    """o* of the argmax rule: the first argmax of e over {e > 0}, -1 when no excess is positive (e = (lo, hi), NaN: impossible)."""
    lo, hi = e
    picked = np.asarray(picked, dtype=np.int64)
    pos_sure = lo > 0                                           # NaN > 0 is False
    pos_maybe = hi > 0
    none = picked < 0
    bad = none & pos_sure.any(axis=-1)
    assert not bad.any(), f'{what}: rows {np.flatnonzero(bad)[:5]} picked -1 with a certainly positive excess'
    bad = ~none & ~pos_maybe.any(axis=-1)
    assert not bad.any(), f'{what}: rows {np.flatnonzero(bad)[:5]} picked an observation with no excess that may be positive'
    decided = np.where(none, ~pos_maybe.any(axis=-1), False)
    live = np.flatnonzero(~none)
    if live.size:
        decided[live] = check_interval_argmax((lo[live], hi[live]), picked[live], pos_maybe[live], what=what)
    return decided


def check_sampled_choice(e, uniforms, picked, what='sampled o*'):
    """
    o* of the sampled rule (NumPy's searchsorted(cdf, u, 'right') over w = max(e, 0), capped at the last positive weight): where every
    excess has a certain sign and every cdf edge lies certainly on one side of u, `picked` is the exact pick.  Elsewhere `picked` is an
    observation whose excess may be positive (or -1 as `check_gap_choice` allows).  Returns the decided rows.
    """
    lo, hi = e
    K, O = lo.shape
    picked = np.asarray(picked, dtype=np.int64)
    decided = np.zeros(K, bool)
    g = LD((O + 1) * (U + U_LD))
    for k in range(K):
        l, h = lo[k], hi[k]
        poss = ~np.isnan(l)
        if not (h[poss] > 0).any():
            assert picked[k] == -1, f'{what}: trial {k} picked {picked[k]} with no excess that may be positive'
            decided[k] = True
            continue
        if picked[k] >= 0:
            assert poss[picked[k]] and h[picked[k]] > 0, f'{what}: trial {k} picked {picked[k]}, whose excess cannot be positive'
        else:
            assert not (l[poss] > 0).any(), f'{what}: trial {k} picked -1 with a certainly positive excess'
        if not np.all((l[poss] > 0) | (h[poss] <= 0)):
            continue
        w_lo = np.where(poss & (l > 0), l, LD(0))
        w_hi = np.where(poss & (h > 0), h, LD(0))
        r_lo, r_hi = np.cumsum(w_lo) * (1 - g), np.cumsum(w_hi) * (1 + g)
        c_lo = r_lo / r_hi[-1] * (1 - 2 * LD(U))
        c_hi = np.minimum(r_hi / r_lo[-1] * (1 + 2 * LD(U)), LD(1))
        uk = LD(uniforms[k])
        below, above = c_hi <= uk, c_lo > uk
        if not np.all(below | above):
            continue
        want = min(int(np.sum(below)), int(np.flatnonzero(w_hi > 0)[-1]))
        decided[k] = True
        assert picked[k] == want, f'{what}: trial {k} picked {picked[k]}, the exact draw at u = {uniforms[k]!r} is {want}'
    return decided


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
