"""
The upper-bound and gap-trial kernels against the extended-precision reference (oracle/highprec.py) at their tile, slab and list-walk
edges: pbvi_support_lists + pbvi_sawtooth_lists and the dense pbvi_sawtooth, pbvi_upper_backup, pbvi_gap_trial_step, pbvi_hsvi_level.

Each stage is checked as a function of its float64 inputs: the device's successor rows and masses are pinned first (rows bitwise the
reference's update, masses bitwise NumPy's sum of the un-normalised projection) and then enter the reference as inputs.  Every value
must lie in its certified interval, every decided choice must be the exact one, and where a path is otherwise invisible (a slab loop)
the launch count of the call (`pbvi_last_launches`) shows that it was taken.
"""
import numpy as np
import pytest

from oracle import highprec as hp
from oracle import pbvi_oracle as orc
from test_gap_solver import choose_np
from test_gpu_backup_edges import device, launches, pairwise, sparse_beliefs, synthetic

pytestmark = pytest.mark.gpu

GAMMA = 0.95
SAW_Q_SLAB = 4096                    # queries per launch of the dense form
FR_SLAB = 65535 * 8                  # rows per launch of few_rows_scores_kernel


@pytest.fixture(scope='module')
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), 'these tests need a CUDA device'
    return torch


# ---- helpers ---------------------------------------------------------------------------------------------------------------------
def cuda(torch, x):
    return torch.as_tensor(np.ascontiguousarray(x), device='cuda')


def support_lists(torch, dev, rows, corner):
    """pbvi_support_lists of `rows`: (idx, val, count, dot) CUDA tensors; the lists hold exactly the positive entries of each row."""
    n, S = rows.shape
    idx = torch.zeros((max(n, 1), S), dtype=torch.int32, device='cuda')
    val = torch.zeros((max(n, 1), S), dtype=torch.float64, device='cuda')
    count = torch.zeros((max(n, 1),), dtype=torch.int32, device='cuda')
    dot = torch.zeros((max(n, 1),), dtype=torch.float64, device='cuda')
    if n:
        dev.support_lists(cuda(torch, rows), cuda(torch, corner), idx[:n], val[:n], count[:n], dot[:n])
        cnt = count.cpu().numpy()
        for i in range(n):
            sup = np.flatnonzero(rows[i] > 0)
            assert cnt[i] == sup.size
            got = idx[i, :cnt[i]].cpu().numpy()
            assert np.array_equal(np.sort(got), sup)
            assert val[i, :cnt[i]].cpu().numpy().tobytes() == rows[i, got].tobytes()
    return idx, val, count, dot


def pinned_successors(model, B, succ, mass):
    """The successor rows are bitwise the reference's update (NaN rows for impossible observations) and the masses bitwise NumPy's sum
    of the un-normalised projection."""
    reach, _, rto, _ = model
    assert np.array_equal(succ, orc.all_successors(reach, rto, B), equal_nan=True)
    n, A, O = mass.shape
    want = np.array([[[np.sum(orc.belief_update(reach, rto, B[i], a, o, normalise=False)) for o in range(O)] for a in range(A)]
                     for i in range(n)])
    assert mass.tobytes() == want.tobytes()


def store_for(rng, S, n_ub, corner, lead=None):
    """n_ub stored beliefs (the first one `lead` when given) with values below their corner value, so that their terms bind."""
    rows = sparse_beliefs(rng, n_ub, S, [S, 40, 5, 1])
    if lead is not None and n_ub:
        rows[0] = lead
    vals = rows @ corner - (0.05 + 0.5 * rng.random(n_ub)) * np.abs(rows @ corner)
    return rows, vals


# ---- sawtooth: list walk and dense ranges ------------------------------------------------------------------------------------------
def sawtooth_both(torch, dev, corner, rows, vals, Q, vals_dev=None):
    """pbvi_sawtooth_lists and pbvi_sawtooth on the same store: both inside the reference's intervals and bitwise equal.  `vals_dev`
    replaces the stored values after the lists are built (a value equal to the device's own dot)."""
    idx, val, count, dot = support_lists(torch, dev, rows, corner)
    if vals_dev is not None:
        vals = vals_dev(dot.cpu().numpy()[:len(rows)])
    n_ub = len(rows)
    lists = dev.sawtooth_lists(cuda(torch, corner), idx, val, count, dot, cuda(torch, vals if n_ub else np.zeros(1)), n_ub,
                               cuda(torch, Q)).cpu().numpy()
    dense = dev.sawtooth(corner, rows, vals, Q).cpu().numpy()
    lo, hi = hp.sawtooth(corner, rows, vals, Q)
    hp.check_interval(lists, (lo, hi), what='sawtooth_lists')
    hp.check_interval(dense, (lo, hi), what='sawtooth')
    assert lists.tobytes() == dense.tobytes()
    return lists, lo, hi


# n_q across the query tile, support counts across the warp, the block and the 1024-entry chunk; the deciding entry is the last state
# of the support ('zero': the only zero ratio of the query; 'nested': the smallest of all-positive ratios); n_ub 0, 1, several
SAW_CASES = pairwise([(1, 7, 8, 9, 17), (1, 255, 256, 257, 1023, 1024, 1025, 2049), ('zero', 'nested'), (0, 1, 6)],
                     cost=lambda c: c[0] * c[1] * max(c[3], 1))


@pytest.mark.parametrize('nq,cnt,mode,n_ub', SAW_CASES)
def test_sawtooth_list_walk_edges(torch_cuda, nq, cnt, mode, n_ub):
    """The deciding stored belief has its support on states 0 .. cnt - 1, so the list entry of the last state is the last of the list
    (entry cnt - 1, in the last 1024-entry chunk); every query also holds 1e-13 entries outside that support (the v0 dot must keep them:
    30 of them move v0 by tens of bounds).  Extra stored beliefs: a query itself, one whose value is its own dot (scale 0), one with
    subnormal entries."""
    torch = torch_cuda
    S = cnt + 40
    model = synthetic(S, 2, 2, 1, seed=cnt + nq)
    dev = device(model)
    rng = np.random.default_rng(cnt * 31 + nq)
    corner = 1.0 + 2.0 * rng.random(S)
    lead = np.zeros(S)
    lead[:cnt] = rng.dirichlet(np.ones(cnt))
    Q = np.zeros((nq, S))
    for k in range(nq):
        Q[k, :cnt] = lead[:cnt] * (1.0 + rng.random(cnt))                # ratios in (1, 2) ...
        Q[k, cnt - 1] = 0.0 if mode == 'zero' else 0.5 * lead[cnt - 1]   # ... but for the last state: 0 or 0.5
        Q[k, cnt + 2: cnt + 32] = 5e-13
        Q[k, cnt + 38] = 0.2
        if k % 3 == 2:
            Q[k, cnt + 36] = 0.3                                          # a state outside the lead's support
        Q[k] /= Q[k].sum()
    rows, vals = store_for(rng, S, n_ub, corner, lead)
    vals_dev = None
    if n_ub > 1:
        rows[1] = Q[0]                                                    # a query equal to a stored belief
        rows[2, :] = 0.0
        rows[2, [cnt + 36, 0]] = [1e-310, 1.0]                            # a subnormal stored entry: 0.3 / 1e-310 overflows to inf
        vals = rows @ corner - (0.05 + 0.5 * rng.random(n_ub)) * np.abs(rows @ corner)

        def vals_dev(dot):
            v = vals.copy()
            v[3] = dot[3]                                                 # scale 0: the term is v0 exactly
            return v
    got, lo, hi = sawtooth_both(torch, dev, corner, rows, vals, Q, vals_dev)
    if n_ub and mode == 'nested':
        v0 = Q @ corner
        assert np.all(got < v0 - 1e-3 * np.abs(v0))                       # the lead's term binds
    dev.close()


@pytest.mark.parametrize('S', [1, 2, 255, 256, 257, 8191, 8192, 8193, 16385])
def test_dense_sawtooth_state_ranges(torch_cuda, S):
    """The dense form compacts each stored belief 8192 states at a time: the deciding state is the last one, in the last range."""
    torch = torch_cuda
    model = synthetic(S, 1, 2, 1, seed=S)
    dev = device(model)
    rng = np.random.default_rng(S)
    corner = 1.0 + rng.random(S)
    lead = rng.dirichlet(np.ones(S))
    Q = np.stack([lead * (1.0 + rng.random(S)) for _ in range(3)])
    Q[:, S - 1] = [0.5 * lead[S - 1], 0.0, 0.25 * lead[S - 1]]
    Q = np.where(Q.sum(1, keepdims=True) > 0, Q, 1.0)
    Q /= Q.sum(1, keepdims=True)
    rows, vals = store_for(rng, S, 4, corner, lead)
    sawtooth_both(torch, dev, corner, rows, vals, Q)
    dev.close()


@pytest.mark.parametrize('nq', [4095, 4096, 4097])
def test_dense_sawtooth_query_slabs(torch_cuda, nq):
    """Queries past 4096 take a second dense launch; the count of the call shows it (v0, one terms launch per slab, row minimum)."""
    torch = torch_cuda
    S = 40
    model = synthetic(S, 1, 2, 1, seed=nq)
    dev = device(model)
    rng = np.random.default_rng(nq)
    corner = 1.0 + rng.random(S)
    Q = sparse_beliefs(rng, nq, S, [S, 9, 3, 1])
    rows, vals = store_for(rng, S, 5, corner)
    rows[0] = Q[-1] * (1.0 + rng.random(S))                              # the last query (second slab) nests in a stored belief
    rows[0] /= rows[0].sum()
    vals[0] = rows[0] @ corner - 0.5
    sawtooth_both(torch, dev, corner, rows, vals, Q)
    dev.sawtooth(corner, rows, vals, Q)
    assert launches(dev) == 2 + -(-nq // SAW_Q_SLAB)
    dev.close()


# ---- pbvi_upper_backup ---------------------------------------------------------------------------------------------------------------
def reward_columns(rng, rbar):
    """Rbar with an all-zero first action column and a last column with a non-zero reward on every state (> 32 for S > 32)."""
    rbar = rbar.copy()
    rbar[:, 0] = 0.0
    rbar[:, -1] = 0.1 + rng.random(rbar.shape[0])
    return rbar


def upper_checked(torch, dev, model, B, F, corner, rows, vals, pin=True):
    """pbvi_upper_backup on B: u, cur and a* against the reference at the device's own successors and masses.  Returns (u, a*, the
    call's launch count)."""
    reach, _, rto, rbar = model
    n_ub = len(rows)
    idx, val, count, dot = support_lists(torch, dev, rows, corner)
    u, cur, act = dev.upper_backup(B, cuda(torch, F), GAMMA, cuda(torch, corner), idx, val, count, dot,
                                   cuda(torch, vals if n_ub else np.zeros(1)), n_ub, want_action=True)
    n_launches = launches(dev)
    u, cur, act = u.cpu().numpy(), cur.cpu().numpy(), act.cpu().numpy()
    succ, mass = [t.cpu().numpy() for t in dev.belief_successors(B)]
    if pin:
        pinned_successors(model, B, succ, mass)
    ref = hp.upper_q(B, rbar, GAMMA, succ, mass, F, corner, rows, vals)
    hp.check_interval(u, ref['u'], what='u')
    hp.check_interval(cur, ref['cur'], what='cur')
    ex, bd = hp.as_center(ref['Q'])
    hp.check_argmax(ex, bd, act, what='a*')
    return u, act, n_launches


# k FIB rows across the 8-row tile; n beliefs across the 128-thread block of upper_q_kernel; (A, O) such that n A O crosses the 8-row
# tile and n A is not a multiple of 8
UB_CASES = pairwise([(1, 7, 8, 9, 17), (1, 3, 127, 128, 129), ((1, 1), (3, 3), (2, 5), (5, 2)), (0, 1, 6)],
                    cost=lambda c: c[0] * c[1] * c[2][0] * c[2][1] * max(1, c[3]))


@pytest.mark.parametrize('k,n,AO,n_ub', UB_CASES)
def test_upper_backup_edges(torch_cuda, k, n, AO, n_ub):
    torch = torch_cuda
    A, O = AO
    S = 48
    rng = np.random.default_rng(k * 1000 + n * 10 + A)
    reach, probs, rto, rbar = synthetic(S, A, O, 1, seed=k + n + A * O)
    model = (reach, probs, rto, reward_columns(rng, rbar))
    dev = device(model)
    B = sparse_beliefs(rng, n, S, [S, 40, 5, 1])
    F = 1.0 + rng.random((k, S)) * 20.0
    corner = F.max(axis=0)
    rows, vals = store_for(rng, S, n_ub, corner)
    if n_ub:
        rows[0] = B[0]                                                    # b itself is stored: its sawtooth term binds for cur
        vals[0] = B[0] @ corner - 3.0
    upper_checked(torch, dev, model, B, F, corner, rows, vals)
    dev.close()


def test_upper_backup_second_few_rows_slab(torch_cuda):
    """90 000 beliefs of a tiger-sized model (S = 2, A = 3, O = 2): 540 000 successors, past the 524 280 rows of one few-rows launch."""
    torch = torch_cuda
    rng = np.random.default_rng(90)
    model = synthetic(2, 3, 2, 1, seed=90)
    dev = device(model)
    n = 90000
    assert n * 3 * 2 > FR_SLAB
    B = rng.dirichlet(np.ones(2), size=n)
    B[::7] = [1.0, 0.0]
    F = 5.0 + rng.random((3, 2))
    corner = F.max(axis=0)
    rows = np.array([[0.3, 0.7], [0.9, 0.1]])
    vals = rows @ corner - 0.5
    u, act, n_big = upper_checked(torch, dev, model, B, F, corner, rows, vals, pin=False)
    n_small = 8 * (65535 // 6)                                            # eight whole successor slabs, 524 256 successors: one launch
    idx, val, count, dot = support_lists(torch, dev, rows, corner)
    dev.upper_backup(B[:n_small], cuda(torch, F), GAMMA, cuda(torch, corner), idx, val, count, dot, cuda(torch, vals), 2)
    assert n_big == launches(dev) + 2 + 1                                 # one more successor slab (projection + normaliser), one more few-rows launch
    tail = dev.upper_backup(B[n_small:], cuda(torch, F), GAMMA, cuda(torch, corner), idx, val, count, dot, cuda(torch, vals), 2)[0]
    assert tail.cpu().numpy().tobytes() == u[n_small:].tobytes()
    dev.close()


# ---- pbvi_gap_trial_step -----------------------------------------------------------------------------------------------------------
def gap_model(rng, S, A, O):
    """A synthetic model in which action 0 has every observation impossible from states 0 .. 2, where it pays 1000: a belief there takes
    a* = 0 and has no possible observation."""
    reach, probs, rto, rbar = synthetic(S, A, O, 1, seed=S + A * O)
    rto = rto.copy()
    rto[:3, 0] = 0.0
    rbar = reward_columns(rng, rbar)
    rbar[:3, 0] = 1000.0
    return reach, probs, rto, rbar


def step_checked(torch, dev, model, B, X, F, corner, rows, vals, theta, uniforms):
    """One pbvi_gap_trial_step against the reference; returns (o*, e computed by NumPy from the device's U and L)."""
    reach, _, rto, rbar = model
    n_ub = len(rows)
    idx, val, count, dot = support_lists(torch, dev, rows, corner)
    lists = (cuda(torch, corner), idx, val, count, dot, cuda(torch, vals if n_ub else np.zeros(1)), n_ub)
    u_ref, _, a_ref = dev.upper_backup(B, cuda(torch, F), GAMMA, *lists, want_action=True)
    out, nxt, U, L = dev.gap_trial_step(B, cuda(torch, X), cuda(torch, F), GAMMA, *lists, theta,
                                        None if uniforms is None else cuda(torch, uniforms), want_bounds=True)
    out, nxt, U, L = [t.cpu().numpy() for t in (out, nxt, U, L)]
    a, o = out[:, 0].astype(np.int64), out[:, 1].astype(np.int64)
    assert np.array_equal(a, a_ref.cpu().numpy()) and out[:, 2].tobytes() == u_ref.cpu().numpy().tobytes()
    K = len(B)
    succ, mass = [t.cpu().numpy() for t in dev.belief_successors(B)]
    sa, ma = succ[np.arange(K), np.maximum(a, 0)], mass[np.arange(K), np.maximum(a, 0)]
    ma = np.where(a[:, None] >= 0, ma, 0.0)
    ref = hp.gap_step(sa, ma, F, corner, rows, vals, X, theta)
    hp.check_interval(U, ref['U'], what='U')
    hp.check_interval(L, ref['L'], what='L')
    e_dev = np.where(ma > 0, ma * ((U - L) - theta), np.nan)
    hp.check_interval(e_dev, ref['e'], what='e')
    for k in range(K):
        uk = None if uniforms is None else uniforms[k]
        assert o[k] == choose_np(e_dev[k], uk), (k, uk)                  # NumPy's rule on the device's own U, L, bit for bit
    sampled = np.zeros(K, bool) if uniforms is None else uniforms >= 0
    hp.check_gap_choice((ref['e'][0][~sampled], ref['e'][1][~sampled]), o[~sampled])
    if sampled.any():
        hp.check_sampled_choice((ref['e'][0][sampled], ref['e'][1][sampled]), uniforms[sampled], o[sampled])
    live = o >= 0
    assert np.all(out[live, 3] == e_dev[live, o[live]])
    hp.check_interval(out[live, 3], (ref['e'][0][live, o[live]], ref['e'][1][live, o[live]]), what='e*')
    dead = ~live
    assert np.all(out[dead, 3] == np.where(np.any(ma[dead] > 0, axis=1), np.nanmax(np.where(ma[dead] > 0, e_dev[dead], -np.inf), axis=1),
                                           -np.inf))
    if live.any():
        want, _ = dev.belief_update(B[live], a[live].astype(np.int32), o[live].astype(np.int32))
        assert nxt[live].tobytes() == want.cpu().numpy().tobytes()
    assert nxt[dead].tobytes() == B[dead].tobytes()
    return o, e_dev


# K across the 128-thread block; N lower rows across the score kernel's 64-column quarter and 256-column tile; O = 1 included
GAP_CASES = pairwise([(1, 127, 128, 129), (1, 63, 64, 65, 257), (1, 2, 5), (0, 4)], cost=lambda c: c[0] * c[1] * c[2] * max(1, c[3]))


@pytest.mark.parametrize('K,N,O,n_ub', GAP_CASES)
def test_gap_trial_step_edges(torch_cuda, K, N, O, n_ub):
    torch = torch_cuda
    S, A = 30, 3
    rng = np.random.default_rng(K * 100 + N + O)
    model = gap_model(rng, S, A, O)
    dev = device(model)
    B = sparse_beliefs(rng, K, S, [S, 12, 3, 1])
    B[0] = 0.0
    B[0, :3] = 1.0 / 3                                                    # a* = 0 with every observation impossible
    F = 30.0 + 10.0 * rng.random((4, S))
    corner = F.max(axis=0)
    X = 5.0 + 20.0 * rng.random((N, S))
    rows, vals = store_for(rng, S, n_ub, corner)
    for theta in (0.0, 1e30):
        o, _ = step_checked(torch, dev, model, B, X, F, corner, rows, vals, theta, None)
        assert o[0] == -1 and (theta == 0.0 or np.all(o == -1))
    # uniforms 0, just below 1, 1 (the cap), above 1, a random one and the argmax rule; then u exactly on the device's cdf values
    uni = np.resize(np.array([0.0, 1.0 - 2.0 ** -53, 1.0, 1.5, float(rng.random()), -1.0]), K)
    o, e_dev = step_checked(torch, dev, model, B, X, F, corner, rows, vals, 0.0, uni)
    on_edge = uni.copy()
    for k in range(K):
        w = np.where(e_dev[k] > 0, e_dev[k], 0.0)
        if np.count_nonzero(w) >= 2:
            cdf = np.cumsum(w)
            cdf /= cdf[-1]
            on_edge[k] = cdf[np.flatnonzero(w)[0]]                        # the first positive cdf value: searchsorted 'right' moves past it
    step_checked(torch, dev, model, B, X, F, corner, rows, vals, 0.0, on_edge)
    dev.close()


# ---- pbvi_hsvi_level ---------------------------------------------------------------------------------------------------------------
def hsvi_checked(torch, dev, model, b, V, corner, rows, vals, keys, kvals, n_stored, conv, may_continue=True):
    """One pbvi_hsvi_level: Q, a*, o* and the gap of the chosen successor against the reference; a successor whose key is stored takes
    the stored value.  Returns (result, meta, successors, masses)."""
    reach, _, rto, rbar = model
    n_ub = len(rows)
    idx, val, count, dot = support_lists(torch, dev, rows, corner)
    succ, mass, res, meta = dev.hsvi_level(cuda(torch, b), cuda(torch, V), GAMMA, cuda(torch, corner), idx, val, count, dot,
                                           cuda(torch, vals if n_ub else np.zeros(1)), n_ub, keys, kvals, n_stored, conv, may_continue)
    succ, mass = succ.cpu().numpy(), mass.cpu().numpy()
    pinned_successors(model, b[None], succ[None], mass[None])
    A, O = mass.shape
    live = mass > 0
    y_lo = np.full((A, O), hp.LD(np.nan))
    y_hi = np.full((A, O), hp.LD(np.nan))
    if live.any():
        y_lo[live], y_hi[live] = hp.sawtooth(corner, rows, vals, succ[live])
        skeys = dev.row_hash(cuda(torch, succ.reshape(A * O, -1))).cpu().numpy().reshape(A, O, 2)
        table = {tuple(k): float(v) for k, v in zip(keys[:n_stored].cpu().numpy(), kvals[:n_stored].cpu().numpy())}
        for a, o in zip(*np.nonzero(live)):
            if tuple(skeys[a, o]) in table:
                y_lo[a, o] = y_hi[a, o] = hp.LD(table[tuple(skeys[a, o])])
    Q = hp.q_values(b[None], rbar, GAMMA, mass[None], y_lo[None], y_hi[None])
    best_a, best_o, max_q, diff = int(res[0]), int(res[1]), float(res[2]), float(res[3])
    ex, bd = hp.as_center(Q)
    hp.check_argmax(ex, bd, [best_a], what='a*')
    hp.check_interval([max_q], (Q[0][:, best_a], Q[1][:, best_a]), what='max Q')
    lo_l, hi_l = np.full(O, hp.LD(np.nan)), np.full(O, hp.LD(np.nan))
    la = live[best_a]
    if la.any():
        lo_l[la], hi_l[la] = hp.max_scores(succ[best_a][la], V)
    ov = hp.excess(mass[best_a][None], (y_lo[best_a][None], y_hi[best_a][None]), (lo_l[None], hi_l[None]), 0.0)
    if la.any():
        hp.check_interval_argmax(ov, [best_o], la[None], what='o*')
        d = hp.excess(np.ones((1, O)), (y_lo[best_a][None], y_hi[best_a][None]), (lo_l[None], hi_l[None]), 0.0)
        hp.check_interval([diff], (d[0][:, best_o], d[1][:, best_o]), what='upper - lower')
    else:
        assert best_o == -1
    return res, meta, succ, mass


@pytest.mark.parametrize('A,O', [(1, 1), (3, 2), (8, 7), (16, 20)])
def test_hsvi_level_edges(torch_cuda, A, O):
    """A O = 1 .. 320 doubles of the choose kernel's shared memory; a stored successor key (its stored value wins); the append on both
    sides of conv_term, at capacity (no append) and with b already stored."""
    torch = torch_cuda
    S = 30
    rng = np.random.default_rng(A * O)
    reach, probs, rto, rbar = synthetic(S, A, O, 1, seed=A * 10 + O)
    model = (reach, probs, rto, reward_columns(rng, rbar) if A > 1 else rbar)
    dev = device(model)
    b = rng.dirichlet(np.ones(S))
    V = rng.random((70, S)) * 5.0
    corner = 10.0 + rng.random(S)
    rows, vals = store_for(rng, S, 5, corner)
    cap = 8
    keys = torch.zeros((cap, 2), dtype=torch.int64, device='cuda')
    kvals = torch.zeros((cap,), dtype=torch.float64, device='cuda')
    # first level: nothing stored, the chosen successor's key then goes into the store with a value below its sawtooth
    res, meta, succ, mass = hsvi_checked(torch, dev, model, b, V, corner, rows, vals, keys, kvals, 0, -1e30)
    assert int(meta[0]) == 1 and kvals[0].item() == float(res[2])                   # appended: (key(b), Q)
    live = np.argwhere(mass > 0)
    a0, o0 = live[-1]
    keys[1] = dev.row_hash(cuda(torch, succ[a0, o0][None]))[0]
    kvals[1] = -7.5
    res, meta, _, _ = hsvi_checked(torch, dev, model, b, V, corner, rows, vals, keys, kvals, 2, -1e30)
    assert int(meta[0]) == 0                                                        # b is stored already
    # b not stored: conv_term just above the chosen gap stops the append, at the gap itself it appends; at capacity it cannot
    keys[0] = 0
    res, meta, _, _ = hsvi_checked(torch, dev, model, b, V, corner, rows, vals, keys, kvals, 2, -1e30)
    diff = float(res[3])
    res, meta, _, _ = hsvi_checked(torch, dev, model, b, V, corner, rows, vals, keys, kvals, 2, float(np.nextafter(diff, np.inf)))
    assert int(meta[0]) == 0 and float(res[3]) == diff
    res, meta, _, _ = hsvi_checked(torch, dev, model, b, V, corner, rows, vals, keys, kvals, 2, diff)
    assert int(meta[0]) == 1 and kvals[2].item() == float(res[2])
    full_keys, full_vals = keys[:3].clone(), kvals[:3].clone()
    full_keys[2] = 0
    res, meta, _, _ = hsvi_checked(torch, dev, model, b, V, corner, rows, vals, full_keys, full_vals, 3, -1e30)
    assert int(meta[0]) == 0 and full_vals[2].item() == kvals[2].item()
    dev.close()
