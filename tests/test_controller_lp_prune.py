"""
LP (convex-combination) dominance of controller nodes, with stochastic successor edges (mixtures).  Checked:
  * pbvi_prune_lp_certificates: keep flags, bounds and counts bitwise those of pbvi_prune_lp; every certificate re-checked in NumPy FP64
    and against HiGHS witness margins;
  * pbvi_controller_evaluate_mixed / pbvi_controller_outcomes_mixed: bitwise the calls without mixtures when there are none, and bitwise
    NumPy restatements (mixture rows, then the sweep in the kernel's order) sweep by sweep / step by step;
  * PolicyGraph.prune_lp on extracted, improved and gap-solved controllers: fewer nodes, bitwise the same value, the certificate without
    re-evaluation, a re-evaluation that does not fall, and roll-outs that agree with the exact outcomes;
  * on the CPU: certificate resolution on hand-made chains, the constructor's checks, the .pg / .mix files, and simulate unchanged for a
    graph without mixtures.
"""
import os
import types

import numpy as np
import pytest

from test_controller_outcomes import outcomes_np, planted
from test_policy_graph import controller_sweep_np
from test_prune_lp import MODELS as LP_MODELS, lp_witness_margins, seeded_solve as lp_seeded_solve, tol_of
from test_upper_bound import fixture_model, seeded_solve


# ---- CPU: certificate resolution ---------------------------------------------------------------------------------------------------
def certs(n, table):
    idx, w = np.full((n, 64), -1, dtype=np.int64), np.zeros((n, 64))
    for i, pairs in table.items():
        for q, (j, lam) in enumerate(pairs):
            idx[i, q], w[i, q] = j, lam
    return idx, w


def check_resolved(res, pruned):
    for i, (nodes, weights) in res.items():
        assert pruned[i] and not np.any(pruned[nodes]) and np.all(np.diff(nodes) > 0)
        assert np.all(weights > 0) and abs(weights.sum() - 1.0) <= 1e-12, (i, weights.sum())


def test_certificates_resolve_through_pruned_chains():
    from pomdp_pbvi_exploration_b200.policy_graph import resolve_certificates
    pruned = np.zeros(8, dtype=bool)
    pruned[[3, 4, 5, 6]] = True
    # 3 -> {0, 4}, 4 -> {1, 5}, 5 -> {2}: a chain through two pruned nodes; 6 -> {3, 7}
    idx, w = certs(8, {3: [(0, 0.5), (4, 0.5)], 4: [(1, 0.25), (5, 0.75)], 5: [(2, 1.0)], 6: [(3, 0.5), (7, 0.5)]})
    res = resolve_certificates(pruned, idx, w)
    check_resolved(res, pruned)
    assert sorted(res) == [3, 4, 5, 6]
    np.testing.assert_array_equal(res[5][0], [2])
    np.testing.assert_array_equal(res[4][0], [1, 2])
    np.testing.assert_allclose(res[4][1], [0.25, 0.75], rtol=0, atol=1e-15)
    np.testing.assert_array_equal(res[3][0], [0, 1, 2])
    np.testing.assert_allclose(res[3][1], [0.5, 0.125, 0.375], rtol=0, atol=1e-15)
    np.testing.assert_array_equal(res[6][0], [0, 1, 2, 7])
    np.testing.assert_allclose(res[6][1], [0.25, 0.0625, 0.1875, 0.5], rtol=0, atol=1e-15)


def test_certificates_resolve_through_cycles_of_pruned_nodes():
    from pomdp_pbvi_exploration_b200.policy_graph import resolve_certificates
    pruned = np.array([False, False, True, True, True])
    # 2 -> {0, 3}, 3 -> {1, 2}, 4 -> {2, 3}: 2 and 3 lean on each other, but each keeps half its weight on a kept node
    idx, w = certs(5, {2: [(0, 0.5), (3, 0.5)], 3: [(1, 0.5), (2, 0.5)], 4: [(2, 0.5), (3, 0.5)]})
    res = resolve_certificates(pruned, idx, w)
    check_resolved(res, pruned)
    # x2 = 0.5 e0 + 0.5 x3, x3 = 0.5 e1 + 0.5 x2  =>  x2 = (2/3) e0 + (1/3) e1, x3 = (1/3) e0 + (2/3) e1
    np.testing.assert_allclose(res[2][1], [2 / 3, 1 / 3], rtol=0, atol=1e-12)
    np.testing.assert_allclose(res[3][1], [1 / 3, 2 / 3], rtol=0, atol=1e-12)
    np.testing.assert_allclose(res[4][1], [0.5, 0.5], rtol=0, atol=1e-12)


def test_random_certificates_resolve_to_convex_combinations_of_kept_nodes():
    from pomdp_pbvi_exploration_b200.policy_graph import resolve_certificates
    rng = np.random.default_rng(3)
    n = 300
    pruned = rng.random(n) < 0.6
    kept = np.flatnonzero(~pruned)
    table = {}
    for i in np.flatnonzero(pruned):
        k = int(rng.integers(1, 8))
        J = rng.choice(np.delete(np.arange(n), i), size=k, replace=False)
        if not np.any(~pruned[J]):
            J[0] = rng.choice(kept)                                # a strict margin: some weight always lands on a kept node
        lam = rng.dirichlet(np.ones(k))
        table[int(i)] = list(zip(J.tolist(), lam.tolist()))
    idx, w = certs(n, table)
    res = resolve_certificates(pruned, idx, w)
    check_resolved(res, pruned)
    assert len(res) == int(pruned.sum())


# ---- CPU: representation -------------------------------------------------------------------------------------------------------
def cpu_model(tag='tiger'):
    model, gamma = fixture_model(tag)
    return model, gamma


def test_constructor_checks_mixtures():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = cpu_model()
    A, O = model.action_count, model.observation_count
    act = np.arange(A)
    succ = np.repeat(np.arange(A)[:, None], O, axis=1)
    good = (np.array([0, 2]), np.array([0, 1]), np.array([0.25, 0.75]))
    pg = PolicyGraph(model, act, np.where(np.arange(O)[None, :] == 0, A, succ), mixtures=good)
    assert pg.mixtures[0].dtype == np.int64 and pg.mixtures[2].dtype == np.float64
    assert PolicyGraph(model, act, succ, mixtures=(np.array([0]), np.zeros(0, np.int64), np.zeros(0))).mixtures is None
    bad = {
        'offsets must rise': (np.array([0, 0, 2]), np.array([0, 1]), np.array([0.5, 0.5])),
        'offsets must rise ': (np.array([1, 2]), np.array([0, 1]), np.array([0.5, 0.5])),
        'one weight per member': (np.array([0, 2]), np.array([0, 1]), np.array([1.0])),
        'members must be nodes': (np.array([0, 2]), np.array([0, A]), np.array([0.5, 0.5])),
        'members must be nodes ': (np.array([0, 2]), np.array([-1, 0]), np.array([0.5, 0.5])),
        'finite and >= 0': (np.array([0, 2]), np.array([0, 1]), np.array([1.5, -0.5])),
        'finite and >= 0 ': (np.array([0, 2]), np.array([0, 1]), np.array([np.nan, 1.0])),
        'sum to 1': (np.array([0, 2]), np.array([0, 1]), np.array([0.5, 0.5 + 1e-11])),
        'integer arrays': (np.array([0.0, 2.0]), np.array([0, 1]), np.array([0.5, 0.5])),
        'tuple': (np.array([0, 2]), np.array([0, 1])),
    }
    for msg, mix in bad.items():
        with pytest.raises(ValueError, match=msg.strip()):
            PolicyGraph(model, act, succ, mixtures=mix)
    with pytest.raises(ValueError, match='successor entries'):
        PolicyGraph(model, act, np.full((A, O), A + 1), mixtures=good)                 # one mixture: entries up to A only
    with pytest.raises(ValueError, match='successor entries'):
        PolicyGraph(model, act, np.full((A, O), A))                                     # no mixtures: entries below A
    assert abs(good[2].sum() - 1.0) == 0.0


def mixed_graph(model, rng, N, M):
    """A random graph with N nodes and M mixtures (without rows), about a third of its edges into mixtures."""
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    A, O = model.action_count, model.observation_count
    sizes = rng.integers(1, 5, size=M)
    off = np.concatenate([[0], np.cumsum(sizes)])
    nodes = rng.integers(0, N, size=int(off[-1]))
    w = np.concatenate([rng.dirichlet(np.ones(k)) for k in sizes])
    for m in range(M):                                              # sums within 1e-12 after a renormalisation
        w[off[m]:off[m + 1]] /= w[off[m]:off[m + 1]].sum()
    succ = rng.integers(0, N, size=(N, O))
    into = rng.random((N, O)) < 0.35
    succ[into] = N + rng.integers(0, M, size=int(into.sum()))
    return PolicyGraph(model, rng.integers(0, A, size=N), succ, mixtures=(off, nodes, w))


def test_pg_and_mix_files_round_trip_bitwise(tmp_path):
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = cpu_model('hallway')
    pg = mixed_graph(model, np.random.default_rng(5), 40, 9)
    pg.save(str(tmp_path), 'g')
    back = PolicyGraph.load(str(tmp_path), 'g', model)
    assert np.array_equal(back.actions, pg.actions) and np.array_equal(back.successors, pg.successors)
    for a, b in zip(back.mixtures, pg.mixtures):
        assert a.dtype == b.dtype and a.tobytes() == b.tobytes()
    first = (tmp_path / 'g.mix').read_text().splitlines()[0].split()
    k = int(first[1])
    assert first[0] == '0' and len(first) == 2 + 2 * k and first[3] == '%.17g' % pg.mixtures[2][0]
    (tmp_path / 'g.mix').write_text('1 1 0 1\n')
    with pytest.raises(ValueError, match='mixture_id'):
        PolicyGraph.load(str(tmp_path), 'g', model)


def test_files_of_a_graph_without_mixtures_are_unchanged(tmp_path):
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = cpu_model('tiger')
    pg = PolicyGraph(model, [0, 1, 2], [[1, 2], [0, 0], [2, 1]])
    pg.save(str(tmp_path), 'g')
    assert sorted(os.listdir(tmp_path)) == ['g.pg']
    assert (tmp_path / 'g.pg').read_bytes() == b'0 0 1 2\n1 1 0 0\n2 2 2 1\n'
    assert PolicyGraph.load(str(tmp_path), 'g', model).mixtures is None


def cpu_rows(pg, node0):
    """Rows for host-only checks: a CPU stand-in for the device (`belief_rows` goes to model.device.device) and the start node."""
    import torch
    model = types.SimpleNamespace(**vars(pg.model))
    model.device = types.SimpleNamespace(device=torch.device('cpu'))
    pg.model = model
    pg.rows = torch.zeros((len(pg), model.state_count), dtype=torch.float64)
    pg.gamma = 0.95
    pg.value = lambda b: (torch.zeros(1, dtype=torch.float64), torch.full((1,), node0, dtype=torch.int32))
    return pg


def simulate_without_mixtures(pg, node0, n, max_steps, seed):
    """The roll-outs of `simulate` as they were before mixtures existed (the same draws in the same order)."""
    m = pg.model
    reach, rto, rbar = np.asarray(m.reachable_states), m.reachable_transitional_observation_table, m.expected_rewards_table
    S, A, O, R = rto.shape
    p = np.asarray(m.start_probabilities, dtype=np.float64)
    rng = np.random.default_rng(seed)
    s = rng.choice(S, size=n, p=p / p.sum())
    node = np.full(n, node0, dtype=np.int64)
    cdf = np.cumsum(rto.reshape(S, A, O * R), axis=2)
    ret, disc = np.zeros(n), 1.0
    for _ in range(max_steps):
        a = pg.actions[node]
        ret += disc * rbar[s, a]
        u = rng.random(n)
        k = np.minimum((cdf[s, a] <= u[:, None]).sum(axis=1), O * R - 1)
        s = reach[s, a, k % R]
        node = pg.successors[node, k // R]
        disc *= pg.gamma
    return ret


def test_simulate_without_mixtures_is_unchanged_for_a_fixed_seed():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = cpu_model('hallway')
    rng = np.random.default_rng(2)
    N = 30
    pg = cpu_rows(PolicyGraph(model, rng.integers(0, model.action_count, N), rng.integers(0, N, (N, model.observation_count))), 4)
    got = pg.simulate(500, 40, seed=9)
    assert got.tobytes() == simulate_without_mixtures(pg, 4, 500, 40, 9).tobytes()


def test_simulate_draws_mixture_members_by_their_weights():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = cpu_model('tiger')
    A, O = model.action_count, model.observation_count
    # node 0 (listen) moves to mixture 0 = {1: 0.2, 2: 0.8} on every observation.  Node 1 listens (Rbar -1 in both states), node 2
    # opens a door (Rbar -100 or 10), so the second reward tells which member was drawn.
    rbar = model.expected_rewards_table
    assert np.all(rbar[:, 0] == -1.0) and not np.any(rbar[:, 1] == -1.0)
    pg = cpu_rows(PolicyGraph(model, [0, 0, 1], [[3] * O, [1] * O, [2] * O], mixtures=([0, 2], [1, 2], [0.2, 0.8])), 0)
    pg.gamma = 1.0
    n = 20000
    second = pg.simulate(n, 2, seed=1) - rbar[0, 0]
    frac = np.mean(second == -1.0)
    assert abs(frac - 0.2) <= 4 * np.sqrt(0.2 * 0.8 / n), frac


def test_improve_rejects_a_graph_with_mixtures():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = cpu_model('tiger')
    O = model.observation_count
    pg = cpu_rows(PolicyGraph(model, [0, 1], [[2] * O, [0] * O], mixtures=([0, 2], [0, 1], [0.5, 0.5])), 0)
    with pytest.raises(ValueError, match='without mixtures'):
        pg.improve(None, 1)
    with pytest.raises(ValueError, match='without mixtures'):
        pg.prune_lp()


# ---- GPU: pbvi_prune_lp_certificates --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('tag', LP_MODELS)
def test_certificates_leave_prune_lp_bitwise_unchanged(tag):
    model, vf, _ = lp_seeded_solve(tag)
    dev = model.device
    k2 = np.flatnonzero(dev.prune_dominated(vf.alpha_vector_array).cpu().numpy())
    import torch
    P = vf.alpha_vector_array[torch.as_tensor(k2, device='cuda')].contiguous()
    keep, bound, counts = dev.prune_lp(P)
    stats = dev.prune_lp_stats()
    keep2, bound2, counts2, idx, w = dev.prune_lp_certificates(P)
    assert dev.prune_lp_stats() == stats
    assert keep2.cpu().numpy().tobytes() == keep.cpu().numpy().tobytes()
    assert bound2.cpu().numpy().tobytes() == bound.cpu().numpy().tobytes()
    assert np.array_equal(counts2, counts)
    rows, idx, w, keep = P.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy(), keep.cpu().numpy()
    tau = tol_of(rows)
    pruned = np.flatnonzero(keep == 0)
    assert np.all(idx[keep != 0] == -1) and np.all(w[keep != 0] == 0.0)
    for i in pruned:
        J = idx[i][idx[i] >= 0]
        k = len(J)
        assert k >= 1 and np.all(idx[i][k:] == -1) and np.all(w[i][k:] == 0.0) and i not in J
        lam = w[i][:k]
        assert np.all(lam >= 0.0) and abs(lam.sum() - 1.0) <= 1e-12
        assert np.all(lam @ rows[J] - rows[i] > tau), (tag, i)
    if len(pruned):
        delta = lp_witness_margins(rows)
        assert np.all(delta[pruned] < 0.0), (tag, delta[pruned].max())


@pytest.mark.gpu
def test_certificates_on_a_set_known_by_construction():
    import torch
    from test_prune_lp import bare_device, tangent_planes
    rng = np.random.default_rng(7)
    S, n_planes, n_comb = 2000, 200, 150
    planes, _ = tangent_planes(S, n_planes, 6, rng)
    comb = np.stack([rng.dirichlet(np.ones(3)) @ planes[rng.choice(n_planes, 3, replace=False)] - 1e-4 for _ in range(n_comb)])
    rows = np.concatenate([planes, comb])
    dev = bare_device(S)
    R = torch.as_tensor(rows, device='cuda')
    keep, bound, counts = dev.prune_lp(R)
    keep2, bound2, counts2, idx, w = dev.prune_lp_certificates(R)
    assert torch.equal(keep, keep2) and bound.cpu().numpy().tobytes() == bound2.cpu().numpy().tobytes() and np.array_equal(counts, counts2)
    idx, w = idx.cpu().numpy(), w.cpu().numpy()
    assert counts[2] == n_comb
    for i in np.flatnonzero(keep.cpu().numpy() == 0):
        J = idx[i][idx[i] >= 0]
        assert np.all(w[i][:len(J)] @ rows[J] - rows[i] > tol_of(rows))


# ---- GPU: the mixed entry points ------------------------------------------------------------------------------------------------
def mixture_np(X, mixtures):
    off, nodes, w = mixtures
    Z = np.empty((len(off) - 1, X.shape[1]))
    for m in range(len(off) - 1):
        z = w[off[m]] * X[nodes[off[m]]]
        for k in range(off[m] + 1, off[m + 1]):
            z = z + w[k] * X[nodes[k]]
        Z[m] = z
    return Z


def random_mixtures(pg, rng, M):
    """pg with M random mixtures over its nodes and about a third of its edges sent to them (rows and gamma kept)."""
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    N, O = len(pg), pg.model.observation_count
    sizes = rng.integers(1, 6, size=M)
    off = np.concatenate([[0], np.cumsum(sizes)])
    w = np.concatenate([rng.dirichlet(np.ones(k)) for k in sizes])
    succ = pg.successors.copy()
    into = rng.random((N, O)) < 0.35
    succ[into] = N + rng.integers(0, M, size=int(into.sum()))
    out = PolicyGraph(pg.model, pg.actions, succ, rows=pg.rows, mixtures=(off, rng.integers(0, N, size=int(off[-1])), w))
    out.gamma = pg.gamma
    return out


def extracted_graph(tag):
    from test_policy_graph import extracted
    model, gamma, _, B, pg, _ = extracted(tag)
    return model, gamma, B, pg


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x3', 'hallway', 'tigergrid'])
def test_mixed_entry_points_without_mixtures_are_the_plain_calls(tag):
    import torch
    model, gamma, B, pg = extracted_graph(tag)
    dev = model.device
    act = torch.as_tensor(pg.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(pg.successors, dtype=torch.int32, device='cuda')
    none = (np.zeros(1, np.int64), np.zeros(0, np.int64), np.zeros(0))
    W0 = pg.rows - 1.0
    a = dev.controller_evaluate(W0, gamma, act, succ, 1e-9, 50)
    b = dev.controller_evaluate_mixed(W0, gamma, act, succ, none, 1e-9, 50)
    assert a[2] == b[2] and torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    m = planted(model)
    q = np.concatenate([model.start_probabilities[None, :], B[:5]])
    nodes = np.arange(len(q)) % len(pg)
    es = np.zeros(model.state_count, np.uint8)
    es[np.asarray(m.end_states)] = 1
    ea = np.zeros(model.action_count, np.uint8)
    x = dev.controller_outcomes(pg.actions, pg.successors, es, ea, gamma, 25, q, nodes)
    y = dev.controller_outcomes_mixed(pg.actions, pg.successors, none, es, ea, gamma, 25, q, nodes)
    assert all(torch.equal(u, v) for u, v in zip(x, y))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x3', 'hallway', 'tigergrid'])
def test_mixed_evaluate_is_the_numpy_restatement_sweep_by_sweep(tag):
    import torch
    model, gamma, B, pg = extracted_graph(tag)
    mg = random_mixtures(pg, np.random.default_rng(17), max(2, len(pg) // 3))
    dev = model.device
    act = torch.as_tensor(mg.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(mg.successors, dtype=torch.int32, device='cuda')
    X = pg.rows.cpu().numpy() - 0.5
    W = X.copy()
    for k in range(1, 5):
        TW = controller_sweep_np(model, mg.actions, mg.successors, np.concatenate([W, mixture_np(W, mg.mixtures)]), gamma)[:len(mg)]
        out, changes, kk = dev.controller_evaluate_mixed(torch.as_tensor(X, device='cuda'), gamma, act, succ, mg.mixtures, 0.0, k)
        assert kk == k
        assert out.cpu().numpy().tobytes() == TW.tobytes(), (tag, k)
        assert float(changes[-1]) == float(np.max(np.abs(TW - W)))
        W = TW
    # mixture_rows (the host's verification path) is the mixture phase's arithmetic
    from pomdp_pbvi_exploration_b200.policy_graph import mixture_rows
    assert mixture_rows(torch.as_tensor(W, device='cuda'), mg.mixtures).cpu().numpy().tobytes() == mixture_np(W, mg.mixtures).tobytes()


def outcomes_mixed_np(model, actions, succ, mixtures, gamma, k):
    """k steps of the outcome recursions with mixtures: each step reads [rows; mixture rows] (outcomes_np's step on extended rows)."""
    N, S = len(actions), model.state_count
    P, M, G = np.zeros((N, S)), np.zeros((N, S)), np.zeros((N, S))
    out = []
    for _ in range(k):
        ext = [np.concatenate([X, mixture_np(X, mixtures)]) for X in (P, M, G)]
        P, M, G = step_np(model, actions, succ, ext, gamma)
        out.append((P, M, G))
    return out


def step_np(model, actions, succ, ext, gamma):
    """One step of the outcome recursions from the rows `ext` = (P, M, G) (extended by mixture rows), in the kernel's order: outcomes_np's
    step with the rows read from `ext`."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, R = reach.shape
    O = rto.shape[2]
    es, ea = np.zeros(S, dtype=bool), np.zeros(A, dtype=bool)
    es[np.asarray(model.end_states, dtype=np.int64)] = True
    ea[np.asarray(model.end_actions, dtype=np.int64)] = True
    P, M, G = ext
    N = len(actions)
    nP, nM, nG = np.empty((N, S)), np.empty((N, S)), np.empty((N, S))
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
    return nP, nM, nG


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'hallway', 'tigergrid'])
def test_mixed_outcomes_are_the_numpy_restatement_step_by_step(tag):
    model, gamma, B, pg = extracted_graph(tag)
    m = planted(model)
    mg = random_mixtures(pg, np.random.default_rng(23), max(2, len(pg) // 3))
    es = np.zeros(m.state_count, np.uint8)
    es[np.asarray(m.end_states)] = 1
    ea = np.zeros(m.action_count, np.uint8)
    ref = outcomes_mixed_np(m, mg.actions, mg.successors, mg.mixtures, gamma, 6)
    plain = outcomes_np(m, pg.actions, pg.successors, gamma, 3)                   # the restatement is outcomes_np's without mixtures
    assert all(x.tobytes() == y.tobytes() for x, y in zip(plain, outcomes_mixed_np(m, pg.actions, pg.successors, ([0, 1], [0], [1.0]),
                                                                                     gamma, 3)[-1]))
    q = np.concatenate([m.start_probabilities[None, :], B[:3]])
    for k in (1, 2, 6):
        P, M, G, series = m.device.controller_outcomes_mixed(mg.actions, mg.successors, mg.mixtures, es, ea, gamma, k, q, np.zeros(len(q)))
        for got, want in zip((P, M, G), ref[k - 1]):
            assert got.cpu().numpy().tobytes() == want.tobytes(), (tag, k)
    assert len(m.end_states) > 0


# ---- GPU: PolicyGraph.prune_lp ------------------------------------------------------------------------------------------------------
_sources = {}


def source_graph(tag, source):
    """(model, gamma, beliefs, evaluated PolicyGraph) from from_value_function, improve or a short GapSolver run."""
    from pomdp_pbvi_exploration_b200 import GapSolver, PolicyGraph
    key = (tag, source)
    if key not in _sources:
        model, vf, hist = seeded_solve(tag)
        gamma = fixture_model(tag)[1]
        B = hist.belief_sets[-1].belief_array.cpu().numpy()
        pg, _ = PolicyGraph.from_value_function(model, vf, B)
        pg.evaluate(gamma, eps=1e-9)
        if source == 'improved':
            pg, _ = pg.improve(B, 2)
        elif source == 'gap':
            pg, _, _ = GapSolver(gamma, 0.01, trials=4, max_depth=10, seed=0).solve(model, max_rounds=3)
        _sources[key] = (model, gamma, B, pg)
    return _sources[key]


def probes(model, B, pg, seed):
    rng = np.random.default_rng(seed)
    Rn = rng.random((64, model.state_count)) ** 4
    Rn /= Rn.sum(axis=1, keepdims=True)
    parts = [model.start_probabilities[None, :], B, Rn]
    if pg.witnesses is not None:
        parts.append(pg.witnesses.cpu().numpy())
    return np.concatenate(parts)


@pytest.mark.gpu
@pytest.mark.parametrize('source', ['extracted', 'improved', 'gap'])
@pytest.mark.parametrize('tag', ['tiger', 'grid4x3', 'hallway', 'tigergrid'])
def test_prune_lp_keeps_value_and_certificate(tag, source):
    import torch
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma, B, pg = source_graph(tag, source)
    rows_before = pg.rows.clone()
    P = probes(model, B, pg, 4)
    before = pg.value(P)[0].cpu().numpy()
    pr = pg.prune_lp()
    st = pr.prune_stats
    assert torch.equal(pg.rows, rows_before) and pg.mixtures is None
    assert len(pr) <= len(pg.prune_dominated()) == st['after_dominated'] and st['nodes_after'] == len(pr)
    assert st['nodes_after'] == st['after_dominated'] - (st['lp_counts'][2] - st['failed'])
    assert pr.gamma == pg.gamma
    assert pr.value(P)[0].cpu().numpy().tobytes() == before.tobytes(), tag
    act = torch.as_tensor(pr.actions, dtype=torch.int32, device='cuda')
    succ = torch.as_tensor(pr.successors, dtype=torch.int32, device='cuda')
    assert pr._residual(pr.rows, gamma, act, succ) <= 0.0                     # W <= T_pi' W in the sweep's arithmetic
    if pr.mixtures is not None:
        W = pr.rows.cpu().numpy()
        TW = controller_sweep_np(model, pr.actions, pr.successors, np.concatenate([W, mixture_np(W, pr.mixtures)]), gamma)[:len(pr)]
        assert np.all(W <= TW)
    fresh = PolicyGraph(model, pr.actions, pr.successors, mixtures=pr.mixtures)
    fresh._initial = pr.rows
    _, h = fresh.evaluate(gamma, eps=1e-9)
    assert float(fresh.value(model.start_probabilities)[0][0]) >= float(before[0]) - h.shift
    if not model.end_states:
        H, n = 60, 10000
        G = float(pr.outcomes(H, gamma=gamma).discounted_return[0])
        ret = pr.simulate(n, H, seed=3)
        se = max(ret.std(ddof=1) / np.sqrt(n), 1e-12 * max(1.0, abs(G)))
        assert abs(ret.mean() - G) <= 4 * se, (tag, source, ret.mean(), G, se)


@pytest.mark.gpu
def test_prune_lp_graph_saves_loads_and_rejects_the_graph_solvers(tmp_path):
    from pomdp_pbvi_exploration_b200 import GapSolver, PolicyGraph
    model, gamma, B, pg = source_graph('hallway', 'extracted')
    pr = pg.prune_lp()
    mg = pr if pr.mixtures is not None else random_mixtures(pr, np.random.default_rng(1), 5)
    mg.save(str(tmp_path), 'g')
    back = PolicyGraph.load(str(tmp_path), 'g', model)
    assert back.rows.cpu().numpy().tobytes() == mg.rows.cpu().numpy().tobytes()
    assert np.array_equal(back.successors, mg.successors)
    for a, b in zip(back.mixtures, mg.mixtures):
        assert a.tobytes() == b.tobytes()
    with pytest.raises(ValueError, match='without mixtures'):
        GapSolver(gamma, 0.01, trials=2, max_depth=3, seed=0).solve(model, max_rounds=1, lower=mg)
    with pytest.raises(ValueError, match='without mixtures'):
        mg.improve(B, 1)
    # prune_dominated keeps mixtures valid and the certificate
    pd = mg.prune_dominated()
    assert pd.value(B)[0].cpu().numpy().tobytes() == mg.value(B)[0].cpu().numpy().tobytes()
    if pd.mixtures is not None:
        import torch
        act = torch.as_tensor(pd.actions, dtype=torch.int32, device='cuda')
        succ = torch.as_tensor(pd.successors, dtype=torch.int32, device='cuda')
        assert mg is not pr or pd._residual(pd.rows, gamma, act, succ) <= 0.0
