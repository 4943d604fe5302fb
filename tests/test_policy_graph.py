"""
Finite-state controllers: the controller sweep (pbvi_controller_sweep) and PolicyGraph (extraction, certified evaluation, simulation,
pomdp-solve files).  Checked against
  * pbvi_backup_assemble on the same tuples (bitwise) and NumPy's reductions of the residual;
  * the exact controller values of small models (the (N*S) x (N*S) linear system);
  * the certificate W <= T_pi W in NumPy, and lower <= upper against UpperBound on default (Rbar-start) solves, negative rewards included;
  * the exact V* of tiger.95 and Monte Carlo roll-outs.
"""
import ctypes

import numpy as np
import pytest

from test_upper_bound import MODELS, fib_of, fixture_model, olfactory_solve, seeded_solve, tiger_exact_value

GOLDEN9 = ['tiger', 'grid4x4', 'grid4x4_noloop', 'tigergrid', 'hallway', 'cheese', 'grid4x3', 'cit', 'synth300']


# ---- CPU ------------------------------------------------------------------------------------------------------------------------
def test_controller_sweep_rejects_bad_arguments_without_a_device():
    from pomdp_pbvi_exploration_b200 import _native
    from pomdp_pbvi_exploration_b200.build import build_library
    build_library()
    lib = _native.load_library()
    buf = (ctypes.c_double * 8)()
    p = ctypes.addressof(buf)
    BAD = _native.PBVI_ERR_BAD_ARG
    args = dict(d_in=p, n=2, actions=p, succ=p, out=p)

    def call(**kw):
        a = dict(args, **kw)
        return lib.pbvi_controller_sweep(kw.get('m'), a['d_in'], a['n'], 0.9, a['actions'], a['succ'], a['out'], None, None)
    assert call() == BAD and b'handle is NULL' in lib.pbvi_last_error()
    for name in ('d_in', 'actions', 'succ', 'out'):
        assert call(**{name: None}) == BAD and b'NULL pointer' in lib.pbvi_last_error(), name
    for n in (0, -3):
        assert call(n=n) == BAD and b'n >= 1' in lib.pbvi_last_error(), n


def test_policy_graph_rejects_out_of_range_nodes():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = fixture_model('tiger')                                      # A = 3, O = 2
    PolicyGraph(model, [0, 2], [[0, 1], [1, 1]])
    with pytest.raises(ValueError, match='actions'):
        PolicyGraph(model, [0, 3], [[0, 1], [1, 1]])
    with pytest.raises(ValueError, match='actions'):
        PolicyGraph(model, [-1, 0], [[0, 1], [1, 1]])
    with pytest.raises(ValueError, match='successor'):
        PolicyGraph(model, [0, 1], [[0, 2], [1, 1]])
    with pytest.raises(ValueError, match='successor'):
        PolicyGraph(model, [0, 1], [[0, -1], [1, 1]])
    with pytest.raises(ValueError):
        PolicyGraph(model, [0, 1], [[0, 1, 0], [1, 1, 0]])                # O columns
    with pytest.raises(ValueError):
        PolicyGraph(model, np.zeros(0, int), np.zeros((0, 2), int))


def test_pomdp_solve_files_of_a_three_node_graph(tmp_path):
    import torch
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, _ = fixture_model('tiger')
    pg = PolicyGraph(model, [0, 2, 1], [[1, 2], [0, 0], [2, 1]])
    pg.rows = torch.tensor([[-1.5, 0.1], [10.0, 1.0 / 3.0], [0.0, -2e-300]], dtype=torch.float64)
    pg.save(str(tmp_path), 'g')
    assert (tmp_path / 'g.pg').read_text() == '0 0 1 2\n1 2 0 0\n2 1 2 1\n'
    assert (tmp_path / 'g.alpha').read_text() == ('0\n-1.5 0.10000000000000001\n\n'
                                                  '2\n10 0.33333333333333331\n\n'
                                                  '1\n0 -2.0000000000000001e-300\n\n')


# ---- NumPy references ------------------------------------------------------------------------------------------------------------
def controller_sweep_np(model, actions, succ, W, gamma):
    """One T_pi application in the kernel's order (r ascending inside, then o ascending, one rounding per operation)."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, R = reach.shape
    O = rto.shape[2]
    out = np.empty_like(W)
    for a in np.unique(actions):
        nodes = np.flatnonzero(actions == a)
        acc = None
        for o in range(O):
            nxt = W[succ[nodes, o]]
            inner = None
            for r in range(R):
                prod = rto[:, a, o, r][None, :] * nxt[:, reach[:, a, r]]
                inner = prod if r == 0 else inner + prod
            term = gamma * inner
            acc = term if o == 0 else acc + term
        out[nodes] = rbar[:, a][None, :] + acc
    return out


def controller_exact_np(model, actions, succ, gamma):
    """V_n = Rbar_{a_n} + gamma sum_{o,r} RTO * V_{succ(n,o)}[reach] solved as one (N*S) x (N*S) linear system."""
    reach, rto, rbar = model.reachable_states, model.reachable_transitional_observation_table, model.expected_rewards_table
    S, A, R = reach.shape
    O = rto.shape[2]
    N = len(actions)
    M = np.eye(N * S)
    rhs = np.empty(N * S)
    s = np.arange(S)
    for n in range(N):
        a = int(actions[n])
        rhs[n * S:(n + 1) * S] = rbar[:, a]
        for o in range(O):
            for r in range(R):
                np.add.at(M, (n * S + s, int(succ[n, o]) * S + reach[:, a, r]), -gamma * rto[:, a, o, r])
    return np.linalg.solve(M, rhs).reshape(N, S)


_graphs = {}
_olf_fib = [None]                  # FIB rows of the olfactory model (computed once by olfactory_solve)


def extracted(tag):
    """(model, gamma, value function, explored beliefs, PolicyGraph, history) of the default (Rbar-start) seeded solve of a fixture, or
    of the olfactory FSVI 10 x 100 solve; the graph is evaluated at eps = 1e-9."""
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    if tag not in _graphs:
        if tag == 'olfactory_fsvi':
            model, gamma, _olf_fib[0], vf, hist = olfactory_solve(10, 100, 0)
        else:
            model, vf, hist = seeded_solve(tag)
            gamma = fixture_model(tag)[1]
        B = hist.belief_sets[-1].belief_array.cpu().numpy()
        pg, stats = PolicyGraph.from_value_function(model, vf, B)
        _, h = pg.evaluate(gamma, eps=1e-9)
        _graphs[tag] = (model, gamma, vf, B, pg, h)
    return _graphs[tag]


# ---- GPU: the sweep kernel ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('tag', MODELS)
def test_controller_sweep_is_backup_assemble(tag):
    import torch
    model, gamma = fixture_model(tag)
    dev = model.device
    A, O, S = model.action_count, model.observation_count, model.state_count
    rng = np.random.default_rng(11)
    for N in (1, 7, 300):                                   # 300 tuples: the action-grouped assemble kernel on R = 1 models
        W = rng.normal(size=(N, S)) * 10
        act = rng.integers(0, A, N).astype(np.int32)
        succ = rng.integers(0, N, (N, O)).astype(np.int32)
        Wt = torch.as_tensor(W, device='cuda')
        out, stats = dev.controller_sweep(Wt, gamma, act, succ, want_stats=True)
        want = dev.backup_assemble(Wt, gamma, act, succ)
        got = out.cpu().numpy()
        assert got.tobytes() == want.cpu().numpy().tobytes(), (tag, N)
        d = got - W
        st = stats.cpu().numpy()
        assert st[0] == np.max(d) and st[1] == np.max(W - got) and st[2] == np.max(np.abs(d)), (tag, N, st)
        assert dev.controller_sweep(Wt, gamma, act, succ).cpu().numpy().tobytes() == got.tobytes()
        if model.reachable_state_count == 1:
            assert np.array_equal(got, controller_sweep_np(model, act, succ, W, gamma)), (tag, N)


# ---- GPU: exact evaluation and the certificate -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'grid4x4', 'grid4x4_noloop', 'cheese', 'grid4x3'])
def test_evaluation_matches_the_exact_controller_value(tag):
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model(tag)
    blind = PolicyGraph.blind(model)
    blind.evaluate(gamma, eps=1e-9)
    for pg in (blind, extracted(tag)[4]):
        exact = controller_exact_np(model, pg.actions, pg.successors, gamma)
        rows = pg.rows.cpu().numpy()
        scale = np.maximum(1.0, np.abs(exact))
        assert np.all(rows <= exact + 1e-9 * scale), (tag, len(pg), float(np.max((rows - exact) / scale)))
        assert np.all(rows >= exact - 1e-5 * scale), (tag, len(pg), float(np.min((rows - exact) / scale)))


def check_certificate(model, gamma, pg):
    W = pg.rows.cpu().numpy()
    TW = controller_sweep_np(model, pg.actions, pg.successors, W, gamma)
    assert np.all(W <= TW + 1e-12 * np.maximum(1.0, np.abs(W))), float(np.max(W - TW))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', MODELS)
def test_certificate_holds_on_every_model(tag):
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model(tag)
    blind = PolicyGraph.blind(model)
    _, hist = blind.evaluate(gamma)
    assert hist.sweeps >= 1 and hist.shift >= 0.0 and hist.residual == hist.residual
    check_certificate(model, gamma, blind)
    if tag != 'olfactory_wrap':                             # its solve is the FSVI one below
        _, _, _, _, pg, _ = extracted(tag)
        check_certificate(model, gamma, pg)


@pytest.mark.gpu
def test_certificate_holds_on_the_olfactory_fsvi_solve():
    model, gamma, _, _, pg, hist = extracted('olfactory_fsvi')
    assert len(pg) > 1 and hist.shift >= 0.0
    check_certificate(model, gamma, pg)


@pytest.mark.gpu
def test_non_contracting_model_is_rejected():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model('tiger', rto_scale=1.1)
    with pytest.raises(ValueError, match='contraction'):
        PolicyGraph.blind(model).evaluate(gamma)


# ---- GPU: soundness against the certified upper bound ----------------------------------------------------------------------------
def check_below_upper(model, pg, ub, B):
    import torch
    R = torch.as_tensor(np.concatenate([model.start_probabilities[None, :], B]), device='cuda')
    lower = pg.value(R)[0].cpu().numpy()
    upper = ub.evaluate(R).cpu().numpy()
    assert np.all(lower <= upper + 1e-9 * np.maximum(1.0, np.abs(upper))), float(np.max(lower - upper))
    return lower, upper


@pytest.mark.gpu
@pytest.mark.parametrize('tag', GOLDEN9)
def test_controller_value_below_upper_bound(tag):
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma, vf, B, pg, _ = extracted(tag)
    fib, _ = fib_of(tag)
    ub = UpperBound(model, fib, gamma)
    check_below_upper(model, pg, ub, B)
    ub.improve(B, passes=2)
    check_below_upper(model, pg, ub, B)
    lower, upper = ub.gap(pg.value_function)
    assert lower == float(pg.value(model.start_probabilities)[0][0]) and lower <= upper + 1e-9 * max(1.0, abs(upper))


@pytest.mark.gpu
def test_controller_value_below_upper_bound_on_olfactory_multi_chunk():
    from pomdp_pbvi_exploration_b200 import UpperBound
    model, gamma, _, B, pg, _ = extracted('olfactory_fsvi')
    ub = UpperBound(model, _olf_fib[0], gamma)
    _, up0 = check_below_upper(model, pg, ub, B)
    ub._chunk_bytes = 64 << 20
    assert ub._chunk(len(B)) < len(B) // 4
    n_dec, _ = ub.improve(B)
    assert n_dec > 0
    _, up1 = check_below_upper(model, pg, ub, B)
    assert np.all(up1 <= up0)


# ---- GPU: quality and simulation -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_tiger_controller_is_near_optimal():
    import torch
    from pomdp_pbvi_exploration_b200 import PolicyGraph, ValueFunction
    model, gamma = fixture_model('tiger')
    dev = model.device
    grid = np.linspace(0.0, 1.0, 101)
    B = torch.as_tensor(np.stack([1 - grid, grid], axis=1), device='cuda')
    vf = ValueFunction(model, np.full((1, 2), float(model.expected_rewards_table.min()) / (1 - gamma)), [0])
    prev = None
    for _ in range(5000):
        out, act, _, _ = dev.backup(B, vf.alpha_vector_array, gamma)
        vf = ValueFunction(model, out, act.cpu().numpy())
        val = dev.max_values(B, vf.alpha_vector_array)[0].cpu().numpy()
        if prev is not None and np.max(np.abs(val - prev)) < 1e-12:
            break
        prev = val
    pg, _ = PolicyGraph.from_value_function(model, vf, B)
    pg.evaluate(gamma, eps=1e-10)
    b0 = model.start_probabilities
    got = float(pg.value(b0)[0][0])
    vstar = float(tiger_exact_value(model, gamma, np.array([b0[1]]))[0])
    assert got <= vstar + 1e-9, (got, vstar)
    assert abs(got - vstar) <= 1e-3 * abs(vstar), (got, vstar, len(pg))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['tiger', 'hallway'])
def test_monte_carlo_agrees_with_the_certified_value(tag):
    model, gamma, _, _, pg, hist = extracted(tag)
    rbar_max = float(np.max(np.abs(model.expected_rewards_table)))
    H = int(np.ceil(np.log(1e-6 * (1 - gamma) / rbar_max) / np.log(gamma))) + 1
    assert gamma ** H * rbar_max / (1 - gamma) < 1e-6
    ret = pg.simulate(4000, H, seed=7)
    assert ret.shape == (4000,)
    mean, se = float(ret.mean()), float(ret.std(ddof=1) / np.sqrt(len(ret)))
    v0 = float(pg.value(model.start_probabilities)[0][0])
    assert abs(mean - v0) <= 5 * se + hist.shift, (tag, mean, se, v0, hist.shift)
    assert np.array_equal(ret, pg.simulate(4000, H, seed=7))


@pytest.mark.gpu
def test_simulate_rejects_leaking_rto_rows():
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma = fixture_model('tiger', rto_scale=0.5)
    pg = PolicyGraph.blind(model)
    pg.evaluate(gamma)
    with pytest.raises(ValueError, match='sum to 1'):
        pg.simulate(10, 5, seed=0)


# ---- GPU: structure, determinism, files ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['hallway', 'olfactory_fsvi'])
def test_extraction_structure_and_determinism(tag):
    import torch
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma, vf, B, pg, _ = extracted(tag)
    dev = model.device
    rows = vf.alpha_vector_array
    N = len(pg)
    assert 1 <= N <= len(vf)
    assert pg.successors.min() >= 0 and pg.successors.max() < N
    assert len(set(pg.source_rows.tolist())) == N
    assert np.array_equal(pg.actions, vf.actions[pg.source_rows])
    assert int(dev.max_values(model.start_probabilities, rows)[1][0]) == pg.source_rows[0]
    best, _ = dev.max_values(pg.witnesses, rows)
    own = (pg.witnesses * rows[torch.as_tensor(pg.source_rows, device=rows.device)]).sum(dim=1)
    best, own = best.cpu().numpy(), own.cpu().numpy()
    assert np.all(own >= best - 1e-9 * np.maximum(1.0, np.abs(best))), float(np.max(best - own))
    pg2, _ = PolicyGraph.from_value_function(model, vf, B)
    pg2.evaluate(gamma, eps=1e-9)
    assert np.array_equal(pg.actions, pg2.actions) and np.array_equal(pg.successors, pg2.successors)
    assert pg.rows.cpu().numpy().tobytes() == pg2.rows.cpu().numpy().tobytes()


@pytest.mark.gpu
def test_save_load_round_trip(tmp_path):
    from pomdp_pbvi_exploration_b200 import PolicyGraph
    model, gamma, _, _, pg, _ = extracted('hallway')
    pg.save(str(tmp_path), 'hallway')
    back = PolicyGraph.load(str(tmp_path), 'hallway', model)
    assert np.array_equal(back.actions, pg.actions) and np.array_equal(back.successors, pg.successors)
    assert back.rows.cpu().numpy().tobytes() == pg.rows.cpu().numpy().tobytes()


@pytest.mark.gpu
def test_extraction_rejects_non_finite_input():
    from pomdp_pbvi_exploration_b200 import PolicyGraph, ValueFunction
    model, _ = fixture_model('tiger')
    with pytest.raises(ValueError):
        PolicyGraph.from_value_function(model, ValueFunction(model, np.array([[0.0, np.inf]]), [0]))
    with pytest.raises(ValueError):
        PolicyGraph.from_value_function(model, ValueFunction(model, np.array([[0.0, 1.0]]), [0]), np.array([[0.5, np.nan]]))
